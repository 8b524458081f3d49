// api.cu -- host side of the C ABI declared in include/nadavca_b200.h: model tables, resident batches, wave
// planning (how many reads' DP matrices fit in HBM at once) and kernel orchestration.  No CPU compute path.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/nadavca_b200.h"
#include "kernels.h"

namespace {

thread_local std::string g_err;
thread_local int g_code = 0;  // code of the last failure on this thread (what the one-shot calls return)

int g_sweep = NVB_SWEEP_AUTO;  // sweep schedule, set by nvb_set_sweep_schedule (tests force both schedules through it)

int fail(int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  g_code = code;
  return code;
}

#define CU(expr)                                                                                      \
  do {                                                                                                \
    cudaError_t _e = (expr);                                                                          \
    if (_e != cudaSuccess)                                                                            \
      return fail(NVB_ECUDA, "CUDA error %s at %s:%d (%s)", cudaGetErrorString(_e), __FILE__, __LINE__, #expr); \
  } while (0)

// Device memory comes from a per-device cache of freed blocks: cudaFree of the ~20 buffers of a batch costs hundreds
// of milliseconds on this driver (measured: 280-650 ms per nvb_batch_destroy of a 1000-read batch), far more than the
// kernels of the batch.  Blocks are handed back to the driver only by nvb_trim_memory() or when an allocation fails.
struct DevicePool {
  std::mutex m;
  std::multimap<size_t, void *> free_blocks;
  size_t cached = 0;
};
DevicePool g_pool[64];

void pool_trim(int device) {
  DevicePool &P = g_pool[device & 63];
  std::lock_guard<std::mutex> lock(P.m);
  for (auto &kv : P.free_blocks) cudaFree(kv.second);
  P.free_blocks.clear();
  P.cached = 0;
}

cudaError_t pool_alloc(void **out, size_t bytes, size_t *capacity, int *device) {
  bytes = (std::max<size_t>(bytes, 1) + 511) & ~(size_t)511;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  *device = dev;
  DevicePool &P = g_pool[dev & 63];
  {
    std::lock_guard<std::mutex> lock(P.m);
    auto it = P.free_blocks.lower_bound(bytes);
    if (it != P.free_blocks.end() && it->first <= bytes + bytes / 4 + (1 << 20)) {
      *out = it->second; *capacity = it->first;
      P.cached -= it->first;
      P.free_blocks.erase(it);
      return cudaSuccess;
    }
  }
  e = cudaMalloc(out, bytes);
  if (e != cudaSuccess) {  // give the cached blocks back and retry once
    cudaGetLastError();
    pool_trim(dev);
    e = cudaMalloc(out, bytes);
  }
  *capacity = bytes;
  return e;
}

void pool_free(void *p, size_t capacity, int device) {
  DevicePool &P = g_pool[device & 63];
  std::lock_guard<std::mutex> lock(P.m);
  P.free_blocks.emplace(capacity, p);
  P.cached += capacity;
}

template <class T>
struct DevBuf {
  T *p = nullptr;
  size_t n = 0;         // elements requested
  size_t capacity = 0;  // bytes of the block
  int device = 0;
  // `owner`: the stream whose kernels may still be reading the current block.  A block that is outgrown goes back to
  // the per-device cache, where any other stream may pick it up, so the owner is drained first (growth is rare: the
  // workspaces only ever grow).
  cudaError_t alloc(size_t count, cudaStream_t owner = nullptr, bool drain = false) {
    if (p && count * sizeof(T) <= capacity) { n = std::max(n, count); return cudaSuccess; }
    if (p && drain) cudaStreamSynchronize(owner);
    release();
    cudaError_t e = pool_alloc((void **)&p, count * sizeof(T), &capacity, &device);
    if (e == cudaSuccess) n = count; else { p = nullptr; capacity = 0; }
    return e;
  }
  void release() {
    if (p) pool_free(p, capacity, device);
    p = nullptr; n = 0; capacity = 0;
  }
  ~DevBuf() { release(); }
};

template <class T>
cudaError_t upload(DevBuf<T> &buf, const T *src, size_t count, cudaStream_t st) {
  cudaError_t e = buf.alloc(count);
  if (e != cudaSuccess) return e;
  if (count == 0) return cudaSuccess;
  return cudaMemcpyAsync(buf.p, src, count * sizeof(T), cudaMemcpyHostToDevice, st);
}

}  // namespace

// DP workspace: owned by the model, ONE PER STREAM, shared by all batches of the model that run on that stream
// (allocating and freeing several GB per batch costs tens of milliseconds per call); it only ever grows and is released
// with the model.  Runs on the same stream are ordered by the stream, runs on different streams never share a
// workspace, so batches of one model may be in flight on several streams at once.
struct Workspace {
  DevBuf<double> pF, sF, dp;   // DP matrices: mantissa planes; path-search scratch rows
  DevBuf<int32_t> pX, sX;      // ... and exponent planes
  DevBuf<uint32_t> records;    // path search: one "new row record" bit per cell (path2.cu)
  DevBuf<double> handoff;      // striped sweep: hand-off rows of band rows too wide for shared memory (rows4.cu)
  size_t bytes() const {
    return pF.capacity + sF.capacity + dp.capacity + pX.capacity + sX.capacity + records.capacity + handoff.capacity;
  }
};

struct nvb_model {
  int device = 0;
  int sm_count = 148;
  ModelDev dev{};
  DevBuf<double> mean, ac, mc;
  mutable std::mutex ws_mutex;
  std::map<cudaStream_t, Workspace> ws;  // std::map: references stay valid while other streams add theirs
  Workspace &workspace(cudaStream_t st) {
    std::lock_guard<std::mutex> lock(ws_mutex);
    return ws[st];
  }
  size_t workspace_bytes() const {
    std::lock_guard<std::mutex> lock(ws_mutex);
    size_t total = 0;
    for (auto &kv : ws) total += kv.second.bytes();
    return total;
  }
};

struct Wave { int b0, b1; int64_t cells; int maxw; };

struct nvb_batch {
  nvb_model *model = nullptr;
  int n_reads = 0;
  int64_t total_ref = 0, total_sig = 0;
  std::vector<int64_t> sig_off, ref_off, ctxb_off, ctxa_off, anc_off;
  // device inputs
  DevBuf<double> d_signal;
  DevBuf<int64_t> d_sig_off, d_ref_off, d_ctxb_off, d_ctxa_off, d_anc_off;
  DevBuf<int32_t> d_ref, d_ctxb, d_ctxa, d_anchors;
  // band geometry
  DevBuf<int32_t> d_bs, d_be, d_flags, d_maxw;
  DevBuf<double> d_row_emis;   // BatchDev::row_emis
  DevBuf<int64_t> d_cell_off, d_summary;
  std::vector<int64_t> cells, w0, wn;  // per read: sum of widths over n+1 band rows, first / last width
  std::vector<int32_t> maxw, flags, no_rotation;  // no_rotation: the read needs the striped sweep (rows4.cu)
  // results
  DevBuf<int32_t> d_events, d_status;
  DevBuf<double> d_ll;
  bool have_events = false, have_ll = false;
  // small per-read arrays of the post-processing calls, kept on the device so that those calls need no
  // synchronisation (re-uploaded only when the host values change)
  DevBuf<int32_t> d_rev;
  DevBuf<int64_t> d_dest;
  std::vector<int32_t> h_rev;
  std::vector<int64_t> h_dest;
  // per-read offsets into the model's DP workspace, valid for the last run
  DevBuf<int64_t> d_mat_base, d_dp_base, d_rec_base;
  int64_t ws_limit = 0;
  int64_t launches = 0;
  int path_pk = 11;  // columns per lane of the path search (path2.cu), from the widest band row of the batch
  // Streams this batch has work on.  Results are read back on `run_stream` (the stream of the latest run); destroying
  // the batch drains every stream that may still be using its buffers -- never the whole device.
  cudaStream_t run_stream = nullptr;
  std::vector<cudaStream_t> streams_used;
  Workspace *last_ws = nullptr;  // workspace of the latest run (nvb_batch_debug_rows)
  void touch(cudaStream_t st) {
    run_stream = st;
    if (std::find(streams_used.begin(), streams_used.end(), st) == streams_used.end()) streams_used.push_back(st);
  }
  void drain() {
    for (cudaStream_t st : streams_used) cudaStreamSynchronize(st);
  }
  // plan of the last run (see prepare_workspace)
  int plan_mode = -1;
  bool plan_dp = false;
  int64_t plan_limit = -1;
  int64_t plan_max[3] = {0, 0, 0};
  std::vector<Wave> plan_waves_cache;
  BatchDev dev{};
  // optional per-stage timing
  bool timing = false;
  std::vector<std::pair<int, std::pair<cudaEvent_t, cudaEvent_t>>> timed;  // (stage, (start, stop))
  ~nvb_batch() {
    for (auto &t : timed) { cudaEventDestroy(t.second.first); cudaEventDestroy(t.second.second); }
  }
};

namespace {
// RAII helper: records a start/stop event pair around one kernel launch when timing is enabled
struct StageTimer {
  nvb_batch *b; cudaStream_t st; cudaEvent_t e0 = nullptr, e1 = nullptr; int stage;
  StageTimer(nvb_batch *batch, int stage_, cudaStream_t stream) : b(batch), st(stream), stage(stage_) {
    if (b->timing) { cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventRecord(e0, st); }
  }
  ~StageTimer() {
    if (b->timing) { cudaEventRecord(e1, st); b->timed.push_back({stage, {e0, e1}}); }
  }
};
}  // namespace

extern "C" {

int nvb_abi_version(void) { return 1; }

const char *nvb_last_error(void) { return g_err.c_str(); }

int nvb_set_sweep_schedule(int schedule) {
  const int before = g_sweep;
  if (schedule == NVB_SWEEP_AUTO || schedule == NVB_SWEEP_ROTATE || schedule == NVB_SWEEP_STRIPES) g_sweep = schedule;
  return before;
}

int nvb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

nvb_model *nvb_model_create(int k, int central_position, int alphabet_size, const double *mean,
                            const double *sigma, int64_t n_kmers, int device) {
  if (k <= 0 || alphabet_size < 2 || central_position < 0 || central_position >= k || !mean || !sigma) {
    fail(NVB_EINVAL, "nvb_model_create: bad arguments");
    return nullptr;
  }
  int64_t expect = 1;
  for (int i = 0; i < k; i++) expect *= alphabet_size;
  if (n_kmers != expect) {
    fail(NVB_EINVAL, "nvb_model_create: expected %lld k-mers, got %lld", (long long)expect, (long long)n_kmers);
    return nullptr;
  }
  if (nvb_device_count() <= device || device < 0) {
    fail(NVB_ECUDA, "nvb_model_create: CUDA device %d not available (no CPU fallback)", device);
    return nullptr;
  }
  if (cudaSetDevice(device) != cudaSuccess) { fail(NVB_ECUDA, "cudaSetDevice(%d) failed", device); return nullptr; }
  nvb_model *m = new nvb_model();
  m->device = device;
  {
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0) m->sm_count = sms;
  }
  std::vector<double> ac(n_kmers), mc(n_kmers);
  for (int64_t i = 0; i < n_kmers; i++) {  // same expressions as kmer_model.cpp:10-13, host libm
    double s = sigma[i];
    ac[i] = log(1 / sqrt(2 * M_PI * s * s));
    mc[i] = 1 / (2 * s * s);
  }
  if (upload(m->mean, mean, (size_t)n_kmers, 0) != cudaSuccess || upload(m->ac, ac.data(), (size_t)n_kmers, 0) != cudaSuccess ||
      upload(m->mc, mc.data(), (size_t)n_kmers, 0) != cudaSuccess || cudaStreamSynchronize(0) != cudaSuccess) {
    fail(NVB_ECUDA, "nvb_model_create: upload failed: %s", cudaGetErrorString(cudaGetLastError()));
    delete m;
    return nullptr;
  }
  m->dev.k = k; m->dev.central = central_position; m->dev.alphabet = alphabet_size; m->dev.n_kmers = n_kmers;
  m->dev.mean = m->mean.p; m->dev.ac = m->ac.p; m->dev.mc = m->mc.p;
  return m;
}

void nvb_model_destroy(nvb_model *model) {
  if (!model) return;
  const int device = model->device;
  cudaSetDevice(device);
  cudaDeviceSynchronize();
  delete model;
  // its workspaces (often several GB) went to the block cache: hand them back to the driver, other allocators
  // (torch) may need the memory
  pool_trim(device);
}

int nvb_model_k(const nvb_model *m) { return m ? m->dev.k : 0; }
int nvb_model_central_position(const nvb_model *m) { return m ? m->dev.central : 0; }
int nvb_model_alphabet_size(const nvb_model *m) { return m ? m->dev.alphabet : 0; }
int64_t nvb_model_workspace_bytes(const nvb_model *m) { return m ? (int64_t)m->workspace_bytes() : 0; }

}  // extern "C"

namespace {

int check_offsets(const int64_t *off, int n, const char *what) {
  if (!off) return fail(NVB_EINVAL, "%s offsets are NULL", what);
  if (off[0] != 0) return fail(NVB_EINVAL, "%s offsets must start at 0", what);
  for (int i = 0; i < n; i++)
    if (off[i + 1] < off[i]) return fail(NVB_EINVAL, "%s offsets are not monotone at read %d", what, i);
  return NVB_OK;
}

// Upload the sequence part of a batch (reference + contexts); enough for expected_signal.
int upload_sequences(nvb_batch *b, int n_reads, const int32_t *reference, const int64_t *reference_off,
                     const int32_t *cb, const int64_t *cb_off, const int32_t *ca, const int64_t *ca_off,
                     cudaStream_t st) {
  int rc;
  if ((rc = check_offsets(reference_off, n_reads, "reference"))) return rc;
  if ((rc = check_offsets(cb_off, n_reads, "context_before"))) return rc;
  if ((rc = check_offsets(ca_off, n_reads, "context_after"))) return rc;
  b->n_reads = n_reads;
  b->ref_off.assign(reference_off, reference_off + n_reads + 1);
  b->ctxb_off.assign(cb_off, cb_off + n_reads + 1);
  b->ctxa_off.assign(ca_off, ca_off + n_reads + 1);
  b->total_ref = b->ref_off[n_reads];
  const int A = b->model->dev.alphabet;
  for (int64_t i = 0; i < b->total_ref; i++)
    if (reference[i] < 0 || reference[i] >= A) return fail(NVB_EINVAL, "reference base %d out of range at %lld", reference[i], (long long)i);
  for (int64_t i = 0; i < b->ctxb_off[n_reads]; i++)
    if (cb[i] < 0 || cb[i] >= A) return fail(NVB_EINVAL, "context_before base out of range");
  for (int64_t i = 0; i < b->ctxa_off[n_reads]; i++)
    if (ca[i] < 0 || ca[i] >= A) return fail(NVB_EINVAL, "context_after base out of range");
  CU(upload(b->d_ref, reference, (size_t)b->total_ref, st));
  CU(upload(b->d_ref_off, reference_off, (size_t)n_reads + 1, st));
  CU(upload(b->d_ctxb, cb, (size_t)b->ctxb_off[n_reads], st));
  CU(upload(b->d_ctxb_off, cb_off, (size_t)n_reads + 1, st));
  CU(upload(b->d_ctxa, ca, (size_t)b->ctxa_off[n_reads], st));
  CU(upload(b->d_ctxa_off, ca_off, (size_t)n_reads + 1, st));
  b->dev.n_reads = n_reads;
  b->dev.ref = b->d_ref.p; b->dev.ref_off = b->d_ref_off.p;
  b->dev.ctxb = b->d_ctxb.p; b->dev.ctxb_off = b->d_ctxb_off.p;
  b->dev.ctxa = b->d_ctxa.p; b->dev.ctxa_off = b->d_ctxa_off.p;
  return NVB_OK;
}

int batch_init(nvb_batch *b, const nvb_reads *r) {
  cudaStream_t st = 0;
  const int n = r->n_reads;
  int rc;
  if (n < 0) return fail(NVB_EINVAL, "n_reads < 0");
  if (r->bandwidth < 0 || r->min_event_length < 0) return fail(NVB_EINVAL, "bandwidth / min_event_length must be >= 0");
  if (r->min_event_length > 6) return fail(NVB_EINVAL, "min_event_length > 6 is not supported");
  if ((rc = check_offsets(r->signal_off, n, "signal"))) return rc;
  if ((rc = check_offsets(r->anchor_off, n, "anchor"))) return rc;
  if ((rc = upload_sequences(b, n, r->reference, r->reference_off, r->context_before, r->context_before_off,
                             r->context_after, r->context_after_off, st)))
    return rc;
  b->sig_off.assign(r->signal_off, r->signal_off + n + 1);
  b->anc_off.assign(r->anchor_off, r->anchor_off + n + 1);
  b->total_sig = b->sig_off[n];
  for (int i = 0; i < n; i++) {
    if (b->sig_off[i + 1] - b->sig_off[i] > 0x7fffff00LL) return fail(NVB_EINVAL, "signal of read %d too long", i);
    if (b->ref_off[i + 1] - b->ref_off[i] > 0x3fffff00LL) return fail(NVB_EINVAL, "reference of read %d too long", i);
  }
  CU(upload(b->d_signal, r->signal, (size_t)b->total_sig, st));
  CU(upload(b->d_sig_off, r->signal_off, (size_t)n + 1, st));
  CU(upload(b->d_anchors, r->anchors, (size_t)b->anc_off[n] * 2, st));
  CU(upload(b->d_anc_off, r->anchor_off, (size_t)n + 1, st));
  CU(b->d_bs.alloc((size_t)b->total_ref + n));
  CU(b->d_be.alloc((size_t)b->total_ref + n));
  CU(b->d_cell_off.alloc((size_t)b->total_ref + 2 * (size_t)n));
  CU(b->d_flags.alloc(n));
  CU(b->d_maxw.alloc(n));
  CU(b->d_summary.alloc((size_t)4 * n));
  CU(b->d_status.alloc(n));
  BatchDev &d = b->dev;
  d.signal = b->d_signal.p; d.sig_off = b->d_sig_off.p;
  d.anchors = b->d_anchors.p; d.anc_off = b->d_anc_off.p;
  d.bandwidth = r->bandwidth; d.mel = r->min_event_length;
  d.bs = b->d_bs.p; d.be = b->d_be.p; d.cell_off = b->d_cell_off.p;
  d.flags = b->d_flags.p; d.max_width = b->d_maxw.p;
  CU(b->d_row_emis.alloc((size_t)4 * std::max<int64_t>(b->total_ref, 1)));
  d.row_emis = b->d_row_emis.p;
  nvbk_band(d, b->d_summary.p, st);
  nvbk_row_emission(b->model->dev, d, b->total_ref, nvbk_emission_scale(), b->d_row_emis.p, st);
  b->launches += 2;
  CU(cudaGetLastError());
  std::vector<int64_t> summary((size_t)4 * n);
  CU(cudaMemcpyAsync(summary.data(), b->d_summary.p, summary.size() * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  b->cells.resize(n); b->w0.resize(n); b->wn.resize(n); b->maxw.resize(n); b->flags.resize(n); b->no_rotation.resize(n);
  for (int i = 0; i < n; i++) {
    b->cells[i] = summary[4 * i];
    b->w0[i] = summary[4 * i + 1];
    b->wn[i] = summary[4 * i + 2];
    b->maxw[i] = (int32_t)(summary[4 * i + 3] & 0xffffffffLL);
    b->flags[i] = ((summary[4 * i + 3] >> 32) & 1) ? NVB_READ_BAD_BAND : 0;
    b->no_rotation[i] = (int32_t)((summary[4 * i + 3] >> 33) & 1);
  }
  int widest = 0;
  for (int i = 0; i < n; i++)
    if (!b->flags[i]) widest = std::max(widest, (int)b->maxw[i]);
  b->path_pk = nvbk_path2_columns_per_lane(widest);
  return NVB_OK;
}

// Forward + backward rows of one wave: the rotating wavefront (rows5.cu) when every read of the wave allows it, else
// the pipelined stripes (rows4.cu).
int run_sweep(nvb_batch *b, Workspace &ws, int mode, const Wave &w, cudaStream_t st) {
  const ModelDev &M = b->model->dev;
  // Measured on B200 (profiles/r02y_sweep_schedules.txt, 32 .. 2000 reads): since the round-2 work on its step loop the
  // rotating wavefront wins at every batch size and in every mode (one read: 7.3 against 10.8 ms for the plain sweep;
  // 1000 reads: 13.2 / 29.2 / 16.4 ms against 23.7 / 30.7 / 27.3 ms plain / transitions / wobble), so it runs whenever
  // the band rows fit its signal window (640 columns) and the band kernel found no read that needs a third slot; the
  // striped sweep keeps the wide and the irregular bands.  One exception: band rows wider than the 352 steps a lane has
  // per row pair keep the second slot of every lane busy (two step bodies per step); then the stripes are faster for
  // the transition and wobble sweeps of SMALL batches (64 reads, band 200: 13.6 / 12.3 ms against 17.6 / 13.2 ms), the
  // rotation still for large ones (512 reads: 22.2 / 17.4 ms against 27.2 / 24.5 ms).
  const int items = 2 * (w.b1 - w.b0);
  const int resident = b->model->sm_count * 16;  // sweep warps of one resident wave
  bool rotate = w.maxw <= 640 && (w.maxw <= 352 || mode == NVB_MODE_PLAIN || 4 * items >= resident);
  if (g_sweep != NVB_SWEEP_AUTO) rotate = w.maxw <= 640 && g_sweep == NVB_SWEEP_ROTATE;
  for (int i = w.b0; i < w.b1 && rotate; i++) rotate = !b->no_rotation[i];
  if (rotate)
    return nvbk_sweep_rotate(M, b->dev, mode, w.b0, w.b1, b->d_mat_base.p, ws.pF.p, ws.pX.p, ws.sF.p, ws.sX.p, st);
  // band rows too wide for the shared-memory hand-off rows of the striped sweep go through global scratch rows
  const int64_t need = nvbk_sweep2_global_handoff_doubles(mode, w.b1 - w.b0, w.maxw);
  if (need > 0 && ws.handoff.alloc((size_t)need, st, true) != cudaSuccess) { cudaGetLastError(); return -2; }
  return nvbk_sweep2(M, b->dev, mode, w.b0, w.b1, w.maxw, b->d_mat_base.p, ws.pF.p, ws.pX.p, ws.sF.p, ws.sX.p,
                     need > 0 ? ws.handoff.p : nullptr, st);
}

int64_t matrix_cells(const nvb_batch *b, int i, int mode) {
  if (b->flags[i]) return 0;
  if (mode == NVB_MODE_TRANS) return 2 * b->cells[i] - b->w0[i] - b->wn[i];
  return b->cells[i];
}


// 32-bit words of record bits the path search keeps for read i (path2.cu): rows x chunks x 32
int64_t record_words(const nvb_batch *b, int i, int mode) {
  if (b->flags[i]) return 0;
  const int64_t n = b->ref_off[i + 1] - b->ref_off[i];
  const int64_t rows = (mode == NVB_MODE_TRANS) ? 2 * n : n + 1;
  const int chunk = 32 * b->path_pk;
  const int64_t nch = (b->maxw[i] + chunk - 1) / chunk;
  return rows * nch * 32;
}

// Split the batch into waves of consecutive reads whose two DP matrices (+ path scratch) fit the workspace limit.
int plan_waves(nvb_batch *b, const Workspace &ws, int mode, bool need_dp, std::vector<Wave> &waves, std::vector<int64_t> &mat_base,
               std::vector<int64_t> &dp_base, std::vector<int64_t> &rec_base, int64_t &max_cells, int64_t &max_dp,
               int64_t &max_rec) {
  int64_t limit = b->ws_limit;
  const int n = b->n_reads;
  if (limit <= 0) {
    // When the whole batch fits the workspace the model already owns, nothing has to be asked of the driver
    // (cudaMemGetInfo costs milliseconds); otherwise plan against 70 % of what is free plus what is already held.
    int64_t cells = 0, dp = 0, rec = 0;
    for (int j = 0; j < n; j++) {
      cells += matrix_cells(b, j, mode);
      if (need_dp) { dp += 2 * (int64_t)b->maxw[j]; rec += record_words(b, j, mode); }
    }
    const bool fits = (size_t)cells * sizeof(double) <= ws.pF.capacity && (size_t)cells * sizeof(double) <= ws.sF.capacity &&
                      (size_t)cells * sizeof(int32_t) <= ws.pX.capacity && (size_t)cells * sizeof(int32_t) <= ws.sX.capacity &&
                      (size_t)dp * sizeof(double) <= ws.dp.capacity && (size_t)rec * sizeof(uint32_t) <= ws.records.capacity;
    if (fits) {
      limit = INT64_MAX;
    } else {
      size_t free_b = 0, total_b = 0;
      CU(cudaMemGetInfo(&free_b, &total_b));
      free_b += ws.bytes();  // what this stream's workspace already holds can be re-used
      limit = (int64_t)(free_b * 0.7);
    }
  }
  mat_base.assign(n, 0); dp_base.assign(n, 0); rec_base.assign(n, 0);
  waves.clear();
  max_cells = 0; max_dp = 0; max_rec = 0;
  int i = 0;
  while (i < n) {
    int64_t cells = 0, dp = 0, rec = 0;
    int maxw = 0;
    int j = i;
    while (j < n) {
      const int64_t c = matrix_cells(b, j, mode), d = need_dp ? 2 * (int64_t)b->maxw[j] : 0;
      const int64_t rw = need_dp ? record_words(b, j, mode) : 0;
      const int64_t bytes = (cells + c) * 2 * (int64_t)(sizeof(double) + sizeof(int32_t)) +
                            (dp + d) * (int64_t)sizeof(double) + (rec + rw) * (int64_t)sizeof(uint32_t);
      if (bytes > limit && j > i) break;
      if (bytes > limit)
        return fail(NVB_ENOMEM, "read %d needs %lld bytes of DP workspace, limit is %lld", j, (long long)bytes, (long long)limit);
      mat_base[j] = cells; dp_base[j] = dp; rec_base[j] = rec;
      cells += c; dp += d; rec += rw;
      if (!b->flags[j]) maxw = std::max(maxw, (int)b->maxw[j]);
      j++;
    }
    waves.push_back({i, j, cells, maxw});
    max_cells = std::max(max_cells, cells);
    max_dp = std::max(max_dp, dp);
    max_rec = std::max(max_rec, rec);
    i = j;
  }
  return NVB_OK;
}

int prepare_workspace(nvb_batch *b, Workspace &ws, int mode, bool need_dp, std::vector<Wave> &waves, cudaStream_t st) {
  std::vector<int64_t> mat_base, dp_base, rec_base;
  int64_t max_cells = 0, max_dp = 0, max_rec = 0;
  // The plan of the previous run is kept: repeating a run needs no host planning, no uploads and no synchronisation,
  // so consecutive runs queue back to back on the stream.
  const bool cached = b->plan_mode == mode && b->plan_dp == need_dp && b->plan_limit == b->ws_limit;
  if (cached) {
    waves = b->plan_waves_cache;
    max_cells = b->plan_max[0]; max_dp = b->plan_max[1]; max_rec = b->plan_max[2];
  } else {
    int rc = plan_waves(b, ws, mode, need_dp, waves, mat_base, dp_base, rec_base, max_cells, max_dp, max_rec);
    if (rc) return rc;
  }
  if (ws.pF.alloc((size_t)max_cells, st, true) != cudaSuccess || ws.sF.alloc((size_t)max_cells, st, true) != cudaSuccess ||
      ws.pX.alloc((size_t)max_cells, st, true) != cudaSuccess || ws.sX.alloc((size_t)max_cells, st, true) != cudaSuccess ||
      ws.dp.alloc((size_t)max_dp, st, true) != cudaSuccess || ws.records.alloc((size_t)max_rec, st, true) != cudaSuccess) {
    cudaGetLastError();
    return fail(NVB_ENOMEM, "cannot allocate %lld bytes of DP workspace",
                (long long)(24 * max_cells + 8 * max_dp + 4 * max_rec));
  }
  if (cached) return NVB_OK;
  CU(upload(b->d_mat_base, mat_base.data(), mat_base.size(), st));
  CU(upload(b->d_dp_base, dp_base.data(), dp_base.size(), st));
  CU(upload(b->d_rec_base, rec_base.data(), rec_base.size(), st));
  // pageable-host uploads above are complete when cudaMemcpyAsync returns only for small sizes; be explicit:
  CU(cudaStreamSynchronize(st));
  b->plan_mode = mode; b->plan_dp = need_dp; b->plan_limit = b->ws_limit;
  b->plan_waves_cache = waves;
  b->plan_max[0] = max_cells; b->plan_max[1] = max_dp; b->plan_max[2] = max_rec;
  return NVB_OK;
}

}  // namespace

extern "C" {

nvb_batch *nvb_batch_create(nvb_model *model, const nvb_reads *reads) {
  g_code = 0;
  if (!model || !reads) { fail(NVB_EINVAL, "nvb_batch_create: NULL argument"); return nullptr; }
  if (cudaSetDevice(model->device) != cudaSuccess) { fail(NVB_ECUDA, "cudaSetDevice failed"); return nullptr; }
  nvb_batch *b = new nvb_batch();
  b->model = model;
  if (batch_init(b, reads) != NVB_OK) { delete b; return nullptr; }
  return b;
}

void nvb_batch_destroy(nvb_batch *batch) {
  if (!batch) return;
  cudaSetDevice(batch->model->device);
  batch->drain();  // its blocks go back to the cache: nothing on the streams it ran on may still be using them
  delete batch;
}

int nvb_trim_memory(int device) {
  if (nvb_device_count() <= device || device < 0) return fail(NVB_ECUDA, "CUDA device %d not available", device);
  CU(cudaSetDevice(device));
  CU(cudaDeviceSynchronize());
  pool_trim(device);
  return NVB_OK;
}

int nvb_batch_set_workspace_limit(nvb_batch *b, int64_t bytes) {
  if (!b) return fail(NVB_EINVAL, "NULL batch");
  b->ws_limit = bytes;
  return NVB_OK;
}

int nvb_batch_refine(nvb_batch *b, int model_transitions, void *stream) {
  if (!b) return fail(NVB_EINVAL, "NULL batch");
  CU(cudaSetDevice(b->model->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int mode = model_transitions ? NVB_MODE_TRANS : NVB_MODE_PLAIN;
  std::vector<Wave> waves;
  Workspace &ws = b->model->workspace(st);
  b->touch(st);
  b->last_ws = &ws;
  int rc = prepare_workspace(b, ws, mode, true, waves, st);
  if (rc) return rc;
  CU(b->d_events.alloc((size_t)2 * b->total_ref, st, true));
  for (const Wave &w : waves) {
    {
      StageTimer t(b, 0, st);
      const int src = run_sweep(b, ws, mode, w, st);
      if (src == -1) return fail(NVB_EINVAL, "min_event_length %d is not supported (maximum 6)", b->dev.mel);
      if (src) return fail(NVB_ENOMEM, "cannot allocate the hand-off rows of the sweep for a band row of %d columns", w.maxw);
    }
    {
      StageTimer t(b, 1, st);
      nvbk_score(w.cells, ws.pF.p, ws.pX.p, ws.sF.p, ws.sX.p, st);
      if (nvbk_path2(b->dev, mode, w.b0, w.b1, b->path_pk, b->d_mat_base.p, ws.pF.p, ws.records.p, b->d_rec_base.p,
                     ws.dp.p, b->d_dp_base.p, w.maxw, b->d_events.p, b->d_status.p, st))
        return fail(NVB_ECUDA, "path kernel: cannot reserve shared memory");
    }
    b->launches += 3;
  }
  CU(cudaGetLastError());
  b->have_events = true;
  return NVB_OK;
}

int nvb_batch_estimate(nvb_batch *b, int model_wobbling, void *stream) {
  if (!b) return fail(NVB_EINVAL, "NULL batch");
  CU(cudaSetDevice(b->model->device));
  cudaStream_t st = (cudaStream_t)stream;
  const ModelDev &M = b->model->dev;
  const int mode = model_wobbling ? NVB_MODE_WOBBLE : NVB_MODE_PLAIN;
  if (M.k + 2 > 32) return fail(NVB_EINVAL, "k = %d is too large for the SNP kernel (needs k+2 <= 32 lanes)", M.k);
  std::vector<Wave> waves;
  Workspace &ws = b->model->workspace(st);
  b->touch(st);
  b->last_ws = &ws;
  int rc = prepare_workspace(b, ws, mode, false, waves, st);
  if (rc) return rc;
  CU(b->d_ll.alloc((size_t)b->total_ref * M.alphabet, st, true));
  nvbk_fill_status(b->dev, b->d_status.p, b->d_ll.p, M.alphabet, st);
  b->launches++;
  for (const Wave &w : waves) {
    {
      StageTimer t(b, 0, st);
      const int src = run_sweep(b, ws, mode, w, st);
      if (src == -1) return fail(NVB_EINVAL, "min_event_length %d is not supported (maximum 6)", b->dev.mel);
      if (src) return fail(NVB_ENOMEM, "cannot allocate the hand-off rows of the sweep for a band row of %d columns", w.maxw);
    }
    {
      StageTimer t(b, 2, st);
      nvbk_no_snp2(M, b->dev, w.b0, w.b1, b->d_mat_base.p, ws.pF.p, ws.pX.p, ws.sF.p, ws.sX.p, b->d_ll.p, st);
    }
    int snp_rc;
    {
      StageTimer t(b, 3, st);
      snp_rc = nvbk_snp2(M, b->dev, model_wobbling, w.b0, w.b1, b->ref_off[w.b0], b->ref_off[w.b1],
                         b->d_mat_base.p, ws.pF.p, ws.pX.p, ws.sF.p, ws.sX.p, b->d_ll.p, st);
    }
    if (snp_rc) return fail(NVB_EINVAL, "SNP kernel configuration not supported");
    b->launches += 3;
  }
  CU(cudaGetLastError());
  b->have_ll = true;
  return NVB_OK;
}

int nvb_batch_get_events(nvb_batch *b, int32_t *events, int32_t *status) {
  if (!b) return fail(NVB_EINVAL, "NULL batch");
  if (!b->have_events) return fail(NVB_ESTATE, "nvb_batch_get_events before nvb_batch_refine");
  CU(cudaSetDevice(b->model->device));
  cudaStream_t st = b->run_stream;  // results are read back behind the run that produced them, on its stream
  if (events) CU(cudaMemcpyAsync(events, b->d_events.p, (size_t)2 * b->total_ref * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  if (status) CU(cudaMemcpyAsync(status, b->d_status.p, (size_t)b->n_reads * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return NVB_OK;
}

int nvb_batch_get_log_likelihoods(nvb_batch *b, double *out, int32_t *status) {
  if (!b) return fail(NVB_EINVAL, "NULL batch");
  if (!b->have_ll) return fail(NVB_ESTATE, "nvb_batch_get_log_likelihoods before nvb_batch_estimate");
  CU(cudaSetDevice(b->model->device));
  cudaStream_t st = b->run_stream;
  if (out) CU(cudaMemcpyAsync(out, b->d_ll.p, (size_t)b->total_ref * b->model->dev.alphabet * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (status) CU(cudaMemcpyAsync(status, b->d_status.p, (size_t)b->n_reads * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return NVB_OK;
}

int nvb_batch_get_bands(nvb_batch *b, int32_t *starts, int32_t *ends) {
  if (!b) return fail(NVB_EINVAL, "NULL batch");
  CU(cudaSetDevice(b->model->device));
  size_t cnt = (size_t)b->total_ref + b->n_reads;
  if (starts) CU(cudaMemcpy(starts, b->d_bs.p, cnt * sizeof(int32_t), cudaMemcpyDeviceToHost));
  if (ends) CU(cudaMemcpy(ends, b->d_be.p, cnt * sizeof(int32_t), cudaMemcpyDeviceToHost));
  return NVB_OK;
}

int nvb_batch_cell_counts(nvb_batch *b, int model_wobbling, int64_t counts[4]) {
  if (!b || !counts) return fail(NVB_EINVAL, "NULL argument");
  CU(cudaSetDevice(b->model->device));
  size_t cnt = (size_t)b->total_ref + b->n_reads;
  std::vector<int32_t> bs(cnt), be(cnt);
  CU(cudaMemcpy(bs.data(), b->d_bs.p, cnt * sizeof(int32_t), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(be.data(), b->d_be.p, cnt * sizeof(int32_t), cudaMemcpyDeviceToHost));
  const int k = b->model->dev.k, cp = b->model->dev.central, A = b->model->dev.alphabet;
  int64_t c0 = 0, c1 = 0, c2 = 0, c3 = 0;
  for (int r = 0; r < b->n_reads; r++) {
    if (b->flags[r]) continue;
    const int n = (int)(b->ref_off[r + 1] - b->ref_off[r]);
    const int32_t *s = bs.data() + b->ref_off[r] + r, *e = be.data() + b->ref_off[r] + r;
    auto W = [&](int j) { return (int64_t)(e[j] - s[j] + 1); };
    for (int rho = 0; rho < 2 * n; rho++) {  // SURVEY.md 8(d)
      int64_t w = (rho % 2 == 0) ? W(rho / 2) : W(rho / 2 + 1);
      if (rho >= 1) c0 += w;
      if (rho <= 2 * n - 2) c0 += w;
    }
    for (int j = 1; j <= n; j++) c1 += W(j);
    for (int j = 0; j < n; j++) c1 += W(j);
    for (int i = 0; i < n; i++) c2 += W(i + 1);
    for (int i = 1; i <= n; i++) c2 += W(i - 1);
    if (model_wobbling) for (int i = 1; i < n; i++) c2 += 2 * W(i);
    const int back = k - cp - 1, fwd = cp;
    for (int i = 0; i < n; i++) {
      int first = std::max(0, i - back), last = std::min(n - 1, i + fwd);
      int64_t c = 0;
      for (int j = first; j <= last; j++) c += W(j + 1) + ((j > 0 && model_wobbling) ? W(j) : 0);
      if (last + 1 < n && model_wobbling) c += W(last);
      c3 += (A - 1) * c;
    }
  }
  counts[0] = c0; counts[1] = c1; counts[2] = c2; counts[3] = c3;
  return NVB_OK;
}

int64_t nvb_batch_launch_count(const nvb_batch *b) { return b ? b->launches : 0; }

int nvb_batch_debug_rows(nvb_batch *b, int read, int plane, double *out_log, int64_t n_cells) {
  if (!b || !out_log || read < 0 || read >= b->n_reads) return fail(NVB_EINVAL, "bad argument");
  if (n_cells != b->cells[read] && n_cells != 2 * b->cells[read] - b->w0[read] - b->wn[read])
    return fail(NVB_EINVAL, "read %d has %lld cells", read, (long long)b->cells[read]);
  if (!b->last_ws) return fail(NVB_ESTATE, "nvb_batch_debug_rows before a run");
  CU(cudaSetDevice(b->model->device));
  CU(cudaStreamSynchronize(b->run_stream));
  const Workspace &ws = *b->last_ws;
  int64_t base = 0;
  CU(cudaMemcpy(&base, b->d_mat_base.p + read, sizeof(int64_t), cudaMemcpyDeviceToHost));
  std::vector<double> f((size_t)n_cells);
  std::vector<int32_t> x((size_t)n_cells);
  CU(cudaMemcpy(f.data(), (plane ? ws.sF.p : ws.pF.p) + base, (size_t)n_cells * sizeof(double), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(x.data(), (plane ? ws.sX.p : ws.pX.p) + base, (size_t)n_cells * sizeof(int32_t), cudaMemcpyDeviceToHost));
  for (int64_t i = 0; i < n_cells; i++)
    out_log[i] = f[i] > 0.0 ? log(f[i]) + x[i] * 0.6931471805599453 : -INFINITY;
  return NVB_OK;
}

int nvb_batch_enable_timing(nvb_batch *b, int on) {
  if (!b) return fail(NVB_EINVAL, "NULL batch");
  b->timing = on != 0;
  return NVB_OK;
}

int nvb_batch_get_timing(nvb_batch *b, double ms[NVB_N_STAGES], int64_t launches[NVB_N_STAGES]) {
  if (!b || !ms || !launches) return fail(NVB_EINVAL, "NULL argument");
  CU(cudaSetDevice(b->model->device));
  b->drain();
  for (int i = 0; i < NVB_N_STAGES; i++) { ms[i] = 0; launches[i] = 0; }
  for (auto &t : b->timed) {
    float x = 0;
    CU(cudaEventElapsedTime(&x, t.second.first, t.second.second));
    ms[t.first] += x;
    launches[t.first] += 1;
    cudaEventDestroy(t.second.first);
    cudaEventDestroy(t.second.second);
  }
  b->timed.clear();
  return NVB_OK;
}

int nvb_measure_fp64_fma_rate(int device, double *fma_per_second) {
  if (!fma_per_second) return fail(NVB_EINVAL, "NULL argument");
  if (nvb_device_count() <= device) return fail(NVB_ECUDA, "CUDA device %d not available", device);
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  DevBuf<double> sink;
  CU(sink.alloc(1));
  const int blocks = prop.multiProcessorCount * 8, iters = 1 << 16;
  nvbk_fp64_fma_probe(1 << 10, blocks, 0, sink.p);  // warm-up
  double best = 0;
  for (int rep = 0; rep < 3; rep++) {
    float ms = nvbk_fp64_fma_probe(iters, blocks, 0, sink.p);
    CU(cudaGetLastError());
    double rate = 8.0 * iters * 256.0 * blocks / (ms * 1e-3);
    best = std::max(best, rate);
  }
  *fma_per_second = best;
  return NVB_OK;
}

int nvb_refine_alignment_batch(nvb_model *model, const nvb_reads *reads, int model_transitions, int32_t *events,
                               int32_t *status) {
  nvb_batch *b = nvb_batch_create(model, reads);
  if (!b) return g_code ? g_code : NVB_EINVAL;  // the code nvb_batch_create failed with (EINVAL / ECUDA / ENOMEM)
  int rc = nvb_batch_refine(b, model_transitions, nullptr);
  if (!rc) rc = nvb_batch_get_events(b, events, status);
  nvb_batch_destroy(b);
  return rc;
}

int nvb_estimate_log_likelihoods_batch(nvb_model *model, const nvb_reads *reads, int model_wobbling, double *out,
                                       int32_t *status) {
  nvb_batch *b = nvb_batch_create(model, reads);
  if (!b) return g_code ? g_code : NVB_EINVAL;
  int rc = nvb_batch_estimate(b, model_wobbling, nullptr);
  if (!rc) rc = nvb_batch_get_log_likelihoods(b, out, status);
  nvb_batch_destroy(b);
  return rc;
}

int nvb_model_expected_signal(nvb_model *model, int32_t n_reads, const int32_t *reference,
                              const int64_t *reference_off, const int32_t *context_before,
                              const int64_t *context_before_off, const int32_t *context_after,
                              const int64_t *context_after_off, double *out) {
  if (!model || !out) return fail(NVB_EINVAL, "NULL argument");
  CU(cudaSetDevice(model->device));
  nvb_batch b;
  b.model = model;
  int rc = upload_sequences(&b, n_reads, reference, reference_off, context_before, context_before_off,
                            context_after, context_after_off, 0);
  if (rc) return rc;
  // the kernel only touches the sequence fields; give the signal offsets a valid array
  b.dev.sig_off = b.d_ref_off.p;
  DevBuf<double> d_out;
  CU(d_out.alloc((size_t)b.total_ref));
  nvbk_expected_signal(model->dev, b.dev, b.total_ref, d_out.p, 0);
  CU(cudaGetLastError());
  CU(cudaMemcpy(out, d_out.p, (size_t)b.total_ref * sizeof(double), cudaMemcpyDeviceToHost));
  return NVB_OK;
}

int nvb_batch_get_alignment_table(nvb_batch *b, const int64_t *start_in_signal, const int64_t *ref_start,
                                  const int64_t *ref_end, const int32_t *reverse, int64_t *out) {
  if (!b || !start_in_signal || !ref_start || !ref_end || !reverse || !out) return fail(NVB_EINVAL, "NULL argument");
  if (!b->have_events) return fail(NVB_ESTATE, "alignment table requested before nvb_batch_refine");
  CU(cudaSetDevice(b->model->device));
  const size_t n = b->n_reads;
  DevBuf<int64_t> d_meta, d_out;
  DevBuf<int32_t> d_rev;
  std::vector<int64_t> meta(3 * n);
  std::copy(start_in_signal, start_in_signal + n, meta.begin());
  std::copy(ref_start, ref_start + n, meta.begin() + n);
  std::copy(ref_end, ref_end + n, meta.begin() + 2 * n);
  cudaStream_t st = b->run_stream;  // behind the refine that produced the events
  CU(upload(d_meta, meta.data(), meta.size(), st));
  CU(upload(d_rev, reverse, n, st));
  CU(d_out.alloc((size_t)3 * b->total_ref));
  nvbk_alignment_table(b->dev, b->d_events.p, b->d_status.p, d_meta.p, d_meta.p + n, d_meta.p + 2 * n, d_rev.p,
                       b->total_ref, d_out.p, st);
  b->launches++;
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out, d_out.p, (size_t)3 * b->total_ref * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));  // the temporaries go back to the block cache on return
  return NVB_OK;
}

int nvb_batch_event_means(nvb_batch *b, double *out) {
  if (!b || !out) return fail(NVB_EINVAL, "NULL argument");
  if (!b->have_events) return fail(NVB_ESTATE, "event means requested before nvb_batch_refine");
  CU(cudaSetDevice(b->model->device));
  DevBuf<double> d_out;
  cudaStream_t st = b->run_stream;  // behind the refine that produced the events
  CU(d_out.alloc((size_t)b->total_ref));
  nvbk_event_means(b->dev, b->d_events.p, b->d_status.p, b->total_ref, d_out.p, st);
  b->launches++;
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out, d_out.p, (size_t)b->total_ref * sizeof(double), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return NVB_OK;
}

int nvb_batch_apply_splines(nvb_batch *b, const double *knots, const double *coefs, const int64_t *spline_off,
                            int degree, void *stream) {
  if (!b || !spline_off) return fail(NVB_EINVAL, "NULL argument");
  if (degree < 1 || degree > 5) return fail(NVB_EINVAL, "spline degree must be 1..5");
  int rc = check_offsets(spline_off, b->n_reads, "spline");
  if (rc) return rc;
  const int64_t total = spline_off[b->n_reads];
  if (total > 0 && (!knots || !coefs)) return fail(NVB_EINVAL, "NULL argument");
  for (int i = 0; i < b->n_reads; i++) {
    const int64_t n = spline_off[i + 1] - spline_off[i];
    if (n != 0 && n < 2 * (degree + 1)) return fail(NVB_EINVAL, "spline of read %d has %lld knots, needs %d", i, (long long)n, 2 * (degree + 1));
  }
  CU(cudaSetDevice(b->model->device));
  cudaStream_t st = (cudaStream_t)stream;
  b->touch(st);
  DevBuf<double> d_knots, d_coefs;
  DevBuf<int64_t> d_off;
  CU(upload(d_knots, knots, (size_t)total, st));
  CU(upload(d_coefs, coefs, (size_t)total, st));
  CU(upload(d_off, spline_off, (size_t)b->n_reads + 1, st));
  nvbk_apply_splines(b->dev, b->d_signal.p, d_knots.p, d_coefs.p, d_off.p, degree, b->total_sig, st);
  b->launches++;
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(st));  // the temporaries go back to the block cache on return
  return NVB_OK;
}

int nvb_batch_get_signal(nvb_batch *b, double *out) {
  if (!b || !out) return fail(NVB_EINVAL, "NULL argument");
  CU(cudaSetDevice(b->model->device));
  CU(cudaMemcpyAsync(out, b->d_signal.p, (size_t)b->total_sig * sizeof(double), cudaMemcpyDeviceToHost, b->run_stream));
  CU(cudaStreamSynchronize(b->run_stream));
  return NVB_OK;
}

int nvb_batch_chunk_values(nvb_batch *b, const int32_t *reverse, double normalization_event_length, double *d_chunks,
                           void *stream) {
  if (!b || !reverse || !d_chunks) return fail(NVB_EINVAL, "NULL argument");
  if (!b->have_ll) return fail(NVB_ESTATE, "chunk values requested before nvb_batch_estimate");
  if (b->model->dev.alphabet != 4) return fail(NVB_EINVAL, "chunk values need alphabet_size == 4");
  CU(cudaSetDevice(b->model->device));
  cudaStream_t st = (cudaStream_t)stream;
  b->touch(st);
  const size_t n = (size_t)b->n_reads;
  if (b->h_rev.size() != n || !std::equal(reverse, reverse + n, b->h_rev.begin())) {
    CU(cudaStreamSynchronize(st));  // an earlier launch may still read the old values
    b->h_rev.assign(reverse, reverse + n);
    CU(upload(b->d_rev, b->h_rev.data(), n, st));
    CU(cudaStreamSynchronize(st));
  }
  nvbk_chunk_values(b->dev, b->d_ll.p, b->d_rev.p, normalization_event_length, b->total_ref, d_chunks, st);
  b->launches++;
  CU(cudaGetLastError());
  return NVB_OK;
}

int nvb_signal_anchors_batch(int device, const nvb_hits *h, int32_t *anchors, int64_t *meta, void *stream) {
  if (!h || !anchors || !meta || h->n_reads < 0) return fail(NVB_EINVAL, "NULL argument");
  if (nvb_device_count() <= device) return fail(NVB_ECUDA, "CUDA device %d not available (no CPU fallback)", device);
  const int n = h->n_reads;
  if (n == 0) return NVB_OK;
  if (!h->cigar_len || !h->cigar_op || !h->cigar_off || !h->mapped_position || !h->reverse || !h->read_sequence ||
      !h->base_to_sample || !h->read_off || !h->n_signal || !h->d_genome || h->bandwidth < 0)
    return fail(NVB_EINVAL, "nvb_signal_anchors_batch: bad argument");
  int rc;
  if ((rc = check_offsets(h->cigar_off, n, "cigar"))) return rc;
  if ((rc = check_offsets(h->read_off, n, "read"))) return rc;
  CU(cudaSetDevice(device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t n_ops = (size_t)h->cigar_off[n], n_bases = (size_t)h->read_off[n];
  DevBuf<int32_t> d_len, d_rev, d_map, d_nsig, d_anchors;
  DevBuf<int8_t> d_op, d_seq;
  DevBuf<int64_t> d_coff, d_pos, d_roff, d_meta;
  CU(upload(d_len, h->cigar_len, n_ops, st));
  CU(upload(d_op, h->cigar_op, n_ops, st));
  CU(upload(d_coff, h->cigar_off, (size_t)n + 1, st));
  CU(upload(d_pos, h->mapped_position, (size_t)n, st));
  CU(upload(d_rev, h->reverse, (size_t)n, st));
  CU(upload(d_seq, h->read_sequence, n_bases, st));
  CU(upload(d_map, h->base_to_sample, n_bases, st));
  CU(upload(d_roff, h->read_off, (size_t)n + 1, st));
  CU(upload(d_nsig, h->n_signal, (size_t)n, st));
  CU(d_anchors.alloc(2 * n_bases));
  CU(d_meta.alloc((size_t)7 * n));
  AnchorBatch A;
  A.n_reads = n;
  A.cigar_len = d_len.p; A.cigar_op = d_op.p; A.cigar_off = d_coff.p; A.mapped_pos = d_pos.p; A.reverse = d_rev.p;
  A.read_seq = d_seq.p; A.mapping = d_map.p; A.read_off = d_roff.p; A.n_signal = d_nsig.p;
  A.genome = h->d_genome; A.genome_len = h->genome_length; A.bandwidth = h->bandwidth;
  nvbk_anchors(A, d_anchors.p, d_meta.p, st);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(anchors, d_anchors.p, 2 * n_bases * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(meta, d_meta.p, (size_t)7 * n * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));  // the temporaries go back to the block cache on return
  return NVB_OK;
}

int nvb_radix_histogram_d(int device, const double *d_values, int64_t n, int absolute_deviation, double shift,
                          uint64_t prefix, int fixed_bits, uint64_t *d_hist, void *stream) {
  if (!d_hist || n < 0 || (n > 0 && !d_values) || fixed_bits < 0 || fixed_bits > 56 || (fixed_bits & 7))
    return fail(NVB_EINVAL, "bad argument");
  if (nvb_device_count() <= device) return fail(NVB_ECUDA, "CUDA device %d not available (no CPU fallback)", device);
  CU(cudaSetDevice(device));
  nvbk_radix_hist(d_values, n, absolute_deviation ? 1 : 0, shift, (unsigned long long)prefix, fixed_bits,
                  (unsigned long long *)d_hist, (cudaStream_t)stream);
  CU(cudaGetLastError());
  return NVB_OK;
}

int nvb_normalize_each(int device, const double *values, const int64_t *off, int32_t n_reads, double lo, double hi,
                       double *out, double *shift_scale, void *stream) {
  if (n_reads < 0 || !off || (n_reads > 0 && (!values || !out))) return fail(NVB_EINVAL, "bad argument");
  if (nvb_device_count() <= device) return fail(NVB_ECUDA, "CUDA device %d not available (no CPU fallback)", device);
  int rc = check_offsets(off, n_reads, "values");
  if (rc) return rc;
  for (int i = 0; i < n_reads; i++)
    if (off[i + 1] - off[i] > 0x7fffff00LL) return fail(NVB_EINVAL, "read %d too long", i);
  CU(cudaSetDevice(device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t total = (size_t)off[n_reads];
  DevBuf<double> d_values, d_out, d_ss;
  DevBuf<int64_t> d_off;
  CU(upload(d_values, values, total, st));
  CU(upload(d_off, off, (size_t)n_reads + 1, st));
  CU(d_out.alloc(total));
  CU(d_ss.alloc((size_t)2 * n_reads));
  nvbk_normalize_each(d_values.p, d_off.p, n_reads, lo, hi, d_out.p, d_ss.p, st);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out, d_out.p, total * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (shift_scale) CU(cudaMemcpyAsync(shift_scale, d_ss.p, (size_t)2 * n_reads * sizeof(double), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return NVB_OK;
}

int nvb_normalize_clip_d(int device, const double *d_values, int64_t n, double shift, double scale, double lo, double hi,
                         double *d_out, void *stream) {
  if (n < 0 || (n > 0 && (!d_values || !d_out))) return fail(NVB_EINVAL, "bad argument");
  if (nvb_device_count() <= device) return fail(NVB_ECUDA, "CUDA device %d not available (no CPU fallback)", device);
  CU(cudaSetDevice(device));
  nvbk_normalize_clip(d_values, n, shift, scale, lo, hi, d_out, (cudaStream_t)stream);
  CU(cudaGetLastError());
  return NVB_OK;
}

int nvb_batch_scatter_add_rows(nvb_batch *b, const double *d_chunks, const int64_t *dest, double *d_rows, void *stream) {
  if (!b || !d_chunks || !dest || !d_rows) return fail(NVB_EINVAL, "NULL argument");
  CU(cudaSetDevice(b->model->device));
  cudaStream_t st = (cudaStream_t)stream;
  b->touch(st);
  const size_t n = (size_t)b->n_reads;
  if (b->h_dest.size() != n || !std::equal(dest, dest + n, b->h_dest.begin())) {
    CU(cudaStreamSynchronize(st));
    b->h_dest.assign(dest, dest + n);
    CU(upload(b->d_dest, b->h_dest.data(), n, st));
    CU(cudaStreamSynchronize(st));
  }
  nvbk_scatter_add_rows(b->dev, d_chunks, b->d_dest.p, b->d_status.p, b->total_ref, d_rows, st);
  b->launches++;
  CU(cudaGetLastError());
  return NVB_OK;
}

int nvb_posterior_rows_d(int device, const double *d_rows, int64_t base_row, int64_t row_lo, int64_t row_hi,
                         const int8_t *d_ref, const int64_t *d_group_off, int32_t n_groups, int k, double snp_prior,
                         double *d_out_rows, void *stream) {
  if (!d_rows || !d_ref || !d_group_off || !d_out_rows || n_groups < 0 || row_hi < row_lo || base_row > row_lo)
    return fail(NVB_EINVAL, "bad argument");
  if (nvb_device_count() <= device) return fail(NVB_ECUDA, "CUDA device %d not available (no CPU fallback)", device);
  CU(cudaSetDevice(device));
  nvbk_posterior_rows(d_rows, base_row, row_lo, row_hi, d_ref, d_group_off, n_groups, k, snp_prior, d_out_rows,
                      (cudaStream_t)stream);
  CU(cudaGetLastError());
  return NVB_OK;
}

}  // extern "C"
