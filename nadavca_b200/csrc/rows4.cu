// rows4.cu -- forward / backward banded DP rows, scaled linear domain (see dp3.cuh), pipelined stripes.
//
// Replaces the driver loops of RefineAlignment (reference nadavca/dtw/dtw.cpp:182-197) and EstimateLogLikelihoods
// (dtw.cpp:48-81) with Node::NextRow (node_next_row.h:6-61).  The rows of a pass are grouped in pairs
// (A-row, B-row): A = the wobble row (dtw.cpp:53-58) or the transition row (dtw.cpp:170-172) in front of base i,
// B = the model row of base i.  A stripe is one LOADER lane plus up to 31 pair lanes of one warp; lane l works one
// column behind lane l-1 and neighbour cells travel by warp shuffle.
//
// One CTA of NW warps works on one (read, direction); warp w takes stripes w, w+NW, ...  A stripe can start as soon
// as the last row of the stripe before it starts to appear, so consecutive stripes overlap in time: the last pair lane
// of a stripe publishes its B-row cells into a shared-memory hand-off row (plus a 64-bit "stripe id | cells ready"
// word), and the LOADER lane of the next stripe consumes them from there, spinning only when it catches up.  With
// NW+1 hand-off rows a buffer is re-used by the warp that consumed it last, so program order alone protects it.
// The band of a default read (W = 301 columns, ~10 new columns per base) makes a 31-pair stripe last ~670 steps
// while a new stripe can start every ~340 steps: two warps per direction keep every warp busy and halve the
// critical path compared with draining each stripe (history/v3_rows_drained_stripes.cu.txt); wider bands use more
// warps.  For batches that fill the GPU, rows5.cu (one rotating wavefront per direction) needs fewer steps.
// Stored rows are written as (mantissa double, exponent int32) planes.
#include "dp3.cuh"
#include "kernels.h"

namespace {

constexpr int PAIRS = NVB_WARP - 1;  // pair lanes per stripe

struct PairGeom {
  int hasA, aband, bband, storeA;
  int64_t aoff, boff;
  int base;  // reference base index of the model row
  int nb;    // base index of the neighbouring model row (the other component of the wobble mixture)
};

template <bool REV>
__device__ __forceinline__ PairGeom pair_geom(const ReadView &v, int mode, int g) {
  PairGeom p;
  const int n = v.n;
  const int i = REV ? n - 1 - g : g;
  p.base = i;
  p.storeA = (mode == NVB_MODE_TRANS);
  if (!REV) {
    p.hasA = (i >= 1) && mode != NVB_MODE_PLAIN;
    p.aband = i; p.bband = i + 1; p.nb = i - 1;
    if (mode == NVB_MODE_TRANS) { p.aoff = trans_row_off(v, 2 * i); p.boff = trans_row_off(v, 2 * i + 1); }
    else { p.aoff = 0; p.boff = v.coff[i + 1]; }
  } else {
    p.hasA = (i <= n - 2) && mode != NVB_MODE_PLAIN;
    p.aband = i + 1; p.bband = i; p.nb = i + 1;
    if (mode == NVB_MODE_TRANS) { p.aoff = trans_row_off(v, 2 * i + 1); p.boff = trans_row_off(v, 2 * i); }
    else { p.aoff = 0; p.boff = v.coff[i]; }
  }
  return p;
}

// Store staging (per warp, shared memory).  A lane owns a row, so storing a cell per lane and step scatters 31
// 8-byte + 31 4-byte writes over 62 cache lines per warp-step; ncu showed that traffic (4-8x sector amplification,
// L1 hit rate of the signal loads 4 %) to be what the sweep waits for.  Instead every lane parks its cell in a
// [32 rows][TS steps] tile and every TS steps the warp writes the tile out row segment by row segment: TS consecutive
// threads write TS consecutive cells of one row.
#ifndef NVB_STRIPE_TS
#define NVB_STRIPE_TS 8
#endif
constexpr int TS = NVB_STRIPE_TS;  // steps per tile: the flush (~270 warp instructions per tile) is amortised over them
constexpr int TSTRIDE = TS + 1;    // padded row stride (conflict-free for the per-step column writes)
struct RowMeta {
  long long off;  // offset of the row's first cell in the matrix planes
  int s, e;       // band of the row (empty for lanes that store nothing)
};
struct StoreTile {
  double *f;      // [32][TSTRIDE]
  int32_t *x;     // [32][TSTRIDE]
  RowMeta *meta;  // [32]
};
constexpr size_t kTileBytes = 32 * TSTRIDE * (sizeof(double) + sizeof(int32_t)) + 32 * sizeof(RowMeta);
constexpr size_t kRingStride = (ring_bytes(4) + 15) / 16 * 16;  // per-warp signal ring (dp3.cuh)

// Write the first `cnt` steps (t0 .. t0+cnt-1) of a tile to the matrix planes.
template <bool REV>
__device__ __forceinline__ void flush_tile(const StoreTile &tile, double *F, int32_t *X, int C0, int t0, int cnt,
                                           int lane) {
  constexpr int RPI = NVB_WARP / TS;  // rows per iteration
  const int kk = lane & (TS - 1);
#pragma unroll
  for (int i = 0; i < NVB_WARP / RPI; i++) {
    const int r = RPI * i + lane / TS;
    const RowMeta m = tile.meta[r];
    const int tt = t0 + kk;
    const int c = REV ? C0 - (tt - r) : C0 + (tt - r);
    if (kk < cnt && c >= m.s && c <= m.e) {
      const long long idx = m.off + (c - m.s);
      F[idx] = tile.f[r * TSTRIDE + kk];
      X[idx] = tile.x[r * TSTRIDE + kk];
    }
  }
}

// Hand-off rows of one CTA in shared memory: NB = NW + 1 buffers of `width` cells each.
struct Handoff {
  double *f;                     // [NB][width]
  int32_t *e;                    // [NB][width]
  volatile unsigned long long *word;  // [NB]  (stripe id + 1) << 32 | cells ready (in sweep order)
  int width, nb;
};

template <int MEL, int MODE, bool REV>
__device__ __forceinline__ void sweep_stripes(const ModelDev &M, const ReadView &v, double *F, int32_t *X, int lane, int warp, int NW,
                              const Handoff &H, const StoreTile &tileB, const StoreTile &tileA, const SignalRing<4> &R,
                              unsigned exp_tab) {
  constexpr int mode = MODE;
  const int n = v.n, N = v.N;
  const double C_E2 = 0.1353352832366127;  // exp(-2): the "/ 2" of kmer_model.cpp:60 is "- 2.0" in log space
  const int n_stripes = (n + PAIRS - 1) / PAIRS;

  // all-ones first row (dtw.cpp:50,66,182,190): written to HBM by warp 0, generated on the fly by stripe 0's loader
  const int j0 = REV ? n : 0;
  if (warp == 0) {
    const int s0 = v.bs[j0], e0 = v.be[j0];
    const int64_t off0 = REV ? ((mode == NVB_MODE_TRANS) ? trans_row_off(v, 2 * n - 1) : v.coff[n]) : 0;
    for (int c = s0 + lane; c <= e0; c += NVB_WARP) { F[off0 + c - s0] = 1.0; X[off0 + c - s0] = 0; }
  }

  for (int s = warp; s < n_stripes; s += NW) {
    const int g0 = s * PAIRS;
    const int npairs = min(PAIRS, n - g0);
    // band of the row this stripe's loader consumes: the initial row, or the B-row of the last pair of stripe s-1
    int ls, le;
    if (s == 0) { ls = v.bs[j0]; le = v.be[j0]; }
    else { const PairGeom pp = pair_geom<REV>(v, mode, g0 - 1); ls = v.bs[pp.bband]; le = v.be[pp.bband]; }
    const int in_buf = (s + H.nb - 1) % H.nb, out_buf = s % H.nb;
    const volatile double *inF = H.f + (size_t)in_buf * H.width;   // volatile: read only after the ready word
    const volatile int32_t *inE = H.e + (size_t)in_buf * H.width;
    double *outF = H.f + (size_t)out_buf * H.width;
    int32_t *outE = H.e + (size_t)out_buf * H.width;
    const unsigned long long in_tag = (unsigned long long)s << 32;         // stripe s-1 publishes tag (s-1)+1 = s
    const unsigned long long out_tag = (unsigned long long)(s + 1) << 32;
    if (lane == 0) H.word[out_buf] = out_tag;  // nothing of this stripe's last row is ready yet
    __syncwarp();

    LaneCfg L;
    lane_cfg_clear(L);
    int ws = 1, awe = 0;  // A-row band, for the stores of the transition rows
    int64_t aoff = 0, boff = 0;
    int storeA = 0, storeB = 0;
    if (lane == 0) {
      L.role = NVB_ROLE_LOADER;
      L.ms = ls; L.me = le;
      const PairGeom pg = pair_geom<REV>(v, mode, g0);
      const int nb = (g0 > 0) ? pg.nb : pg.base;  // emission of the model row before the stripe
      lane_set_emission_row(L, v.emis + 4 * (size_t)nb);
    } else if (lane <= npairs) {
      const PairGeom pg = pair_geom<REV>(v, mode, g0 + lane - 1);
      L.role = NVB_ROLE_PAIR;
      lane_set_emission_row(L, v.emis + 4 * (size_t)pg.base);
      ws = v.bs[pg.aband]; awe = v.be[pg.aband];
      L.ms = v.bs[pg.bband]; L.me = v.be[pg.bband];
      aoff = pg.aoff; boff = pg.boff; storeA = pg.storeA && pg.hasA; storeB = 1;
      if (pg.hasA) {
        L.ws = ws; L.we = awe;
        if (mode == NVB_MODE_TRANS) {  // GetTransitionDistribution (kmer_model.cpp:64-94): constant 0.01, or 0
          const double mo = v.emis[4 * (size_t)pg.nb];
          const bool dead = (mo == L.mu);
          L.pc = dead ? 0.0 : 0.01 * 64.0;  // 0.01 as mantissa 0.64 and exponent -6 (an exact rescaling)
          L.kc = dead ? NVB_EZERO : -6;
        } else {
          L.cm = C_E2; L.abias = 0;
        }
      }
    }
    {
      RowMeta mb;
      mb.off = boff; mb.s = storeB ? L.ms : 1; mb.e = storeB ? L.me : 0;
      tileB.meta[lane] = mb;
      if (MODE == NVB_MODE_TRANS) {
        RowMeta ma;
        ma.off = aoff; ma.s = storeA ? ws : 1; ma.e = storeA ? awe : 0;
        tileA.meta[lane] = ma;
      }
    }
    __syncwarp();
    const bool publishes = (lane == npairs) && (s + 1 < n_stripes);  // last pair lane feeds the next stripe
    const int C0 = REV ? le : ls;
    const int endcol = __shfl_sync(NVB_FULL, REV ? L.ms : L.me, npairs);
    const int T = (REV ? C0 - endcol : endcol - C0) + npairs + 1;

    LaneState<MEL> S;
    lane_reset(S);
    LaneOut out;
    out.f = 0.0; out.E = NVB_EZERO; out.p = 1.0; out.k = 0;
    auto sample_index = [&](int t) {
      const int c = REV ? C0 - (t - lane) : C0 + (t - lane);
      return min(max(REV ? c : c - 1, 0), N - 1);
    };
    // signal window of the warp (dp3.cuh): 32 consecutive samples sliding by one per step, staged by TMA bulk copies
    auto stage = [&](int t) {  // the steps t .. t+TS read (and evaluate one step ahead) these samples
      const int lo = REV ? C0 - t - TS : C0 + t - NVB_WARP, hi = REV ? C0 - t + NVB_WARP - 1 : C0 + t + TS - 1;
      ring_advance<REV, 4>(R, min(max(lo, 0), N - 1), min(max(hi, 0), N - 1), min(max(lo - (REV ? 32 : 8), 0), N - 1),
                           min(max(hi + (REV ? 8 : 32), 0), N - 1), lane);
    };
    ring_reset(R, lane);  // every stripe starts at its own band start
    stage(0);
    double p_cur;
    int k_cur;
    lane_emit(L, exp_tab, ring_read(R, sample_index(0)), p_cur, k_cur);  // emissions are evaluated one step ahead
    unsigned ready = 0;  // cells of the hand-off row known to be ready (sweep order)
    const unsigned row_cells = (unsigned)(le - ls + 1);
    for (int t = 0; t < T; t++) {
      // The loader (lane 0) consumes hand-off cell t at step t.  Every 16 steps the whole warp (uniform branch, no
      // divergence around the shuffles) makes sure the producer is at least 16 cells ahead of that, sleeping otherwise.
      if (s > 0 && (t & 15) == 0 && (unsigned)t < row_cells) {
        const unsigned need = min((unsigned)t + 16u, row_cells);
        unsigned backoff = 256;  // ns; a stripe starts ~340 producer steps (~200 us) before its first cell exists
        while (ready < need) {
          const unsigned long long w = H.word[in_buf];
          ready = ((w >> 32) == (in_tag >> 32)) ? (unsigned)w : 0u;
          if (ready < need) {
            __nanosleep(backoff);
            backoff = min(backoff * 2, 4096u);
          }
        }
      }
      const int c = REV ? C0 - (t - lane) : C0 + (t - lane);
      if ((t & (TS - 1)) == 0 && t > 0) stage(t);
      // the emission of step t+1 needs only its sample: it overlaps the state update of step t, which waits for the
      // neighbour's shuffle
      const double p = p_cur;
      const int kk = k_cur;
      lane_emit(L, exp_tab, ring_read(R, sample_index(t + 1)), p_cur, k_cur);
      LaneOut in = shfl_up_out<MODE>(out);
      XD aout;
      lane_update<MEL, MODE, false, false>(L, S, c, p, kk, in, 1.0, 0, out, aout);
      if (lane == 0) {
        const bool inb = (c >= L.ms && c <= L.me);
        out.f = inb ? 1.0 : 0.0;
        out.E = inb ? 0 : NVB_EZERO;
        if (inb && s > 0) {
          out.f = inF[c - L.ms];
          out.E = inE[c - L.ms];
        }
      } else {
        const bool inb = (c >= L.ms && c <= L.me);
        if (publishes && inb) {
          outF[c - L.ms] = out.f;
          outE[c - L.ms] = out.E;
          // the ready count is published every 8 cells (and at the end of the row): a fence per cell would wait for
          // this step's HBM stores as well; the consumer runs ~340 steps behind, so the coarser count costs nothing
          const unsigned done = (unsigned)(REV ? L.me - c : c - L.ms) + 1u;
          if ((done & 7u) == 0u || done == (unsigned)(L.me - L.ms + 1)) {
            __threadfence_block();
            H.word[out_buf] = out_tag | (unsigned long long)done;
          }
        }
      }
      // park this step's cells; every TS steps the warp writes the tiles out with coalesced row segments
      const int k = t & (TS - 1);
      tileB.f[lane * TSTRIDE + k] = out.f;
      tileB.x[lane * TSTRIDE + k] = out.E;
      if (MODE == NVB_MODE_TRANS) {
        tileA.f[lane * TSTRIDE + k] = aout.f;
        tileA.x[lane * TSTRIDE + k] = aout.e;
      }
      if (k == TS - 1 || t == T - 1) {
        __syncwarp();
        flush_tile<REV>(tileB, F, X, C0, t - k, k + 1, lane);
        if (MODE == NVB_MODE_TRANS) flush_tile<REV>(tileA, F, X, C0, t - k, k + 1, lane);
        __syncwarp();
      }
      if ((t & NVB_RENORM_MASK) == NVB_RENORM_MASK) lane_renorm(S);
    }
    __syncwarp();
  }
  ring_drain(R);
}

template <int MEL, int MODE>
__global__ void __launch_bounds__(224, 4) sweep4_kernel(ModelDev M, BatchDev B, int b0, int n_items, int NW, int width,
                                                     const int64_t *mat_base, double *pF, int32_t *pX, double *sF,
                                                     int32_t *sX, double *g_handoff) {
  extern __shared__ unsigned long long smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x;  // (read, direction)
  const unsigned exp_tab = exp_table_init();
  if (item >= n_items) return;
  const int b = b0 + (item >> 1);
  if (B.flags[b]) return;
  Handoff H;
  H.nb = NW + 1;
  H.width = width;
  H.word = smem_raw;                                   // [nb] (padded to 8 words)
  unsigned char *tiles;
  if (g_handoff == nullptr) {
    H.f = reinterpret_cast<double *>(smem_raw + 8);    // nb <= 8
    H.e = reinterpret_cast<int32_t *>(H.f + (size_t)H.nb * width);
    tiles = reinterpret_cast<unsigned char *>(H.e + (size_t)H.nb * width);
  } else {
    // band rows too wide for shared memory: the hand-off rows of this (read, direction) live in global scratch
    // (2 * nb * width doubles per item).  Producer and consumer are warps of the same CTA, so the block-scope fence
    // in front of the ready word and the volatile reads behind it order the accesses exactly as in shared memory.
    H.f = g_handoff + (size_t)item * 2 * H.nb * width;
    H.e = reinterpret_cast<int32_t *>(H.f + (size_t)H.nb * width);
    tiles = reinterpret_cast<unsigned char *>(smem_raw + 8);
  }
  // per-warp store tiles behind the hand-off rows (B rows, and A rows for the transition sweep)
  auto make_tile = [&](int index) {
    unsigned char *p = tiles + (size_t)index * kTileBytes;
    StoreTile t;
    t.f = reinterpret_cast<double *>(p);
    t.meta = reinterpret_cast<RowMeta *>(t.f + 32 * TSTRIDE);
    t.x = reinterpret_cast<int32_t *>(t.meta + 32);
    return t;
  };
  constexpr int TPW = (MODE == NVB_MODE_TRANS) ? 2 : 1;  // tiles per warp: B rows, plus A rows for the transition sweep
  const StoreTile tileB = make_tile(TPW * warp), tileA = make_tile(TPW * warp + TPW - 1);
  // per-warp signal ring (4 chunks of 32 samples + mbarriers + state) behind the tiles
  SignalRing<4> R;
  unsigned char *rings = tiles + (size_t)TPW * NW * kTileBytes;
  rings += (16 - (smem_u32(rings) & 15u)) & 15u;  // cp.async.bulk needs a 16-byte aligned destination
  ring_init(R, rings + (size_t)warp * kRingStride, B.signal, B.sig_off[b], B.sig_off[B.n_reads], lane);
  if (threadIdx.x < H.nb) H.word[threadIdx.x] = 0ull;
  __syncthreads();
  ReadView v = read_view(B, b);
  const int64_t base = mat_base[b];
  if (item & 1) sweep_stripes<MEL, MODE, true>(M, v, sF + base, sX + base, lane, warp, NW, H, tileB, tileA, R, exp_tab);
  else sweep_stripes<MEL, MODE, false>(M, v, pF + base, pX + base, lane, warp, NW, H, tileB, tileA, R, exp_tab);
}

// Node::TotalLikelihood(prefix[n], suffix[n]) (dtw.cpp:83-85); suffix[n] is all ones.  Two passes over the row:
// largest exponent, then the mantissa sum relative to it.
__global__ void __launch_bounds__(128) no_snp2_kernel(ModelDev M, BatchDev B, int b0, int n_items,
                                                      const int64_t *mat_base, const double *pF, const int32_t *pX,
                                                      const double *sF, const int32_t *sX, double *out_ll) {
  const int wic = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * (blockDim.x >> 5) + wic;
  if (item >= n_items) return;
  const int b = b0 + item;
  if (B.flags[b]) return;
  ReadView v = read_view(B, b);
  const int n = v.n;
  const int64_t off = mat_base[b] + v.coff[n];
  const int w = v.be[n] - v.bs[n] + 1;
  int emax = NVB_EZERO;
  for (int i = lane; i < w; i += NVB_WARP) {
    const double f = pF[off + i] * sF[off + i];
    if (f > 0.0) emax = max(emax, pX[off + i] + sX[off + i]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) emax = max(emax, __shfl_xor_sync(NVB_FULL, emax, o));
  double acc = 0.0;
  for (int i = lane; i < w; i += NVB_WARP) {
    const double f = pF[off + i] * sF[off + i];
    if (f > 0.0) acc += f * pow2neg(pX[off + i] + sX[off + i] - emax);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(NVB_FULL, acc, o);
  const double total = log_ext(acc, emax);
  const int A = M.alphabet;
  double *out = out_ll + B.ref_off[b] * A;
  for (int i = lane; i < n; i += NVB_WARP) out[(int64_t)i * A + v.ref[i]] = total;
}

template <int MEL, int MODE>
int launch_mode(const ModelDev &M, const BatchDev &B, int b0, int n_items, int NW, int width, size_t smem,
                const int64_t *mb, double *pF, int32_t *pX, double *sF, int32_t *sX, double *gh, cudaStream_t st) {
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(sweep4_kernel<MEL, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return -2;
  sweep4_kernel<MEL, MODE><<<n_items, NW * NVB_WARP, smem, st>>>(M, B, b0, n_items, NW, width, mb, pF, pX, sF, sX, gh);
  return 0;
}

template <int MEL>
int launch_sweep4(const ModelDev &M, const BatchDev &B, int mode, int b0, int n_items, int NW, int width, size_t smem,
                  const int64_t *mb, double *pF, int32_t *pX, double *sF, int32_t *sX, double *gh, cudaStream_t st) {
  switch (mode) {
    case NVB_MODE_PLAIN: return launch_mode<MEL, NVB_MODE_PLAIN>(M, B, b0, n_items, NW, width, smem, mb, pF, pX, sF, sX, gh, st);
    case NVB_MODE_TRANS: return launch_mode<MEL, NVB_MODE_TRANS>(M, B, b0, n_items, NW, width, smem, mb, pF, pX, sF, sX, gh, st);
    default: return launch_mode<MEL, NVB_MODE_WOBBLE>(M, B, b0, n_items, NW, width, smem, mb, pF, pX, sF, sX, gh, st);
  }
}

// Launch geometry of the striped sweep for a wave whose widest band row has wave_maxw columns.
struct SweepPlan {
  int NW, width;
  size_t smem;
  bool global_handoff;
};

SweepPlan plan_sweep(int mode, int wave_maxw) {
  SweepPlan p;
  // warps per (read, direction): a stripe lasts ~W + 12*31 steps, a new one can start every ~11*31 steps
  p.width = (wave_maxw + 1) & ~1;  // keeps the int32 plane 8-byte aligned
  int NW = (wave_maxw + 12 * PAIRS + 11 * PAIRS - 1) / (11 * PAIRS);
  NW = NW < 1 ? 1 : (NW > 7 ? 7 : NW);
  const int tiles_per_warp = (mode == NVB_MODE_TRANS) ? 2 : 1;
  auto tile_bytes = [&](int nw) { return (size_t)64 + 16 + (size_t)nw * (tiles_per_warp * kTileBytes + kRingStride); };
  auto bytes = [&](int nw) { return tile_bytes(nw) + (size_t)(nw + 1) * p.width * (sizeof(double) + sizeof(int32_t)); };
  const size_t limit = 200 * 1024;
  p.global_handoff = bytes(1) > limit;  // not even two hand-off rows fit (band rows beyond ~8.5k columns)
  if (!p.global_handoff)
    while (NW > 1 && bytes(NW) > limit) NW--;
  p.NW = NW;
  p.smem = p.global_handoff ? tile_bytes(NW) : bytes(NW);
  return p;
}

}  // namespace

double nvbk_emission_scale() { return NVB_EXP_SCALE; }

// Doubles of global scratch the striped sweep needs for its hand-off rows (0 when they fit shared memory).
int64_t nvbk_sweep2_global_handoff_doubles(int mode, int n_reads, int wave_maxw) {
  const SweepPlan p = plan_sweep(mode, wave_maxw);
  return p.global_handoff ? (int64_t)2 * n_reads * 2 * (p.NW + 1) * p.width : 0;
}

// wave_maxw: widest band row among the reads [b0, b1).  Returns -1 for an unsupported min_event_length, -2 when the
// shared-memory reservation fails.
int nvbk_sweep2(const ModelDev &M, const BatchDev &B, int mode, int b0, int b1, int wave_maxw,
                const int64_t *d_mat_base, double *pF, int32_t *pX, double *sF, int32_t *sX, double *g_handoff,
                cudaStream_t st) {
  const int n_items = 2 * (b1 - b0);
  if (n_items <= 0) return 0;
  const SweepPlan p = plan_sweep(mode, wave_maxw);
  if (p.global_handoff && g_handoff == nullptr) return -2;
  double *gh = p.global_handoff ? g_handoff : nullptr;
  const int NW = p.NW, width = p.width;
  const size_t smem = p.smem;
  switch (B.mel) {
    case 0: return launch_sweep4<0>(M, B, mode, b0, n_items, NW, width, smem, d_mat_base, pF, pX, sF, sX, gh, st);
    case 1: return launch_sweep4<1>(M, B, mode, b0, n_items, NW, width, smem, d_mat_base, pF, pX, sF, sX, gh, st);
    case 2: return launch_sweep4<2>(M, B, mode, b0, n_items, NW, width, smem, d_mat_base, pF, pX, sF, sX, gh, st);
    case 3: return launch_sweep4<3>(M, B, mode, b0, n_items, NW, width, smem, d_mat_base, pF, pX, sF, sX, gh, st);
    case 4: return launch_sweep4<4>(M, B, mode, b0, n_items, NW, width, smem, d_mat_base, pF, pX, sF, sX, gh, st);
    case 5: return launch_sweep4<5>(M, B, mode, b0, n_items, NW, width, smem, d_mat_base, pF, pX, sF, sX, gh, st);
    case 6: return launch_sweep4<6>(M, B, mode, b0, n_items, NW, width, smem, d_mat_base, pF, pX, sF, sX, gh, st);
    default: return -1;
  }
}

void nvbk_no_snp2(const ModelDev &M, const BatchDev &B, int b0, int b1, const int64_t *d_mat_base, const double *pF,
                  const int32_t *pX, const double *sF, const int32_t *sX, double *d_out_ll, cudaStream_t st) {
  const int n_items = b1 - b0;
  if (n_items <= 0) return;
  no_snp2_kernel<<<(n_items + 3) / 4, 128, 0, st>>>(M, B, b0, n_items, d_mat_base, pF, pX, sF, sX, d_out_ll);
}
