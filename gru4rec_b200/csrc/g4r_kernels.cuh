// g4r_kernels.cuh -- device code of the GRU4Rec session-parallel training step for sm_100a.
//
// One mini-batch (reference: one call of the compiled Theano `train_function`, gru4rec.py:584,623) is a
// fixed sequence of phases.  Each phase is a __device__ function parameterised on (cta, n_cta) so the same
// code runs either as one kernel per phase (CUDA-graph replay; easy to profile with ncu) or inside the
// persistent cooperative kernel (g4r_persistent.cuh) with grid barriers between phases.
//
// Data layout (all fp32, row-major, leading dimension padded to a multiple of 4 floats so every row is
// a whole number of 16-byte vectors; padding columns are zero and stay zero):
//   item tables   Wy [I x ldL], By [I], E [I x ldE], Wx0 [I x ld3] (no-embedding mode) + acc/vel twins
//   dense         Wx[l] [in x ld3], Wh[l] [L x ldL], Wrz[l] [L x ld2], Bh[l] [ld3] + acc/vel twins
//   hidden state  H[l] [B x ldL] in PHYSICAL lanes; a step addresses lane b through slot[b]
//   score columns are processed in (item, position)-sorted order so that all duplicates of an item are
//   adjacent and owned by one CTA (deterministic sparse Adagrad without atomics); the plan kernel builds
//   that order for a whole window of steps off the critical path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/g4r.h"

#define G4R_EPS_ADA 1e-6f
#define G4R_EPS_LOG 1e-24f
#define G4R_NSTAT 8

struct ActSpec { int kind; float p1, p2; };
constexpr int MG_CAP = 256;          // steps per multi-GPU window (g4r_multi.cuh)
struct MgDev {                       // device pointers of the multi-GPU state
  int R, rank;
  int *gItem, *gPos, *gM, *gX;       // gathered per-rank sorted columns [R][MG_CAP][NP], batch sizes [R][MG_CAP], inputs [R][MG_CAP][B]
  int *mEnt, *mItem, *mCbeg;         // merged columns per step: entry = rank << 20 | col ; [MG_CAP][R*NP], chunks [MG_CAP][NCH+1]
  int *mTot;                         // [MG_CAP] merged length
  int *xEnt, *xItem, *xTot;          // merged input rows per step: entry = rank << 16 | lane ; [MG_CAP][R*B]
  float *DSYall, *DBYall, *INall;    // gathered gradients of one step [R][NP][ldL], [R][NP], [R][B][ldin]
  float* gradFlat; size_t gradCount; // dense gradients, contiguous (all-reduced in place)
};

struct MgTensor { float *p, *acc, *vel; size_t goff; int count; };
struct TsBuf {                 // device buffers of the tensor-core step (owned by the handle's workspace)
  unsigned char *A1, *A2, *A3, *A4, *A5, *A6, *A7, *A8;      // left operands  (rows x K) as hi|lo blocks
  unsigned char *W1, *W2, *W3, *W4, *B3, *B4, *B5, *B8a, *B8b;   // right operands (n x K)
  float *P, *P1, *Pa, *Pb;                                   // partial tiles of the split-K products: main stream, dSy (side 1), dense gradients (side 2)
  float *O, *bias;                                           // scores / dL/do [Bpad x ldO] (lane-major), bias of the sorted columns [NP]
  int ldO;
  int Mpad, Lk2, Lk1, Lk3, Nk, Bk;                           // padded extents: lanes; K = 2L, L, 3L, columns, lanes (multiples of 32)
  int Lp;                                                    // L rounded up to the 256-wide N tile (segments of B8a)
};
// tiling of one tensor-core product (g4r_tcstep.cuh): N tile, tile counts, K splits, leading dimension / size of the partial tiles.
// cluster_cap > 0: the K splits of a tile form a thread-block cluster (power of two <= cap, divides the 128 tile rows)
struct TsShape { int NT, m_tiles, n_tiles, ksplit, ldP; size_t p_floats; };
static inline TsShape ts_shape(int rows, int cols, int chunks, int n_sm, int cluster_cap) {
  TsShape t;
  t.NT = cols > 128 ? 256 : 128;
  t.m_tiles = (rows + 127) / 128; t.n_tiles = (cols + t.NT - 1) / t.NT;
  const int tiles = t.m_tiles * t.n_tiles;
  int ks = (n_sm - 8) / tiles;                              // about one CTA per SM
  if (ks > chunks) ks = chunks;
  if (ks < 1) ks = 1;
  if (cluster_cap > 0) {
    int p2 = 1;
    while (p2 * 2 <= ks && p2 * 2 <= cluster_cap) p2 *= 2;
    t.ksplit = p2;
  } else {
    const int cps = (chunks + ks - 1) / ks;
    t.ksplit = (chunks + cps - 1) / cps;                    // no empty splits
  }
  t.ldP = t.n_tiles * t.NT;
  t.p_floats = (size_t)t.ksplit * t.m_tiles * 128 * t.ldP;
  return t;
}

// ---- row-sharded multi-GPU state (g4r_shard.cuh): item tables live only on their owner (row i -> rank i % R, local row i / R);
// peers read parameter rows and write gradient rows through peer-mapped pointers (cudaIpc) inside the persistent kernel ----
constexpr int MGS_MAXR = 8;            // ranks of one NVSwitch box
constexpr int MGS_FLAG_STRIDE = 32;    // one cross-GPU flag per 128-byte line
constexpr int MGS_GRU_CTAS = 48;       // == FK_G (g4r_fast.cuh)
enum { MGF_ROWS = 0, MGF_APPLIED = MGS_MAXR, MGF_IN = 2 * MGS_MAXR, MGF_INAPPLIED = 3 * MGS_MAXR, MGF_DENSE = 4 * MGS_MAXR,
       MGF_COUNT = 4 * MGS_MAXR + MGS_MAXR * MGS_GRU_CTAS };
struct ShardDev {
  int R, rank, rows_local, ldW;        // ldW = ldL + 4: a table row is [Wy row | By | 0 0 0] so that one bulk copy brings both
  int NA, DSL;                         // CTAs that apply the owned rows; capacity (floats) of one GRU CTA's dense-gradient slice
  float* W[MGS_MAXR];                  // [rows_local x ldW] parameter shard of every rank (index = rank; own entry = local memory)
  float* Wx[MGS_MAXR];                 // [rows_local x ld3] input-side table shard (no-embedding mode)
  // exchange buffers: every float travels as an 8-byte (value, lock-step sequence) pair -- data and flag in one store
  float* inbox[MGS_MAXR];              // [2][R][NP][ldW] pairs: gradient rows (dSy | dby) written by rank r for the columns it scored
  float* inboxIn[MGS_MAXR];            // [2][R][B][ld3] pairs: gradient rows of the gathered input rows
  float* denseIn[MGS_MAXR];            // [2][R][MGS_GRU_CTAS][DSL] pairs: dense-gradient slices
  float* mgInLL[MGS_MAXR];             // [2][B][ld3] pairs: input rows of the next mini-batch, pushed by their owners
  unsigned int* flags[MGS_MAXR];       // [MGF_COUNT][MGS_FLAG_STRIDE] sequence flags, written by peers, polled locally
  float *W_acc, *W_vel, *Wx_acc, *Wx_vel;   // optimizer state of the owned rows (local)
  float* mgIn;                         // [B][ld3] input rows of the current mini-batch, gathered from their owners
  const int *aEnt, *aItem, *aCbeg;     // merged plan of the rows this rank owns: entries (rank << 20 | column) [CAP][R*NP], chunks [CAP][NA+1]
  const int *xEnt, *xItem, *xTot;      // owned input rows: entries (rank << 16 | lane) [CAP][R*B], count [CAP]
  const int *gX, *gM;                  // all ranks' inputs / batch sizes of the window [R][MG_CAP][B], [R][MG_CAP]
  int* abort;                          // set when a cross-GPU wait timed out
};
// synchronisation counters of the role-specialised kernel (g4r_fast.cuh), one per 128-byte line
struct FastSync {                   // one counter per 128-byte line
  unsigned int bar;      unsigned int p0[31];
  unsigned int stats;    unsigned int p1[31];
  unsigned int h_ready;  unsigned int p2[31];
  unsigned int b1_done;  unsigned int p3[31];
  unsigned int grp;      unsigned int p4[31];
  unsigned int in_done;  unsigned int p5[31];
  unsigned int rows;     unsigned int p6[31];   // k_fast_t: chunk-row (Wy / By) updates of a step complete
};
struct GridBar { unsigned int count; unsigned int gen; unsigned int pad[30]; };   // grid barrier state (persistent mode)

struct LayerDev {
  int L, ldL, ld2, ld3;
  int in_dim, ld_in;       // in_dim==0: layer 0 of no-embedding mode (input rows gathered from Wx0, no matmul)
  float *Wx, *Wx_acc, *Wx_vel;
  float *Wh, *Wh_acc, *Wh_vel;
  float *Wrz, *Wrz_acc, *Wrz_vel;
  float *Bh, *Bh_acc, *Bh_vel;
  float *Wx_g, *Wh_g, *Wrz_g, *Bh_g;   // multi-GPU: dense gradients are exported here (all-reduced) instead of applied
  float *H;                // training hidden state, physical lanes [B x ldL]
  float *Hold, *r, *z, *ah, *ht, *y;   // forward saves, compact lanes [Bmax x ldL]
  float *dvec;             // [Bmax x ld3]  (da_h | da_r | da_z)
  float *dy;               // [Bmax x ldL]  upstream gradient wrt this layer's (dropped) output
  const float* in;         // [Bmax x ld_in] input activations (layer>0: y of the layer below; layer 0: in0)
};

struct ModelDev {
  int n_items, n_layers, B, Bld, S, mode;   // mode: 0 none, 1 embed, 2 shared
  int L, ldL;                               // last layer
  int in0_dim, ld_in0;                      // width of gathered input rows for embed/shared
  int NP;                                   // capacity of score columns per step (B + S rounded up to 4)
  int NCH;                                  // number of column chunks (CTAs of the score phases)
  int loss; ActSpec fact, hact;
  float p_drop_h, p_drop_e, lr, mom, lmbd, bpreg, logq, alpha;
  int adapt; int nn_top1;                   // nn_top1 = M + n_sample term handled at run time (uses S_cfg)
  float ap1, ap1c, ap2, ap2c;               // adapt_params[0], 1 - [0], [1], 1 - [1] (rmsprop / adadelta / adam, gru4rec.py:300-381)
  float grad_cap, smoothing;                // gru4rec.py:386-389, 226-228 / 232-234
  const float* gscale;                      // grad_cap > 0: device scalar every gradient is multiplied with before its update (else nullptr)
  float* gnorm2;                            // grad_cap > 0: sum of squares of all gradients of the step
  float* stat2;                             // smoothing > 0: [NCH x B x 2] partial (sum -log(p + eps), sum p / (p + eps)) per chunk
  int S_cfg;
  int export_only;                          // multi-GPU: compute gradients only; the merged update is applied after the exchange
  uint32_t drop_seed;
  LayerDev layer[G4R_MAX_LAYERS];
  float *Wy, *Wy_acc, *Wy_vel; float *By, *By_acc, *By_vel;
  float *E, *E_acc, *E_vel;                 // embed mode table (none mode: layer[0].Wx is the table)
  float *Sx, *in0, *dSx;                    // [Bmax x ld_in0] gathered rows, dropped input, grad wrt gathered rows
  float *snapAcc, *snapVel;                 // shared mode: acc/vel rows of X taken before the Wy update
  const float *logP0t, *logP0s;             // logq * log(P0) for targets, logq * log(P0**alpha) for samples
  // step scratch
  float *O;                                 // [NP x Bld] pre-activation scores, column-major (col*Bld + b)
  float *DSY; float *DBY;                   // [NP x ldL], [NP]
  float *part;                              // [NCH x Bmax x ldL] partial dL/dh per chunk
  float *stat;                              // [NCH x Bmax x NSTAT]
  float *RS;                                // [Bmax x NSTAT] final row statistics
  float *cost;                              // [CAP]
  int   *nanflag;
  // device-resident window of the schedule + plans
  int CAP;
  const int *wX, *wY, *wSlot, *wM, *wSti, *wXnext; const uint8_t *wF, *wXflag; const uint32_t* wG;
  int *pItem, *pPos, *pTcol, *pCbeg;
  int* pKey;                                // sharded multi-GPU: owner-major sort key (owner * n_items + item) of every sorted column
  int shardR;                               // > 0: tables are row-sharded over shardR ranks (columns sorted owner-major, equal chunks)
  const int* ST;                            // sample store [rows x S] int32
};

// ------------------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ float act_fwd(const ActSpec a, float x) {
  switch (a.kind) {
    case G4R_ACT_LINEAR: return x;
    case G4R_ACT_RELU: return fmaxf(x, 0.f);
    case G4R_ACT_TANH: return tanhf(x);
    case G4R_ACT_LEAKY: return x >= 0.f ? x : a.p1 * x;
    case G4R_ACT_ELU: return x >= 0.f ? x : a.p1 * (expf(x) - 1.0f);
    case G4R_ACT_SELU: return a.p1 * (x >= 0.f ? x : a.p2 * (expf(x) - 1.0f));
    default: return x;
  }
}
// derivative given pre-activation x and output y
__device__ __forceinline__ float act_der(const ActSpec a, float x, float y) {
  switch (a.kind) {
    case G4R_ACT_LINEAR: return 1.f;
    case G4R_ACT_RELU: return x > 0.f ? 1.f : 0.f;
    case G4R_ACT_TANH: return 1.f - y * y;
    case G4R_ACT_LEAKY: return x >= 0.f ? 1.f : a.p1;
    case G4R_ACT_ELU: return x >= 0.f ? 1.f : a.p1 * expf(x);
    case G4R_ACT_SELU: return a.p1 * (x >= 0.f ? 1.f : a.p2 * expf(x));
    default: return 1.f;
  }
}

__host__ __device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16; return x;
}
// dropout mask/retain for element idx of stream `stream` at global step `gstep` (definition shared with the oracle)
__device__ __forceinline__ float drop_scale(uint32_t seed, uint32_t gstep, uint32_t stream, uint32_t idx, float retain) {
  uint32_t k = mix32(seed ^ (0x9E3779B9U * (stream + 1U)));
  k = mix32(k + gstep);
  uint32_t r = mix32(k + idx);
  float u = (float)(r >> 8) * (1.0f / 16777216.0f);
  return u < retain ? __fdiv_rn(1.0f, retain) : 0.f;
}
#define G4R_STREAM_EMBED 100u

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
// read-only path: for arrays the running kernel never writes (lets the compiler hoist the load above unrelated stores)
__device__ __forceinline__ float4 ldn4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// ------------------------------------------------------------------------------------------------
// generic CTA-tile GEMM accumulate: acc[TM][TN] += sum_k A(m,k) * B(k,n) for the thread's micro tile of a
// BM x BN CTA tile.  A(m,k), B(k,n) are fetched through functors (bounds handled by the functor).
// ------------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------------
// CTA-tile GEMM pieces.  A tile operand is always "32 x 128": 32 = the tile's M (or N) extent, 128 = a K slab,
// stored in shared memory as [128][33].  ONE non-inlined loader serves every operand of every phase (the
// persistent kernels execute each phase once per mini-batch, so code size == instruction-cache misses).
//   element(i32, i128) = base[row(i32) * s32 + (o128 + i128) * s128] * (mul ? mul[same index] : 1)
//   row(i32) = rowidx ? rowidx[i32] (negative -> 0.0) : o32 + i32 ;   masked outside lim32 / lim128
// All 16 global loads of a thread are issued into registers before the first shared-memory store.
// ------------------------------------------------------------------------------------------------
constexpr int GB = 32;    // tile edge
constexpr int GK = 128;   // K slab
constexpr int GT = 2;     // micro tile
constexpr int GEMM_THREADS = (GB / GT) * (GB / GT);   // 256
struct TileSrc {
  const float* base; const float* mul; const int* rowidx;
  long long s32, s128; int o32, o128, lim32, lim128; int fast128;
};
__device__ __forceinline__ void tile_load(float* sdst, const TileSrc t) {
  constexpr int NE = GB * GK / GEMM_THREADS;   // 16
  const int tid = threadIdx.x;
  float r[NE];
#pragma unroll
  for (int j = 0; j < NE; j++) {
    const int i = tid + j * GEMM_THREADS;
    const int i32 = t.fast128 ? i / GK : i % GB;
    const int i128 = t.fast128 ? i % GK : i / GB;
    long long row = t.rowidx ? (long long)t.rowidx[i32] : (long long)(t.o32 + i32);
    const bool ok = row >= 0 && (t.rowidx ? true : (t.o32 + i32 < t.lim32)) && (t.o128 + i128 < t.lim128);
    float v = 0.f;
    if (ok) {
      const long long off = row * t.s32 + (long long)(t.o128 + i128) * t.s128;
      v = t.base[off];
      if (t.mul) v *= t.mul[off];
    }
    r[j] = v;
  }
#pragma unroll
  for (int j = 0; j < NE; j++) {
    const int i = tid + j * GEMM_THREADS;
    const int i32 = t.fast128 ? i / GK : i % GB;
    const int i128 = t.fast128 ? i % GK : i / GB;
    sdst[i128 * (GB + 1) + i32] = r[j];
  }
}
// acc[2][2] += A-tile x B-tile over kmax slab entries (A: 32 = m, B: 32 = n)
__device__ __forceinline__ void tile_mma(float (&acc)[GT][GT], const float* sA, const float* sB, int kmax) {
  const int tx = threadIdx.x % (GB / GT), ty = threadIdx.x / (GB / GT);
#pragma unroll 2
  for (int k = 0; k < kmax; k++) {
    const float a0 = sA[k * (GB + 1) + ty * GT], a1 = sA[k * (GB + 1) + ty * GT + 1];
    const float b0 = sB[k * (GB + 1) + tx * GT], b1 = sB[k * (GB + 1) + tx * GT + 1];
    acc[0][0] = fmaf(a0, b0, acc[0][0]); acc[0][1] = fmaf(a0, b1, acc[0][1]);
    acc[1][0] = fmaf(a1, b0, acc[1][0]); acc[1][1] = fmaf(a1, b1, acc[1][1]);
  }
}
// full K loop: acc += A x B with both operands described by TileSrc (o128 is advanced per slab)
__device__ __forceinline__ void tile_gemm(float (&acc)[GT][GT], TileSrc a, TileSrc b, int K, float* sA, float* sB) {
  for (int k0 = 0; k0 < K; k0 += GK) {
    a.o128 = k0; b.o128 = k0;
    __syncthreads();
    tile_load(sA, a);
    tile_load(sB, b);
    __syncthreads();
    tile_mma(acc, sA, sB, min(GK, K - k0));
  }
}

// stage `nrows` rows of `kw` float4 into shared memory, NU 16-byte loads in flight per thread before any store
template <int NU, class FRow>
__device__ __forceinline__ void stage_rows_n(float* sdst, int sld, int nrows, int kw, FRow rowptr) {
  const int total = nrows * kw;
  for (int i0 = 0; i0 < total; i0 += NU * (int)blockDim.x) {
    float4 v[NU];
#pragma unroll
    for (int u = 0; u < NU; u++) {
      const int i = i0 + u * (int)blockDim.x + (int)threadIdx.x;
      v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i < total) { const float* rp = rowptr(i / kw); if (rp) v[u] = ld4(rp + (i % kw) * 4); }
    }
#pragma unroll
    for (int u = 0; u < NU; u++) {
      const int i = i0 + u * (int)blockDim.x + (int)threadIdx.x;
      if (i < total) st4(sdst + (i / kw) * sld + (i % kw) * 4, v[u]);
    }
  }
}
template <class FRow>
__device__ __forceinline__ void stage_rows4(float* sdst, int sld, int nrows, int kw, FRow rowptr) {
  const int total = nrows * kw;
  for (int i0 = 0; i0 < total; i0 += 4 * (int)blockDim.x) {
    float4 v[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int i = i0 + u * (int)blockDim.x + (int)threadIdx.x;
      v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i < total) { const float* rp = rowptr(i / kw); if (rp) v[u] = ld4(rp + (i % kw) * 4); }
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int i = i0 + u * (int)blockDim.x + (int)threadIdx.x;
      if (i < total) st4(sdst + (i / kw) * sld + (i % kw) * 4, v[u]);
    }
  }
}
// ------------------------------------------------------------------------------------------------
// The Adagrad(+momentum) update, written once: every kernel that trains calls these helpers (only the column role of
// k_fast_t keeps an inline copy, which avoids a register spill there).  They take the gradient already scaled
// (grad_scale).  The sparse and dense step tails are different formulas on purpose.
// ------------------------------------------------------------------------------------------------
// Adagrad scaling of one gradient against the OLD accumulator a0 (gru4rec.py:335-340): a = a0 + g^2, returns g / sqrt(a + eps)
__device__ __forceinline__ float adagrad_scale(float g, float a0, float& a) {
  a = a0 + g * g;
  return __fdiv_rn(g, sqrtf(a + G4R_EPS_ADA));
}
// sparse step of one duplicate-group member (gru4rec.py:407-431): lmbd uses p0, the row before the update; the parameter
// accumulates every member's step in ps, the velocity vl is the last member's
__device__ __forceinline__ void sparse_step(const ModelDev& md, float gs, float p0, float v0, float& ps, float& vl, bool mom) {
  const float d = md.lmbd > 0.f ? md.lr * (gs + md.lmbd * p0) : md.lr * gs;
  if (mom) { vl = md.mom * v0 - d; ps += vl; } else ps -= d;
}
// dense step (gru4rec.py:390-406): returns the new parameter; v is the velocity, read and written only with momentum
__device__ __forceinline__ float dense_step(const ModelDev& md, float gs, float p0, float& v, bool mom) {
  if (mom) { v = md.mom * v - md.lr * (gs + md.lmbd * p0); return p0 + v; }
  return p0 * (1.0f - md.lr * md.lmbd) - md.lr * gs;
}
// Adagrad(+momentum) of one element of an item row with the gradients of its duplicate group added in position order:
// every member is scaled against the old accumulator a0, acc / velocity keep the last member's, the parameter accumulates
struct SparseUpd {
  float p0, a0, v0, ps, al, vl;
  __device__ __forceinline__ void begin(float p, float a, float v) { p0 = p; a0 = a; v0 = v; ps = p; al = 0.f; vl = 0.f; }
  __device__ __forceinline__ void add(const ModelDev& md, float g, bool ada, bool mom) {
    sparse_step(md, ada ? adagrad_scale(g, a0, al) : g, p0, v0, ps, vl, mom);
  }
};
// the same on a 16-byte quad of a row; plmbd is the row the lmbd term uses (the parameter row itself unless given).
// One branch per condition covers all four components: written per component (SparseUpd::add four times), the compiler
// turns the lmbd / mom branches into selects, which changes the FMA contraction of `ps -= d` and so the rounding.
struct SparseUpd4 {
  float4 p0, a0, v0, ps, al, vl;
  __device__ __forceinline__ void begin(float4 p, float4 a, float4 v, float4 plmbd) { p0 = plmbd; a0 = a; v0 = v; ps = p; al = make_float4(0.f, 0.f, 0.f, 0.f); vl = al; }
  __device__ __forceinline__ void begin(float4 p, float4 a, float4 v) { begin(p, a, v, p); }
  __device__ __forceinline__ void add(const ModelDev& md, float4 g, bool ada, bool mom) {
    if (ada) { g.x = adagrad_scale(g.x, a0.x, al.x); g.y = adagrad_scale(g.y, a0.y, al.y); g.z = adagrad_scale(g.z, a0.z, al.z); g.w = adagrad_scale(g.w, a0.w, al.w); }
    float4 d;
    if (md.lmbd > 0.f) { d.x = md.lr * (g.x + md.lmbd * p0.x); d.y = md.lr * (g.y + md.lmbd * p0.y); d.z = md.lr * (g.z + md.lmbd * p0.z); d.w = md.lr * (g.w + md.lmbd * p0.w); }
    else { d.x = md.lr * g.x; d.y = md.lr * g.y; d.z = md.lr * g.z; d.w = md.lr * g.w; }
    if (mom) {
      vl.x = md.mom * v0.x - d.x; vl.y = md.mom * v0.y - d.y; vl.z = md.mom * v0.z - d.z; vl.w = md.mom * v0.w - d.w;
      ps.x += vl.x; ps.y += vl.y; ps.z += vl.z; ps.w += vl.w;
    } else { ps.x -= d.x; ps.y -= d.y; ps.z -= d.z; ps.w -= d.w; }
  }
};

// ------------------------------------------------------------------------------------------------
// Adaptive scalers other than Adagrad (gru4rec.py:300-329 adam, 341-366 adadelta, 367-381 rmsprop) and the update that follows
// (gru4rec.py:390-431), for ONE element of a parameter with n gradient contributions in position order (n = 1: dense).
// Only for adapt > G4R_ADAPT_ADAGRAD: Adagrad and plain SGD call the helpers above directly.
// Sparse ("sampled") parameters use the reference's duplicate-accurate forms: the decayed state receives the squared
// gradients of ALL duplicates, every duplicate is scaled with that common state (and adam's sparse first moment accumulates
// grad**2 -- sic, gru4rec.py:325); velocity: last duplicate wins; parameter: all duplicates accumulate.
// States of an element: s0 = acc, s1 = upd (adadelta) | meang (adam), s2 = countt (adam).
// ------------------------------------------------------------------------------------------------
struct OptE { float p, s0, s1, s2, v; };
__device__ __forceinline__ float grad_scale(const ModelDev& md) { return md.gscale ? *md.gscale : 1.0f; }
template <bool SPARSE, class FG>
__device__ __forceinline__ void opt_elem(const ModelDev& md, OptE& e, float p0l, int n, FG gk) {
  const float gsc = grad_scale(md);
  const int ad = md.adapt;
  const bool mom = md.mom > 0.f;
  float A = e.s0, sclr = 1.f, common = 0.f;
  if (ad == G4R_ADAPT_RMSPROP || ad == G4R_ADAPT_ADADELTA) {
    A = e.s0 * md.ap1;
    for (int k = 0; k < n; k++) { const float g = gk(k) * gsc; A += md.ap1c * g * g; }
    if (ad == G4R_ADAPT_ADADELTA) {
      sclr = __fdiv_rn(e.s1 + G4R_EPS_ADA, A + G4R_EPS_ADA);
      float U = e.s1 * md.ap1;
      for (int k = 0; k < n; k++) { const float g = gk(k) * gsc; U += md.ap1c * sclr * g * g; }
      e.s1 = U;
      sclr = sqrtf(sclr);
    } else sclr = __fdiv_rn(1.0f, sqrtf(A + G4R_EPS_ADA));
    e.s0 = A;
  } else if (ad == G4R_ADAPT_ADAM) {
    A = e.s0 * md.ap2;
    float Mg = e.s1 * md.ap1;
    for (int k = 0; k < n; k++) { const float g = gk(k) * gsc; A += md.ap2c * g * g; Mg += md.ap1c * (SPARSE ? g * g : g); }
    const float ct = e.s2 + 1.0f;
    const float bias = 1.0f - powf(md.ap1, ct);
    common = __fdiv_rn(__fdiv_rn(Mg, bias), sqrtf(__fdiv_rn(A, bias)) + G4R_EPS_ADA);
    e.s0 = A; e.s1 = Mg; e.s2 = ct;
  }
  const float v0 = e.v;
  float ps = e.p, vl = e.v;
  for (int k = 0; k < n; k++) {
    const float g = gk(k) * gsc;
    float gs;
    if (ad == G4R_ADAPT_RMSPROP) gs = g * sclr;
    else if (ad == G4R_ADAPT_ADADELTA) gs = g * sclr;
    else gs = common;
    if (SPARSE) sparse_step(md, gs, p0l, v0, ps, vl, mom);
    else ps = dense_step(md, gs, e.p, vl, mom);         // dense: one member (n = 1), so vl is still v0 here
  }
  e.p = ps; e.v = vl;
}
// number of adaptive state arrays per parameter (they sit one after the other, `stride` elements apart, behind `*.acc`)
__host__ __device__ inline int opt_states(int adapt) { return adapt == G4R_ADAPT_ADAM ? 3 : (adapt == G4R_ADAPT_ADADELTA ? 2 : (adapt == G4R_ADAPT_NONE ? 0 : 1)); }
// generic (any scaler) row update: one row of `ld` elements, n members, element-wise over the lanes of a warp / threads of a CTA
template <class FG>
__device__ __forceinline__ void opt_row_generic(const ModelDev& md, float* prow, float* arow, size_t ast, float* vrow, const float* p0row, int ld,
                                                int n, int t0, int tstep, bool write_state, FG grow /* (member k, column c) -> gradient */) {
  const int ns = opt_states(md.adapt);
  for (int c = t0; c < ld; c += tstep) {
    OptE e;
    e.p = prow[c];
    e.s0 = ns > 0 ? arow[c] : 0.f; e.s1 = ns > 1 ? arow[ast + c] : 0.f; e.s2 = ns > 2 ? arow[2 * ast + c] : 0.f;
    e.v = vrow ? vrow[c] : 0.f;
    opt_elem<true>(md, e, p0row ? p0row[c] : e.p, n, [&](int k) { return grow(k, c); });
    prow[c] = e.p;
    if (write_state) {
      if (ns > 0) arow[c] = e.s0;
      if (ns > 1) arow[ast + c] = e.s1;
      if (ns > 2) arow[2 * ast + c] = e.s2;
      if (vrow) vrow[c] = e.v;
    }
  }
}

// dense Adagrad(+momentum) on one element (gru4rec.py:330-340,390-406)
__device__ __forceinline__ void dense_update(const ModelDev& md, float* p, float* acc, float* vel, float g, size_t ast = 0) {
  if (md.adapt > G4R_ADAPT_ADAGRAD) {
    const int ns = opt_states(md.adapt);
    OptE e;
    e.p = *p; e.s0 = acc[0]; e.s1 = ns > 1 ? acc[ast] : 0.f; e.s2 = ns > 2 ? acc[2 * ast] : 0.f; e.v = vel ? *vel : 0.f;
    opt_elem<false>(md, e, e.p, 1, [&](int) { return g; });
    *p = e.p; acc[0] = e.s0;
    if (ns > 1) acc[ast] = e.s1;
    if (ns > 2) acc[2 * ast] = e.s2;
    if (vel) *vel = e.v;
    return;
  }
  g *= grad_scale(md);
  float gs = g;
  if (md.adapt == G4R_ADAPT_ADAGRAD) gs = adagrad_scale(g, *acc, *acc);
  const bool mom = md.mom > 0.f;
  float v = mom ? *vel : 0.f;
  *p = dense_step(md, gs, *p, v, mom);
  if (mom) *vel = v;
}

// ------------------------------------------------------------------------------------------------
// phase G0: gather input rows for embedding modes (gru4rec.py:440-443 / 450-451), one warp per lane
// ------------------------------------------------------------------------------------------------
__device__ void phase_gather_in(const ModelDev& md, int s, bool train, int cta, int ncta) {
  const int M = md.wM[s];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const float* tab = (md.mode == 2) ? md.Wy : md.E;
  const int ld = md.ld_in0, W = md.in0_dim;
  const uint32_t gstep = md.wG[s];
  const float retain = 1.0f - md.p_drop_e;
  for (int b = cta * nwarp + warp; b < M; b += ncta * nwarp) {
    const int item = md.wX[(size_t)s * md.B + b];
    const float* row = tab + (size_t)item * ld;
    for (int c4 = lane; c4 < ld / 4; c4 += 32) {
      float4 v = ld4(row + c4 * 4);
      st4(md.Sx + (size_t)b * ld + c4 * 4, v);
      if (train && md.p_drop_e > 0.f) {
        const uint32_t base = (uint32_t)(b * W + c4 * 4);
        v.x *= (c4 * 4 + 0 < W) ? drop_scale(md.drop_seed, gstep, G4R_STREAM_EMBED, base + 0, retain) : 0.f;
        v.y *= (c4 * 4 + 1 < W) ? drop_scale(md.drop_seed, gstep, G4R_STREAM_EMBED, base + 1, retain) : 0.f;
        v.z *= (c4 * 4 + 2 < W) ? drop_scale(md.drop_seed, gstep, G4R_STREAM_EMBED, base + 2, retain) : 0.f;
        v.w *= (c4 * 4 + 3 < W) ? drop_scale(md.drop_seed, gstep, G4R_STREAM_EMBED, base + 3, retain) : 0.f;
      }
      st4(md.in0 + (size_t)b * ld + c4 * 4, v);
      if (train && md.mode == 2) {
        if (md.Wy_acc) st4(md.snapAcc + (size_t)b * ld + c4 * 4, ld4(md.Wy_acc + (size_t)item * ld + c4 * 4));
        if (md.Wy_vel) st4(md.snapVel + (size_t)b * ld + c4 * 4, ld4(md.Wy_vel + (size_t)item * ld + c4 * 4));
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// phase F1: rz = sigmoid(vec[:, L:] + H @ Wrz)  (gru4rec.py:460 / 473).  Tile = 32 lanes x 32 gate columns.
// Hsrc: hidden-state array this pass reads/writes (training H or evaluation H), physical lanes.
// flags bit1: zero the lane's state before the step (evaluation.py:136-139).
// ------------------------------------------------------------------------------------------------
__device__ void phase_f1(const ModelDev& md, int li, int s, float* Hsrc, int tile, float* sA, float* sB) {
  const LayerDev& ly = md.layer[li];
  const int M = md.wM[s];
  const int L = ly.L;
  const int ntn = (2 * L + GB - 1) / GB;
  const int tn = tile % ntn, tm = tile / ntn;
  const int m0 = tm * GB, n0 = tn * GB;
  if (m0 >= M) return;
  __shared__ int sSlot[GB], sXi[GB];
  const float* __restrict__ Hs = Hsrc;
  const float* __restrict__ Wrz = ly.Wrz;
  const float* __restrict__ Wx = ly.Wx;
  const float* __restrict__ Bh = ly.Bh;
  const bool gathered = ly.in_dim == 0;
  // row metadata once (index -> data chains would otherwise repeat inside every load loop)
  if (threadIdx.x < GB) {
    const int b = m0 + threadIdx.x;
    int sl = -1, x = 0;
    if (b < M) {
      sl = (md.wF[(size_t)s * md.B + b] & 2) ? -1 : md.wSlot[(size_t)s * md.B + b];
      if (gathered) x = md.wX[(size_t)s * md.B + b];
    }
    sSlot[threadIdx.x] = sl; sXi[threadIdx.x] = x;
  }
  __syncthreads();
  const int tx = threadIdx.x % (GB / GT), ty = threadIdx.x / (GB / GT);
  // epilogue operands are independent of the GEMM: issue their loads first
  float pre[GT][GT];
#pragma unroll
  for (int i = 0; i < GT; i++)
#pragma unroll
    for (int j = 0; j < GT; j++) {
      const int b = m0 + ty * GT + i, c = n0 + tx * GT + j;
      float v = 0.f;
      if (b < M && c < 2 * L) {
        v = Bh[L + c];
        if (gathered) v += Wx[(size_t)sXi[ty * GT + i] * ly.ld3 + L + c];
      }
      pre[i][j] = v;
    }
  float acc[GT][GT] = {};
  tile_gemm(acc, TileSrc{Hs, nullptr, sSlot, ly.ldL, 1, 0, 0, GB, L, 1}, TileSrc{Wrz, nullptr, nullptr, 1, ly.ld2, n0, 0, 2 * L, L, 0}, L, sA, sB);
  if (!gathered)
    tile_gemm(acc, TileSrc{ly.in, nullptr, nullptr, ly.ld_in, 1, m0, 0, M, ly.in_dim, 1},
              TileSrc{Wx + L, nullptr, nullptr, 1, ly.ld3, n0, 0, 2 * L, ly.in_dim, 0}, ly.in_dim, sA, sB);
#pragma unroll
  for (int i = 0; i < GT; i++) {
    const int b = m0 + ty * GT + i;
    if (b >= M) continue;
#pragma unroll
    for (int j = 0; j < GT; j++) {
      const int c = n0 + tx * GT + j;
      if (c >= 2 * L) continue;
      const float g = sigmoidf_(acc[i][j] + pre[i][j]);
      if (c < L) ly.r[(size_t)b * ly.ldL + c] = g; else ly.z[(size_t)b * ly.ldL + (c - L)] = g;
    }
  }
  // the tiles of column block 0 also materialise the compact copy of the old hidden state (16-byte vectors)
  if (tn == 0) {
    float* __restrict__ Ho = ly.Hold;
    const int q4 = ly.ldL / 4;
    for (int i0 = 0; i0 < GB * q4; i0 += 4 * (int)blockDim.x) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int i = i0 + u * (int)blockDim.x + (int)threadIdx.x;
        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < GB * q4) { const int sl = sSlot[i / q4]; if (sl >= 0) v[u] = ld4(Hs + (size_t)sl * ly.ldL + (i % q4) * 4); }
      }
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int i = i0 + u * (int)blockDim.x + (int)threadIdx.x;
        if (i < GB * q4 && m0 + i / q4 < M) st4(Ho + (size_t)(m0 + i / q4) * ly.ldL + (i % q4) * 4, v[u]);
      }
    }
  }
}
__device__ __forceinline__ int f1_tiles(const ModelDev& md, int li, int Bmax) {
  return ((2 * md.layer[li].L + GB - 1) / GB) * ((Bmax + GB - 1) / GB);
}

// ------------------------------------------------------------------------------------------------
// phase F2: h~ = act((H*r) @ Wh + vec[:, :L]); h = (1-z) H + z h~; dropout; H_new (gru4rec.py:461-466)
// ------------------------------------------------------------------------------------------------
__device__ void phase_f2(const ModelDev& md, int li, int s, float* Hsrc, bool train, int tile, float* sA, float* sB) {
  const LayerDev& ly = md.layer[li];
  const int M = md.wM[s];
  const int L = ly.L;
  const int ntn = (L + GB - 1) / GB;
  const int tn = tile % ntn, tm = tile / ntn;
  const int m0 = tm * GB, n0 = tn * GB;
  if (m0 >= M) return;
  __shared__ int sSlot2[GB], sXi2[GB], sFl2[GB];
  const float* __restrict__ Hold = ly.Hold;
  const float* __restrict__ Rr = ly.r;
  const float* __restrict__ Zz = ly.z;
  const float* __restrict__ Wh = ly.Wh;
  const float* __restrict__ Wx = ly.Wx;
  const float* __restrict__ Bh = ly.Bh;
  const bool gathered = ly.in_dim == 0;
  if (threadIdx.x < GB) {
    const int b = m0 + threadIdx.x;
    int sl = 0, x = 0, f = 0;
    if (b < M) { sl = md.wSlot[(size_t)s * md.B + b]; f = md.wF[(size_t)s * md.B + b]; if (gathered) x = md.wX[(size_t)s * md.B + b]; }
    sSlot2[threadIdx.x] = sl; sXi2[threadIdx.x] = x; sFl2[threadIdx.x] = f;
  }
  __syncthreads();
  const int tx = threadIdx.x % (GB / GT), ty = threadIdx.x / (GB / GT);
  float pre[GT][GT], pz[GT][GT], ph[GT][GT];
#pragma unroll
  for (int i = 0; i < GT; i++)
#pragma unroll
    for (int j = 0; j < GT; j++) {
      const int b = m0 + ty * GT + i, c = n0 + tx * GT + j;
      float v = 0.f, z = 0.f, ho = 0.f;
      if (b < M && c < L) {
        v = Bh[c];
        if (gathered) v += Wx[(size_t)sXi2[ty * GT + i] * ly.ld3 + c];
        z = Zz[(size_t)b * ly.ldL + c];
        ho = Hold[(size_t)b * ly.ldL + c];
      }
      pre[i][j] = v; pz[i][j] = z; ph[i][j] = ho;
    }
  float acc[GT][GT] = {};
  tile_gemm(acc, TileSrc{Hold, Rr, nullptr, ly.ldL, 1, m0, 0, M, L, 1}, TileSrc{Wh, nullptr, nullptr, 1, ly.ldL, n0, 0, L, L, 0}, L, sA, sB);
  if (!gathered)
    tile_gemm(acc, TileSrc{ly.in, nullptr, nullptr, ly.ld_in, 1, m0, 0, M, ly.in_dim, 1},
              TileSrc{Wx, nullptr, nullptr, 1, ly.ld3, n0, 0, L, ly.in_dim, 0}, ly.in_dim, sA, sB);
  const uint32_t gstep = md.wG[s];
  const float retain = 1.0f - md.p_drop_h;
#pragma unroll
  for (int i = 0; i < GT; i++) {
    const int b = m0 + ty * GT + i;
    if (b >= M) continue;
#pragma unroll
    for (int j = 0; j < GT; j++) {
      const int c = n0 + tx * GT + j;
      if (c >= L) continue;
      const float v = acc[i][j] + pre[i][j];
      const float ht = act_fwd(md.hact, v);
      const float z = pz[i][j];
      float h = (1.0f - z) * ph[i][j] + z * ht;
      if (train && md.p_drop_h > 0.f) h *= drop_scale(md.drop_seed, gstep, (uint32_t)li, (uint32_t)(b * L + c), retain);
      ly.ah[(size_t)b * ly.ldL + c] = v;
      ly.ht[(size_t)b * ly.ldL + c] = ht;
      ly.y[(size_t)b * ly.ldL + c] = h;
      Hsrc[(size_t)sSlot2[ty * GT + i] * ly.ldL + c] = (train && (sFl2[ty * GT + i] & 1)) ? 0.f : h;
    }
  }
}
__device__ __forceinline__ int f2_tiles(const ModelDev& md, int li, int Bmax) {
  return ((md.layer[li].L + GB - 1) / GB) * ((Bmax + GB - 1) / GB);
}

// ------------------------------------------------------------------------------------------------
// phase S1: sampled scores o = h @ Sy^T + by (- logq correction) for this CTA's column chunk, plus the
// chunk's partial row statistics of the loss.  (gru4rec.py:482-496, 225-248)
// ------------------------------------------------------------------------------------------------
constexpr int SC_CT = 16;    // columns per sub tile
constexpr int SC_TB = 32;    // lanes per row tile
constexpr int SC_KT = 128;   // feature slab
constexpr int SC_LDS = SC_KT + 4;
constexpr int SC_THREADS = 256;

struct RowStat { float m, Z, A, Q, D, T, aux; };

__device__ __forceinline__ bool loss_pairwise(int loss) { return loss == G4R_LOSS_BPR_MAX || loss == G4R_LOSS_TOP1_MAX || loss == G4R_LOSS_BPR || loss == G4R_LOSS_TOP1; }
__device__ __forceinline__ bool loss_softmaxneg(int loss) { return loss == G4R_LOSS_BPR_MAX || loss == G4R_LOSS_TOP1_MAX; }

// merge (m,Z,A,Q,D) of two partial softmax-weighted sums
__device__ __forceinline__ void stat_merge(float& m, float& Z, float& A, float& Q, float& D, float m2, float Z2, float A2, float Q2, float D2) {
  const float mn = fmaxf(m, m2);
  const float e1 = (m == -INFINITY) ? 0.f : expf(m - mn), e2 = (m2 == -INFINITY) ? 0.f : expf(m2 - mn);
  Z = Z * e1 + Z2 * e2; A = A * e1 + A2 * e2; Q = Q * e1 + Q2 * e2; D = D * e1 + D2 * e2; m = mn;
}

// accumulate one score column into a row's running statistics (online softmax-style merge)
__device__ __forceinline__ void stat_add_elem(const ModelDev& md, float o, bool is_t, float t, float& m, float& Z, float& A, float& Q, float& D, float& T, float& has) {
  if (md.loss == G4R_LOSS_XE || md.loss == G4R_LOSS_XE_LOGIT) {
    stat_merge(m, Z, A, Q, D, o, 1.f, 0.f, 0.f, 0.f);
    if (is_t) { T = o; has = 1.f; }
    return;
  }
  const float y = act_fwd(md.fact, o);
  if (is_t) has = 1.f;
  if (md.loss == G4R_LOSS_BPR_MAX) {
    if (!is_t) { const float sg = sigmoidf_(t - y); stat_merge(m, Z, A, Q, D, y, 1.f, sg, y * y, sg * (1.f - sg)); }
  } else if (md.loss == G4R_LOSS_TOP1_MAX) {
    if (!is_t) { const float a1 = sigmoidf_(y - t), b1 = sigmoidf_(y * y); stat_merge(m, Z, A, Q, D, y, 1.f, a1 + b1, 0.f, a1 * (1.f - a1)); }
  } else if (md.loss == G4R_LOSS_BPR) {
    const float sg = sigmoidf_(t - y);
    A += -logf(sg);
    if (!is_t) D += 1.f - sg;
  } else {  // TOP1
    const float a1 = sigmoidf_(y - t), b1 = sigmoidf_(y * y);
    A += a1 + b1;
    if (!is_t) D += a1 * (1.f - a1);
  }
}
__device__ __forceinline__ void stat_combine(const ModelDev& md, float& m, float& Z, float& A, float& Q, float& D, float& T, float& has,
                                             float m2, float Z2, float A2, float Q2, float D2, float T2, float has2) {
  if (md.loss == G4R_LOSS_BPR || md.loss == G4R_LOSS_TOP1) { A += A2; D += D2; }
  else stat_merge(m, Z, A, Q, D, m2, Z2, A2, Q2, D2);
  if (has2 > 0.f) { T = T2; has = 1.f; }
}

__device__ void phase_score(const ModelDev& md, int s, int chunk, float* smem) {
  const int M = md.wM[s];
  const int* cbeg = md.pCbeg + (size_t)s * (md.NCH + 1);
  const int cb = cbeg[chunk], ce = cbeg[chunk + 1];
  if (cb >= ce) {   // empty chunk: neutral partial statistics
    for (int b = threadIdx.x; b < M; b += blockDim.x) {
      float* st = md.stat + ((size_t)chunk * md.B + b) * G4R_NSTAT;
      st[0] = -INFINITY; st[1] = 0.f; st[2] = 0.f; st[3] = 0.f; st[4] = 0.f; st[5] = 0.f; st[6] = 0.f; st[7] = 0.f;
    }
    return;
  }
  const int ldL = md.ldL;
  const float* __restrict__ Y = md.layer[md.n_layers - 1].y;
  const float* __restrict__ Wy = md.Wy;
  const float* __restrict__ By = md.By;
  const int* __restrict__ pItem = md.pItem + (size_t)s * md.NP;
  const int* __restrict__ pPos = md.pPos + (size_t)s * md.NP;
  const int* __restrict__ tcol = md.pTcol + (size_t)s * md.B;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float* sY = smem;                              // [SC_TB][SC_LDS]
  float* sS = sY + SC_TB * SC_LDS;               // [SC_CT][SC_LDS]
  float* sT = sS + SC_CT * SC_LDS;               // [Bmax] target activations (pairwise losses)
  float* sRun = sT + md.Bld;                     // [Bmax][8] running row statistics of this chunk
  float* sPart = sRun + (size_t)md.Bld * 8;      // [8][SC_TB][8] per-warp statistics of the current tile
  float* sBias = sPart + 8 * SC_TB * 8;          // [SC_CT] bias (- logq correction) of the sub tile's columns
  int* sIt = reinterpret_cast<int*>(sBias + SC_CT);   // [SC_CT] items, [SC_CT] positions
  const bool pw = loss_pairwise(md.loss);
  for (int b = tid; b < M; b += SC_THREADS) {
    float* r = sRun + b * 8;
    r[0] = -INFINITY; r[1] = 0.f; r[2] = 0.f; r[3] = 0.f; r[4] = 0.f; r[5] = 0.f; r[6] = 0.f; r[7] = 0.f;
  }
  // --- target activations t_b = f(o_b,target) for pairwise losses; four rows per warp in flight
  if (pw) {
    for (int bq = warp * 4; bq < M; bq += (SC_THREADS / 32) * 4) {
      int item[4];
#pragma unroll
      for (int q = 0; q < 4; q++) item[q] = (bq + q < M) ? md.wY[(size_t)s * md.B + bq + q] : -1;
      float a[4] = {0.f, 0.f, 0.f, 0.f};
      for (int c4 = lane; c4 < ldL / 4; c4 += 32) {
        float4 w[4], y[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
          w[q] = make_float4(0.f, 0.f, 0.f, 0.f); y[q] = w[q];
          if (item[q] >= 0) { w[q] = ld4(Wy + (size_t)item[q] * ldL + c4 * 4); y[q] = ld4(Y + (size_t)(bq + q) * ldL + c4 * 4); }
        }
#pragma unroll
        for (int q = 0; q < 4; q++) { a[q] = fmaf(w[q].x, y[q].x, a[q]); a[q] = fmaf(w[q].y, y[q].y, a[q]); a[q] = fmaf(w[q].z, y[q].z, a[q]); a[q] = fmaf(w[q].w, y[q].w, a[q]); }
      }
      float bias[4];
#pragma unroll
      for (int q = 0; q < 4; q++) {
        bias[q] = 0.f;
        if (lane == 0 && item[q] >= 0) { bias[q] = By[item[q]]; if (md.logq > 0.f) bias[q] -= md.logP0t[item[q]]; }
      }
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const float v = warp_sum(a[q]);
        if (lane == 0 && item[q] >= 0) sT[bq + q] = act_fwd(md.fact, v + bias[q]);
      }
    }
  }
  // --- scores, sub tile by sub tile
  for (int j0 = cb; j0 < ce; j0 += SC_CT) {
    const int nj = min(SC_CT, ce - j0);
    __syncthreads();
    if (tid < nj) {
      const int item = pItem[j0 + tid], pos = pPos[j0 + tid];
      float bz = By[item];
      if (md.logq > 0.f) bz -= (pos < M) ? md.logP0t[item] : md.logP0s[item];
      sIt[tid] = item; sBias[tid] = bz;
    }
    __syncthreads();
    for (int b0 = 0; b0 < M; b0 += SC_TB) {
      float acc0 = 0.f, acc1 = 0.f;
      for (int k0 = 0; k0 < ldL; k0 += SC_KT) {
        const int kw = min(SC_KT, ldL - k0) / 4;       // float4 per row in this slab
        if (k0 > 0) __syncthreads();
        {
          int myit[4];   // item ids of the rows this thread stages (read before any shared store)
          stage_rows4(sY, SC_LDS, SC_TB, kw, [&](int rr) -> const float* { return (b0 + rr < M) ? Y + (size_t)(b0 + rr) * ldL + k0 : nullptr; });
          (void)myit;
          stage_rows4(sS, SC_LDS, nj, kw, [&](int rr) -> const float* { return Wy + (size_t)sIt[rr] * ldL + k0; });
        }
        __syncthreads();
        const float* yr = sY + lane * SC_LDS;
        const float* s0 = sS + warp * SC_LDS;
        const float* s1 = sS + (warp + 8) * SC_LDS;
        const bool h0 = warp < nj, h1 = warp + 8 < nj;
        for (int c4 = 0; c4 < kw; c4++) {
          const float4 y = ld4(yr + c4 * 4);
          if (h0) { const float4 w = ld4(s0 + c4 * 4); acc0 = fmaf(y.x, w.x, acc0); acc0 = fmaf(y.y, w.y, acc0); acc0 = fmaf(y.z, w.z, acc0); acc0 = fmaf(y.w, w.w, acc0); }
          if (h1) { const float4 w = ld4(s1 + c4 * 4); acc1 = fmaf(y.x, w.x, acc1); acc1 = fmaf(y.y, w.y, acc1); acc1 = fmaf(y.z, w.z, acc1); acc1 = fmaf(y.w, w.w, acc1); }
        }
      }
      // this thread: lane b = b0 + lane, columns warp and warp + 8 of the sub tile
      const int b = b0 + lane;
      float m = -INFINITY, Z = 0.f, A = 0.f, Q = 0.f, D = 0.f, T = 0.f, has = 0.f;
      if (b < M) {
        const int tc = tcol[b];
        const float t = pw ? sT[b] : 0.f;
#pragma unroll
        for (int q = 0; q < 2; q++) {
          const int jj = warp + q * 8;
          if (jj < nj) {
            const float o = (q ? acc1 : acc0) + sBias[jj];
            md.O[(size_t)(j0 + jj) * md.Bld + b] = o;
            stat_add_elem(md, o, tc == j0 + jj, t, m, Z, A, Q, D, T, has);
          }
        }
      }
      float* pp = sPart + ((size_t)warp * SC_TB + lane) * 8;
      pp[0] = m; pp[1] = Z; pp[2] = A; pp[3] = Q; pp[4] = D; pp[5] = T; pp[6] = has;
      __syncthreads();
      if (tid < SC_TB && b0 + tid < M) {
        float* r = sRun + (size_t)(b0 + tid) * 8;
        float rm = r[0], rZ = r[1], rA = r[2], rQ = r[3], rD = r[4], rT = r[5], rh = r[6];
#pragma unroll
        for (int w = 0; w < 8; w++) {
          const float* q = sPart + ((size_t)w * SC_TB + tid) * 8;
          stat_combine(md, rm, rZ, rA, rQ, rD, rT, rh, q[0], q[1], q[2], q[3], q[4], q[5], q[6]);
        }
        r[0] = rm; r[1] = rZ; r[2] = rA; r[3] = rQ; r[4] = rD; r[5] = rT; r[6] = rh;
      }
      __syncthreads();
    }
  }
  for (int b = tid; b < M; b += SC_THREADS) {
    float* st = md.stat + ((size_t)chunk * md.B + b) * G4R_NSTAT;
    const float* r = sRun + (size_t)b * 8;
    st4(st, make_float4(r[0], r[1], r[2], r[3]));
    st4(st + 4, make_float4(r[4], r[5], r[6], pw ? sT[b] : 0.f));
  }
}
__host__ __device__ inline size_t score_smem_bytes(int Bld) {
  return (size_t)(SC_TB * SC_LDS + SC_CT * SC_LDS + Bld + Bld * 8 + 8 * SC_TB * 8 + SC_CT + 2 * SC_CT + 32) * sizeof(float);
}

// final row statistics RS[b] = {m, Z, A', Q', D', t or target score, loss_b} from the merged sums (gru4rec.py:225-248)
__device__ __forceinline__ void stats_finalize(const ModelDev& md, int b, int M, int N, float m, float Z, float A, float Q, float D, float T, float tt) {
  float* rs = md.RS + (size_t)b * G4R_NSTAT;
  float loss = 0.f;
  if (md.loss == G4R_LOSS_XE) {
    const float pt = __fdiv_rn(expf(T - m), Z);
    loss = -logf(pt + G4R_EPS_LOG);
    rs[0] = m; rs[1] = Z; rs[5] = T; rs[2] = pt;
  } else if (md.loss == G4R_LOSS_XE_LOGIT) {
    loss = logf(Z) - (T - m);
    rs[0] = m; rs[1] = Z; rs[5] = T;
  } else if (md.loss == G4R_LOSS_BPR_MAX) {
    const float Ap = __fdiv_rn(A, Z), Qp = __fdiv_rn(Q, Z), Dp = __fdiv_rn(D, Z);
    loss = -logf(Ap + G4R_EPS_LOG) + md.bpreg * Qp;
    rs[0] = m; rs[1] = Z; rs[2] = Ap; rs[3] = Qp; rs[4] = Dp; rs[5] = tt;
  } else if (md.loss == G4R_LOSS_TOP1_MAX) {
    const float Ap = __fdiv_rn(A, Z), Dp = __fdiv_rn(D, Z);
    loss = Ap;
    rs[0] = m; rs[1] = Z; rs[2] = Ap; rs[4] = Dp; rs[5] = tt;
  } else if (md.loss == G4R_LOSS_BPR) {
    loss = A;
    rs[4] = D; rs[5] = tt;
  } else {  // TOP1 (gru4rec.py:242-244): mean over the N columns, last term over M + n_sample; the reference subtracts a
    // COLUMN from the row-mean vector, which broadcasts to [M x M] before the sum: everything is M times the row expression
    const float c = sigmoidf_(tt * tt);
    loss = (float)M * (__fdiv_rn(A, (float)N) - __fdiv_rn(c, (float)(M + md.S_cfg)));
    rs[4] = D; rs[5] = tt;
  }
  rs[6] = loss;
}

// ------------------------------------------------------------------------------------------------
// phase S2: combine the chunk statistics of lane b (one CTA per lane; fixed combine order => deterministic)
// RS[b] = {m, Z, A', Q', D', t_or_targetO, loss_b}
// ------------------------------------------------------------------------------------------------
__device__ void phase_stats(const ModelDev& md, int s, int cta, int ncta, float* smem) {
  const int M = md.wM[s];
  const int sti = md.wSti[s];
  const int N = M + (sti >= 0 ? md.S : 0);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = blockDim.x >> 5;
  float* sW = smem;   // [nwarp][8]
  for (int b = cta; b < M; b += ncta) {
    float m = -INFINITY, Z = 0.f, A = 0.f, Q = 0.f, D = 0.f, T = 0.f, has = 0.f, tt = 0.f;
    for (int c = tid; c < md.NCH; c += blockDim.x) {
      const float* st = md.stat + ((size_t)c * md.B + b) * G4R_NSTAT;
      const float4 u = ld4(st), v = ld4(st + 4);
      stat_combine(md, m, Z, A, Q, D, T, has, u.x, u.y, u.z, u.w, v.x, v.y, v.z);
      if (c == 0) tt = v.w;      // chunk 0 is never empty
    }
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {   // fixed butterfly order
      const float m2 = __shfl_xor_sync(0xffffffffu, m, o), Z2 = __shfl_xor_sync(0xffffffffu, Z, o), A2 = __shfl_xor_sync(0xffffffffu, A, o),
                  Q2 = __shfl_xor_sync(0xffffffffu, Q, o), D2 = __shfl_xor_sync(0xffffffffu, D, o), T2 = __shfl_xor_sync(0xffffffffu, T, o),
                  h2 = __shfl_xor_sync(0xffffffffu, has, o);
      stat_combine(md, m, Z, A, Q, D, T, has, m2, Z2, A2, Q2, D2, T2, h2);
    }
    tt = __shfl_sync(0xffffffffu, tt, 0);
    __syncthreads();
    if (lane == 0) { float* w = sW + warp * 8; w[0] = m; w[1] = Z; w[2] = A; w[3] = Q; w[4] = D; w[5] = T; w[6] = has; w[7] = tt; }
    __syncthreads();
    if (tid == 0) {
      tt = sW[7];
      for (int w = 1; w < nwarp; w++) { const float* q = sW + w * 8; stat_combine(md, m, Z, A, Q, D, T, has, q[0], q[1], q[2], q[3], q[4], q[5], q[6]); }
      if (loss_softmaxneg(md.loss)) stat_merge(m, Z, A, Q, D, 0.f, 0.f, 0.f, 0.f, 0.f);   // the zeroed diagonal takes part in the max (gru4rec.py:200-202)
      stats_finalize(md, b, M, N, m, Z, A, Q, D, T, tt);
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// label smoothing (cross-entropy losses): second statistics pass over the scores once the row maximum / normaliser are final
//   S2a  per chunk and lane: sum_j l(j) (l = -log(p_j + eps) for softmax outputs, the log-softmax itself for xe_logit) and
//        sum_j p_j / (p_j + eps)
//   S2b  one CTA per lane merges the chunks in a fixed order and rewrites the lane's loss
// ------------------------------------------------------------------------------------------------
__device__ void phase_stats2a(const ModelDev& md, int s, int chunk) {
  const int M = md.wM[s];
  const int* cbeg = md.pCbeg + (size_t)s * (md.NCH + 1);
  const int cb = cbeg[chunk], ce = cbeg[chunk + 1];
  for (int b = threadIdx.x; b < M; b += blockDim.x) {
    const float m = md.RS[(size_t)b * G4R_NSTAT], Z = md.RS[(size_t)b * G4R_NSTAT + 1];
    float s1 = 0.f, f = 0.f;
    for (int j = cb; j < ce; j++) {
      const float o = md.O[(size_t)j * md.Bld + b];
      if (md.loss == G4R_LOSS_XE) { const float p = __fdiv_rn(expf(o - m), Z); s1 += -logf(p + G4R_EPS_LOG); f += __fdiv_rn(p, p + G4R_EPS_LOG); }
      else s1 += logf(Z) - (o - m);
    }
    md.stat2[((size_t)chunk * md.B + b) * 2] = s1;
    md.stat2[((size_t)chunk * md.B + b) * 2 + 1] = f;
  }
}
__device__ void phase_stats2b(const ModelDev& md, int s, int cta, int ncta, float* smem) {
  const int M = md.wM[s];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = blockDim.x >> 5;
  for (int b = cta; b < M; b += ncta) {
    float s1 = 0.f, f = 0.f;
    for (int c = tid; c < md.NCH; c += blockDim.x) { s1 += md.stat2[((size_t)c * md.B + b) * 2]; f += md.stat2[((size_t)c * md.B + b) * 2 + 1]; }
    for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); f += __shfl_xor_sync(0xffffffffu, f, o); }
    __syncthreads();
    if (lane == 0) { smem[warp * 2] = s1; smem[warp * 2 + 1] = f; }
    __syncthreads();
    if (tid == 0) {
      s1 = 0.f; f = 0.f;
      for (int w = 0; w < nwarp; w++) { s1 += smem[w * 2]; f += smem[w * 2 + 1]; }
      float* rs = md.RS + (size_t)b * G4R_NSTAT;
      const float n_out = (float)(M + md.S_cfg);
      const float c1 = 1.0f - __fdiv_rn(n_out, n_out - 1.0f) * md.smoothing, c2 = __fdiv_rn(md.smoothing, n_out - 1.0f);
      rs[3] = f;
      if (md.loss == G4R_LOSS_XE) rs[6] = c1 * (-logf(rs[2] + G4R_EPS_LOG)) + c2 * s1;
      else rs[6] = c1 * (logf(rs[1]) - (rs[5] - rs[0])) + c2 * s1;
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// grad_cap (gru4rec.py:386-389): global L2 norm over the dense gradients and the per-position gradients of the gathered rows;
// every gradient is scaled by cap / norm when norm >= cap.  One CTA, fixed summation order.
// ------------------------------------------------------------------------------------------------
__device__ void phase_gradnorm(const ModelDev& md, int s, const float* dense_flat, size_t dense_count, float* gscale, float* smem) {
  const int M = md.wM[s];
  const int N = M + (md.wSti[s] >= 0 ? md.S : 0);
  float a = 0.f;
  const int tid = threadIdx.x, nt = blockDim.x;
  for (size_t i = tid; i < (size_t)N * md.ldL; i += nt) { const float g = md.DSY[i]; a += g * g; }
  for (int i = tid; i < N; i += nt) { const float g = md.DBY[i]; a += g * g; }
  const float* G = md.mode == 0 ? md.layer[0].dvec : md.dSx;
  const int ldg = md.mode == 0 ? md.layer[0].ld3 : md.ld_in0;
  for (int i = tid; i < M * ldg; i += nt) { const float g = G[i]; a += g * g; }
  for (size_t i = tid; i < dense_count; i += nt) { const float g = dense_flat[i]; a += g * g; }
  a = warp_sum(a);
  if ((tid & 31) == 0) smem[tid >> 5] = a;
  __syncthreads();
  if (tid == 0) {
    float t = 0.f;
    for (int w = 0; w < (nt >> 5); w++) t += smem[w];
    const float norm = sqrtf(t);
    gscale[0] = norm >= md.grad_cap ? __fdiv_rn(md.grad_cap, norm) : 1.0f;
  }
}

// dL/do for element (b, column j) given final row statistics (already divided by batch_size)
__device__ __forceinline__ float loss_grad_elem(const ModelDev& md, const float* rs, float o, bool is_t, int M, int N) {
  const float invB = __fdiv_rn(1.0f, (float)md.B);
  if (md.smoothing > 0.f && (md.loss == G4R_LOSS_XE || md.loss == G4R_LOSS_XE_LOGIT)) {
    // label smoothing (gru4rec.py:226-228, 232-234): loss_i = c1 * l(target) + c2 * sum_j l(j), n_out = M + n_sample
    const float n_out = (float)(M + md.S_cfg);
    const float c1 = 1.0f - __fdiv_rn(n_out, n_out - 1.0f) * md.smoothing, c2 = __fdiv_rn(md.smoothing, n_out - 1.0f);
    const float p = __fdiv_rn(expf(o - rs[0]), rs[1]);
    if (md.loss == G4R_LOSS_XE) {
      const float f = __fdiv_rn(p, p + G4R_EPS_LOG), ft = __fdiv_rn(rs[2], rs[2] + G4R_EPS_LOG);
      return (-c2 * f - (is_t ? c1 * ft : 0.f) + p * (c2 * rs[3] + c1 * ft)) * invB;       // rs[3] = sum_j p_j / (p_j + eps)
    }
    return (-(c2 + (is_t ? c1 : 0.f)) + p * (c2 * (float)N + c1)) * invB;
  }
  if (md.loss == G4R_LOSS_XE) {
    const float p = __fdiv_rn(expf(o - rs[0]), rs[1]);
    const float fac = __fdiv_rn(rs[2], rs[2] + G4R_EPS_LOG);
    return fac * (p - (is_t ? 1.f : 0.f)) * invB;
  }
  if (md.loss == G4R_LOSS_XE_LOGIT) {
    const float p = __fdiv_rn(expf(o - rs[0]), rs[1]);
    return (p - (is_t ? 1.f : 0.f)) * invB;
  }
  const float y = act_fwd(md.fact, o);
  const float fd = act_der(md.fact, o, y);
  const float t = rs[5];
  float dy;
  if (md.loss == G4R_LOSS_BPR_MAX) {
    const float Ap = rs[2], Qp = rs[3], Dp = rs[4];
    const float invA = __fdiv_rn(1.0f, Ap + G4R_EPS_LOG);
    if (is_t) dy = -invA * Dp;
    else {
      const float sj = __fdiv_rn(expf(y - rs[0]), rs[1]);
      const float sg = sigmoidf_(t - y);
      const float dLds = -invA * sg + md.bpreg * y * y;
      const float mean = -invA * Ap + md.bpreg * Qp;
      dy = sj * (dLds - mean) + invA * sj * sg * (1.f - sg) + 2.f * md.bpreg * y * sj;
    }
  } else if (md.loss == G4R_LOSS_TOP1_MAX) {
    const float Ap = rs[2], Dp = rs[4];
    if (is_t) dy = -Dp;
    else {
      const float sj = __fdiv_rn(expf(y - rs[0]), rs[1]);
      const float a1 = sigmoidf_(y - t), b1 = sigmoidf_(y * y);
      dy = sj * ((a1 + b1) - Ap) + sj * a1 * (1.f - a1) + sj * b1 * (1.f - b1) * 2.f * y;
    }
  } else if (md.loss == G4R_LOSS_BPR) {
    if (is_t) dy = -rs[4];
    else dy = 1.f - sigmoidf_(t - y);
  } else {  // TOP1 (M times the row expression, see the statistics phase)
    const float invN = __fdiv_rn(1.0f, (float)N);
    if (is_t) {
      const float c = sigmoidf_(t * t);
      dy = -rs[4] * invN + c * (1.f - c) * 2.f * t * invN - __fdiv_rn(c * (1.f - c) * 2.f * t, (float)(M + md.S_cfg));
    } else {
      const float a1 = sigmoidf_(y - t), b1 = sigmoidf_(y * y);
      dy = (a1 * (1.f - a1) + b1 * (1.f - b1) * 2.f * y) * invN;
    }
    dy *= (float)M;
  }
  return dy * fd * invB;
}

// ------------------------------------------------------------------------------------------------
// phase S3: loss gradient for this chunk's columns, dSy / dby rows, partial dL/dh, then the sparse
// Adagrad(+momentum) update of the chunk's Wy / By rows (gru4rec.py:383-384 grads, 407-431 updates).
// Duplicates of an item are adjacent (sorted plan) and handled sequentially in position order:
// acc / velocity keep the LAST occurrence (set_subtensor), the parameter accumulates all (inc_subtensor).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void sparse_row_update(const ModelDev& md, float* __restrict__ prow, float* __restrict__ arow, float* __restrict__ vrow,
                                                  const float* gsrc, int gstride, int n_members, int lane, int ld, bool ada, bool mom, size_t ast = 0) {
  // one item, n_members duplicate positions (in position order): gsrc + k*gstride is the gradient row of member k
  if (md.adapt > G4R_ADAPT_ADAGRAD) {
    opt_row_generic(md, prow, arow, ast, vrow, nullptr, ld, n_members, lane, 32, true, [&](int k, int c) { return gsrc[(size_t)k * gstride + c]; });
    return;
  }
  const float gsc = grad_scale(md);
  for (int c4 = lane; c4 < ld / 4; c4 += 32) {
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    SparseUpd4 u;
    u.begin(ld4(prow + c4 * 4), ada ? ld4(arow + c4 * 4) : z, mom ? ld4(vrow + c4 * 4) : z);
    for (int k = 0; k < n_members; k++) {
      float4 g = ld4(gsrc + (size_t)k * gstride + c4 * 4);
      g.x *= gsc; g.y *= gsc; g.z *= gsc; g.w *= gsc;
      u.add(md, g, ada, mom);
    }
    st4(prow + c4 * 4, u.ps);
    if (ada) st4(arow + c4 * 4, u.al);
    if (mom) st4(vrow + c4 * 4, u.vl);
  }
}

// sparse update of the Wy / By rows of column chunk `chunk` (gru4rec.py:407-431): one warp per item group, members in position
// order.  gD / gDby: gradient rows of the chunk's columns (row j - cb of a shared-memory block, or the global DSY / DBY arrays)
__device__ __forceinline__ void chunk_rows_update(const ModelDev& md, const int* __restrict__ pItem, int cb, int ce, const float* gD, int gDld, int gDoff,
                                                  const float* gDby) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const int ldL = md.ldL;
  const bool ada = md.adapt == G4R_ADAPT_ADAGRAD;
  const bool mom = md.mom > 0.f;
  const size_t astW = (size_t)md.n_items * ldL, astB = (size_t)md.n_items;
  for (int j = cb + warp; j < ce; j += nwarp) {
    const int item = pItem[j];
    if (j > cb && pItem[j - 1] == item) continue;          // not a group start
    int je = j + 1;
    while (je < ce && pItem[je] == item) je++;
    const float* gsrc = gD + (size_t)(j - gDoff) * gDld;
    sparse_row_update(md, md.Wy + (size_t)item * ldL, md.Wy_acc ? md.Wy_acc + (size_t)item * ldL : nullptr,
                      md.Wy_vel ? md.Wy_vel + (size_t)item * ldL : nullptr, gsrc, gDld, je - j, lane, ldL, ada, mom, astW);
    if (md.adapt > G4R_ADAPT_ADAGRAD) {
      if (lane == 0) opt_row_generic(md, md.By + item, md.By_acc + item, astB, md.By_vel ? md.By_vel + item : nullptr, nullptr, 1, je - j, 0, 1, true,
                                     [&](int k, int) { return gDby[j - gDoff + k]; });
    } else if (lane == 0) {   // By (gru4rec.py:486-489)
      const float gsc = grad_scale(md);
      SparseUpd u;
      u.begin(md.By[item], ada ? md.By_acc[item] : 0.f, mom ? md.By_vel[item] : 0.f);
      for (int jj = j; jj < je; jj++) u.add(md, gDby[jj - gDoff] * gsc, ada, mom);
      md.By[item] = u.ps;
      if (ada) md.By_acc[item] = u.al;
      if (mom) md.By_vel[item] = u.vl;
    }
  }
}

__device__ void phase_lossgrad(const ModelDev& md, int s, int chunk, float* smem) {
  const int M = md.wM[s];
  const int sti = md.wSti[s];
  const int N = M + (sti >= 0 ? md.S : 0);
  const int* cbeg = md.pCbeg + (size_t)s * (md.NCH + 1);
  const int cb = cbeg[chunk], ce = cbeg[chunk + 1];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int ldL = md.ldL;
  const int Bp = md.Bld;
  float* sY = smem;                              // [SC_TB][SC_LDS]
  float* sS = sY + SC_TB * SC_LDS;               // [SC_CT][SC_LDS]
  float* sG = sS + SC_CT * SC_LDS;               // [SC_CT][Bp]
  float* sRS = sG + (size_t)SC_CT * Bp;          // [Bp][8] final row statistics
  float* sD = sRS + (size_t)Bp * 8;              // [SC_CT][ldL] dSy rows of the current sub tile
  float* sDby = sD + (size_t)SC_CT * ldL;        // [SC_CT]
  int* sIt = reinterpret_cast<int*>(sDby + SC_CT);   // [SC_CT] items of the sub tile
  int* sTc = sIt + SC_CT;                        // [Bp] target column of each lane
  // final row statistics (+ the step's cost, by chunk 0 in fixed order)
  for (int i = tid; i < M * 2; i += SC_THREADS) st4(sRS + i * 4, ld4(md.RS + i * 4));
  for (int b = tid; b < M; b += SC_THREADS) sTc[b] = md.pTcol[(size_t)s * md.B + b];
  __syncthreads();
  if (chunk == 0 && tid == 0) {
    float c = 0.f;
    for (int b = 0; b < M; b++) c += sRS[b * 8 + 6];
    c = __fdiv_rn(c, (float)md.B);            // cost = loss / batch_size (gru4rec.py:577)
    md.cost[s] = c;
    if (c != c) atomicExch(md.nanflag, 1);
  }
  float* part = md.part + (size_t)chunk * md.B * ldL;
  if (cb >= ce) {   // empty chunk: its partial dL/dh must read as zero
    for (int i = tid; i < M * ldL; i += SC_THREADS) part[i] = 0.f;
    return;
  }
  const float* __restrict__ Y = md.layer[md.n_layers - 1].y;
  const float* __restrict__ Wy = md.Wy;
  const int* __restrict__ pItem = md.pItem + (size_t)s * md.NP;
  const bool single = (ce - cb) <= SC_CT && !md.export_only;   // whole chunk in one sub tile: the dSy rows stay in shared memory
  for (int j0 = cb; j0 < ce; j0 += SC_CT) {
    const int nj = min(SC_CT, ce - j0);
    __syncthreads();
    if (tid < SC_CT) sIt[tid] = tid < nj ? pItem[j0 + tid] : 0;
    // gradients of the sub tile: g[b][jj] = dL/do
    for (int i0 = 0; i0 < SC_CT * Bp; i0 += 4 * SC_THREADS) {
      float ov[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int i = i0 + u * SC_THREADS + tid;
        const int jj = i / Bp, b = i % Bp;
        ov[u] = (i < SC_CT * Bp && jj < nj && b < M) ? md.O[(size_t)(j0 + jj) * Bp + b] : 0.f;
      }
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int i = i0 + u * SC_THREADS + tid;
        const int jj = i / Bp, b = i % Bp;
        if (i < SC_CT * Bp) sG[i] = (jj < nj && b < M) ? loss_grad_elem(md, sRS + (size_t)b * 8, ov[u], sTc[b] == j0 + jj, M, N) : 0.f;
      }
    }
    __syncthreads();
    for (int jj = warp; jj < nj; jj += SC_THREADS / 32) {    // dby
      float a = 0.f;
      for (int b = lane; b < M; b += 32) a += sG[jj * Bp + b];
      a = warp_sum(a);
      if (lane == 0) { sDby[jj] = a; md.DBY[j0 + jj] = a; }
    }
    for (int k0 = 0; k0 < ldL; k0 += SC_KT) {
      const int kw = min(SC_KT, ldL - k0) / 4;
      stage_rows4(sS, SC_LDS, nj, kw, [&](int rr) -> const float* { return Wy + (size_t)sIt[rr] * ldL + k0; });
      float4 d0 = make_float4(0.f, 0.f, 0.f, 0.f), d1 = d0;     // dSy for columns warp, warp+8 at feature quad `lane`
      for (int b0 = 0; b0 < M; b0 += SC_TB) {
        if (b0 > 0) __syncthreads();
        stage_rows4(sY, SC_LDS, SC_TB, kw, [&](int rr) -> const float* { return (b0 + rr < M) ? Y + (size_t)(b0 + rr) * ldL + k0 : nullptr; });
        __syncthreads();
        if (lane < kw) {
          const int nb = min(SC_TB, M - b0);
          for (int bb = 0; bb < nb; bb++) {     // dSy_j[k] += sum_b g[b][j] * y[b][k]
            const float4 y = ld4(sY + bb * SC_LDS + lane * 4);
            const float g0 = sG[warp * Bp + b0 + bb], g1 = sG[(warp + 8) * Bp + b0 + bb];
            d0.x = fmaf(g0, y.x, d0.x); d0.y = fmaf(g0, y.y, d0.y); d0.z = fmaf(g0, y.z, d0.z); d0.w = fmaf(g0, y.w, d0.w);
            d1.x = fmaf(g1, y.x, d1.x); d1.y = fmaf(g1, y.y, d1.y); d1.z = fmaf(g1, y.z, d1.z); d1.w = fmaf(g1, y.w, d1.w);
          }
          // partial dL/dh[b][k] (+)= sum_j g[b][j] * Sy_j[k] : this warp handles lanes b0 + warp + 8*q
          for (int bb = warp; bb < SC_TB && b0 + bb < M; bb += SC_THREADS / 32) {
            float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int jj = 0; jj < nj; jj++) {
              const float g = sG[jj * Bp + b0 + bb];
              const float4 w = ld4(sS + jj * SC_LDS + lane * 4);
              a.x = fmaf(g, w.x, a.x); a.y = fmaf(g, w.y, a.y); a.z = fmaf(g, w.z, a.z); a.w = fmaf(g, w.w, a.w);
            }
            float* dst = part + (size_t)(b0 + bb) * ldL + k0 + lane * 4;
            if (j0 > cb) { const float4 o = ld4(dst); a.x += o.x; a.y += o.y; a.z += o.z; a.w += o.w; }
            st4(dst, a);
          }
        }
      }
      if (lane < kw) {
        if (warp < nj) { st4(sD + (size_t)warp * ldL + k0 + lane * 4, d0); if (!single) st4(md.DSY + (size_t)(j0 + warp) * ldL + k0 + lane * 4, d0); }
        if (warp + 8 < nj) { st4(sD + (size_t)(warp + 8) * ldL + k0 + lane * 4, d1); if (!single) st4(md.DSY + (size_t)(j0 + warp + 8) * ldL + k0 + lane * 4, d1); }
      }
      __syncthreads();
    }
  }
  __syncthreads();
  if (md.export_only) return;     // multi-GPU: DSY / DBY are exchanged and the merged update is applied by k_mg_apply_rows
  // ---- sparse update of this chunk's item groups
  if (single) chunk_rows_update(md, pItem, cb, ce, sD, ldL, cb, sDby);
  else chunk_rows_update(md, pItem, cb, ce, md.DSY, ldL, 0, md.DBY);
}
// grad_cap: second pass -- the rows of the chunk are updated from the exported gradient rows, scaled by the global-norm factor
__device__ void phase_apply_rows(const ModelDev& md, int s, int chunk) {
  const int* cbeg = md.pCbeg + (size_t)s * (md.NCH + 1);
  const int cb = cbeg[chunk], ce = cbeg[chunk + 1];
  if (cb >= ce) return;
  chunk_rows_update(md, md.pItem + (size_t)s * md.NP, cb, ce, md.DSY, md.ldL, 0, md.DBY);
}
__host__ __device__ inline size_t lossgrad_smem_bytes(int Bld, int ldL) {
  return (size_t)(SC_TB * SC_LDS + SC_CT * SC_LDS + SC_CT * Bld + Bld * 8 + SC_CT * ldL + SC_CT + SC_CT + Bld + 32) * sizeof(float);
}

// ------------------------------------------------------------------------------------------------
// phase B1: elementwise part of the GRU backward (SURVEY Appendix A): dh, dz, dh~, da_h, da_z
// ------------------------------------------------------------------------------------------------
__device__ void phase_b1(const ModelDev& md, int li, int s, int cta, int ncta, int nch_override = 0) {
  const int NCHp = nch_override > 0 ? nch_override : md.NCH;      // partial dL/dh blocks to sum (tensor-core step: K splits)
  const LayerDev& ly = md.layer[li];
  const int M = md.wM[s];
  const int L = ly.L, ldL = ly.ldL;
  const bool last = (li == md.n_layers - 1);
  const uint32_t gstep = md.wG[s];
  const float retain = 1.0f - md.p_drop_h;
  const float* __restrict__ part = md.part;
  const float* __restrict__ Ht = ly.ht;
  const float* __restrict__ Ho = ly.Hold;
  const float* __restrict__ Zz = ly.z;
  const float* __restrict__ Ah = ly.ah;
  const float* __restrict__ Dy = ly.dy;
  // eight lanes cooperate on one element: each sums every 8th chunk partial (independent loads), fixed-order tree
  const int sub = threadIdx.x & 7;
  const int grp = (cta * blockDim.x + threadIdx.x) >> 3, ngrp = (ncta * blockDim.x) >> 3;
  const size_t cs = (size_t)md.B * ldL;
  const int E = M * L;
  for (int e0 = 0; e0 < E; e0 += ngrp) {
    const int e = e0 + grp;
    const bool ok = e < E;
    const int b = ok ? e / L : 0, c = ok ? e % L : 0;
    const size_t o = (size_t)b * ldL + c;
    float ht = 0.f, ho = 0.f, z = 0.f, ah = 0.f, dy = 0.f;
    if (ok && sub == 0) { ht = Ht[o]; ho = Ho[o]; z = Zz[o]; ah = Ah[o]; if (!last) dy = Dy[o]; }
    if (last) {
      float d = 0.f;
      if (ok) {
        for (int c0 = 0; c0 < NCHp; c0 += 64) {      // 8 independent loads in flight per lane, fixed summation order
          float v[8];
#pragma unroll
          for (int u = 0; u < 8; u++) { const int ch = c0 + sub + 8 * u; v[u] = ch < NCHp ? part[(size_t)ch * cs + o] : 0.f; }
          d += ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
        }
      }
      d += __shfl_xor_sync(0xffffffffu, d, 4); d += __shfl_xor_sync(0xffffffffu, d, 2); d += __shfl_xor_sync(0xffffffffu, d, 1);
      dy = d;
    }
    if (ok && sub == 0) {
      float dh = dy;
      if (md.p_drop_h > 0.f) dh *= drop_scale(md.drop_seed, gstep, (uint32_t)li, (uint32_t)(b * L + c), retain);
      const float dz = dh * (ht - ho);
      const float dht = dh * z;
      const float dah = dht * act_der(md.hact, ah, ht);
      ly.dvec[(size_t)b * ly.ld3 + c] = dah;
      ly.dvec[(size_t)b * ly.ld3 + 2 * L + c] = dz * z * (1.f - z);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// phase B2: d(H*r) = da_h @ Wh^T ; dr = d(H*r) * H ; da_r = dr r (1-r)
// ------------------------------------------------------------------------------------------------
__device__ void phase_b2(const ModelDev& md, int li, int s, int tile, float* sA, float* sB) {
  const LayerDev& ly = md.layer[li];
  const int M = md.wM[s];
  const int L = ly.L;
  const int ntn = (L + GB - 1) / GB;
  const int tn = tile % ntn, tm = tile / ntn;
  const int m0 = tm * GB, n0 = tn * GB;
  if (m0 >= M) return;
  float acc[GT][GT] = {};
  tile_gemm(acc, TileSrc{ly.dvec, nullptr, nullptr, ly.ld3, 1, m0, 0, M, L, 1}, TileSrc{ly.Wh, nullptr, nullptr, ly.ldL, 1, n0, 0, L, L, 1}, L, sA, sB);   // Wh^T
  const int tx = threadIdx.x % (GB / GT), ty = threadIdx.x / (GB / GT);
#pragma unroll
  for (int i = 0; i < GT; i++) {
    const int b = m0 + ty * GT + i;
    if (b >= M) continue;
#pragma unroll
    for (int j = 0; j < GT; j++) {
      const int c = n0 + tx * GT + j;
      if (c >= L) continue;
      const size_t o = (size_t)b * ly.ldL + c;
      const float r = ly.r[o];
      ly.dvec[(size_t)b * ly.ld3 + L + c] = acc[i][j] * ly.Hold[o] * r * (1.f - r);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// phase B3: gradient wrt the layer input: din = dvec @ Wx^T (only layers with an input matmul).
// layer > 0: becomes dy of the layer below.  layer 0 (embed/shared): dSx = din * embed-dropout mask.
// ------------------------------------------------------------------------------------------------
__device__ void phase_b3(const ModelDev& md, int li, int s, int tile, float* sA, float* sB) {
  const LayerDev& ly = md.layer[li];
  const int M = md.wM[s];
  const int L = ly.L, K = 3 * L, IN = ly.in_dim;
  const int ntn = (IN + GB - 1) / GB;
  const int tn = tile % ntn, tm = tile / ntn;
  const int m0 = tm * GB, n0 = tn * GB;
  if (m0 >= M) return;
  float acc[GT][GT] = {};
  tile_gemm(acc, TileSrc{ly.dvec, nullptr, nullptr, ly.ld3, 1, m0, 0, M, K, 1}, TileSrc{ly.Wx, nullptr, nullptr, ly.ld3, 1, n0, 0, IN, K, 1}, K, sA, sB);   // Wx^T
  const int tx = threadIdx.x % (GB / GT), ty = threadIdx.x / (GB / GT);
  const uint32_t gstep = md.wG[s];
  const float retain = 1.0f - md.p_drop_e;
#pragma unroll
  for (int i = 0; i < GT; i++) {
    const int b = m0 + ty * GT + i;
    if (b >= M) continue;
#pragma unroll
    for (int j = 0; j < GT; j++) {
      const int c = n0 + tx * GT + j;
      if (c >= IN) continue;
      float v = acc[i][j];
      if (li > 0) md.layer[li - 1].dy[(size_t)b * md.layer[li - 1].ldL + c] = v;
      else {
        if (md.p_drop_e > 0.f) v *= drop_scale(md.drop_seed, gstep, G4R_STREAM_EMBED, (uint32_t)(b * IN + c), retain);
        md.dSx[(size_t)b * md.ld_in0 + c] = v;
      }
    }
  }
}
__device__ __forceinline__ int b3_tiles(const ModelDev& md, int li, int Bmax) {
  return ((md.layer[li].in_dim + GB - 1) / GB) * ((Bmax + GB - 1) / GB);
}

// ------------------------------------------------------------------------------------------------
// phase D: dense weight gradients fused with their Adagrad(+momentum) update (gru4rec.py:390-406)
//   dWh = (H*r)^T da_h ; dWrz = H^T da_rz ; dWx = in^T dvec ; dBh = sum_b dvec
// job space: [Wh tiles | Wrz tiles | Wx tiles | Bh blocks]
// ------------------------------------------------------------------------------------------------
struct DenseJobs { int nWh, nWrz, nWx, nBh; };
__host__ __device__ inline DenseJobs dense_jobs(int L, int in_dim) {
  DenseJobs j;
  const int tl = (L + GB - 1) / GB;
  j.nWh = tl * tl;
  j.nWrz = tl * ((2 * L + GB - 1) / GB);
  j.nWx = in_dim > 0 ? ((in_dim + GB - 1) / GB) * ((3 * L + GB - 1) / GB) : 0;
  j.nBh = (3 * L + GEMM_THREADS - 1) / GEMM_THREADS;
  return j;
}
__device__ void phase_dense(const ModelDev& md, int li, int s, int job, float* sA, float* sB) {
  const LayerDev& ly = md.layer[li];
  const int M = md.wM[s];
  const int L = ly.L;
  const DenseJobs dj = dense_jobs(L, ly.in_dim);
  const int tx = threadIdx.x % (GB / GT), ty = threadIdx.x / (GB / GT);
  float acc[GT][GT] = {};
  if (job < dj.nWh) {
    const int ntn = (L + GB - 1) / GB;
    const int m0 = (job / ntn) * GB, n0 = (job % ntn) * GB;
    tile_gemm(acc, TileSrc{ly.Hold, ly.r, nullptr, 1, ly.ldL, m0, 0, L, M, 0}, TileSrc{ly.dvec, nullptr, nullptr, 1, ly.ld3, n0, 0, L, M, 0}, M, sA, sB);
#pragma unroll
    for (int i = 0; i < GT; i++)
#pragma unroll
      for (int j = 0; j < GT; j++) {
        const int rr = m0 + ty * GT + i, c = n0 + tx * GT + j;
        if (rr < L && c < L) { const size_t o = (size_t)rr * ly.ldL + c; if (md.export_only) ly.Wh_g[o] = acc[i][j]; else dense_update(md, ly.Wh + o, ly.Wh_acc ? ly.Wh_acc + o : nullptr, ly.Wh_vel ? ly.Wh_vel + o : nullptr, acc[i][j], (size_t)L * ly.ldL); }
      }
    return;
  }
  job -= dj.nWh;
  if (job < dj.nWrz) {
    const int ntn = (2 * L + GB - 1) / GB;
    const int m0 = (job / ntn) * GB, n0 = (job % ntn) * GB;
    tile_gemm(acc, TileSrc{ly.Hold, nullptr, nullptr, 1, ly.ldL, m0, 0, L, M, 0}, TileSrc{ly.dvec + L, nullptr, nullptr, 1, ly.ld3, n0, 0, 2 * L, M, 0}, M, sA, sB);
#pragma unroll
    for (int i = 0; i < GT; i++)
#pragma unroll
      for (int j = 0; j < GT; j++) {
        const int rr = m0 + ty * GT + i, c = n0 + tx * GT + j;
        if (rr < L && c < 2 * L) { const size_t o = (size_t)rr * ly.ld2 + c; if (md.export_only) ly.Wrz_g[o] = acc[i][j]; else dense_update(md, ly.Wrz + o, ly.Wrz_acc ? ly.Wrz_acc + o : nullptr, ly.Wrz_vel ? ly.Wrz_vel + o : nullptr, acc[i][j], (size_t)L * ly.ld2); }
      }
    return;
  }
  job -= dj.nWrz;
  if (job < dj.nWx) {
    const int IN = ly.in_dim;
    const int ntn = (3 * L + GB - 1) / GB;
    const int m0 = (job / ntn) * GB, n0 = (job % ntn) * GB;
    tile_gemm(acc, TileSrc{ly.in, nullptr, nullptr, 1, ly.ld_in, m0, 0, IN, M, 0}, TileSrc{ly.dvec, nullptr, nullptr, 1, ly.ld3, n0, 0, 3 * L, M, 0}, M, sA, sB);
#pragma unroll
    for (int i = 0; i < GT; i++)
#pragma unroll
      for (int j = 0; j < GT; j++) {
        const int rr = m0 + ty * GT + i, c = n0 + tx * GT + j;
        if (rr < IN && c < 3 * L) { const size_t o = (size_t)rr * ly.ld3 + c; if (md.export_only) ly.Wx_g[o] = acc[i][j]; else dense_update(md, ly.Wx + o, ly.Wx_acc ? ly.Wx_acc + o : nullptr, ly.Wx_vel ? ly.Wx_vel + o : nullptr, acc[i][j], (size_t)IN * ly.ld3); }
      }
    return;
  }
  job -= dj.nWx;
  {
    const int c = job * GEMM_THREADS + threadIdx.x;
    if (c < 3 * L) {
      float g = 0.f;
      for (int b = 0; b < M; b++) g += ly.dvec[(size_t)b * ly.ld3 + c];
      if (md.export_only) ly.Bh_g[c] = g; else dense_update(md, ly.Bh + c, ly.Bh_acc ? ly.Bh_acc + c : nullptr, ly.Bh_vel ? ly.Bh_vel + c : nullptr, g, (size_t)ly.ld3);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// phase X: sparse update of the gathered INPUT rows (gru4rec.py:407-431 applied to Wx0[X] / E[X] / Wy[X]).
// One CTA per duplicate group of X (chain through wXnext); members processed in position order.
// ------------------------------------------------------------------------------------------------
__device__ void phase_sparse_in(const ModelDev& md, int s, int b, bool apply_pass = false) {
  const int M = md.wM[s];
  if (b >= M || (md.export_only && !apply_pass)) return;
  const uint8_t xf = md.wXflag[(size_t)s * md.B + b];
  if (!(xf & 1)) return;                      // not the first position of its group
  const int item = md.wX[(size_t)s * md.B + b];
  const int* xnext = md.wXnext + (size_t)s * md.B;
  float *tab, *tacc, *tvel; const float* G; int ld, ldg;
  if (md.mode == 0) { const LayerDev& l0 = md.layer[0]; tab = l0.Wx; tacc = l0.Wx_acc; tvel = l0.Wx_vel; G = l0.dvec; ld = l0.ld3; ldg = l0.ld3; }
  else if (md.mode == 1) { tab = md.E; tacc = md.E_acc; tvel = md.E_vel; G = md.dSx; ld = md.ld_in0; ldg = md.ld_in0; }
  else { tab = md.Wy; tacc = md.Wy_acc; tvel = md.Wy_vel; G = md.dSx; ld = md.ldL; ldg = md.ld_in0; }
  const bool ada = md.adapt == G4R_ADAPT_ADAGRAD, mom = md.mom > 0.f;
  const bool shared = md.mode == 2;
  const bool write_state = !(shared && (xf & 2));     // shared: a later (Y / sample) occurrence owns acc / velocity
  float* prow = tab + (size_t)item * ld;
  if (md.adapt > G4R_ADAPT_ADAGRAD) {                 // rmsprop / adadelta / adam (no-embedding and separate-embedding modes)
    __shared__ int s_mem[64];
    __shared__ int s_n;
    if (threadIdx.x == 0) { int n = 0; for (int bb = b; bb >= 0 && n < 64; bb = xnext[bb]) s_mem[n++] = bb; s_n = n; }
    __syncthreads();
    opt_row_generic(md, prow, tacc + (size_t)item * ld, (size_t)md.n_items * ld, tvel ? tvel + (size_t)item * ld : nullptr, nullptr, ld, s_n,
                    (int)threadIdx.x, (int)blockDim.x, true, [&](int k, int c) { return G[(size_t)s_mem[k] * ldg + c]; });
    __syncthreads();
    return;
  }
  const float gsc = grad_scale(md);
  for (int c4 = threadIdx.x; c4 < ld / 4; c4 += blockDim.x) {
    const float4 pcur = ld4(prow + c4 * 4);
    float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), v0 = a0, p0 = pcur;
    if (shared) {
      p0 = ld4(md.Sx + (size_t)b * ldg + c4 * 4);         // row value before the Wy update (sparam)
      if (ada) a0 = ld4(md.snapAcc + (size_t)b * ldg + c4 * 4);
      if (mom) v0 = ld4(md.snapVel + (size_t)b * ldg + c4 * 4);
    } else {
      if (ada) a0 = ld4(tacc + (size_t)item * ld + c4 * 4);
      if (mom) v0 = ld4(tvel + (size_t)item * ld + c4 * 4);
    }
    SparseUpd4 u;
    u.begin(pcur, a0, v0, p0);
    for (int bb = b; bb >= 0; bb = xnext[bb]) {
      float4 g = ld4(G + (size_t)bb * ldg + c4 * 4);
      g.x *= gsc; g.y *= gsc; g.z *= gsc; g.w *= gsc;
      u.add(md, g, ada, mom);
    }
    st4(prow + c4 * 4, u.ps);
    if (write_state) {
      if (ada) st4(tacc + (size_t)item * ld + c4 * 4, u.al);
      if (mom) st4(tvel + (size_t)item * ld + c4 * 4, u.vl);
    }
  }
}
