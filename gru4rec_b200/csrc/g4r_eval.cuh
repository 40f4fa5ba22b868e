// g4r_eval.cuh -- scoring path: evaluate_gpu's compiled function (evaluation.py:57-76) and predict
// (gru4rec.py:699-710).  Full-catalogue scores are never materialised for evaluation: each CTA scores a tile of
// consecutive items against all lanes and counts how many beat / tie the lane's target score.
// Included at the end of g4r_lib.cu (uses its handle type and helper macros).
#pragma once
#include "g4r_eval_tc.cuh"

constexpr int EV_IT = 64;     // items per CTA tile
constexpr int EV_TB = 32;     // lanes per row tile
constexpr int EV_KT = 128;    // feature slab
constexpr int EV_LDS = EV_KT + 4;
constexpr int EV_THREADS = 256;

#include "g4r_topk.cuh"

// mode 'tiebreaking' (evaluation.py:55,65): yhat += U(0,1) * 1e-10 before the standard ranking.  The reference draws the noise
// from Theano's MRG stream (not reproducible offline); here it is a counter hash of (evaluation step, lane, score column), so
// the target's own column carries the same noise in the target score and in the tile and never beats itself.
__device__ __forceinline__ float tie_noise(unsigned int seed, int s, int b, unsigned int col) {
  unsigned int k = mix32(seed ^ (0x9E3779B9U * (unsigned int)(s + 1)));
  k = mix32(k + (unsigned int)b * 0x85EBCA6BU);
  return (float)(mix32(k + col) >> 8) * (1.0f / 16777216.0f) * 1e-10f;
}

// target score of every lane, computed with the same sequential k order as the tile kernel (bitwise equal)
__global__ void __launch_bounds__(128) k_eval_tgt(int slot, int s, float* tgt, int* cnt, unsigned int tie, int subset_mode, int lohi_stride) {
  const ModelDev& md = MD;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  const int M = md.wM[s];
  if (b >= M) return;
  const int item = md.wY[(size_t)s * md.B + b];
  const float* yr = md.layer[md.n_layers - 1].y + (size_t)b * md.ldL;
  const float* wr = md.Wy + (size_t)item * md.ldL;
  float a = 0.f;
#pragma unroll 8
  for (int c4 = 0; c4 < md.ldL / 4; c4++) {          // loads batched by the unroll, the fma chain keeps its order
    const float4 y = ld4(yr + c4 * 4), w = ld4(wr + c4 * 4);
    a = fmaf(y.x, w.x, a); a = fmaf(y.y, w.y, a); a = fmaf(y.z, w.z, a); a = fmaf(y.w, w.w, a);
  }
  float sc = a + md.By[item];
  const float pre = sc;
  if (md.fact.kind <= G4R_ACT_SELU) sc = act_fwd(md.fact, sc);
  if (lohi_stride > 0) {      // tcgen05 ranking: the two pre-activation thresholds of this lane (g4r_eval_tc.cuh)
    float lo, hi;
    tc_thresholds(md.fact, md.fact.kind <= G4R_ACT_SELU, sc, pre, lo, hi);
    tgt[lohi_stride + b] = lo; tgt[2 * lohi_stride + b] = hi;
  }
  if (tie) sc += tie_noise(tie, s, b, subset_mode ? 0x40000000U + (unsigned int)b : (unsigned int)item);
  tgt[b] = sc;
  cnt[b * 2 + 0] = 0; cnt[b * 2 + 1] = 0;
}

// `subset` (evaluate_gpu(items=...), evaluation.py:52-56): the competitors are the n_cand listed items instead of the catalogue
template <bool WRITE>
__global__ void __launch_bounds__(EV_THREADS) k_eval_score(int slot, int s, const float* __restrict__ tgt, int* cnt, float* out,
                                                           const int* __restrict__ subset, int n_cand, unsigned int tie = 0u) {
  const ModelDev& md = MD;
  extern __shared__ __align__(16) float smem[];
  float* sY = smem;                        // [EV_TB][EV_LDS]
  float* sW = sY + EV_TB * EV_LDS;         // [EV_IT][EV_LDS]
  int* sCnt = reinterpret_cast<int*>(sW + EV_IT * EV_LDS);   // [EV_TB][2]
  const int M = md.wM[s];
  const int I = subset ? n_cand : md.n_items, ldL = md.ldL;
  const int i0 = blockIdx.x * EV_IT;
  const int ni = min(EV_IT, I - i0);
  auto item_of = [&](int pos) -> int { return subset ? subset[pos] : pos; };
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* Y = md.layer[md.n_layers - 1].y;
  const bool hoist = ldL <= EV_KT;
  if (hoist) {
    const int kw = ldL / 4;
    for (int i = tid; i < EV_IT * kw; i += EV_THREADS) {
      const int rr = i / kw, c4 = i % kw;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (rr < ni) v = ld4(md.Wy + (size_t)item_of(i0 + rr) * ldL + c4 * 4);
      st4(sW + rr * EV_LDS + c4 * 4, v);
    }
  }
  for (int b0 = 0; b0 < M; b0 += EV_TB) {
    float acc[8];
#pragma unroll
    for (int q = 0; q < 8; q++) acc[q] = 0.f;
    if (tid < EV_TB * 2) sCnt[tid] = 0;
    for (int k0 = 0; k0 < ldL; k0 += EV_KT) {
      const int kw = min(EV_KT, ldL - k0) / 4;
      __syncthreads();
      for (int i = tid; i < EV_TB * kw; i += EV_THREADS) {
        const int rr = i / kw, c4 = i % kw;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (b0 + rr < M) v = ld4(Y + (size_t)(b0 + rr) * ldL + k0 + c4 * 4);
        st4(sY + rr * EV_LDS + c4 * 4, v);
      }
      if (!hoist) {
        for (int i = tid; i < EV_IT * kw; i += EV_THREADS) {
          const int rr = i / kw, c4 = i % kw;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (rr < ni) v = ld4(md.Wy + (size_t)item_of(i0 + rr) * ldL + k0 + c4 * 4);
          st4(sW + rr * EV_LDS + c4 * 4, v);
        }
      }
      __syncthreads();
      const float* yr = sY + lane * EV_LDS;
      for (int c4 = 0; c4 < kw; c4++) {
        const float4 y = ld4(yr + c4 * 4);
#pragma unroll
        for (int q = 0; q < 8; q++) {
          const float4 w = ld4(sW + (warp + 8 * q) * EV_LDS + c4 * 4);
          acc[q] = fmaf(y.x, w.x, acc[q]); acc[q] = fmaf(y.y, w.y, acc[q]); acc[q] = fmaf(y.z, w.z, acc[q]); acc[q] = fmaf(y.w, w.w, acc[q]);
        }
      }
    }
    const int b = b0 + lane;
    if (b < M) {
      int gt = 0, eq = 0;
      const float t = WRITE ? 0.f : tgt[b];
#pragma unroll
      for (int q = 0; q < 8; q++) {
        const int it = i0 + warp + 8 * q;
        if (warp + 8 * q < ni) {
          float sc = acc[q] + md.By[item_of(it)];
          if (WRITE) out[(size_t)b * I + it] = sc;
          else {
            if (md.fact.kind <= G4R_ACT_SELU) sc = act_fwd(md.fact, sc);
            if (tie) sc += tie_noise(tie, s, b, (unsigned int)it);
            gt += sc > t; eq += sc == t;
          }
        }
      }
      if (!WRITE) { if (gt) atomicAdd(&sCnt[lane * 2], gt); if (eq) atomicAdd(&sCnt[lane * 2 + 1], eq); }
    }
    __syncthreads();
    if (!WRITE && tid < EV_TB * 2) {
      const int bb = b0 + tid / 2;
      if (bb < M && sCnt[tid]) atomicAdd(&cnt[bb * 2 + (tid & 1)], sCnt[tid]);
    }
  }
}
static size_t eval_smem_bytes() { return (size_t)(EV_TB * EV_LDS + EV_IT * EV_LDS) * sizeof(float) + EV_TB * 2 * sizeof(int) + 64; }

// ranks + per-cutoff sums (evaluation.py:60-75), accumulated in double on the device
__global__ void __launch_bounds__(256) k_eval_rank(int slot, int s, const int* cnt, const int* cut, int n_cut, int mode, double* sums) {
  const ModelDev& md = MD;
  if (blockIdx.x != 0) return;
  const int M = md.wM[s];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  __shared__ double red[8][2];
  // one cut-off at a time: lanes strided over the threads, double sums reduced in a fixed order (deterministic)
  for (int j = 0; j < n_cut; j++) {
    double hit = 0.0, rr = 0.0;
    for (int b = tid; b < M; b += blockDim.x) {
      const int gt = cnt[b * 2], eq = cnt[b * 2 + 1];
      double rank;
      if (mode == 1) rank = (double)(gt + eq);
      else if (mode == 2) rank = (double)gt + 0.5 * (double)(eq - 1) + 1.0;
      else rank = (double)(gt + 1);
      if (rank <= (double)cut[j]) { hit += 1.0; rr += 1.0 / rank; }
    }
    for (int o = 16; o > 0; o >>= 1) { hit += __shfl_xor_sync(0xffffffffu, hit, o); rr += __shfl_xor_sync(0xffffffffu, rr, o); }
    __syncthreads();
    if (lane == 0) { red[warp][0] = hit; red[warp][1] = rr; }
    __syncthreads();
    if (tid == 0) {
      double h = 0.0, r = 0.0;
      for (int w = 0; w < (int)(blockDim.x >> 5); w++) { h += red[w][0]; r += red[w][1]; }
      sums[j] += h; sums[n_cut + j] += r;
    }
  }
}

// final activation of the predict path (gru4rec.py:499-505): elementwise, softmax, or softmax for softmax_logit
__global__ void __launch_bounds__(256) k_predict_act(int slot, float* out, int batch) {
  const ModelDev& md = MD;
  const int b = blockIdx.x;
  if (b >= batch) return;
  float* row = out + (size_t)b * md.n_items;
  const int I = md.n_items;
  __shared__ float red[32];
  if (md.fact.kind <= G4R_ACT_SELU) {
    for (int i = threadIdx.x; i < I; i += blockDim.x) row[i] = act_fwd(md.fact, row[i]);
    return;
  }
  float m = -INFINITY;
  for (int i = threadIdx.x; i < I; i += blockDim.x) m = fmaxf(m, row[i]);
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  m = red[0];
  for (int w = 1; w < (int)(blockDim.x >> 5); w++) m = fmaxf(m, red[w]);
  __syncthreads();
  float z = 0.f;
  for (int i = threadIdx.x; i < I; i += blockDim.x) z += expf(row[i] - m);
  z = warp_sum(z);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = z;
  __syncthreads();
  z = 0.f;
  for (int w = 0; w < (int)(blockDim.x >> 5); w++) z += red[w];
  for (int i = threadIdx.x; i < I; i += blockDim.x) row[i] = __fdiv_rn(expf(row[i] - m), z);
}

struct EvalCtx {
  ModelDev mde;
  int Be = 0;
  int *hX = nullptr, *hY = nullptr, *hSlot = nullptr, *hM = nullptr, *hSti = nullptr; uint8_t* hF = nullptr; uint32_t* hG = nullptr;
  int *dX = nullptr, *dY = nullptr, *dSlot = nullptr, *dM = nullptr, *dSti = nullptr; uint8_t* dF = nullptr; uint32_t* dG = nullptr;
  int* dCut = nullptr; double* dSums = nullptr; float* dOut = nullptr; size_t out_cap = 0;
  int cap = 0;
  int slot = -1;
  int* dCand = nullptr; int n_cand = 0; size_t cand_cap = 0;     // candidate subset of evaluate_gpu(items=...), item indices
  unsigned char *dAsplit = nullptr, *dBsplit = nullptr;           // tcgen05 path: hi / lo TF32 operand blocks (g4r_eval_tc.cuh)
  // g4r_predict_topk (g4r_topk.cuh): its own candidate list (the evaluation subset above is left alone), the per-partition lists,
  // the results, and per k the lane-buffer size and CTAs per SM of k_topk_score (0 = not yet computed)
  int* dTkCand = nullptr; size_t tk_cand_cap = 0;
  float* dTkK = nullptr; int* dTkI = nullptr; size_t tk_part_cap = 0;
  float* dTkMZ = nullptr; size_t tk_mz_cap = 0;
  int* dTkItems = nullptr; float* dTkScores = nullptr; size_t tk_out_cap = 0;
  int tk_cap[TK_MAX_K + 1] = {}, tk_occ[TK_MAX_K + 1] = {};
};

static void eval_release(g4r_handle* h) {
  if (!h->eval_ctx) return;
  EvalCtx& e = *static_cast<EvalCtx*>(h->eval_ctx);
  cudaFreeHost(e.hX); cudaFreeHost(e.hY); cudaFreeHost(e.hSlot); cudaFreeHost(e.hF); cudaFreeHost(e.hM); cudaFreeHost(e.hSti); cudaFreeHost(e.hG);
  cudaFree(e.dX); cudaFree(e.dY); cudaFree(e.dSlot); cudaFree(e.dF); cudaFree(e.dM); cudaFree(e.dSti); cudaFree(e.dG);
  cudaFree(e.dCut); cudaFree(e.dSums); if (e.dOut) cudaFree(e.dOut); if (e.dCand) cudaFree(e.dCand);
  if (e.dAsplit) cudaFree(e.dAsplit); if (e.dBsplit) cudaFree(e.dBsplit);
  cudaFree(e.dTkCand); cudaFree(e.dTkK); cudaFree(e.dTkI); cudaFree(e.dTkMZ); cudaFree(e.dTkItems); cudaFree(e.dTkScores);
  slot_free(e.slot);
  delete static_cast<EvalCtx*>(h->eval_ctx);
  h->eval_ctx = nullptr;
}

static int eval_ctx(g4r_handle* h, EvalCtx** out) {
  if (h->eval_ctx) { *out = static_cast<EvalCtx*>(h->eval_ctx); return G4R_OK; }
  EvalCtx e;
  e.Be = h->cfg.eval_batch_size > 0 ? h->cfg.eval_batch_size : h->cfg.batch_size;
  e.cap = 512;
  const size_t nb = (size_t)e.cap * e.Be;
  CK(cudaMallocHost(&e.hX, nb * sizeof(int))); CK(cudaMallocHost(&e.hY, nb * sizeof(int))); CK(cudaMallocHost(&e.hSlot, nb * sizeof(int)));
  CK(cudaMallocHost(&e.hF, nb)); CK(cudaMallocHost(&e.hM, e.cap * sizeof(int))); CK(cudaMallocHost(&e.hSti, e.cap * sizeof(int))); CK(cudaMallocHost(&e.hG, e.cap * sizeof(uint32_t)));
  CK(cudaMalloc(&e.dX, nb * sizeof(int))); CK(cudaMalloc(&e.dY, nb * sizeof(int))); CK(cudaMalloc(&e.dSlot, nb * sizeof(int)));
  CK(cudaMalloc(&e.dF, nb)); CK(cudaMalloc(&e.dM, e.cap * sizeof(int))); CK(cudaMalloc(&e.dSti, e.cap * sizeof(int))); CK(cudaMalloc(&e.dG, e.cap * sizeof(uint32_t)));
  CK(cudaMalloc(&e.dCut, 64 * sizeof(int))); CK(cudaMalloc(&e.dSums, 128 * sizeof(double)));
  e.mde = h->md;
  e.mde.B = e.Be;
  e.mde.wX = e.dX; e.mde.wY = e.dY; e.mde.wSlot = e.dSlot; e.mde.wM = e.dM; e.mde.wSti = e.dSti; e.mde.wF = e.dF; e.mde.wG = e.dG;
  e.slot = slot_alloc();
  if (e.slot < 0) FAIL(G4R_ERR_STATE, "too many live g4r handles in this process");
  CK(slot_upload(e.slot, e.mde, h->stream));
  cudaFuncSetAttribute(k_eval_score<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)eval_smem_bytes());
  cudaFuncSetAttribute(k_eval_score<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)eval_smem_bytes());
  int smem_optin = 0;       // k_topk_score: its lane buffers may take all the shared memory a CTA can have (topk_shape)
  if (cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->cfg.device) != cudaSuccess ||
      cudaFuncSetAttribute(k_topk_score, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin) != cudaSuccess) cudaGetLastError();
  if (cudaFuncSetAttribute(k_eval_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(TcSmem)) != cudaSuccess) cudaGetLastError();
  h->eval_ctx = new EvalCtx(e);
  *out = static_cast<EvalCtx*>(h->eval_ctx);
  return G4R_OK;
}

static int eval_forward(g4r_handle* h, EvalCtx* e, int s) {
  const ModelDev& md = e->mde;
  cudaStream_t st = h->stream;
  if (md.mode != 0) { k_gather_in<<<std::max(1, (e->Be + 7) / 8), 256, 0, st>>>(e->slot, nullptr, s, 0); h->launches++; }
  for (int li = 0; li < md.n_layers; li++) {
    const LayerDev& ly = md.layer[li];
    k_f1<<<tiles2(2 * ly.L, e->Be), GEMM_THREADS, 0, st>>>(e->slot, nullptr, s, li, h->He[li]);
    k_f2<<<tiles2(ly.L, e->Be), GEMM_THREADS, 0, st>>>(e->slot, nullptr, s, li, h->He[li], 0);
    h->launches += 2;
  }
  return G4R_OK;
}

extern "C" int g4r_eval_schedule(g4r_handle* h, const g4r_schedule* s, const int32_t* cut_off, int32_t n_cut, int32_t mode,
                                 double* recall_sum, double* mrr_sum, int64_t* n_events) {
  if (!h || !s || !cut_off || n_cut <= 0 || n_cut > 64 || !recall_sum || !mrr_sum) return G4R_ERR_INVALID;
  if (mode < 0 || mode > 3) FAIL(G4R_ERR_INVALID, "eval mode must be 0 (standard), 1 (conservative), 2 (median) or 3 (tiebreaking)");
  const unsigned int tie = mode == 3 ? 0x5bd1e995u : 0u;
  cudaSetDevice(h->cfg.device);
  EvalCtx* e = nullptr;
  int rc = eval_ctx(h, &e);
  if (rc) return rc;
  if (s->B > e->Be) FAIL(G4R_ERR_INVALID, "schedule batch size exceeds eval_batch_size");
  const int Be = e->Be, Bs = s->B, I = h->md.n_items;
  cudaStream_t st = h->stream;
  for (int i = 0; i < h->md.n_layers; i++) CK(cudaMemsetAsync(h->He[i], 0, (size_t)Be * h->md.layer[i].ldL * sizeof(float), st));   // gru4rec.py:731-733
  CK(cudaMemcpyAsync(e->dCut, cut_off, n_cut * sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(e->dSums, 0, 128 * sizeof(double), st));
  // tensor-core scoring (full-catalogue ranking of a wide batch): the item table is split once per evaluation into hi / lo
  // TF32 operand blocks; cfg.eval_tc: 1 forces the fp32 FFMA tiles, 2 forces tcgen05
  const int tc_chunks = (h->md.L + 1 + TC_KC - 1) / TC_KC,      // + the bias column
             tc_tiles = (I + TC_N - 1) / TC_N, tc_lblocks = (Be + TC_M - 1) / TC_M;
  const bool tc_possible = e->n_cand == 0 && mode != 3 && h->cfg.eval_tc != 1 && (h->cfg.eval_tc == 2 || (Bs >= 64 && I >= 2048));
  if (tc_possible) {
    if (!e->dAsplit) CK(cudaMalloc(&e->dAsplit, (size_t)tc_lblocks * tc_chunks * 2 * TC_A_BYTES));     // hidden states: blocks of 128 lanes
    if (!e->dBsplit) CK(cudaMalloc(&e->dBsplit, (size_t)tc_tiles * tc_chunks * 2 * TC_B_BYTES));       // item table: blocks of 256 items
    k_tc_split<TC_N><<<dim3(tc_tiles, tc_chunks), 256, 0, st>>>(h->md.Wy, I, h->md.ldL, h->md.L, e->dBsplit, tc_chunks, h->md.By, 0.f);
    h->launches++;
  }
  int64_t done = 0;
  while (done < s->n_steps) {
    const int64_t w = std::min<int64_t>(e->cap, s->n_steps - done);
    CK(cudaStreamSynchronize(st));   // staging buffers are reused
    for (int64_t i = 0; i < w; i++) {   // the window arrays are strided by the engine's scoring lanes
      memcpy(e->hX + i * Be, s->X.data() + (done + i) * Bs, (size_t)Bs * sizeof(int));
      memcpy(e->hY + i * Be, s->Y.data() + (done + i) * Bs, (size_t)Bs * sizeof(int));
      memcpy(e->hSlot + i * Be, s->slots.data() + (done + i) * Bs, (size_t)Bs * sizeof(int));
      memcpy(e->hF + i * Be, s->F.data() + (done + i) * Bs, (size_t)Bs);
    }
    memcpy(e->hM, s->M.data() + done, (size_t)w * sizeof(int));
    for (int64_t i = 0; i < w; i++) {
      e->hSti[i] = -1; e->hG[i] = 0;
      const int M = e->hM[i];
      for (int b = 0; b < M; b++) {
        const int x = e->hX[i * Be + b], y = e->hY[i * Be + b];
        if (x < 0 || x >= I || y < 0 || y >= I) FAIL(G4R_ERR_INDEX, "Index out of bounds");
      }
    }
    CK(cudaMemcpyAsync(e->dX, e->hX, (size_t)w * Be * sizeof(int), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(e->dY, e->hY, (size_t)w * Be * sizeof(int), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(e->dSlot, e->hSlot, (size_t)w * Be * sizeof(int), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(e->dF, e->hF, (size_t)w * Be, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(e->dM, e->hM, (size_t)w * sizeof(int), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(e->dSti, e->hSti, (size_t)w * sizeof(int), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(e->dG, e->hG, (size_t)w * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    // two streams: the GRU forward of mini-batch i+1 (st) overlaps the ranking of mini-batch i (rk).  The ranking reads the
    // hidden output only in its first kernels (target scores, operand split -- or the fp32 tile kernel itself), after which the
    // forward stream may overwrite it; everything the ranking kernels share (target scores, counters, operand blocks, metric
    // sums) is ordered by the ranking stream itself, so the sums accumulate in mini-batch order as before.
    cudaStream_t rk = h->side;
    for (int64_t i = 0; i < w; i++) {
      eval_forward(h, e, (int)i);
      CK(cudaEventRecord(h->ts_ev[0], st)); CK(cudaStreamWaitEvent(rk, h->ts_ev[0], 0));
      k_eval_tgt<<<(Be + 31) / 32, 32, 0, rk>>>(e->slot, (int)i, h->dTgt, h->dRankCnt, tie, e->n_cand > 0 ? 1 : 0, tc_possible ? Be : 0);
      const int n_comp = e->n_cand > 0 ? e->n_cand : I;
      const int M_i = e->hM[i];
      const bool tc = tc_possible && (h->cfg.eval_tc == 2 || M_i >= 64);
      if (tc) {
        k_tc_split<TC_M><<<dim3((M_i + TC_M - 1) / TC_M, tc_chunks), 256, 0, rk>>>(h->md.layer[h->md.n_layers - 1].y, M_i, h->md.ldL, h->md.L, e->dAsplit, tc_chunks, nullptr, 1.0f);
        CK(cudaEventRecord(h->ts_ev[1], rk));
        k_eval_tc<<<std::min(tc_tiles, h->n_sm), TC_THREADS, sizeof(TcSmem), rk>>>(e->slot, (int)i, h->dTgt, Be, h->dRankCnt, e->dAsplit, e->dBsplit);
        h->launches++;
      } else {
        k_eval_score<false><<<(n_comp + EV_IT - 1) / EV_IT, EV_THREADS, eval_smem_bytes(), rk>>>(e->slot, (int)i, h->dTgt, h->dRankCnt, nullptr, e->n_cand > 0 ? e->dCand : nullptr, e->n_cand, tie);
        CK(cudaEventRecord(h->ts_ev[1], rk));
      }
      CK(cudaStreamWaitEvent(st, h->ts_ev[1], 0));        // the hidden output of this mini-batch has been consumed
      k_eval_rank<<<1, 256, 0, rk>>>(e->slot, (int)i, h->dRankCnt, e->dCut, n_cut, mode, e->dSums);
      h->launches += 3;
    }
    CK(cudaEventRecord(h->ts_ev[2], rk)); CK(cudaStreamWaitEvent(st, h->ts_ev[2], 0));   // window complete before its staging is reused
    CK(cudaGetLastError());
    done += w;
  }
  std::vector<double> sums(128);
  CK(cudaMemcpyAsync(sums.data(), e->dSums, 128 * sizeof(double), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  for (int j = 0; j < n_cut; j++) { recall_sum[j] = sums[j]; mrr_sum[j] = sums[n_cut + j]; }
  if (n_events) *n_events = s->n_events;
  return G4R_OK;
}

// evaluate_gpu(items=...) (evaluation.py:52-56,84-100): the targets are ranked against this candidate list (item indices,
// duplicates allowed as in the reference) instead of the whole catalogue; n = 0 restores the full-catalogue ranking.
extern "C" int g4r_set_eval_items(g4r_handle* h, const int64_t* items, int64_t n) {
  if (!h || n < 0 || (n > 0 && !items)) return G4R_ERR_INVALID;
  cudaSetDevice(h->cfg.device);
  EvalCtx* e = nullptr;
  int rc = eval_ctx(h, &e);
  if (rc) return rc;
  if (n == 0) { e->n_cand = 0; return G4R_OK; }
  if (n > (int64_t)1 << 30) FAIL(G4R_ERR_INVALID, "too many candidate items");
  std::vector<int> tmp((size_t)n);
  for (int64_t i = 0; i < n; i++) {
    if (items[i] < 0 || items[i] >= h->md.n_items) FAIL(G4R_ERR_INDEX, "Index out of bounds");
    tmp[(size_t)i] = (int)items[i];
  }
  if (e->cand_cap < (size_t)n) { if (e->dCand) cudaFree(e->dCand); e->dCand = nullptr; e->cand_cap = 0; CK(cudaMalloc(&e->dCand, (size_t)n * sizeof(int))); e->cand_cap = (size_t)n; }
  CK(cudaMemcpyAsync(e->dCand, tmp.data(), (size_t)n * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  e->n_cand = (int)n;
  return G4R_OK;
}

extern "C" int g4r_predict(g4r_handle* h, const int32_t* X, int32_t batch, const uint8_t* reset_mask, float* out) {
  if (!h || !X || !out) return G4R_ERR_INVALID;
  cudaSetDevice(h->cfg.device);
  EvalCtx* e = nullptr;
  int rc = eval_ctx(h, &e);
  if (rc) return rc;
  const int Be = e->Be, I = h->md.n_items;
  if (batch <= 0 || batch > Be) FAIL(G4R_ERR_INVALID, "predict batch exceeds eval_batch_size");
  cudaStream_t st = h->stream;
  for (int b = 0; b < Be; b++) {
    e->hX[b] = b < batch ? X[b] : -1; e->hY[b] = 0; e->hSlot[b] = b;
    e->hF[b] = (b < batch && reset_mask && reset_mask[b]) ? 2 : 0;
    if (b < batch && (X[b] < 0 || X[b] >= I)) FAIL(G4R_ERR_INDEX, "Index out of bounds");
  }
  e->hM[0] = batch; e->hSti[0] = -1; e->hG[0] = 0;
  CK(cudaMemcpyAsync(e->dX, e->hX, (size_t)Be * sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(e->dY, e->hY, (size_t)Be * sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(e->dSlot, e->hSlot, (size_t)Be * sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(e->dF, e->hF, (size_t)Be, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(e->dM, e->hM, sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(e->dSti, e->hSti, sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(e->dG, e->hG, sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  const size_t need = (size_t)batch * I;
  if (e->out_cap < need) { if (e->dOut) cudaFree(e->dOut); CK(cudaMalloc(&e->dOut, need * sizeof(float))); e->out_cap = need; }
  eval_forward(h, e, 0);
  k_eval_score<true><<<(I + EV_IT - 1) / EV_IT, EV_THREADS, eval_smem_bytes(), st>>>(e->slot, 0, nullptr, nullptr, e->dOut, nullptr, 0);
  k_predict_act<<<batch, 256, 0, st>>>(e->slot, e->dOut, batch);
  h->launches += 2;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, e->dOut, need * sizeof(float), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return G4R_OK;
}

// Lane-buffer size of k_topk_score for this k: k + one tile at least, grown by whole tiles while the CTAs per SM stay the same
// (more slack = fewer cuts of the buffers).  Partitions of the catalogue per lane block: enough CTAs to fill the SMs once.
static int topk_shape(g4r_handle* h, EvalCtx* e, int k, int* cap, int* occ) {
  if (!e->tk_cap[k]) {
    int smem_optin = 0, o1 = 0;
    CK(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->cfg.device));
    int c = k + EV_IT;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o1, k_topk_score, EV_THREADS, topk_score_smem_bytes(c)));
    if (o1 < 1) FAIL(G4R_ERR_CUDA, "k_topk_score does not fit on a multiprocessor");
    for (int more = 0; more < 16; more++) {
      const size_t sm = topk_score_smem_bytes(c + EV_IT);
      int o = 0;
      if (sm > (size_t)smem_optin) break;
      CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, k_topk_score, EV_THREADS, sm));
      if (o < o1) break;
      c += EV_IT;
    }
    e->tk_cap[k] = c; e->tk_occ[k] = o1;
  }
  *cap = e->tk_cap[k]; *occ = e->tk_occ[k];
  return G4R_OK;
}

extern "C" int g4r_predict_topk(g4r_handle* h, const int32_t* X, int32_t batch, const uint8_t* reset_mask,
                                const int64_t* cand, int64_t n_cand, int32_t k, int32_t* items_out, float* scores_out) {
  if (!h || !X || !items_out || !scores_out || n_cand < 0 || (n_cand > 0 && !cand)) return G4R_ERR_INVALID;
  cudaSetDevice(h->cfg.device);
  EvalCtx* e = nullptr;
  int rc = eval_ctx(h, &e);
  if (rc) return rc;
  const int Be = e->Be, I = h->md.n_items;
  if (batch <= 0 || batch > Be) FAIL(G4R_ERR_INVALID, "predict batch exceeds eval_batch_size");
  if (n_cand > (int64_t)1 << 30) FAIL(G4R_ERR_INVALID, "too many candidate items");
  const int n_comp = n_cand > 0 ? (int)n_cand : I;
  if (k < 1 || k > TK_MAX_K || k > n_comp) FAIL(G4R_ERR_INVALID, "k must be in 1 .. min(256, number of candidate items)");
  for (int b = 0; b < batch; b++)
    if (X[b] < 0 || X[b] >= I) FAIL(G4R_ERR_INDEX, "Index out of bounds");
  cudaStream_t st = h->stream;
  if (n_cand > 0) {
    std::vector<int> tmp((size_t)n_cand);
    for (int64_t i = 0; i < n_cand; i++) {
      if (cand[i] < 0 || cand[i] >= I) FAIL(G4R_ERR_INDEX, "Index out of bounds");
      tmp[(size_t)i] = (int)cand[i];
    }
    std::vector<uint8_t> seen((size_t)I, 0);
    for (const int c : tmp) {
      if (seen[c]) FAIL(G4R_ERR_INVALID, "duplicate candidate item");
      seen[c] = 1;
    }
    if (e->tk_cand_cap < (size_t)n_cand) { cudaFree(e->dTkCand); e->dTkCand = nullptr; e->tk_cand_cap = 0; CK(cudaMalloc(&e->dTkCand, (size_t)n_cand * sizeof(int))); e->tk_cand_cap = (size_t)n_cand; }
    CK(cudaMemcpyAsync(e->dTkCand, tmp.data(), (size_t)n_cand * sizeof(int), cudaMemcpyHostToDevice, st));
  }
  int cap = 0, occ = 0;
  rc = topk_shape(h, e, k, &cap, &occ);
  if (rc) return rc;
  const int lblocks = (batch + EV_TB - 1) / EV_TB, tiles = (n_comp + EV_IT - 1) / EV_IT;
  // one wave of CTAs; each partition at least one tile; at most 16384 partial entries per lane for the merge
  const int parts = std::max(1, std::min({h->n_sm * occ / lblocks, tiles, 16384 / k}));
  const size_t n_part = (size_t)batch * parts * k, n_mz = (size_t)batch * parts * 2, n_out = (size_t)batch * k;
  if (e->tk_part_cap < n_part) {
    cudaFree(e->dTkK); cudaFree(e->dTkI); e->dTkK = nullptr; e->dTkI = nullptr; e->tk_part_cap = 0;
    CK(cudaMalloc(&e->dTkK, n_part * sizeof(float))); CK(cudaMalloc(&e->dTkI, n_part * sizeof(int))); e->tk_part_cap = n_part;
  }
  if (e->tk_mz_cap < n_mz) { cudaFree(e->dTkMZ); e->dTkMZ = nullptr; e->tk_mz_cap = 0; CK(cudaMalloc(&e->dTkMZ, n_mz * sizeof(float))); e->tk_mz_cap = n_mz; }
  if (e->tk_out_cap < n_out) {
    cudaFree(e->dTkItems); cudaFree(e->dTkScores); e->dTkItems = nullptr; e->dTkScores = nullptr; e->tk_out_cap = 0;
    CK(cudaMalloc(&e->dTkItems, n_out * sizeof(int))); CK(cudaMalloc(&e->dTkScores, n_out * sizeof(float))); e->tk_out_cap = n_out;
  }
  // lanes staged exactly as g4r_predict stages them: one event per lane, reset_mask -> flag 2 (zero the lane first)
  for (int b = 0; b < Be; b++) {
    e->hX[b] = b < batch ? X[b] : -1; e->hY[b] = 0; e->hSlot[b] = b;
    e->hF[b] = (b < batch && reset_mask && reset_mask[b]) ? 2 : 0;
  }
  e->hM[0] = batch; e->hSti[0] = -1; e->hG[0] = 0;
  CK(cudaMemcpyAsync(e->dX, e->hX, (size_t)Be * sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(e->dY, e->hY, (size_t)Be * sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(e->dSlot, e->hSlot, (size_t)Be * sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(e->dF, e->hF, (size_t)Be, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(e->dM, e->hM, sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(e->dSti, e->hSti, sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(e->dG, e->hG, sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  eval_forward(h, e, 0);
  k_topk_score<<<dim3(lblocks, parts), EV_THREADS, topk_score_smem_bytes(cap), st>>>(e->slot, n_cand > 0 ? e->dTkCand : nullptr, n_comp, k, cap,
                                                                                     e->dTkK, e->dTkI, e->dTkMZ);
  k_topk_merge<<<batch, TK_MERGE_THREADS, 0, st>>>(e->slot, parts, k, e->dTkK, e->dTkI, e->dTkMZ, e->dTkItems, e->dTkScores);
  h->launches += 2;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(items_out, e->dTkItems, n_out * sizeof(int), cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(scores_out, e->dTkScores, n_out * sizeof(float), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return G4R_OK;
}

// hidden state of the scoring path (predict_next_batch zeroes it when the batch size changes, gru4rec.py:696-697)
extern "C" int g4r_reset_eval_hidden(g4r_handle* h) {
  if (!h) return G4R_ERR_INVALID;
  cudaSetDevice(h->cfg.device);
  const int Be = h->cfg.eval_batch_size > 0 ? h->cfg.eval_batch_size : h->cfg.batch_size;
  for (int i = 0; i < h->md.n_layers; i++) CK(cudaMemsetAsync(h->He[i], 0, (size_t)Be * h->md.layer[i].ldL * sizeof(float), h->stream));
  return G4R_OK;
}
