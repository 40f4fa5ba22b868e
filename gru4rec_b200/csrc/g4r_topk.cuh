// g4r_topk.cuh -- per-lane top-k of the predict scores without materialising the [batch x n_items] matrix
// (g4r_predict_topk, g4r_eval.cuh).  Two kernels:
//   k_topk_score  grid (lane blocks of EV_TB, item partitions): scores the partition's item tiles against the lanes' last-layer
//                 output, keeps a candidate buffer per lane in shared memory and writes each lane's sorted partial top-k (plus, for
//                 the softmax family, the partition's (max, sum of exp) of the logits);
//   k_topk_merge  one CTA per lane: merges the partitions' lists in a fixed order and writes the final items and scores.
// Order of candidates: score descending, item index ascending on ties; the selected set and its order therefore do not depend on
// the grid shape, the partitioning or the order of the shared-memory atomics.
// Included from g4r_eval.cuh (uses EV_* and the helpers of g4r_kernels.cuh).
#pragma once

constexpr int TK_MAX_K = 256;
constexpr int TK_MERGE_THREADS = 256;
constexpr int TK_MERGE_CAP = TK_MAX_K + TK_MERGE_THREADS;       // merge buffer: k kept + room for one round of admissions
constexpr int TK_NONE = 0x7fffffff;                              // item index of an empty slot (ranks after every real item)

// (ka, ia) ranks before (kb, ib): higher score, or the same score and a lower item index.  A NaN score ranks nowhere.
__device__ __forceinline__ bool tk_before(float ka, int ia, float kb, int ib) { return ka > kb || (ka == kb && ia < ib); }

// Sorts the first n entries of (K, I) into candidate order with one warp.  Bitonic network in its "mirror" form: every
// compare-exchange moves the better entry to the lower position, so the virtual padding up to the next power of two (empty slots,
// which rank last) never has to be stored or touched.
__device__ void tk_warp_sort(float* K, int* I, int n) {
  const int lane = threadIdx.x & 31;
  int N = 1;
  while (N < n) N <<= 1;
  auto cx = [&](int i, int j) {
    if (j >= n) return;
    const float ki = K[i], kj = K[j];
    const int ii = I[i], ij = I[j];
    if (tk_before(kj, ij, ki, ii)) { K[i] = kj; K[j] = ki; I[i] = ij; I[j] = ii; }
  };
  for (int size = 2; size <= N; size <<= 1) {
    const int half = size >> 1;
    for (int t = lane; t < N / 2; t += 32) {
      const int i = (t / half) * size + (t % half);
      cx(i, i ^ (size - 1));
    }
    __syncwarp();
    for (int stride = size >> 2; stride > 0; stride >>= 1) {
      for (int t = lane; t < N / 2; t += 32) {
        const int i = 2 * t - (t & (stride - 1));
        cx(i, i + stride);
      }
      __syncwarp();
    }
  }
}

// Keeps the best k of the n entries of a buffer (one warp): sort, cut to k, and make the k-th entry the admission threshold
// (an empty slot while fewer than k entries have been seen, so everything is admitted).  *cnt may have counted past the end of
// a full buffer; the caller passes n = min(*cnt, capacity).
__device__ void tk_compact(float* K, int* I, int n, int* cnt, float* thrK, int* thrI, int k) {
  __syncwarp();                                             // every lane has read the count before lane 0 rewrites it
  tk_warp_sort(K, I, n);
  if ((threadIdx.x & 31) == 0) {
    const int m = min(n, k);
    *cnt = m;
    *thrK = m == k ? K[k - 1] : -INFINITY;
    *thrI = m == k ? I[k - 1] : TK_NONE;
  }
  __syncwarp();
}

// cap: entries per lane buffer (k kept + at least one tile of admissions)
static size_t topk_score_smem_bytes(int cap) {
  return (size_t)(EV_TB * EV_LDS + EV_IT * EV_LDS) * sizeof(float)          // sY, sW
         + (size_t)EV_TB * cap * (sizeof(float) + sizeof(int))             // candidate buffers
         + (size_t)EV_TB * 3 * sizeof(int) + 2 * 8 * EV_TB * sizeof(float) + 64;
}

// The tile loop repeats k_eval_score's arithmetic (same smem staging, same sequential-k fmaf chain per score, then + By), so every
// pre-activation score is bitwise equal to what g4r_predict writes.  It is a separate copy because the loop nest is inverted:
// k_eval_score holds one item tile per CTA and walks the lanes; here a CTA holds one block of lanes (their hidden output staged
// once when it fits one slab) and walks the item tiles of its partition, which is what lets the candidate buffers stay resident.
// parts: number of partitions (gridDim.y); the partition p covers item tiles [p * T / parts, (p + 1) * T / parts).
// cap >= k + EV_IT: a full buffer is cut back to k, which leaves room for every admission of a tile that did not fit.
__global__ void __launch_bounds__(EV_THREADS) k_topk_score(int slot, const int* __restrict__ subset, int n_cand, int k, int cap,
                                                           float* __restrict__ pK, int* __restrict__ pI, float* __restrict__ pMZ) {
  const ModelDev& md = MD;
  extern __shared__ __align__(16) float smem[];
  float* sY = smem;                                         // [EV_TB][EV_LDS]
  float* sW = sY + EV_TB * EV_LDS;                          // [EV_IT][EV_LDS]
  float* bK = sW + EV_IT * EV_LDS;                          // [EV_TB][cap]
  int* bI = reinterpret_cast<int*>(bK + EV_TB * cap);       // [EV_TB][cap]
  int* sCnt = bI + EV_TB * cap;                             // [EV_TB]
  int* sThrI = sCnt + EV_TB;                                // [EV_TB]
  float* sThrK = reinterpret_cast<float*>(sThrI + EV_TB);   // [EV_TB]
  float* sMZ = sThrK + EV_TB;                               // [2][8][EV_TB] per-warp softmax partials
  const int M = md.wM[0];
  const int I = subset ? n_cand : md.n_items, ldL = md.ldL;
  const int b0 = blockIdx.x * EV_TB, parts = gridDim.y, p = blockIdx.y;
  const int T = (I + EV_IT - 1) / EV_IT;
  const int t_beg = (int)((long long)p * T / parts), t_end = (int)((long long)(p + 1) * T / parts);
  auto item_of = [&](int pos) -> int { return subset ? subset[pos] : pos; };
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* Y = md.layer[md.n_layers - 1].y;
  const bool elementwise = md.fact.kind <= G4R_ACT_SELU;
  const bool hoist = ldL <= EV_KT;
  if (tid < EV_TB) { sCnt[tid] = 0; sThrK[tid] = -INFINITY; sThrI[tid] = TK_NONE; }
  if (hoist) {
    const int kw = ldL / 4;
    for (int i = tid; i < EV_TB * kw; i += EV_THREADS) {
      const int rr = i / kw, c4 = i % kw;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (b0 + rr < M) v = ld4(Y + (size_t)(b0 + rr) * ldL + c4 * 4);
      st4(sY + rr * EV_LDS + c4 * 4, v);
    }
  }
  const int b = b0 + lane;
  float lm = -INFINITY, lz = 0.f;                           // softmax family: running (max, sum of exp) of this thread's logits
  for (int t = t_beg; t < t_end; t++) {
    const int i0 = t * EV_IT;
    const int ni = min(EV_IT, I - i0);
    float acc[8];
#pragma unroll
    for (int q = 0; q < 8; q++) acc[q] = 0.f;
    for (int k0 = 0; k0 < ldL; k0 += EV_KT) {
      const int kw = min(EV_KT, ldL - k0) / 4;
      __syncthreads();
      if (!hoist) {
        for (int i = tid; i < EV_TB * kw; i += EV_THREADS) {
          const int rr = i / kw, c4 = i % kw;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (b0 + rr < M) v = ld4(Y + (size_t)(b0 + rr) * ldL + k0 + c4 * 4);
          st4(sY + rr * EV_LDS + c4 * 4, v);
        }
      }
      for (int i = tid; i < EV_IT * kw; i += EV_THREADS) {
        const int rr = i / kw, c4 = i % kw;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (rr < ni) v = ld4(md.Wy + (size_t)item_of(i0 + rr) * ldL + k0 + c4 * 4);
        st4(sW + rr * EV_LDS + c4 * 4, v);
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
    // admission: only entries that rank before the current k-th can be in the final top-k (equal scores with a lower index do).
    // An entry that finds its buffer full stays pending; full buffers are cut back to k and the pending entries retried against
    // the new threshold (the second pass always has room: at most EV_IT entries of a lane are pending).
    unsigned int pend = 0u;
    if (b < M) {
#pragma unroll
      for (int q = 0; q < 8; q++) {
        if (warp + 8 * q < ni) {
          float sc = acc[q] + md.By[item_of(i0 + warp + 8 * q)];
          if (elementwise) sc = act_fwd(md.fact, sc);
          else if (sc > lm) { lz = lz * expf(lm - sc) + 1.f; lm = sc; }
          else lz += expf(sc - lm);
          acc[q] = sc;
          pend |= 1u << q;
        }
      }
    }
    for (;;) {
      if (pend) {
        const float tK = sThrK[lane];
        const int tI = sThrI[lane];
#pragma unroll
        for (int q = 0; q < 8; q++) {
          if (!(pend >> q & 1u)) continue;
          const int it = item_of(i0 + warp + 8 * q);
          if (!tk_before(acc[q], it, tK, tI)) { pend &= ~(1u << q); continue; }
          const int pos = atomicAdd(&sCnt[lane], 1);
          if (pos < cap) { bK[lane * cap + pos] = acc[q]; bI[lane * cap + pos] = it; pend &= ~(1u << q); }
        }
      }
      if (!__syncthreads_or(pend != 0u)) break;
      for (int l = warp; l < EV_TB; l += 8) {
        const int n = min(sCnt[l], cap);
        if (n == cap) tk_compact(bK + l * cap, bI + l * cap, n, &sCnt[l], &sThrK[l], &sThrI[l], k);
      }
      __syncthreads();
    }
  }
  __syncthreads();
  for (int l = warp; l < EV_TB; l += 8) {
    if (b0 + l >= M) continue;
    tk_compact(bK + l * cap, bI + l * cap, min(sCnt[l], cap), &sCnt[l], &sThrK[l], &sThrI[l], k);
    const int n = sCnt[l];
    const size_t o = ((size_t)(b0 + l) * parts + p) * k;
    for (int j = lane; j < k; j += 32) {
      pK[o + j] = j < n ? bK[l * cap + j] : -INFINITY;
      pI[o + j] = j < n ? bI[l * cap + j] : TK_NONE;
    }
  }
  if (!elementwise) {                                       // per-partition (max, sum of exp), warps combined in a fixed order
    sMZ[warp * EV_TB + lane] = lm; sMZ[(8 + warp) * EV_TB + lane] = lz;
    __syncthreads();
    if (warp == 0 && b < M) {
      float m = -INFINITY, z = 0.f;
      for (int w = 0; w < 8; w++) m = fmaxf(m, sMZ[w * EV_TB + lane]);
      for (int w = 0; w < 8; w++) {
        const float zw = sMZ[(8 + w) * EV_TB + lane];
        if (zw > 0.f) z += zw * expf(sMZ[w * EV_TB + lane] - m);
      }
      pMZ[((size_t)b * parts + p) * 2 + 0] = m; pMZ[((size_t)b * parts + p) * 2 + 1] = z;
    }
  }
}

// One CTA per lane: the parts x k partial lists are admitted against the running k-th entry, depth-major (the best entry of every
// partition first), so the threshold tightens early; the final order is the candidate order.  Elementwise activations return the
// ranking value itself; the softmax family returns expf(x - m) / z with (m, z) merged over the partitions in partition order.
__global__ void __launch_bounds__(TK_MERGE_THREADS) k_topk_merge(int slot, int parts, int k, const float* __restrict__ pK,
                                                                 const int* __restrict__ pI, const float* __restrict__ pMZ,
                                                                 int* __restrict__ items_out, float* __restrict__ scores_out) {
  const ModelDev& md = MD;
  __shared__ float bK[TK_MERGE_CAP];
  __shared__ int bI[TK_MERGE_CAP];
  __shared__ int sCnt, sThrI;
  __shared__ float sThrK, sM, sZ;
  const int b = blockIdx.x, tid = threadIdx.x;
  const int n = parts * k, cap = k + TK_MERGE_THREADS;
  const float* K = pK + (size_t)b * n;
  const int* Ii = pI + (size_t)b * n;
  if (tid == 0) { sCnt = 0; sThrK = -INFINITY; sThrI = TK_NONE; }
  __syncthreads();
  for (int r0 = 0; r0 < n; r0 += TK_MERGE_THREADS) {
    const int f = r0 + tid;
    float kk = -INFINITY;
    int ii = TK_NONE;
    if (f < n) { const int e = (f % parts) * k + f / parts; kk = K[e]; ii = Ii[e]; }
    bool pend = ii != TK_NONE;
    for (;;) {
      if (pend) {
        if (!tk_before(kk, ii, sThrK, sThrI)) pend = false;
        else {
          const int pos = atomicAdd(&sCnt, 1);
          if (pos < cap) { bK[pos] = kk; bI[pos] = ii; pend = false; }
        }
      }
      if (!__syncthreads_or(pend)) break;
      if (tid < 32) tk_compact(bK, bI, min(sCnt, cap), &sCnt, &sThrK, &sThrI, k);
      __syncthreads();
    }
  }
  if (tid < 32) tk_compact(bK, bI, min(sCnt, cap), &sCnt, &sThrK, &sThrI, k);
  const bool elementwise = md.fact.kind <= G4R_ACT_SELU;
  if (!elementwise && tid == 0) {
    const float* mz = pMZ + (size_t)b * parts * 2;
    float m = -INFINITY, z = 0.f;
    for (int q = 0; q < parts; q++) m = fmaxf(m, mz[q * 2]);
    for (int q = 0; q < parts; q++) if (mz[q * 2 + 1] > 0.f) z += mz[q * 2 + 1] * expf(mz[q * 2] - m);
    sM = m; sZ = z;
  }
  __syncthreads();
  const int cnt = sCnt;
  for (int j = tid; j < k; j += TK_MERGE_THREADS) {
    const bool real = j < cnt;
    const float x = real ? bK[j] : -INFINITY;
    items_out[(size_t)b * k + j] = real ? bI[j] : -1;
    scores_out[(size_t)b * k + j] = elementwise ? x : __fdiv_rn(expf(x - sM), sZ);
  }
}
