// g4r_fast.cuh -- role-specialised persistent kernel for the headline shape family:
//   no-embedding mode, one GRU layer, L <= 120 (step_mode 3: L <= 128), batch <= 32, every score-column chunk <= 32 columns.
// (step_mode 2; anything else runs k_persistent / the per-phase kernels, which share all numerics.)
//
// Why: at B=32, L=100 a mini-batch is ~8 dependent phases over ~6 MB; time is memory/barrier latency.  This kernel
//  * keeps every CTA a "column CTA" owning one chunk of score columns; the chunk's Wy / Adagrad / momentum rows and
//    the target rows are PREFETCHED with TMA bulk copies (cp.async.bulk -> mbarrier complete_tx) while the GRU
//    phases of the previous step run, so the score phase starts with its operands already in shared memory;
//  * folds the row-statistics combine into the score->gradient barrier (the last CTA to arrive combines);
//  * runs the GRU phases on a group of G CTAs with group barriers; the other CTAs only wait for `h_ready`;
//  * uses monotonic release/acquire counters (no resets, no separate fences) for all synchronisation.
//
// What is computed (reference hidasib/GRU4Rec, same formulas as the generic phases in g4r_kernels.cuh):
//   F1 / F2   GRU layer in no-embedding mode, gru4rec.py:459-466 (vec = Wx0[X] + Bh, column blocks h~ | r | z, :460-462),
//             hidden dropout and the reset of finished sessions (:464-466)
//   scores    o = h Sy^T + by (- logq log P), gru4rec.py:480-496; final activations :189-223
//   stats     row statistics of the losses, gru4rec.py:225-248 (softmax_neg with the zeroed diagonal :199-203)
//   lossgrad  dL/do of SURVEY appendix A (the reference differentiates symbolically, :383-384), dSy, dby, partial dL/dh
//   update    sparse Adagrad (+momentum) with the duplicate rules of gru4rec.py:335-340,407-431 on the chunk's rows,
//             dense Adagrad (+momentum) of Wh / Wrz / Bh, :330-334,390-406, input rows Wx0[X] :407-431
#pragma once

constexpr int FK_THREADS = 512;
constexpr int FK_NW = FK_THREADS / 32;   // warps per CTA
constexpr int FK_G = 48;            // CTAs that run the GRU phases
constexpr int FK_CT = 32;           // max columns per chunk
constexpr int FK_Q = FK_CT / FK_NW;  // columns per warp
constexpr int FK_B = 32;            // max lanes
static_assert(FK_THREADS / 16 == FK_B, "statistics mapping: 16 threads per lane");
constexpr int FK_LDS = 132;         // shared row stride (floats) for L <= 128: conflict-free 16-byte accesses


__device__ __forceinline__ void red_release_add(unsigned int* p, unsigned int v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int atom_acqrel_add(unsigned int* p, unsigned int v) {
  unsigned int old;
  asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
  return old;
}
__device__ __forceinline__ void wait_ge(const unsigned int* p, unsigned int target) {
  while (ld_acquire_u32(p) < target) { }
}
// ---- mbarrier + TMA bulk copy (1-D, no tensor map): rows of ld*4 bytes, 16-byte aligned ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned int bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned int parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra.uni WAIT_DONE;\n\t"
      "bra.uni WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t}\n" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_row(void* sdst, const void* gsrc, unsigned int bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(smem_u32(sdst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

struct FastSmem {
  // column role
  alignas(128) float sY[FK_B * FK_LDS];          // h of the step (all lanes)
  float sS[FK_CT * FK_LDS];         // Wy rows of the chunk (TMA)
  float sAcc[FK_CT * FK_LDS];       // Adagrad rows (TMA)
  float sVel[FK_CT * FK_LDS];       // momentum rows (TMA)
  float sTW[FK_B * FK_LDS];         // target rows (TMA; pairwise losses)
  float sD[FK_CT * FK_LDS];         // dSy rows
  float sG[FK_CT * FK_B];           // dL/do
  float sO[FK_CT * FK_B];           // scores o
  float sRS[FK_B * 8];
  float sPart[FK_NW * FK_B * 8];
  float sT[FK_B];                   // target activations
  float sBias[FK_CT], sByP[FK_CT], sByA[FK_CT], sByV[FK_CT], sDby[FK_CT], sTB[FK_B];
  int sIt[2][FK_CT], sPos[2][FK_CT], sTc[2][FK_B], sYit[2][FK_B], sCb[2][2];
  int sFlag[4];
  alignas(8) unsigned long long mbar;
  unsigned long long sTs[2];        // %globaltimer around F1's wait for the helper CTAs (stamped runs only)
  // GRU role: thin-slab phases (every GRU CTA owns a few output columns / rows and stages the full 32-lane operand)
  alignas(16) float gA[FK_B * 388];             // staged [32 x <=384] operand (H, Hold*r, da_h, dvec)
  alignas(16) float gW[8 * FK_LDS + FK_NW * FK_B * 5 + 16 * FK_B];      // this CTA's weight slab (<= 8 columns/rows of length <= 128) + reduction scratch
  int gIdx[3 * FK_B];               // slot, item, flags of the lanes
};

// loads the index metadata of step s into buffer `buf` (plain loads; consumed much later)
template <class SM>
__device__ __forceinline__ void fk_load_idx(const ModelDev& md, SM& sm, int s, int n_steps, int chunk, int buf) {
  const int tid = threadIdx.x;
  if (s >= n_steps) return;
  const int M = md.wM[s];
  const int* cbeg = md.pCbeg + (size_t)s * (md.NCH + 1);
  const bool hc = chunk < md.NCH;
  const int cb = hc ? cbeg[chunk] : 0, ce = hc ? cbeg[chunk + 1] : 0;
  if (tid < FK_CT) {
    int it = 0, pos = 0;
    if (cb + tid < ce) { it = md.pItem[(size_t)s * md.NP + cb + tid]; pos = md.pPos[(size_t)s * md.NP + cb + tid]; }
    sm.sIt[buf][tid] = it; sm.sPos[buf][tid] = pos;
  }
  if (tid >= 32 && tid < 32 + FK_B) {
    const int b = tid - 32;
    sm.sTc[buf][b] = b < M ? md.pTcol[(size_t)s * md.B + b] : -1;
    sm.sYit[buf][b] = b < M ? md.wY[(size_t)s * md.B + b] : 0;
  }
  if (tid == 64) { sm.sCb[buf][0] = cb; sm.sCb[buf][1] = ce; }
}

// issue the TMA prefetch of step s (rows are final once the previous step's updates are complete; k_fast_t updates a
// chunk's rows after arriving at the last column barrier, so it acquires FastSync::rows before calling this)
template <class SM>
__device__ __forceinline__ void fk_prefetch_rows(const ModelDev& md, SM& sm, int s, int n_steps, int buf, bool pw) {
  if (s >= n_steps) return;
  const int tid = threadIdx.x;
  const int M = md.wM[s];
  const int cb = sm.sCb[buf][0], ce = sm.sCb[buf][1];
  const int nj = ce - cb;
  const bool ada = md.adapt == G4R_ADAPT_ADAGRAD, mom = md.mom > 0.f;
  const unsigned int rowb = (unsigned int)md.ldL * 4u;
  uint64_t* bar = reinterpret_cast<uint64_t*>(&sm.mbar);
  // bulk copies are issued one per thread-instruction; spreading them over the warps (lane 0 of each) keeps the issue
  // off the critical path (one warp issuing ~80 copies took 2.3 us)
  const int ntab = 1 + (ada ? 1 : 0) + (mom ? 1 : 0);
  const int ncopy = nj * ntab + (pw ? M : 0);
  if (tid == 0) {
    const unsigned int total = rowb * (unsigned int)ncopy;
    asm volatile("fence.proxy.async.global;" ::: "memory");
    if (total > 0) mbar_expect_tx(bar, total);
    else asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
  }
  if ((tid & 31) == 0) {
    for (int i = tid >> 5; i < ncopy; i += FK_NW) {
      if (i < nj * ntab) {
        const int j = i / ntab, t = i % ntab;
        const size_t off = (size_t)sm.sIt[buf][j] * md.ldL;
        if (t == 0) tma_row(sm.sS + j * FK_LDS, md.Wy + off, rowb, bar);
        else if (t == 1 && ada) tma_row(sm.sAcc + j * FK_LDS, md.Wy_acc + off, rowb, bar);
        else tma_row(sm.sVel + j * FK_LDS, md.Wy_vel + off, rowb, bar);
      } else {
        const int b = i - nj * ntab;
        tma_row(sm.sTW + b * FK_LDS, md.Wy + (size_t)sm.sYit[buf][b] * md.ldL, rowb, bar);
      }
    }
  }
  if (false) {
  } else if (tid >= 64 && tid < 64 + FK_CT) {
    const int j = tid - 64;
    if (j < nj) {
      const int it = sm.sIt[buf][j];
      float bz = md.By[it];
      sm.sByP[j] = bz;
      if (md.logq > 0.f) bz -= (sm.sPos[buf][j] < M) ? md.logP0t[it] : md.logP0s[it];
      sm.sBias[j] = bz;
      sm.sByA[j] = ada ? md.By_acc[it] : 0.f;
      sm.sByV[j] = mom ? md.By_vel[it] : 0.f;
    }
  } else if (tid >= 96 && tid < 96 + FK_B) {
    const int b = tid - 96;
    if (pw && b < M) {
      const int it = sm.sYit[buf][b];
      float bz = md.By[it];
      if (md.logq > 0.f) bz -= md.logP0t[it];
      sm.sTB[b] = bz;
    }
  }
}

// the TMA prefetch of step s + 1 once every CTA's chunk-row update of step s is complete
template <class SM>
__device__ __forceinline__ void fk_wait_rows_prefetch(const ModelDev& md, SM& sm, FastSync* fs, int s, int n_steps, int buf, bool pw, int ncta) {
  if (s + 1 >= n_steps) return;
  if (threadIdx.x == 0) wait_ge(&fs->rows, (unsigned int)(s + 1) * (unsigned int)ncta);
  __syncthreads();
  fk_prefetch_rows(md, sm, s + 1, n_steps, buf ^ 1, pw);
}
__device__ __forceinline__ void fk_group_barrier(FastSync* fs, unsigned int& gepoch) {
  __syncthreads();
  gepoch += 1;
  if (threadIdx.x == 0) { red_release_add(&fs->grp, 1u); wait_ge(&fs->grp, gepoch * FK_G); }
  __syncthreads();
}
// the same barrier split in two, so that work which needs no other CTA runs while the group arrives
__device__ __forceinline__ void fk_group_arrive(FastSync* fs, unsigned int& gepoch) {
  __syncthreads();
  gepoch += 1;
  if (threadIdx.x == 0) red_release_add(&fs->grp, 1u);
}
__device__ __forceinline__ void fk_group_wait(FastSync* fs, unsigned int gepoch) {
  if (threadIdx.x == 0) wait_ge(&fs->grp, gepoch * FK_G);
  __syncthreads();
}

// ---------------- thin-slab GRU phases (no-embedding mode, one layer, M <= 32, L <= 128) ----------------
// ncu on the 32x32-tile kernels showed ~2000 instructions per warp at ~8.6 cycles each (2 warps per scheduler):
// the GRU phases are instruction-latency bound.  Here the work of a phase is spread over all FK_G CTAs (a few
// output columns each), the reduction dimension is split over the 8 warps, and every thread issues a few dozen FMAs.
template <class SM>
__device__ __forceinline__ void fk_stage_lanes(const ModelDev& md, SM& sm, int s, int M) {
  if (threadIdx.x < FK_B) {
    const int b = threadIdx.x;
    sm.gIdx[b] = b < M ? md.wSlot[(size_t)s * md.B + b] : -1;
    sm.gIdx[FK_B + b] = b < M ? md.wX[(size_t)s * md.B + b] : 0;
    sm.gIdx[2 * FK_B + b] = b < M ? md.wF[(size_t)s * md.B + b] : 0;
  }
  __syncthreads();
}
// acc[j] (j < W) for lane b = tid % 32 over the k-slice of warp tid / 32: sum_k A[b][k] * Wt[j][k]
template <int W>
__device__ __forceinline__ void fk_slab_dot(float (&acc)[W], const float* sAop, int lda, const float* sWt, int K) {
  const int b = threadIdx.x & 31, ks = threadIdx.x >> 5;
  const int kq = (K + 3) / 4;                      // float4 count along k
  const int per = (kq + FK_NW - 1) / FK_NW;
  const int q0 = ks * per, q1 = min(kq, q0 + per);
#pragma unroll
  for (int j = 0; j < W; j++) acc[j] = 0.f;
  for (int q = q0; q < q1; q++) {
    const float4 a = ld4(sAop + b * lda + q * 4);
#pragma unroll
    for (int j = 0; j < W; j++) {
      const float4 w = ld4(sWt + j * FK_LDS + q * 4);
      acc[j] = fmaf(a.x, w.x, acc[j]); acc[j] = fmaf(a.y, w.y, acc[j]); acc[j] = fmaf(a.z, w.z, acc[j]); acc[j] = fmaf(a.w, w.w, acc[j]);
    }
  }
}
// cross-warp reduction of acc[W] per lane: red[ks][b][j] -> thread (b, j) sums the 8 slices in fixed order
template <int W>
__device__ __forceinline__ float fk_slab_reduce(const float (&acc)[W], float* red, int jsel) {
  const int b = threadIdx.x & 31, ks = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < W; j++) red[(ks * FK_B + b) * W + j] = acc[j];
  __syncthreads();
  float v = 0.f;
  if (jsel < W) {
#pragma unroll
    for (int k = 0; k < FK_NW; k++) v += red[(k * FK_B + b) * W + jsel];
  }
  return v;
}
constexpr int FK_W1 = 5;    // rz columns per CTA   (ceil(2*128 / 48) = 6 would also fit; 2L <= 240 with 48 CTAs)
constexpr int FK_W2 = 3;    // h / dHr columns per CTA (L <= 144)

// stage H rows of the lanes (fk_stage_lanes done; zero for out-of-range lanes) for F1
__device__ __forceinline__ void fk_f1_stage_h(const LayerDev& ly, FastSmem& sm) {
  const int ldL = ly.ldL;
  stage_rows4(sm.gA, FK_LDS, FK_B, ldL / 4, [&](int rr) -> const float* { const int sl = sm.gIdx[rr]; return sl >= 0 ? ly.H + (size_t)sl * ldL : nullptr; });
}
// F1: rz = sigmoid(Wx0[X][L:3L] + Bh[L:3L] + H @ Wrz) for this CTA's FK_W1 columns; CTA 0 also writes Hold
// inrows != nullptr (row-sharded multi-GPU): the gathered input rows Wx0[X] of the step sit in a local [B x ld3] buffer
// staged: the lanes (fk_stage_lanes), the H rows (fk_f1_stage_h) and the transposed weight slab gW[j][k] = Wrz[k][c0 + j]
// (zero outside j < W, k < L) are already in shared memory, otherwise they are staged from global memory here
// stamp: the %globaltimer around the wait for the helper CTAs goes to sm.sTs (equal stamps when no wait was needed)
__device__ void fk_f1(const ModelDev& md, FastSmem& sm, int s, int cta, const unsigned int* wait_ctr, unsigned int wait_target, const float* inrows = nullptr,
                      bool staged = false, bool stamp = false) {
  const LayerDev& ly = md.layer[0];
  const int M = md.wM[s], L = ly.L, ldL = ly.ldL, tid = threadIdx.x;
  const int c0 = cta * FK_W1;
  if (c0 >= 2 * L) return;
  const int W = min(FK_W1, 2 * L - c0);
  if (!staged) fk_stage_lanes(md, sm, s, M);
  // if the helper CTAs' input-row updates are already complete, the epilogue operand is fetched before the product instead
  // of after it
  if (tid == 0) sm.sFlag[3] = (!wait_ctr || ld_acquire_u32(wait_ctr) >= wait_target) ? 1 : 0;
  const int kw = ldL / 4;
  if (!staged) {
    fk_f1_stage_h(ly, sm);
    for (int i = tid; i < FK_W1 * FK_LDS; i += FK_THREADS) {
      const int j = i / FK_LDS, k = i % FK_LDS;
      sm.gW[i] = (j < W && k < L) ? ly.Wrz[(size_t)k * ly.ld2 + c0 + j] : 0.f;
    }
  }
  const int b = tid & 31, jsel = tid >> 5;
  __syncthreads();
  const bool early = sm.sFlag[3] != 0;
  float pre = 0.f;
  if (early && jsel < W && b < M) pre = (inrows ? inrows[(size_t)b * ly.ld3 + L + c0 + jsel] : ly.Wx[(size_t)sm.gIdx[FK_B + b] * ly.ld3 + L + c0 + jsel]) + ly.Bh[L + c0 + jsel];
  float acc[FK_W1];
  fk_slab_dot<FK_W1>(acc, sm.gA, FK_LDS, sm.gW, L);
  const float v = fk_slab_reduce<FK_W1>(acc, sm.gW + 8 * FK_LDS, jsel);
  // otherwise the gathered input rows are still in flight on the helper CTAs (previous step's update): wait now, after
  // the H @ Wrz part, then fetch the epilogue operands (gathered row element + bias)
  if (stamp && tid == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); sm.sTs[0] = t_; }
  if (!early) {
    if (tid == 0) wait_ge(wait_ctr, wait_target);
    __syncthreads();
    if (jsel < W && b < M) pre = (inrows ? inrows[(size_t)b * ly.ld3 + L + c0 + jsel] : ly.Wx[(size_t)sm.gIdx[FK_B + b] * ly.ld3 + L + c0 + jsel]) + ly.Bh[L + c0 + jsel];
  }
  if (stamp && tid == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); sm.sTs[1] = t_; }
  if (jsel < W && b < M) {
    const int c = c0 + jsel;
    const float g = sigmoidf_(v + pre);
    if (c < L) ly.r[(size_t)b * ldL + c] = g; else ly.z[(size_t)b * ldL + (c - L)] = g;
  }
  if (cta == 0) {
    for (int i = tid; i < FK_B * kw; i += FK_THREADS) {
      const int rr = i / kw, c4 = i % kw;
      if (rr < M) st4(ly.Hold + (size_t)rr * ldL + c4 * 4, ld4(sm.gA + rr * FK_LDS + c4 * 4));
    }
  }
}
// F2: h~ = act(Wx0[X][0:L] + Bh[0:L] + (H*r) @ Wh), h, dropout, H_new for this CTA's FK_W2 columns
// staged: the lanes of step s (fk_stage_lanes) and the transposed slab Wt[j][k] = Wh[k][c0 + j] (zero outside j < W, k < L)
// are already in shared memory, the slab at rows FK_W1.. of gW (after F1's Wrz rows); otherwise both are staged here, the slab
// from global memory to rows 0..
__device__ void fk_f2(const ModelDev& md, FastSmem& sm, int s, int cta, const float* inrows = nullptr, bool staged = false) {
  const LayerDev& ly = md.layer[0];
  const int M = md.wM[s], L = ly.L, ldL = ly.ldL, tid = threadIdx.x;
  const int c0 = cta * FK_W2;
  if (c0 >= L) return;
  const int W = min(FK_W2, L - c0);
  if (!staged) fk_stage_lanes(md, sm, s, M);
  const int kw = ldL / 4;
  // stage H*r
  for (int i0 = 0; i0 < FK_B * kw; i0 += 2 * FK_THREADS) {
    float4 hv[2], rv[2];
#pragma unroll
    for (int u = 0; u < 2; u++) {
      const int i = i0 + u * FK_THREADS + tid;
      hv[u] = make_float4(0.f, 0.f, 0.f, 0.f); rv[u] = hv[u];
      if (i < FK_B * kw) {
        const int rr = i / kw, c4 = i % kw;   // Hold (compact copy written by CTA 0 in F1): H itself is being overwritten
        if (rr < M) { hv[u] = ld4(ly.Hold + (size_t)rr * ldL + c4 * 4); rv[u] = ld4(ly.r + (size_t)rr * ldL + c4 * 4); }
      }
    }
#pragma unroll
    for (int u = 0; u < 2; u++) {
      const int i = i0 + u * FK_THREADS + tid;
      if (i < FK_B * kw) st4(sm.gA + (i / kw) * FK_LDS + (i % kw) * 4, make_float4(hv[u].x * rv[u].x, hv[u].y * rv[u].y, hv[u].z * rv[u].z, hv[u].w * rv[u].w));
    }
  }
  if (!staged) {
    for (int i = tid; i < FK_W2 * FK_LDS; i += FK_THREADS) {
      const int j = i / FK_LDS, k = i % FK_LDS;
      sm.gW[i] = (j < W && k < L) ? ly.Wh[(size_t)k * ldL + c0 + j] : 0.f;
    }
  }
  const int b = tid & 31, jsel = tid >> 5;
  float pre = 0.f, z = 0.f, ho = 0.f;
  if (jsel < W && b < M) {
    const int c = c0 + jsel;
    pre = (inrows ? inrows[(size_t)b * ly.ld3 + c] : ly.Wx[(size_t)sm.gIdx[FK_B + b] * ly.ld3 + c]) + ly.Bh[c];
    z = ly.z[(size_t)b * ldL + c];
    ho = ly.Hold[(size_t)b * ldL + c];
  }
  __syncthreads();
  float acc[FK_W2];
  fk_slab_dot<FK_W2>(acc, sm.gA, FK_LDS, sm.gW + (staged ? FK_W1 * FK_LDS : 0), L);
  const float v0 = fk_slab_reduce<FK_W2>(acc, sm.gW + 8 * FK_LDS, jsel);
  if (jsel < W && b < M) {
    const int c = c0 + jsel;
    const float v = v0 + pre;
    const float ht = act_fwd(md.hact, v);
    float h = (1.0f - z) * ho + z * ht;
    if (md.p_drop_h > 0.f) h *= drop_scale(md.drop_seed, md.wG[s], 0u, (uint32_t)(b * L + c), 1.0f - md.p_drop_h);
    ly.ah[(size_t)b * ldL + c] = v;
    ly.ht[(size_t)b * ldL + c] = ht;
    ly.y[(size_t)b * ldL + c] = h;
    ly.H[(size_t)sm.gIdx[b] * ldL + c] = (sm.gIdx[2 * FK_B + b] & 1) ? 0.f : h;
  }
}
// B2: d(H*r)[b][c] = sum_j da_h[b][j] Wh[c][j]; da_r = d(H*r) * Hold * r (1-r) for this CTA's FK_W2 columns
__device__ void fk_b2(const ModelDev& md, FastSmem& sm, int s, int cta) {
  const LayerDev& ly = md.layer[0];
  const int M = md.wM[s], L = ly.L, ldL = ly.ldL, tid = threadIdx.x;
  const int c0 = cta * FK_W2;
  if (c0 >= L) return;
  const int W = min(FK_W2, L - c0);
  const int kw = ldL / 4;
  __syncthreads();
  stage_rows4(sm.gA, FK_LDS, FK_B, kw, [&](int rr) -> const float* { return rr < M ? ly.dvec + (size_t)rr * ly.ld3 : nullptr; });
  stage_rows4(sm.gW, FK_LDS, W, kw, [&](int rr) -> const float* { return ly.Wh + (size_t)(c0 + rr) * ldL; });
  const int b = tid & 31, jsel = tid >> 5;
  float ho = 0.f, r = 0.f;
  if (jsel < W && b < M) { ho = ly.Hold[(size_t)b * ldL + c0 + jsel]; r = ly.r[(size_t)b * ldL + c0 + jsel]; }
  __syncthreads();
  float acc[FK_W2];
  fk_slab_dot<FK_W2>(acc, sm.gA, FK_LDS, sm.gW, L);
  const float v = fk_slab_reduce<FK_W2>(acc, sm.gW + 8 * FK_LDS, jsel);
  if (jsel < W && b < M) ly.dvec[(size_t)b * ly.ld3 + L + c0 + jsel] = v * ho * r * (1.f - r);
}
// D: dense Adagrad(+momentum) of Wh / Wrz / Bh, owned by the forward column owners.  GRU CTA `cta` updates exactly the
// weights it multiplies with in F1 / F2 of the next step, so the updated slab feeds those products from shared memory:
//   e = j L + k            (j < FK_W1)  Wrz[k][c0 + j], c0 = FK_W1 cta    grad sum_b Hold[b][k] dvec[b][L + c0 + j]
//   e = (FK_W1 + j) L + k  (j < FK_W2)  Wh[k][c2 + j],  c2 = FK_W2 cta    grad sum_b (Hold r)[b][k] dvec[b][c2 + j]
//   e = FK_WD L + j                     Bh[L + c0 + j] (j < FK_W1), Bh[c2 + j - FK_W1]     grad sum_b of the same column
// Only this CTA reads or writes these values, except Wh, which B2 reads by rows before the group barrier that follows it.
// Per element the arithmetic is the generic dense update's: the lanes summed in order with fmaf (the bias: plain sums), then
// adagrad_scale and dense_step.  The Wr columns (and Bh_r) need da_r from every CTA's B2 and run after that barrier
// (phase 1); everything else runs while the CTA waits for it (phase 0).
constexpr int FK_WD = FK_W1 + FK_W2;                 // slab rows: F1 columns, then F2 columns
constexpr int FK_DNE = FK_WD * 120 + FK_WD;          // owned elements per GRU CTA at L <= 120
static_assert(3 * FK_DNE <= FK_NW * FK_B * 8, "owned parameter / Adagrad / momentum values fit sPart");
static_assert(2 * FK_B * FK_LDS <= FK_B * 388, "Hold * r fits behind the staged H rows in gA");
static_assert(FK_WD * FK_B <= FK_CT * FK_B, "owned dvec columns fit sG");

// owned element e: parameter / Adagrad / momentum pointers, slab row j, weight row k (-1: bias); false if e is past the layer
__device__ __forceinline__ bool fk_own(const LayerDev& ly, int cta, int e, float*& p, float*& pa, float*& pv, int& j, int& k) {
  const int L = ly.L, c0 = cta * FK_W1, c2 = cta * FK_W2;
  size_t off;
  if (e < FK_WD * L) { j = e / L; k = e % L; }
  else { j = e - FK_WD * L; k = -1; if (j >= FK_WD) return false; }
  if (j < FK_W1 ? c0 + j >= 2 * L : c2 + j - FK_W1 >= L) return false;
  if (k < 0) {
    off = j < FK_W1 ? (size_t)(L + c0 + j) : (size_t)(c2 + j - FK_W1);
    p = ly.Bh + off; pa = ly.Bh_acc ? ly.Bh_acc + off : nullptr; pv = ly.Bh_vel ? ly.Bh_vel + off : nullptr;
  } else if (j < FK_W1) {
    off = (size_t)k * ly.ld2 + c0 + j;
    p = ly.Wrz + off; pa = ly.Wrz_acc ? ly.Wrz_acc + off : nullptr; pv = ly.Wrz_vel ? ly.Wrz_vel + off : nullptr;
  } else {
    off = (size_t)k * ly.ldL + c2 + j - FK_W1;
    p = ly.Wh + off; pa = ly.Wh_acc ? ly.Wh_acc + off : nullptr; pv = ly.Wh_vel ? ly.Wh_vel + off : nullptr;
  }
  return true;
}
// phase of slab row j: 1 for the Wr columns (their gradient needs da_r), 0 otherwise
__device__ __forceinline__ int fk_own_phase(int L, int cta, int j) { return (j < FK_W1 && cta * FK_W1 + j < L) ? 1 : 0; }

// While the CTA waits for b1_done: Hold(s) and Hold * r(s) into shared memory (F1 of step s + 1 overwrites both in global
// memory after the B2 group barrier), and the owned parameter / Adagrad / momentum values (final: no other CTA writes them).
// All loads are issued before the first store, so the whole staging costs one round trip.
__device__ void fk_dense_stage(const ModelDev& md, FastSmem& sm, int s, int cta) {
  const LayerDev& ly = md.layer[0];
  const int M = md.wM[s], L = ly.L, ldL = ly.ldL, kw = ldL / 4, tid = threadIdx.x;
  if (cta * FK_W1 >= 2 * L) return;                 // no F1 columns (and so no F2 columns either)
  const bool ada = md.adapt == G4R_ADAPT_ADAGRAD, mom = md.mom > 0.f;
  constexpr int NU = 2;                             // M * kw <= 32 * 32 quads and FK_DNE elements: two per thread
  static_assert(NU * FK_THREADS >= FK_B * 32 && NU * FK_THREADS >= FK_DNE, "fk_dense_stage covers one pass");
  float4 hv[NU], rv[NU];
  float p0[NU], a0[NU], v0[NU];
#pragma unroll
  for (int u = 0; u < NU; u++) {
    const int i = u * FK_THREADS + tid;
    hv[u] = make_float4(0.f, 0.f, 0.f, 0.f); rv[u] = hv[u];
    if (i < M * kw) { const size_t o = (size_t)(i / kw) * ldL + (i % kw) * 4; hv[u] = ld4(ly.Hold + o); rv[u] = ld4(ly.r + o); }
    float *p, *pa, *pv; int j, k;
    p0[u] = 0.f; a0[u] = 0.f; v0[u] = 0.f;
    if (fk_own(ly, cta, i, p, pa, pv, j, k)) {
      p0[u] = *p;
      if (ada && pa) a0[u] = *pa;
      if (mom && pv) v0[u] = *pv;
    }
  }
  float* sHr = sm.gA + FK_B * FK_LDS;
#pragma unroll
  for (int u = 0; u < NU; u++) {
    const int i = u * FK_THREADS + tid;
    if (i < M * kw) {
      const int o = (i / kw) * FK_LDS + (i % kw) * 4;
      st4(sm.sD + o, hv[u]);
      st4(sHr + o, make_float4(hv[u].x * rv[u].x, hv[u].y * rv[u].y, hv[u].z * rv[u].z, hv[u].w * rv[u].w));
    }
    if (i < FK_DNE) { sm.sPart[i] = p0[u]; sm.sPart[FK_DNE + i] = a0[u]; sm.sPart[2 * FK_DNE + i] = v0[u]; }
  }
}
// this thread's element of the owned dvec columns of phase ph (tid = j * FK_B + b), for fk_dense_put_dcol
__device__ __forceinline__ float fk_dense_dcol(const LayerDev& ly, int M, int cta, int ph) {
  const int j = threadIdx.x / FK_B, b = threadIdx.x % FK_B, L = ly.L, c0 = cta * FK_W1, c2 = cta * FK_W2;
  if (j >= FK_WD || b >= M || fk_own_phase(L, cta, j) != ph) return 0.f;
  if (j < FK_W1 ? c0 + j >= 2 * L : c2 + j - FK_W1 >= L) return 0.f;
  return ly.dvec[(size_t)b * ly.ld3 + (j < FK_W1 ? L + c0 + j : c2 + j - FK_W1)];
}
__device__ __forceinline__ void fk_dense_put_dcol(FastSmem& sm, const LayerDev& ly, int cta, int ph, float v) {
  const int j = threadIdx.x / FK_B;
  if (j < FK_WD && fk_own_phase(ly.L, cta, j) == ph) sm.sG[threadIdx.x] = v;
}
// gradient and update of the owned elements of phase ph (fk_dense_stage and fk_dense_put_dcol of the phase done).  The new
// weights go to the slab rows gW[j][k] (zero elsewhere) that F1 / F2 multiply with, and to global memory; the Wh
// parameters only in phase 1, once every CTA has passed B2.
__device__ void fk_dense_update(const ModelDev& md, FastSmem& sm, int s, int cta, int ph) {
  const LayerDev& ly = md.layer[0];
  const int M = md.wM[s], L = ly.L, tid = threadIdx.x;
  if (cta * FK_W1 >= 2 * L) return;
  const bool ada = md.adapt == G4R_ADAPT_ADAGRAD, mom = md.mom > 0.f;
  const float* sHr = sm.gA + FK_B * FK_LDS;
  if (ph == 0) {
    for (int i = tid; i < FK_WD * FK_LDS; i += FK_THREADS) {
      const int j = i / FK_LDS, k = i % FK_LDS;
      float *p, *pa, *pv; int jj, kk;
      if (k >= L || !fk_own(ly, cta, j * L, p, pa, pv, jj, kk)) sm.gW[i] = 0.f;
    }
  }
  for (int e = tid; e < FK_WD * L + FK_WD; e += FK_THREADS) {
    float *p, *pa, *pv; int j, k;
    if (!fk_own(ly, cta, e, p, pa, pv, j, k) || fk_own_phase(L, cta, j) != ph) continue;
    const float* dc = sm.sG + j * FK_B;
    float g = 0.f;
    if (k >= 0) {
      const float* a = (j < FK_W1 ? sm.sD : sHr) + k;
      for (int b = 0; b < M; b++) g = fmaf(a[b * FK_LDS], dc[b], g);
    } else {
      for (int b = 0; b < M; b++) g = g + dc[b];
    }
    float gs = g;
    if (ada) gs = adagrad_scale(g, sm.sPart[FK_DNE + e], *pa);
    float v = sm.sPart[2 * FK_DNE + e];
    const float pn = dense_step(md, gs, sm.sPart[e], v, mom);
    if (mom) *pv = v;
    if (k >= 0) sm.gW[j * FK_LDS + k] = pn;
    if (k < 0 || j < FK_W1) *p = pn;
  }
  if (ph == 1) {
    const int c2 = cta * FK_W2, W2 = max(0, min(FK_W2, L - c2));
    for (int i = tid; i < W2 * L; i += FK_THREADS) {
      const int k = i / W2, j = i % W2;
      ly.Wh[(size_t)k * ly.ldL + c2 + j] = sm.gW[(FK_W1 + j) * FK_LDS + k];
    }
  }
}

// Input-row update of lane b on a helper (non-GRU) CTA, concurrent with the dense update of the GRU group: it starts when
// the GRU group has passed its B2 barrier (dvec complete) and only touches Wx0 rows, which the dense phase never reads.
template <class SM>
__device__ void fk_sparse_in(const ModelDev& md, SM& sm, int s, int b) {
  const LayerDev& ly = md.layer[0];
  const int M = md.wM[s];
  if (b >= M) return;
  const uint8_t xf = md.wXflag[(size_t)s * md.B + b];
  if (!(xf & 1)) return;                                // not the first position of its duplicate group
  const int ld3 = ly.ld3, tid = threadIdx.x;
  const int item = md.wX[(size_t)s * md.B + b];
  const int* xnext = md.wXnext + (size_t)s * md.B;
  if (tid == 0) { int n = 0; for (int bb = b; bb >= 0 && n < FK_B; bb = xnext[bb]) sm.gIdx[n++] = bb; sm.gIdx[FK_B] = n; }
  __syncthreads();
  const int nmem = sm.gIdx[FK_B];
  const bool ada = md.adapt == G4R_ADAPT_ADAGRAD, mom = md.mom > 0.f;
  float* prow = ly.Wx + (size_t)item * ld3;
  for (int c4 = tid; c4 < ld3 / 4; c4 += FK_THREADS) {
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    SparseUpd4 u;
    u.begin(ld4(prow + c4 * 4), ada ? ld4(ly.Wx_acc + (size_t)item * ld3 + c4 * 4) : z, mom ? ld4(ly.Wx_vel + (size_t)item * ld3 + c4 * 4) : z);
    for (int k = 0; k < nmem; k++) u.add(md, ld4(ly.dvec + (size_t)sm.gIdx[k] * ld3 + c4 * 4), ada, mom);
    st4(prow + c4 * 4, u.ps);
    if (ada) st4(ly.Wx_acc + (size_t)item * ld3 + c4 * 4, u.al);
    if (mom) st4(ly.Wx_vel + (size_t)item * ld3 + c4 * 4, u.vl);
  }
}

// Same update when the CTA owns exactly one lane: everything that does not depend on this step's gradients (duplicate
// chain, parameter / Adagrad / momentum row) is fetched BEFORE waiting for the dvec rows, so that only one load round trip
// separates the GRU role's "dvec complete" signal from the row update.
template <class SM>
__device__ void fk_sparse_in_one(const ModelDev& md, SM& sm, int s, int b, const unsigned int* ctr, unsigned int target) {
  const LayerDev& ly = md.layer[0];
  const int M = md.wM[s], ld3 = ly.ld3, tid = threadIdx.x;
  const bool act = b < M && (md.wXflag[(size_t)s * md.B + b] & 1);       // first position of its duplicate group
  const int item = act ? md.wX[(size_t)s * md.B + b] : 0;
  const bool ada = md.adapt == G4R_ADAPT_ADAGRAD, mom = md.mom > 0.f;
  if (act && tid == 0) {
    const int* xnext = md.wXnext + (size_t)s * md.B;
    int n = 0; for (int bb = b; bb >= 0 && n < FK_B; bb = xnext[bb]) sm.gIdx[n++] = bb; sm.gIdx[FK_B] = n;
  }
  float* prow = ly.Wx + (size_t)item * ld3;
  const int c4 = tid;
  const bool mine = act && c4 < ld3 / 4;                                   // ld3 / 4 <= 96 quads: one pass
  float4 p0 = make_float4(0.f, 0.f, 0.f, 0.f), a0 = p0, v0 = p0;
  if (mine) {
    p0 = ld4(prow + c4 * 4);
    if (ada) a0 = ld4(ly.Wx_acc + (size_t)item * ld3 + c4 * 4);
    if (mom) v0 = ld4(ly.Wx_vel + (size_t)item * ld3 + c4 * 4);
  }
  if (tid == 0) wait_ge(ctr, target);
  __syncthreads();
  if (mine) {
    const int nmem = sm.gIdx[FK_B];
    SparseUpd4 u;
    u.begin(p0, a0, v0);
    for (int k = 0; k < nmem; k++) u.add(md, ld4(ly.dvec + (size_t)sm.gIdx[k] * ld3 + c4 * 4), ada, mom);
    st4(prow + c4 * 4, u.ps);
    if (ada) st4(ly.Wx_acc + (size_t)item * ld3 + c4 * 4, u.al);
    if (mom) st4(ly.Wx_vel + (size_t)item * ld3 + c4 * 4, u.vl);
  }
}

// B1 (fast kernel): every CTA reduces a contiguous run of dL/dh elements; lanes = consecutive elements (coalesced),
// warps = slices of the chunk partials, cross-warp sum in shared memory in fixed order; then da_h / da_z.
template <bool CL, class SM>
__device__ void fk_b1(const ModelDev& md, SM& sm, int s, int cta, int ncta) {
  const LayerDev& ly = md.layer[0];
  const int M = md.wM[s], L = ly.L, ldL = ly.ldL;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int E = M * ldL;                                  // padded elements (padding columns are zero everywhere)
  const int per = ((E + ncta - 1) / ncta + 31) / 32 * 32; // elements per CTA, multiple of 32
  const int e0 = cta * per;
  float* red = sm.sPart;                                  // [FK_NW][per]  (per <= 128 for M*ldL <= 4096*... checked on host)
  const size_t cs = (size_t)md.B * ldL;
  // forward saves of this thread's output element (per <= 128 <= FK_THREADS: at most one element per thread), fetched up
  // front so that their round trip overlaps the loads of the chunk partials
  float pht = 0.f, pho = 0.f, pz = 0.f, pah = 0.f;
  if (!CL && tid < per && e0 + tid < E && (e0 + tid) % ldL < L) {
    const size_t o = (size_t)((e0 + tid) / ldL) * ldL + (e0 + tid) % ldL;
    pht = ly.ht[o]; pho = ly.Hold[o]; pz = ly.z[o]; pah = ly.ah[o];
  }
  for (int eb = 0; eb < per; eb += 32) {
    const int e = e0 + eb + lane;
    float d = 0.f;
    if (e < E) {
      float v[10];
#pragma unroll
      for (int u = 0; u < 10; u++) { const int ch = warp + FK_NW * u; v[u] = ch < md.NCH ? md.part[(size_t)ch * cs + e] : 0.f; }
      d = (((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]))) + (v[8] + v[9]);
    }
    red[warp * per + eb + lane] = d;
  }
  __syncthreads();
  for (int i = tid; i < per; i += FK_THREADS) {
    const int e = e0 + i;
    if (e >= E) continue;
    const int b = e / ldL, c = e % ldL;
    if (c >= L) continue;
    float dy = 0.f;
#pragma unroll
    for (int w = 0; w < FK_NW; w++) dy += red[w * per + i];
    const size_t o = (size_t)b * ldL + c;
    if (CL) { ly.dy[o] = dy; continue; }     // cluster variant: the GRU cluster owns ht / z / ah and derives da_h, da_z itself
    const float ht = pht, ho = pho, z = pz, ah = pah;
    float dh = dy;
    if (md.p_drop_h > 0.f) dh *= drop_scale(md.drop_seed, md.wG[s], 0u, (uint32_t)(b * L + c), 1.0f - md.p_drop_h);
    const float dz = dh * (ht - ho);
    const float dah = dh * z * act_der(md.hact, ah, ht);
    ly.dvec[(size_t)b * ly.ld3 + c] = dah;
    ly.dvec[(size_t)b * ly.ld3 + 2 * L + c] = dz * z * (1.f - z);
  }
}

#include "g4r_fastc.cuh"

// CL = false: GRU phases on a 48-CTA group with global group barriers (step_mode 2).
// CL = true : launched with thread-block clusters; the GRU phases run on cluster 0 (g4r_fastc.cuh, step_mode 3).
template <bool CL>
__global__ void __launch_bounds__(FK_THREADS, 1) k_fast_t(int slot, int n_steps, FastSync* fs, unsigned long long* tstamp) {
  using SM = typename std::conditional<CL, FastSmemC, FastSmem>::type;
  extern __shared__ __align__(128) unsigned char fk_raw[];
  SM& sm = *reinterpret_cast<SM*>(fk_raw);
  const ModelDev& md = MD;
  const LayerDev& ly = md.layer[0];
  const int cta = blockIdx.x, ncta = gridDim.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int chunk = cta;                       // CTAs beyond the number of chunks own no columns
  const bool has_chunk = chunk < md.NCH;
  const int G = CL ? (int)cl_size() : FK_G;    // CTAs of the GRU role
  const bool gru = cta < G;
  const bool pw = loss_pairwise(md.loss);
  const bool ada = md.adapt == G4R_ADAPT_ADAGRAD, mom = md.mom > 0.f;
  const int L = md.L, ldL = md.ldL, B = md.B;
  const int kw = ldL / 4;
  uint64_t* bar = reinterpret_cast<uint64_t*>(&sm.mbar);
  unsigned int bar_epoch = 0, gepoch = 0, stats_target = 0;
  const int in_ctas = min(B, ncta - G);        // helper CTAs [G, G + in_ctas) update the gathered input rows
#ifdef G4R_CF_FINE
#define FK_FTS(s_) ((tstamp && cta == 0 && (s_) < 500 && n_steps >= 1000) ? tstamp + (size_t)((s_) + 500) * 16 : nullptr)
#define FK_STAMP_OK(s_) ((s_) < 500)
#else
#define FK_FTS(s_) ((unsigned long long*)nullptr)
#define FK_STAMP_OK(s_) true
#endif
#define FK_STAMP(k) do { if (tstamp && cta == 0 && tid == 0 && FK_STAMP_OK(s)) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); tstamp[(size_t)s * 16 + (k)] = t_; } } while (0)
// fine stamps of the column phases; in step_mode 2 the GRU role reuses their slots (1, 4, 9, 10, 11, 12)
#define FK_STAMP_CL(k) do { if (CL) FK_STAMP(k); } while (0)
  if (tid == 0) { mbar_init(bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  fk_load_idx(md, sm, 0, n_steps, chunk, 0);
  __syncthreads();
  fk_prefetch_rows(md, sm, 0, n_steps, 0, pw);
  // GRU forward of step 0
  ClusterCtx cc = {0, 1, 0, 0};
  if constexpr (CL) {
    if (gru) {
      cc = cf_init(md, sm);
      cf_load_resident(md, sm, cc);
      if (n_steps > 0) {
        fk_stage_lanes(md, sm, 0, md.wM[0]);
        cf_f1(md, sm, cc, 0, false, nullptr, 0u, nullptr);
        cf_f2(md, sm, cc, 0, nullptr);
        __syncthreads();
        if (tid == 0) red_release_add(&fs->h_ready, 1u);
      }
    }
  } else {
    if (gru) {
      fk_f1(md, sm, 0, cta, nullptr, 0u);
      fk_group_barrier(fs, gepoch);
      fk_f2(md, sm, 0, cta);
      __syncthreads();
      if (tid == 0) red_release_add(&fs->h_ready, 1u);
    }
  }
  for (int s = 0; s < n_steps; s++) {
    const int buf = s & 1;
    const int M = md.wM[s];
    const int sti = md.wSti[s];
    const int N = M + (sti >= 0 ? md.S : 0);
    FK_STAMP(0);
    // indices of the NEXT step (consumed after this step's last barrier)
    fk_load_idx(md, sm, s + 1, n_steps, chunk, buf ^ 1);
    // ---- wait for h(s), stage it ----
    if (tid == 0) wait_ge(&fs->h_ready, (unsigned int)(s + 1) * (unsigned int)G);
    __syncthreads();
    stage_rows4(sm.sY, FK_LDS, FK_B, kw, [&](int rr) -> const float* { return rr < M ? ly.y + (size_t)rr * ldL : nullptr; });
    mbar_wait(bar, (unsigned int)(s & 1));      // prefetched rows of this step have landed
    __syncthreads();
    FK_STAMP_CL(1);
    const int cb = sm.sCb[buf][0], ce = sm.sCb[buf][1];
    const int nj = ce - cb;
    // ---- scores + partial statistics ----
    if (pw) {                                   // target activations: warp per 4 lanes
      for (int b = warp; b < FK_B; b += FK_NW) {
        if (b < M) {
          float a = 0.f;
          if (lane < kw) {
            const float4 y = ld4(sm.sY + b * FK_LDS + lane * 4), w = ld4(sm.sTW + b * FK_LDS + lane * 4);
            a = fmaf(w.x, y.x, a); a = fmaf(w.y, y.y, a); a = fmaf(w.z, y.z, a); a = fmaf(w.w, y.w, a);
          }
          a = warp_sum(a);
          if (lane == 0) sm.sT[b] = act_fwd(md.fact, a + sm.sTB[b]);
        }
      }
    }
    {
      float accq[FK_Q];
#pragma unroll
      for (int q = 0; q < FK_Q; q++) accq[q] = 0.f;
      const float* yr = sm.sY + lane * FK_LDS;
      for (int c4 = 0; c4 < kw; c4++) {
        const float4 y = ld4(yr + c4 * 4);
#pragma unroll
        for (int q = 0; q < FK_Q; q++) {
          if (warp + FK_NW * q < nj) {
            const float4 w = ld4(sm.sS + (warp + FK_NW * q) * FK_LDS + c4 * 4);
            accq[q] = fmaf(y.x, w.x, accq[q]); accq[q] = fmaf(y.y, w.y, accq[q]); accq[q] = fmaf(y.z, w.z, accq[q]); accq[q] = fmaf(y.w, w.w, accq[q]);
          }
        }
      }
      FK_STAMP_CL(9);
#pragma unroll
      for (int q = 0; q < FK_Q; q++) {
        const int jj = warp + q * FK_NW;
        if (jj < nj && lane < M) sm.sO[jj * FK_B + lane] = accq[q] + sm.sBias[jj];
      }
      __syncthreads();                          // sT and sO complete
      // chunk statistics of lane b by 16 threads (column jj = sub, sub + 16): row max first, then plain sums -- one expf
      // per column instead of an exp-rescaling merge per element
      {
        const int b = tid >> 4, sub = tid & 15;            // FK_THREADS / 16 == FK_B lanes
        const bool okb = b < M;
        const int tc = okb ? sm.sTc[buf][b] : -1;
        const float t = (pw && okb) ? sm.sT[b] : 0.f;
        float yv[2]; bool use[2], ist[2];
        float mloc = -INFINITY;
        const bool smx = loss_softmaxneg(md.loss), xe = (md.loss == G4R_LOSS_XE || md.loss == G4R_LOSS_XE_LOGIT);
#pragma unroll
        for (int q = 0; q < 2; q++) {
          const int jj = sub + 16 * q;
          use[q] = okb && jj < nj;
          ist[q] = use[q] && (tc == cb + jj);
          const float o = use[q] ? sm.sO[jj * FK_B + b] : 0.f;
          yv[q] = xe ? o : act_fwd(md.fact, o);
          if (use[q] && (xe || (smx && !ist[q]))) mloc = fmaxf(mloc, yv[q]);
        }
#pragma unroll
        for (int o = 1; o < 16; o <<= 1) mloc = fmaxf(mloc, __shfl_xor_sync(0xffffffffu, mloc, o));
        float Z = 0.f, A = 0.f, Q = 0.f, D = 0.f, T = 0.f, has = 0.f;
#pragma unroll
        for (int q = 0; q < 2; q++) {
          if (!use[q]) continue;
          const float y = yv[q];
          if (ist[q]) has = 1.f;
          if (xe) { Z += expf(y - mloc); if (ist[q]) T = y; }
          else if (md.loss == G4R_LOSS_BPR_MAX) { if (!ist[q]) { const float e = expf(y - mloc), sg = sigmoidf_(t - y); Z += e; A += sg * e; Q += y * y * e; D += sg * (1.f - sg) * e; } }
          else if (md.loss == G4R_LOSS_TOP1_MAX) { if (!ist[q]) { const float e = expf(y - mloc), a1 = sigmoidf_(y - t), b1 = sigmoidf_(y * y); Z += e; A += (a1 + b1) * e; D += a1 * (1.f - a1) * e; } }
          else if (md.loss == G4R_LOSS_BPR) { const float sg = sigmoidf_(t - y); A += -logf(sg); if (!ist[q]) D += 1.f - sg; }
          else { const float a1 = sigmoidf_(y - t), b1 = sigmoidf_(y * y); A += a1 + b1; if (!ist[q]) D += a1 * (1.f - a1); }
        }
#pragma unroll
        for (int o = 1; o < 16; o <<= 1) {
          Z += __shfl_xor_sync(0xffffffffu, Z, o); A += __shfl_xor_sync(0xffffffffu, A, o); Q += __shfl_xor_sync(0xffffffffu, Q, o);
          D += __shfl_xor_sync(0xffffffffu, D, o); T += __shfl_xor_sync(0xffffffffu, T, o); has += __shfl_xor_sync(0xffffffffu, has, o);
        }
        if (has_chunk && okb && sub == 0) {
          float* st = md.stat + ((size_t)chunk * md.B + b) * G4R_NSTAT;
          st4(st, make_float4(mloc, Z, A, Q));
          st4(st + 4, make_float4(D, T, has > 0.f ? 1.f : 0.f, pw ? t : 0.f));
        }
      }
    }
    // ---- barrier B2, then lane b's statistics are combined by CTA b (all lanes in parallel, fixed merge order) ----
    __syncthreads();
    FK_STAMP_CL(10);
    bar_epoch += 1;
    if (tid == 0) { red_release_add(&fs->bar, 1u); wait_ge(&fs->bar, bar_epoch * (unsigned int)ncta); }
    __syncthreads();
    if (cta < M) {
      // lane b = cta: row max over the chunk maxima, one rescale exp per chunk, then plain sums (fixed shuffle / warp order)
      const int b = cta;
      const bool maxed = !(md.loss == G4R_LOSS_BPR || md.loss == G4R_LOSS_TOP1);
      float mc = -INFINITY, Z = 0.f, A = 0.f, Q = 0.f, D = 0.f, T = 0.f, has = 0.f, tt = 0.f;
      if (tid < md.NCH) {
        const float* st = md.stat + ((size_t)tid * md.B + b) * G4R_NSTAT;
        const float4 u = ld4(st), v = ld4(st + 4);
        mc = u.x; Z = u.y; A = u.z; Q = u.w; D = v.x; T = v.y; has = v.z;
        if (tid == 0) tt = v.w;
      }
      float mg = mc;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) mg = fmaxf(mg, __shfl_xor_sync(0xffffffffu, mg, o));
      if (lane == 0) sm.sPart[warp] = mg;
      __syncthreads();
      mg = sm.sPart[0];
      for (int w = 1; w < FK_NW; w++) mg = fmaxf(mg, sm.sPart[w]);
      if (loss_softmaxneg(md.loss)) mg = fmaxf(mg, 0.f);          // the zeroed diagonal takes part in the max (gru4rec.py:200-202)
      if (maxed) {
        const float sc = (mc == -INFINITY) ? 0.f : expf(mc - mg);
        Z *= sc; A *= sc; Q *= sc; D *= sc;
      }
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        Z += __shfl_xor_sync(0xffffffffu, Z, o); A += __shfl_xor_sync(0xffffffffu, A, o); Q += __shfl_xor_sync(0xffffffffu, Q, o);
        D += __shfl_xor_sync(0xffffffffu, D, o); T += __shfl_xor_sync(0xffffffffu, T, o); has += __shfl_xor_sync(0xffffffffu, has, o);
      }
      __syncthreads();
      if (lane == 0) { float* w = sm.sPart + 32 + warp * 8; w[0] = Z; w[1] = A; w[2] = Q; w[3] = D; w[4] = T; w[5] = has; w[6] = tt; }
      __syncthreads();
      if (tid == 0) {
        tt = sm.sPart[32 + 6];
        for (int w = 1; w < FK_NW; w++) { const float* q = sm.sPart + 32 + w * 8; Z += q[0]; A += q[1]; Q += q[2]; D += q[3]; T += q[4]; }
        const float m = mg;
        float* rs = md.RS + (size_t)b * G4R_NSTAT;
        float loss = 0.f, r0 = m, r1 = Z, r2 = 0.f, r3 = 0.f, r4 = 0.f, r5 = tt;
        if (md.loss == G4R_LOSS_XE) { const float pt = __fdiv_rn(expf(T - m), Z); loss = -logf(pt + G4R_EPS_LOG); r2 = pt; r5 = T; }
        else if (md.loss == G4R_LOSS_XE_LOGIT) { loss = logf(Z) - (T - m); r5 = T; }
        else if (md.loss == G4R_LOSS_BPR_MAX) { r2 = __fdiv_rn(A, Z); r3 = __fdiv_rn(Q, Z); r4 = __fdiv_rn(D, Z); loss = -logf(r2 + G4R_EPS_LOG) + md.bpreg * r3; }
        else if (md.loss == G4R_LOSS_TOP1_MAX) { r2 = __fdiv_rn(A, Z); r4 = __fdiv_rn(D, Z); loss = r2; }
        else if (md.loss == G4R_LOSS_BPR) { loss = A; r4 = D; }
        else { const float c = sigmoidf_(tt * tt); loss = (float)M * (__fdiv_rn(A, (float)N) - __fdiv_rn(c, (float)(M + md.S_cfg))); r4 = D; }
        st4(rs, make_float4(r0, r1, r2, r3));
        st4(rs + 4, make_float4(r4, r5, loss, 0.f));
        red_release_add(&fs->stats, 1u);
      }
    }
    stats_target += (unsigned int)M;
    if (tid == 0) wait_ge(&fs->stats, stats_target);
    __syncthreads();
    FK_STAMP(2);
    // ---- loss gradient, dSy, partial dL/dh, sparse update of this chunk's rows ----
    if (tid < M * 2) st4(sm.sRS + tid * 4, ld4(md.RS + tid * 4));
    __syncthreads();
    if (chunk == 0 && tid == 0) {
      float c = 0.f;
      for (int b = 0; b < M; b++) c += sm.sRS[b * 8 + 6];
      c = __fdiv_rn(c, (float)md.B);
      md.cost[s] = c;
      if (c != c) atomicExch(md.nanflag, 1);
    }
    FK_STAMP_CL(11);
    for (int i = tid; i < FK_CT * FK_B; i += FK_THREADS) {
      const int jj = i / FK_B, b = i % FK_B;
      sm.sG[i] = (jj < nj && b < M) ? loss_grad_elem(md, sm.sRS + (size_t)b * 8, sm.sO[i], sm.sTc[buf][b] == cb + jj, M, N) : 0.f;
    }
    __syncthreads();
    for (int jj = warp; jj < nj; jj += FK_THREADS / 32) {
      float a = (lane < M) ? sm.sG[jj * FK_B + lane] : 0.f;
      a = warp_sum(a);
      if (lane == 0) sm.sDby[jj] = a;
    }
    FK_STAMP_CL(12);
    float* part = md.part + (size_t)(has_chunk ? chunk : 0) * md.B * ldL;
    if (has_chunk) {
      // dSy[j][quad] = sum_b g[b][j] y[b][quad]: one thread per (column, 16-byte feature quad), all nj*kw pairs in parallel
      for (int t = tid; t < nj * kw; t += FK_THREADS) {
        const int jj = t / kw, q4 = t % kw;
        float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int bb = 0; bb < M; bb++) {
          const float4 y = ld4(sm.sY + bb * FK_LDS + q4 * 4);
          const float g = sm.sG[jj * FK_B + bb];
          d.x = fmaf(g, y.x, d.x); d.y = fmaf(g, y.y, d.y); d.z = fmaf(g, y.z, d.z); d.w = fmaf(g, y.w, d.w);
        }
        st4(sm.sD + jj * FK_LDS + q4 * 4, d);
      }
      // partial dL/dh[b][quad] = sum_j g[b][j] Sy_j[quad]: one thread per (lane, quad)
      for (int t = tid; t < M * kw; t += FK_THREADS) {
        const int bb = t / kw, q4 = t % kw;
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int jj = 0; jj < nj; jj++) {
          const float g = sm.sG[jj * FK_B + bb];
          const float4 w = ld4(sm.sS + jj * FK_LDS + q4 * 4);
          a.x = fmaf(g, w.x, a.x); a.y = fmaf(g, w.y, a.y); a.z = fmaf(g, w.z, a.z); a.w = fmaf(g, w.w, a.w);
        }
        st4(part + (size_t)bb * ldL + q4 * 4, a);
      }
    }
    if (has_chunk && nj == 0) for (int i = tid; i < M * ldL; i += FK_THREADS) part[i] = 0.f;
    // ---- barrier B3: partial dL/dh complete.  Arrive, update the chunk's rows while the others arrive, then wait ----
    __syncthreads();
    FK_STAMP(13);
    bar_epoch += 1;
    if (tid == 0) red_release_add(&fs->bar, 1u);
    // sparse update from shared memory (rows prefetched before the step): one warp per duplicate group.  Nothing before the
    // next step's prefetch reads these rows, which waits for fs->rows.  Written out rather than with SparseUpd4 / SparseUpd,
    // which cost this kernel a 16-byte register spill; same arithmetic.
    for (int j = warp; j < nj; j += FK_THREADS / 32) {
      const int item = sm.sIt[buf][j];
      if (j > 0 && sm.sIt[buf][j - 1] == item) continue;
      int je = j + 1;
      while (je < nj && sm.sIt[buf][je] == item) je++;
      if (lane < kw) {
        const float4 p0 = ld4(sm.sS + j * FK_LDS + lane * 4);
        float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), v0 = a0, al = a0, vl = a0;
        if (ada) a0 = ld4(sm.sAcc + j * FK_LDS + lane * 4);
        if (mom) v0 = ld4(sm.sVel + j * FK_LDS + lane * 4);
        float4 ps = p0;
        for (int k = j; k < je; k++) {
          const float4 g = ld4(sm.sD + k * FK_LDS + lane * 4);
          float4 gs = g;
          if (ada) {
            al.x = a0.x + g.x * g.x; al.y = a0.y + g.y * g.y; al.z = a0.z + g.z * g.z; al.w = a0.w + g.w * g.w;
            gs.x = __fdiv_rn(g.x, sqrtf(al.x + G4R_EPS_ADA)); gs.y = __fdiv_rn(g.y, sqrtf(al.y + G4R_EPS_ADA));
            gs.z = __fdiv_rn(g.z, sqrtf(al.z + G4R_EPS_ADA)); gs.w = __fdiv_rn(g.w, sqrtf(al.w + G4R_EPS_ADA));
          }
          float4 d;
          if (md.lmbd > 0.f) { d.x = md.lr * (gs.x + md.lmbd * p0.x); d.y = md.lr * (gs.y + md.lmbd * p0.y); d.z = md.lr * (gs.z + md.lmbd * p0.z); d.w = md.lr * (gs.w + md.lmbd * p0.w); }
          else { d.x = md.lr * gs.x; d.y = md.lr * gs.y; d.z = md.lr * gs.z; d.w = md.lr * gs.w; }
          if (mom) {
            vl.x = md.mom * v0.x - d.x; vl.y = md.mom * v0.y - d.y; vl.z = md.mom * v0.z - d.z; vl.w = md.mom * v0.w - d.w;
            ps.x += vl.x; ps.y += vl.y; ps.z += vl.z; ps.w += vl.w;
          } else { ps.x -= d.x; ps.y -= d.y; ps.z -= d.z; ps.w -= d.w; }
        }
        const size_t off = (size_t)item * ldL + lane * 4;
        st4(md.Wy + off, ps);
        if (ada) st4(md.Wy_acc + off, al);
        if (mom) st4(md.Wy_vel + off, vl);
      }
      if (lane == 0) {
        const float p0 = sm.sByP[j];
        float a0 = sm.sByA[j], v0 = sm.sByV[j], al = 0.f, vl = 0.f, ps = p0;
        for (int k = j; k < je; k++) {
          const float g = sm.sDby[k];
          float gs = g;
          if (ada) { al = a0 + g * g; gs = __fdiv_rn(g, sqrtf(al + G4R_EPS_ADA)); }
          const float d = md.lmbd > 0.f ? md.lr * (gs + md.lmbd * p0) : md.lr * gs;
          if (mom) { vl = md.mom * v0 - d; ps += vl; } else ps -= d;
        }
        md.By[item] = ps;
        if (ada) md.By_acc[item] = al;
        if (mom) md.By_vel[item] = vl;
      }
    }
    __syncthreads();
    if (tid == 0) red_release_add(&fs->rows, 1u);
    FK_STAMP(14);
    if (tid == 0) wait_ge(&fs->bar, bar_epoch * (unsigned int)ncta);
    __syncthreads();
    FK_STAMP(3);
    // ---- b1 on every CTA, then prefetch the next step's rows ----
    fk_b1<CL>(md, sm, s, cta, ncta);
    __syncthreads();
    if (tid == 0) red_release_add(&fs->b1_done, 1u);
    FK_STAMP(15);
    // prefetch of the next step's rows, which any CTA may have updated inside its B3 window (the GRU CTAs of step_mode 2
    // issue it inside the B2 group-barrier window instead)
    if (CL || !gru) fk_wait_rows_prefetch(md, sm, fs, s, n_steps, buf, pw, ncta);
    FK_STAMP_CL(4);
    if constexpr (!CL) {
      if (gru) {                                  // during the b1_done wait: operands of the dense update, lanes of the next step
        fk_dense_stage(md, sm, s, cta);
        if (s + 1 < n_steps) fk_stage_lanes(md, sm, s + 1, md.wM[s + 1]);
      }
    }
    // ---- GRU role: backward, dense update, forward of the next step ----
    if constexpr (CL) {
      if (gru) {
        if (s + 1 < n_steps) fk_stage_lanes(md, sm, s + 1, md.wM[s + 1]);
        cf_backward(md, sm, cc, fs, s, ncta, s + 1 < n_steps, (tstamp && cta == 0 && FK_STAMP_OK(s)) ? tstamp + (size_t)s * 16 : nullptr, FK_FTS(s));
        FK_STAMP(6);
        if (s + 1 < n_steps) {
          cf_f1(md, sm, cc, s + 1, true, &fs->in_done, (unsigned int)(s + 1) * (unsigned int)in_ctas, FK_FTS(s));
          FK_STAMP(7);
          cf_f2(md, sm, cc, s + 1, FK_FTS(s));
          __syncthreads();
          if (tid == 0) red_release_add(&fs->h_ready, 1u);
        } else {
          cl_wait();                                   // matches the arrive left pending by cf_backward
        }
        FK_STAMP(8);
      } else if (cta < G + in_ctas) {
        const unsigned int tgt = (unsigned int)(s + 1) * (unsigned int)G;           // dvec rows of the step complete
        if (in_ctas == B && ly.ld3 / 4 <= FK_THREADS) fk_sparse_in_one(md, sm, s, cta - G, &fs->grp, tgt);
        else {
          if (tid == 0) wait_ge(&fs->grp, tgt);
          __syncthreads();
          for (int b = cta - G; b < B; b += in_ctas) { fk_sparse_in(md, sm, s, b); __syncthreads(); }
        }
        __syncthreads();
        if (tid == 0) red_release_add(&fs->in_done, 1u);
      }
    } else if (gru) {
      if (tid == 0) wait_ge(&fs->b1_done, (unsigned int)(s + 1) * (unsigned int)ncta);
      __syncthreads();
      const float dc0 = fk_dense_dcol(ly, M, cta, 0);  // da_h / da_z columns of the owned slab: in flight during b2
      fk_b2(md, sm, s, cta);
      fk_group_arrive(fs, gepoch);       // epoch 2*s + 2: all of dvec (da_r included) is complete -> the helper CTAs poll this counter
      FK_STAMP(5);
      if (s + 1 < n_steps) {                     // the prefetch, inside the window: wait for every CTA's row update...
        if (tid == 0) wait_ge(&fs->rows, (unsigned int)(s + 1) * (unsigned int)ncta);
        __syncthreads();
      }
      FK_STAMP(4);
      fk_prefetch_rows(md, sm, s + 1, n_steps, buf ^ 1, pw);   // ...then issue the copies
      FK_STAMP(10);
      fk_dense_put_dcol(sm, ly, cta, 0, dc0);
      __syncthreads();
      fk_dense_update(md, sm, s, cta, 0);
      if (s + 1 < n_steps && cta * FK_W1 < 2 * L) fk_f1_stage_h(ly, sm);
      FK_STAMP(1);
      fk_group_wait(fs, gepoch);
      FK_STAMP(9);
      const float dc1 = fk_dense_dcol(ly, M, cta, 1);  // da_r columns
      fk_dense_put_dcol(sm, ly, cta, 1, dc1);
      __syncthreads();
      fk_dense_update(md, sm, s, cta, 1);
      __syncthreads();
      FK_STAMP(6);
      if (s + 1 < n_steps) {
        fk_f1(md, sm, s + 1, cta, &fs->in_done, (unsigned int)(s + 1) * (unsigned int)in_ctas, nullptr, true, tstamp && cta == 0);   // waits for the helper CTAs' input-row updates
        fk_group_barrier(fs, gepoch);
        FK_STAMP(7);
        if (tstamp && cta == 0 && tid == 0 && FK_STAMP_OK(s)) { tstamp[(size_t)s * 16 + 11] = sm.sTs[0]; tstamp[(size_t)s * 16 + 12] = sm.sTs[1]; }
        fk_f2(md, sm, s + 1, cta, nullptr, true);
        __syncthreads();
        if (tid == 0) red_release_add(&fs->h_ready, 1u);
      }
      FK_STAMP(8);
    } else if (cta < FK_G + in_ctas) {
      // the GRU group's barrier after B2 is its (2 s + 2)-th group barrier (1 in the prologue, then B2 / f1 per step)
      if (tid == 0) wait_ge(&fs->grp, (unsigned int)(2 * s + 2) * FK_G);
      __syncthreads();
      for (int b = cta - FK_G; b < B; b += in_ctas) { fk_sparse_in(md, sm, s, b); __syncthreads(); }
      __syncthreads();
      if (tid == 0) red_release_add(&fs->in_done, 1u);
    }
  }
  if constexpr (CL) { if (gru) cf_store_resident(md, sm, cc); }
#undef FK_STAMP
#undef FK_STAMP_CL
}
