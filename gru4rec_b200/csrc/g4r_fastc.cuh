// g4r_fastc.cuh -- GRU phases of the role-specialised kernel on ONE thread-block cluster (step_mode 3).
//
// The 48-CTA GRU group of k_fast pays four global-memory group barriers (~1.2 us each) and an L2 round trip per
// phase for a 32 x 100 GRU.  Here the GRU side lives on cluster 0 (CS CTAs, CS = 8):
//  * every CTA owns a slice K_c of the hidden units (whole 16-byte quads) and keeps the matching columns of Wh and
//    Wrz (r and z blocks) together with their Adagrad / momentum state RESIDENT in shared memory for the whole window
//    (read once at kernel start, written back at kernel end): the dense update never touches global memory;
//  * phases exchange data through distributed shared memory (st.shared::cluster pushes) and hardware cluster
//    barriers (barrier.cluster, ~0.2 us) instead of L2 + global counters;
//  * per mini-batch: reduce-scatter of d(H*r) partials (1 barrier), all-gather of H*r (1 barrier + 1 split barrier).
// Column CTAs, helper CTAs (input-row update) and all numerics formulas are shared with k_fast.
//
// Reference formulas (hidasib/GRU4Rec): cf_f1 = rz gates, gru4rec.py:460-462 (r | z column blocks of Wrz, vec[:, L:]);
// cf_f2 = candidate, new state, dropout, reset, :463-466; cf_backward = GRU backward of SURVEY appendix A (the reference uses
// T.grad, :383-384: dh -> dz, dh~ -> da_h; d(H*r) = da_h Wh^T -> da_r) followed by the dense Adagrad (+momentum) update of
// gru4rec.py:330-334,390-406 on the resident columns.
#pragma once

constexpr int FC_SL = 17;        // row stride of the [32 x <=16] slice buffers (conflict-free with lane = batch row)
constexpr int FC_PH = 16;        // max hidden units per cluster CTA (L <= 128 with 8 CTAs)
constexpr int FC_PS = 20;        // row stride of the push staging buffer (16-byte aligned rows)

struct FastSmemC {
  // column role (same fields as FastSmem); during the GRU phases sY / sD / (sG,sO,sPart) are reused, see below
  alignas(128) float sY[FK_B * FK_LDS];          // h of the step | GRU phases: cH  = Hold / H rows (all lanes, all units)
  float sS[FK_CT * FK_LDS];
  float sAcc[FK_CT * FK_LDS];
  float sVel[FK_CT * FK_LDS];
  float sTW[FK_B * FK_LDS];
  float sD[FK_CT * FK_LDS];                      // dSy rows        | GRU phases: cHr = Hold * r (all lanes, all units)
  float sG[FK_CT * FK_B];                        // dL/do           | GRU backward: cRed[src][unit][lane] (sG, sO, sPart contiguous)
  float sO[FK_CT * FK_B];
  float sPart[2048];
  float sRS[FK_B * 8];
  float sT[FK_B];
  float sBias[FK_CT], sByP[FK_CT], sByA[FK_CT], sByV[FK_CT], sDby[FK_CT], sTB[FK_B];
  int sIt[2][FK_CT], sPos[2][FK_CT], sTc[2][FK_B], sYit[2][FK_B], sCb[2][2];
  int sFlag[4];
  alignas(8) unsigned long long mbar;
  int gIdx[3 * FK_B];
  // cluster GRU role
  int cQ0[17];                                   // first quad of every rank's unit slice (cQ0[CS] = number of quads)
  int cOwn[32];                                  // owning rank of every quad
  alignas(16) float rP[3 * FC_PH * FK_LDS];      // resident columns: [0,16) Wh[:, k0+j] | [16,32) Wrz[:, k0+j] | [32,48) Wrz[:, L+k0+j]
  float rA[3 * FC_PH * FK_LDS];                  // their Adagrad accumulators
  float rV[3 * FC_PH * FK_LDS];                  // their momentum buffers
  float rB[3][3 * FC_PH];                        // Bh slice (h~ | r | z) : value, accumulator, momentum
  float cR[FK_B * FC_SL], cZ[FK_B * FC_SL], cHt[FK_B * FC_SL], cAh[FK_B * FC_SL], cHo[FK_B * FC_SL];   // forward saves of the slice
  float cDh[FK_B * FC_SL], cDr[FK_B * FC_SL], cDz[FK_B * FC_SL];                                       // da_h, da_r, da_z of the slice
  alignas(16) float cPush[FK_B * FC_PS];         // staging of the H*r slice before the 16-byte pushes
};
static_assert(sizeof(FastSmemC) <= 232448, "FastSmemC exceeds the 227 KB shared memory of one CTA");
static_assert(offsetof(FastSmemC, sO) == offsetof(FastSmemC, sG) + sizeof(float) * FK_CT * FK_B, "cRed region must be contiguous");
static_assert(offsetof(FastSmemC, sPart) == offsetof(FastSmemC, sO) + sizeof(float) * FK_CT * FK_B, "cRed region must be contiguous");
static_assert(FK_CT * FK_B * 2 + 2048 >= 8 * FC_PH * FK_B, "cRed region too small");

struct ClusterCtx { int rk, CS, k0, nk; };
// fine-grained %globaltimer stamps of the cluster phases (debug builds with -DG4R_CF_FINE only)
#ifdef G4R_CF_FINE
#define CF_T(k) do { if (fts && threadIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); fts[k] = t_; } } while (0)
#else
#define CF_T(k) do { } while (0)
#endif

__device__ __forceinline__ unsigned int cl_rank() { unsigned int r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ unsigned int cl_size() { unsigned int r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cl_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cl_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t cl_map(const void* p, unsigned int rank) {
  uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(rank)); return r;
}
__device__ __forceinline__ void cl_st(uint32_t addr, float v) { asm volatile("st.shared::cluster.f32 [%0], %1;" :: "r"(addr), "f"(v) : "memory"); }
__device__ __forceinline__ void cl_st4(uint32_t addr, float4 v) {
  asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" :: "r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// unit slices: the kw = ldL/4 quads are dealt to the CS ranks in contiguous runs of floor/ceil(kw / CS) quads
__device__ __forceinline__ ClusterCtx cf_init(const ModelDev& md, FastSmemC& sm) {
  ClusterCtx cc;
  cc.rk = (int)cl_rank(); cc.CS = (int)cl_size();
  const int kw = md.layer[0].ldL / 4;
  if (threadIdx.x <= (unsigned)cc.CS && threadIdx.x < 17) sm.cQ0[threadIdx.x] = (int)threadIdx.x * kw / cc.CS;
  __syncthreads();
  if (threadIdx.x < 32) {
    int o = 0;
    for (int r = 0; r < cc.CS; r++) if ((int)threadIdx.x >= sm.cQ0[r]) o = r;
    sm.cOwn[threadIdx.x] = o;
  }
  cc.k0 = 4 * sm.cQ0[cc.rk];
  cc.nk = 4 * (sm.cQ0[cc.rk + 1] - sm.cQ0[cc.rk]);
  __syncthreads();
  return cc;
}

// resident columns <-> global (once per window each)
__device__ void cf_load_resident(const ModelDev& md, FastSmemC& sm, const ClusterCtx& cc) {
  const LayerDev& ly = md.layer[0];
  const int L = ly.L, tid = threadIdx.x;
  for (int i = tid; i < 3 * FC_PH * FK_LDS; i += FK_THREADS) {
    const int q = i / FK_LDS, k = i % FK_LDS, t = q / FC_PH, j = q % FC_PH;
    const int c = cc.k0 + j;
    float p = 0.f, a = 0.f, v = 0.f;
    if (j < cc.nk && c < L && k < L) {
      if (t == 0) {
        const size_t o = (size_t)k * ly.ldL + c;
        p = ly.Wh[o]; if (ly.Wh_acc) a = ly.Wh_acc[o]; if (ly.Wh_vel) v = ly.Wh_vel[o];
      } else {
        const size_t o = (size_t)k * ly.ld2 + (t == 2 ? L : 0) + c;
        p = ly.Wrz[o]; if (ly.Wrz_acc) a = ly.Wrz_acc[o]; if (ly.Wrz_vel) v = ly.Wrz_vel[o];
      }
    }
    sm.rP[i] = p; sm.rA[i] = a; sm.rV[i] = v;
  }
  if (tid < 3 * FC_PH) {
    const int t = tid / FC_PH, j = tid % FC_PH, c = cc.k0 + j;
    float p = 0.f, a = 0.f, v = 0.f;
    if (j < cc.nk && c < L) { const int o = t * L + c; p = ly.Bh[o]; if (ly.Bh_acc) a = ly.Bh_acc[o]; if (ly.Bh_vel) v = ly.Bh_vel[o]; }
    sm.rB[0][tid] = p; sm.rB[1][tid] = a; sm.rB[2][tid] = v;
  }
  __syncthreads();
}
__device__ void cf_store_resident(const ModelDev& md, FastSmemC& sm, const ClusterCtx& cc) {
  const LayerDev& ly = md.layer[0];
  const int L = ly.L, tid = threadIdx.x;
  __syncthreads();
  for (int i = tid; i < 3 * FC_PH * FK_LDS; i += FK_THREADS) {
    const int q = i / FK_LDS, k = i % FK_LDS, t = q / FC_PH, j = q % FC_PH;
    const int c = cc.k0 + j;
    if (j < cc.nk && c < L && k < L) {
      if (t == 0) {
        const size_t o = (size_t)k * ly.ldL + c;
        ly.Wh[o] = sm.rP[i]; if (ly.Wh_acc) ly.Wh_acc[o] = sm.rA[i]; if (ly.Wh_vel) ly.Wh_vel[o] = sm.rV[i];
      } else {
        const size_t o = (size_t)k * ly.ld2 + (t == 2 ? L : 0) + c;
        ly.Wrz[o] = sm.rP[i]; if (ly.Wrz_acc) ly.Wrz_acc[o] = sm.rA[i]; if (ly.Wrz_vel) ly.Wrz_vel[o] = sm.rV[i];
      }
    }
  }
  if (tid < 3 * FC_PH) {
    const int t = tid / FC_PH, j = tid % FC_PH, c = cc.k0 + j;
    if (j < cc.nk && c < L) { const int o = t * L + c; ly.Bh[o] = sm.rB[0][tid]; if (ly.Bh_acc) ly.Bh_acc[o] = sm.rB[1][tid]; if (ly.Bh_vel) ly.Bh_vel[o] = sm.rB[2][tid]; }
  }
}

// F1 of step s on the cluster: r, z of the slice; pushes Hold * r to every CTA of the cluster.
// `pending`: a barrier.cluster.arrive was already issued by this CTA (after the dense update of the previous step) and
// the H rows of the step are already staged in cH (cf_backward prefetched them during the dense update).
__device__ void cf_f1(const ModelDev& md, FastSmemC& sm, const ClusterCtx& cc, int s, bool pending, const unsigned int* wait_ctr, unsigned int wait_target, unsigned long long* fts) {
  const LayerDev& ly = md.layer[0];
  const int M = md.wM[s], L = ly.L, ldL = ly.ldL, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int kw = ldL / 4, nk = cc.nk;
  float* cH = sm.sY;
  float* cHr = sm.sD;
  // H rows of the step's lanes (zero rows for empty lanes); gIdx of step s was staged by the caller
  if (!pending) stage_rows4(cH, FK_LDS, FK_B, kw, [&](int rr) -> const float* { const int sl = sm.gIdx[rr]; return sl >= 0 ? ly.H + (size_t)sl * ldL : nullptr; });
  // the gathered input rows of this step may still be in flight on the helper CTAs (previous step's update): if they are
  // already done (the usual case), the epilogue operands are fetched now and their latency hides behind the product
  if (tid == 0) sm.sFlag[3] = (!wait_ctr || ld_acquire_u32(wait_ctr) >= wait_target) ? 1 : 0;
  __syncthreads();
  const bool early = sm.sFlag[3] != 0;
  CF_T(8);
  // this thread: lane b = lane, slice columns qi = warp and warp + 16 out of [r_0..r_nk-1 | z_0..z_nk-1]
  float acc[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
  const float* wrow[2]; bool has[2]; float pre[2] = {0.f, 0.f};
#pragma unroll
  for (int u = 0; u < 2; u++) {
    const int qi = warp + 16 * u;
    has[u] = qi < 2 * nk;
    wrow[u] = sm.rP + (size_t)(qi < nk ? FC_PH + qi : 2 * FC_PH + (qi - nk)) * FK_LDS;
    if (!has[u]) wrow[u] = sm.rP;
    const bool isr = qi < nk;
    const int c = cc.k0 + (isr ? qi : qi - nk);
    if (early && has[u] && lane < M && c < L) pre[u] = ly.Wx[(size_t)sm.gIdx[FK_B + lane] * ly.ld3 + (isr ? L : 2 * L) + c];
  }
  {
    const float* hr = cH + lane * FK_LDS;
    for (int c4 = 0; c4 < kw; c4++) {
      const float4 y = ld4(hr + c4 * 4);
#pragma unroll
      for (int u = 0; u < 2; u++) {
        if (has[u]) {
          const float4 w = ld4(wrow[u] + c4 * 4);
          acc[u][0] = fmaf(y.x, w.x, acc[u][0]); acc[u][1] = fmaf(y.y, w.y, acc[u][1]);
          acc[u][0] = fmaf(y.z, w.z, acc[u][0]); acc[u][1] = fmaf(y.w, w.w, acc[u][1]);
        }
      }
    }
  }
  CF_T(9);
  // the gathered input rows of this step may still be in flight on the helper CTAs (previous step's update)
  if (!early) { if (tid == 0) wait_ge(wait_ctr, wait_target); __syncthreads(); }
  CF_T(10);
#pragma unroll
  for (int u = 0; u < 2; u++) {
    const int qi = warp + 16 * u;
    if (!has[u]) continue;
    const bool isr = qi < nk;
    const int j = isr ? qi : qi - nk, c = cc.k0 + j;
    float g = 0.f, ho = 0.f;
    if (lane < M && c < L) {
      if (!early) pre[u] = ly.Wx[(size_t)sm.gIdx[FK_B + lane] * ly.ld3 + (isr ? L : 2 * L) + c];
      g = sigmoidf_(acc[u][0] + acc[u][1] + (pre[u] + sm.rB[0][(isr ? FC_PH : 2 * FC_PH) + j]));
      if (isr) { ho = cH[lane * FK_LDS + c]; ly.r[(size_t)lane * ldL + c] = g; ly.Hold[(size_t)lane * ldL + c] = ho; }
    }
    if (isr) { sm.cR[lane * FC_SL + j] = g; sm.cHo[lane * FC_SL + j] = ho; sm.cPush[lane * FC_PS + j] = ho * g; }
    else sm.cZ[lane * FC_SL + j] = g;
  }
  // every CTA of the cluster must be done reading H*r of the previous step (its dense update) before the pushes
  CF_T(11);
  if (!pending) cl_arrive();
  cl_wait();
  __syncthreads();
  CF_T(12);
  {
    const int nq = nk / 4;
    for (int i = tid; i < FK_B * nq; i += FK_THREADS) {
      const int b = i / nq, jq = i % nq;
      const float4 v = ld4(sm.cPush + b * FC_PS + jq * 4);
      const float* dst = cHr + b * FK_LDS + cc.k0 + jq * 4;
      for (int t = 0; t < cc.CS; t++) cl_st4(cl_map(dst, (unsigned)t), v);
    }
  }
  CF_T(13);
  cl_arrive();
  cl_wait();
  CF_T(14);
}

// F2 of step s on the cluster: h~, h, dropout, H_new for the slice (one column per warp)
__device__ void cf_f2(const ModelDev& md, FastSmemC& sm, const ClusterCtx& cc, int s, unsigned long long* fts) {
  const LayerDev& ly = md.layer[0];
  const int M = md.wM[s], L = ly.L, ldL = ly.ldL, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int kw = ldL / 4;
  const float* cHr = sm.sD;
  const int j = warp, c = cc.k0 + j;
  const bool on = j < cc.nk && c < L && lane < M;
  float pre = 0.f;
  if (on) pre = ly.Wx[(size_t)sm.gIdx[FK_B + lane] * ly.ld3 + c] + sm.rB[0][j];
  float a0 = 0.f, a1 = 0.f;
  if (j < cc.nk) {
    const float* hr = cHr + lane * FK_LDS;
    const float* wr = sm.rP + (size_t)j * FK_LDS;
    for (int c4 = 0; c4 < kw; c4++) {
      const float4 y = ld4(hr + c4 * 4), w = ld4(wr + c4 * 4);
      a0 = fmaf(y.x, w.x, a0); a1 = fmaf(y.y, w.y, a1); a0 = fmaf(y.z, w.z, a0); a1 = fmaf(y.w, w.w, a1);
    }
  }
  if (on) {
    const float v = a0 + a1 + pre;
    const float ht = act_fwd(md.hact, v);
    const float z = sm.cZ[lane * FC_SL + j], ho = sm.cHo[lane * FC_SL + j];
    float h = (1.0f - z) * ho + z * ht;
    if (md.p_drop_h > 0.f) h *= drop_scale(md.drop_seed, md.wG[s], 0u, (uint32_t)(lane * L + c), 1.0f - md.p_drop_h);
    sm.cAh[lane * FC_SL + j] = v;
    sm.cHt[lane * FC_SL + j] = ht;
    ly.y[(size_t)lane * ldL + c] = h;
    ly.H[(size_t)sm.gIdx[lane] * ldL + c] = (sm.gIdx[2 * FK_B + lane] & 1) ? 0.f : h;
  }
  CF_T(15);
}

// Backward of step s on the cluster + dense update of the resident columns.  Leaves one barrier.cluster.arrive pending.
__device__ void cf_backward(const ModelDev& md, FastSmemC& sm, const ClusterCtx& cc, FastSync* fs, int s, int ncta, bool have_next, unsigned long long* ts, unsigned long long* fts) {
  const LayerDev& ly = md.layer[0];
  const int M = md.wM[s], L = ly.L, ldL = ly.ldL, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int kw = ldL / 4, nk = cc.nk;
  float* cH = sm.sY;
  float* cHr = sm.sD;
  float* cRed = sm.sG;
  CF_T(0);
  // (a) Hold and r of the step (all lanes, all units; written by the cluster in F1) -- independent of dL/dh, issued first
  float4 hv[2], rv[2];
#pragma unroll
  for (int u = 0; u < 2; u++) {
    const int i = tid + u * FK_THREADS;
    hv[u] = make_float4(0.f, 0.f, 0.f, 0.f); rv[u] = hv[u];
    if (i < FK_B * kw) {
      const int rr = i / kw, c4 = i % kw;
      if (rr < M) { hv[u] = ld4(ly.Hold + (size_t)rr * ldL + c4 * 4); rv[u] = ld4(ly.r + (size_t)rr * ldL + c4 * 4); }
    }
  }
  // (b) dL/dh of the step is complete when every CTA has finished its part of the reduction
  if (tid == 0) wait_ge(&fs->b1_done, (unsigned int)(s + 1) * (unsigned int)ncta);
  __syncthreads();
  CF_T(1);
  const int b = lane, j = warp, c = cc.k0 + j;
  const bool on = j < nk && c < L && b < M;
  float dyv = 0.f;
  if (on) dyv = ly.dy[(size_t)b * ldL + c];
#pragma unroll
  for (int u = 0; u < 2; u++) {
    const int i = tid + u * FK_THREADS;
    if (i < FK_B * kw) {
      const int rr = i / kw, c4 = i % kw;
      st4(cH + rr * FK_LDS + c4 * 4, hv[u]);
      st4(cHr + rr * FK_LDS + c4 * 4, make_float4(hv[u].x * rv[u].x, hv[u].y * rv[u].y, hv[u].z * rv[u].z, hv[u].w * rv[u].w));
    }
  }
  if (j < FC_PH) {
    float dah = 0.f, daz = 0.f;
    if (on) {
      const float ht = sm.cHt[b * FC_SL + j], ho = sm.cHo[b * FC_SL + j], z = sm.cZ[b * FC_SL + j], ah = sm.cAh[b * FC_SL + j];
      float dh = dyv;
      if (md.p_drop_h > 0.f) dh *= drop_scale(md.drop_seed, md.wG[s], 0u, (uint32_t)(b * L + c), 1.0f - md.p_drop_h);
      const float dz = dh * (ht - ho);
      dah = dh * z * act_der(md.hact, ah, ht);
      daz = dz * z * (1.f - z);
      ly.dvec[(size_t)b * ly.ld3 + c] = dah;
      ly.dvec[(size_t)b * ly.ld3 + 2 * L + c] = daz;
    }
    sm.cDh[b * FC_SL + j] = dah; sm.cDz[b * FC_SL + j] = daz;
  }
  __syncthreads();
  CF_T(2);
  // (c) partial d(H*r)[b][k] = sum_{j in slice} da_h[b][j] Wh[k][k0+j] for ALL k, pushed to the owner of k
  float dhr[FC_PH];                                   // da_h of lane `lane` (rows of Wh beyond the slice are zero in rP)
#pragma unroll
  for (int jj = 0; jj < FC_PH; jj++) dhr[jj] = sm.cDh[lane * FC_SL + jj];
  for (int k = warp; k < L; k += FK_NW) {
    float a = 0.f, a2 = 0.f;
#pragma unroll
    for (int jj = 0; jj < FC_PH; jj += 2) { a = fmaf(dhr[jj], sm.rP[jj * FK_LDS + k], a); a2 = fmaf(dhr[jj + 1], sm.rP[(jj + 1) * FK_LDS + k], a2); }
    a += a2;
    const int owner = sm.cOwn[k >> 2];
    const int kk = k - 4 * sm.cQ0[owner];
    cl_st(cl_map(cRed + (cc.rk * FC_PH + kk) * FK_B + lane, (unsigned)owner), a);
  }
  CF_T(3);
  cl_arrive();
  cl_wait();
  CF_T(4);
  // (d) da_r of the slice
  if (j < FC_PH) {
    float dar = 0.f;
    if (on) {
      float v = 0.f;
      for (int src = 0; src < cc.CS; src++) v += cRed[(src * FC_PH + j) * FK_B + b];
      const float ho = sm.cHo[b * FC_SL + j], r = sm.cR[b * FC_SL + j];
      dar = v * ho * r * (1.f - r);
      ly.dvec[(size_t)b * ly.ld3 + L + c] = dar;
    }
    sm.cDr[b * FC_SL + j] = dar;
  }
  __syncthreads();
  if (tid == 0) red_release_add(&fs->grp, 1u);        // dvec rows complete -> the helper CTAs update the gathered input rows
  if (ts && tid == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); ts[5] = t_; }
  CF_T(5);
  // (e) gradients of the resident columns (warp = unit j of the slice, lane = quad of the reduction index k) + update
  const bool ada = md.adapt == G4R_ADAPT_ADAGRAD, mom = md.mom > 0.f;
  // H rows of the NEXT step (final since its F2): loaded now, stored into cH after the dense update has read Hold from it
  float4 hn[2];
#pragma unroll
  for (int u = 0; u < 2; u++) {
    const int i = tid + u * FK_THREADS;
    hn[u] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (have_next && i < FK_B * kw) { const int sl = sm.gIdx[i / kw]; if (sl >= 0) hn[u] = ld4(ly.H + (size_t)sl * ldL + (i % kw) * 4); }
  }
  float sbh = 0.f, sbr = 0.f, sbz = 0.f;             // bias gradients of unit j (same summation order as the matrices)
  if (j < nk && lane < kw) {
    float4 gh = make_float4(0.f, 0.f, 0.f, 0.f), gr = gh, gz = gh;
    for (int bb = 0; bb < M; bb++) {
      const float4 a = ld4(cHr + bb * FK_LDS + lane * 4), h4 = ld4(cH + bb * FK_LDS + lane * 4);
      const float dh = sm.cDh[bb * FC_SL + j], dr = sm.cDr[bb * FC_SL + j], dz = sm.cDz[bb * FC_SL + j];
      sbh += dh; sbr += dr; sbz += dz;
      gh.x = fmaf(a.x, dh, gh.x); gh.y = fmaf(a.y, dh, gh.y); gh.z = fmaf(a.z, dh, gh.z); gh.w = fmaf(a.w, dh, gh.w);
      gr.x = fmaf(h4.x, dr, gr.x); gr.y = fmaf(h4.y, dr, gr.y); gr.z = fmaf(h4.z, dr, gr.z); gr.w = fmaf(h4.w, dr, gr.w);
      gz.x = fmaf(h4.x, dz, gz.x); gz.y = fmaf(h4.y, dz, gz.y); gz.z = fmaf(h4.z, dz, gz.z); gz.w = fmaf(h4.w, dz, gz.w);
    }
#pragma unroll
    for (int t = 0; t < 3; t++) {
      const float4 g4 = t == 0 ? gh : (t == 1 ? gr : gz);
      const int o = (t * FC_PH + j) * FK_LDS + lane * 4;
      const float ge[4] = {g4.x, g4.y, g4.z, g4.w};
#pragma unroll
      for (int e = 0; e < 4; e++) {
        const float g = ge[e], p0 = sm.rP[o + e];
        float gs = g;
        if (ada) gs = adagrad_scale(g, sm.rA[o + e], sm.rA[o + e]);
        sm.rP[o + e] = dense_step(md, gs, p0, sm.rV[o + e], mom);
      }
    }
  }
  CF_T(6);
  if (j < nk && lane < 3 && c < L) {
    float g = lane == 0 ? sbh : (lane == 1 ? sbr : sbz);
    if (lane >= kw) {                                   // fewer than 3 quads: this lane did not run the loop above
      const float* d = lane == 0 ? sm.cDh : (lane == 1 ? sm.cDr : sm.cDz);
      g = 0.f;
      for (int bb = 0; bb < M; bb++) g += d[bb * FC_SL + j];
    }
    const int o = lane * FC_PH + j;
    const float p0 = sm.rB[0][o];
    float gs = g;
    if (ada) gs = adagrad_scale(g, sm.rB[1][o], sm.rB[1][o]);
    sm.rB[0][o] = dense_step(md, gs, p0, sm.rB[2][o], mom);
  }
  __syncthreads();
  cl_arrive();          // this CTA no longer reads H*r of step s
#pragma unroll
  for (int u = 0; u < 2; u++) {
    const int i = tid + u * FK_THREADS;
    if (have_next && i < FK_B * kw) st4(cH + (i / kw) * FK_LDS + (i % kw) * 4, hn[u]);
  }
  CF_T(7);
}
