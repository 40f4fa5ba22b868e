// g4r_shard.cuh -- multi-GPU training with ROW-SHARDED item tables and the exchange INSIDE the persistent kernel
// (SURVEY section 8e; the reference is single-device, .theanorc_gru4rec:3, so the semantics are the ones stated in
// g4r_multi.cuh: one lock step = the mini-batches of all ranks as ONE list of positions in (rank, position) order under
// the single-GPU duplicate rules of gru4rec.py:335-340,407-431; dense gradients are summed).
//
// Layout: row i of Wy / By / Wx0 (and their Adagrad / momentum state) lives ONLY on rank i % R, local row i / R, inside a
// library-owned cudaMalloc segment that every peer maps through cudaIpc.  A table row is [Wy row | By | 0 0 0] so that one
// bulk copy brings the bias along.  Dense GRU weights are replicated.
//
// One lock step on every rank, all inside k_fast_mg (the role-specialised kernel of g4r_fast.cuh):
//   columns  every CTA owns an equal slice of the rank's sorted score columns; the parameter rows are fetched from their
//            OWNERS with TMA bulk copies over NVLink (peer-mapped addresses) while the GRU phases run;
//   export   the dSy|dby rows are stored straight into the owner's inbox (16-byte peer stores), fence.sys, sequence flag;
//   apply    68 "apply" CTAs of the owner wait for all ranks' flags and update the owned rows from the merged plan
//            (item, rank, position order; Adagrad / momentum state: last occurrence; parameter: all occurrences);
//   inputs   32 helper CTAs do the same for the gathered input rows Wx0[X] and fetch the rows of the next step;
//   dense    every GRU CTA pushes its slice of the dense gradient to all peers, sums the R slices in rank order (replicas stay
//            bit-identical) and applies Adagrad / momentum.
// Cross-GPU synchronisation = monotonic sequence flags in peer memory (st.release.sys / ld.acquire.sys), every poll with a
// time-out that raises an abort flag instead of hanging the box.  NCCL is used only for the per-window all-gather of the
// (model independent) sorted column lists.  Included from g4r_lib.cu after g4r_fast.cuh and g4r_multi.cuh.
#pragma once

constexpr unsigned long long MGS_TIMEOUT_NS = 4000000000ull;   // 4 s per cross-GPU wait

__device__ __forceinline__ unsigned int ld_acquire_sys_u32(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys_u32(unsigned int* p, unsigned int v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ float4 ld_volatile4(const float* p) {
  float4 v;
  asm volatile("ld.volatile.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long mgs_timer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// wait until the sequence flag *p (written by a peer GPU) reaches `target`; gives up after MGS_TIMEOUT_NS
__device__ __forceinline__ void wait_sys_ge(const unsigned int* p, unsigned int target, int* abort) {
  if ((int)(ld_acquire_sys_u32(p) - target) >= 0) return;
  const unsigned long long t0 = mgs_timer();
  unsigned int spins = 0;
  while ((int)(ld_acquire_sys_u32(p) - target) < 0) {
    if ((++spins & 127u) == 0) {
      if (*(volatile int*)abort) return;
      if (mgs_timer() - t0 > MGS_TIMEOUT_NS) { atomicExch(abort, 1); return; }
    }
  }
}
// warp 0 of the CTA: lane q < R waits for flag `first + q` of the local page (lane `skip` does not wait)
__device__ __forceinline__ void mgs_wait_flags(const ShardDev& sh, int first, int skip, unsigned int target) {
  if (threadIdx.x < 32) {
    const int q = threadIdx.x;
    if (q < sh.R && q != skip) wait_sys_ge(sh.flags[sh.rank] + (size_t)(first + q) * MGS_FLAG_STRIDE, target, sh.abort);
    __syncwarp();
  }
}
// ---- "LL" exchange: 8-byte (value, sequence) pairs.  A pair is written by ONE store, so data and flag travel together over
// NVLink: the receiver polls the data itself -- no system-scope fence, no separate flag, one one-way latency per exchange.
// The sequence is the lock-step number (>= 1, strictly increasing per slot), the slots are double buffered by its parity.
__device__ __forceinline__ void ll_store4(float* dst_pairs, float4 v, unsigned int seq) {
  asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" :: "l"(dst_pairs), "r"(__float_as_uint(v.x)), "r"(seq), "r"(__float_as_uint(v.y)), "r"(seq) : "memory");
  asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" :: "l"(dst_pairs + 4), "r"(__float_as_uint(v.z)), "r"(seq), "r"(__float_as_uint(v.w)), "r"(seq) : "memory");
}
__device__ __forceinline__ float4 ll_load4(const float* src_pairs, unsigned int seq, int* abort) {
  uint4 a, b;
  unsigned int spins = 0; unsigned long long t0 = 0;
  while (true) {
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w) : "l"(src_pairs) : "memory");
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "l"(src_pairs + 4) : "memory");
    if (a.y == seq && a.w == seq && b.y == seq && b.w == seq) break;
    if ((++spins & 127u) == 0) {
      if (*(volatile int*)abort) break;
      const unsigned long long t = mgs_timer();
      if (t0 == 0) t0 = t;
      if (t - t0 > MGS_TIMEOUT_NS) { atomicExch(abort, 1); break; }
    }
  }
  return make_float4(__uint_as_float(a.x), __uint_as_float(a.z), __uint_as_float(b.x), __uint_as_float(b.z));
}
__device__ __forceinline__ float ll_load1(const float* src_pair, unsigned int seq, int* abort) {
  uint2 a;
  unsigned int spins = 0; unsigned long long t0 = 0;
  while (true) {
    asm volatile("ld.volatile.global.v2.u32 {%0, %1}, [%2];" : "=r"(a.x), "=r"(a.y) : "l"(src_pair) : "memory");
    if (a.y == seq) break;
    if ((++spins & 127u) == 0) {
      if (*(volatile int*)abort) break;
      const unsigned long long t = mgs_timer();
      if (t0 == 0) t0 = t;
      if (t - t0 > MGS_TIMEOUT_NS) { atomicExch(abort, 1); break; }
    }
  }
  return __uint_as_float(a.x);
}
// local counter wait that also gives up when the step was aborted
__device__ __forceinline__ void wait_ge_abortable(const unsigned int* p, unsigned int target, int* abort) {
  unsigned int spins = 0;
  while (ld_acquire_u32(p) < target) { if ((++spins & 1023u) == 0 && *(volatile int*)abort) return; }
}

struct FastSmemMG : FastSmem {
  ShardDev sh;
  int sOw[2][FK_CT], sLoc[2][FK_CT], sYow[2][FK_B], sYloc[2][FK_B];
};
// second set of local counters of the sharded kernel (one per 128-byte line)
struct FastSyncMG {
  unsigned int exp_done;   unsigned int p0[31];
  unsigned int apply_done; unsigned int p1[31];
  unsigned int h1;         unsigned int p2[31];
  unsigned int h2;         unsigned int p3[31];
};

__device__ __forceinline__ void fk_load_idx_mg(const ModelDev& md, FastSmemMG& sm, int s, int n_steps, int chunk, int buf) {
  const int tid = threadIdx.x;
  if (s >= n_steps) return;
  const int M = md.wM[s], R = sm.sh.R;
  const int* cbeg = md.pCbeg + (size_t)s * (md.NCH + 1);
  const bool hc = chunk < md.NCH;
  const int cb = hc ? cbeg[chunk] : 0, ce = hc ? cbeg[chunk + 1] : 0;
  if (tid < FK_CT) {
    int it = 0, pos = 0;
    if (cb + tid < ce) { it = md.pItem[(size_t)s * md.NP + cb + tid]; pos = md.pPos[(size_t)s * md.NP + cb + tid]; }
    sm.sIt[buf][tid] = it; sm.sPos[buf][tid] = pos;
    sm.sOw[buf][tid] = it % R; sm.sLoc[buf][tid] = it / R;
  }
  if (tid >= 32 && tid < 32 + FK_B) {
    const int b = tid - 32;
    const int y = b < M ? md.wY[(size_t)s * md.B + b] : 0;
    sm.sTc[buf][b] = b < M ? md.pTcol[(size_t)s * md.B + b] : -1;
    sm.sYit[buf][b] = y; sm.sYow[buf][b] = y % R; sm.sYloc[buf][b] = y / R;
  }
  if (tid == 64) { sm.sCb[buf][0] = cb; sm.sCb[buf][1] = ce; }
}

// TMA prefetch of step s: the chunk's parameter rows (and the target rows) come from their owners' shards over NVLink
__device__ __forceinline__ void fk_prefetch_mg(const ModelDev& md, FastSmemMG& sm, int s, int n_steps, int buf, bool pw) {
  if (s >= n_steps) return;
  const int tid = threadIdx.x;
  const int M = md.wM[s];
  const int nj = sm.sCb[buf][1] - sm.sCb[buf][0];
  const int ldW = sm.sh.ldW;
  const unsigned int rowb = (unsigned int)ldW * 4u;
  uint64_t* bar = reinterpret_cast<uint64_t*>(&sm.mbar);
  const int ncopy = nj + (pw ? M : 0);
  if (tid == 0) {
    const unsigned int total = rowb * (unsigned int)ncopy;
    if (total > 0) mbar_expect_tx(bar, total);
    else asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
  }
  if ((tid & 31) == 0) {
    asm volatile("fence.proxy.async.global;" ::: "memory");
    for (int i = tid >> 5; i < ncopy; i += FK_NW) {
      if (i < nj) tma_row(sm.sS + i * FK_LDS, sm.sh.W[sm.sOw[buf][i]] + (size_t)sm.sLoc[buf][i] * ldW, rowb, bar);
      else { const int b = i - nj; tma_row(sm.sTW + b * FK_LDS, sm.sh.W[sm.sYow[buf][b]] + (size_t)sm.sYloc[buf][b] * ldW, rowb, bar); }
    }
  }
}

// owner side: merged update of the rows of apply-chunk `a` (one warp per item group, members in (rank, position) order)
__device__ void mgs_apply_rows(const ModelDev& md, FastSmemMG& sm, int s, int a, int par, unsigned int T) {
  const ShardDev& sh = sm.sh;
  const int R = sh.R, ldW = sh.ldW, nq = ldW / 4;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int* cbeg = sh.aCbeg + (size_t)s * (sh.NA + 1);
  const int cb = cbeg[a], ce = cbeg[a + 1];
  const int* ent = sh.aEnt + (size_t)s * R * md.NP;
  const int* it = sh.aItem + (size_t)s * R * md.NP;
  const bool ada = md.adapt == G4R_ADAPT_ADAGRAD, mom = md.mom > 0.f;
  const float* inb = sh.inbox[sh.rank] + (size_t)par * R * md.NP * ldW * 2;      // (value, sequence) pairs
  float* W = sh.W[sh.rank];
  for (int j = cb + warp; j < ce; j += FK_NW) {
    const int item = it[j];
    if (j > cb && it[j - 1] == item) continue;
    int je = j + 1;
    while (je < ce && it[je] == item) je++;
    const size_t ro = (size_t)(item / R) * ldW;
    for (int q4 = lane; q4 < nq; q4 += 32) {
      const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      SparseUpd4 u;
      u.begin(ld4(W + ro + q4 * 4), ada ? ld4(sh.W_acc + ro + q4 * 4) : z, mom ? ld4(sh.W_vel + ro + q4 * 4) : z);
      for (int k = j; k < je; k++) {
        const int e = ent[k];
        u.add(md, ll_load4(inb + (((size_t)(e >> 20) * md.NP + (size_t)(e & 0xfffff)) * ldW + q4 * 4) * 2, T, sh.abort), ada, mom);
      }
      st4(W + ro + q4 * 4, u.ps);
      if (ada) st4(sh.W_acc + ro + q4 * 4, u.al);
      if (mom) st4(sh.W_vel + ro + q4 * 4, u.vl);
    }
  }
}
// owner side: merged update of the owned input rows; helper `hb` of `nh` takes the groups that start at j = hb, hb + nh, ...
__device__ void mgs_apply_inputs(const ModelDev& md, FastSmemMG& sm, int s, int hb, int nh, int par, unsigned int T) {
  const ShardDev& sh = sm.sh;
  const LayerDev& ly = md.layer[0];
  const int R = sh.R, ld3 = ly.ld3, B = md.B, tid = threadIdx.x;
  const int xt = sh.xTot[s];
  const int* ent = sh.xEnt + (size_t)s * R * B;
  const int* it = sh.xItem + (size_t)s * R * B;
  const bool ada = md.adapt == G4R_ADAPT_ADAGRAD, mom = md.mom > 0.f;
  const float* inb = sh.inboxIn[sh.rank] + (size_t)par * R * B * ld3 * 2;       // (value, sequence) pairs
  float* Tb = sh.Wx[sh.rank];
  for (int j = hb; j < xt; j += nh) {
    const int item = it[j];
    if (j > 0 && it[j - 1] == item) continue;
    int je = j + 1;
    while (je < xt && it[je] == item) je++;
    const size_t ro = (size_t)(item / R) * ld3;
    for (int q4 = tid; q4 < ld3 / 4; q4 += FK_THREADS) {
      const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      SparseUpd4 u;
      u.begin(ld4(Tb + ro + q4 * 4), ada ? ld4(sh.Wx_acc + ro + q4 * 4) : z, mom ? ld4(sh.Wx_vel + ro + q4 * 4) : z);
      for (int k = j; k < je; k++) {
        const int e = ent[k];
        u.add(md, ll_load4(inb + (((size_t)(e >> 16) * B + (size_t)(e & 0xffff)) * ld3 + q4 * 4) * 2, T, sh.abort), ada, mom);
      }
      st4(Tb + ro + q4 * 4, u.ps);
      if (ada) st4(sh.Wx_acc + ro + q4 * 4, u.al);
      if (mom) st4(sh.Wx_vel + ro + q4 * 4, u.vl);
    }
  }
}
// fetch input row X(s)[b] from its owner into the local buffer the GRU phases read
__device__ __forceinline__ void mgs_gather_input(const ModelDev& md, FastSmemMG& sm, int s, int b) {
  const ShardDev& sh = sm.sh;
  const int ld3 = md.layer[0].ld3;
  if (b >= md.wM[s]) return;
  const int x = md.wX[(size_t)s * md.B + b];
  const float* src = sh.Wx[x % sh.R] + (size_t)(x / sh.R) * ld3;
  for (int q4 = threadIdx.x; q4 < ld3 / 4; q4 += FK_THREADS) st4(sh.mgIn + (size_t)b * ld3 + q4 * 4, ld_volatile4(src + q4 * 4));
}

// owner side, after the input rows of lock step T - 1 are applied: push the rows the ranks need for the NEXT mini-batch (window
// step s1) straight into their buffers -- the owner knows every rank's inputs of the whole window (gathered schedule)
__device__ void mgs_push_inputs(const ModelDev& md, FastSmemMG& sm, int s1, int hb, int nh, unsigned int T1) {
  const ShardDev& sh = sm.sh;
  const int R = sh.R, ld3 = md.layer[0].ld3, B = md.B, tid = threadIdx.x;
  const int par1 = (int)(T1 & 1u);
  const int xt = sh.xTot[s1];
  const int* ent = sh.xEnt + (size_t)s1 * R * B;
  const int* it = sh.xItem + (size_t)s1 * R * B;
  const float* Tb = sh.Wx[sh.rank];
  for (int j = hb; j < xt; j += nh) {
    const int e = ent[j], r = e >> 16, b = e & 0xffff;
    const float* row = Tb + (size_t)(it[j] / R) * ld3;
    float* dst = sh.mgInLL[r] + ((size_t)par1 * B + b) * ld3 * 2;
    for (int q4 = tid; q4 < ld3 / 4; q4 += FK_THREADS) ll_store4(dst + q4 * 8, __ldcg(reinterpret_cast<const float4*>(row + q4 * 4)), T1);
  }
}
// requester side: lane b's input row of lock step T1 arrives in the LL buffer; copy it to the plain buffer the GRU phases read
__device__ __forceinline__ void mgs_receive_input(const ModelDev& md, FastSmemMG& sm, int s1, int b, unsigned int T1) {
  const ShardDev& sh = sm.sh;
  const int ld3 = md.layer[0].ld3;
  if (b >= md.wM[s1]) return;
  const float* src = sh.mgInLL[sh.rank] + ((size_t)(T1 & 1u) * md.B + b) * ld3 * 2;
  for (int q4 = threadIdx.x; q4 < ld3 / 4; q4 += FK_THREADS) st4(sh.mgIn + (size_t)b * ld3 + q4 * 4, ll_load4(src + q4 * 8, T1, sh.abort));
}

// dense gradients of this GRU CTA's slab, summed over the ranks (pushed to every peer, added in rank order), then Adagrad(+momentum)
__device__ void fk_dense_mg(const ModelDev& md, FastSmemMG& sm, int s, int cta, unsigned int T, int par) {
  const ShardDev& sh = sm.sh;
  const LayerDev& ly = md.layer[0];
  const int M = md.wM[s], L = ly.L, ldL = ly.ldL, ld3 = ly.ld3, tid = threadIdx.x;
  const int Rr = (L + FK_G - 1) / FK_G;
  const int k0 = cta * Rr;
  const int nr = max(0, min(Rr, L - k0));
  const int CB = (3 * L + FK_G - 1) / FK_G;
  const int cb0 = cta * CB, ncb = max(0, min(CB, 3 * L - cb0));
  const int nWh = nr * L, nWrz = nr * 2 * L, total = nWh + nWrz + ncb;
  float* sHo = sm.gW;
  float* sHr = sm.gW + 8 * FK_B;
  float* sGd = sm.sD;                        // the column role's dSy scratch is idle during the GRU phases
  const int R = sh.R, me = sh.rank;
  __syncthreads();
  if (total > 0) {
    stage_rows_n<5>(sm.gA, 388, FK_B, ld3 / 4, [&](int rr) -> const float* { return rr < M ? ly.dvec + (size_t)rr * ld3 : nullptr; });
    for (int i = tid; i < nr * FK_B; i += FK_THREADS) {
      const int rr = i / FK_B, b = i % FK_B;
      float ho = 0.f, r = 0.f;
      if (b < M) { ho = ly.Hold[(size_t)b * ldL + k0 + rr]; r = ly.r[(size_t)b * ldL + k0 + rr]; }
      sHo[i] = ho; sHr[i] = ho * r;
    }
  }
  __syncthreads();
  for (int o = tid; o < total; o += FK_THREADS) {
    float g = 0.f;
    if (o < nWh) { const float* av = sHr + (o / L) * FK_B; const float* bv = sm.gA + o % L; for (int b = 0; b < M; b++) g = fmaf(av[b], bv[b * 388], g); }
    else if (o < nWh + nWrz) { const int q = o - nWh; const float* av = sHo + (q / (2 * L)) * FK_B; const float* bv = sm.gA + L + q % (2 * L); for (int b = 0; b < M; b++) g = fmaf(av[b], bv[b * 388], g); }
    else { const float* bv = sm.gA + cb0 + (o - nWh - nWrz); for (int b = 0; b < M; b++) g += bv[b * 388]; }
    sGd[o] = g;
  }
  __syncthreads();
  const int t4 = (total + 3) / 4;
  for (int i = tid; i < (R - 1) * t4; i += FK_THREADS) {
    const int qi = i / t4, q = qi < me ? qi : qi + 1, c4 = i % t4;
    ll_store4(sh.denseIn[q] + (((size_t)(par * R + me) * FK_G + cta) * sh.DSL + c4 * 4) * 2, ld4(sGd + c4 * 4), T);
  }
  const bool ada = md.adapt == G4R_ADAPT_ADAGRAD, mom = md.mom > 0.f;
  const float* din = sh.denseIn[me] + ((size_t)par * R * FK_G * sh.DSL + (size_t)cta * sh.DSL) * 2;
  for (int o = tid; o < total; o += FK_THREADS) {
    // the R - 1 peer slices of this output: all pair loads are issued back to back (independent), then the sequences are checked;
    // only the pairs that have not arrived yet are polled again
    uint2 pr[MGS_MAXR];
    unsigned int pending = 0;
#pragma unroll
    for (int q = 0; q < MGS_MAXR; q++) {
      pr[q] = make_uint2(0u, T);
      if (q < R && q != me) asm volatile("ld.volatile.global.v2.u32 {%0, %1}, [%2];" : "=r"(pr[q].x), "=r"(pr[q].y) : "l"(din + ((size_t)q * FK_G * sh.DSL + o) * 2) : "memory");
    }
#pragma unroll
    for (int q = 0; q < MGS_MAXR; q++) if (q < R && q != me && pr[q].y != T) pending |= 1u << q;
    if (pending) {
#pragma unroll
      for (int q = 0; q < MGS_MAXR; q++)
        if (pending & (1u << q)) pr[q].x = __float_as_uint(ll_load1(din + ((size_t)q * FK_G * sh.DSL + o) * 2, T, sh.abort));
    }
    float g = 0.f;
#pragma unroll
    for (int q = 0; q < MGS_MAXR; q++) if (q < R) g += (q == me) ? sGd[o] : __uint_as_float(pr[q].x);      // rank order: identical on every rank
    float *p, *pa, *pv;
    if (o < nWh) { const size_t off = (size_t)(k0 + o / L) * ldL + o % L; p = ly.Wh + off; pa = ly.Wh_acc ? ly.Wh_acc + off : nullptr; pv = ly.Wh_vel ? ly.Wh_vel + off : nullptr; }
    else if (o < nWh + nWrz) { const int q = o - nWh; const size_t off = (size_t)(k0 + q / (2 * L)) * ly.ld2 + q % (2 * L); p = ly.Wrz + off; pa = ly.Wrz_acc ? ly.Wrz_acc + off : nullptr; pv = ly.Wrz_vel ? ly.Wrz_vel + off : nullptr; }
    else { const int c = cb0 + (o - nWh - nWrz); p = ly.Bh + c; pa = ly.Bh_acc ? ly.Bh_acc + c : nullptr; pv = ly.Bh_vel ? ly.Bh_vel + c : nullptr; }
    const float p0 = *p;
    float gs = g;
    if (ada) gs = adagrad_scale(g, *pa, *pa);
    float v = mom ? *pv : 0.f;
    *p = dense_step(md, gs, p0, v, mom);
    if (mom) *pv = v;
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// the sharded role-specialised kernel: one cooperative launch per window on every rank
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(FK_THREADS, 1) k_fast_mg(int slot, int n_steps, FastSync* fs, FastSyncMG* fm, const ShardDev* shp, unsigned int gbase, unsigned long long* tstamp) {
  extern __shared__ __align__(128) unsigned char fk_raw[];
  FastSmemMG& sm = *reinterpret_cast<FastSmemMG*>(fk_raw);
  const ModelDev& md = MD;
  const LayerDev& ly = md.layer[0];
  const int cta = blockIdx.x, ncta = gridDim.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  {
    const int* src = reinterpret_cast<const int*>(shp);
    int* dst = reinterpret_cast<int*>(&sm.sh);
    for (int i = tid; i < (int)(sizeof(ShardDev) / sizeof(int)); i += FK_THREADS) dst[i] = src[i];
  }
  __syncthreads();
  const ShardDev& sh = sm.sh;
  const int R = sh.R, me = sh.rank, ldW = sh.ldW;
  const int G = FK_G;
  const bool gru = cta < G;
  // the GRU CTAs own no score columns here (md.NCH <= ncta - G chunks start at CTA G): their critical chain b2 -> dense
  // exchange -> f1 -> f2 must not wait for system-scope fences of exported rows
  const int chunk = gru ? md.NCH : cta - G;
  const bool has_chunk = chunk < md.NCH;
  const bool pw = loss_pairwise(md.loss);
  const int L = md.L, ldL = md.ldL, B = md.B;
  (void)L;
  const int kw = ldL / 4;
  const int in_ctas = min(B, ncta - G - R);     // helper CTAs [G, G + in_ctas): input rows
  const int A0 = G + in_ctas;                   // apply CTAs [A0, ncta)
  const int NA = ncta - A0;                     // == sh.NA
  const bool helper = !gru && cta < A0;
  const bool applier = cta >= A0;
  uint64_t* bar = reinterpret_cast<uint64_t*>(&sm.mbar);
  unsigned int bar_epoch = 0, gepoch = 0, stats_target = 0;
  // %globaltimer stamps (16 slots per step): GRU CTA 0 -> 0..6, first helper -> 8..13, first apply CTA -> 14..15
#define MG_STAMP(c_, k) do { if (tstamp && cta == (c_) && tid == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); tstamp[(size_t)s * 16 + (k)] = t_; } } while (0)
  if (tid == 0) { mbar_init(bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  if (!gru) {
    fk_load_idx_mg(md, sm, 0, n_steps, chunk, 0);
    __syncthreads();
    // every owner has applied all lock steps of the previous windows before its rows are read
    mgs_wait_flags(sh, MGF_APPLIED, -1, gbase);
    __syncthreads();
    fk_prefetch_mg(md, sm, 0, n_steps, 0, pw);
  }
  if (helper && n_steps > 0) {
    mgs_wait_flags(sh, MGF_INAPPLIED, -1, gbase);
    __syncthreads();
    mgs_gather_input(md, sm, 0, cta - G);
    __syncthreads();
    if (tid == 0) red_release_add(&fs->in_done, 1u);
  }
  if (gru && n_steps > 0) {
    fk_f1(md, sm, 0, cta, &fs->in_done, (unsigned int)in_ctas, sh.mgIn);
    fk_group_barrier(fs, gepoch);
    fk_f2(md, sm, 0, cta, sh.mgIn);
    __syncthreads();
    if (tid == 0) red_release_add(&fs->h_ready, 1u);
  }
  for (int s = 0; s < n_steps; s++) {
    const int buf = s & 1;
    const int M = md.wM[s];
    const int sti = md.wSti[s];
    const int N = M + (sti >= 0 ? md.S : 0);
    const unsigned int T = gbase + (unsigned int)s + 1u;        // sequence number of this lock step
    const int par = (int)((gbase + (unsigned int)s) & 1u);      // inbox parity
    int cb = 0, nj = 0;
    MG_STAMP(0, 0);
    if (!gru) {
    fk_load_idx_mg(md, sm, s + 1, n_steps, chunk, buf ^ 1);
    // ---- wait for h(s), stage it; the prefetched rows have landed ----
    if (tid == 0) wait_ge(&fs->h_ready, (unsigned int)(s + 1) * (unsigned int)G);
    __syncthreads();
    stage_rows4(sm.sY, FK_LDS, FK_B, kw, [&](int rr) -> const float* { return rr < M ? ly.y + (size_t)rr * ldL : nullptr; });
    mbar_wait(bar, (unsigned int)(s & 1));
    cb = sm.sCb[buf][0];
    nj = sm.sCb[buf][1] - cb;
    if (tid < FK_CT && tid < nj) {                  // bias = By (row tail) - logq correction (gru4rec.py:494-495)
      float bz = sm.sS[tid * FK_LDS + ldL];
      if (md.logq > 0.f) bz -= (sm.sPos[buf][tid] < M) ? md.logP0t[sm.sIt[buf][tid]] : md.logP0s[sm.sIt[buf][tid]];
      sm.sBias[tid] = bz;
    }
    if (tid >= 64 && tid < 64 + FK_B && pw && tid - 64 < M) {
      const int b = tid - 64;
      float bz = sm.sTW[b * FK_LDS + ldL];
      if (md.logq > 0.f) bz -= md.logP0t[sm.sYit[buf][b]];
      sm.sTB[b] = bz;
    }
    __syncthreads();
    // ---- scores + partial statistics (as k_fast) ----
    if (pw) {
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
#pragma unroll
      for (int q = 0; q < FK_Q; q++) {
        const int jj = warp + q * FK_NW;
        if (jj < nj && lane < M) sm.sO[jj * FK_B + lane] = accq[q] + sm.sBias[jj];
      }
      __syncthreads();
      {
        const int b = tid >> 4, sub = tid & 15;
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
        float Z = 0.f, A = 0.f, Q = 0.f, D = 0.f, Tt = 0.f, has = 0.f;
#pragma unroll
        for (int q = 0; q < 2; q++) {
          if (!use[q]) continue;
          const float y = yv[q];
          if (ist[q]) has = 1.f;
          if (xe) { Z += expf(y - mloc); if (ist[q]) Tt = y; }
          else if (md.loss == G4R_LOSS_BPR_MAX) { if (!ist[q]) { const float e = expf(y - mloc), sg = sigmoidf_(t - y); Z += e; A += sg * e; Q += y * y * e; D += sg * (1.f - sg) * e; } }
          else if (md.loss == G4R_LOSS_TOP1_MAX) { if (!ist[q]) { const float e = expf(y - mloc), a1 = sigmoidf_(y - t), b1 = sigmoidf_(y * y); Z += e; A += (a1 + b1) * e; D += a1 * (1.f - a1) * e; } }
          else if (md.loss == G4R_LOSS_BPR) { const float sg = sigmoidf_(t - y); A += -logf(sg); if (!ist[q]) D += 1.f - sg; }
          else { const float a1 = sigmoidf_(y - t), b1 = sigmoidf_(y * y); A += a1 + b1; if (!ist[q]) D += a1 * (1.f - a1); }
        }
#pragma unroll
        for (int o = 1; o < 16; o <<= 1) {
          Z += __shfl_xor_sync(0xffffffffu, Z, o); A += __shfl_xor_sync(0xffffffffu, A, o); Q += __shfl_xor_sync(0xffffffffu, Q, o);
          D += __shfl_xor_sync(0xffffffffu, D, o); Tt += __shfl_xor_sync(0xffffffffu, Tt, o); has += __shfl_xor_sync(0xffffffffu, has, o);
        }
        if (has_chunk && okb && sub == 0) {
          float* st = md.stat + ((size_t)chunk * md.B + b) * G4R_NSTAT;
          st4(st, make_float4(mloc, Z, A, Q));
          st4(st + 4, make_float4(D, Tt, has > 0.f ? 1.f : 0.f, pw ? t : 0.f));
        }
      }
    }
    }   // !gru
    // ---- barrier, then lane b's statistics are combined by CTA b ----
    __syncthreads();
    bar_epoch += 1;
    if (tid == 0) { red_release_add(&fs->bar, 1u); wait_ge(&fs->bar, bar_epoch * (unsigned int)ncta); }
    __syncthreads();
    if (cta < M) {
      const int b = cta;
      const bool maxed = !(md.loss == G4R_LOSS_BPR || md.loss == G4R_LOSS_TOP1);
      float mc = -INFINITY, Z = 0.f, A = 0.f, Q = 0.f, D = 0.f, Tt = 0.f, has = 0.f, tt = 0.f;
      if (tid < md.NCH) {
        const float* st = md.stat + ((size_t)tid * md.B + b) * G4R_NSTAT;
        const float4 u = ld4(st), v = ld4(st + 4);
        mc = u.x; Z = u.y; A = u.z; Q = u.w; D = v.x; Tt = v.y; has = v.z;
        if (tid == 0) tt = v.w;
      }
      float mg = mc;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) mg = fmaxf(mg, __shfl_xor_sync(0xffffffffu, mg, o));
      if (lane == 0) sm.sPart[warp] = mg;
      __syncthreads();
      mg = sm.sPart[0];
      for (int w = 1; w < FK_NW; w++) mg = fmaxf(mg, sm.sPart[w]);
      if (loss_softmaxneg(md.loss)) mg = fmaxf(mg, 0.f);
      if (maxed) {
        const float sc = (mc == -INFINITY) ? 0.f : expf(mc - mg);
        Z *= sc; A *= sc; Q *= sc; D *= sc;
      }
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        Z += __shfl_xor_sync(0xffffffffu, Z, o); A += __shfl_xor_sync(0xffffffffu, A, o); Q += __shfl_xor_sync(0xffffffffu, Q, o);
        D += __shfl_xor_sync(0xffffffffu, D, o); Tt += __shfl_xor_sync(0xffffffffu, Tt, o); has += __shfl_xor_sync(0xffffffffu, has, o);
      }
      __syncthreads();
      if (lane == 0) { float* w = sm.sPart + 32 + warp * 8; w[0] = Z; w[1] = A; w[2] = Q; w[3] = D; w[4] = Tt; w[5] = has; w[6] = tt; }
      __syncthreads();
      if (tid == 0) {
        tt = sm.sPart[32 + 6];
        for (int w = 1; w < FK_NW; w++) { const float* q = sm.sPart + 32 + w * 8; Z += q[0]; A += q[1]; Q += q[2]; D += q[3]; Tt += q[4]; }
        const float m = mg;
        float* rs = md.RS + (size_t)b * G4R_NSTAT;
        float loss = 0.f, r0 = m, r1 = Z, r2 = 0.f, r3 = 0.f, r4 = 0.f, r5 = tt;
        if (md.loss == G4R_LOSS_XE) { const float pt = __fdiv_rn(expf(Tt - m), Z); loss = -logf(pt + G4R_EPS_LOG); r2 = pt; r5 = Tt; }
        else if (md.loss == G4R_LOSS_XE_LOGIT) { loss = logf(Z) - (Tt - m); r5 = Tt; }
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
    if (!gru) {
    if (tid == 0) wait_ge(&fs->stats, stats_target);
    __syncthreads();
    // ---- loss gradient, dSy, partial dL/dh ----
    if (tid < M * 2) st4(sm.sRS + tid * 4, ld4(md.RS + tid * 4));
    __syncthreads();
    if (chunk == 0 && tid == 0) {
      float c = 0.f;
      for (int b = 0; b < M; b++) c += sm.sRS[b * 8 + 6];
      c = __fdiv_rn(c, (float)md.B);
      md.cost[s] = c;
      if (c != c) atomicExch(md.nanflag, 1);
    }
    for (int i = tid; i < FK_CT * FK_B; i += FK_THREADS) {
      const int jj = i / FK_B, b = i % FK_B;
      sm.sG[i] = (jj < nj && b < M) ? loss_grad_elem(md, sm.sRS + (size_t)b * 8, sm.sO[i], sm.sTc[buf][b] == cb + jj, M, N) : 0.f;
    }
    __syncthreads();
    for (int jj = warp; jj < nj; jj += FK_NW) {
      float a = (lane < M) ? sm.sG[jj * FK_B + lane] : 0.f;
      a = warp_sum(a);
      if (lane == 0) sm.sDby[jj] = a;
    }
    float* part = md.part + (size_t)(has_chunk ? chunk : 0) * md.B * ldL;
    if (has_chunk) {
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
    __syncthreads();
    // ---- export: dSy | dby rows go straight into the owners' inboxes (peer stores over NVLink) ----
    for (int t = tid; t < nj * (kw + 1); t += FK_THREADS) {
      const int jj = t / (kw + 1), q4 = t % (kw + 1);
      const float4 v = q4 < kw ? ld4(sm.sD + jj * FK_LDS + q4 * 4) : make_float4(sm.sDby[jj], 0.f, 0.f, 0.f);
      ll_store4(sh.inbox[sm.sOw[buf][jj]] + (((size_t)(par * R + me) * md.NP + (size_t)(cb + jj)) * ldW + q4 * 4) * 2, v, T);
    }
    if (has_chunk && nj == 0) for (int i = tid; i < M * ldL; i += FK_THREADS) part[i] = 0.f;
    }   // !gru
    // ---- barrier: partial dL/dh complete (local visibility only; the peer stores are fenced after b1) ----
    __syncthreads();
    bar_epoch += 1;
    if (tid == 0) { red_release_add(&fs->bar, 1u); wait_ge(&fs->bar, bar_epoch * (unsigned int)ncta); }
    __syncthreads();
    MG_STAMP(0, 1);
    fk_b1<false>(md, sm, s, cta, ncta);
    __syncthreads();
    if (tid == 0) red_release_add(&fs->b1_done, 1u);
    if (gru) {
      if (tid == 0) wait_ge(&fs->b1_done, (unsigned int)(s + 1) * (unsigned int)ncta);
      __syncthreads();
      MG_STAMP(0, 2);
      fk_b2(md, sm, s, cta);
      fk_group_barrier(fs, gepoch);      // epoch 3 s + 2: dvec complete -> the helper CTAs poll this counter
      MG_STAMP(0, 3);
      fk_dense_mg(md, sm, s, cta, T, par);
      fk_group_barrier(fs, gepoch);
      MG_STAMP(0, 4);
      if (s + 1 < n_steps) {
        fk_f1(md, sm, s + 1, cta, &fs->in_done, (unsigned int)(s + 2) * (unsigned int)in_ctas, sh.mgIn);
        fk_group_barrier(fs, gepoch);
        MG_STAMP(0, 5);
        fk_f2(md, sm, s + 1, cta, sh.mgIn);
        __syncthreads();
        if (tid == 0) red_release_add(&fs->h_ready, 1u);
      }
      MG_STAMP(0, 6);
    } else if (helper) {
      const int hb = cta - G;
      // dvec rows of the step are complete when the GRU group has passed its (3 s + 2)-th barrier
      if (tid == 0) wait_ge(&fs->grp, (unsigned int)(3 * s + 2) * FK_G);
      __syncthreads();
      MG_STAMP(G, 8);
      if (hb < M) {
        const int x = md.wX[(size_t)s * B + hb];
        float* dst = sh.inboxIn[x % R] + (((size_t)(par * R + me) * B + hb) * ly.ld3) * 2;
        for (int q4 = tid; q4 < ly.ld3 / 4; q4 += FK_THREADS) ll_store4(dst + q4 * 8, ld4(ly.dvec + (size_t)hb * ly.ld3 + q4 * 4), T);
      }
      MG_STAMP(G, 9);
      mgs_apply_inputs(md, sm, s, hb, in_ctas, par, T);       // polls the (value, sequence) pairs of the rows it needs
      __syncthreads();
      MG_STAMP(G, 10);
      if (tid == 0) { red_release_add(&fm->h2, 1u); wait_ge_abortable(&fm->h2, (unsigned int)(s + 1) * (unsigned int)in_ctas, sh.abort); }
      __syncthreads();
      MG_STAMP(G, 11);
      if (s + 1 < n_steps) {
        mgs_push_inputs(md, sm, s + 1, hb, in_ctas, T + 1u);   // owned rows of the next mini-batch -> their requesters
        MG_STAMP(G, 12);
        mgs_receive_input(md, sm, s + 1, hb, T + 1u);
        __syncthreads();
        if (tid == 0) red_release_add(&fs->in_done, 1u);
        MG_STAMP(G, 13);
      }
      if (hb < R && tid == 0) st_release_sys_u32(sh.flags[hb] + (size_t)(MGF_INAPPLIED + me) * MGS_FLAG_STRIDE, T);   // next window's prologue gathers after this
      mgs_wait_flags(sh, MGF_APPLIED, -1, T);
      __syncthreads();
      fk_prefetch_mg(md, sm, s + 1, n_steps, buf ^ 1, pw);
    } else if (applier) {
      const int a = cta - A0;
      MG_STAMP(A0, 14);
      mgs_apply_rows(md, sm, s, a, par, T);       // polls the (value, sequence) pairs of the gradient rows it needs
      __syncthreads();
      if (tid == 0) red_release_add(&fm->apply_done, 1u);
      MG_STAMP(A0, 15);
      if (a < R && tid == 0) {
        wait_ge_abortable(&fm->apply_done, (unsigned int)(s + 1) * (unsigned int)NA, sh.abort);
        st_release_sys_u32(sh.flags[a] + (size_t)(MGF_APPLIED + me) * MGS_FLAG_STRIDE, T);
      }
      mgs_wait_flags(sh, MGF_APPLIED, -1, T);
      __syncthreads();
      fk_prefetch_mg(md, sm, s + 1, n_steps, buf ^ 1, pw);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// per-window merged plans of the rows this rank owns (model independent; off the critical path)
// ---------------------------------------------------------------------------------------------------------------------
struct MgsPlan {
  int R, rank, NP, B, NA, n_items;
  const int *gKey, *gM, *gX;     // gathered [R][MG_CAP][NP], [R][MG_CAP], [R][MG_CAP][B]
  const int* wSti; int S;
  int *ownLo, *ownHi;            // [MG_CAP][R]
  int *aEnt, *aItem, *aCbeg, *aTot;
  int *xEnt, *xItem, *xTot;
};
__device__ __forceinline__ int mgs_lower_bound(const int* a, int lo, int hi, int key) {   // first index in [lo, hi) with a[i] >= key
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (a[mid] < key) lo = mid + 1; else hi = mid; }
  return lo;
}
__global__ void __launch_bounds__(32) k_mgs_bounds(MgsPlan p, int n_steps) {
  const int s = blockIdx.x, q = threadIdx.x;
  if (s >= n_steps) return;
  const int S = p.wSti[s] >= 0 ? p.S : 0;
  int cnt = 0;
  if (q < p.R) {
    const int* list = p.gKey + ((size_t)q * MG_CAP + s) * p.NP;
    const int Nq = p.gM[q * MG_CAP + s] + S;
    const int lo = mgs_lower_bound(list, 0, Nq, p.rank * p.n_items);
    const int hi = mgs_lower_bound(list, lo, Nq, (p.rank + 1) * p.n_items);
    p.ownLo[s * p.R + q] = lo; p.ownHi[s * p.R + q] = hi;
    cnt = hi - lo;
  }
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if (q == 0) p.aTot[s] = cnt;
}
__global__ void __launch_bounds__(256) k_mgs_plan(MgsPlan p, int n_steps) {
  const int s = blockIdx.y;
  if (s >= n_steps) return;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= p.R * p.NP) return;
  const int r = idx / p.NP, j = idx % p.NP;
  const int lo_r = p.ownLo[s * p.R + r], hi_r = p.ownHi[s * p.R + r];
  if (j < lo_r || j >= hi_r) return;
  const int key = p.gKey[((size_t)r * MG_CAP + s) * p.NP + j];
  int g = j - lo_r;
  for (int q = 0; q < p.R; q++) {
    if (q == r) continue;
    const int* other = p.gKey + ((size_t)q * MG_CAP + s) * p.NP;
    const int lo_q = p.ownLo[s * p.R + q], hi_q = p.ownHi[s * p.R + q];
    // q < r: its equal keys sort before mine (count <= key); q > r: only smaller keys
    g += mgs_lower_bound(other, lo_q, hi_q, q < r ? key + 1 : key) - lo_q;
  }
  const size_t base = (size_t)s * p.R * p.NP;
  p.aEnt[base + g] = (r << 20) | j;
  p.aItem[base + g] = key - p.rank * p.n_items;
}
__global__ void __launch_bounds__(256) k_mgs_plan2(MgsPlan p, int n_steps) {
  extern __shared__ __align__(16) unsigned long long keys[];
  const int s = blockIdx.x;
  if (s >= n_steps) return;
  const int tid = threadIdx.x;
  const int tot = p.aTot[s];
  const int* it = p.aItem + (size_t)s * p.R * p.NP;
  for (int c = tid; c <= p.NA; c += blockDim.x) {
    int j = (int)(((long long)c * tot + p.NA - 1) / p.NA);
    if (c == p.NA) j = tot;
    while (j > 0 && j < tot && it[j] == it[j - 1]) j++;
    p.aCbeg[(size_t)s * (p.NA + 1) + c] = min(j, tot);
  }
  int npow2 = 1;
  while (npow2 < p.R * p.B) npow2 <<= 1;
  __shared__ int s_cnt;
  if (tid == 0) s_cnt = 0;
  __syncthreads();
  for (int i = tid; i < npow2; i += blockDim.x) {
    unsigned long long key = ~0ULL;
    if (i < p.R * p.B) {
      const int r = i / p.B, b = i % p.B;
      if (b < p.gM[r * MG_CAP + s]) {
        const int x = p.gX[((size_t)r * MG_CAP + s) * p.B + b];
        if (x % p.R == p.rank) { key = ((unsigned long long)(unsigned)x << 32) | (unsigned)((r << 16) | b); atomicAdd(&s_cnt, 1); }
      }
    }
    keys[i] = key;
  }
  __syncthreads();
  for (int k = 2; k <= npow2; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < npow2; i += blockDim.x) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const unsigned long long a = keys[i], b = keys[ixj];
          if ((a > b) == ((i & k) == 0)) { keys[i] = b; keys[ixj] = a; }
        }
      }
      __syncthreads();
    }
  const int xt = s_cnt;
  for (int i = tid; i < xt; i += blockDim.x) {
    p.xEnt[(size_t)s * p.R * p.B + i] = (int)(keys[i] & 0xffffffffu);
    p.xItem[(size_t)s * p.R * p.B + i] = (int)(keys[i] >> 32);
  }
  if (tid == 0) p.xTot[s] = xt;
}

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
struct ShardSeg {                       // offsets (bytes) inside the peer-mapped segment; identical on every rank
  size_t W = 0, W_acc = 0, W_vel = 0, Wx = 0, Wx_acc = 0, Wx_vel = 0, inbox = 0, inboxIn = 0, denseIn = 0, mgInLL = 0, flags = 0, total = 0;
  int rows_local = 0, ldW = 0, DSL = 0;
};
struct ShardHost {
  ShardSeg seg;
  char* base = nullptr;                 // this rank's segment (cudaMalloc)
  char* peer[MGS_MAXR] = {};            // mapped bases (own entry = base)
  bool opened = false;
  ShardDev dev; ShardDev* dDev = nullptr;
  FastSyncMG* dSync = nullptr;
  MgsPlan plan;
  unsigned int lock_steps = 0;          // lock steps completed so far (sequence base of the next window)
  int NA = 0;
};

static bool shard_eligible(const g4r_config& c, int n_sm) {
  if (c.world_size < 2 || c.world_size > MGS_MAXR) return false;
  if (c.mg_replicated == 1) return false;                         // caller forces the replicated NCCL path
  if (c.constrained_embedding || c.embedding > 0 || c.n_layers != 1) return false;
  const int L = c.layers[0], B = c.batch_size, R = c.world_size;
  if (round4(L) > 124 || B > FK_B || 2 * L > FK_W1 * FK_G || L > FK_W2 * FK_G) return false;
  if (B < R) return false;                                       // the first R helper CTAs send the input-row flags
  if (n_sm < FK_G + std::min(B, n_sm - FK_G - R) + R) return false;
  if ((long long)c.world_size * c.n_items >= (1ll << 31)) return false;
  if (c.adapt != G4R_ADAPT_ADAGRAD && c.adapt != G4R_ADAPT_NONE) return false;
  if (c.grad_cap > 0.f || c.smoothing > 0.f) return false;
  if (c.step_mode != 2) return false;
  const int gen_len = (c.n_sample > 0 && c.sample_store > 0) ? c.sample_store / c.n_sample : 0;
  const int NP = round4(B + (gen_len > 1 ? c.n_sample : 0));
  const int NCH = std::max(1, std::min(n_sm, (NP + 3) / 4));
  if ((NP + NCH - 1) / NCH > FK_CT) return false;
  return true;
}
static ShardSeg shard_segment(const g4r_config& c) {
  ShardSeg sg;
  const int R = c.world_size, L = c.layers[0], B = c.batch_size;
  const int ldL = round4(L), ld3 = round4(3 * L);
  const bool ada = c.adapt == G4R_ADAPT_ADAGRAD, mom = c.momentum > 0.f;
  const int gen_len = (c.n_sample > 0 && c.sample_store > 0) ? c.sample_store / c.n_sample : 0;
  const int NP = round4(B + (gen_len > 1 ? c.n_sample : 0));
  sg.rows_local = (c.n_items + R - 1) / R;
  sg.ldW = ldL + 4;
  const int Rr = (L + FK_G - 1) / FK_G, CB = (3 * L + FK_G - 1) / FK_G;
  sg.DSL = round4(Rr * 3 * L + CB);
  size_t off = 0;
  auto take = [&](size_t bytes) { off = align_up(off, 256); size_t o = off; off += bytes; return o; };
  const size_t tw = (size_t)sg.rows_local * sg.ldW * 4, tx = (size_t)sg.rows_local * ld3 * 4;
  sg.W = take(tw); sg.W_acc = ada ? take(tw) : 0; sg.W_vel = mom ? take(tw) : 0;
  sg.Wx = take(tx); sg.Wx_acc = ada ? take(tx) : 0; sg.Wx_vel = mom ? take(tx) : 0;
  sg.inbox = take((size_t)2 * R * NP * sg.ldW * 8);          // (value, sequence) pairs
  sg.inboxIn = take((size_t)2 * R * B * ld3 * 8);
  sg.denseIn = take((size_t)2 * R * FK_G * sg.DSL * 8);
  sg.mgInLL = take((size_t)2 * B * ld3 * 8);
  sg.flags = take((size_t)MGF_COUNT * MGS_FLAG_STRIDE * 4);
  sg.total = align_up(off, 256);
  return sg;
}
static ShardHost* shard_of(g4r_handle* h) { return static_cast<ShardHost*>(h->shard); }

static void shard_release(g4r_handle* h) {
  ShardHost* sh = shard_of(h);
  if (!sh) return;
  for (int q = 0; q < MGS_MAXR; q++) if (sh->peer[q] && sh->peer[q] != sh->base) cudaIpcCloseMemHandle(sh->peer[q]);
  if (sh->base) cudaFree(sh->base);
  delete sh;
  h->shard = nullptr;
}

// 64-byte cudaIpcMemHandle_t of this rank's segment
extern "C" int g4r_mg_ipc_handle(g4r_handle* h, char* out64) {
  if (!h || !out64) return G4R_ERR_INVALID;
  ShardHost* sh = shard_of(h);
  if (!sh) FAIL(G4R_ERR_STATE, "handle is not row-sharded");
  cudaSetDevice(h->cfg.device);
  cudaIpcMemHandle_t mh;
  CK(cudaIpcGetMemHandle(&mh, sh->base));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t size");
  memcpy(out64, &mh, 64);
  return G4R_OK;
}
extern "C" int g4r_mg_sharded(const g4r_handle* h) { return (h && h->shard) ? 1 : 0; }

// maps the segments of all ranks (handles in rank order, 64 bytes each) and publishes the peer pointers to the device
extern "C" int g4r_mg_ipc_open(g4r_handle* h, const char* handles, int32_t world) {
  if (!h || !handles) return G4R_ERR_INVALID;
  ShardHost* sh = shard_of(h);
  if (!sh) FAIL(G4R_ERR_STATE, "handle is not row-sharded");
  if (world != h->cfg.world_size) FAIL(G4R_ERR_INVALID, "world size mismatch");
  if (sh->opened) return G4R_OK;
  cudaSetDevice(h->cfg.device);
  const int R = world, me = h->cfg.rank;
  for (int q = 0; q < R; q++) {
    if (q == me) { sh->peer[q] = sh->base; continue; }
    cudaIpcMemHandle_t mh; memcpy(&mh, handles + (size_t)q * 64, 64);
    void* p = nullptr;
    CK(cudaIpcOpenMemHandle(&p, mh, cudaIpcMemLazyEnablePeerAccess));
    sh->peer[q] = (char*)p;
  }
  ShardDev& d = sh->dev;
  for (int q = 0; q < R; q++) {
    d.W[q] = (float*)(sh->peer[q] + sh->seg.W); d.Wx[q] = (float*)(sh->peer[q] + sh->seg.Wx);
    d.inbox[q] = (float*)(sh->peer[q] + sh->seg.inbox); d.inboxIn[q] = (float*)(sh->peer[q] + sh->seg.inboxIn);
    d.denseIn[q] = (float*)(sh->peer[q] + sh->seg.denseIn); d.flags[q] = (unsigned int*)(sh->peer[q] + sh->seg.flags);
    d.mgInLL[q] = (float*)(sh->peer[q] + sh->seg.mgInLL);
  }
  CK(cudaMemcpyAsync(sh->dDev, &d, sizeof(ShardDev), cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  sh->opened = true;
  return G4R_OK;
}

// pure host arithmetic of the ownership map (for tests of the host logic; no device needed)
extern "C" int g4r_mg_owner(int64_t item, int32_t world) { return world > 0 ? (int)(item % world) : 0; }
extern "C" int64_t g4r_mg_local_row(int64_t item, int32_t world) { return world > 0 ? item / world : item; }
extern "C" int64_t g4r_mg_shard_rows(int64_t n_items, int32_t world, int32_t rank) { return world > 0 ? (n_items - rank + world - 1) / world : n_items; }
extern "C" int g4r_mg_segment_bytes(const g4r_config* cfg, size_t* total, size_t* inbox_bytes, size_t* inbox_in_bytes, size_t* dense_bytes) {
  if (!cfg || cfg->world_size < 2 || cfg->n_layers != 1) return G4R_ERR_INVALID;
  const ShardSeg sg = shard_segment(*cfg);
  if (total) *total = sg.total;
  if (inbox_bytes) *inbox_bytes = sg.inboxIn - sg.inbox;
  if (inbox_in_bytes) *inbox_in_bytes = sg.denseIn - sg.inboxIn;
  if (dense_bytes) *dense_bytes = sg.mgInLL - sg.denseIn;
  return G4R_OK;
}

// per-window plan exchange: all-gather of the ranks' sorted column lists (NCCL), merged plan of the rows this rank owns
static int mgs_plan_window(g4r_handle* h, int64_t n) {
  ShardHost* sh = shard_of(h);
  if (!h->mg_host || !static_cast<MgHost*>(h->mg_host)->ready) FAIL(G4R_ERR_STATE, "multi-GPU handle: call g4r_mg_init first");
  MgHost& m = *static_cast<MgHost*>(h->mg_host);
  if (n > MG_CAP) FAIL(G4R_ERR_INVALID, "row-sharded handle: at most MG_CAP steps per window");
  const ModelDev& md = h->md;
  cudaStream_t st = h->stream;
  const int R = sh->dev.R, NP = md.NP, B = md.B;
  const MgDev& mg = m.dev;
  NC(g_nccl.GroupStart());
  NC(g_nccl.AllGather(md.pKey, mg.gItem, (size_t)MG_CAP * NP, ncclInt32, m.comm, st));
  NC(g_nccl.AllGather(md.wM, mg.gM, (size_t)MG_CAP, ncclInt32, m.comm, st));
  NC(g_nccl.AllGather(md.wX, mg.gX, (size_t)MG_CAP * B, ncclInt32, m.comm, st));
  NC(g_nccl.GroupEnd());
  k_mgs_bounds<<<(unsigned)n, 32, 0, st>>>(sh->plan, (int)n);
  k_mgs_plan<<<dim3((R * NP + 255) / 256, (unsigned)n), 256, 0, st>>>(sh->plan, (int)n);
  int npow2 = 1; while (npow2 < R * B) npow2 <<= 1;
  k_mgs_plan2<<<(unsigned)n, 256, (size_t)npow2 * 8, st>>>(sh->plan, (int)n);
  h->launches += 3;
  CK(cudaGetLastError());
  return G4R_OK;
}
// one window of n lock steps (n <= MG_CAP, identical on every rank): ONE cooperative launch per rank
static int mgs_run_window(g4r_handle* h, int64_t n) {
  ShardHost* sh = shard_of(h);
  if (!sh->opened) FAIL(G4R_ERR_STATE, "row-sharded handle: peer segments not mapped (g4r_mg_ipc_open)");
  cudaStream_t st = h->stream;
  CK(cudaMemsetAsync(h->dFastSync, 0, sizeof(FastSync), st));
  CK(cudaMemsetAsync(sh->dSync, 0, sizeof(FastSyncMG), st));
  int slot = h->slot, nst = (int)n; FastSync* fsp = h->dFastSync; FastSyncMG* fmp = sh->dSync; const ShardDev* sdp = sh->dDev; unsigned int gbase = sh->lock_steps;
  unsigned long long* ts = h->stamp_on ? h->dStamp : nullptr;
  void* args[] = {&slot, &nst, &fsp, &fmp, &sdp, &gbase, &ts};
  CK(cudaLaunchCooperativeKernel((void*)k_fast_mg, dim3(h->pk_blocks), dim3(FK_THREADS), args, sizeof(FastSmemMG), st));
  h->launches += 1; h->fast_windows++;
  sh->lock_steps += (unsigned int)n;
  if (h->gen_len > 0) h->sample_ptr += n;
  h->global_step += (uint32_t)n;
  return G4R_OK;
}

// called by g4r_create for a row-sharded configuration: allocates the peer-mappable segment, registers the sharded tensors
static int shard_create(g4r_handle* h) {
  const g4r_config& c = h->cfg;
  ShardHost* sh = new ShardHost();
  h->shard = sh;
  sh->seg = shard_segment(c);
  if (cudaMalloc(&sh->base, sh->seg.total) != cudaSuccess) { h->err = "cudaMalloc of the sharded segment failed"; return G4R_ERR_CUDA; }
  CK(cudaMemsetAsync(sh->base, 0, sh->seg.total, h->stream));
  const ModelDev& md = h->md;
  const int R = c.world_size, B = md.B, L = md.L, ldL = md.ldL, ld3 = md.layer[0].ld3;
  const bool ada = c.adapt == G4R_ADAPT_ADAGRAD, mom = c.momentum > 0.f;
  sh->NA = h->n_sm - FK_G - std::min(B, h->n_sm - FK_G - R);
  // workspace carve-outs
  char* w = (char*)align_up((size_t)h->shard_ws, 256);
  int* ownLo = (int*)w; w += (size_t)MG_CAP * R * sizeof(int);
  int* ownHi = (int*)w; w += (size_t)MG_CAP * R * sizeof(int);
  w = (char*)align_up((size_t)w, 256); sh->dDev = (ShardDev*)w; w += align_up(sizeof(ShardDev), 256);
  sh->dSync = (FastSyncMG*)w; w += align_up(sizeof(FastSyncMG), 256);
  float* mgIn = (float*)w; w += (size_t)B * ld3 * sizeof(float);
  if ((size_t)(w - h->shard_ws) > h->shard_ws_bytes) { h->err = "internal: sharded workspace carve-out too small"; return G4R_ERR_STATE; }
  ShardDev& d = sh->dev;
  memset(&d, 0, sizeof(d));
  d.R = R; d.rank = c.rank; d.rows_local = sh->seg.rows_local; d.ldW = sh->seg.ldW; d.NA = sh->NA; d.DSL = sh->seg.DSL;
  d.W_acc = ada ? (float*)(sh->base + sh->seg.W_acc) : nullptr; d.W_vel = mom ? (float*)(sh->base + sh->seg.W_vel) : nullptr;
  d.Wx_acc = ada ? (float*)(sh->base + sh->seg.Wx_acc) : nullptr; d.Wx_vel = mom ? (float*)(sh->base + sh->seg.Wx_vel) : nullptr;
  d.mgIn = mgIn;
  const MgDev& mg = h->mgdev;
  d.aEnt = mg.mEnt; d.aItem = mg.mItem; d.aCbeg = mg.mCbeg; d.xEnt = mg.xEnt; d.xItem = mg.xItem; d.xTot = mg.xTot; d.gX = mg.gX; d.gM = mg.gM;
  d.abort = md.nanflag + 3;
  MgsPlan& p = sh->plan;
  p.R = R; p.rank = c.rank; p.NP = md.NP; p.B = B; p.NA = sh->NA; p.n_items = c.n_items;
  p.gKey = mg.gItem; p.gM = mg.gM; p.gX = mg.gX; p.wSti = md.wSti; p.S = md.S; p.ownLo = ownLo; p.ownHi = ownHi;
  p.aEnt = mg.mEnt; p.aItem = mg.mItem; p.aCbeg = mg.mCbeg; p.aTot = mg.mTot; p.xEnt = mg.xEnt; p.xItem = mg.xItem; p.xTot = mg.xTot;
  // tensors: logical shapes as on one GPU; rows are scattered over the ranks
  auto reg = [&](const std::string& name, size_t off, int64_t cols, int64_t ld, size_t col0) {
    TensorInfo t; t.ptr = (float*)(sh->base + off) + col0; t.rows = c.n_items; t.cols = cols; t.ld = ld; t.sharded = true; t.seg_off = off + col0 * sizeof(float);
    h->tensors[name] = t;
  };
  reg("Wy", sh->seg.W, L, sh->seg.ldW, 0); reg("By", sh->seg.W, 1, sh->seg.ldW, ldL);
  if (ada) { reg("Wy.acc", sh->seg.W_acc, L, sh->seg.ldW, 0); reg("By.acc", sh->seg.W_acc, 1, sh->seg.ldW, ldL); }
  if (mom) { reg("Wy.vel", sh->seg.W_vel, L, sh->seg.ldW, 0); reg("By.vel", sh->seg.W_vel, 1, sh->seg.ldW, ldL); }
  reg("Wx0", sh->seg.Wx, 3 * L, ld3, 0);
  if (ada) reg("Wx0.acc", sh->seg.Wx_acc, 3 * L, ld3, 0);
  if (mom) reg("Wx0.vel", sh->seg.Wx_vel, 3 * L, ld3, 0);
  if (cudaFuncSetAttribute(k_fast_mg, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FastSmemMG)) != cudaSuccess) { h->err = "k_fast_mg: shared memory opt-in failed"; return G4R_ERR_CUDA; }
  int per_sm = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_fast_mg, FK_THREADS, sizeof(FastSmemMG));
  if (per_sm < 1 || h->pk_blocks <= 0) { h->err = "k_fast_mg cannot be co-resident (cooperative launch / shared memory)"; return G4R_ERR_INVALID; }
  return G4R_OK;
}

// scatter / gather of a sharded tensor between a full host matrix and the ranks' shards
static int shard_set_tensor(g4r_handle* h, const TensorInfo& t, const float* host) {
  const int R = h->cfg.world_size, me = h->cfg.rank;
  const int64_t rows_q = (t.rows - me + R - 1) / R;
  if (rows_q <= 0) return G4R_OK;
  CK(cudaMemcpy2DAsync(t.ptr, t.ld * sizeof(float), host + (size_t)me * t.cols, (size_t)R * t.cols * sizeof(float), t.cols * sizeof(float), rows_q, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return G4R_OK;
}
static int shard_get_tensor(g4r_handle* h, const TensorInfo& t, float* host) {
  ShardHost* sh = shard_of(h);
  if (!sh->opened) FAIL(G4R_ERR_STATE, "row-sharded tensor: peer segments are not mapped yet (g4r_mg_ipc_open)");
  const int R = h->cfg.world_size;
  for (int q = 0; q < R; q++) {
    const int64_t rows_q = (t.rows - q + R - 1) / R;
    if (rows_q <= 0) continue;
    const float* src = (const float*)(sh->peer[q] + t.seg_off);
    CK(cudaMemcpy2DAsync(host + (size_t)q * t.cols, (size_t)R * t.cols * sizeof(float), src, t.ld * sizeof(float), t.cols * sizeof(float), rows_q, cudaMemcpyDeviceToHost, h->stream));
  }
  CK(cudaStreamSynchronize(h->stream));
  return G4R_OK;
}
