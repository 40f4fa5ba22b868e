// g4r_multi.cuh -- synchronous data parallelism over the GPUs of one box (SURVEY section 8e), round-1 design:
//   * every rank runs its own B lanes (its own sessions, its own negative samples) through the single-GPU phases in
//     "export" mode: row gradients (dSy, dby, input-row gradients) and dense gradients are produced, nothing is applied;
//   * NCCL over NVLink: all-gather of the row gradients, all-reduce (sum) of the flat dense-gradient buffer;
//   * every rank then applies the IDENTICAL merged update to its replica of the parameters: the positions of all ranks
//     are treated as one list in (rank, position) order with the single-GPU duplicate rules (Adagrad / momentum state:
//     last occurrence wins; parameter: all occurrences accumulate), so replicas stay bit-identical and the result equals
//     the oracle run on the concatenated mini-batch.
// The merged order is model independent: per window the ranks' sorted column lists are all-gathered once and merged on
// the device by rank arithmetic (k_mg_plan), off the critical path.
// Included from g4r_lib.cu.  Modes: no-embedding and separate-embedding (constrained embedding: next round).
#pragma once
#include <nccl.h>     // types only: the library is resolved at run time (dlopen) so that libg4r.so has no load-time
#include <dlfcn.h>    // dependency on a particular libnccl (PyTorch bundles its own libnccl.so.2)

struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;
static bool nccl_load() {
  if (g_nccl.lib) return true;
  void* l = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);     // already-loaded copy (e.g. PyTorch's) is reused by SONAME
  if (!l) l = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!l) return false;
  g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))dlsym(l, "ncclGetUniqueId");
  g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))dlsym(l, "ncclCommInitRank");
  g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))dlsym(l, "ncclCommDestroy");
  g_nccl.AllGather = (decltype(g_nccl.AllGather))dlsym(l, "ncclAllGather");
  g_nccl.AllReduce = (decltype(g_nccl.AllReduce))dlsym(l, "ncclAllReduce");
  g_nccl.GroupStart = (decltype(g_nccl.GroupStart))dlsym(l, "ncclGroupStart");
  g_nccl.GroupEnd = (decltype(g_nccl.GroupEnd))dlsym(l, "ncclGroupEnd");
  g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))dlsym(l, "ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.CommDestroy || !g_nccl.AllGather || !g_nccl.AllReduce || !g_nccl.GroupStart ||
      !g_nccl.GroupEnd || !g_nccl.GetErrorString) return false;
  g_nccl.lib = l;
  return true;
}


// merged position of every (rank, column): own index + for each other rank the number of its columns that sort before
__global__ void __launch_bounds__(256) k_mg_plan(ModelDev md, MgDev mg, int n_steps) {
  const int s = blockIdx.y;
  if (s >= n_steps) return;
  const int NP = md.NP;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;      // over R * NP
  if (idx >= mg.R * NP) return;
  const int r = idx / NP, j = idx % NP;
  const int S = md.wSti[s] >= 0 ? md.S : 0;                    // same on every rank
  const int Nr = mg.gM[r * MG_CAP + s] + S;
  if (j >= Nr) return;
  const int* mine = mg.gItem + ((size_t)r * MG_CAP + s) * NP;
  const int item = mine[j];
  int g = j;
  for (int q = 0; q < mg.R; q++) {
    if (q == r) continue;
    const int* other = mg.gItem + ((size_t)q * MG_CAP + s) * NP;
    const int Nq = mg.gM[q * MG_CAP + s] + S;
    int lo = 0, hi = Nq;                                       // q < r: count items <= item ; q > r: count items < item
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      const int v = other[mid];
      if (q < r ? (v <= item) : (v < item)) lo = mid + 1; else hi = mid;
    }
    g += lo;
  }
  const size_t base = (size_t)s * mg.R * NP;
  mg.mEnt[base + g] = (r << 20) | j;
  mg.mItem[base + g] = item;
  if (idx == 0) {
    int tot = 0;
    for (int q = 0; q < mg.R; q++) tot += mg.gM[q * MG_CAP + s] + S;
    mg.mTot[s] = tot;
  }
}
// chunk boundaries of the merged list (never split an item group) and the merged, sorted input rows
__global__ void __launch_bounds__(256) k_mg_plan2(ModelDev md, MgDev mg, int n_steps) {
  extern __shared__ __align__(16) unsigned long long keys[];
  const int s = blockIdx.x;
  if (s >= n_steps) return;
  const int tid = threadIdx.x;
  const int NP = md.NP, B = md.B, R = mg.R;
  int tot = 0;
  const int S = md.wSti[s] >= 0 ? md.S : 0;
  for (int q = 0; q < R; q++) tot += mg.gM[q * MG_CAP + s] + S;
  const int* it = mg.mItem + (size_t)s * R * NP;
  for (int c = tid; c <= md.NCH; c += blockDim.x) {
    int j = (int)(((long long)c * tot + md.NCH - 1) / md.NCH);
    if (c == md.NCH) j = tot;
    while (j > 0 && j < tot && it[j] == it[j - 1]) j++;
    mg.mCbeg[(size_t)s * (md.NCH + 1) + c] = min(j, tot);
  }
  // input rows: bitonic sort of (item, rank, lane)
  int npow2 = 1;
  while (npow2 < R * B) npow2 <<= 1;
  int xt = 0;
  for (int i = tid; i < npow2; i += blockDim.x) {
    unsigned long long key = ~0ULL;
    if (i < R * B) {
      const int r = i / B, b = i % B;
      if (b < mg.gM[r * MG_CAP + s]) key = ((unsigned long long)(unsigned)mg.gX[((size_t)r * MG_CAP + s) * B + b] << 32) | (unsigned)((r << 16) | b);
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
  for (int q = 0; q < R; q++) xt += mg.gM[q * MG_CAP + s];
  for (int i = tid; i < xt; i += blockDim.x) {
    mg.xEnt[(size_t)s * R * B + i] = (int)(keys[i] & 0xffffffffu);
    mg.xItem[(size_t)s * R * B + i] = (int)(keys[i] >> 32);
  }
  if (tid == 0) mg.xTot[s] = xt;
}

// one item, members given by entry list: gradient row of member k = gbase + (rank_k * rstride + idx_k) * gld
__device__ __forceinline__ void mg_row_update(const ModelDev& md, float* prow, float* arow, float* vrow, const int* ent, int n, int shift, int mask,
                                              const float* gbase, size_t rstride, int gld, int lane, int ld, bool ada, bool mom) {
  for (int c4 = lane; c4 < ld / 4; c4 += 32) {
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    SparseUpd4 u;
    u.begin(ld4(prow + c4 * 4), ada ? ld4(arow + c4 * 4) : z, mom ? ld4(vrow + c4 * 4) : z);
    for (int k = 0; k < n; k++) {
      const int e = ent[k];
      u.add(md, ld4(gbase + ((size_t)(e >> shift) * rstride + (size_t)(e & mask)) * gld + c4 * 4), ada, mom);
    }
    st4(prow + c4 * 4, u.ps);
    if (ada) st4(arow + c4 * 4, u.al);
    if (mom) st4(vrow + c4 * 4, u.vl);
  }
}

// merged sparse update of Wy / By for the chunk of the merged column list owned by this CTA
__global__ void __launch_bounds__(256) k_mg_apply_rows(int slot, MgDev mg, const int* base, int off) {
  const ModelDev& md = MD;
  const int s = STEP_IDX;
  const int* cbeg = mg.mCbeg + (size_t)s * (md.NCH + 1);
  const int cb = cbeg[blockIdx.x], ce = cbeg[blockIdx.x + 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int* ent = mg.mEnt + (size_t)s * mg.R * md.NP;
  const int* it = mg.mItem + (size_t)s * mg.R * md.NP;
  const bool ada = md.adapt == G4R_ADAPT_ADAGRAD, mom = md.mom > 0.f;
  for (int j = cb + warp; j < ce; j += blockDim.x >> 5) {
    const int item = it[j];
    if (j > cb && it[j - 1] == item) continue;
    int je = j + 1;
    while (je < ce && it[je] == item) je++;
    mg_row_update(md, md.Wy + (size_t)item * md.ldL, md.Wy_acc ? md.Wy_acc + (size_t)item * md.ldL : nullptr, md.Wy_vel ? md.Wy_vel + (size_t)item * md.ldL : nullptr,
                  ent + j, je - j, 20, 0xfffff, mg.DSYall, (size_t)md.NP, md.ldL, lane, md.ldL, ada, mom);
    if (lane == 0) {
      SparseUpd u;
      u.begin(md.By[item], ada ? md.By_acc[item] : 0.f, mom ? md.By_vel[item] : 0.f);
      for (int k = j; k < je; k++) {
        const int e = ent[k];
        u.add(md, mg.DBYall[(size_t)(e >> 20) * md.NP + (e & 0xfffff)], ada, mom);
      }
      md.By[item] = u.ps;
      if (ada) md.By_acc[item] = u.al;
      if (mom) md.By_vel[item] = u.vl;
    }
  }
}
// merged sparse update of the gathered input rows (Wx0 in no-embedding mode, E in embedding mode): one CTA per group
__global__ void __launch_bounds__(128) k_mg_apply_in(int slot, MgDev mg, const int* base, int off) {
  const ModelDev& md = MD;
  const int s = STEP_IDX;
  const int tot = mg.xTot[s];
  const int j = blockIdx.x;
  if (j >= tot) return;
  const int* it = mg.xItem + (size_t)s * mg.R * md.B;
  const int item = it[j];
  if (j > 0 && it[j - 1] == item) return;
  int je = j + 1;
  while (je < tot && it[je] == item) je++;
  const int* ent = mg.xEnt + (size_t)s * mg.R * md.B;
  float *tab, *tacc, *tvel; int ld;
  if (md.mode == 0) { const LayerDev& l0 = md.layer[0]; tab = l0.Wx; tacc = l0.Wx_acc; tvel = l0.Wx_vel; ld = l0.ld3; }
  else { tab = md.E; tacc = md.E_acc; tvel = md.E_vel; ld = md.ld_in0; }
  const bool ada = md.adapt == G4R_ADAPT_ADAGRAD, mom = md.mom > 0.f;
  const int lane = threadIdx.x;        // all 128 threads stride over the 16-byte columns of the row
  for (int c4 = lane; c4 < ld / 4; c4 += 128) {
    float* prow = tab + (size_t)item * ld;
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    SparseUpd4 u;
    u.begin(ld4(prow + c4 * 4), ada ? ld4(tacc + (size_t)item * ld + c4 * 4) : z, mom ? ld4(tvel + (size_t)item * ld + c4 * 4) : z);
    for (int k = j; k < je; k++) {
      const int e = ent[k];
      u.add(md, ld4(mg.INall + ((size_t)(e >> 16) * md.B + (size_t)(e & 0xffff)) * ld + c4 * 4), ada, mom);
    }
    st4(prow + c4 * 4, u.ps);
    if (ada) st4(tacc + (size_t)item * ld + c4 * 4, u.al);
    if (mom) st4(tvel + (size_t)item * ld + c4 * 4, u.vl);
  }
}

struct MgHost {
  ncclComm_t comm = nullptr;
  MgDev dev;
  bool ready = false;
  cudaGraphExec_t graphU = nullptr, graph1 = nullptr; int64_t launches_per_step = 0;
};

#define NC(call) do { ncclResult_t r_ = (call); if (r_ != ncclSuccess) { h->err = std::string(#call) + ": " + g_nccl.GetErrorString(r_); return G4R_ERR_CUDA; } } while (0)

extern "C" int g4r_mg_unique_id(char* out128) {
  if (!nccl_load()) return G4R_ERR_STATE;
  ncclUniqueId id;
  if (g_nccl.GetUniqueId(&id) != ncclSuccess) return G4R_ERR_CUDA;
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
  memcpy(out128, &id, 128);
  return G4R_OK;
}

extern "C" int g4r_mg_init(g4r_handle* h, const char* id128) {
  if (!h || !id128) return G4R_ERR_INVALID;
  const int R = h->cfg.world_size, rank = h->cfg.rank;
  if (R < 2) FAIL(G4R_ERR_INVALID, "world_size < 2");
  if (h->md.mode == 2) FAIL(G4R_ERR_INVALID, "multi-GPU with constrained_embedding is not implemented yet");
  if (!h->mg_alloc) FAIL(G4R_ERR_STATE, "handle was created without multi-GPU buffers");
  if (!nccl_load()) FAIL(G4R_ERR_STATE, "libnccl.so.2 could not be loaded");
  cudaSetDevice(h->cfg.device);
  if (!h->mg_host) h->mg_host = new MgHost();
  MgHost& m = *static_cast<MgHost*>(h->mg_host);
  ncclUniqueId id; memcpy(&id, id128, 128);
  NC(g_nccl.CommInitRank(&m.comm, R, id, rank));
  m.dev = h->mgdev;
  m.ready = true;
  if (!h->shard) h->md.export_only = 1;      // replicated path: gradients only, merged update after the NCCL exchange
  CK(slot_upload(h->slot, h->md, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return G4R_OK;
}
static void mg_release(g4r_handle* h) {
  if (!h->mg_host) return;
  MgHost* m = static_cast<MgHost*>(h->mg_host);
  if (m->graphU) cudaGraphExecDestroy(m->graphU);
  if (m->graph1) cudaGraphExecDestroy(m->graph1);
  if (m->comm) g_nccl.CommDestroy(m->comm);
  delete m;
  h->mg_host = nullptr;
}

// one window of n steps (n <= MG_CAP; identical n on every rank)
static int mg_run_window(g4r_handle* h, int64_t n) {
  MgHost& m = *static_cast<MgHost*>(h->mg_host);
  const ModelDev& md = h->md;
  const MgDev& mg = m.dev;
  cudaStream_t st = h->stream;
  const int R = mg.R, NP = md.NP, B = md.B;
  // window metadata of all ranks (model independent): sorted columns, batch sizes, inputs
  NC(g_nccl.GroupStart());
  NC(g_nccl.AllGather(md.pItem, mg.gItem, (size_t)MG_CAP * NP, ncclInt32, m.comm, st));
  NC(g_nccl.AllGather(md.wM, mg.gM, (size_t)MG_CAP, ncclInt32, m.comm, st));
  NC(g_nccl.AllGather(md.wX, mg.gX, (size_t)MG_CAP * B, ncclInt32, m.comm, st));
  NC(g_nccl.GroupEnd());
  k_mg_plan<<<dim3((R * NP + 255) / 256, (unsigned)n), 256, 0, st>>>(md, mg, (int)n);
  int npow2 = 1; while (npow2 < R * B) npow2 <<= 1;
  k_mg_plan2<<<(unsigned)n, 256, (size_t)npow2 * 8, st>>>(md, mg, (int)n);
  h->launches += 2;
  CK(cudaGetLastError());
  const LayerDev& l0 = md.layer[0];
  const float* in_local = md.mode == 0 ? l0.dvec : md.dSx;
  const int in_ld = md.mode == 0 ? l0.ld3 : md.ld_in0;
  const std::vector<MgTensor>& tens = h->mg_tensors;
  // one lock-step mini-batch: local gradients -> NCCL exchange -> merged update (window-relative step = *base + off)
  auto enqueue = [&](const int* base, int off) -> int {
    enqueue_train_step(h, base, off);                     // export mode: gradients only
    NC(g_nccl.GroupStart());
    NC(g_nccl.AllGather(md.DSY, mg.DSYall, (size_t)NP * md.ldL, ncclFloat32, m.comm, st));
    NC(g_nccl.AllGather(md.DBY, mg.DBYall, (size_t)NP, ncclFloat32, m.comm, st));
    NC(g_nccl.AllGather(in_local, mg.INall, (size_t)B * in_ld, ncclFloat32, m.comm, st));
    NC(g_nccl.AllReduce(mg.gradFlat, mg.gradFlat, mg.gradCount, ncclFloat32, ncclSum, m.comm, st));
    NC(g_nccl.GroupEnd());
    k_mg_apply_rows<<<md.NCH, 256, 0, st>>>(h->slot, mg, base, off);
    k_mg_apply_in<<<R * B, 128, 0, st>>>(h->slot, mg, base, off);
    for (const MgTensor& t : tens) k_apply_dense<<<(t.count + 255) / 256, 256, 0, st>>>(h->slot, t.p, t.acc, t.vel, mg.gradFlat + t.goff, t.count);
    h->launches += 2 + (int64_t)tens.size();
    return G4R_OK;
  };
  constexpr int MG_UNROLL = 8;
  if (!m.graphU) {      // capture kernels + collectives of MG_UNROLL steps (and of one step) once; replay per window
    for (int pass = 0; pass < 2; pass++) {
      const int unroll = pass == 0 ? MG_UNROLL : 1;
      cudaGraph_t g = nullptr;
      const int64_t l0c = h->launches;
      CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
      for (int i = 0; i < unroll; i++) { int rc = enqueue(h->dStepBase, i); if (rc) { cudaStreamEndCapture(st, &g); return rc; } }
      k_advance<<<1, 32, 0, st>>>(h->dStepBase, unroll);
      CK(cudaStreamEndCapture(st, &g));
      CK(cudaGraphInstantiate(pass == 0 ? &m.graphU : &m.graph1, g, 0));
      cudaGraphDestroy(g);
      m.launches_per_step = (h->launches - l0c) / unroll;
      h->launches = l0c;
    }
  }
  CK(cudaMemsetAsync(h->dStepBase, 0, sizeof(int), st));
  int64_t i = 0;
  for (; i + MG_UNROLL <= n; i += MG_UNROLL) CK(cudaGraphLaunch(m.graphU, st));
  for (; i < n; i++) CK(cudaGraphLaunch(m.graph1, st));
  h->launches += n * m.launches_per_step;
  CK(cudaGetLastError());
  if (h->gen_len > 0) h->sample_ptr += n;
  h->global_step += (uint32_t)n;
  return G4R_OK;
}
