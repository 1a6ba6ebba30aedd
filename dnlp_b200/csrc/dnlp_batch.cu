// Batched (multi-start) engine behind the C-ABI: the same tape evaluated at B points in lock step.
// See include/dnlp_b200.h (dnlp_batch_*) and dnlp_batch_kernels.cuh.
#include "../../include/dnlp_b200.h"
#include "dnlp_batch_kernels.cuh"
#include "dnlp_batch_kkt.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <string>
#include <vector>

namespace {
thread_local std::string g_batch_create_error;

#define CKB(call)                                                                          \
  do {                                                                                     \
    cudaError_t e_ = (call);                                                               \
    if (e_ != cudaSuccess) {                                                               \
      char buf_[512];                                                                      \
      snprintf(buf_, sizeof buf_, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__,      \
               cudaGetErrorString(e_));                                                    \
      err = buf_;                                                                          \
      return 1;                                                                            \
    }                                                                                      \
  } while (0)

struct BInstr {
  dnlp_instr_desc d;
  bool has_f2 = false;
  int gemm_group = -1;               // index into dnlp_batch::groups when this GEMV runs in a grouped launch
  dnlp::GemmDesc *one_desc = nullptr;   // device descriptor for launching this GEMV on its own
  int32_t *smallk_slots = nullptr;   // device: the K slots every row combines (tall-skinny GEMM path)
};
}  // namespace

struct dnlp_batch {
  int device = 0, sm_count = 148, B = 0;
  int64_t n = 0, m = 0, nslots = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  double *V = nullptr;                   // nslots x B, batch fastest
  double *out[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};      // len x B, batch fastest
  double *out_const[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  int64_t out_len[6] = {0, 0, 0, 0, 0, 0};
  double *stage = nullptr;               // staging for layout changes (max(len) x B)
  int64_t stage_len = 0;
  std::vector<BInstr> instrs;
  // independent dense maps of identical shape (the k+1 quad forms of a QCQP) launched as one grid
  struct GemmGroup { std::vector<int32_t> members; dnlp::GemmDesc *descs = nullptr; int64_t M = 0, K = 0; };
  std::vector<GemmGroup> groups;
  std::vector<int32_t> prog[DNLP_NPROG];
  std::vector<void *> owned;
  int64_t launches = 0;
  std::string err;
  // dense KKT systems of the lock-step interior-point driver (dnlp_batch_kkt_*); slot b of every array is start b
  struct Kkt {
    int64_t N = 0, M = 0, ntgt = 0, nnzH = 0;
    int32_t *ti = nullptr, *tj = nullptr, *sp = nullptr, *src = nullptr;   // targets and their sources, pattern order
    double *K = nullptr, *Dg = nullptr, *Wd = nullptr, *work = nullptr;
    double *sigma = nullptr, *dw = nullptr, *dc = nullptr, *rhs = nullptr, *sol = nullptr, *wq = nullptr;
    int32_t *starts = nullptr, *inertia = nullptr;
    std::vector<void *> owned;
  } kkt;
  void kkt_free() {
    for (void *p : kkt.owned) cudaFree(p);
    kkt = Kkt();
  }

  template <typename T>
  int upload(const T *host, int64_t count, T **dev) {
    *dev = nullptr;
    if (count <= 0 || host == nullptr) return 0;
    void *p = nullptr;
    CKB(cudaMalloc(&p, (size_t)count * sizeof(T)));
    owned.push_back(p);
    CKB(cudaMemcpy(p, host, (size_t)count * sizeof(T), cudaMemcpyHostToDevice));
    *dev = static_cast<T *>(p);
    return 0;
  }
  int grid_for(int64_t items) const {
    int64_t need = (items + 255) / 256, cap = (int64_t)sm_count * 8;
    return (int)(need < 1 ? 1 : (need > cap ? cap : need));
  }
  // the launch sequence of every program mask, captured once and replayed as one CUDA graph: a slice of
  // 512 starts per GPU spends as long launching its ~25 short kernels as running them otherwise
  struct MaskGraph { cudaGraphExec_t exec = nullptr; int64_t nlaunch = 0; };
  MaskGraph graphs[64];
  bool graphs_enabled = true;
  bool dmma_k8 = false;          // m16n8k8 DMMA shape instead of m8n8k4 (A/B: DNLP_DMMA_K8)
  double *split_scratch = nullptr;         // partial sums of the term-split long-row kernel
  unsigned int *split_tickets = nullptr;
  int64_t split_scratch_len = 0, split_ticket_len = 0;
  int launch(const BInstr &I);
  int run_program(int p);
  int run_union(int32_t prog_mask);
  int issue_union(int32_t prog_mask);
  int reset_outputs();
  int put(const double *host, double *dev_batch_major, int64_t len);
  int get(int space, double *host);
};

namespace {
using namespace dnlp;

template <int F, bool Bn>
void launch_belem_t(const dnlp_batch *o, const dnlp_instr_desc &d, int grid) {
  belem_kernel<F, Bn><<<grid, 256, 0, o->stream>>>(o->V, d.a_off, d.a_stride, d.b_off, d.b_stride, d.dst_off,
                                                  d.count, d.param, o->B, d.dst_stride > 0 ? d.dst_stride : 1, d.post_scale);
}
bool launch_belem(const dnlp_batch *o, const dnlp_instr_desc &d, int grid) {
  switch (d.fcode) {
#define U(F) case F: launch_belem_t<F, false>(o, d, grid); return true;
#define Bn(F) case F: launch_belem_t<F, true>(o, d, grid); return true;
    U(F_EXP) U(F_LOG) U(F_ENTR) U(F_NEG_LOG_M1) U(F_RECIP) U(F_NEG_RECIP) U(F_NEG_RECIP_SQ)
    U(F_LOGISTIC) U(F_LOGISTIC_D1) U(F_LOGISTIC_D2) U(F_POW)
    U(F_SIN) U(F_COS) U(F_NEG_SIN) U(F_NEG_COS) U(F_TAN) U(F_TAN_D1) U(F_TAN_D2)
    U(F_SINH) U(F_COSH) U(F_TANH) U(F_TANH_D1) U(F_TANH_D2)
    U(F_ASINH) U(F_ASINH_D1) U(F_ASINH_D2) U(F_ATANH) U(F_ATANH_D1) U(F_ATANH_D2)
    U(F_XEXP) U(F_XEXP_D1) U(F_XEXP_D2)
    Bn(F_REL_ENTR) Bn(F_LOG_RATIO_P1) Bn(F_DIV) Bn(F_DIV_SQ) Bn(F_DIV_CUBE)
#undef U
#undef Bn
    default: return false;
  }
}
}  // namespace

int dnlp_batch::launch(const BInstr &I) {
  const dnlp_instr_desc &d = I.d;
  if (d.count <= 0) return 0;
  double *dst = (d.dst_space == DNLP_DST_V) ? V + d.dst_off * B : out[d.dst_space] + d.dst_off * B;
  switch (d.kind) {
    case DNLP_ELEM:
      if (!launch_belem(this, d, grid_for(d.count * B))) { err = "unknown elementwise function code"; return 1; }
      break;
    case DNLP_POLY: {
      if (I.smallk_slots) {
        const int threads = B >= 256 ? 256 : ((B + 31) / 32) * 32;
        // starts per thread: every register slot must carry a real start (a slice of 512 starts per GPU
        // ran the 4-slot build half empty: 0.170 ms instead of the 0.09 ms its 0.54 GB of output needs)
        const int nb = B > 2 * threads ? 4 : (B > threads ? 2 : 1);
        const int bchunks = (B + threads * nb - 1) / (threads * nb);
        int64_t want_blocks = (int64_t)sm_count * 8;
        int64_t rblocks = want_blocks / bchunks > 0 ? want_blocks / bchunks : 1;
        int rows_per_block = (int)((d.count + rblocks - 1) / rblocks);
        if (rows_per_block < 1) rows_per_block = 1;
        const int64_t blocks = ((d.count + rows_per_block - 1) / rows_per_block) * bchunks;
#define SKN(Lc, Nb) bsmallk_kernel<Lc, Nb><<<(int)blocks, threads, 0, stream>>>(                      \
            V, dst, d.coef, I.smallk_slots, d.pos, d.count, d.accumulate, B, rows_per_block)
#define SK(Lc) case Lc: if (nb == 4) SKN(Lc, 4); else if (nb == 2) SKN(Lc, 2); else SKN(Lc, 1); break;
        switch (d.row_len) {
          SK(2) SK(3) SK(4) SK(5) SK(6) SK(7) SK(8) SK(9) SK(10) SK(11) SK(12) SK(13) SK(14) SK(15) SK(16)
          default: err = "small-K kernel: unsupported row length"; return 1;
        }
#undef SK
#undef SKN
        break;
      }
      if (d.count > 0 && d.nterms / d.count >= 128) {
        const int64_t blocks = d.count * ((B + 31) / 32);
        // very few (row, start-chunk) pairs: the terms of a row are split over KS CTAs as well
        const int64_t mean_terms = d.nterms / d.count;
        int KS = (int)((int64_t)sm_count * 2 / (blocks > 0 ? blocks : 1));
        if (KS > mean_terms / 32) KS = (int)(mean_terms / 32);
        if (KS > 32) KS = 32;
        if (KS >= 2 && (int64_t)KS * d.count * B <= split_scratch_len && blocks <= split_ticket_len) {
          if (I.has_f2)
            bpoly_long_split_kernel<true, 8><<<(int)(blocks * KS), 256, 0, stream>>>(V, dst, d.ptr, d.row_len, d.coef, d.f1, d.f2, d.pos, d.count, d.accumulate, B, KS, split_scratch, split_tickets);
          else
            bpoly_long_split_kernel<false, 8><<<(int)(blocks * KS), 256, 0, stream>>>(V, dst, d.ptr, d.row_len, d.coef, d.f1, d.f2, d.pos, d.count, d.accumulate, B, KS, split_scratch, split_tickets);
          break;
        }
        // few (row, start-chunk) pairs: 16 warps split the terms; enough of them to fill the machine: 8
        if (blocks <= (int64_t)sm_count * 2) {
          if (I.has_f2)
            bpoly_long_kernel<true, 16><<<(int)blocks, 512, 0, stream>>>(V, dst, d.ptr, d.row_len, d.coef, d.f1, d.f2, d.pos, d.count, d.accumulate, B);
          else
            bpoly_long_kernel<false, 16><<<(int)blocks, 512, 0, stream>>>(V, dst, d.ptr, d.row_len, d.coef, d.f1, d.f2, d.pos, d.count, d.accumulate, B);
        } else {
          const int64_t cap = (int64_t)sm_count * 8;
          const int grid = (int)(blocks < cap ? blocks : cap);
          if (I.has_f2)
            bpoly_long_kernel<true, 8><<<grid, 256, 0, stream>>>(V, dst, d.ptr, d.row_len, d.coef, d.f1, d.f2, d.pos, d.count, d.accumulate, B);
          else
            bpoly_long_kernel<false, 8><<<grid, 256, 0, stream>>>(V, dst, d.ptr, d.row_len, d.coef, d.f1, d.f2, d.pos, d.count, d.accumulate, B);
        }
        break;
      }
      const int threads = B >= 256 ? 256 : ((B + 31) / 32) * 32;
      const int bchunks = (B + threads - 1) / threads;
      int64_t blocks = d.count * bchunks, cap = (int64_t)sm_count * 16;
      int grid = (int)(blocks < cap ? blocks : cap);
      if (I.has_f2)
        bpoly_kernel<true><<<grid, threads, 0, stream>>>(V, dst, d.ptr, d.row_len, d.coef, d.f1, d.f2, d.pos, d.count, d.accumulate, B);
      else
        bpoly_kernel<false><<<grid, threads, 0, stream>>>(V, dst, d.ptr, d.row_len, d.coef, d.f1, d.f2, d.pos, d.count, d.accumulate, B);
      break;
    }
    case DNLP_GEMV: {
      // (a GEMV that belongs to a group never reaches here: run_union launches the group once)
      const int tiles = (int)(((d.count + GM - 1) / GM) * ((B + GN - 1) / GN));
      const int cap = sm_count * 4;
      if (dmma_k8)
        bgemm_dmma_kernel<true><<<tiles < cap ? tiles : cap, 128, BGEMM_SMEM, stream>>>(I.one_desc, 1, (int)d.count, B, (int)d.ncols);
      else
        bgemm_dmma_kernel<false><<<tiles < cap ? tiles : cap, 128, BGEMM_SMEM, stream>>>(I.one_desc, 1, (int)d.count, B, (int)d.ncols);
      break;
    }
    case DNLP_SCALE:
      bscale_kernel<<<grid_for(d.count * B), 256, 0, stream>>>(V, d.s_slot, d.coef, dst, d.pos, d.count, d.accumulate, B);
      break;
    default:
      err = "unknown instruction kind";
      return 1;
  }
  ++launches;
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) { err = std::string("kernel launch failed: ") + cudaGetErrorString(e); return 1; }
  return 0;
}

int dnlp_batch::run_program(int p) {
  for (int32_t id : prog[p]) if (launch(instrs[id])) return 1;
  return 0;
}

int dnlp_batch::run_union(int32_t prog_mask) {
  prog_mask &= 63;
  if (!graphs_enabled) return issue_union(prog_mask);
  MaskGraph &G = graphs[prog_mask];
  if (!G.exec) {
    const int64_t before = launches;
    CKB(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
    const int rc = issue_union(prog_mask);
    cudaGraph_t g = nullptr;
    cudaError_t ce = cudaStreamEndCapture(stream, &g);
    if (rc) { if (g) cudaGraphDestroy(g); cudaGetLastError(); return 1; }
    if (ce != cudaSuccess) { err = std::string("graph capture failed: ") + cudaGetErrorString(ce); return 1; }
    G.nlaunch = launches - before;
    launches = before;
    CKB(cudaGraphInstantiate(&G.exec, g, 0));
    cudaGraphDestroy(g);
  }
  CKB(cudaGraphLaunch(G.exec, stream));
  launches += G.nlaunch;
  return 0;
}

int dnlp_batch::issue_union(int32_t prog_mask) {
  // there is no per-x cache in batch mode: run every needed instruction exactly once
  std::vector<uint8_t> need(instrs.size(), 0);
  for (int p = 0; p < DNLP_NPROG; ++p)
    if (prog_mask & (1 << p))
      for (int32_t id : prog[p]) need[id] = 1;
  std::vector<uint8_t> group_done(groups.size(), 0);
  for (size_t id = 0; id < instrs.size(); ++id) {     // ids are in topological order
    if (!need[id]) continue;
    const int gi = instrs[id].gemm_group;
    if (gi >= 0) {
      if (group_done[gi]) continue;
      // all members read only x: running the not-needed ones as well is harmless and keeps one launch
      GemmGroup &G = groups[gi];
      const int64_t tiles = ((G.M + GM - 1) / GM) * ((B + GN - 1) / GN) * (int64_t)G.members.size();
      const int64_t cap = (int64_t)sm_count * 4;
      if (dmma_k8)
        bgemm_dmma_kernel<true><<<(int)(tiles < cap ? tiles : cap), 128, BGEMM_SMEM, stream>>>(
            G.descs, (int)G.members.size(), (int)G.M, B, (int)G.K);
      else
        bgemm_dmma_kernel<false><<<(int)(tiles < cap ? tiles : cap), 128, BGEMM_SMEM, stream>>>(
            G.descs, (int)G.members.size(), (int)G.M, B, (int)G.K);
      ++launches;
      cudaError_t e = cudaPeekAtLastError();
      if (e != cudaSuccess) { err = std::string("kernel launch failed: ") + cudaGetErrorString(e); return 1; }
      group_done[gi] = 1;
      continue;
    }
    if (launch(instrs[id])) return 1;
  }
  return 0;
}

int dnlp_batch::put(const double *host, double *dev, int64_t len) {
  if (len <= 0) return 0;
  CKB(cudaMemcpyAsync(stage, host, (size_t)len * B * sizeof(double), cudaMemcpyHostToDevice, stream));
  const int64_t tiles = ((len + 31) / 32) * ((B + 31) / 32);
  to_batch_major_kernel<<<(int)(tiles < sm_count * 8 ? tiles : sm_count * 8), 256, 0, stream>>>(stage, dev, len, B);
  ++launches;
  return 0;
}

int dnlp_batch::get(int space, double *host) {
  const int64_t len = out_len[space];
  if (host == nullptr || len <= 0) return 0;
  const int64_t tiles = ((len + 31) / 32) * ((B + 31) / 32);
  from_batch_major_kernel<<<(int)(tiles < sm_count * 8 ? tiles : sm_count * 8), 256, 0, stream>>>(out[space], stage, len, B);
  ++launches;
  CKB(cudaMemcpyAsync(host, stage, (size_t)len * B * sizeof(double), cudaMemcpyDeviceToHost, stream));
  return 0;
}

extern "C" {

void dnlp_batch_destroy(dnlp_batch *o) {
  if (!o) return;
  cudaSetDevice(o->device);
  if (o->stream) cudaStreamSynchronize(o->stream);
  for (auto &g : o->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
  o->kkt_free();
  for (void *p : o->owned) cudaFree(p);
  if (o->ev0) cudaEventDestroy(o->ev0);
  if (o->ev1) cudaEventDestroy(o->ev1);
  if (o->stream) cudaStreamDestroy(o->stream);
  delete o;
}

static int batch_create_impl(dnlp_batch *o, const dnlp_tape_desc *t) {
  if (o == nullptr) { g_batch_create_error = "batch handle is NULL (closed or never created)"; return 1; }
  std::string &err = o->err;
  CKB(cudaSetDevice(o->device));
  cudaDeviceProp prop;
  CKB(cudaGetDeviceProperties(&prop, o->device));
  o->sm_count = prop.multiProcessorCount;
  CKB(cudaStreamCreateWithFlags(&o->stream, cudaStreamNonBlocking));
  CKB(cudaEventCreate(&o->ev0));
  CKB(cudaEventCreate(&o->ev1));
  o->n = t->n; o->m = t->m; o->nslots = t->nslots;
  const int B = o->B;
  void *p = nullptr;
  CKB(cudaMalloc(&p, (size_t)(t->nslots + 2) * B * sizeof(double)));
  o->owned.push_back(p);
  o->V = static_cast<double *>(p);
  CKB(cudaMemset(o->V, 0, (size_t)(t->nslots + 2) * B * sizeof(double)));
  if (t->n_params > 0 && t->params) {          // every start sees the same parameter values
    double *pd = nullptr;
    if (o->upload(t->params, t->n_params, &pd)) return 1;
    bfill_kernel<<<o->grid_for(t->n_params * (int64_t)B), 256, 0, o->stream>>>(pd, o->V + (t->n + 1 + t->m) * (int64_t)B, t->n_params, B);
  }
  const int64_t lens[6] = {0, 1, t->n, t->m, t->nnz_jac, t->nnz_hess};
  const double *consts[6] = {nullptr, &t->f_const, t->grad_const, t->g_const, t->jac_const, t->hess_const};
  int64_t maxlen = t->n > t->m ? t->n : t->m;
  for (int s = 1; s < 6; ++s) {
    o->out_len[s] = lens[s];
    if (lens[s] > maxlen) maxlen = lens[s];
    CKB(cudaMalloc(&p, (size_t)(lens[s] + 2) * B * sizeof(double)));
    o->owned.push_back(p);
    o->out[s] = static_cast<double *>(p);
    if (lens[s] > 0 && consts[s]) { if (o->upload(consts[s], lens[s], &o->out_const[s])) return 1; }
  }
  o->split_scratch_len = (int64_t)32 * 64 * B;          // KS <= 32 slices x up to 64 long rows x B starts
  o->split_ticket_len = 64 * (int64_t)((B + 31) / 32) + 64;
  CKB(cudaMalloc(&p, (size_t)o->split_scratch_len * sizeof(double)));
  o->owned.push_back(p);
  o->split_scratch = static_cast<double *>(p);
  CKB(cudaMalloc(&p, (size_t)o->split_ticket_len * sizeof(unsigned int)));
  o->owned.push_back(p);
  o->split_tickets = static_cast<unsigned int *>(p);
  CKB(cudaMemset(o->split_tickets, 0, (size_t)o->split_ticket_len * sizeof(unsigned int)));
  o->stage_len = maxlen + 2;
  CKB(cudaMalloc(&p, (size_t)o->stage_len * B * sizeof(double)));
  o->owned.push_back(p);
  o->stage = static_cast<double *>(p);

  o->instrs.resize(t->n_instr);
  for (int i = 0; i < t->n_instr; ++i) {
    const dnlp_instr_desc &h = t->instrs[i];
    BInstr &D = o->instrs[i];
    D.d = h;
    D.d.ptr = nullptr; D.d.coef = nullptr; D.d.f1 = nullptr; D.d.f2 = nullptr; D.d.pos = nullptr; D.d.Q = nullptr;
    D.d.qpos = nullptr;                       // (SPMVJ only lives in the union program of the single-start engine)
    if (h.kind == DNLP_POLY) {
      if (h.ptr) { if (o->upload(h.ptr, h.count + 1, const_cast<int64_t **>(&D.d.ptr))) return 1; }
      if (o->upload(h.coef, h.nterms, const_cast<double **>(&D.d.coef))) return 1;
      if (o->upload(h.f1, h.nterms, const_cast<int32_t **>(&D.d.f1))) return 1;
      if (h.f2) { if (o->upload(h.f2, h.nterms, const_cast<int32_t **>(&D.d.f2))) return 1; }
      D.has_f2 = h.f2 != nullptr;
      // every row combines the same <= 16 slots?  (uniform rows, single factor)
      if (!h.ptr && !h.f2 && h.row_len >= 2 && h.row_len <= 16 && h.count >= 1024) {
        bool same = true;
        for (int64_t r = 1; r < h.count && same; ++r)
          for (int j = 0; j < h.row_len; ++j)
            if (h.f1[r * h.row_len + j] != h.f1[j]) { same = false; break; }
        if (same) { if (o->upload(h.f1, (int64_t)h.row_len, &D.smallk_slots)) return 1; }
      }
    } else if (h.kind == DNLP_GEMV) {
      if (o->upload(h.Q, h.count * h.ncols, const_cast<double **>(&D.d.Q))) return 1;
    } else if (h.kind == DNLP_SCALE) {
      if (o->upload(h.coef, h.count, const_cast<double **>(&D.d.coef))) return 1;
    }
    if ((h.kind == DNLP_POLY || h.kind == DNLP_SCALE) && h.pos) {
      if (o->upload(h.pos, h.count, const_cast<int32_t **>(&D.d.pos))) return 1;
    }
  }
  for (int q = 0; q < DNLP_NPROG; ++q) o->prog[q].assign(t->prog[q], t->prog[q] + t->prog_len[q]);
  // group the dense maps that depend on x only and share a shape
  for (int i = 0; i < t->n_instr; ++i) {
    const dnlp_instr_desc &d = o->instrs[i].d;
    if (d.kind != DNLP_GEMV) continue;
    {
      double *dst = (d.dst_space == DNLP_DST_V) ? o->V + d.dst_off * B : o->out[d.dst_space] + d.dst_off * B;
      dnlp::GemmDesc one{d.Q, o->V + d.x_off * B, dst, d.alpha};
      if (o->upload(&one, 1, &o->instrs[i].one_desc)) return 1;
    }
    if (d.level != 0 || d.dst_space != DNLP_DST_V) continue;
    int gi = -1;
    for (size_t g = 0; g < o->groups.size(); ++g)
      if (o->groups[g].M == d.count && o->groups[g].K == d.ncols) { gi = (int)g; break; }
    if (gi < 0) { o->groups.emplace_back(); gi = (int)o->groups.size() - 1; o->groups[gi].M = d.count; o->groups[gi].K = d.ncols; }
    o->groups[gi].members.push_back(i);
  }
  for (size_t g = 0; g < o->groups.size(); ++g) {
    auto &G = o->groups[g];
    if (G.members.size() < 2) continue;                 // a lone map keeps the plain path
    std::vector<dnlp::GemmDesc> hd;
    for (int32_t id : G.members) {
      const dnlp_instr_desc &d = o->instrs[id].d;
      hd.push_back(dnlp::GemmDesc{d.Q, o->V + d.x_off * B, o->V + d.dst_off * B, d.alpha});
      o->instrs[id].gemm_group = (int)g;
    }
    if (o->upload(hd.data(), (int64_t)hd.size(), &G.descs)) return 1;
  }
  if (const char *e = getenv("DNLP_BATCH_NO_GRAPHS")) o->graphs_enabled = atoi(e) == 0;
  if (const char *e = getenv("DNLP_DMMA_K8")) o->dmma_k8 = atoi(e) != 0;
  if (o->reset_outputs()) return 1;
  CKB(cudaFuncSetAttribute(dnlp::bgemm_dmma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dnlp::BGEMM_SMEM));
  CKB(cudaFuncSetAttribute(dnlp::bgemm_dmma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dnlp::BGEMM_SMEM));
  CKB(cudaStreamSynchronize(o->stream));
  return 0;
}

int dnlp_batch_create(const dnlp_tape_desc *t, int device, int32_t batch, dnlp_batch **out) {
  *out = nullptr;
  if (batch <= 0) { g_batch_create_error = "batch must be positive"; return 1; }
  dnlp_batch *o = new dnlp_batch();
  o->device = device;
  o->B = batch;
  if (batch_create_impl(o, t)) {
    g_batch_create_error = o->err;
    dnlp_batch_destroy(o);
    return 1;
  }
  *out = o;
  return 0;
}

const char *dnlp_batch_last_error(dnlp_batch *o) { return o ? o->err.c_str() : g_batch_create_error.c_str(); }

}  // extern "C"

int dnlp_batch::reset_outputs() {
  for (int s = 1; s < 6; ++s) {
    if (out_len[s] <= 0) continue;
    if (out_const[s]) {
      bfill_kernel<<<grid_for(out_len[s] * B), 256, 0, stream>>>(out_const[s], out[s], out_len[s], B);
      ++launches;
    } else {
      CKB(cudaMemsetAsync(out[s], 0, (size_t)out_len[s] * B * sizeof(double), stream));
    }
  }
  return 0;
}

extern "C" {

int dnlp_batch_upload(dnlp_batch *o, const double *X, const double *LAM, const double *SIGMA) {
  if (o == nullptr) { g_batch_create_error = "batch handle is NULL (closed or never created)"; return 1; }
  std::string &err = o->err;
  CKB(cudaSetDevice(o->device));
  if (o->put(X, o->V, o->n)) return 1;
  if (SIGMA) CKB(cudaMemcpyAsync(o->V + o->n * o->B, SIGMA, (size_t)o->B * sizeof(double), cudaMemcpyHostToDevice, o->stream));
  if (LAM && o->m > 0) { if (o->put(LAM, o->V + (o->n + 1) * o->B, o->m)) return 1; }
  CKB(cudaStreamSynchronize(o->stream));
  return 0;
}

int dnlp_batch_eval(dnlp_batch *o, const double *X, const double *LAM, const double *SIGMA,
                    double *F, double *GRAD, double *G, double *JAC, double *HESS) {
  if (o == nullptr) { g_batch_create_error = "batch handle is NULL (closed or never created)"; return 1; }
  std::string &err = o->err;
  CKB(cudaSetDevice(o->device));
  if (o->put(X, o->V, o->n)) return 1;
  const bool want_h = HESS != nullptr;
  if (want_h) {
    if (!SIGMA || (o->m > 0 && !LAM)) { err = "hessian requested without multipliers"; return 1; }
    CKB(cudaMemcpyAsync(o->V + o->n * o->B, SIGMA, (size_t)o->B * sizeof(double), cudaMemcpyHostToDevice, o->stream));
    if (o->m > 0) { if (o->put(LAM, o->V + (o->n + 1) * o->B, o->m)) return 1; }
  }
  double *outs[6] = {nullptr, F, GRAD, G, JAC, HESS};
  int32_t mask = 0;
  for (int p = 0; p < 5; ++p)
    if (outs[p + 1]) mask |= 1 << p;
  if (o->run_union(mask)) return 1;
  for (int s = 1; s < 6; ++s)
    if (outs[s]) {
      if (o->get(s, outs[s])) return 1;
      CKB(cudaStreamSynchronize(o->stream));      // the staging buffer is reused by the next output
    }
  CKB(cudaStreamSynchronize(o->stream));
  return 0;
}

int dnlp_batch_run_device(dnlp_batch *o, int32_t prog_mask, int32_t iters, float *elapsed_ms) {
  if (o == nullptr) { g_batch_create_error = "batch handle is NULL (closed or never created)"; return 1; }
  std::string &err = o->err;
  CKB(cudaSetDevice(o->device));
  CKB(cudaEventRecord(o->ev0, o->stream));
  for (int it = 0; it < iters; ++it)
    if (o->run_union(prog_mask)) return 1;
  CKB(cudaEventRecord(o->ev1, o->stream));
  CKB(cudaEventSynchronize(o->ev1));
  float ms = 0.f;
  CKB(cudaEventElapsedTime(&ms, o->ev0, o->ev1));
  if (elapsed_ms) *elapsed_ms = ms;
  return 0;
}

int dnlp_batch_read_output(dnlp_batch *o, int32_t space, double *out) {
  if (o == nullptr) { g_batch_create_error = "batch handle is NULL (closed or never created)"; return 1; }
  std::string &err = o->err;
  CKB(cudaSetDevice(o->device));
  if (space < 1 || space > 5) { err = "bad output id"; return 1; }
  if (o->get(space, out)) return 1;
  CKB(cudaStreamSynchronize(o->stream));
  return 0;
}

int dnlp_batch_profile_instrs(dnlp_batch *o, int32_t p, int32_t iters, float *ms_per_instr) {
  if (o == nullptr) { g_batch_create_error = "batch handle is NULL (closed or never created)"; return 1; }
  std::string &err = o->err;
  CKB(cudaSetDevice(o->device));
  for (size_t i = 0; i < o->instrs.size(); ++i) ms_per_instr[i] = 0.f;
  for (int32_t id : o->prog[p]) if (o->launch(o->instrs[id])) return 1;
  CKB(cudaStreamSynchronize(o->stream));
  for (int it = 0; it < iters; ++it)
    for (int32_t id : o->prog[p]) {
      CKB(cudaEventRecord(o->ev0, o->stream));
      if (o->launch(o->instrs[id])) return 1;
      CKB(cudaEventRecord(o->ev1, o->stream));
      CKB(cudaEventSynchronize(o->ev1));
      float ms = 0.f;
      CKB(cudaEventElapsedTime(&ms, o->ev0, o->ev1));
      ms_per_instr[id] += ms / (float)iters;
    }
  return 0;
}

// CUDA-event time of every GROUPED GEMM launch (the k+1 independent quad_form maps of a QCQP as one grid):
// ms_per_group[g], flops_per_group[g]; returns the number of groups (<= max_groups) or -1.
int dnlp_batch_profile_groups(dnlp_batch *o, int32_t iters, float *ms_per_group, double *flops_per_group, int32_t max_groups) {
  if (o == nullptr) { g_batch_create_error = "batch handle is NULL (closed or never created)"; return -1; }
  if (cudaSetDevice(o->device) != cudaSuccess) return -1;
  int ng = 0;
  for (size_t gi = 0; gi < o->groups.size() && ng < max_groups; ++gi) {
    auto &G = o->groups[gi];
    if (G.members.size() < 2) continue;
    const int64_t tiles = ((G.M + dnlp::GM - 1) / dnlp::GM) * ((o->B + dnlp::GN - 1) / dnlp::GN) * (int64_t)G.members.size();
    const int64_t cap = (int64_t)o->sm_count * 4;
    const int grid = (int)(tiles < cap ? tiles : cap);
    auto go = [&]() {
      if (o->dmma_k8) dnlp::bgemm_dmma_kernel<true><<<grid, 128, dnlp::BGEMM_SMEM, o->stream>>>(G.descs, (int)G.members.size(), (int)G.M, o->B, (int)G.K);
      else dnlp::bgemm_dmma_kernel<false><<<grid, 128, dnlp::BGEMM_SMEM, o->stream>>>(G.descs, (int)G.members.size(), (int)G.M, o->B, (int)G.K);
    };
    go();
    cudaEventRecord(o->ev0, o->stream);
    for (int it = 0; it < iters; ++it) go();
    cudaEventRecord(o->ev1, o->stream);
    if (cudaEventSynchronize(o->ev1) != cudaSuccess) return -1;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, o->ev0, o->ev1);
    ms_per_group[ng] = ms / (float)(iters > 0 ? iters : 1);
    flops_per_group[ng] = 2.0 * (double)G.M * (double)G.K * (double)o->B * (double)G.members.size();
    ++ng;
  }
  return ng;
}

int64_t dnlp_batch_kernel_launches(dnlp_batch *o) { return o ? o->launches : -1; }

int dnlp_batch_kkt_setup(dnlp_batch *o, int64_t ns, const int32_t *slack_rows, const int32_t *jac_rows,
                         const int32_t *jac_cols, const int32_t *hess_rows, const int32_t *hess_cols) {
  if (o == nullptr) { g_batch_create_error = "batch handle is NULL (closed or never created)"; return 1; }
  std::string &err = o->err;
  CKB(cudaSetDevice(o->device));
  CKB(cudaStreamSynchronize(o->stream));
  o->kkt_free();
  const int64_t n = o->n, m = o->m, nnzJ = o->out_len[4], nnzH = o->out_len[5];
  if (ns < 0 || ns > m) { err = "kkt_setup: the number of slack rows must lie in [0, m]"; return 1; }
  const int64_t N = n + ns, M = N + m, B = o->B;
  // the scatter map: every lower-triangle target (i, j) of K with its sources in pattern order
  std::map<int64_t, std::vector<int32_t>> tgt;
  for (int64_t i = 0; i < M; ++i) tgt[i * M + i];
  std::vector<char> seen(m > 0 ? m : 1, 0);
  for (int64_t s = 0; s < ns; ++s) {
    const int32_t r = slack_rows[s];
    if (r < 0 || r >= m || seen[r]) { err = "kkt_setup: slack rows must be distinct constraint rows"; return 1; }
    seen[r] = 1;
  }
  for (int64_t k = 0; k < nnzH; ++k) {
    const int64_t r = hess_rows[k], c = hess_cols[k];
    if (r < 0 || r >= n || c < 0 || c >= n) { err = "kkt_setup: Hessian pattern entry out of range"; return 1; }
    tgt[std::max(r, c) * M + std::min(r, c)].push_back((int32_t)k);
  }
  for (int64_t k = 0; k < nnzJ; ++k) {
    const int64_t r = jac_rows[k], c = jac_cols[k];
    if (r < 0 || r >= m || c < 0 || c >= n) { err = "kkt_setup: Jacobian pattern entry out of range"; return 1; }
    tgt[(N + r) * M + c].push_back((int32_t)(nnzH + k));
  }
  for (int64_t s = 0; s < ns; ++s) tgt[(N + slack_rows[s]) * M + n + s].push_back(-1);
  std::vector<int32_t> ti, tj, sp(1, 0), src;
  for (auto &kv : tgt) {
    ti.push_back((int32_t)(kv.first / M));
    tj.push_back((int32_t)(kv.first % M));
    src.insert(src.end(), kv.second.begin(), kv.second.end());
    sp.push_back((int32_t)src.size());
  }
  // refuse what does not fit: the B dense systems dominate
  const double kbytes = (double)B * (double)M * (double)M * 8.0;
  const double vbytes = (double)B * (double)(9 * M + 2 * N + 4) * 8.0 + (double)(3 * ti.size() + src.size() + 1) * 4.0;
  size_t free_b = 0, total_b = 0;
  CKB(cudaMemGetInfo(&free_b, &total_b));
  if (kbytes + vbytes > 0.95 * (double)free_b) {
    char buf[320];
    snprintf(buf, sizeof buf, "kkt_setup: the dense KKT systems need B*(N+m)^2*8 = %lld*%lld^2*8 = %.3e bytes "
             "(+%.3e for vectors) but the device has %.3e bytes free; use fewer starts per batch",
             (long long)B, (long long)M, kbytes, vbytes, (double)free_b);
    err = buf;
    return 1;
  }
  auto &Q = o->kkt;
  Q.N = N; Q.M = M; Q.ntgt = (int64_t)ti.size(); Q.nnzH = nnzH;
  auto alloc = [&](size_t bytes, void **p) -> int {
    CKB(cudaMalloc(p, bytes < 8 ? 8 : bytes));
    Q.owned.push_back(*p);
    return 0;
  };
  auto up = [&](const std::vector<int32_t> &h, int32_t **d) -> int {
    if (alloc(h.size() * sizeof(int32_t), (void **)d)) return 1;
    CKB(cudaMemcpyAsync(*d, h.data(), h.size() * sizeof(int32_t), cudaMemcpyHostToDevice, o->stream));
    return 0;
  };
  if (up(ti, &Q.ti) || up(tj, &Q.tj) || up(sp, &Q.sp) || up(src, &Q.src)) { o->kkt_free(); return 1; }
  if (alloc((size_t)B * M * M * 8, (void **)&Q.K) || alloc((size_t)B * M * 8, (void **)&Q.Dg) ||
      alloc((size_t)B * N * 8, (void **)&Q.Wd) || alloc((size_t)B * 3 * M * 8, (void **)&Q.work) ||
      alloc((size_t)B * N * 8, (void **)&Q.sigma) || alloc((size_t)B * 8, (void **)&Q.dw) ||
      alloc((size_t)B * 8, (void **)&Q.dc) || alloc((size_t)B * M * 8, (void **)&Q.rhs) ||
      alloc((size_t)B * M * 8, (void **)&Q.sol) || alloc((size_t)B * 8, (void **)&Q.wq) ||
      alloc((size_t)B * 4, (void **)&Q.starts) || alloc((size_t)B * 3 * 4, (void **)&Q.inertia)) {
    o->kkt_free();
    return 1;
  }
  CKB(cudaStreamSynchronize(o->stream));
  return 0;
}

int dnlp_batch_kkt_solve(dnlp_batch *o, int32_t count, const int32_t *starts, const double *sigma, const double *dw,
                         const double *dc, const double *rhs, double *sol, int32_t *inertia, double *wquad,
                         float *elapsed_ms) {
  if (o == nullptr) { g_batch_create_error = "batch handle is NULL (closed or never created)"; return 1; }
  std::string &err = o->err;
  auto &Q = o->kkt;
  if (Q.M == 0) { err = "kkt_solve: call dnlp_batch_kkt_setup first"; return 1; }
  if (count < 0 || count > o->B) { err = "kkt_solve: count must lie in [0, batch]"; return 1; }
  if (count == 0) { if (elapsed_ms) *elapsed_ms = 0.f; return 0; }
  std::vector<char> seen(o->B, 0);
  for (int c = 0; c < count; ++c) {
    if (starts[c] < 0 || starts[c] >= o->B || seen[starts[c]]) { err = "kkt_solve: start ids must be distinct and in [0, batch)"; return 1; }
    seen[starts[c]] = 1;
  }
  CKB(cudaSetDevice(o->device));
  const int64_t N = Q.N, M = Q.M;
  cudaStream_t st = o->stream;
  CKB(cudaMemcpyAsync(Q.starts, starts, (size_t)count * 4, cudaMemcpyHostToDevice, st));
  if (N > 0) CKB(cudaMemcpyAsync(Q.sigma, sigma, (size_t)count * N * 8, cudaMemcpyHostToDevice, st));
  CKB(cudaMemcpyAsync(Q.dw, dw, (size_t)count * 8, cudaMemcpyHostToDevice, st));
  CKB(cudaMemcpyAsync(Q.dc, dc, (size_t)count * 8, cudaMemcpyHostToDevice, st));
  CKB(cudaMemcpyAsync(Q.rhs, rhs, (size_t)count * M * 8, cudaMemcpyHostToDevice, st));
  CKB(cudaEventRecord(o->ev0, st));
  const int64_t cap = (int64_t)o->sm_count * 8;
  int64_t g = ((int64_t)count * M * M + 255) / 256;
  dnlp_kkt::kkt_zero_kernel<<<(int)(g < cap ? g : cap), 256, 0, st>>>(Q.K, Q.starts, count, M * M);
  g = (Q.ntgt * count + 255) / 256;
  dnlp_kkt::kkt_scatter_kernel<<<(int)(g < cap ? g : cap), 256, 0, st>>>(
      Q.K, Q.Dg, Q.Wd, o->out[4], o->out[5], o->B, Q.ti, Q.tj, Q.sp, Q.src, Q.ntgt, Q.nnzH, Q.starts, count,
      Q.sigma, Q.dw, Q.dc, N, M);
  dnlp_kkt::kkt_ldl_kernel<<<count, dnlp_kkt::THREADS, 0, st>>>(Q.K, Q.starts, M, Q.inertia, Q.work, 3 * M);
  dnlp_kkt::kkt_solve_kernel<<<count, dnlp_kkt::THREADS, 0, st>>>(Q.K, Q.Dg, Q.Wd, Q.starts, M, N, Q.inertia, Q.rhs,
                                                                  Q.sol, Q.wq, Q.work);
  o->launches += 4;
  CKB(cudaPeekAtLastError());
  CKB(cudaEventRecord(o->ev1, st));
  CKB(cudaMemcpyAsync(sol, Q.sol, (size_t)count * M * 8, cudaMemcpyDeviceToHost, st));
  CKB(cudaMemcpyAsync(inertia, Q.inertia, (size_t)count * 3 * 4, cudaMemcpyDeviceToHost, st));
  CKB(cudaMemcpyAsync(wquad, Q.wq, (size_t)count * 8, cudaMemcpyDeviceToHost, st));
  CKB(cudaStreamSynchronize(st));
  float ms = 0.f;
  CKB(cudaEventElapsedTime(&ms, o->ev0, o->ev1));
  if (elapsed_ms) *elapsed_ms = ms;
  return 0;
}

int dnlp_batch_kkt_matrix(dnlp_batch *o, int32_t start, double *out) {
  if (o == nullptr) { g_batch_create_error = "batch handle is NULL (closed or never created)"; return 1; }
  std::string &err = o->err;
  auto &Q = o->kkt;
  if (Q.M == 0) { err = "kkt_matrix: call dnlp_batch_kkt_setup first"; return 1; }
  if (start < 0 || start >= o->B) { err = "kkt_matrix: start id out of range"; return 1; }
  CKB(cudaSetDevice(o->device));
  const int64_t M = Q.M;
  std::vector<double> dg(M);
  CKB(cudaMemcpyAsync(out, Q.K + (int64_t)start * M * M, (size_t)M * M * 8, cudaMemcpyDeviceToHost, o->stream));
  CKB(cudaMemcpyAsync(dg.data(), Q.Dg + (int64_t)start * M, (size_t)M * 8, cudaMemcpyDeviceToHost, o->stream));
  CKB(cudaStreamSynchronize(o->stream));
  for (int64_t i = 0; i < M; ++i) {         // the strict upper triangle and the saved diagonal are K as assembled
    out[i * M + i] = dg[i];
    for (int64_t j = 0; j < i; ++j) out[i * M + j] = out[j * M + i];
  }
  return 0;
}

}  // extern "C"
