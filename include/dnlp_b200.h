/*
 * dnlp_b200 - C ABI of the B200-native NLP oracle.
 *
 * Drop-in boundary: these entry points replace, one for one, the seven callbacks
 * of the reference's `Oracles` object that cyipopt / Knitro drive
 * (/root/reference/cvxpy/reductions/solvers/nlp_solvers/nlp_solver.py:181-427;
 *  consumers: ipopt_nlpif.py:143-170, knitro_nlpif.py:211-309).
 *
 *   Oracles.__init__           nlp_solver.py:182-203   -> dnlp_create
 *   Oracles.objective          nlp_solver.py:212-216   -> dnlp_eval_f
 *   Oracles.gradient           nlp_solver.py:218-235   -> dnlp_eval_grad
 *   Oracles.constraints        nlp_solver.py:237-244   -> dnlp_eval_g
 *   Oracles.jacobian           nlp_solver.py:278-307   -> dnlp_eval_jac
 *   Oracles.hessian            nlp_solver.py:394-421   -> dnlp_eval_hess
 *   Oracles.jacobianstructure  nlp_solver.py:309-335   -> host arrays produced once by the DAG
 *   Oracles.hessianstructure   nlp_solver.py:374-392      compiler (dnlp_b200/compiler.py); the
 *                                                         library only stores nnz counts
 *
 * Plain pointers and sizes only; no exceptions cross the ABI.  Every function
 * returning int returns 0 on success, non-zero otherwise (dnlp_last_error gives text).
 * All arithmetic is fp64, all slot / position indices int32, row pointers int64.
 *
 * Ownership: the oracle owns its device buffers, stream and events.  `x`, `lam` and
 * output pointers are caller-owned host memory (pageable or pinned) that is read /
 * written only during the call; every call is complete (stream-synchronised) on return.
 * Threading: one oracle is used from one thread at a time (callbacks arrive serially).
 */
#ifndef DNLP_B200_H
#define DNLP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dnlp_oracle dnlp_oracle;

/* instruction kinds */
enum { DNLP_ELEM = 1, DNLP_POLY = 2, DNLP_GEMV = 3, DNLP_SCALE = 4, DNLP_SPMVJ = 5 };
/* destinations: the value buffer V or one of the five outputs */
enum { DNLP_DST_V = 0, DNLP_DST_F = 1, DNLP_DST_GRAD = 2, DNLP_DST_G = 3, DNLP_DST_JAC = 4, DNLP_DST_HESS = 5 };
/* programs */
enum { DNLP_PROG_F = 0, DNLP_PROG_GRAD = 1, DNLP_PROG_G = 2, DNLP_PROG_JAC = 3, DNLP_PROG_HESS = 4,
       DNLP_PROG_ALL = 5, DNLP_NPROG = 6 };

/* One tape instruction (host pointers; dnlp_create copies everything to HBM). */
typedef struct {
  int32_t kind;
  int32_t dst_space;
  int64_t dst_off;
  int64_t count;
  /* ELEM: dst[k] = F(V[a_off + k*a_stride], V[b_off + k*b_stride]; param) */
  int32_t fcode;
  int32_t a_stride;
  int32_t b_stride;
  int32_t accumulate;     /* POLY/SCALE: dst += instead of dst = */
  double param;
  int64_t a_off;
  int64_t b_off;
  /* POLY: dst[pos?[k]] = sum_{t in ptr[k]..ptr[k+1]} coef[t] * V[f1[t]] * V[f2[t]]   (index -1 = 1.0) */
  const int64_t *ptr;     /* count+1 entries, or NULL when every row has row_len terms */
  const double *coef;     /* nterms */
  const int32_t *f1;      /* nterms */
  const int32_t *f2;      /* nterms, or NULL when no term has a second factor */
  const int32_t *pos;     /* count entries or NULL (identity) */
  int64_t nterms;
  int32_t row_len;        /* uniform row length when ptr == NULL */
  int32_t uses_lam;       /* depends on (sigma, lambda): never cached across calls */
  int32_t level;          /* 0 = reads only x / lambda (no instruction feeds it) */
  int32_t dep_mask;       /* what the result depends on, transitively: 1 = x, 2 = sigma, 4 = lambda, 8 = parameters */
  /* GEMV: dst[i] = alpha * sum_j Q[i*ncols + j] * V[x_off + j] */
  const double *Q;
  int64_t ncols;
  int64_t x_off;
  double alpha;
  /* SCALE: dst[pos?[k]] = V[s_slot] * coef[k] */
  int64_t s_slot;
  /* data dependencies: ids of the instructions whose V ranges this one reads.  Independent
   * instructions become parallel branches of the CUDA graph that replays a launch sequence. */
  const int32_t *deps;
  int64_t n_deps;
  /* ELEM: dst[k * dst_stride] = post_scale * F(...).  dst_stride 2 = the interleaved (value, derivative)
   * pair layout that SPMVJ gathers with one 16-byte load. */
  int32_t dst_stride;
  int32_t reserved0;
  double post_scale;
  /* SPMVJ (fused constraint value + Jacobian fill; ptr / coef / f1 / pos as for POLY, f1 even slots):
   *   G[pos?[k]] = sum_t coef[t] * V[f1[t]],   JAC[qpos[t]] = coef[t] * V[f1[t] + 1]   (qpos -1 = skip) */
  const int32_t *qpos;    /* nterms */
} dnlp_instr_desc;

typedef struct {
  int64_t n;              /* variables */
  int64_t m;              /* constraints */
  int64_t nslots;         /* length of V: n + 1 + m + temporaries */
  int64_t nnz_jac;
  int64_t nnz_hess;
  int32_t n_instr;
  const dnlp_instr_desc *instrs;
  const int32_t *prog[DNLP_NPROG];   /* instruction ids in execution order */
  int32_t prog_len[DNLP_NPROG];
  /* compile-time constant part of every output (entries owned by an instruction are overwritten) */
  double f_const;
  const double *grad_const;   /* n */
  const double *g_const;      /* m */
  const double *jac_const;    /* nnz_jac */
  const double *hess_const;   /* nnz_hess */
  /* Parameter values (cvxpy Parameters: constants whose value may change between solves) occupy
   * V[n + 1 + m, n + 1 + m + n_params); instructions that read them carry dep_mask bit 8. */
  int64_t n_params;
  const double *params;       /* n_params initial values */
} dnlp_tape_desc;

int dnlp_device_count(void);
const char *dnlp_version(void);
int dnlp_device_synchronize(int device);       /* cudaDeviceSynchronize on `device` (timing brackets of callers) */

int dnlp_create(const dnlp_tape_desc *tape, int device, dnlp_oracle **out);
void dnlp_destroy(dnlp_oracle *o);
const char *dnlp_last_error(dnlp_oracle *o);   /* o may be NULL: error of the last failed create */

/* ---- the callbacks (host buffers in, host buffers out) ---- */
int dnlp_eval_f(dnlp_oracle *o, const double *x, double *f);
int dnlp_eval_grad(dnlp_oracle *o, const double *x, double *grad /* n */);
int dnlp_eval_g(dnlp_oracle *o, const double *x, double *g /* m */);
int dnlp_eval_jac(dnlp_oracle *o, const double *x, double *vals /* nnz_jac */);
int dnlp_eval_hess(dnlp_oracle *o, const double *x, const double *lam /* m */, double sigma,
                   double *vals /* nnz_hess */);
/* all five at one (x, lam, sigma): one upload, shared forward sweep, outputs may be NULL to skip the copy */
int dnlp_eval_all(dnlp_oracle *o, const double *x, const double *lam, double sigma,
                  double *f, double *grad, double *g, double *jac, double *hess);

/* ---- parameters: new values for the slots V[n+1+m ..); invalidates exactly what depends on them (no recompilation) ---- */
int dnlp_set_params(dnlp_oracle *o, const double *values, int64_t count);

/* ---- constant-entry elision (reference quirk Q5: affine Jacobian rows never change) ----
 * dnlp_set_dynamic registers, for one output (DNLP_DST_GRAD..DNLP_DST_HESS), the positions of the
 * entries that depend on x / lambda.  dnlp_eval_dyn then runs program `prog` and copies ONLY those
 * entries, compacted in `pos` order, to `compact`; the caller keeps the constant entries (it got
 * them once from the compiler) and scatters the compact values into its array. */
int dnlp_set_dynamic(dnlp_oracle *o, int32_t dst_space, const int32_t *pos, int64_t count);
int dnlp_eval_dyn(dnlp_oracle *o, int32_t prog, const double *x, const double *lam, double sigma,
                  double *compact);

/* ---- eager delivery of the x-only outputs ----
 * The caller names the (pinned) host arrays it passes to dnlp_eval_f / _grad / _g / _jac (or, for an
 * output with registered dynamic positions, the compact array it passes to dnlp_eval_dyn).  With
 * `eager` != 0 the first callback at a NEW x computes f, grad, g and J together and copies them to
 * those arrays on a second stream: the D2H of the later callbacks' results overlaps the solver's own
 * work, the staging of lambda and its H2D (PCIe is full duplex); a later callback at the same x only
 * waits for its copy.  The Hessian (needs lambda, sigma) keeps its own call. */
int dnlp_bind_outputs(dnlp_oracle *o, double *f, double *grad, double *g, double *jac, int32_t eager);

/* ---- device-resident results (multi-GPU assembly: outputs are reduced / gathered over NVLink
 *      without a host round trip) ----
 * dnlp_run stages the inputs and executes program `prog`, leaving the result in HBM;
 * dnlp_output_ptr returns the device address of a full output array (length n, m, nnz_jac, nnz_hess). */
int dnlp_run(dnlp_oracle *o, int32_t prog, const double *x, const double *lam, double sigma);
void *dnlp_output_ptr(dnlp_oracle *o, int32_t dst_space);

/* ---- pinned host memory for callers that want true async copies ---- */
void *dnlp_host_alloc(int64_t bytes);
void dnlp_host_free(void *p);

/* ---- device-resident execution and measurement (bench.py / tests) ----
 * dnlp_upload_point puts (x, lam, sigma) into HBM; dnlp_run_device then executes the programs in
 * `prog_mask` (bit i = program i) `iters` times back to back with every cache invalidated before each
 * iteration and returns the CUDA-event time of the whole loop in ms.
 * dnlp_profile_instrs times every instruction of one program with its own event pair. */
int dnlp_upload_point(dnlp_oracle *o, const double *x, const double *lam, double sigma);
int dnlp_run_device(dnlp_oracle *o, int32_t prog_mask, int32_t iters, float *elapsed_ms);
int dnlp_profile_instrs(dnlp_oracle *o, int32_t prog, int32_t iters, float *ms_per_instr /* n_instr */);
int dnlp_read_output(dnlp_oracle *o, int32_t dst_space, double *out);   /* D2H of one output array */
int64_t dnlp_kernel_launches(dnlp_oracle *o);                           /* launches since create */
const char *dnlp_instr_kernel(dnlp_oracle *o, int32_t instr);           /* kernel name of an executed instruction */
int dnlp_set_cache(dnlp_oracle *o, int32_t enabled);                    /* x-keyed forward cache on/off */
int dnlp_set_graphs(dnlp_oracle *o, int32_t enabled);                   /* CUDA-graph replay of launch sequences on/off */
int dnlp_set_parallel(dnlp_oracle *o, int32_t enabled);                 /* parallel graph branches for independent instructions on/off */
int dnlp_set_windows(dnlp_oracle *o, int32_t enabled);                  /* shared-memory gather windows (SpMV against a short vector) on/off */

/* ---- batched multi-start evaluation (BASELINE config 4; the reference's serial `best_of` loop,
 *      cvxpy/problems/problem.py:1249-1275, evaluates one start at a time) ----
 * The same tape is evaluated at `batch` independent points in lock step.  Host arrays hold one
 * start per contiguous block: X[b*n + i], LAM[b*m + j], SIGMA[b], and likewise every output
 * (F[b], GRAD[b*n + i], G[b*m + j], JAC[b*nnz_jac + k], HESS[b*nnz_hess + k]).  A NULL output is
 * skipped together with its program.  Dense quad_form maps become FP64 tensor-core GEMMs. */
typedef struct dnlp_batch dnlp_batch;
int dnlp_batch_create(const dnlp_tape_desc *tape, int device, int32_t batch, dnlp_batch **out);
void dnlp_batch_destroy(dnlp_batch *b);
const char *dnlp_batch_last_error(dnlp_batch *b);
int dnlp_batch_eval(dnlp_batch *b, const double *X, const double *LAM, const double *SIGMA,
                    double *F, double *GRAD, double *G, double *JAC, double *HESS);
int dnlp_batch_upload(dnlp_batch *b, const double *X, const double *LAM, const double *SIGMA);
int dnlp_batch_run_device(dnlp_batch *b, int32_t prog_mask, int32_t iters, float *elapsed_ms);
int dnlp_batch_read_output(dnlp_batch *b, int32_t dst_space, double *out);   /* D2H of one output, start-major */
int dnlp_batch_profile_instrs(dnlp_batch *b, int32_t prog, int32_t iters, float *ms_per_instr);
int dnlp_batch_profile_groups(dnlp_batch *b, int32_t iters, float *ms_per_group, double *flops_per_group,
                              int32_t max_groups);   /* grouped DMMA GEMM launches, timed with CUDA events */
int64_t dnlp_batch_kernel_launches(dnlp_batch *b);
const char *dnlp_batch_instr_kernel(dnlp_batch *b, int32_t instr);   /* kernel variant of an executed instruction, e.g.
                                                                          "bsmallk_kernel<9, 2>"; "" if never run */

/* ---- batched KKT systems of the lock-step interior-point driver (dnlp_b200/lockstep_ipm.py) ----
 * Per start b, with z = (x, slacks) of length N = n + ns and M = N + m:
 *   K_b = [[ W_b + diag(Sigma_b) + dw_b I ,  A_b' ],   W_b: the Hessian output HESS (lower-triangle pattern, mirrored,
 *          [ A_b                          , -dc_b I ]]       duplicates summed in pattern order), zero on the slack block
 *   A_b = [J_b, -P]: J_b from output JAC, column n + s of P is a 1 in constraint row slack_rows[s].
 * dnlp_batch_kkt_setup builds the scatter maps from the patterns (host arrays) and allocates B dense M x M systems;
 * it fails with a message naming B*M^2*8 bytes when they do not fit.  dnlp_batch_kkt_solve assembles K for `count`
 * distinct start ids from the HESS and JAC outputs the last run left in HBM, factors it as LDL' without pivoting
 * (order [x / slack block, constraint block]) and returns per start the inertia (n+, n-, n0) from the signs of D
 * (a pivot d_j with |d_j| <= 1e-11 (|K_jj| + sum_k L_jk^2 |d_k|) counts as zero).  For a start whose inertia is (N, m, 0) it solves K sol = rhs,
 * refines once against K and returns the solution and dz' W dz (dz = sol[:N]); the solution row and wquad are NaN
 * when the inertia differs, the result is not finite, or its normwise backward error exceeds 1e-8.
 * Inputs and outputs are start-major: sigma[c*N + i], rhs / sol[c*M + i], inertia[3c + k].  *elapsed_ms: CUDA-event
 * time of assembly + factorisation + solve.  dnlp_batch_kkt_matrix copies the assembled K of one start (M x M). */
int dnlp_batch_kkt_setup(dnlp_batch *b, int64_t ns, const int32_t *slack_rows, const int32_t *jac_rows,
                         const int32_t *jac_cols, const int32_t *hess_rows, const int32_t *hess_cols);
int dnlp_batch_kkt_solve(dnlp_batch *b, int32_t count, const int32_t *starts, const double *sigma, const double *dw,
                         const double *dc, const double *rhs, double *sol, int32_t *inertia, double *wquad,
                         float *elapsed_ms);
int dnlp_batch_kkt_matrix(dnlp_batch *b, int32_t start, double *out);

/* Quasi-Newton mode (hessian_approximation = "limited-memory" of the lock-step driver): W_b is a dense damped-BFGS
 * matrix per start kept in HBM instead of the HESS output, its lower triangle packed batch fastest (entry (i, j <= i)
 * of start b at (i(i+1)/2 + j) * B + b).  dnlp_batch_kkt_setup_qn builds the scatter map from the JAC pattern, the
 * slack -1 entries and the packed W (no HESS source), allocates the K and W workspaces and sets every W_b = I; it
 * fails with a message naming B*(N+m)^2*8 and B*n(n+1)/2*8 bytes when they do not fit, or when n(n+1)/2 plus the
 * Jacobian entries exceed the int32 range.  It and dnlp_batch_kkt_setup replace each other's state.
 * dnlp_batch_kkt_solve and dnlp_batch_kkt_matrix work in both modes.
 * dnlp_batch_qn_update applies the damped BFGS update of the test-suite's stand-in to `count` distinct start ids:
 * S and Y are start-major (S[c*n + i]); applied[c] = 0 when s'Ws > 0 fails (NaN included) and W_b is left unchanged.
 * *elapsed_ms: CUDA-event time of the update's kernels.  dnlp_batch_qn_matrix copies W_b as a full n x n matrix. */
int dnlp_batch_kkt_setup_qn(dnlp_batch *b, int64_t ns, const int32_t *slack_rows, const int32_t *jac_rows,
                            const int32_t *jac_cols);
int dnlp_batch_qn_update(dnlp_batch *b, int32_t count, const int32_t *starts, const double *S, const double *Y,
                         int32_t *applied, float *elapsed_ms);
int dnlp_batch_qn_matrix(dnlp_batch *b, int32_t start, double *out);

/* ---- row-sharded evaluation across the GPUs of one node (BASELINE config 3; SURVEY.md 8e) ----
 * One process per GPU.  The reference has no counterpart (it is single-process NumPy); the surface
 * mirrors the callbacks above, evaluated collectively: every rank runs the local tape of its rows,
 * entries several ranks contribute to are summed by a one-shot all-reduce over peer memory (NVLink
 * P2P stores + flags; ncclAllReduce for payloads above 16384 doubles), entries owned by one rank are
 * stored by their owner straight into the root's copy of the global output array.
 * The caller brings its own rendezvous (any way to all-gather a few hundred bytes between the ranks). */
typedef struct dnlp_comm dnlp_comm;
typedef struct dnlp_shard dnlp_shard;
int dnlp_comm_unique_id(char *out128);                    /* rank 0: ncclGetUniqueId (libnccl is dlopen'ed) */
int dnlp_comm_create(const char *nccl_id /* 128 bytes or NULL: no NCCL */, int rank, int world, int device,
                     dnlp_comm **out);
void dnlp_comm_destroy(dnlp_comm *c);
const char *dnlp_comm_last_error(dnlp_comm *c);
int dnlp_comm_has_nccl(dnlp_comm *c);
int dnlp_comm_ipc_handle(dnlp_comm *c, char *out64);      /* cudaIpcMemHandle_t of this rank's exchange area */
int dnlp_comm_open_peers(dnlp_comm *c, const char *handles /* world x 64 bytes, rank order */);
int dnlp_comm_allreduce_host(dnlp_comm *c, double *vec, int64_t count);   /* sum over ranks, in place */

int dnlp_shard_create(dnlp_oracle *local, dnlp_comm *comm, int root, dnlp_shard **out);
void dnlp_shard_destroy(dnlp_shard *s);
const char *dnlp_shard_last_error(dnlp_shard *s);
int dnlp_shard_set_output(dnlp_shard *s, int32_t dst_space, int64_t n_shared_total, const int32_t *shared_src,
                          const int32_t *shared_global_pos, int64_t n_owned, const int32_t *owned_pos,
                          const int32_t *owned_global_pos, int64_t global_len, const double *global_const,
                          int64_t n_dyn, const int32_t *dyn_global_pos);
int dnlp_shard_root_handles(dnlp_shard *s, char *out384);           /* root: IPC handles of its global arrays */
int dnlp_shard_open_root(dnlp_shard *s, const char *handles384);    /* every rank: map them */
int dnlp_shard_set_layout(dnlp_shard *s, int32_t n_xruns, const int64_t *xsrc, const int64_t *xlen,
                          int32_t n_lruns, const int64_t *lsrc, const int64_t *llen);   /* eval then takes GLOBAL x / lambda */
int dnlp_shard_eval(dnlp_shard *s, int32_t prog, const double *x_local, const double *lam_local, double sigma,
                    double *host_out /* root only */);
int dnlp_shard_run_device(dnlp_shard *s, int32_t prog_mask, int32_t iters, float *elapsed_ms);

/* Shared-host delivery of a sharded output (csrc/dnlp_shard.cu): the global output array lives in one POSIX
 * shared-memory segment page-locked by every rank; each GPU copies the runs it owns into it over its own
 * PCIe link and host-side epoch counters (the control segment) tell every rank when all slices have landed,
 * so EVERY rank's callback returns the full global array.  Only for outputs without summed entries whose
 * owned entries form contiguous runs; every rank must make the same sequence of dnlp_shard_eval calls.
 * `create` = 1 on exactly one rank, which returns before the others attach; after all have attached the
 * creator removes the names (dnlp_shard_share_unlink).  *host_array stays valid after dnlp_shard_destroy, until
 * dnlp_shard_share_release.  The reference has no counterpart: it evaluates the
 * whole problem in one process (cvxpy/reductions/solvers/nlp_solvers/nlp_solver.py:200-377). */
int dnlp_shard_share_control(dnlp_shard *s, const char *shm_name, int32_t create);
int dnlp_shard_share_output(dnlp_shard *s, int32_t dst_space, const char *shm_name, int32_t create, int64_t n_runs,
                            const int64_t *local_start, const int64_t *global_start, const int64_t *length,
                            double **host_array);
int dnlp_shard_share_unlink(const char *shm_name);
int dnlp_shard_share_reset(dnlp_shard *s);      /* a peer could not attach: back to the device-side route */
/* Worker loop: only the root runs the solver (the reference drives its callbacks from one cyipopt.Problem,
 * ipopt_nlpif.py:143-170).  The root posts every callback - program id (-1: leave the loop), x, lambda, sigma -
 * into shared host memory before it evaluates; the other ranks block in dnlp_shard_wait_command (0 = command
 * received, 2 = timeout_s passed, call again, 1 = a rank failed) and then make the same dnlp_shard_eval call on the
 * shared copies *x_host / *lam_host - or with NULL for a vector the flags report as unchanged since the previous
 * command (dnlp_shard_eval then keeps the point / multipliers it has, no compare). */
int dnlp_shard_share_inputs(dnlp_shard *s, const char *shm_x, const char *shm_lam, int32_t create, int64_t n_global,
                            int64_t m_global, double **x_host, double **lam_host);
int dnlp_shard_post_command(dnlp_shard *s, int32_t prog, const double *x, const double *lam, double sigma,
                            int32_t force, int32_t *flags);   /* *flags: 1 = x changed | 2 = lambda changed */
int dnlp_shard_wait_command(dnlp_shard *s, double timeout_s, int32_t *prog, double *sigma, int32_t *flags);
int dnlp_shard_share_release(double *host_array, int64_t count);   /* unpin + unmap; the array outlives dnlp_shard_destroy */

#ifdef __cplusplus
}
#endif
#endif /* DNLP_B200_H */
