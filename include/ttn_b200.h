/*
 * ttn_b200.h — C ABI of libttn_b200.so: the B200 (sm_100a) implementation of TensorTrainNumerics.jl's
 * core-contraction hot path.
 *
 * The reference (pure Julia, v1.1.3) has no FFI of its own; this header defines the boundary its hot-path
 * methods bind to through `ccall` (see INTEGRATION.md for the Julia shim).  Every entry point names the
 * reference function it replaces (file:line relative to the reference repository root).
 *
 * Conventions
 *  - All functions return an int status: 0 = ok, else one of the TTN_E* codes; ttn_last_error() gives the text.
 *    No C++ exception crosses this boundary.  Status -> reference exception mapping:
 *      TTN_EDIM      AssertionError("Incompatible dimensions")   src/tt_operations.jl:11,102
 *      TTN_ECENTER   DimensionMismatch("Impossible orthogonalization")  src/tt_tools.jl:513
 *      TTN_EARG      AssertionError (sweeps >= 1, k in 1:N-1)     src/tt_tools.jl:744,773
 *      TTN_ESCHED    AssertionError("Sweep schedule error")       src/solvers/dmrg.jl:513, als.jl:263, mals.jl:347
 *      TTN_ECUDA     ErrorException(ttn_last_error())
 *  - dtype: TTN_F64 (Julia Float64) or TTN_C128 (Julia ComplexF64, interleaved re/im = cuDoubleComplex).
 *  - Host arrays are dense column-major exactly as Julia stores them:
 *      TT core  X_k[s,a,b]   of size (n_k, r_{k-1}, r_k):        ptr[s + n*(a + r_{k-1}*b)]      src/tt_tools.jl:23-29
 *      MPO core A_k[i,j,a,b] of size (n_k, n_k, R_{k-1}, R_k):   ptr[i + n*(j + n*(a + R_{k-1}*b))]  src/tt_tools.jl:48-54
 *  - Host memory stays owned by the caller; the library copies in/out and owns all device memory behind the
 *    opaque handles, so whole sweeps run without host round trips of tensor data.
 *  - One context per HOST THREAD: every thread that calls the library owns a compute stream, a copy stream, an allocation
 *    cache and its own counters, and must call ttn_init itself.  Calls are blocking for their thread.  Handles are used and
 *    released by the thread that created them (an uploaded operator may be READ by several threads).  Two threads working on
 *    independent trains overlap on the GPU.  One process drives one GPU.
 *  - There is no CPU fallback: without a CUDA device ttn_init fails with TTN_ECUDA.
 */
#ifndef TTN_B200_H
#define TTN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TTN_OK 0
#define TTN_EDIM 1
#define TTN_EARG 2
#define TTN_ECENTER 3
#define TTN_ESCHED 4
#define TTN_ENOTCONV 5
#define TTN_ECUDA 6
#define TTN_EINTERNAL 7

#define TTN_F64 0
#define TTN_C128 1

typedef struct ttn_ttv_s* ttn_ttv; /* device-resident TTvector  (src/tt_tools.jl:23-29)  */
typedef struct ttn_tto_s* ttn_tto; /* device-resident TToperator (src/tt_tools.jl:48-54) */

/* ---- library lifetime ------------------------------------------------------------------------------ */
int ttn_init(int device);                 /* selects the device, creates the calling thread's stream and memory cache */
int ttn_shutdown(void);
const char* ttn_last_error(void);
int ttn_version(void);
int ttn_synchronize(void);
long long ttn_launch_count(void);         /* kernels launched by the library since ttn_reset_launch_count */
int ttn_reset_launch_count(void);
void* ttn_stream(void);                   /* cudaStream_t the library launches on (for event timing) */
/* per-kernel-family CUDA-event timing on the library stream (bench.py's roofline pass; adds two event records per launch).
 * families: 0 gemm, 1 copy/permute, 2 apply, 3 qr panel, 4 qr reflector apply, 5 jacobi, 6 reductions/axpy, 7 gather/norms */
#define TTN_NFAMILIES 8
/* run-time switches between two live paths on the same input (for tests that compare them): "gram_compress" (1: Gram path
 * of tt_compress! for truncerr == 0, csrc/heig.cu), "gram_jacobi_min" (columns from which the Gram-block Jacobi serves large
 * SVDs), "gemm_bulk" (1: TMA-staged Float64 big tile when the operands allow it), "gemm_thin" (1: streaming kernel for
 * right-multiplications with N, K <= 32); "reset_flops" clears the flop counters; read-only counters through
 * ttn_get_option: "gemm_flops", "heig_flops", "gram_calls", "gram_fallbacks", "gram_last_flags".  Per host thread, like the context. */
int ttn_set_option(const char* key, double value);
int ttn_get_option(const char* key, double* value);
int ttn_last_jacobi_sweeps(void);        /* diagnostics: sweeps of the most recent Jacobi SVD */
int ttn_profile(int enable);              /* clears the records and switches profiling on/off */
int ttn_profile_read(double* ms /* 8 */, long long* counts /* 8 */);

/* ---- containers -------------------------------------------------------------------------------------- */
/* TTvector(N, ttv_vec, ttv_dims, ttv_rks, ttv_ot): rks has d+1 entries, ot d entries (may be NULL = zeros).
 * `batch` > 1 uploads `batch` TTs of identical dims/ranks; cores[k] then points to (n, r_l, r_r, batch). */
int ttn_ttv_upload(int dtype, int d, const int64_t* dims, const int64_t* rks, const int64_t* ot,
                   const void* const* cores, int batch, ttn_ttv* out);
/* Asynchronous variants for pipelines over batches of trains (cfg5): the copies run on the library's copy stream and overlap
 * the compute stream.  Host buffers must be page-locked and stay valid until the copy has completed.  A handle returned by
 * ttn_ttv_upload_async may be passed to ttn_apply / ttn_apply_compress / ttn_compress / ttn_ttv_download(_async) / ttn_ttv_free
 * right away (they make the compute stream wait for the upload); before any other entry point call ttn_ttv_wait.  After
 * ttn_ttv_download_async the host buffers are valid once ttn_copy_synchronize has returned; ttn_ttv_free may be called at once
 * (the release is ordered after the copy). */
int ttn_ttv_upload_async(int dtype, int d, const int64_t* dims, const int64_t* rks, const int64_t* ot,
                         const void* const* cores, int batch, ttn_ttv* out);
int ttn_ttv_wait(ttn_ttv x);
int ttn_ttv_download_async(ttn_ttv x, void* const* cores);
int ttn_copy_synchronize(void);
int ttn_ttv_info(ttn_ttv x, int* dtype, int* d, int* batch);
int ttn_ttv_ranks(ttn_ttv x, int64_t* rks /* d+1 */);
int ttn_ttv_dims(ttn_ttv x, int64_t* dims /* d */);
int ttn_ttv_ot(ttn_ttv x, int64_t* ot /* d */);
int ttn_ttv_download(ttn_ttv x, void* const* cores);
int ttn_ttv_copy(ttn_ttv x, ttn_ttv* out);                       /* Base.copy, src/tt_tools.jl:172-178 */
int ttn_ttv_complex(ttn_ttv x, ttn_ttv* out);                    /* Base.complex, src/tt_tools.jl:63-65 */
int ttn_ttv_free(ttn_ttv x);
int ttn_tto_upload(int dtype, int d, const int64_t* dims, const int64_t* rks, const void* const* cores, ttn_tto* out);
int ttn_tto_complex(ttn_tto A, ttn_tto* out);                    /* Base.complex, src/tt_tools.jl:59-61 */
int ttn_tto_info(ttn_tto A, int* dtype, int* d);
int ttn_tto_ranks(ttn_tto A, int64_t* rks /* d+1 */);            /* tto_rks, src/tt_tools.jl:52 */
int ttn_tto_dims(ttn_tto A, int64_t* dims /* d */);              /* tto_dims, src/tt_tools.jl:51 */
int ttn_tto_download(ttn_tto A, void* const* cores);             /* cores back as (n_k, n_k, R_{k-1}, R_k) column-major, src/tt_tools.jl:50 */
int ttn_tto_free(ttn_tto A);

/* ---- TT algebra -------------------------------------------------------------------------------------- */
/* y = A * x                      *(A::TToperator, v::TTvector), src/tt_operations.jl:101-111 */
int ttn_apply(ttn_tto A, ttn_ttv x, ttn_ttv* y);
/* dot(a, b) (conj on a), out = {re, im} per batch element     src/tt_operations.jl:239-250 */
int ttn_dot(ttn_ttv a, ttn_ttv b, double* out);
/* norm(a) per batch element                                     src/tt_operations.jl:465-470 */
int ttn_norm(ttn_ttv a, double* out);
/* z = x + y                                                     src/tt_operations.jl:10-35 */
int ttn_add(ttn_ttv x, ttn_ttv y, ttn_ttv* z);
/* y = (re + i*im) * x  (scales the first core with ot == 0)     src/tt_operations.jl:256-266 */
int ttn_scale(ttn_ttv x, double re, double im, ttn_ttv* y);

/* ---- canonicalisation and rounding ------------------------------------------------------------------- */
/* y = orthogonalize(x; i = center), center is 1-based          src/tt_tools.jl:511-543 */
int ttn_orthogonalize(ttn_ttv x, int center, ttn_ttv* y);
/* tt_compress!(x, max_bond; truncerr, sweeps): in place.       src/tt_tools.jl:772-789 with the `_svdtrunc`
 * method of src/tt_cross_interpolation.jl:149-166.  The reference's discarded orthogonalize (tt_tools.jl:769)
 * is not executed.  sigma_out (optional, may be NULL) receives, for batch element 0, the retained singular
 * values of every bond step, each step padded to `sigma_stride` doubles (2*(d-1)*sweeps steps). */
int ttn_compress(ttn_ttv x, int64_t max_bond, double truncerr, int sweeps, double* sigma_out, int64_t sigma_stride);
/* y = tt_compress!(A * x, max_bond; truncerr, sweeps): `*(A, v)` (src/tt_operations.jl:101-111) fused into the first pass of
 * `tt_compress!` (src/tt_tools.jl:772-789).  With truncerr == 0 the product cores (n, R r, R' r') are consumed by the two-site
 * merges without being written to memory; results equal ttn_apply followed by ttn_compress (same sigma_out layout). */
int ttn_apply_compress(ttn_tto A, ttn_ttv x, int64_t max_bond, double truncerr, int sweeps, double* sigma_out, int64_t sigma_stride,
                       ttn_ttv* y);
/* _tt_bond_truncate!(x, k; max_bond, truncerr), k 1-based; mutates x; if y != NULL also returns
 * orthogonalize(x; i = k) as the reference does.                src/tt_tools.jl:743-770 */
int ttn_bond_truncate(ttn_ttv x, int k, int64_t max_bond, double truncerr, ttn_ttv* y);

/* ---- site surgery: the other users of the two-site truncated split (single trains, in place) ----------
 * `mode` selects the rank rule of the caller: 0 = keep sigma_j > tol * sigma_1 (all if tol <= 0), the rule of
 * `_swap_adjacent_sites` / `to_qtt` (src/qtt_tools.jl:680-685, 286-289); 1 = the `_svdtrunc` tail-norm rule with
 * the `max_bond` cap (src/tt_cross_interpolation.jl:149-166) used by `_ttm_swap!`.  Split: U | S*Vt. */
/* _swap_adjacent_sites(cores[k], cores[k+1]; threshold)   src/qtt_tools.jl:660-694  (driver `reorder`, :731-774)
 * _ttm_swap!(cores, rks, k; tol, rmax)                     src/tt_operations.jl:366-383
 * Contracts sites k, k+1 (1-based), exchanges their physical indices and re-factorises. */
int ttn_swap_sites(ttn_ttv x, int k, int mode, int64_t max_bond, double tol);
/* _ttm_contract!(cores, rks, k): core_k[s] <- core_k[s] * core_{k+1}[s], site k+1 removed (equal physical dims).
 *                                                          src/tt_operations.jl:385-397 */
int ttn_merge_sites_diag(ttn_ttv x, int k);
/* one split of `to_qtt`: site k with n_k = coarse * fine becomes sites (coarse, fine), s = fine_idx + coarse_idx * fine.
 *                                                          src/qtt_tools.jl:270-298 */
int ttn_split_site(ttn_ttv x, int k, int64_t coarse, int mode, int64_t max_bond, double tol);

/* ---- alternating solvers ----------------------------------------------------------------------------- */
typedef struct {
  int N;                       /* window size for dmrg_* (1 or 2); ignored by als/mals */
  double tol;                  /* SVD truncation tolerance (mals: sv_trunc, dmrg: cut_off_index) */
  const int64_t* sweep_schedule; int n_sweep_schedule;
  const int64_t* rmax_schedule;  int n_rmax_schedule;
  int64_t rmax;                /* mals_linsolve rmax */
  int sweep_count;             /* als_linsolve: number of half sweeps (src/solvers/als.jl:198-222) */
  int it_solver;               /* linear local problems: 0 = dense direct solve (K_full + `\`, as the reference) while the
                                * window has at most max(itslv_thresh, 2048) unknowns, matrix-free GMRES beyond; 1 = always GMRES */
  int linsolv_maxiter;         /* Krylov iteration cap per local solve */
  double linsolv_tol;          /* Krylov tolerance per local solve */
  int itslv_thresh;            /* see it_solver (dmrg.jl:92-177); eigen problems are always solved by Lanczos */
  int krylovdim;               /* Lanczos / GMRES subspace size (KrylovKit default 30) */
  int symmetrize;              /* dmrg_*: apply 0.5*(K + K^T) like src/solvers/dmrg.jl:241 (1) or K only (0) */
} ttn_solver_params;
int ttn_solver_params_default(ttn_solver_params* p);

/* als_linsolve(A, b, x0; sweep_count)            src/solvers/als.jl:161-225;  residual (optional) = ||Ax-b||/||b|| */
int ttn_als_linsolve(ttn_tto A, ttn_ttv b, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* residual);
/* als_eigsolve(A, x0; sweep_schedule, rmax_schedule)  src/solvers/als.jl:251-321;  E: capacity cap_E, n_E written */
int ttn_als_eigsolve(ttn_tto A, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* E, int cap_E, int* n_E);
/* als_gen_eigsolv(A, S, x0; sweep_schedule, rmax_schedule): lowest pair of A x = lambda S x, S Hermitian positive definite.
 * The local pencil is solved densely as the reference's K_eiggenmin does (src/solvers/als.jl:89-102, driver :344-440). */
int ttn_als_gen_eigsolv(ttn_tto A, ttn_tto S, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* E, int cap_E, int* n_E);
/* mals_linsolve(A, b, x0; tol, rmax)             src/solvers/mals.jl:240-309 */
int ttn_mals_linsolve(ttn_tto A, ttn_ttv b, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* residual);
/* mals_eigsolve(A, x0; tol, sweep_schedule, rmax_schedule)   src/solvers/mals.jl:335-425 */
int ttn_mals_eigsolve(ttn_tto A, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* E, int64_t* r_hist, int cap_E,
                      int* n_E);
/* dmrg_linsolve(A, b, x0; N, tol, sweep_schedule, rmax_schedule)   src/solvers/dmrg.jl:385-473 */
int ttn_dmrg_linsolve(ttn_tto A, ttn_ttv b, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* residual);
/* dmrg_eigsolve(A, x0; N, tol, sweep_schedule, rmax_schedule)      src/solvers/dmrg.jl:501-578 */
int ttn_dmrg_eigsolve(ttn_tto A, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* E, int64_t* r_hist, int cap_E,
                      int* n_E);

typedef struct {
  int two_site;                /* 0: tdvp (src/solvers/tdvp.jl:154-203), 1: tdvp2 (:303-357) */
  const double* steps; int n_steps;
  int normalize, sweeps, imaginary_time;
  int64_t max_bond; double truncerr;      /* tdvp2 only */
  int krylovdim; double krylov_tol; int krylov_maxiter;   /* KrylovKit.exponentiate stand-in */
} ttn_tdvp_params;
int ttn_tdvp_params_default(ttn_tdvp_params* p);
int ttn_tdvp(ttn_tto H, ttn_ttv u0, const ttn_tdvp_params* p, ttn_ttv* u);

/* ---- kernel-level entry points (parity tests, benchmarks) -------------------------------------------- */
/* strided-batched GEMM on device pointers: C = alpha*op(A)*op(B) + beta*C  (element strides; batch strides bA/bB/bC, 0 for an
   operand shared by the whole batch).  Any batch >= 1 is accepted: beyond 65535 products it runs as several launches. */
int ttn_gemm(int dtype, int M, int N, int K, const void* A, int64_t sAm, int64_t sAk, int conjA, const void* B, int64_t sBk,
             int64_t sBn, int conjB, void* C, int64_t sCm, int64_t sCn, double alpha, double beta, int batch, int64_t bA,
             int64_t bB, int64_t bC);
/* two-site effective-operator matvec  Y[a,b,c] = sum G[y,a,d] Amid[y,b,e,z] V[d,e,f] H[z,c,f]  on HOST arrays in the
 * reference layouts (src/solvers/dmrg.jl:239-244); symmetrize as in ttn_solver_params. */
int ttn_matvec2_host(int dtype, int w_l, int w_r, int chi_l, int chi_r, int nn, const void* G, const void* Amid, const void* H,
                     const void* V, void* Y, int symmetrize);
/* device-resident matvec for benchmarking: prepare once, apply many times */
typedef struct ttn_matvec_s* ttn_matvec;
int ttn_matvec2_create(int dtype, int w_l, int w_r, int chi_l, int chi_r, int nn, const void* G, const void* Amid,
                       const void* H, ttn_matvec* out);
int ttn_matvec2_apply(ttn_matvec mv, const void* V_dev, void* Y_dev);   /* device pointers, (chi_l, nn, chi_r) */
int ttn_matvec2_free(ttn_matvec mv);
/* ---- the same matvec sharded over the GPUs of one NVLink node (one process per GPU; SURVEY.md section 8(e)) ----------
 * Rank `rank` of `nranks` owns the slice c in [c0, c0+cp) of the right environment's bra index (ttn_shard_range) and
 * computes Y[:, :, c0:c0+cp] with no reduction; the epilogue of its last GEMM stores the tiles into the result
 * buffers of every peer (P2P over NVLink), so after ttn_shard_matvec_apply the complete vector is resident on every
 * rank (stream-ordered).  Peer buffers are exchanged as CUDA IPC handles: each rank calls _handles (192 bytes: two
 * result buffers + the epoch flags), the host side all-gathers them (MPI.jl / torch.distributed) and calls _bind with
 * the nranks x 192 bytes in rank order.  Without _bind (or nranks == 1) only the local slice is written.
 * G, Amid, H are HOST arrays in the reference layouts (dmrg.jl:27-46); every rank passes the full arrays. */
typedef struct ttn_shard_matvec_s* ttn_shard_matvec;
int ttn_shard_range(int chi, int rank, int nranks, int* c0, int* cp);
int ttn_shard_matvec_create(int dtype, int w_l, int w_r, int chi_l, int chi_r, int nn, const void* G, const void* Amid,
                            const void* H, int rank, int nranks, ttn_shard_matvec* out);
int ttn_shard_matvec_handles(ttn_shard_matvec mv, void* handles192);
int ttn_shard_matvec_bind(ttn_shard_matvec mv, const void* all_handles);
/* *Y_dev: library-owned full vector.  The exchange waits for every peer's epoch flag for at most TTN_SHARD_TIMEOUT_S
 * seconds (default 60); after a timeout the sticky error of ttn_shard_matvec_error is set and Y is INVALID — callers of
 * this kernel-level entry point must poll it before consuming Y (ttn_shard_eigsolve checks it itself and fails with
 * TTN_ECUDA). */
int ttn_shard_matvec_apply(ttn_shard_matvec mv, const void* V_dev, void** Y_dev);
/* lowest eigenpair of the sharded operator (KrylovKit.eigsolve(..., :SR) stand-in, dmrg.jl:245): x_dev start vector in,
 * eigenvector out (identical on every rank); the Lanczos recurrence is replicated, only the matvec is distributed */
int ttn_shard_eigsolve(ttn_shard_matvec mv, void* x_dev, int krylovdim, int maxiter, double tol, double* theta, int* matvecs);
int ttn_shard_matvec_slice(ttn_shard_matvec mv, int* c0, int* cp);
int ttn_shard_matvec_error(ttn_shard_matvec mv, int* err);    /* 1 if an epoch wait timed out (a peer died) */
int ttn_shard_matvec_free(ttn_shard_matvec mv);

/* ---- DMRG over several GPUs of one node (one process per GPU): the sweep of src/solvers/dmrg.jl:501-578 runs replicated
 * on every rank (identical data, environment updates and two-site SVDs replicated), the Lanczos matvec of every bond step
 * (dmrg.jl:239-245) is sharded on the bra index of the right environment and exchanged through the fused all-gather
 * epilogue over NVLink peer memory.  The exchange buffers live in a context created ONCE (max_elems >= chi_max^2 n^N
 * elements), exported as 2 x 192 bytes of CUDA IPC handles and bound to the handles of all ranks (rank-major). */
typedef struct ttn_shard_ctx_s* ttn_shard_ctx;
int ttn_shard_ctx_create(int dtype, int64_t max_elems, int rank, int nranks, ttn_shard_ctx* out);
int ttn_shard_ctx_handles(ttn_shard_ctx c, void* handles384);
int ttn_shard_ctx_bind(ttn_shard_ctx c, const void* all_handles);
int ttn_shard_ctx_free(ttn_shard_ctx c);
int ttn_dmrg_eigsolve_sharded(ttn_tto A, ttn_ttv x0, const ttn_solver_params* p, ttn_shard_ctx sc, ttn_ttv* x, double* E,
                              int64_t* r_hist, int cap_E, int* n_E);
/* environment updates on HOST arrays, reference layouts (src/solvers/dmrg.jl:27-35) */
int ttn_env_left_host(int dtype, int n, int w_l, int w_r, int r_l, int r_r, const void* G, const void* x, const void* A,
                      void* Gout);
int ttn_env_right_host(int dtype, int n, int w_l, int w_r, int r_l, int r_r, const void* H, const void* x, const void* A,
                       void* Hout);
/* truncated SVD of a host matrix (column-major m x n): `_svdtrunc` src/tt_cross_interpolation.jl:149-166.
 * Returns U (m x r), s (r), Vt (r x n) into caller buffers sized for r = min(m,n); *r_out = retained rank. */
int ttn_svdtrunc_host(int dtype, int m, int n, const void* A, int64_t max_bond, double truncerr, void* U, double* s, void* Vt,
                      int* r_out);
/* thin QR of a host matrix (column-major m x n): Q (m x k), R (k x n), k = min(m,n) */
/* Top `nev` eigenpairs (descending) of `batch` Hermitian PSD matrices G (n x n column-major each, host): the engine of the
 * Gram path of tt_compress! (csrc/heig.cu; replaces `svd` of src/tt_cross_interpolation.jl:150 when truncerr == 0).
 * flags[b] != 0: the fast path declines this matrix (clusters / accuracy), callers fall back to the Jacobi SVD. */
int ttn_heig_host(int dtype, int n, int nev, int batch, const void* G, double* lam, void* U, int* flags);
int ttn_qr_host(int dtype, int m, int n, const void* A, void* Q, void* R);
/* The truncation rules of the path on a host spectrum `s` (sorted descending, `len` values); pure host code, callable without
 * a device.  rule 0: `_svdtrunc` tail-norm rule + `max_bond` cap (src/tt_cross_interpolation.jl:149-166); 1: `sv_trunc`
 * (src/solvers/mals.jl:42-56), number of retained values; 2: `cut_off_index` (src/solvers/dmrg.jl:179-185); 3: relative
 * threshold `s_j > tol * s_1` (src/qtt_tools.jl:680-685). */
int ttn_rank_rule(int rule, const double* s, int len, double tol, int64_t max_bond, int* r);
/* r_and_d_to_rks(rks, dims; rmax), src/tt_tools.jl:407-425 (host; `rks` and `out` hold d + 1 values) */
int ttn_r_and_d_to_rks(const int64_t* rks, const int64_t* dims, int d, int64_t rmax, int64_t* out);

/* device memory helpers for benchmarks */
int ttn_dev_alloc(size_t bytes, void** out);
int ttn_dev_free(void* p);
int ttn_h2d(void* dst, const void* src, size_t bytes);
int ttn_d2h(void* dst, const void* src, size_t bytes);

#ifdef __cplusplus
}
#endif
#endif /* TTN_B200_H */
