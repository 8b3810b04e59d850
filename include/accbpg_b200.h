/*
 * accbpg_b200.h -- C ABI of the B200-native accbpg hot path (libaccbpg_b200.so).
 *
 * The reference (DredderGun/accbpg_and_fw) is pure Python/NumPy and has no FFI:
 * its boundary is the duck-typed operator protocol between the driver loops and
 * the f / h / lmo objects (accbpg/functions.py:10-24, :199-235,
 * accbpg/functions_lmo.py:137-160).  Each entry point below replaces the NumPy
 * body of one of those operator methods; the citation next to it is the
 * reference code it stands in for.  INTEGRATION.md shows the ctypes stub a
 * maintainer of the reference would add to route the method to the entry point.
 *
 * Conventions
 *   - every `const double*` / `double*` named d_* or documented "device" is a
 *     device pointer to IEEE float64; matrices are row-major (C order) with an
 *     explicit leading dimension in elements;
 *   - `stream` is a cudaStream_t passed as void*; nothing synchronises except
 *     accbpg_ctx_read(), so results that are host scalars in the reference are
 *     written to a device slot (`d_out`) and fetched with accbpg_ctx_read();
 *   - data-dependent failures that the reference raises as AssertionError /
 *     ValueError are reported as bits OR-ed into the context's status word
 *     (ACCBPG_ST_*), fetched by the same accbpg_ctx_read();
 *   - return value: 0 ok, ACCBPG_E_ARG bad argument, ACCBPG_E_CUDA a CUDA call
 *     failed (text from accbpg_last_error());
 *   - no entry point allocates device memory except accbpg_ctx_create();
 *     matrix-sized scratch is caller-provided after a *_workspace_bytes() query;
 *   - all reductions use a fixed tree (no floating-point atomics): results are
 *     bit-reproducible run to run for a given shape and GPU.
 */
#ifndef ACCBPG_B200_H
#define ACCBPG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ACCBPG_ABI_VERSION 7

/* return codes */
#define ACCBPG_OK      0
#define ACCBPG_E_ARG   1
#define ACCBPG_E_CUDA  2

/* status bits (device-side precondition checks of the reference) */
#define ACCBPG_ST_X_NEGATIVE     0x001u  /* DOptimalObj: x.min() >= 0            functions.py:45  */
#define ACCBPG_ST_NOT_PD         0x002u  /* slogdet sign <= 0 -> ValueError      functions.py:49  */
#define ACCBPG_ST_ARG_NOT_POS    0x004u  /* Burg: x.min()>0, y.min()>0           functions.py:243,252,270 */
#define ACCBPG_ST_PROX_NOT_POS   0x008u  /* Burg prox: g.min()>0 / >-lamda       functions.py:261,296 */
#define ACCBPG_ST_ARG_NEGATIVE   0x010u  /* Shannon: x.min()>=0, y.min()>=0      functions.py:406,419,436 */
#define ACCBPG_ST_Y_NOT_POS      0x020u  /* ShannonSimplex div_prox: y.min()>0   functions.py:488 */
#define ACCBPG_ST_NEWTON_MAXIT   0x040u  /* Burg-simplex root-find hit the iteration guard (never in the reference) */

/* ---- library ---------------------------------------------------------- */
int         accbpg_abi_version(void);
const char* accbpg_last_error(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
uint64_t    accbpg_launch_count(void);

/* optional per-kernel timing with CUDA events on the launching stream (bench.py's roofline line).
 * ids 0..accbpg_prof_count()-1, names from accbpg_prof_name(); prof_read waits for the recorded events,
 * returns the summed duration and the number of bracketed launches since the last read, and resets them. */
int         accbpg_prof_enable(int on);
int         accbpg_prof_count(void);
const char* accbpg_prof_name(int id);
int         accbpg_prof_read(int id, double* total_ms, int64_t* count);

/* ---- context: small device scratch (reduction partials, 256 scalar slots,
 *      status word) + pinned host mirror.  One per device/thread of control. */
int     accbpg_ctx_create(void** ctx);
int     accbpg_ctx_destroy(void* ctx);
double* accbpg_ctx_slots(void* ctx);            /* device pointer to 256 float64 result slots */
int     accbpg_ctx_sm_count(void* ctx);
/* copy count (<= 256) float64 results from device address d_src (the context's slots or any
 * caller-owned device buffer the kernels were told to write to) and the status word to the
 * host through pinned memory, wait for the stream, clear the status word.  This is the only
 * synchronising entry point.  d_src / h_out may be NULL when count == 0. */
int     accbpg_ctx_read(void* ctx, void* stream, const double* d_src, int count,
                        double* h_out, uint32_t* h_status);

/* Deferred form of accbpg_ctx_read: _async enqueues the copy (and the read-and-clear of the status word) behind the
 * work already on the stream and returns a ticket; _wait blocks until that copy has landed.  The drivers use it to
 * enqueue iteration k+1 while iteration k is still running, so the GPU never waits for the host between iterations.
 * At most ACCBPG_READ_RING tickets may be outstanding; tickets are reused round-robin. */
#define ACCBPG_READ_RING 8
int     accbpg_ctx_read_async(void* ctx, void* stream, const double* d_src, int count, int* ticket);
int     accbpg_ctx_read_wait(void* ctx, int ticket, int count, double* h_out, uint32_t* h_status);

/* ---- iterate arithmetic inlined in the drivers (accbpg/algorithms.py:147,150,
 *      243,250,369,374,478,483; np.dot at :53,168,260,279,387,406;
 *      algorithms_fw.py:39,231) ---------------------------------------- */
/* out = a*x + b*y  (two rounded products, one rounded add: same as NumPy) */
int accbpg_vec_axpby(void* ctx, void* stream, int64_t n, double a, const double* d_x,
                     double b, const double* d_y, double* d_out);
/* out = x + a*(s - x)   algorithms_fw.py:34,54,231 */
int accbpg_vec_step_toward(void* ctx, void* stream, int64_t n, const double* d_x,
                           const double* d_s, double a, double* d_out);
int accbpg_vec_dot(void* ctx, void* stream, int64_t n, const double* d_x, const double* d_y, double* d_out);
/* d_out = dot(g, a - b) without the temporary */
int accbpg_vec_dot_diff(void* ctx, void* stream, int64_t n, const double* d_g, const double* d_a,
                        const double* d_b, double* d_out);
/* d_out = sum (a - b)^2: ||s - x||^2 of the (L0,L1) Frank-Wolfe step rules (algorithms_fw.py:297, :396) */
int accbpg_vec_sqdist(void* ctx, void* stream, int64_t n, const double* d_a, const double* d_b, double* d_out);
int accbpg_vec_sum(void* ctx, void* stream, int64_t n, const double* d_x, double* d_out);
/* d_out[0] = min(x), d_out[1] = max(x) */
int accbpg_vec_minmax(void* ctx, void* stream, int64_t n, const double* d_x, double* d_out);
/* d_out[0] = value, d_out[1] = (double) first index attaining it; want_max = 0 argmin, 1 argmax */
int accbpg_vec_argext(void* ctx, void* stream, int64_t n, const double* d_x, int want_max, double* d_out);

/* out (p x q, row-major) = u v^T: the rank-one vertex of lmo_nuclear_norm_ball (functions_lmo.py:4-13) */
int accbpg_mat_outer(void* ctx, void* stream, int64_t p, const double* d_u, int64_t q, const double* d_v, double* d_out);

/* ---- Burg entropy kernels  h(x) = -sum log x   (accbpg/functions.py:238-356) */
#define ACCBPG_BURG_PLAIN   0   /* BurgEntropy.prox_map        functions.py:255-262 */
#define ACCBPG_BURG_L1      1   /* BurgEntropyL1.prox_map      functions.py:290-298 */
#define ACCBPG_BURG_L2      2   /* BurgEntropyL2.prox_map      functions.py:316-323 */
int accbpg_burg_value(void* ctx, void* stream, int64_t n, const double* d_x, double* d_out);        /* :242-244 */
int accbpg_burg_gradient(void* ctx, void* stream, int64_t n, const double* d_x, double* d_out_vec); /* :246-248 */
int accbpg_burg_divergence(void* ctx, void* stream, int64_t n, const double* d_x, const double* d_y,
                           double* d_out);                                                          /* :250-253 */
/* prox_map(g, L) when d_y == NULL, div_prox_map(y, g, L) = prox_map(g - L*(-1/y), L) otherwise (:264-271) */
int accbpg_burg_prox(void* ctx, void* stream, int64_t n, int kind, double lamda,
                     const double* d_y, const double* d_g, double L, double* d_out_vec);
/* BurgEntropySimplex.prox_map / inherited div_prox_map (functions.py:336-356): one persistent kernel replays cmin,
 * bisection and Newton with the iterate in registers; the grid-wide sums of a step go through a slot table (every block
 * gathers the block partials itself, or above 128 blocks a leader block adds them and posts the total in one slot;
 * value + round token per 16-byte store, block-order adds): no host round trip and no grid barrier per Newton step.
 * d_info (3 slots, may be NULL): bisection steps, Newton steps, final c. */
int accbpg_burg_simplex_prox(void* ctx, void* stream, int64_t n, const double* d_y, const double* d_g,
                             double L, double eps, double* d_out_vec, double* d_info);
/* column-sharded building block of the same root-find, on one rank's slice:
 * d_gg = (g [+ L/y]) / L, d_out[0] = min(gg). */
int accbpg_burg_simplex_prepare(void* ctx, void* stream, int64_t n, const double* d_y, const double* d_g,
                                double L, double* d_gg, double* d_out);
/* the same root-find without a host round trip: every rank all-gathers the slices of gg (padding entries +inf),
 * runs the whole recurrence of functions.py:341-356 on the gathered vector with the kernel of accbpg_burg_simplex_prox
 * -- the result does not depend on how the columns are sharded -- and finishes its own slice, out = 1/(gg + c), with
 * the c left on the device.  d_info (3 slots): bisection steps, Newton steps, c. */
int accbpg_burg_simplex_root(void* ctx, void* stream, int64_t n, const double* d_gg, double eps, double* d_info);
int accbpg_burg_simplex_finish_dev(void* ctx, void* stream, int64_t n, const double* d_gg, const double* d_c,
                                   double* d_out_vec);
/* The column-sharded prox with the gather over NVLink peer memory instead of an NCCL all-gather, in two calls.
 * push: the preparing kernel stores this rank's slice of gg = (g [+ L/y]) / L (d_y may be NULL), padded with +inf up to
 * `width`, into segment `rank` of EVERY rank's gathered vector (and into d_gg_local for
 * accbpg_burg_simplex_finish_dev) and releases a flag word on every rank.  root: a one-warp kernel waits for the
 * `world` flags, then the recurrence of functions.py:341-356 runs on the gathered world*width vector exactly as in
 * accbpg_burg_simplex_root (d_info likewise).  peer_gg / peer_flags: host arrays of `world` device pointers to every
 * rank's symmetric buffers (2*world*width doubles, double-buffered on the epoch's parity; world uint64, zeroed once);
 * epoch 1, 2, 3, ... per push/root pair on these buffers, the same on every rank. */
int accbpg_burg_simplex_push_peer(void* ctx, void* stream, int64_t n_local, int64_t width, const double* d_y,
                                  const double* d_g, double L, int rank, int world, void* const* peer_gg,
                                  void* const* peer_flags, uint64_t epoch, double* d_gg_local);
int accbpg_burg_simplex_root_peer(void* ctx, void* stream, int64_t width, double eps, int rank, int world,
                                  void* const* peer_gg, void* const* peer_flags, uint64_t epoch, double* d_info);
/* Sum `count` (<= 15) per-rank partial scalars at d_in over the ranks through peer memory, in rank order, into d_out
 * (may equal d_in) (the batched divergence / dot-product partials of a driver iteration, algorithms.py:53,153-154,...):
 * one small kernel instead of an NCCL all-reduce.  The exchange also carries every rank's status word and ORs them into
 * the local one, so an assertion of the reference that fails on one rank's slice is raised on every rank at the same
 * read.  peer_tab: every rank's 2*world*16 doubles; peer_flags: world uint64, zeroed once. */
int accbpg_peer_sum_scalars(void* ctx, void* stream, const double* d_in, double* d_out, int count, int rank, int world,
                            void* const* peer_tab, void* const* peer_flags, uint64_t epoch);
/* The same status exchange for the NCCL / gloo fallback: export writes the status word as a float64 into d_slot (which
 * the caller all-reduces with max), import ORs the reduced value back into the local status word. */
int accbpg_ctx_status_export(void* ctx, void* stream, double* d_slot);
int accbpg_ctx_status_import(void* ctx, void* stream, const double* d_slot);
/* The column-sharded LMO's reduction (functions_lmo.py:153-158 with the columns split over ranks): the lowest
 * (value, global index) pair over the ranks, ties to the lowest index, in place on the two doubles at d_pair.  Tables
 * as accbpg_peer_sum_scalars. */
int accbpg_peer_argmin_pair(void* ctx, void* stream, double* d_pair, int rank, int world, void* const* peer_tab,
                            void* const* peer_flags, uint64_t epoch);
/* In-place all-reduce(sum) of n doubles over peer memory (the m-vector A x of PoissonRegression / KLdivRegression,
 * functions.py:102-158, and other replicated sums): every rank stores its vector into slot `rank` of every rank's
 * buffer, releases a flag word there, waits for the `world` flags and adds the slots in rank order.  peer_buf: every
 * rank's 2*world*cap doubles (cap >= n); peer_flags: world uint64, zeroed once. */
int accbpg_peer_sum_vector(void* ctx, void* stream, double* d_x, int64_t n, int64_t cap, int rank, int world,
                           void* const* peer_buf, void* const* peer_flags, uint64_t epoch);

/* ---- Shannon entropy kernels  h(x) = sum x log x   (accbpg/functions.py:398-490) */
int accbpg_shannon_value(void* ctx, void* stream, int64_t n, const double* d_x, double delta, double* d_out);   /* :405-408 */
int accbpg_shannon_gradient(void* ctx, void* stream, int64_t n, const double* d_x, double delta,
                            double* d_out_vec);                                                                  /* :410-413 */
int accbpg_shannon_divergence(void* ctx, void* stream, int64_t n, const double* d_x, const double* d_y,
                              double delta, double* d_out);                                                      /* :415-421 */
/* exp(-(lamda+g)/L - 1) when d_y == NULL (:423-428, :458-462), y*exp(-(lamda+g)/L) otherwise (:430-438, :464-466).
 * normalize != 0: divide by the sum (ShannonEntropySimplex :475-490); d_sum_out (1 slot) receives the
 * un-normalised sum.  normalize == 2: write the un-normalised vector and the sum only (sharded use). */
int accbpg_shannon_prox(void* ctx, void* stream, int64_t n, double lamda, const double* d_y,
                        const double* d_g, double L, int normalize, double* d_out_vec, double* d_sum_out);
/* out = x * scale (finishes the sharded simplex normalisation: scale = 1/sum is NOT used; out = x / denom) */
int accbpg_vec_divide(void* ctx, void* stream, int64_t n, const double* d_x, double denom, double* d_out_vec);

/* ---- linear minimisation oracle over the simplex (accbpg/functions_lmo.py:137-160) */
/* s = 1e-15 everywhere, s[first argmin g] = radius; d_out[0] = min g, d_out[1] = index */
int accbpg_lmo_simplex(void* ctx, void* stream, int64_t n, const double* d_g, double radius,
                       double* d_s_vec, double* d_out);
/* s = fill everywhere except s[idx] = radius (sharded use: each rank fills its slice) */
int accbpg_lmo_fill_vertex(void* ctx, void* stream, int64_t n, double fill, int64_t idx, double radius,
                           double* d_s_vec);
/* elementwise LMOs: l_inf ball  c - r*sign(g)  (functions_lmo.py:106-134); l2 ball  c - r*g/||g||
 * (:16-51, norm supplied by the caller from accbpg_vec_dot); box  where(g<0, upper, lower) (:190-212) */
int accbpg_lmo_linf(void* ctx, void* stream, int64_t n, const double* d_g, double radius,
                    const double* d_center, double* d_s_vec);
int accbpg_lmo_l2(void* ctx, void* stream, int64_t n, const double* d_g, double radius, double gnorm,
                  const double* d_center, double* d_s_vec);
int accbpg_lmo_box(void* ctx, void* stream, int64_t n, const double* d_g, const double* d_lower,
                   const double* d_upper, double* d_s_vec);

/* ---- D-optimal design objective  f(x) = -log det(H diag(x) H^T)
 *      (DOptimalObj.func_grad, accbpg/functions.py:43-59).  H is m x n_local row-major. */
/* The workspace must be ZERO-FILLED once after allocation and then left to the library (it keeps the progress
 * counters of the data-flow Cholesky chain and the never-written upper part of L^{-1} there from call to call). */
size_t accbpg_dopt_workspace_bytes(int m, int64_t n_local);
/* K1: M = H diag(x) H^T as an FP64 DMMA SYRK (lower tiles, split over n, fixed-order reduce), written
 * as a full symmetric m x m matrix with leading dimension m.  Sets ST_X_NEGATIVE if some x < 0. */
int accbpg_dopt_gram(void* ctx, void* stream, const double* d_H, int m, int64_t n_local, int64_t ldh,
                     const double* d_x, void* d_ws, double* d_M);
/* Column-sharded form of K1 with the cross-GPU sum fused behind the SYRK over NVLink peer memory instead of an NCCL
 * all-reduce (reference: the same HXHT, accbpg/functions.py:153, when H's columns live on several GPUs).  The split
 * reduction that ends the SYRK stores each summed lower-triangle element straight into slot `rank` of EVERY rank's
 * receive buffer (remote stores), the last CTA raises this rank's flag word on every rank; a second kernel waits for the
 * `world` flags and sums the received matrices in rank order into d_M (full, mirrored) - all ranks end with bit-identical
 * M.  peer_recv / peer_flags: host arrays of `world` device pointers to every rank's symmetric buffers
 * (2*world*m*m doubles - double-buffered on epoch parity - and `world` uint64 flag words, zero-initialised once; e.g.
 * torch.distributed._symmetric_memory buffer_ptrs); epoch: 1, 2, 3, ..., one per call on these buffers, the same on
 * every rank.  world <= 16.  A rank that waits longer than two minutes for a peer traps. */
int accbpg_dopt_gram_allreduce(void* ctx, void* stream, const double* d_H, int m, int64_t n_local, int64_t ldh,
                               const double* d_x, void* d_ws, int rank, int world, void* const* peer_recv,
                               void* const* peer_flags, uint64_t epoch, double* d_M);
/* Gram matrix of a simplex vertex s (s = fill everywhere, s[i] = radius: lmo_simplex, functions_lmo.py:153-158) from
 * d_G = H H^T of the local columns:  fill*G + (radius - fill) h_i h_i^T.  d_idx: device double holding the GLOBAL column
 * index the LMO chose (accbpg_lmo_simplex's d_out[1]); columns outside [col_offset, col_offset + n_local) add nothing.
 * Lets FW_alg_div_step (algorithms_fw.py:6-75) form M(x + alpha(s - x)) = (1-alpha) M(x) + alpha M(s) without a SYRK. */
int accbpg_dopt_vertex_gram(void* ctx, void* stream, const double* d_H, int m, int64_t n_local, int64_t ldh,
                            const double* d_G, double fill, const double* d_idx, int64_t col_offset, double radius,
                            double* d_out);
/* K2 (+K3): blocked Cholesky M = L L^T (right-looking over 64-wide block columns, two launches for the whole chain:
 * one CTA walks the critical path - panel product, diagonal update, in-warp 64x64 factor and inverse - while a second
 * grid does every other 64x64 tile job as its operands become final, on progress counters in global memory), out of place (d_M symmetric m x m is only read); d_out[0] = -log det M =
 * -sum log(pivot).  d_L (m x m, may be NULL) receives the lower factor, zero above the diagonal.  want_inverse != 0
 * also leaves L^{-1} in the workspace for accbpg_dopt_grad: the block forward substitution rides in the same launches
 * as the factorisation.  Sets ST_NOT_PD on a pivot <= 0.  d_ws is the dopt workspace (any n_local). */
int accbpg_dopt_factor(void* ctx, void* stream, int m, const double* d_M, double* d_L, int want_inverse, void* d_ws,
                       double* d_out);
/* K4: g_j = -|| L^{-1} h_j ||^2 for the local columns, with the L^{-1} that the last accbpg_dopt_factor(want_inverse = 1)
 * on this workspace left there: a DMMA triangular GEMM whose epilogue reduces squared column norms
 * (M^{-1}H is never materialised). */
int accbpg_dopt_grad(void* ctx, void* stream, const double* d_H, int m, int64_t n_local, int64_t ldh, void* d_ws,
                     double* d_g);
/* whole func_grad on one GPU: flag 0 value, 1 gradient, 2 both (value always computed, as in the reference) */
int accbpg_dopt_func_grad(void* ctx, void* stream, const double* d_H, int m, int64_t n, int64_t ldh,
                          const double* d_x, int flag, void* d_ws, double* d_f_out, double* d_g);

/* f(xf) and (f(yg), grad f(yg)) in one call (flag_y = 1 or 2): what one accelerated iteration needs (F[k] = f(x_k)
 * and the gradient at y_k, accbpg/algorithms.py:135,148 / :231,245 / :347,371).  The value-only Cholesky overlaps the
 * gradient chain on the context's side stream; results and status bits are identical to two separate calls. */
int accbpg_dopt_pair(void* ctx, void* stream, const double* d_H, int m, int64_t n_local, int64_t ldh,
                     const double* d_xf, const double* d_yg, int flag_y, void* d_ws, double* d_fx_out,
                     double* d_fy_out, double* d_g);

/* Same evaluation from Gram matrices the caller already holds (M(x) is linear in x: the drivers form
 * M((1-t)x + t z) = (1-t)M(x) + t M(z) with accbpg_vec_axpby instead of another SYRK).  d_Mx may be NULL
 * (then only (f(y), grad f(y)) is produced); flag_y 0 / 1 / 2. */
int accbpg_dopt_pair_from_gram(void* ctx, void* stream, const double* d_H, int m, int64_t n_local, int64_t ldh,
                               const double* d_Mx, const double* d_My, int flag_y, void* d_ws, double* d_fx_out,
                               double* d_fy_out, double* d_g);

/* ---- the same objective on a SPARSE design matrix (D_opt_libsvm, accbpg/applications.py:17-33, which densifies the
 *      LIBSVM data with .toarray('C'); parser accbpg/utils.py:22-95).  H (m x n, one column per sample) stays in
 *      compressed-column form: d_colptr[n+1], d_rowidx[nnz] (feature index, 0-based), d_vals[nnz]; m <= 128.
 *      K1 and K4 read the sparse columns; K2 / K3 are accbpg_dopt_factor on the dense m x m Gram matrix, with the
 *      workspace of accbpg_dopt_sparse_workspace_bytes(m) (zero-filled once, like the dense one). */
size_t accbpg_dopt_sparse_workspace_bytes(int m);
int accbpg_dopt_sparse_gram(void* ctx, void* stream, const int64_t* d_colptr, const int* d_rowidx, const double* d_vals,
                            int m, int64_t n, const double* d_x, void* d_ws, double* d_M);
/* g_j = -|| L^{-1} h_j ||^2 over the nonzeros of column j, with the L^{-1} the last accbpg_dopt_factor(want_inverse = 1)
 * left in d_ws */
int accbpg_dopt_sparse_grad(void* ctx, void* stream, const int64_t* d_colptr, const int* d_rowidx, const double* d_vals,
                            int m, int64_t n, void* d_ws, double* d_g);

/* ---- small shapes: the WHOLE BPG solve in one launch (accbpg/algorithms.py:11-72 with DOptimalObj, functions.py:27-59,
 *      and BurgEntropySimplex, functions.py:326-356).  When H and the m x m factor fit in the shared memory of one SM
 *      (accbpg_dopt_bpg_small_smem_bytes(m, n) != 0; BASELINE configs[0], 80 x 200, does) one persistent CTA - or a
 *      cluster of 2 / 4 CTAs that share the columns of H and exchange through distributed shared memory - runs every
 *      iteration - Gram matrix, factorisation, gradient, Burg-simplex prox, divergence, line-search test, stopping test -
 *      with the control flow of the reference's loop.  d_x: x0 in, last iterate out.  d_F / d_Ls: maxitrs entries each;
 *      d_info[0] = entries written (k + 1), [1] = line-search trials, [2] = last L, [3] = Newton steps of all prox calls,
 *      [4..9] = SM clocks spent in: diagonal-block inverses, gradient, prox, divergence + dot, Gram matrix, factorisation
 *      (d_info has 16 doubles).
 *      linesearch = 0: L stays fixed (algorithms.py:57-58).  Assertions of the reference arrive in the status word. */
size_t accbpg_dopt_bpg_small_smem_bytes(int m, int64_t n);
int accbpg_dopt_bpg_small(void* ctx, void* stream, const double* d_H, int m, int64_t n, int64_t ldh, double* d_x, double L,
                          double ls_ratio, int linesearch, int maxitrs, double epsilon, double eps_prox, double* d_F,
                          double* d_Ls, double* d_info);

/* ---- small shapes: the WHOLE ABPG (accbpg/algorithms.py:94-180) or ABPG_gain (:295-420) solve in one launch, with
 *      DOptimalObj and BurgEntropySimplex, on the machinery of accbpg_dopt_bpg_small (one CTA or a cluster of 2 / 4,
 *      Gram matrix, factorisation, in-place gradient, Burg-simplex root-find) in a shared-memory plan of its own (three
 *      more vectors: accbpg_dopt_abpg_small_smem_bytes).  Every point is evaluated from scratch, as the reference does
 *      (no carried Gram images).  Per trip: y = (1-theta) x- + theta z- (:147, :369), f(y) and g = grad f(y)
 *      (functions.py:43-58), z = div_prox_map(z-, g, theta^(gamma-1) [G] L) (functions.py:341-356),
 *      x = (1-theta) x- + theta z (:150, :374), D(x, y) and D(z, z-), and for ABPG_gain's line search f(x) (:387),
 *      which for the accepted trip is F[k+1].  ABPG, and ABPG_gain with checkdiv, evaluate F[k+1] = f(x_{k+1}) at the
 *      top of the next iteration.
 *      The decisions are those of accbpg_linreg_abpg_small: theta = gamma/(k+gamma), solve_theta (:75-91) when
 *      theta_eq, the alpha form (:367) for ABPG_gain otherwise; G /= ls_dec per iteration and G *= ls_inc per rejected
 *      trip; checkdiv; restart rules 'f' and 'g' (:168, :406; ABPG from k = 1, ABPG_gain from k = 0); the stop
 *      D(z, z-) < epsilon.  Every CTA takes them from the same bits; the scalar and elementwise expressions round like
 *      the host's arithmetic.
 *      driver: ACCBPG_SMALL_DRV_*; restart_rule: ACCBPG_SMALL_RESTART_* (both defined below).  G0, ls_inc, ls_dec and
 *      checkdiv are read by ABPG_gain only.  eps_prox: BurgEntropySimplex's root-find tolerance.
 *      d_x: x0 in, last iterate out.  d_hist: 7 rows of maxitrs doubles, row r at d_hist + r * maxitrs: [0] F, [1] G
 *      (ABPG) or Gain (ABPG_gain), [2] Gdiv (ABPG_gain; the previous value when a trip stops on D(z, z-) < epsilon),
 *      [3] theta, [4] D(x, y), [5] D(z, z-), [6] T (%globaltimer nanoseconds at the top of the iteration since the kernel
 *      started).  d_info (16 doubles): [0] entries written, [1] trips, [2] cluster size, [3] 1 when the very first trip
 *      stopped on D(z, z-) < epsilon, where the reference's Gdr is unbound (the solve ends there), [4] the last G (ABPG)
 *      or gain (ABPG_gain), [5] Newton steps of all root-finds.  Status bits as accbpg_dopt_bpg_small's; the first one
 *      ends the solve.  ACCBPG_E_ARG on NULL pointers, a shape that does not fit, ldh < n, non-finite or non-positive L,
 *      gamma, G0, ls_inc, ls_dec or eps_prox, maxitrs < 1, an unknown driver or restart rule. */
size_t accbpg_dopt_abpg_small_smem_bytes(int m, int64_t n);
int accbpg_dopt_abpg_small(void* ctx, void* stream, int driver, const double* d_H, int m, int64_t n, int64_t ldh,
                           double* d_x, double L, double gamma, int maxitrs, double epsilon, double eps_prox,
                           int theta_eq, int restart, int restart_rule, double G0, double ls_inc, double ls_dec,
                           int checkdiv, double* d_hist, double* d_info);

/* ---- Poisson / KL regression objectives (accbpg/functions.py:102-120, :140-158).  A is m x n_local. */
#define ACCBPG_LINREG_POISSON 0   /* f = sum b log(b/Ax) + Ax - b ; r = 1 - b/Ax   */
#define ACCBPG_LINREG_KL      1   /* f = sum Ax log(Ax/b) - Ax + b ; r = log(Ax/b) */
size_t accbpg_linreg_workspace_bytes(int64_t m, int64_t n_local);
/* K5: Ax (local partial product when A is a column slab) */
int accbpg_linreg_matvec(void* ctx, void* stream, const double* d_A, int64_t m, int64_t n_local, int64_t lda,
                         const double* d_x, void* d_ws, double* d_Ax);
/* K7: objective value and the residual vector r that the gradient needs (d_r may be NULL) */
int accbpg_linreg_value_resid(void* ctx, void* stream, int kind, int64_t m, const double* d_Ax,
                              const double* d_b, double* d_f_out, double* d_r);
/* K6: g = A^T r, one pass over A (the reference materialises an m x n broadcast product) */
int accbpg_linreg_rmatvec(void* ctx, void* stream, const double* d_A, int64_t m, int64_t n_local, int64_t lda,
                          const double* d_r, void* d_ws, double* d_g);

/* ---- small shapes: the WHOLE BPG solve in one launch (accbpg/algorithms.py:11-72) with PoissonRegression /
 *      KLdivRegression (functions.py:85-158) and a Burg or Shannon kernel (functions.py:238-323, :398-490).  When A and
 *      the solve's vectors fit in the shared memory of one SM - or of a cluster of 2, 4 or 8 CTAs, each holding a
 *      contiguous slice of A's columns, the smallest that fits - one persistent launch runs every iteration: gradient
 *      A^T r(Ax) from the carried A x (:112, :150), div_prox_map (:264-271, :290-298, :316-323, :430-438, :464-466,
 *      :475-490), A x1 and f(x1), dot(g, x1 - x) and divergence (:250-253, :415-421), the line-search test
 *      (algorithms.py:53), the stopping test (algorithms.py:66).  The per-CTA partials of A x and of the n-sums are added
 *      in rank order through distributed shared memory: two solves of one instance are bit-identical.
 *      d_x: x0 in, last iterate out.  d_F, d_Ls, d_T: maxitrs entries each; d_T[k] = %globaltimer nanoseconds at the top
 *      of iteration k since the kernel started.  d_info (16 doubles): [0] entries written, [1] line-search trials,
 *      [2] last L, [3] cluster size.  lamda: the kernel's lambda (0 for BURG, SHANNON, SHANNON_SIMPLEX); delta: the
 *      Shannon kernels' delta (unused for Burg).  linesearch = 0: L stays fixed (algorithms.py:57-58).
 *      The reference's assertions arrive in the status word (the operator path's bits) and end the solve at that
 *      iteration. */
#define ACCBPG_SMALL_H_BURG             0   /* BurgEntropy             functions.py:238-271 */
#define ACCBPG_SMALL_H_BURG_L1          1   /* BurgEntropyL1           functions.py:274-298 */
#define ACCBPG_SMALL_H_BURG_L2          2   /* BurgEntropyL2           functions.py:301-323 */
#define ACCBPG_SMALL_H_SHANNON          3   /* ShannonEntropy          functions.py:398-438 */
#define ACCBPG_SMALL_H_SHANNON_L1       4   /* ShannonEntropyL1        functions.py:441-466 */
#define ACCBPG_SMALL_H_SHANNON_SIMPLEX  5   /* ShannonEntropySimplex   functions.py:469-490 */
/* 0 when no cluster of <= 8 CTAs holds A (m x n doubles) and the solve's vectors in shared memory */
size_t accbpg_linreg_bpg_small_smem_bytes(int64_t m, int64_t n);
/* kind: ACCBPG_LINREG_POISSON / _KL; hkind: ACCBPG_SMALL_H_* */
int accbpg_linreg_bpg_small(void* ctx, void* stream, int kind, const double* d_A, int64_t m, int64_t n, int64_t lda,
                            const double* d_b, int hkind, double lamda, double delta, double* d_x, double L,
                            double ls_ratio, int linesearch, int maxitrs, double epsilon,
                            double* d_F, double* d_Ls, double* d_T, double* d_info);

/* ---- small shapes: the WHOLE ABPG (accbpg/algorithms.py:94-180) or ABPG_gain (:295-420) solve in one launch, on the
 *      instances and kernels of accbpg_linreg_bpg_small, in a shared-memory plan of its own (more vectors: a cluster
 *      may be larger than BPG's for one shape).  It follows the drivers' default evaluation scheme (linear images):
 *      A x- and A z- are carried, A y and A x are their combinations (:147, :150, :369, :374), A z is one matvec per
 *      trip, and A x is re-formed from x at the end of every iteration k with (k+1) % reanchor_every == 0.  Per trip:
 *      f(y) and g = A^T r(A y) (:112, :150), z = div_prox_map(z-, g, theta^(gamma-1) [G] L), x, D(x, y), D(z, z-)
 *      (:250-253, :415-421), and for ABPG_gain the gain line search (:387) with G /= ls_dec per iteration and
 *      G *= ls_inc per rejected trip; theta = gamma/(k+gamma), solve_theta (:75-91) when theta_eq, the alpha form
 *      (:367) otherwise; checkdiv; restart rules 'f' and 'g' (:168, :406; ABPG from k = 1, ABPG_gain from k = 0);
 *      the stop D(z, z-) < epsilon.  All decisions are taken redundantly in every CTA from
 *      the same exchanged bits.
 *      driver: ACCBPG_SMALL_DRV_*; restart_rule: ACCBPG_SMALL_RESTART_* (the reference never restarts on other rules).
 *      G0, ls_inc, ls_dec and checkdiv are read by ABPG_gain only.
 *      d_x: x0 in, last iterate out.  d_hist: 7 rows of maxitrs doubles, row r at d_hist + r * maxitrs:
 *      [0] F, [1] G (ABPG) or Gain (ABPG_gain), [2] Gdiv (ABPG_gain; the previous value when a trip stops on
 *      D(z, z-) < epsilon), [3] theta, [4] D(x, y), [5] D(z, z-), [6] T (%globaltimer nanoseconds at the top of the
 *      iteration since the kernel started).  d_info (16 doubles): [0] entries written, [1] trips, [2] cluster size,
 *      [3] 1 when the very first trip stopped on D(z, z-) < epsilon, where the reference's Gdr is unbound (the solve
 *      ends there), [4] the last G (ABPG) or gain (ABPG_gain).  Assertions arrive in the status word as for BPG and end
 *      the solve.  ACCBPG_E_ARG on NULL pointers, a shape that does not fit, non-finite or non-positive L, gamma, G0,
 *      ls_inc or ls_dec, maxitrs < 1 or reanchor_every < 1. */
#define ACCBPG_SMALL_DRV_ABPG        0
#define ACCBPG_SMALL_DRV_ABPG_GAIN   1
#define ACCBPG_SMALL_RESTART_NONE    0
#define ACCBPG_SMALL_RESTART_F       1   /* F[k] > F[k-1]                algorithms.py:168, :406 */
#define ACCBPG_SMALL_RESTART_G       2   /* dot(g, x - x-) > 0           algorithms.py:168, :406 */
/* 0 when no cluster of <= 8 CTAs holds A and the accelerated solve's vectors in shared memory (host only) */
size_t accbpg_linreg_abpg_small_smem_bytes(int64_t m, int64_t n);
int accbpg_linreg_abpg_small(void* ctx, void* stream, int driver, int kind, const double* d_A, int64_t m, int64_t n,
                             int64_t lda, const double* d_b, int hkind, double lamda, double delta, double* d_x,
                             double L, double gamma, int maxitrs, double epsilon, int theta_eq, int restart,
                             int restart_rule, double G0, double ls_inc, double ls_dec, int checkdiv,
                             int reanchor_every, double* d_hist, double* d_info);

/* ---- D_opt_FW / D_opt_FW_away (accbpg/D_opt_alg.py:9-88, :91-185) -------
 * State lives in caller-owned device buffers: x, w (n), Hinv (m x m, ld m), a control block of
 * ACCBPG_FW_CTRL_DOUBLES float64 (layout: enum FwCtrl in csrc/fw.cu, mirrored by dopt_fw.py) and four
 * history arrays of maxitrs float64 (F, SP, SN, T; T holds %globaltimer nanoseconds). */
#define ACCBPG_FW_CTRL_DOUBLES 32
size_t accbpg_fw_workspace_bytes(int m, int64_t n);   /* zero-filled once by the caller, like the D-opt workspace it contains */
/* setup (D_opt_alg.py:39-45 / :123-129): M = V diag(x0) V^T, Hinv = M^{-1}, w_j = v_j^T Hinv v_j,
 * ctrl <- {log det M, not stopped}.  Sets the ST_X_NEGATIVE / ST_NOT_PD status bits like func_grad. */
int accbpg_fw_setup(void* ctx, void* stream, const double* d_V, int m, int64_t n, int64_t ldv,
                    const double* d_x0, void* d_ws, double* d_Hinv, double* d_w, double* d_ctrl);
/* enqueue iterations k_start .. k_start+k_count-1 of the loop (:51-82 / :135-179): argmax w; masked argmin + step
 * rule + history entry + gather of the chosen column; u = Hinv v; Hinv <- (Hinv -/+ c u u^T)/(1 -/+ t); the single
 * pass over V that forms u^T V and updates w and x.  When V is 16-byte aligned with even n and ldv, n < 2^31,
 * m <= 4096 and at least three 32 KB ring stages fit in shared memory next to three vectors of m doubles, this is ONE
 * persistent launch for the whole batch (one CTA per SM; the pass is fed by tensor copies into a shared-memory
 * ring, decisions and u are exchanged between the CTAs); otherwise two launches per iteration chained by
 * programmatic dependent launch.  Same bits either way.
 * away = 0: D_opt_FW, 1: D_opt_FW_away.  Once the optimality test fires (ctrl[0] = 1, ctrl[1] = k) the
 * remaining iterations are not executed; ctrl[14] counts the history entries written. */
int accbpg_fw_run(void* ctx, void* stream, const double* d_V, int m, int64_t n, int64_t ldv, int away, double eps,
                  int k_start, int k_count, void* d_ws, double* d_Hinv, double* d_x, double* d_w, double* d_ctrl,
                  double* d_hist_F, double* d_hist_SP, double* d_hist_SN, double* d_hist_T);


/* Column-sharded building blocks of the same loop (D_opt_alg.py:9-185 with V split by columns over the ranks;
 * Hinv, the control block and the histories are replicated).  A selection record (accbpg_fw_record_bytes() bytes)
 * carries a rank's arg-max, support arg-min and first off-support entry with their GLOBAL indices and the w / x values
 * the step rule needs.  Per iteration k the caller runs
 *   accbpg_fw_decide(k, all ranks' records)  ->  all-reduce(sum) of d_vcol (only the owner of the chosen column
 *   contributes non-zeros)  ->  accbpg_fw_step(k): u = Hinv v, the local pass over V, the rank-one update of Hinv and
 *   the record of the updated local slice  ->  all-gather of the records.
 * The decision merges the records in rank order with the lowest-index tie-break, so the vertex sequence does not
 * depend on the number of ranks. */
size_t accbpg_fw_record_bytes(void);
int accbpg_fw_setup_from_gram(void* ctx, void* stream, const double* d_V, int m, int64_t n_local, int64_t ldv,
                              const double* d_M, void* d_ws, double* d_Hinv, double* d_w, double* d_ctrl);
int accbpg_fw_select_local(void* ctx, void* stream, int64_t n_local, int64_t col_offset, int away, const double* d_x,
                           const double* d_w, void* d_ws, int m, void* d_record_out);
int accbpg_fw_decide(void* ctx, void* stream, const double* d_V, int m, int64_t n_local, int64_t ldv, int64_t col_offset,
                     int away, double eps, int k, const void* d_records, int world, void* d_ws, double* d_ctrl,
                     double* d_hist_F, double* d_hist_SP, double* d_hist_SN, double* d_hist_T, double* d_vcol);
int accbpg_fw_step(void* ctx, void* stream, const double* d_V, int m, int64_t n_local, int64_t ldv, int64_t col_offset,
                   int away, int k, void* d_ws, double* d_Hinv, const double* d_vcol, double* d_x, double* d_w,
                   double* d_ctrl, void* d_record_out);
/* The column-sharded loop with both exchanges over NVLink peer memory instead of NCCL (D_opt_alg.py:52-82 / :136-179
 * per iteration, as accbpg_fw_run): iterations k_start .. k_start+k_count-1 enqueued in one call, three launches each.
 * The tail of every pass stores this rank's selection record into slot `rank` of EVERY rank's record buffer and releases
 * a flag word there; the deciding kernel of the next iteration waits for the `world` flags, merges the records in rank
 * order and decides (replicated); the rank that owns the chosen column stores it into every rank's column buffer and
 * releases the column flag, on which u = Hinv v waits.  peer_rec / peer_col / peer_flags: host arrays of `world` device
 * pointers to every rank's symmetric buffers - 2*world records, 2*m doubles, world+1 uint64 (zero-initialised once; one
 * set of buffers per run, k_start = 0 first).  Records and columns are double-buffered on the iteration's parity.
 * d_Hinv, d_ctrl and the histories are replicated; d_x, d_w are this rank's slices. */
int accbpg_fw_run_peer(void* ctx, void* stream, const double* d_V, int m, int64_t n_local, int64_t ldv,
                       int64_t col_offset, int away, double eps, int k_start, int k_count, int rank, int world,
                       void* const* peer_rec, void* const* peer_col, void* const* peer_flags, void* d_ws,
                       double* d_Hinv, double* d_x, double* d_w, double* d_ctrl, double* d_hist_F, double* d_hist_SP,
                       double* d_hist_SN, double* d_hist_T);

#ifdef __cplusplus
}
#endif
#endif /* ACCBPG_B200_H */
