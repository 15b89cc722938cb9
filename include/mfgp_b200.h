/* mfgp_b200.h -- C-ABI of the B200-native hot path of mfgp-coverage (libmfgp_b200.so).
 *
 * The reference (pure Python) has no FFI; its seam is the Python call surface of gaussian_process.py and
 * simulator.py.  Each entry point below names the reference call site it replaces (file:line under the
 * reference repository).  Conventions:
 *   - every pointer is a caller-owned DEVICE pointer unless the parameter name ends in `_host`;
 *   - sizes are int64_t, parameters are EVALUATED (non-log) doubles in `mfgp_params`;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*) unless documented as blocking;
 *   - return value: 0 = ok, negative = MFGP_ERR_*; no exceptions, no allocation inside (workspaces are
 *     caller-provided, sizes from mfgp_workspace_bytes);
 *   - matrices are row-major fp64; the training set is ordered [X_L ; X_H] as in gaussian_process.py:527-528;
 *   - `npad` is the training size N = NL + NH rounded up to a multiple of MFGP_TILE (64); factor / inverse
 *     buffers are npad x npad with leading dimension `ld` >= npad, padding rows/cols hold the identity.
 */
#ifndef MFGP_B200_H
#define MFGP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MFGP_TILE 64

#define MFGP_OK 0
#define MFGP_ERR_INVALID (-1)   /* bad argument (null pointer, size, alignment) */
#define MFGP_ERR_NOT_SPD (-2)   /* Cholesky hit a non-positive pivot: numpy raises LinAlgError here */
#define MFGP_ERR_CUDA (-3)      /* a CUDA runtime call failed; see mfgp_last_error */
#define MFGP_ERR_EMPTY_CELL (-4)/* a Voronoi cell holds no grid point: np.amax([]) raises ValueError here */

/* Evaluated hyper-parameters.  gaussian_process.py:132,:248-251 (SF) and :411-416,:510-514 (MF):
 * scale = exp(hyp[1|4]), length = exp(hyp[2|5]), rho = exp(hyp[6]), noise = exp(hyp[3] | hyp[7], hyp[8]) added to the
 * diagonal UN-squared, jitter = 1e-8 (:42,:298).  Means are passed evaluated so both the current exp() convention and
 * the 2020 raw convention of the logged goldens can be served.  Single fidelity: multi = 0, NL = 0, *_L ignored. */
typedef struct mfgp_params {
    double s_L, l_L;        /* lofi kernel: output scale, length scale          */
    double s_H, l_H;        /* hifi (or the only) kernel                          */
    double rho;             /* AR1 cross-fidelity scale                           */
    double noise_L, noise_H;
    double mean_L, mean_H;
    double jitter;
    int32_t multi;          /* 1 = two-level AR1 MFGP, 0 = SFGP                   */
    int32_t reserved;
} mfgp_params;

const char* mfgp_version(void);
const char* mfgp_last_error(void);          /* text of the last CUDA error seen by this thread */
int64_t mfgp_debug_chol_trace(int64_t* out, int64_t max_tasks);   /* diagnostics: per-chain-task time stamps of the tiled Cholesky (MFGP_DF_TRACE=1) */
int64_t mfgp_launch_count(void);            /* kernels launched by this library since load (bench.py's gpu_launches) */
int64_t mfgp_npad(int64_t n);               /* n rounded up to MFGP_TILE (at least MFGP_TILE)  */
int64_t mfgp_workspace_bytes(int64_t npad); /* scratch needed by mfgp_cholesky / mfgp_tri_inverse (one buffer serves both) */

/* ---- GP fit: replaces SFGP.updt_info gaussian_process.py:229-255 and MFGP.updt_info :493-529 ------------------- */

/* K[npad,ld] = training covariance + (noise + jitter) I; padding = identity.  Only the 64x64 tiles on or below the
 * diagonal are written (K is symmetric and mfgp_cholesky* read the lower triangle).  Also writes the scaled
 * training coordinates Tt[npad,4] = (x/l_L, y/l_L, x/l_H, y/l_H) used by mfgp_posterior (:77-78 divides before
 * differencing).  Replaces the K assembly at gaussian_process.py:253 / :523-528. */
int mfgp_build_train_cov(const double* Xt, int64_t NL, int64_t NH, const mfgp_params* p_host,
                         double* K, int64_t npad, int64_t ld, double* Tt, void* stream);

/* In-place lower Cholesky of K[npad,ld] (np.linalg.cholesky at gaussian_process.py:254 / :529).  Blocked, trailing
 * updates on FP64 tensor cores (DMMA).  Also writes the inverses of the 64x64 diagonal blocks into the diagonal
 * blocks of W (may be NULL).  `info` (device int32): 0, 1 + index of the first non-positive pivot, or -1 (internal error:
 * the tile-dataflow kernel gave up waiting for a tile).  `work`: mfgp_workspace_bytes(npad) bytes; it holds the kernel's
 * ticket counter and per-tile ready flags, so calls that use DIFFERENT work buffers may overlap freely (other streams,
 * other host threads); a work buffer must not be shared by calls that can run concurrently.  A call that returns
 * MFGP_ERR_INVALID (odd ld / ldw / ldb / ldm, a base pointer off 16-byte alignment, a short workspace, ...) enqueues
 * nothing: info, K, W and work keep their contents.  The same holds for mfgp_cholesky_solve[_gram] (also Bm, M). */
int mfgp_cholesky(double* K, int64_t npad, int64_t ld, double* W, int64_t ldw, int32_t* info, void* work,
                  void* stream);

/* W[npad,ldw] = L^-1 (lower; strict upper part zeroed), by recursive block doubling on DMMA.  Needs the diagonal
 * 64x64 blocks of W already inverted by mfgp_cholesky.  Stands in for the four general solves at
 * gaussian_process.py:141,:145 / :431,:434. */
int mfgp_tri_inverse(const double* L, int64_t npad, int64_t ld, double* W, int64_t ldw, void* work, void* stream);

/* z[npad] = W (y - mean): y[N] raw observations ordered [y_L ; y_H]; centring as gaussian_process.py:133 / :419-424. */
int mfgp_whiten(const double* W, int64_t npad, int64_t ldw, const double* y, int64_t NL, int64_t NH,
                const mfgp_params* p_host, double* z, void* stream);

/* Bordered (append-only) factor update: replaces the refit inside SFGP.updt gaussian_process.py:257-268 and
 * MFGP.updt_hifi :531-542 when samples were only APPENDED.  The reference appends new points at the END of [X_L; X_H]
 * and refactors from scratch (:266-268, :540-542); the leading block of L is unchanged, so only the 64-row blocks that
 * hold rows [NL+NH_old, NL+NH_new) of L, W = L^-1 and z are recomputed (left-looking, split-K DMMA tile products).
 * Xt / y must already hold all NL+NH_new points; K, W, Tt, z must be the buffers of the standing factorisation, with
 * leading dimensions >= mfgp_npad(NL+NH_new).  `work`: mfgp_append_workspace_bytes(npad) bytes. */
int mfgp_cholesky_append(const double* Xt, int64_t NL, int64_t NH_old, int64_t NH_new, const mfgp_params* p_host,
                         double* K, int64_t ld, double* W, int64_t ldw, const double* y, double* z, double* Tt,
                         int32_t* info, void* work, int64_t work_bytes, void* stream);
int64_t mfgp_append_workspace_bytes(int64_t npad);

/* ---- GP posterior: replaces SFGP.predict gaussian_process.py:121-148 and MFGP.predict :401-438 ------------------ */

/* mu[G] = mean_H + psi^T K^-1 (y-m), var[G] = k(0) - |W psi|^2 for the G points Xs[G,2].  Fused: psi tiles are
 * generated on chip, multiplied by W on DMMA and reduced; psi / V never reach HBM.  N = NL+NH may be 0 (prior).
 * If Vc != NULL the whitened cross-covariance V = W psi^T is also stored, Vc[n*ldv + g] (for choi_greedy); if
 * qred != NULL the variance reduction |W psi|^2 is stored as well (var = k(0) - qred loses it when qred ~ ulp). */
int mfgp_posterior(const double* Xs, int64_t G, const double* Tt, int64_t NL, int64_t NH,
                   const double* W, int64_t npad, int64_t ldw, const double* z, const mfgp_params* p_host,
                   double* mu, double* var, double* qred, double* Vc, int64_t ldv, void* stream);

/* Tensor-product grids (every grid of the reference: distribution.py:337-339 builds `[[i, j] for i in g for j in g]`).
 * The RBF kernel is separable per axis, so psi[g][n] = TLx[ix][n]*TLy[iy][n] + THx[ix][n]*THy[iy][n] with
 * (ix, iy) = divmod(g, ny) and the scales / rho / padding folded into the x tables: 2 flops per element instead of two
 * fp64 exp, which matters because exp and DMMA share the FP64 pipe.  mfgp_grid_tables fills the four tables
 * ([nx|ny][ldt], ldt >= npad) from the axis values ux[nx], uy[ny] after every fit; mfgp_posterior_grid is
 * mfgp_posterior for the flat x-major index range [g_lo, g_lo + G) (grid sharding passes a sub-range). */
int mfgp_grid_tables(const double* ux, int64_t nx, const double* uy, int64_t ny, const double* Tt, int64_t NL, int64_t NH,
                     int64_t npad, const mfgp_params* p_host, double* TLx, double* TLy, double* THx, double* THy,
                     int64_t ldt, void* stream);
int mfgp_posterior_grid(int64_t ny, int64_t g_lo, int64_t G, const double* TLx, const double* TLy, const double* THx,
                        const double* THy, int64_t ldt, int64_t NL, int64_t NH, const double* W, int64_t npad,
                        int64_t ldw, const double* z, const mfgp_params* p_host, double* mu, double* var, double* qred,
                        double* Vc, int64_t ldv, void* stream);

/* Incremental posterior after mfgp_cholesky_append: rows [row_lo, NL+NH) of V = W psi are new since mu / var / qred
 * were last computed; only their contributions are formed and ADDED (mu += v_new . z_new, var -= |v_new|^2,
 * qred += |v_new|^2).  Equal to a from-scratch mfgp_posterior up to rounding (~1e-13 k(0)); cost ~ G (N - row_lo) N
 * instead of G N^2 / 2.  0 < row_lo < NL+NH. */
int mfgp_posterior_update(const double* Xs, int64_t G, const double* Tt, int64_t NL, int64_t NH,
                          const double* W, int64_t npad, int64_t ldw, const double* z, const mfgp_params* p_host,
                          int64_t row_lo, double* mu, double* var, double* qred, double* Vc, int64_t ldv, void* stream);
int mfgp_posterior_grid_update(int64_t ny, int64_t g_lo, int64_t G, const double* TLx, const double* TLy,
                               const double* THx, const double* THy, int64_t ldt, int64_t NL, int64_t NH, const double* W,
                               int64_t npad, int64_t ldw, const double* z, const mfgp_params* p_host, int64_t row_lo,
                               double* mu, double* var, double* qred, double* Vc, int64_t ldv, void* stream);

/* Factored posterior for whole columns [ix0, ix0+ncols) of a tensor-product grid ux[nx] x uy[ny] (x-major).  Each axis
 * factor of the separable RBF cross-covariance is an entire function of the grid coordinate; its Chebyshev interpolant of
 * order rx / ry (per kernel part: L = lofi, H = hifi) on [xlo,xhi] / [ylo,yhi] reproduces the factor tables to rounding
 * (~5e-15 entrywise at the orders chosen by the host), which turns the G triangular products v = W psi of mfgp_posterior
 * into ONE product W B with R = ryL*rxL' + ryH*rxH' (~2.5k) columns plus per-column 64x64 Gram matrices: ~4e10 MAC
 * instead of 8.8e12 at 1 M points / N = 4096, same mean and variance to ~2e-14 k(0).  Nothing of the training covariance
 * is approximated.  Outputs are flat over the requested columns: mu / var / qred[(ix-ix0)*ny + iy].  ryL, ryH multiples
 * of 4, every order <= 64 (both parts share one expansion of max(rxL, rxH) x max(ryL, ryH) terms); single fidelity:
 * rxL = ryL = 0, NL = 0.  `chunk_cols` columns are processed per
 * pass (bounds the workspace).  No V cache: callers that need V (choi_greedy) use mfgp_posterior_grid. */
int mfgp_posterior_grid_factored(const double* ux, int64_t nx, const double* uy, int64_t ny, int64_t ix0, int64_t ncols,
                                 const double* Xt, int64_t NL, int64_t NH, const double* W, int64_t npad, int64_t ldw,
                                 const double* z, const mfgp_params* p_host, int64_t rxL, int64_t ryL, int64_t rxH, int64_t ryH,
                                 double xlo, double xhi, double ylo, double yhi, int64_t chunk_cols,
                                 double* mu, double* var, double* qred, double* Gstore, double* Hz_store, void* work,
                                 int64_t work_bytes, void* stream);
/* Gstore[ncols, 64, 64] / Hz_store[mfgp_factored_rhs_cols] (both optional in the full forms) keep the per-column Gram
 * matrices G'(ix) and z^T Y, so that after mfgp_cholesky_append only the NEW rows [row_lo, NL+NH) of Y = W B have to be
 * formed: G'(ix) += Y'_new^T Y'_new, then every grid point is re-evaluated (a 64 x 64 quadratic form per point).  Same
 * results as the full form to rounding; ~7e8 MAC + the evaluation pass instead of 4e10 MAC at c4 with 64 new samples. */
int mfgp_posterior_grid_factored_update(const double* ux, int64_t nx, const double* uy, int64_t ny, int64_t ix0, int64_t ncols,
                                        const double* Xt, int64_t NL, int64_t NH, int64_t row_lo, const double* W, int64_t npad,
                                        int64_t ldw, const double* z, const mfgp_params* p_host, int64_t rxL, int64_t ryL,
                                        int64_t rxH, int64_t ryH, double xlo, double xhi, double ylo, double yhi,
                                        int64_t chunk_cols, double* mu, double* var, double* qred, double* Gstore,
                                        double* Hz_store, void* work, int64_t work_bytes, void* stream);
int64_t mfgp_factored_workspace_bytes(int64_t npad, int64_t ncols, int64_t ny, int64_t rxL, int64_t ryL, int64_t rxH,
                                      int64_t ryH, int64_t chunk_cols);

/* Fused fit + factored posterior (the from-scratch iteration of the reference, simulator.py:888-892, on a tensor grid):
 *   mfgp_build_train_cov  ->  mfgp_factored_prepare (B = [B_L | B_H | y - mean], mfgp_factored_rhs_cols columns)
 *   ->  mfgp_cholesky_solve (K -> L in place, diagonal-block inverses into W, Ball -> L^-1 Ball: ONE persistent
 *       tile-dataflow kernel, chol_dataflow_kernel in csrc/gp_fit.cu; its ticket counter and ready flags live in `work`,
 *       mfgp_cholesky_solve_workspace_bytes(npad, R) bytes of caller memory, so the call is re-entrant per work buffer)
 *   ->  mfgp_posterior_grid_factored_solved (steps 4-6; z_out receives the whitened observations).
 * Neither the explicit inverse (mfgp_tri_inverse) nor the product W B is formed; run mfgp_tri_inverse afterwards only if W
 * is needed (dense posterior, mfgp_cholesky_append, choi_greedy).  Same geometry / order arguments and the same `work`
 * buffer for prepare and solved.  ldY (row stride of Yall) is a multiple of 64 from the layout's own right-hand-side count
 * (mfgp_factored_rhs_cols[_trunc]) up to mfgp_factored_rhs_cols(rxL, ryL, rxH, ryH); a larger one is MFGP_ERR_INVALID
 * (mfgp_factored_gram_target: NULL), since the Gram route keeps M = Yall^T Yall at that stride inside `work`. */
int64_t mfgp_factored_rhs_cols(int64_t rxL, int64_t ryL, int64_t rxH, int64_t ryH);
int mfgp_factored_prepare(const double* ux, int64_t nx, const double* uy, int64_t ny, int64_t ix0, int64_t ncols,
                          const double* Xt, const double* y, int64_t NL, int64_t NH, int64_t npad, const mfgp_params* p_host,
                          int64_t rxL, int64_t ryL, int64_t rxH, int64_t ryH, double xlo, double xhi, double ylo, double yhi,
                          int64_t chunk_cols, double* Ball, int64_t ldB, void* work, int64_t work_bytes, void* stream);
int64_t mfgp_cholesky_solve_workspace_bytes(int64_t npad, int64_t R);
int mfgp_cholesky_solve(double* K, int64_t npad, int64_t ld, double* W, int64_t ldw, int32_t* info, double* Bm, int64_t ldb,
                        int64_t R, void* work, int64_t work_bytes, void* stream);
int mfgp_posterior_grid_factored_solved(const double* ux, int64_t nx, const double* uy, int64_t ny, int64_t ix0, int64_t ncols,
                                        const double* Xt, int64_t NL, int64_t NH, int64_t npad, const mfgp_params* p_host,
                                        int64_t rxL, int64_t ryL, int64_t rxH, int64_t ryH, double xlo, double xhi, double ylo,
                                        double yhi, int64_t chunk_cols, const double* Yall, int64_t ldY, double* z_out,
                                        double* mu, double* var, double* qred, double* Gstore, double* Hz_store, void* work,
                                        int64_t work_bytes, void* stream);

/* The same sequence with the Gram product of steps 4 + 5 folded into the factorisation kernel.  The Gram route of the
 * factored posterior needs M = Yall^T Yall (R x R; csrc/gp_factored.cu); mfgp_cholesky_solve_gram accumulates its 64x64
 * tiles with low-priority tasks of the SAME tile-dataflow kernel -- group of block rows by group, in a fixed order, so M is
 * deterministic -- in the CTA slots that the factorisation leaves idle while it waits on its chain of diagonal blocks:
 *   M = mfgp_factored_gram_target(...)   pointer into the prepare `work` buffer where the posterior call expects M, or NULL
 *                                         when steps 4 + 5 will take the direct route (then use the plain pair above);
 *   mfgp_cholesky_solve_gram(..., M, ldm = ldb = R, work of mfgp_cholesky_solve_gram_workspace_bytes(npad, R) bytes, ...);
 *   mfgp_posterior_grid_factored_solved_gram(...)   same arguments as _solved; skips the product and its reduction.
 * M == NULL in mfgp_cholesky_solve_gram is mfgp_cholesky_solve.
 *
 * Truncated column layout (optional, `kx`: HOST array of max(ryL, ryH) int32, or NULL for the uniform layout).  Term (l, k) of the
 * expansion -- T_l(ty) T_k(tx) -- has a coefficient bounded by a_y[l] a_x[k], and both factors decay super-exponentially (the
 * axis factors are entire functions), so the far corner of the rx x ry block is below rounding: per y term l only the first
 * kx[l] x terms (a multiple of 4, 4 <= kx[l] <= round_up(max(rxL, rxH), 4)) are kept; the right-hand-side matrix shrinks to
 * mfgp_factored_rhs_cols_trunc(ry, kx) columns (c4: 1344 -> 896) at the same entrywise accuracy -- the caller picks kx from the
 * same coefficient envelopes that gave it the orders (mfgp_coverage_b200/_engine.py: chebyshev_truncation).  Only the Gram route
 * reads this layout: give the same kx to mfgp_factored_prepare_trunc, mfgp_factored_gram_target (which then never returns
 * NULL for a valid geometry) and mfgp_posterior_grid_factored_solved_gram; Gstore / Hz_store must be NULL. */
int64_t mfgp_factored_rhs_cols_trunc(int64_t ry, const int32_t* kx);
int mfgp_posterior_grid_factored_trunc(const double* ux, int64_t nx, const double* uy, int64_t ny, int64_t ix0, int64_t ncols,
                                       const double* Xt, int64_t NL, int64_t NH, const double* W, int64_t npad, int64_t ldw,
                                       const double* z, const mfgp_params* p_host, int64_t rxL, int64_t ryL, int64_t rxH, int64_t ryH,
                                       double xlo, double xhi, double ylo, double yhi, int64_t chunk_cols, const int32_t* kx,
                                       double* mu, double* var, double* qred, double* Gstore, double* Hz_store, void* work,
                                       int64_t work_bytes, void* stream);   /* mfgp_posterior_grid_factored with the layout above */
int mfgp_factored_prepare_trunc(const double* ux, int64_t nx, const double* uy, int64_t ny, int64_t ix0, int64_t ncols,
                                const double* Xt, const double* y, int64_t NL, int64_t NH, int64_t npad, const mfgp_params* p_host,
                                int64_t rxL, int64_t ryL, int64_t rxH, int64_t ryH, double xlo, double xhi, double ylo, double yhi,
                                int64_t chunk_cols, const int32_t* kx, double* Ball, int64_t ldB, void* work, int64_t work_bytes,
                                void* stream);
double* mfgp_factored_gram_target(int64_t nx, int64_t ny, int64_t ix0, int64_t ncols, int64_t NL, int64_t NH, int64_t npad,
                                  const mfgp_params* p_host, int64_t rxL, int64_t ryL, int64_t rxH, int64_t ryH,
                                  int64_t chunk_cols, const int32_t* kx, int64_t ldY, void* work, int64_t work_bytes);
int64_t mfgp_cholesky_solve_gram_workspace_bytes(int64_t npad, int64_t R);
int mfgp_cholesky_solve_gram(double* K, int64_t npad, int64_t ld, double* W, int64_t ldw, int32_t* info, double* Bm, int64_t ldb,
                             int64_t R, double* M, int64_t ldm, void* work, int64_t work_bytes, void* stream);
int mfgp_posterior_grid_factored_solved_gram(const double* ux, int64_t nx, const double* uy, int64_t ny, int64_t ix0,
                                             int64_t ncols, const double* Xt, int64_t NL, int64_t NH, int64_t npad,
                                             const mfgp_params* p_host, int64_t rxL, int64_t ryL, int64_t rxH, int64_t ryH,
                                             double xlo, double xhi, double ylo, double yhi, int64_t chunk_cols,
                                             const int32_t* kx, const double* Yall, int64_t ldY, double* z_out, double* mu,
                                             double* var, double* qred, double* Gstore, double* Hz_store, void* work,
                                             int64_t work_bytes, void* stream);

/* ---- coverage step: replaces simulator.py in_polygon :105-124, compute_loss :194-228, compute_centroids :231-283,
 *      compute_max_var :286-323, compute_sample_clusters :377-412 ------------------------------------------------ */

/* One pass over the grid for up to two bounded-Voronoi partitions:
 *   partition C ("lloyd", seeds_c[Ac,2]): cent[Ac,4] = {sum w, sum w*x, sum w*y, count},
 *                                          amax_val[Ac], amax_idx[Ac] = per-cell max of var and its FIRST grid index
 *                                          (np.argmax semantics; -1 for an empty cell);
 *   partition P ("loss",  seeds_p[Ap,2]): lossp[Ap,2] = {sum |x-seed|^2 f, count}.
 * Membership: nearest seed when the two smallest squared distances differ by more than tie_tol, otherwise the
 * reference's exact crossings test (matplotlib point_in_path, restated) against the cell polygons
 * poly_xy[nvert,2] / poly_off[A+1] (Qhull vertex order; nvert == poly_off[A]); a point may then fall in 0, 1 or several cells, exactly as in
 * the reference.  tie_tol = +inf forces the crossings test everywhere.  w / var / f / member_* may be NULL to skip
 * the corresponding output; Ac or Ap may be 0.  member_c[G, ceil(Ac/64)] receives the membership bit masks.
 * `base_index` is added to grid indices (grid sharding).  Deterministic (no floating-point atomics).
 * Arg-max ties (amax_k0, amax_rel): two variances are tied when they differ by at most amax_rel * (amax_k0 - smaller),
 * a tolerance relative to the variance REDUCTION; ties go to the LOWEST index (np.argmax returns the first index).
 * This reproduces both ways the reference's variances tie: bit-identical values at mirror-image points of a symmetric
 * prior (tolerance >> arithmetic noise) and the 1-ulp plateaus of k0 - q far from all data (tolerance << 1 ulp, exact
 * compare).  amax_rel = 0: plain first-index arg-max.  Callers in simulator.py pass k(0) and 1e-10.
 * tie_count (optional device int32): receives the number of (point, partition) pairs whose membership the crossings test
 * decided (nearest-seed gap <= tie_tol).  0 means the result does not depend on the polygon vertices at all -- the
 * drop-in then never needs host Qhull for that iteration (cells clipped on the device, cov_voronoi_clip). */
int cov_assign_reduce(const double* xy, const double* w, const double* var, const double* f, int64_t G,
                      int64_t base_index,
                      const double* seeds_c, int64_t Ac, const double* poly_xy_c, const int32_t* poly_off_c, int64_t nvert_c,
                      const double* seeds_p, int64_t Ap, const double* poly_xy_p, const int32_t* poly_off_p, int64_t nvert_p,
                      double tie_tol, double amax_k0, double amax_rel,
                      double* cent, double* amax_val, int64_t* amax_idx, double* lossp,
                      uint64_t* member_c, int32_t* tie_count, void* work, int64_t work_bytes, void* stream);
int64_t cov_workspace_bytes(int64_t G, int64_t Ac, int64_t Ap);

/* The same pass for a tensor-product grid stored x-major (point g = ix*ny + iy; every grid of the reference:
 * distribution.py:337-339) or a whole-column slice of one (grid sharding): G must be a multiple of ny.  Uses the
 * column-sweep kernel -- a warp owns 32 consecutive iy and walks the columns, each lane accumulates privately for the
 * cell it is in, no shuffles in the loop -- and returns exactly what cov_assign_reduce returns (sums in a different,
 * equally fixed order).  No membership output; tie_tol must be finite (nearest-seed cells). */
int cov_assign_reduce_grid(const double* xy, const double* w, const double* var, const double* f, int64_t G, int64_t ny,
                           int64_t base_index,
                           const double* seeds_c, int64_t Ac, const double* poly_xy_c, const int32_t* poly_off_c, int64_t nvert_c,
                           const double* seeds_p, int64_t Ap, const double* poly_xy_p, const int32_t* poly_off_p, int64_t nvert_p,
                           double tie_tol, double amax_k0, double amax_rel,
                           double* cent, double* amax_val, int64_t* amax_idx, double* lossp,
                           int32_t* tie_count, void* work, int64_t work_bytes, void* stream);

/* Bounded Voronoi cells on the device (replaces voronoi_bounded simulator.py:154-191 + poly_area :127-136 where host Qhull
 * is the bottleneck -- replicate sweeps, device-resident loops): cell i = the box [xmin-eps/2, xmax+eps/2] x
 * [ymin-eps/2, ymax+eps/2] clipped by the bisectors with all other seeds, which IS the reference's mirrored-seed diagram
 * restricted to its first A cells.  Output in cov_assign_reduce's layout: poly_xy[<= cap_vertices, 2], poly_off[A+1],
 * plus areas[A] (shoelace).  Vertices agree with Qhull's to ~1e-13; only grid points exactly on a bisector can be
 * classified differently, so parity runs keep Qhull.  flag[0] = 1 (and NaN areas) if a polygon outgrew the capacity. */
int64_t cov_voronoi_clip_workspace_bytes(int64_t A);
int cov_voronoi_clip(const double* seeds, int64_t A, double xmin, double xmax, double ymin, double ymax, double eps,
                     double* poly_xy, int32_t* poly_off, int64_t cap_vertices, double* areas, int32_t* flag, void* work,
                     int64_t work_bytes, void* stream);

/* O(A) finishing of cov_assign_reduce's partial sums with the reference's arithmetic (simulator.py:215-219, :256-271):
 * out[0] = loss, out[1+2i], out[2+2i] = centroid i clamped to [xmin,xmax] x [ymin,ymax], out[1+2Ac+i] = max variance of
 * cell i, out[1+3Ac+i] = its arg-max grid index as a double (-1: empty cell), out[1+4Ac .. 4+4Ac] = the values of up
 * to four device int32 flags (may be NULL: e.g. mfgp_cholesky's `info`, cov_voronoi_clip's `flag`, cov_assign_reduce's
 * tie_count), so ONE D2H copy of 5 + 4 Ac doubles brings a whole iteration's result and its error state back. */
int cov_finish(const double* cent, const double* areas_c, int64_t Ac, const double* lossp, const double* areas_p, int64_t Ap,
               const double* amax_val, const int64_t* amax_idx, double xmin, double xmax, double ymin, double ymax,
               const int32_t* flag0, const int32_t* flag1, const int32_t* flag2, const int32_t* flag3, double* out,
               void* stream);

/* Global first-index argmax of v[G] (np.argmax at simulator.py:352): out_val[1], out_idx[1]. */
int cov_argmax(const double* v, int64_t G, int64_t base_index, double k0, double rel, double* out_val, int64_t* out_idx,
               void* work, int64_t work_bytes, void* stream);

/* ---- Choi greedy sample planner: replaces compute_sample_points simulator.py:326-374 ---------------------------- */

/* Greedy max-variance selection on the cached V (rows [0,n0) valid, capacity rows `cap`, row stride ldv >= G):
 * while max(var) > threshold: j = first argmax (tie rule as above with k0 = k(0), rel = tie_rel); append the bordered-
 * Cholesky row for x_j (hifi level, pseudo-observation = current mean, so mu is unchanged); qred += v^2 and
 * var = k(0) - qred (recomputed, never decremented: the reference re-predicts from scratch).  Picks (grid indices) go to picks_host[<= max_picks];
 * returns the number of picks (>= 0) or a negative error.  BLOCKING (synchronises `stream` once per pick). */
int64_t choi_greedy(const double* Xs, int64_t G, double* Vc, int64_t ldv, int64_t n0, int64_t cap, double* var,
                    double* qred, const mfgp_params* p_host, double threshold, double tie_rel, int64_t max_picks,
                    int64_t* picks_host,
                    void* work, int64_t work_bytes, void* stream);

/* Grid-sharded form of choi_greedy: every rank of a process group owns the whole-column slice [base, base + G) of the
 * grid, its V cache Vc[cap, ldv] (rows [0,n0) valid), var[G] and qred[G].  One pick is
 *   choi_shard_append -> choi_shard_propose -> all-gather of the send slots (caller, rank order) -> choi_shard_select;
 * planning starts with choi_shard_begin (arg-max of the slice's var + the first propose) -> all-gather -> select.
 * A send slot is cap + 4 doubles: [value, index bits (int64), x_j, y_j, V[0:n, j - base]] of the shard's first-index
 * arg-max (global index; -1: no candidate, or planning is done -- every rank still joins every exchange).  The select
 * folds the `world` slots of recv[world, cap + 4] in rank order with the tie rule of choi_greedy (a tie goes to the lowest
 * global index), applies its loop condition (value > threshold, max_picks, cap), records the pick and stages the winner's
 * slot for the next append.  It is deterministic, so every rank that sees the same slots holds the same state.  Nothing
 * synchronises except choi_shard_status (BLOCKING): status_host[3] = {n, picks, done}, and, if picks_host != NULL, the
 * picks since begin (global grid indices, up to cap of them).  `work`: choi_shard_workspace_bytes(G, cap) bytes, the
 * same buffer and the same (G, cap) for every call between two begins.  G > 0 (every shard owns at least one column). */
int64_t choi_shard_workspace_bytes(int64_t G, int64_t cap);
int choi_shard_begin(const double* Xs, int64_t G, int64_t base, const double* Vc, int64_t ldv, int64_t n0, int64_t cap,
                     const double* var, const mfgp_params* p_host, double tie_rel, double* send, void* work,
                     int64_t work_bytes, void* stream);
int choi_shard_append(const double* Xs, int64_t G, int64_t base, double* Vc, int64_t ldv, int64_t cap, double* var,
                      double* qred, const mfgp_params* p_host, double tie_rel, void* work, int64_t work_bytes, void* stream);
int choi_shard_propose(const double* Xs, int64_t G, int64_t base, const double* Vc, int64_t ldv, int64_t cap,
                       const mfgp_params* p_host, double tie_rel, double* send, void* work, int64_t work_bytes, void* stream);
int choi_shard_select(const double* recv, int64_t world, int64_t G, int64_t cap, const mfgp_params* p_host, double threshold,
                      double tie_rel, int64_t max_picks, void* work, int64_t work_bytes, void* stream);
int choi_shard_status(int64_t G, int64_t cap, const void* work, int64_t work_bytes, int64_t* status_host, int64_t* picks_host,
                      void* stream);

/* ---- batched replicate stepper: the loop bodies of simulator.py periodic :618-785, todescato :788-954, lloyd :508-616 for many
 *      independent runs of one experiment (runner.py:100, :131-147 fans the replicates out over a process pool) ----------------- */

/* State of a batch of R runs; every pointer is a caller-owned device buffer with a leading run dimension.
 * Shared by the runs: grid xy[G,2] (x-major tensor grid ux[nx] x uy[ny]), truth f[G].  Per run: training set Xt[cap,2], y[cap]
 * (first NL rows: the lofi prior), W[cap,cap] = L^-1 (lower) and z[cap] of the standing fit, axis-factor tables
 * T{x,y}{L,H}[cap][nx|ny] (exp(-0.5 ((u - U_n) / l)^2) per training point n), standing posterior mu[G] / var[G], positions /
 * previous positions / Lloyd seeds pos, prev, cen [A,2], pos_idx[A] (grid index of the position or -1), prob[A], explore[A],
 * counters Ncur, knew, status (0 ok, k > 0: pivot k-1 not positive, -4: empty cell, -1: capacity), noise_used, nsamples,
 * ties[iterations] (grid points within TIE_TOL/10 of a bisector, per iteration).  Random numbers drawn by the host in the
 * order the reference consumes them: noise[max_samples] (N(0, sigma_n) per sample, :707), unif[iterations, A] (:943).
 * Logs: log_loss[iterations], log_agent[iterations, A, 11] (X, Y, XMax, YMax, VarMax, Var0, XCentroid, YCentroid, ProbExplore,
 * Explore, Distance: the reference's agent row), log_sample[max_samples, 5] (Iteration, Agent, X, Y, Sample). */
typedef struct mfgp_batch {
    int64_t runs, G, nx, ny, A, NL, cap, algo /* 0 lloyd, 1 periodic, 2 todescato, 3 choi */, iterations, max_samples;
    double xmin, xmax, ymin, ymax, eps, tie_tol, amax_rel;
    const double* xy; const double* f; const double* ux; const double* uy;
    double* Xt; double* y; double* W; double* z;
    double* TxL; double* TyL; double* TxH; double* TyH;
    double* mu; double* var;
    double* pos; double* prev; double* cen;
    int64_t* pos_idx;
    double* prob; int32_t* explore;
    int32_t* Ncur; int32_t* knew; int32_t* status; int32_t* noise_used; int32_t* nsamples; int32_t* ties;
    const double* noise; const double* unif;
    double* log_loss; double* log_agent; double* log_sample;
    /* Choi only (algo 3; NULL otherwise).  Planner: q[G] per run (variance reduction |W psi_g|^2 of the rows in use),
     * picks[cap] (grid indices of the period's picks in selection order, planned rows Ncur + k), nplan (picks so far),
     * plan_state (0 planning, 1 done, 2 stopped at cap: grow the buffers, reset to 0, resume), pmask[cap] (cells of each
     * pick, bit c = agent c), ccount[A] (picks per cell), cties (picks within TIE_TOL/10 of a bisector in this period).
     * Tours: tour_off[runs*A+1] (tour of (run r, agent c) = tour[tour_off[r*A+c] .. tour_off[r*A+c+1]), grid indices),
     * tour_cur[runs*A] (next entry to visit). */
    double* q; int64_t* picks; int32_t* nplan; int32_t* plan_state; int32_t* pmask; int32_t* ccount; int32_t* cties;
    int32_t* tour_off; int32_t* tour_cur; int64_t* tour;
} mfgp_batch;

/* One iteration of every run: take the exploring agents' samples (:698-713), append them to the model by a block-bordered
 * update of W and z (the reference refits, gaussian_process.py:266-268 / :540-542), add the new rows to the standing
 * posterior (:723), evaluate both partitions -- loss (:194-228), centroids (:231-283), per-cell max variance (:286-323) --
 * write the log rows (:740-768), decide (:771-775, :942-943) and move (:777-782).  Three launches, no host involvement
 * between iterations: the whole run can be captured in one CUDA graph.  b_host / p_host are read on the host. */
int mfgp_batch_step(const mfgp_batch* b_host, const mfgp_params* p_host, int64_t iteration, void* stream);

/* ---- batched Choi (algo 3): per period plan (compute_sample_points :326-374), cluster (compute_sample_clusters :377-412)
 *      and tours (compute_sample_tsp :415-454) for every run, then the period's iterations through mfgp_batch_step ---- */

/* Start of a period: q[g] = |W psi_g|^2 over the rows [0, Ncur) of every run, nplan = 0, plan_state = 0 (1 for a stopped run). */
int mfgp_batch_choi_begin(const mfgp_batch* b_host, const mfgp_params* p_host, void* stream);

/* `rounds` pick rounds without a host synchronisation.  A round advances every planning run by one pick: first-index arg-max
 * of k(0) - q with the tie rule of cov_argmax; if it exceeds `threshold`, the pick is appended to the run's factor as the
 * temporary row Ncur + nplan (bordered update; Ncur, z, mu and var are not touched) and q += v^2 with v the new row of
 * W Psi.  A run whose rows would exceed cap stops with plan_state 2; a non-positive pivot sets status (as the stepper). */
int mfgp_batch_choi_plan(const mfgp_batch* b_host, const mfgp_params* p_host, double threshold, int64_t rounds, void* stream);

/* Cells of every pick in the partition seeded by cen (device-clipped bounded Voronoi cells; nearest seed, the crossings
 * test within TIE_TOL of a bisector): pmask, ccount, cties. */
int mfgp_batch_choi_cluster(const mfgp_batch* b_host, void* stream);

/* Tours of all runs x agents: the clusters (picks of a cell in selection order) are gathered at b->tour_off (the caller's
 * prefix sum of ccount, n_total entries, largest n_max) into pts[n_total,2] / gidx[n_total], ordered by choi_tsp_tours
 * into ord[n_total] (work / work_bytes: as choi_tsp_tours), and stored as grid indices in b->tour; tour_cur = tour_off. */
int mfgp_batch_choi_tours(const mfgp_batch* b_host, int64_t n_total, int64_t n_max, double* pts, int64_t* gidx, int32_t* ord,
                          void* work, int64_t work_bytes, void* stream);

/* ---- hyper-parameter training: replaces SFGP.likelihood / MFGP.likelihood gaussian_process.py:81-105, :344-384 and the
 *      autograd gradient behind SFGP.train / MFGP.train :107-119, :386-399 ------------------------------------------- */

/* Negative log marginal likelihood and its analytic gradient for the model whose fit is standing in (L, W, z, Tt) --
 * i.e. after mfgp_build_train_cov -> mfgp_cholesky -> mfgp_tri_inverse -> mfgp_whiten with the hyper-parameters in
 * question (means under the exp() convention of :89, :356-357):
 *   out[0] = 1/2 z.z + sum log diag L + 1/2 N log 2 pi            (:102-104, :381-383)
 *   out[1 + k] = d out[0] / d hyp[k] for the LOG-scaled hyper-parameters in the reference's order --
 *   [mu_lo, s^2_lo, L_lo, mu_hi, s^2_hi, L_hi, rho, noise_lo, noise_hi] (multi) or [mu, s^2, L, noise] (single; out[5..9] = 0):
 *   1/2 sum_ij (K^-1 - alpha alpha^T)_ij dK_ij/dh - alpha . dm/dh with alpha = W^T z, K^-1 = W^T W (DMMA tile product) and
 *   the dK/dh terms re-evaluated on the fly in one sweep over the lower triangle.  out: 10 doubles (device).
 *   `work`: mfgp_nlml_workspace_bytes(npad) bytes. */
int64_t mfgp_nlml_workspace_bytes(int64_t npad);
int mfgp_nlml_grad(const double* L, int64_t npad, int64_t ld, const double* W, int64_t ldw, const double* z, const double* Tt,
                   int64_t NL, int64_t NH, const mfgp_params* p_host, double* out, void* work, int64_t work_bytes,
                   void* stream);

/* ---- Choi tour planner: replaces compute_sample_tsp simulator.py:415-454 ------------------------------------------ */

/* Visiting order of every agent's sample points.  The reference calls mlrose.TSPOpt + mlrose.genetic_alg(mutation_prob=0.2,
 * max_attempts=100, random_state=2) per cluster (:435-438); mlrose is an unpinned third-party host routine, so its tour
 * order is not reproducible.  This entry minimises the same objective (length of the closed tour) deterministically:
 * nearest-neighbour construction from point 0 of the cluster (ties -> lowest index), then best-improvement 2-opt with
 * position 0 fixed (ties -> lowest (i, j)) until no segment reversal gains more than 1e-12.  One CTA per cluster, all
 * clusters in one launch.  pts[n_total,2]: the clusters' points back to back; off[A+1]: cluster c owns points
 * [off[c], off[c+1]); n_max = size of the largest cluster; order[n_total]: order[off[c] + k] = LOCAL index (within
 * cluster c) of the k-th point of its tour; moves[A] (optional): 2-opt moves applied.  `work`: only read when
 * n_max > 4096 (choi_tsp_workspace_bytes(n_total) bytes).  Bit-identical to the CPU statement oracle/tsp.py. */
int64_t choi_tsp_workspace_bytes(int64_t n_total);
int choi_tsp_tours(const double* pts, const int32_t* off, int64_t A, int64_t n_total, int64_t n_max, int32_t* order,
                   int32_t* moves, void* work, int64_t work_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MFGP_B200_H */
