// Batched replicate stepper: many INDEPENDENT coverage runs on small grids advance one iteration per launch sequence.
// Replaces, for the replicate sweeps of the reference (runner.py:131-147: Pool.map over 100+ simulations of the same
// experiment; BASELINE config 5: 512 periodic_hmf runs on 64x64 grids), the per-run loop body of simulator.py
// periodic :618-785 / todescato :788-954 / lloyd :508-616:
//     take samples (:698-713)  ->  updt_hifi / updt (:716-721)  ->  predict (:723)  ->  compute_loss, compute_centroids,
//     compute_max_var (:725-733)  ->  log rows (:740-768)  ->  decision (:771-775)  ->  move (:777-782).
// One run at a time this loop is launch-bound (~20 small kernels + host Python per iteration, ~0.5 ms); here THREE launches
// step every run of the batch, the loop state never leaves the device, and the host is not involved between iterations
// (the three launches of an iteration can be replayed from a CUDA graph):
//   batch_append_kernel     one CTA per run: the exploring agents' samples (truth at the position's grid index + the run's
//                           pre-drawn noise), block-bordered update of W = L^-1 and z (the reference refits from scratch,
//                           gaussian_process.py:266-268, :540-542; appended rows only change the trailing block), axis-factor
//                           table rows of the new points;
//   batch_posterior_kernel  the standing posterior takes the new rows' contribution: mu += v_new . z_new, var -= |v_new|^2,
//                           v_new = W_new psi with the separable cross-covariance read from the per-run axis tables;
//   batch_coverage_kernel   one CTA per run: both bounded-Voronoi partitions clipped in place (cov_device.cuh), membership
//                           of every grid point (nearest seed; the reference's crossings test within TIE_TOL of a bisector),
//                           per-cell sums / arg-max with the tie rule of argmax.cuh in a fixed order, O(A) finishing with the
//                           reference's arithmetic, log rows, explore decision, position update.
// Randomness is drawn on the host in the order the reference consumes it and uploaded once (uniforms of todescato's
// Bernoulli draws :943, the N(0, sigma_n) sample noise :707).  Dynamics (centroids, arg-max points, decisions, samples) do
// not depend on how exact bisector ties are resolved (the Lloyd partition is seeded by centroids); the LOSS of an iteration
// whose agents sit on grid points may hold grid points exactly on a bisector, which the reference resolves through Qhull's
// vertex rounding -- those (run, iteration) pairs are counted in `ties` for the host to re-evaluate if it needs them bit-exact.
#include <cfloat>

#include "argmax.cuh"
#include "batched.cuh"
#include "cov_device.cuh"

namespace mfgp {

// training covariance entry between a NEW hifi point (x, y) and training point n of the run -- the operations of
// build_train_cov_kernel (gp_fit.cu), i.e. of gaussian_process.py:523-528 / :253
__device__ __forceinline__ double bt_cov(const DevParams& p, double xi, double yi, double xj, double yj, bool jL) {
    if (p.multi) {
        const double kL = rbf_scaled(xi / p.l_L, yi / p.l_L, xj / p.l_L, yj / p.l_L, p.s_L);
        if (jL) return p.rho * kL;
        const double kH = rbf_scaled(xi / p.l_H, yi / p.l_H, xj / p.l_H, yj / p.l_H, p.s_H);
        return __dadd_rn(__dmul_rn(p.rho2, kL), kH);
    }
    return rbf_scaled(xi / p.l_H, yi / p.l_H, xj / p.l_H, yj / p.l_H, p.s_H);
}

// ---- step 1: samples + block-bordered update of W = L^-1 ---------------------------------------------------------------------
// With K_new = [[K, k], [k^T, kk]], l = W k (N x q), S = kk - l^T l = C C^T:   L_new = [[L, 0], [l^T, C]],
// W_new = [[W, 0], [-C^-1 l^T W, C^-1]],  z_new = W_new,rows (y - m).  q <= A new points per iteration.
__global__ void __launch_bounds__(BT_THREADS) batch_append_kernel(BatchArgs a, int it) {
    extern __shared__ __align__(16) double bsm[];
    __shared__ int s_agent[BT_MAXA];
    __shared__ int s_q, s_N;
    __shared__ double s_S[BT_MAXA][BT_MAXA], s_Ci[BT_MAXA][BT_MAXA], s_xn[BT_MAXA][2];
    const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = BT_THREADS / 32;
    const int cap = a.cap, A = a.A;
    if (tid == 0) {
        int q = 0;
        if (a.status[r] == 0 && a.algo != 0)
            for (int i = 0; i < A; i++)
                if (a.explore[r * A + i]) s_agent[q++] = i;
        s_N = a.Ncur[r];
        if (q > 0 && (s_N + q > cap || a.noise_used[r] + q > a.max_samples)) { a.status[r] = -1; q = 0; }
        s_q = q;
        a.knew[r] = q;
    }
    __syncthreads();
    const int q = s_q, N = s_N;
    if (q == 0) return;
    double* Xt = a.Xt + (int64_t)r * cap * 2;
    double* yv = a.y + (int64_t)r * cap;
    double* W = a.W + (int64_t)r * cap * cap;
    double* z = a.z + (int64_t)r * cap;
    double* kv = bsm;                       // [q][cap]  covariance of the new points with the old ones
    double* lv = bsm + (int64_t)A * cap;            // [q][cap]  l = W k
    if (tid < q) {          // reference simulator.py:698-713: sample = truth at the position's grid point + N(0, sigma_n)
        const int ag = s_agent[tid];
        const long long gi = a.pos_idx[r * A + ag];
        const int used = a.noise_used[r];
        const double sx = a.xy[2 * gi], sy = a.xy[2 * gi + 1];
        const double sample = a.f[gi] + a.noise[(int64_t)r * a.max_samples + used + tid];
        Xt[2 * (N + tid)] = sx; Xt[2 * (N + tid) + 1] = sy;
        yv[N + tid] = sample;
        s_xn[tid][0] = sx; s_xn[tid][1] = sy;
        double* row = a.log_sample + ((int64_t)r * a.max_samples + used + tid) * 5;
        row[0] = (double)it; row[1] = (double)ag; row[2] = sx; row[3] = sy; row[4] = sample;
    }
    __syncthreads();
    if (tid == 0) { a.noise_used[r] += q; a.nsamples[r] += q; }
    for (int e = tid; e < q * N; e += BT_THREADS) {
        const int j = e / N, n = e % N;
        kv[j * cap + n] = bt_cov(a.p, s_xn[j][0], s_xn[j][1], Xt[2 * n], Xt[2 * n + 1], n < a.NL);
    }
    if (tid < q * q) {
        const int j = tid / q, j2 = tid % q;
        double v = a.p.multi ? __dadd_rn(__dmul_rn(a.p.rho2, rbf_scaled(s_xn[j][0] / a.p.l_L, s_xn[j][1] / a.p.l_L, s_xn[j2][0] / a.p.l_L,
                                                                        s_xn[j2][1] / a.p.l_L, a.p.s_L)),
                                         rbf_scaled(s_xn[j][0] / a.p.l_H, s_xn[j][1] / a.p.l_H, s_xn[j2][0] / a.p.l_H, s_xn[j2][1] / a.p.l_H, a.p.s_H))
                                : rbf_scaled(s_xn[j][0] / a.p.l_H, s_xn[j][1] / a.p.l_H, s_xn[j2][0] / a.p.l_H, s_xn[j2][1] / a.p.l_H, a.p.s_H);
        if (j == j2) { v = v + a.p.noise_H; v = v + a.p.jitter; }
        s_S[j][j2] = v;
    }
    __syncthreads();
    // l[n][j] = sum_{m <= n} W[n][m] k[m][j]: a warp per row, lanes over m (coalesced), fixed butterfly
    for (int n = warp; n < N; n += nwarp) {
        double acc[BT_MAXA];
#pragma unroll
        for (int j = 0; j < BT_MAXA; j++) acc[j] = 0.0;
        const double* wr = W + (int64_t)n * cap;
#pragma unroll 4
        for (int m = lane; m <= n; m += 32) {         // (unrolled: four loads of W in flight per lane; same order of the sums)
            const double w = wr[m];
#pragma unroll
            for (int j = 0; j < BT_MAXA; j++)
                if (j < q) acc[j] = fma(w, kv[j * cap + m], acc[j]);
        }
#pragma unroll
        for (int j = 0; j < BT_MAXA; j++)
            if (j < q) {
                const double s = warp_sum_d(acc[j]);
                if (lane == 0) lv[j * cap + n] = s;
            }
    }
    __syncthreads();
    // S = kk - l^T l
    for (int e = warp; e < q * q; e += nwarp) {
        const int j = e / q, j2 = e % q;
        double s = 0.0;
        for (int n = lane; n < N; n += 32) s = fma(lv[j * cap + n], lv[j2 * cap + n], s);
        s = warp_sum_d(s);
        if (lane == 0) s_S[j][j2] -= s;
    }
    __syncthreads();
    if (tid == 0) {          // C = chol(S) (lower), Ci = C^-1; np.linalg.cholesky raises on a non-positive pivot (:254, :529)
        int bad = 0;
        for (int j = 0; j < q && !bad; j++) {
            for (int j2 = 0; j2 <= j; j2++) {
                double s = s_S[j][j2];
                for (int t = 0; t < j2; t++) s -= s_S[j][t] * s_S[j2][t];
                if (j == j2) {
                    if (!(s > 0.0)) { bad = N + j + 1; break; }
                    s_S[j][j] = sqrt(s);
                } else {
                    s_S[j][j2] = s / s_S[j2][j2];
                }
            }
        }
        if (bad) a.status[r] = bad;
        for (int j = 0; j < q; j++)
            for (int j2 = 0; j2 < q; j2++) s_Ci[j][j2] = 0.0;
        if (!bad)
            for (int c = 0; c < q; c++) {          // column c of C^-1 by forward substitution
                for (int j = c; j < q; j++) {
                    double s = (j == c) ? 1.0 : 0.0;
                    for (int t = c; t < j; t++) s -= s_S[j][t] * s_Ci[t][c];
                    s_Ci[j][c] = s / s_S[j][j];
                }
            }
        s_q = bad ? 0 : q;
    }
    __syncthreads();
    if (s_q == 0) { if (tid == 0) a.knew[r] = 0; return; }
    // t[j][m] = sum_{n >= m} l[n][j] W[n][m]  (a thread per column m: coalesced over m for every n), then
    // W_new[j][m] = -sum_{j2 <= j} Ci[j][j2] t[j2][m]
    for (int m = tid; m < N; m += BT_THREADS) {
        double t[BT_MAXA];
#pragma unroll
        for (int j = 0; j < BT_MAXA; j++) t[j] = 0.0;
#pragma unroll 4
        for (int n = m; n < N; n++) {
            const double w = W[(int64_t)n * cap + m];
#pragma unroll
            for (int j = 0; j < BT_MAXA; j++)
                if (j < q) t[j] = fma(lv[j * cap + n], w, t[j]);
        }
#pragma unroll
        for (int j = 0; j < BT_MAXA; j++)
            if (j < q) {
                double s = 0.0;
#pragma unroll
                for (int j2 = 0; j2 < BT_MAXA; j2++)
                    if (j2 <= j) s = fma(s_Ci[j][j2], t[j2], s);
                W[(int64_t)(N + j) * cap + m] = -s;
            }
    }
    if (tid < q * q) {
        const int j = tid / q, j2 = tid % q;
        W[(int64_t)(N + j) * cap + N + j2] = (j2 <= j) ? s_Ci[j][j2] : 0.0;
    }
    // axis-factor table rows of the new points: e(u, U) = exp(-0.5 ((u - U) / l)^2) with the division first (:77-78)
    for (int e = tid; e < q * (a.nx + a.ny); e += BT_THREADS) {
        const int j = e / (a.nx + a.ny), i = e % (a.nx + a.ny);
        const bool isx = i < a.nx;
        const double u = isx ? a.ux[i] : a.uy[i - a.nx], U = s_xn[j][isx ? 0 : 1];
        const double dH = u / a.p.l_H - U / a.p.l_H;
        const int64_t row = (int64_t)r * cap + N + j;
        if (isx) a.TxH[row * a.nx + i] = exp(-0.5 * (dH * dH)); else a.TyH[row * a.ny + (i - a.nx)] = exp(-0.5 * (dH * dH));
        if (a.p.multi) {
            const double dL = u / a.p.l_L - U / a.p.l_L;
            if (isx) a.TxL[row * a.nx + i] = exp(-0.5 * (dL * dL)); else a.TyL[row * a.ny + (i - a.nx)] = exp(-0.5 * (dL * dL));
        }
    }
    __syncthreads();
    // z_new[j] = W_new[j][:] (y - m): a warp per new row
    for (int j = warp; j < q; j += nwarp) {
        const double* wr = W + (int64_t)(N + j) * cap;
        double s = 0.0;
        for (int m = lane; m < N + q; m += 32) s = fma(wr[m], yv[m] - (m < a.NL ? a.p.mean_L : a.p.mean_H), s);
        s = warp_sum_d(s);
        if (lane == 0) z[N + j] = s;
    }
    if (tid == 0) a.Ncur[r] = N + q;
}

// ---- step 2: the standing posterior takes the new rows ---------------------------------------------------------------------
__global__ void __launch_bounds__(BT_THREADS) batch_posterior_kernel(BatchArgs a) {
    const int r = blockIdx.y;
    const int q = a.knew[r];
    if (q == 0 || a.status[r] != 0) return;
    const int g = blockIdx.x * BT_THREADS + threadIdx.x;
    if (g >= a.G) return;
    const int Nn = a.Ncur[r], N0 = Nn - q, cap = a.cap;
    const int ix = g / a.ny, iy = g % a.ny;
    const double* W = a.W + (int64_t)r * cap * cap + (int64_t)N0 * cap;
    const double* TxH = a.TxH + (int64_t)r * cap * a.nx;
    const double* TyH = a.TyH + (int64_t)r * cap * a.ny;
    const double* TxL = a.TxL + (int64_t)r * cap * a.nx;
    const double* TyL = a.TyL + (int64_t)r * cap * a.ny;
    double v[BT_MAXA];
#pragma unroll
    for (int j = 0; j < BT_MAXA; j++) v[j] = 0.0;
    const double cLL = a.p.rho * a.p.s_L, cLH = a.p.rho2 * a.p.s_L;      // gaussian_process.py:426-429
    for (int n = 0; n < Nn; n++) {
        double psi = 0.0;
        if (n >= a.NL) psi = a.p.s_H * (__ldg(TxH + (int64_t)n * a.nx + ix) * __ldg(TyH + (int64_t)n * a.ny + iy));
        if (a.p.multi) psi = fma(n < a.NL ? cLL : cLH, __ldg(TxL + (int64_t)n * a.nx + ix) * __ldg(TyL + (int64_t)n * a.ny + iy), psi);
#pragma unroll
        for (int j = 0; j < BT_MAXA; j++)
            if (j < q) v[j] = fma(__ldg(W + (int64_t)j * cap + n), psi, v[j]);
    }
    const double* z = a.z + (int64_t)r * cap + N0;
    double dm = 0.0, dq = 0.0;
#pragma unroll
    for (int j = 0; j < BT_MAXA; j++)
        if (j < q) { dm = fma(v[j], z[j], dm); dq = fma(v[j], v[j], dq); }
    a.mu[(int64_t)r * a.G + g] += dm;
    a.var[(int64_t)r * a.G + g] -= dq;
}

// The same update with PT consecutive grid points (same ix) per thread: the q loads of W_new[:, n] and the two x-table entries of
// a training point serve PT points, the y-table entries come as 16-byte loads -- 14 loads for 44 FMAs (q = 8, PT = 4) instead of
// 12 for 11.  Per point the same operations in the same order as batch_posterior_kernel: bitwise the same results.
template <int QM, int PT>          // q <= QM appended rows, PT in {2, 4} points per thread (ny % PT == 0)
__global__ void __launch_bounds__(BT_THREADS) batch_posterior_tiled_kernel(BatchArgs a) {
    const int r = blockIdx.y;
    const int q = a.knew[r];
    if (q == 0 || a.status[r] != 0) return;
    const int g = (blockIdx.x * BT_THREADS + threadIdx.x) * PT;
    if (g >= a.G) return;
    const int Nn = a.Ncur[r], N0 = Nn - q, cap = a.cap;
    const int ix = g / a.ny, iy = g % a.ny;
    const double* W = a.W + (int64_t)r * cap * cap + (int64_t)N0 * cap;
    const double* TxH = a.TxH + (int64_t)r * cap * a.nx + ix;
    const double* TyH = a.TyH + (int64_t)r * cap * a.ny + iy;
    const double* TxL = a.TxL + (int64_t)r * cap * a.nx + ix;
    const double* TyL = a.TyL + (int64_t)r * cap * a.ny + iy;
    double v[QM][PT];
#pragma unroll
    for (int j = 0; j < QM; j++)
#pragma unroll
        for (int p = 0; p < PT; p++) v[j][p] = 0.0;
    const double cLL = a.p.rho * a.p.s_L, cLH = a.p.rho2 * a.p.s_L;      // gaussian_process.py:426-429
    for (int n = 0; n < Nn; n++) {
        double psi[PT];
#pragma unroll
        for (int p = 0; p < PT; p++) psi[p] = 0.0;
        if (n >= a.NL) {
            const double tx = __ldg(TxH + (int64_t)n * a.nx);
#pragma unroll
            for (int p = 0; p < PT; p += 2) {
                const double2 ty = __ldg(reinterpret_cast<const double2*>(TyH + (int64_t)n * a.ny + p));
                psi[p] = a.p.s_H * (tx * ty.x); psi[p + 1] = a.p.s_H * (tx * ty.y);
            }
        }
        if (a.p.multi) {
            const double c = n < a.NL ? cLL : cLH, tx = __ldg(TxL + (int64_t)n * a.nx);
#pragma unroll
            for (int p = 0; p < PT; p += 2) {
                const double2 ty = __ldg(reinterpret_cast<const double2*>(TyL + (int64_t)n * a.ny + p));
                psi[p] = fma(c, tx * ty.x, psi[p]); psi[p + 1] = fma(c, tx * ty.y, psi[p + 1]);
            }
        }
#pragma unroll
        for (int j = 0; j < QM; j++)
            if (j < q) {
                const double w = __ldg(W + (int64_t)j * cap + n);
#pragma unroll
                for (int p = 0; p < PT; p++) v[j][p] = fma(w, psi[p], v[j][p]);
            }
    }
    const double* z = a.z + (int64_t)r * cap + N0;
#pragma unroll
    for (int p = 0; p < PT; p++) {
        double dm = 0.0, dq = 0.0;
#pragma unroll
        for (int j = 0; j < QM; j++)
            if (j < q) { dm = fma(v[j][p], z[j], dm); dq = fma(v[j][p], v[j][p], dq); }
        a.mu[(int64_t)r * a.G + g + p] += dm;
        a.var[(int64_t)r * a.G + g + p] -= dq;
    }
}

// ---- step 3: coverage step, finishing, log, decision, move -------------------------------------------------------------------
constexpr int BC_SLOTS = 8;          // per cell: sum w, sum w x, sum w y, count, max var, arg-max index, loss sum, loss count
constexpr int BC_MAXV = 24;          // a cell of <= 16 seeds in a box has at most 4 + 15 vertices

__global__ void __launch_bounds__(BT_THREADS) batch_coverage_kernel(BatchArgs a, int it) {
    extern __shared__ __align__(16) unsigned short s_mask[];    // [2][G] membership bit masks (Lloyd partition, loss partition)
    __shared__ double s_seed[2][BT_MAXA][2];                    // [0]: Lloyd partition (centroids), [1]: loss partition (positions)
    __shared__ double s_poly[2][BT_MAXA][2 * BC_MAXV];
    __shared__ int s_cnt[2][BT_MAXA];
    __shared__ double s_area[2][BT_MAXA];
    __shared__ double s_buf[BT_THREADS / 32][256];
    __shared__ double s_tot[BT_MAXA][BC_SLOTS];
    __shared__ int s_ties, s_bad;
    const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = BT_THREADS / 32;
    const int A = a.A;
    if (a.status[r] != 0) return;
    double* pos = a.pos + (int64_t)r * A * 2;
    double* prev = a.prev + (int64_t)r * A * 2;
    double* cen = a.cen + (int64_t)r * A * 2;
    const bool thompson = a.algo == 4;          // both partitions seeded by the positions; the draw stage moves the agents
    if (tid < 2 * A) { s_seed[0][tid >> 1][tid & 1] = thompson ? pos[tid] : cen[tid]; s_seed[1][tid >> 1][tid & 1] = pos[tid]; }
    if (thompson) {          // grid index of the training rows this iteration appended (every agent samples, in agent order)
        const int q = a.knew[r];
        if (tid < q) a.rowidx[(int64_t)r * a.cap + a.Ncur[r] - q + tid] = (int)a.pos_idx[r * A + tid];
    }
    if (tid == 0) { s_ties = 0; s_bad = 0; }
    __syncthreads();
    // bounded Voronoi cells of both partitions: the box inflated by eps/2 clipped by the bisectors (simulator.py:154-191)
    const double h = 0.5 * a.eps;
    for (int c = warp; c < 2 * A; c += nwarp) {
        const int part = c / A, i = c % A;
        bool overflow = false;
        int which = 0;
        const int n = vc_clip_cell(&s_seed[part][0][0], A, i, a.xmin - h, a.xmax + h, a.ymin - h, a.ymax + h, s_buf[warp], lane, overflow, which);
        const double* px = s_buf[warp] + 128 * which;
        const double* py = px + 64;
        if (n > BC_MAXV) overflow = true;
        for (int v = lane; v < n && v < BC_MAXV; v += 32) { s_poly[part][i][2 * v] = px[v]; s_poly[part][i][2 * v + 1] = py[v]; }
        if (lane == 0) {
            double s1 = 0.0, s2 = 0.0;
            for (int v = 0; v < n; v++) {
                const int u = (v + n - 1) % n;
                s1 += px[v] * py[u];
                s2 += py[v] * px[u];
            }
            s_cnt[part][i] = n < BC_MAXV ? n : BC_MAXV;
            s_area[part][i] = 0.5 * fabs(s1 - s2);
            if (overflow) s_bad = 1;
        }
        __syncwarp();
    }
    __syncthreads();
    const double* w = (a.algo == 0) ? a.f : a.mu + (int64_t)r * a.G;
    const double* var = a.var + (int64_t)r * a.G;
    const bool with_var = a.algo != 0;
    const TieRule tol{a.p.k0, a.amax_rel};
    // pass 1: membership masks of every grid point in both partitions
    int hard = 0;
    for (int g = tid; g < a.G; g += BT_THREADS) {
        const double x = a.xy[2 * g], y = a.xy[2 * g + 1];
#pragma unroll
        for (int part = 0; part < 2; part++) {
            double best = DBL_MAX, second = DBL_MAX;
            int bi = 0;
            for (int c = 0; c < A; c++) {
                const double dx = x - s_seed[part][c][0], dy = y - s_seed[part][c][1];
                const double d = fma(dx, dx, dy * dy);
                if (d < best) { second = best; best = d; bi = c; }
                else if (d < second) second = d;
            }
            const double gap = second - best;
            unsigned mask = 0;
            if (gap > a.tie_tol) {
                mask = 1u << bi;
            } else {                                   // within TIE_TOL of a bisector: the reference's crossings test decides
                if (!(gap > 0.1 * a.tie_tol)) hard++;
                for (int c = 0; c < A; c++)
                    if (crossings_inside(s_poly[part][c], s_cnt[part][c], x, y)) mask |= 1u << c;
            }
            s_mask[part * a.G + g] = (unsigned short)mask;
            if (thompson && part == 0) a.cmask[(int64_t)r * a.G + g] = (unsigned short)mask;
        }
    }
    if (hard) atomicAdd(&s_ties, hard);
    __syncthreads();
    // pass 2: a warp per cell; lanes stride over the grid in index order, one fixed butterfly per quantity
    for (int c = warp; c < A; c += nwarp) {
        double sw = 0.0, swx = 0.0, swy = 0.0, sl = 0.0;
        int cn = 0, ln = 0;
        ArgMax am{0.0, -1};
        const unsigned short bit = (unsigned short)(1u << c);
        const double sx = s_seed[1][c][0], sy = s_seed[1][c][1];
        for (int g = lane; g < a.G; g += 32) {
            if (s_mask[g] & bit) {
                const double x = a.xy[2 * g], y = a.xy[2 * g + 1], wv = w[g];
                sw += wv; swx += wv * x; swy += wv * y; cn++;
                if (with_var) am = argmax_combine(am, ArgMax{var[g], (long long)g}, tol);
            }
            if (s_mask[a.G + g] & bit) {
                const double dx = a.xy[2 * g] - sx, dy = a.xy[2 * g + 1] - sy;
                sl += __dmul_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), a.f[g]);     // simulator.py:215-216
                ln++;
            }
        }
        const double t0 = warp_sum_d(sw), t1 = warp_sum_d(swx), t2 = warp_sum_d(swy), t3 = warp_sum_d(sl);
        const int n0 = __reduce_add_sync(0xffffffffu, cn), n1 = __reduce_add_sync(0xffffffffu, ln);
        const ArgMax m = with_var ? argmax_warp(am, tol) : ArgMax{0.0, -1};
        if (lane == 0) {
            double* o = s_tot[c];
            o[0] = t0; o[1] = t1; o[2] = t2; o[3] = (double)n0; o[4] = m.v; o[5] = __longlong_as_double(m.i); o[6] = t3; o[7] = (double)n1;
            if (with_var && m.i < 0) s_bad = 2;          // np.amax([]) raises ValueError (simulator.py:312)
        }
    }
    __syncthreads();
    if (tid == 0) {
        a.ties[(int64_t)r * a.iterations + it] = s_ties;
        if (s_bad) a.status[r] = (s_bad == 2) ? -4 : -5;
        double loss = 0.0;                                 // simulator.py:215-219, cell order
        for (int c = 0; c < A; c++) loss += (s_tot[c][6] / s_tot[c][7]) * s_area[1][c];
        a.log_loss[(int64_t)r * a.iterations + it] = loss;
    }
    if (tid < A) {          // centroid (simulator.py:256-271), log row (:740-768), decision (:771-775 / :942-943), move (:777-782)
        const int i = tid;
        const double n = s_tot[i][3], ar = s_area[0][i];
        const double f_int = (s_tot[i][0] / n) * ar;
        double cx = ((s_tot[i][1] / n) * ar) / f_int, cy = ((s_tot[i][2] / n) * ar) / f_int;
        if (cx < a.xmin) cx = a.xmin;
        if (cx > a.xmax) cx = a.xmax;
        if (cy < a.ymin) cy = a.ymin;
        if (cy > a.ymax) cy = a.ymax;
        const double px = pos[2 * i], py = pos[2 * i + 1];
        const double ddx = px - prev[2 * i], ddy = py - prev[2 * i + 1];
        const double dist = sqrt(ddx * ddx + ddy * ddy);
        const long long gi = __double_as_longlong(s_tot[i][5]);
        const double mv = with_var ? s_tot[i][4] : 0.0;
        const double axm = (with_var && gi >= 0) ? a.xy[2 * gi] : 0.0, aym = (with_var && gi >= 0) ? a.xy[2 * gi + 1] : 0.0;
        double* row = a.log_agent + (((int64_t)r * a.iterations + it) * A + i) * BT_LOGC;
        row[0] = px; row[1] = py; row[2] = axm; row[3] = py; row[4] = mv; row[5] = with_var ? a.p.k0 : 0.0;
        row[6] = cx; row[7] = cy; row[8] = a.prob[r * A + i]; row[9] = (double)a.explore[r * A + i]; row[10] = dist;
        if (thompson) {          // every agent samples from the next iteration on; the draw stage fills XCentroid / YCentroid
            row[8] = 1.0; row[9] = 1.0;
            a.prob[r * A + i] = 1.0;
            a.explore[r * A + i] = 1;
            a.ccell[((int64_t)r * A + i) * 2] = n;
            a.ccell[((int64_t)r * A + i) * 2 + 1] = ar;
            return;
        }
        int ex = 0;
        double pr = 0.0;
        long long tgi = -1;
        if (a.algo == 1) { ex = ((it / 5) % 2 == 0) ? 1 : 0; pr = (double)ex; }
        else if (a.algo == 2) {
            pr = sqrt(mv / (a.p.k0 * (double)A));              // todescato_prob, simulator.py:457-467
            ex = a.unif[((int64_t)r * a.iterations + it) * A + i] < pr ? 1 : 0;
        }
        else if (a.algo == 3) {          // Choi: explore while the tour has points left, visit its next point (simulator.choi)
            const int k = r * A + i, cur = a.tour_cur[k];
            ex = cur < a.tour_off[k + 1] ? 1 : 0;
            pr = (double)ex;
            if (ex) { tgi = a.tour[cur]; a.tour_cur[k] = cur + 1; }
        }
        a.prob[r * A + i] = pr;
        a.explore[r * A + i] = ex;
        prev[2 * i] = px; prev[2 * i + 1] = py;
        if (a.algo == 0 || !ex) { pos[2 * i] = cx; pos[2 * i + 1] = cy; a.pos_idx[r * A + i] = -1; }
        else if (a.algo == 3) { pos[2 * i] = a.xy[2 * tgi]; pos[2 * i + 1] = a.xy[2 * tgi + 1]; a.pos_idx[r * A + i] = tgi; }
        else { pos[2 * i] = axm; pos[2 * i + 1] = aym; a.pos_idx[r * A + i] = gi; }
        cen[2 * i] = cx; cen[2 * i + 1] = cy;
    }
}


// ---- Choi (algo 3): the per-period planner, clusters and tours of every run ---------------------------------------------------
// The greedy planner of compute_sample_points (simulator.py:326-374) picks arg-max_g (k0 - q[g]) until it is <= threshold,
// each pick conditioning a COPY of the model on one more hifi point.  Here a pick is appended to the run's own factor as the
// temporary row Ncur + k (q = 1 case of the bordered update of batch_append_kernel); Ncur does not move, so the run's model is
// unchanged and the next real sample overwrites the row.  The planner's variance is k0 - q with q = |W psi|^2 accumulated from
// a recomputation at the period start, never the stepper's decremented var: far from the data q ~ ulp(k0), and the first
// index of the top 1-ulp plateau is what the reference picks (argmax.cuh).

constexpr int CQ_ROWS = 8;

// period start: q[g] = |W psi_g|^2 over the rows [0, Ncur) of the run; rows of W in CQ_ROWS-row strips, psi recomputed per strip
__global__ void __launch_bounds__(BT_THREADS) batch_choi_q_kernel(BatchArgs a) {
    const int r = blockIdx.y;
    const int g = blockIdx.x * BT_THREADS + threadIdx.x;
    if (blockIdx.x == 0 && threadIdx.x == 0) { a.nplan[r] = 0; a.plan_state[r] = a.status[r] != 0 ? 1 : 0; }
    if (g >= a.G) return;
    const int N = a.Ncur[r], cap = a.cap, ix = g / a.ny, iy = g % a.ny;
    const double* W = a.W + (int64_t)r * cap * cap;
    double q = 0.0;
    for (int n0 = 0; n0 < N; n0 += CQ_ROWS) {
        const int hi = min(n0 + CQ_ROWS, N);
        double acc[CQ_ROWS];
#pragma unroll
        for (int j = 0; j < CQ_ROWS; j++) acc[j] = 0.0;
        for (int m = 0; m < hi; m++) {
            const double psi = bt_psi(a, r, m, ix, iy);
#pragma unroll
            for (int j = 0; j < CQ_ROWS; j++)
                if (n0 + j < hi && m <= n0 + j) acc[j] = fma(__ldg(W + (int64_t)(n0 + j) * cap + m), psi, acc[j]);
        }
#pragma unroll
        for (int j = 0; j < CQ_ROWS; j++)
            if (n0 + j < hi) q = fma(acc[j], acc[j], q);
    }
    a.q[(int64_t)r * a.G + g] = q;
}

// one pick of every planning run: arg-max, bordered append of the pick as row n = Ncur + k, q += v^2 with v = W[n, :] psi
__global__ void __launch_bounds__(BT_THREADS) batch_choi_pick_kernel(BatchArgs a, double threshold) {
    extern __shared__ __align__(16) double csm[];      // kv[cap] (covariance with rows < n), l[cap] = W kv, w[cap] = new row of W
    __shared__ double s_v[BT_THREADS / 32];
    __shared__ long long s_i[BT_THREADS / 32];
    __shared__ double s_ci;
    __shared__ int s_go;
    const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = BT_THREADS / 32;
    if (a.plan_state[r] != 0 || a.status[r] != 0) return;
    const int cap = a.cap, k = a.nplan[r], n = a.Ncur[r] + k;
    const TieRule tol{a.p.k0, a.amax_rel};
    double* q = a.q + (int64_t)r * a.G;
    ArgMax best{0.0, -1};
    for (int g = tid; g < a.G; g += BT_THREADS) best = argmax_combine(best, ArgMax{a.p.k0 - q[g], (long long)g}, tol);
    best = argmax_warp(best, tol);
    if (lane == 0) { s_v[warp] = best.v; s_i[warp] = best.i; }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < nwarp; w++) best = argmax_combine(best, ArgMax{s_v[w], s_i[w]}, tol);
        int go = 0;
        if (!(best.v > threshold)) a.plan_state[r] = 1;                   // while max var > threshold (:345)
        else if (n + 1 > cap) a.plan_state[r] = 2;                       // the host grows the buffers and resumes
        else { a.picks[(int64_t)r * cap + k] = best.i; go = 1; }
        s_go = go;
        s_i[0] = best.i;
    }
    __syncthreads();
    if (!s_go) return;
    const long long pick = s_i[0];
    const double xs = a.xy[2 * pick], ys = a.xy[2 * pick + 1];
    double* Xt = a.Xt + (int64_t)r * cap * 2;
    double* W = a.W + (int64_t)r * cap * cap;
    double* kv = csm;
    double* lv = csm + cap;
    double* wn = csm + 2 * cap;
    const int pix = (int)(pick / a.ny), piy = (int)(pick % a.ny);      // the pick is a grid point: its covariances are table entries
    for (int m = tid; m < n; m += BT_THREADS) kv[m] = bt_psi(a, r, m, pix, piy);
    __syncthreads();
    for (int nn = warp; nn < n; nn += nwarp) {          // l = W kv: a warp per row
        const double* wr = W + (int64_t)nn * cap;
        double s = 0.0;
        for (int m = lane; m <= nn; m += 32) s = fma(wr[m], kv[m], s);
        s = warp_sum_d(s);
        if (lane == 0) lv[nn] = s;
    }
    __syncthreads();
    if (warp == 0) {          // d^2 = k(x, x) + noise_H + jitter - l.l; np.linalg.cholesky raises on a non-positive pivot
        double s = 0.0;
        for (int m = lane; m < n; m += 32) s = fma(lv[m], lv[m], s);
        s = warp_sum_d(s);
        if (lane == 0) {
            const double xh = xs / a.p.l_H, yh = ys / a.p.l_H;
            double kk = rbf_scaled(xh, yh, xh, yh, a.p.s_H);
            if (a.p.multi) {
                const double xl = xs / a.p.l_L, yl = ys / a.p.l_L;
                kk = __dadd_rn(__dmul_rn(a.p.rho2, rbf_scaled(xl, yl, xl, yl, a.p.s_L)), kk);
            }
            kk = kk + a.p.noise_H;
            kk = kk + a.p.jitter;
            const double d2 = kk - s;
            if (!(d2 > 0.0)) { a.status[r] = n + 1; s_ci = 0.0; }
            else s_ci = 1.0 / sqrt(d2);
        }
    }
    __syncthreads();
    const double ci = s_ci;
    if (ci == 0.0) return;
    for (int m = tid; m < n; m += BT_THREADS) {        // W[n][m] = -ci sum_{nn >= m} l[nn] W[nn][m]
        double t = 0.0;
        for (int nn = m; nn < n; nn++) t = fma(lv[nn], W[(int64_t)nn * cap + m], t);
        const double w = -(ci * t);
        wn[m] = w;
        W[(int64_t)n * cap + m] = w;
    }
    if (tid == 0) {
        wn[n] = ci;
        W[(int64_t)n * cap + n] = ci;
        Xt[2 * n] = xs; Xt[2 * n + 1] = ys;
        a.nplan[r] = k + 1;
    }
    for (int i = tid; i < a.nx + a.ny; i += BT_THREADS) {      // axis-table rows of the pick (batch_append_kernel)
        const bool isx = i < a.nx;
        const double u = isx ? a.ux[i] : a.uy[i - a.nx], U = isx ? xs : ys;
        const double dH = u / a.p.l_H - U / a.p.l_H;
        const int64_t row = (int64_t)r * cap + n;
        if (isx) a.TxH[row * a.nx + i] = exp(-0.5 * (dH * dH)); else a.TyH[row * a.ny + (i - a.nx)] = exp(-0.5 * (dH * dH));
        if (a.p.multi) {
            const double dL = u / a.p.l_L - U / a.p.l_L;
            if (isx) a.TxL[row * a.nx + i] = exp(-0.5 * (dL * dL)); else a.TyL[row * a.ny + (i - a.nx)] = exp(-0.5 * (dL * dL));
        }
    }
    __syncthreads();
    for (int g = tid; g < a.G; g += BT_THREADS) {
        const int ix = g / a.ny, iy = g % a.ny;
        double v = 0.0;
        for (int m = 0; m <= n; m++) v = fma(wn[m], bt_psi(a, r, m, ix, iy), v);
        q[g] += v * v;
    }
}

// cells of the period's picks in the partition seeded by the centroids (simulator.py:651-653, :377-412): nearest seed, and
// within TIE_TOL of a bisector the crossings test against the device-clipped cells (pass 1 of batch_coverage_kernel).  A pick
// in no cell is dropped, a pick in several cells joins each of them.  Hard ties (gap <= TIE_TOL/10) are counted: there the
// reference's Qhull vertices decide, and the host re-runs such runs on the single-run path.
__global__ void __launch_bounds__(BT_THREADS) batch_choi_cluster_kernel(BatchArgs a) {
    __shared__ double s_seed[BT_MAXA][2];
    __shared__ double s_poly[BT_MAXA][2 * BC_MAXV];
    __shared__ int s_cnt[BT_MAXA];
    __shared__ double s_buf[BT_THREADS / 32][256];
    __shared__ int s_ties, s_bad;
    const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = BT_THREADS / 32;
    const int A = a.A, cap = a.cap;
    const int k = a.status[r] == 0 ? a.nplan[r] : 0;
    if (tid < 2 * A) s_seed[tid >> 1][tid & 1] = a.cen[(int64_t)r * A * 2 + tid];
    if (tid == 0) { s_ties = 0; s_bad = 0; }
    __syncthreads();
    const double h = 0.5 * a.eps;
    for (int i = warp; i < A && k > 0; i += nwarp) {
        bool overflow = false;
        int which = 0;
        const int nv = vc_clip_cell(&s_seed[0][0], A, i, a.xmin - h, a.xmax + h, a.ymin - h, a.ymax + h, s_buf[warp], lane, overflow, which);
        const double* px = s_buf[warp] + 128 * which;
        const double* py = px + 64;
        if (nv > BC_MAXV) overflow = true;
        for (int v = lane; v < nv && v < BC_MAXV; v += 32) { s_poly[i][2 * v] = px[v]; s_poly[i][2 * v + 1] = py[v]; }
        if (lane == 0) {
            s_cnt[i] = nv < BC_MAXV ? nv : BC_MAXV;
            if (overflow) s_bad = 1;
        }
        __syncwarp();
    }
    __syncthreads();
    int hard = 0;
    for (int j = tid; j < k; j += BT_THREADS) {
        const long long g = a.picks[(int64_t)r * cap + j];
        const double x = a.xy[2 * g], y = a.xy[2 * g + 1];
        double best = DBL_MAX, second = DBL_MAX;
        int bi = 0;
        for (int c = 0; c < A; c++) {
            const double dx = x - s_seed[c][0], dy = y - s_seed[c][1];
            const double d = fma(dx, dx, dy * dy);
            if (d < best) { second = best; best = d; bi = c; }
            else if (d < second) second = d;
        }
        const double gap = second - best;
        unsigned mask = 0;
        if (gap > a.tie_tol) {
            mask = 1u << bi;
        } else {
            if (!(gap > 0.1 * a.tie_tol)) hard++;
            for (int c = 0; c < A; c++)
                if (crossings_inside(s_poly[c], s_cnt[c], x, y)) mask |= 1u << c;
        }
        a.pmask[(int64_t)r * cap + j] = (int)mask;
    }
    if (hard) atomicAdd(&s_ties, hard);
    __syncthreads();
    for (int c = warp; c < A; c += nwarp) {
        int cn = 0;
        for (int j = lane; j < k; j += 32) cn += (a.pmask[(int64_t)r * cap + j] >> c) & 1;
        cn = __reduce_add_sync(0xffffffffu, cn);
        if (lane == 0) a.ccount[r * A + c] = cn;
    }
    if (tid == 0) {
        a.cties[r] = s_ties;
        if (s_bad) a.status[r] = -5;
    }
}

// cluster (r, c) = the picks of run r in cell c, in selection order, at tour_off[r*A + c]: coordinates for the tour planner
__global__ void batch_choi_gather_kernel(BatchArgs a, double* pts, long long* gidx) {
    const int rc = blockIdx.x * blockDim.x + threadIdx.x;
    if (rc >= a.runs * a.A) return;
    const int r = rc / a.A, c = rc % a.A, cap = a.cap;
    int o = a.tour_off[rc];
    a.tour_cur[rc] = o;
    if (a.ccount[rc] == 0) return;
    const int k = a.nplan[r];
    for (int j = 0; j < k; j++)
        if ((a.pmask[(int64_t)r * cap + j] >> c) & 1) {
            const long long g = a.picks[(int64_t)r * cap + j];
            pts[2 * (int64_t)o] = a.xy[2 * g]; pts[2 * (int64_t)o + 1] = a.xy[2 * g + 1];
            gidx[o++] = g;
        }
}

// tour of (r, c) as grid indices in visiting order (ord: local indices from tsp_tours_kernel)
__global__ void batch_choi_order_kernel(BatchArgs a, const long long* gidx, const int32_t* ord) {
    const int rc = blockIdx.x * blockDim.x + threadIdx.x;
    if (rc >= a.runs * a.A) return;
    const int o0 = a.tour_off[rc], o1 = a.tour_off[rc + 1];
    for (int t = o0; t < o1; t++) a.tour[t] = gidx[o0 + ord[t]];
}

bool batch_valid(const mfgp_batch* b, const mfgp_params* p_host) {
    return b && p_host && b->runs > 0 && b->A > 0 && b->A <= BT_MAXA && b->G > 0 && b->nx * b->ny == b->G && b->cap > 0 &&
           b->algo >= 0 && b->algo <= 4 && (b->algo != 3 || (b->tour_off && b->tour_cur)) &&
           (b->algo != 4 || (b->seed && b->cmask && b->ccell && b->rowidx));
}

BatchArgs batch_args(const mfgp_batch* b, const mfgp_params* p_host) {
    BatchArgs a{};
    a.runs = (int)b->runs; a.G = (int)b->G; a.nx = (int)b->nx; a.ny = (int)b->ny; a.A = (int)b->A; a.NL = (int)b->NL;
    a.cap = (int)b->cap; a.algo = (int)b->algo; a.iterations = (int)b->iterations; a.max_samples = (int)b->max_samples;
    a.xmin = b->xmin; a.xmax = b->xmax; a.ymin = b->ymin; a.ymax = b->ymax; a.eps = b->eps; a.tie_tol = b->tie_tol;
    a.amax_rel = b->amax_rel; a.p = make_dev_params(*p_host);
    a.xy = b->xy; a.f = b->f; a.ux = b->ux; a.uy = b->uy; a.Xt = b->Xt; a.y = b->y; a.W = b->W; a.z = b->z;
    a.TxL = b->TxL; a.TyL = b->TyL; a.TxH = b->TxH; a.TyH = b->TyH; a.mu = b->mu; a.var = b->var; a.pos = b->pos; a.prev = b->prev;
    a.cen = b->cen; a.pos_idx = reinterpret_cast<long long*>(b->pos_idx); a.prob = b->prob; a.explore = b->explore;
    a.Ncur = b->Ncur; a.knew = b->knew; a.status = b->status; a.noise_used = b->noise_used; a.nsamples = b->nsamples;
    a.ties = b->ties; a.noise = b->noise; a.unif = b->unif; a.log_loss = b->log_loss; a.log_agent = b->log_agent;
    a.log_sample = b->log_sample;
    a.q = b->q; a.picks = reinterpret_cast<long long*>(b->picks); a.nplan = b->nplan; a.plan_state = b->plan_state;
    a.pmask = b->pmask; a.ccount = b->ccount; a.cties = b->cties; a.tour_off = b->tour_off; a.tour_cur = b->tour_cur;
    a.tour = reinterpret_cast<long long*>(b->tour);
    a.seed = reinterpret_cast<const long long*>(b->seed); a.cmask = reinterpret_cast<unsigned short*>(b->cmask); a.ccell = b->ccell;
    a.rowidx = b->rowidx;
    return a;
}

}  // namespace mfgp

using namespace mfgp;

// Layout of the caller-provided state block (doubles unless noted), per run r and in this order:
//   Xt[cap*2] y[cap] W[cap*cap] z[cap] TxL[cap*nx] TyL[cap*ny] TxH[cap*nx] TyH[cap*ny] mu[G] var[G] pos[2A] prev[2A] cen[2A]
//   prob[A] | int64: pos_idx[A] | int32: explore[A] Ncur knew status noise_used nsamples ties[iterations]
// (the host module mfgp-coverage_b200/_batched.py owns the buffers; this file only receives pointers)
extern "C" {

/* struct mfgp_batch: include/mfgp_b200.h */

int mfgp_batch_step(const mfgp_batch* b, const mfgp_params* p_host, int64_t iteration, void* stream) {
    if (!batch_valid(b, p_host) || iteration < 0 || iteration >= b->iterations) return MFGP_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const BatchArgs a = batch_args(b, p_host);
    if (a.algo != 0) {
        const size_t smem = sizeof(double) * 2 * (size_t)a.A * (size_t)a.cap;
        if (smem > 200 * 1024) return MFGP_ERR_INVALID;
        MFGP_CUDA_CHECK(cudaFuncSetAttribute(batch_append_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        batch_append_kernel<<<a.runs, BT_THREADS, smem, st>>>(a, (int)iteration);
        MFGP_LAUNCH_CHECK();
        // (the tables' rows must be 16-byte aligned for the tiled kernels: ny even; their point tiles must not straddle a column)
        if (a.A <= 8 && a.ny % 4 == 0 && a.G % 4 == 0)
            batch_posterior_tiled_kernel<8, 4><<<dim3((unsigned)((a.G / 4 + BT_THREADS - 1) / BT_THREADS), (unsigned)a.runs), BT_THREADS, 0, st>>>(a);
        else if (a.ny % 2 == 0 && a.G % 2 == 0)
            batch_posterior_tiled_kernel<BT_MAXA, 2><<<dim3((unsigned)((a.G / 2 + BT_THREADS - 1) / BT_THREADS), (unsigned)a.runs), BT_THREADS, 0, st>>>(a);
        else
            batch_posterior_kernel<<<dim3((unsigned)((a.G + BT_THREADS - 1) / BT_THREADS), (unsigned)a.runs), BT_THREADS, 0, st>>>(a);
        MFGP_LAUNCH_CHECK();
    }
    const size_t msmem = sizeof(unsigned short) * 2 * (size_t)a.G;
    if (msmem > 160 * 1024) return MFGP_ERR_INVALID;
    MFGP_CUDA_CHECK(cudaFuncSetAttribute(batch_coverage_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msmem));
    batch_coverage_kernel<<<a.runs, BT_THREADS, msmem, st>>>(a, (int)iteration);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}


static bool choi_valid(const mfgp_batch* b, const mfgp_params* p_host) {
    return batch_valid(b, p_host) && b->algo == 3 && b->q && b->picks && b->nplan && b->plan_state && b->pmask && b->ccount &&
           b->cties;
}

int mfgp_batch_choi_begin(const mfgp_batch* b, const mfgp_params* p_host, void* stream) {
    if (!choi_valid(b, p_host)) return MFGP_ERR_INVALID;
    const BatchArgs a = batch_args(b, p_host);
    batch_choi_q_kernel<<<dim3((unsigned)((a.G + BT_THREADS - 1) / BT_THREADS), (unsigned)a.runs), BT_THREADS, 0,
                          static_cast<cudaStream_t>(stream)>>>(a);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

int mfgp_batch_choi_plan(const mfgp_batch* b, const mfgp_params* p_host, double threshold, int64_t rounds, void* stream) {
    if (!choi_valid(b, p_host) || rounds < 0) return MFGP_ERR_INVALID;
    const BatchArgs a = batch_args(b, p_host);
    const size_t smem = sizeof(double) * 3 * (size_t)a.cap;
    if (smem > 200 * 1024) return MFGP_ERR_INVALID;
    MFGP_CUDA_CHECK(cudaFuncSetAttribute(batch_choi_pick_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    for (int64_t i = 0; i < rounds; i++) {
        batch_choi_pick_kernel<<<a.runs, BT_THREADS, smem, static_cast<cudaStream_t>(stream)>>>(a, threshold);
        MFGP_LAUNCH_CHECK();
    }
    return MFGP_OK;
}

int mfgp_batch_choi_cluster(const mfgp_batch* b, void* stream) {
    mfgp_params dummy{};
    if (!b || !choi_valid(b, &dummy)) return MFGP_ERR_INVALID;
    const BatchArgs a = batch_args(b, &dummy);
    batch_choi_cluster_kernel<<<a.runs, BT_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(a);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

int mfgp_batch_choi_tours(const mfgp_batch* b, int64_t n_total, int64_t n_max, double* pts, int64_t* gidx, int32_t* ord,
                          void* work, int64_t work_bytes, void* stream) {
    mfgp_params dummy{};
    if (!b || !choi_valid(b, &dummy) || n_total < 0 || n_max < 0 || n_max > n_total) return MFGP_ERR_INVALID;
    if (n_total > 0 && (!pts || !gidx || !ord || !b->tour)) return MFGP_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const BatchArgs a = batch_args(b, &dummy);
    const int nrc = a.runs * a.A;
    batch_choi_gather_kernel<<<(nrc + 127) / 128, 128, 0, st>>>(a, pts, reinterpret_cast<long long*>(gidx));
    MFGP_LAUNCH_CHECK();
    if (n_total == 0) return MFGP_OK;
    const int rc = choi_tsp_tours(pts, b->tour_off, nrc, n_total, n_max, ord, nullptr, work, work_bytes, stream);
    if (rc != MFGP_OK) return rc;
    batch_choi_order_kernel<<<(nrc + 127) / 128, 128, 0, st>>>(a, reinterpret_cast<const long long*>(gidx), ord);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

}  // extern "C"
