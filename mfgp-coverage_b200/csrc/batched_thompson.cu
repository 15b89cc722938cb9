// Batched Thompson sampling (stepper algo 4): the draw stage of simulator.thompson for every run of a batch, after the
// iteration's mfgp_batch_step (samples appended, posterior updated, both partitions seeded by the positions, log row).
//
// Per run r and draw s = agent i, the pathwise posterior draw of mfgp_grid_sample_coef (gp_sample_grid.cu),
//
//   F_s(g) = mu(g) + f_s(g) - k(g, X) beta_s,   beta_s = W^T W (f_s(X) + sqrt(noise_n + jitter) eta_s),
//
// f_s the prior draw whose Chebyshev coefficients on the plan's box are sqrt(s_P) Qx_P Xi_P Qy_P^T per kernel part (AR1:
// C_prior = rho C_L + C_H, lofi rows see C_L).  Agent i needs only sum_{g in cell i} F_i(g) {1, x, y}: each grid point is
// evaluated for the draw of its own cell, never for all S draws, and nothing per grid point is written out.
//   bt_prior_kernel  (run, draw) per CTA: normals Xi from the counter-based generator, coefficients C_prior / C_L in shared
//                    memory, Hc[ix][l] = sum_k T_k(tx_ix) C_prior[l][k] for every grid column, and the right-hand side
//                    f_s(X_n) + sd_n eta[n][s] (grid rows read the prior from Hc, the off-grid prior rows expand it in full)
//   bt_beta_kernel   run per CTA: u = W rhs, beta = W^T u over the lower triangle of the run's W, the A right-hand sides
//                    sharing every load of W (the loop structure of batch_append_kernel)
//   bt_cell_kernel   run per CTA: F of every grid point for the draw of each cell it belongs to (mu from the stepper's mean,
//                    the prior from Hc, k(g, X_n) from the exact axis tables), per-thread cell sums in a fixed order, fixed
//                    butterflies, cov_finish's arithmetic (NaN for an empty cell), snap_to_grid in agent order, the move.
// No floating-point atomics: a run's results do not depend on the batch it is in.
//
// Normals: Philox4x32-10 (Salmon et al., SC'11) keyed by the run's 64-bit seed, counter (row, agent, iteration, 0); the
// first 64 output bits give u1 in (0, 1], the last 64 u2 in [0, 1), and the normal is sqrt(-2 ln u1) cos(2 pi u2).  Rows
// follow mfgp_grid_sample_coef's layout: lofi block Xi_L[i][j] at row i * ryL + j, hifi block after it, then one noise row
// per training point.
#include <cmath>

#include "batched.cuh"

namespace mfgp {

struct ThompsonArgs {
    BatchArgs a;
    int it;
    int rx[2], ry[2];                      // per kernel part (0 lofi, 1 hifi)
    const double* Qx[2]; const double* Qy[2];
    double sq[2];                          // sqrt(s_P)
    int first;                             // 0: both parts (multi-fidelity), 1: hifi only
    int rxm, rym, kpad, R, d0;             // merged orders, C row pitch, ry * kpad, prior rows of the normals
    double bxlo, bxhi, bylo, byhi;
    double sdL, sdH;                       // sqrt(noise + jitter) of lofi / hifi rows
    double* Hc;                            // [runs][A][nx][rym]
    double* rhs;                           // [runs][A][cap]
    double* beta;                          // [runs][A][cap]
};

__device__ __forceinline__ double bt_normal(unsigned long long seed, int it, int row, int agent) {
    unsigned c0 = (unsigned)row, c1 = (unsigned)agent, c2 = (unsigned)it, c3 = 0u;
    unsigned k0 = (unsigned)seed, k1 = (unsigned)(seed >> 32);
#pragma unroll
    for (int i = 0; i < 10; i++) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    const unsigned long long a53 = ((((unsigned long long)c0) << 32) | c1) >> 11;
    const unsigned long long b53 = ((((unsigned long long)c2) << 32) | c3) >> 11;
    const double u1 = (double)(a53 + 1ull) * 0x1p-53, u2 = (double)b53 * 0x1p-53;
    return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
}

// sum_l T_l(t) h[l], l < r, by the Chebyshev recurrence (the basis of cheb_basis_kernel)
__device__ __forceinline__ double cheb_dot(double t, const double* __restrict__ h, int r) {
    double f = 0.0, t0 = 1.0, t1 = t;
    for (int l = 0; l < r; l++) {
        f = fma(t0, h[l], f);
        const double t2 = 2.0 * t * t1 - t0;
        t0 = t1; t1 = t2;
    }
    return f;
}

__global__ void __launch_bounds__(BT_THREADS) bt_prior_kernel(ThompsonArgs t) {
    extern __shared__ __align__(16) double tsm[];
    const BatchArgs& a = t.a;
    const int s = blockIdx.x, r = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = BT_THREADS / 32;
    if (a.status[r] != 0) return;
    const int P_ = t.rym + 1;
    double* X = tsm;                       // Xi[i][j]
    double* T = X + t.rxm * P_;            // (Qx Xi)[k][j]
    double* Cp = T + t.rxm * P_;           // C_prior[l * kpad + k]
    double* CL = Cp + t.R;                 // C_L
    const unsigned long long seed = (unsigned long long)a.seed[r];
    for (int e = tid; e < t.R; e += BT_THREADS) { Cp[e] = 0.0; CL[e] = 0.0; }
    for (int P = t.first; P < 2; P++) {    // prior_coef_kernel's products
        const int rx = t.rx[P], ry = t.ry[P], off = P ? t.rx[0] * t.ry[0] : 0;
        const double* Qx = t.Qx[P];
        const double* Qy = t.Qy[P];
        __syncthreads();
        for (int e = tid; e < rx * ry; e += BT_THREADS) X[(e / ry) * P_ + e % ry] = bt_normal(seed, t.it, off + e, s);
        __syncthreads();
        for (int e = tid; e < rx * ry; e += BT_THREADS) {
            const int k = e / ry, j = e % ry;
            double v = 0.0;
            for (int i = 0; i < rx; i++) v = fma(Qx[k * rx + i], X[i * P_ + j], v);
            T[k * P_ + j] = v;
        }
        __syncthreads();
        for (int e = tid; e < rx * ry; e += BT_THREADS) {
            const int l = e / rx, k = e % rx;
            double c = 0.0;
            for (int j = 0; j < ry; j++) c = fma(T[k * P_ + j], Qy[l * ry + j], c);
            c *= t.sq[P];
            const int o = l * t.kpad + k;
            if (P == 0) { CL[o] = c; Cp[o] = a.p.rho * c; }
            else Cp[o] += c;
        }
    }
    __syncthreads();
    const double xs = t.bxlo + t.bxhi, xd = t.bxhi - t.bxlo, ys = t.bylo + t.byhi, yd = t.byhi - t.bylo;
    double* Hc = t.Hc + ((int64_t)r * a.A + s) * a.nx * t.rym;
    for (int e = tid; e < a.nx * t.rym; e += BT_THREADS) {
        const int ix = e / t.rym, l = e % t.rym;
        Hc[e] = cheb_dot((2.0 * a.ux[ix] - xs) / xd, Cp + l * t.kpad, t.rxm);
    }
    __syncthreads();                       // Hc (global) is read back by this CTA below
    const int N = a.Ncur[r];
    const int* rowidx = a.rowidx + (int64_t)r * a.cap;
    const double* Xt = a.Xt + (int64_t)r * a.cap * 2;
    double* rhs = t.rhs + ((int64_t)r * a.A + s) * a.cap;
    for (int n = warp; n < N; n += nwarp) {          // off-grid rows (the prior points): a warp per row, lanes over l
        if (rowidx[n] >= 0) continue;
        const double tx = (2.0 * Xt[2 * n] - xs) / xd, ty = (2.0 * Xt[2 * n + 1] - ys) / yd;
        const double* C = n < a.NL ? CL : Cp;
        double f = 0.0;
        for (int l = lane; l < t.rym; l += 32) {
            double u0 = 1.0, u1 = ty;
            for (int j = 0; j < l; j++) {
                const double u2 = 2.0 * ty * u1 - u0;
                u0 = u1; u1 = u2;
            }
            f = fma(u0, cheb_dot(tx, C + l * t.kpad, t.rxm), f);
        }
        f = warp_sum_d(f);
        if (lane == 0) rhs[n] = f + (n < a.NL ? t.sdL : t.sdH) * bt_normal(seed, t.it, t.d0 + n, s);
    }
    for (int n = tid; n < N; n += BT_THREADS) {      // grid rows: the prior from the grid evaluation
        const int g = rowidx[n];
        if (g < 0) continue;
        const double ty = (2.0 * a.uy[g % a.ny] - ys) / yd;
        const double f = cheb_dot(ty, Hc + (int64_t)(g / a.ny) * t.rym, t.rym);
        rhs[n] = f + (n < a.NL ? t.sdL : t.sdH) * bt_normal(seed, t.it, t.d0 + n, s);
    }
}

__global__ void __launch_bounds__(BT_THREADS) bt_beta_kernel(ThompsonArgs t) {
    extern __shared__ __align__(16) double bsm[];
    const BatchArgs& a = t.a;
    const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = BT_THREADS / 32;
    if (a.status[r] != 0) return;
    const int N = a.Ncur[r], cap = a.cap, A = a.A;
    double* v = bsm;                       // [A][cap] right-hand sides
    double* u = bsm + (int64_t)A * cap;    // [A][cap] W v
    for (int e = tid; e < A * N; e += BT_THREADS) {
        const int j = e / N, n = e % N;
        v[j * cap + n] = t.rhs[((int64_t)r * A + j) * cap + n];
    }
    __syncthreads();
    const double* W = a.W + (int64_t)r * cap * cap;
    for (int n = warp; n < N; n += nwarp) {          // u[j][n] = sum_{m <= n} W[n][m] v[j][m]: a warp per row
        double acc[BT_MAXA];
#pragma unroll
        for (int j = 0; j < BT_MAXA; j++) acc[j] = 0.0;
        const double* wr = W + (int64_t)n * cap;
#pragma unroll 4
        for (int m = lane; m <= n; m += 32) {
            const double w = wr[m];
#pragma unroll
            for (int j = 0; j < BT_MAXA; j++)
                if (j < A) acc[j] = fma(w, v[j * cap + m], acc[j]);
        }
#pragma unroll
        for (int j = 0; j < BT_MAXA; j++)
            if (j < A) {
                const double sum = warp_sum_d(acc[j]);
                if (lane == 0) u[j * cap + n] = sum;
            }
    }
    __syncthreads();
    // beta[j][m] = sum_{n >= m} W[n][m] u[j][n]: a thread per column, the warp's rows from its first column on (coalesced);
    // entries above the diagonal are never read (W's upper part is not written)
    for (int m = tid; m < N; m += BT_THREADS) {
        double b[BT_MAXA];
#pragma unroll
        for (int j = 0; j < BT_MAXA; j++) b[j] = 0.0;
#pragma unroll 4
        for (int n = m & ~31; n < N; n++) {
            const double w = n >= m ? W[(int64_t)n * cap + m] : 0.0;
#pragma unroll
            for (int j = 0; j < BT_MAXA; j++)
                if (j < A) b[j] = fma(w, u[j * cap + n], b[j]);
        }
#pragma unroll
        for (int j = 0; j < BT_MAXA; j++)
            if (j < A) t.beta[((int64_t)r * A + j) * cap + m] = b[j];
    }
}

// np.argmin(np.abs(u - v)): the first index of the smallest distance
__device__ __forceinline__ int nearest_index(const double* __restrict__ u, int n, double v) {
    int best = 0;
    double d = fabs(u[0] - v);
    for (int i = 1; i < n; i++) {
        const double e = fabs(u[i] - v);
        if (e < d) { d = e; best = i; }
    }
    return best;
}

__global__ void __launch_bounds__(BT_THREADS) bt_cell_kernel(ThompsonArgs t) {
    extern __shared__ __align__(16) double csm2[];    // beta [A][N]
    __shared__ double s_red[BT_THREADS / 32][BT_MAXA][3];
    __shared__ double s_tgt[BT_MAXA][2];
    __shared__ int s_g[BT_MAXA][4];                     // target (ix, iy) or -1, fallback (ix, iy)
    __shared__ int s_fin[BT_MAXA][2];
    const BatchArgs& a = t.a;
    const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (a.status[r] != 0) return;
    const int N = a.Ncur[r], A = a.A, cap = a.cap;
    for (int e = tid; e < A * N; e += BT_THREADS) {
        const int j = e / N, n = e % N;
        csm2[j * N + n] = t.beta[((int64_t)r * A + j) * cap + n];
    }
    __syncthreads();
    double s0[BT_MAXA], s1[BT_MAXA], s2[BT_MAXA];
#pragma unroll
    for (int j = 0; j < BT_MAXA; j++) s0[j] = s1[j] = s2[j] = 0.0;
    const double ys = t.bylo + t.byhi, yd = t.byhi - t.bylo;
    const unsigned short* cm = a.cmask + (int64_t)r * a.G;
    const double* mu = a.mu + (int64_t)r * a.G;
    const double* Hc = t.Hc + (int64_t)r * A * a.nx * t.rym;
    for (int g = tid; g < a.G; g += BT_THREADS) {
        unsigned m = cm[g];
        if (!m) continue;
        const int ix = g / a.ny, iy = g % a.ny;
        const double x = a.xy[2 * g], y = a.xy[2 * g + 1], base = mu[g], ty = (2.0 * a.uy[iy] - ys) / yd;
        while (m) {                                    // the cells of the point: one, or several on a bisector
            const int c = __ffs(m) - 1;
            m &= m - 1;
            const double f = cheb_dot(ty, Hc + ((int64_t)c * a.nx + ix) * t.rym, t.rym);
            const double* bc = csm2 + c * N;
            double kb = 0.0;
#pragma unroll 4
            for (int n = 0; n < N; n++) kb = fma(bt_psi(a, r, n, ix, iy), bc[n], kb);
            const double F = (base + f) - kb;
#pragma unroll
            for (int j = 0; j < BT_MAXA; j++)
                if (j == c) { s0[j] += F; s1[j] = fma(F, x, s1[j]); s2[j] = fma(F, y, s2[j]); }
        }
    }
#pragma unroll
    for (int j = 0; j < BT_MAXA; j++)
        if (j < A) {
            const double v0 = warp_sum_d(s0[j]), v1 = warp_sum_d(s1[j]), v2 = warp_sum_d(s2[j]);
            if (lane == 0) { s_red[warp][j][0] = v0; s_red[warp][j][1] = v1; s_red[warp][j][2] = v2; }
        }
    __syncthreads();
    double* pos = a.pos + (int64_t)r * A * 2;
    if (tid < A) {          // cov_finish's arithmetic, then the two candidate grid points of snap_to_grid
        const int i = tid;
        double m0 = 0.0, m1 = 0.0, m2 = 0.0;
        for (int w = 0; w < BT_THREADS / 32; w++) { m0 += s_red[w][i][0]; m1 += s_red[w][i][1]; m2 += s_red[w][i][2]; }
        const double n = a.ccell[((int64_t)r * A + i) * 2], area = a.ccell[((int64_t)r * A + i) * 2 + 1];
        const double f_int = __dmul_rn(__ddiv_rn(m0, n), area);
        double cx = __ddiv_rn(__dmul_rn(__ddiv_rn(m1, n), area), f_int);
        double cy = __ddiv_rn(__dmul_rn(__ddiv_rn(m2, n), area), f_int);
        if (cx < a.xmin) cx = a.xmin;
        if (cx > a.xmax) cx = a.xmax;
        if (cy < a.ymin) cy = a.ymin;
        if (cy > a.ymax) cy = a.ymax;
        s_tgt[i][0] = cx; s_tgt[i][1] = cy;
        const bool ok = isfinite(cx) && isfinite(cy);
        s_g[i][0] = ok ? nearest_index(a.ux, a.nx, cx) : -1;
        s_g[i][1] = ok ? nearest_index(a.uy, a.ny, cy) : -1;
        s_g[i][2] = nearest_index(a.ux, a.nx, pos[2 * i]);
        s_g[i][3] = nearest_index(a.uy, a.ny, pos[2 * i + 1]);
    }
    __syncthreads();
    if (tid == 0) {          // in agent order: a target taken by a lower-index agent (or NaN) falls back to the position's point
        for (int i = 0; i < A; i++) {
            int gx = s_g[i][0], gy = s_g[i][1];
            bool take = gx >= 0;
            for (int k = 0; k < i && take; k++)
                if (s_fin[k][0] == gx && s_fin[k][1] == gy) take = false;
            if (!take) { gx = s_g[i][2]; gy = s_g[i][3]; }
            s_fin[i][0] = gx; s_fin[i][1] = gy;
        }
    }
    __syncthreads();
    if (tid < A) {
        const int i = tid;
        const long long gi = (long long)s_fin[i][0] * a.ny + s_fin[i][1];
        double* prev = a.prev + (int64_t)r * A * 2;
        double* cen = a.cen + (int64_t)r * A * 2;
        prev[2 * i] = pos[2 * i]; prev[2 * i + 1] = pos[2 * i + 1];
        pos[2 * i] = a.xy[2 * gi]; pos[2 * i + 1] = a.xy[2 * gi + 1];
        a.pos_idx[r * A + i] = gi;
        cen[2 * i] = s_tgt[i][0]; cen[2 * i + 1] = s_tgt[i][1];
        double* row = a.log_agent + (((int64_t)r * a.iterations + t.it) * A + i) * BT_LOGC;
        row[6] = s_tgt[i][0]; row[7] = s_tgt[i][1];
    }
}

__global__ void bt_normals_kernel(const long long* __restrict__ seed, int A, int it, int rows, double* __restrict__ out) {
    const int r = blockIdx.y;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (int64_t)rows * A) return;
    out[(int64_t)r * rows * A + e] = bt_normal((unsigned long long)seed[r], it, (int)(e / A), (int)(e % A));
}

inline int64_t ts_rup(int64_t v, int64_t m) { return (v + m - 1) / m * m; }

static bool thompson_valid(const mfgp_batch* b, const mfgp_params* p) {
    if (!batch_valid(b, p) || b->algo != 4 || b->runs > 65535 || !b->ux || !b->uy || !b->QxH || !b->QyH) return false;
    if (b->rxH < 1 || b->ryH < 1 || b->rxH > 64 || b->ryH > 64) return false;
    if (p->multi ? (b->rxL < 1 || b->ryL < 1 || b->rxL > 64 || b->ryL > 64 || !b->QxL || !b->QyL) : (b->rxL || b->ryL || b->NL))
        return false;
    return b->bxhi > b->bxlo && b->byhi > b->bylo && std::isfinite(b->bxhi - b->bxlo) && std::isfinite(b->byhi - b->bylo);
}

static int64_t thompson_work_doubles(const mfgp_batch* b) {
    const int64_t rym = b->ryL > b->ryH ? b->ryL : b->ryH;
    return ts_rup(b->runs * b->A * b->nx * rym, 2) + 2 * ts_rup(b->runs * b->A * b->cap, 2);
}

}  // namespace mfgp

using namespace mfgp;

extern "C" int64_t mfgp_batch_thompson_workspace_bytes(const mfgp_batch* b) {
    if (!b || b->runs <= 0 || b->A <= 0 || b->nx <= 0 || b->cap <= 0 || b->ryH < 0 || b->ryL < 0) return 0;
    return thompson_work_doubles(b) * 8 + 256;
}

extern "C" int mfgp_batch_thompson(const mfgp_batch* b, const mfgp_params* p_host, int64_t iteration, void* work,
                                   int64_t work_bytes, void* stream) {
    if (!b || !p_host || !thompson_valid(b, p_host) || iteration < 0 || iteration >= b->iterations) return MFGP_ERR_INVALID;
    if (!work || (reinterpret_cast<uintptr_t>(work) & 15) || work_bytes < thompson_work_doubles(b) * 8) return MFGP_ERR_INVALID;
    const int64_t beta_smem = 8 * 2 * b->A * b->cap;
    if (beta_smem > 200 * 1024) return MFGP_ERR_INVALID;      // the sample append's staging limit (mfgp_batch_step)
    ThompsonArgs t{};
    t.a = batch_args(b, p_host);
    const bool multi = p_host->multi != 0;
    t.it = (int)iteration;
    t.rx[0] = (int)b->rxL; t.ry[0] = (int)b->ryL; t.rx[1] = (int)b->rxH; t.ry[1] = (int)b->ryH;
    t.Qx[0] = b->QxL; t.Qy[0] = b->QyL; t.Qx[1] = b->QxH; t.Qy[1] = b->QyH;
    t.sq[0] = multi ? std::sqrt(p_host->s_L) : 0.0; t.sq[1] = std::sqrt(p_host->s_H);
    t.first = multi ? 0 : 1;
    t.rxm = t.rx[0] > t.rx[1] ? t.rx[0] : t.rx[1];
    t.rym = t.ry[0] > t.ry[1] ? t.ry[0] : t.ry[1];
    t.kpad = (int)ts_rup(t.rxm, 4);
    t.R = t.rym * t.kpad;
    t.d0 = t.rx[0] * t.ry[0] + t.rx[1] * t.ry[1];
    t.bxlo = b->bxlo; t.bxhi = b->bxhi; t.bylo = b->bylo; t.byhi = b->byhi;
    t.sdL = std::sqrt(t.a.p.noise_L + t.a.p.jitter); t.sdH = std::sqrt(t.a.p.noise_H + t.a.p.jitter);
    double* wp = static_cast<double*>(work);
    t.Hc = wp;
    t.rhs = t.Hc + ts_rup(b->runs * b->A * b->nx * t.rym, 2);
    t.beta = t.rhs + ts_rup(b->runs * b->A * b->cap, 2);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int prior_smem = (int)(8 * (2 * t.rxm * (t.rym + 1) + 2 * t.R));
    MFGP_CUDA_CHECK(cudaFuncSetAttribute(bt_prior_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, prior_smem));
    bt_prior_kernel<<<dim3((unsigned)b->A, (unsigned)b->runs), BT_THREADS, prior_smem, st>>>(t);
    MFGP_LAUNCH_CHECK();
    MFGP_CUDA_CHECK(cudaFuncSetAttribute(bt_beta_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)beta_smem));
    bt_beta_kernel<<<(unsigned)b->runs, BT_THREADS, (size_t)beta_smem, st>>>(t);
    MFGP_LAUNCH_CHECK();
    const int cell_smem = (int)(beta_smem / 2);
    MFGP_CUDA_CHECK(cudaFuncSetAttribute(bt_cell_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, cell_smem));
    bt_cell_kernel<<<(unsigned)b->runs, BT_THREADS, (size_t)cell_smem, st>>>(t);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

extern "C" int mfgp_batch_thompson_normals(const mfgp_batch* b, int64_t iteration, int64_t rows, double* out, void* stream) {
    if (!b || b->algo != 4 || !b->seed || !out || b->runs <= 0 || b->runs > 65535 || b->A <= 0 || b->A > BT_MAXA ||
        iteration < 0 || iteration >= b->iterations || rows <= 0 || rows * b->A >= (1LL << 31))
        return MFGP_ERR_INVALID;
    const int64_t n = rows * b->A;
    bt_normals_kernel<<<dim3((unsigned)((n + 255) / 256), (unsigned)b->runs), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const long long*>(b->seed), (int)b->A, (int)iteration, (int)rows, out);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}
