// Joint posterior draws over whole tensor-product grids by pathwise conditioning (Matheron's rule):
//
//   f_post(.) = mean_H + f(.) + k(., X) K^-1 (y - m - f(X) - eps),     f a prior draw, eps ~ N(0, diag(noise + jitter))
//
// is an exact draw from the posterior of the latent f_H.  No posterior covariance is formed or factored.
//
// Prior draw: per kernel part P (lofi, hifi), g_P ~ N(0, K_P,x (x) K_P,y) at the r_x x r_y tensor of Chebyshev nodes of a box
// that covers the grid and the training points, interpolated.  In coefficient space C_P = sqrt(s_P) Qx_P Xi_P Qy_P^T with
// Q = DCT K_nodes^(1/2) (host, r <= 64) and Xi_P a block of the caller's standard normals.  AR1: f_L = g_L, f_H = rho f_L + g_H;
// lofi training rows see f_L, hifi rows and the grid see f_H.
//
// mfgp_grid_sample_coef: one coefficient matrix per draw, ry x kpad in the merged basis T_l(ty) T_k(tx) of gp_factored.cu,
//   prior_coef_kernel    C_L,s and C_prior,s = rho C_L,s + C_H,s                          (~r^3 per draw)
//   train_basis_kernel   Phi[n][(l, k)] = T_l(ty_n) T_k(tx_n)
//   gemm_f64 x 2         f_s(X_n) = Phi C_s^T  (C_L for lofi rows, C_prior for hifi rows)
//   residual_kernel      R[n][s] = y_n - m_n - f_s(X_n) - sqrt(noise_n + jitter) eta[n][s]
//   gemm_f64 x 2         alpha = W^T (W R)     (W = L^-1 of the standing fit, lower triangular)
//   gemm_f64             D = B^T alpha         (B: build_B_merged_kernel, the cross-covariance's coefficients on the box)
//   combine_kernel       C_s = C_prior,s + D_s
// mfgp_grid_sample_eval: F[g][s] = mean_H + sum_l Uy[iy][l] sum_k Ux[ix][k] C_s[l][k] for whole columns,
//   gemm_f64             Hc[ix][s][l] = sum_k Ux[ix][k] C_s[l][k]
//   grid_sample_eval_kernel  F tile (64 iy x 64 draws) = Uy tile Hc[ix]^T on DMMA, mean added, 16-byte stores.
// Every sum runs in a fixed order: the same inputs give the same bits, and a column slice gives the same bits as the whole grid.
#include <cmath>

#include "cheb.cuh"
#include "common.cuh"
#include "gemm_f64.cuh"

namespace mfgp {

constexpr int SG_RP = 64;                  // padding of the coefficient count R = ry * kpad (rows of D, columns of B / Phi)

// ---- prior coefficients: one CTA per draw ------------------------------------------------------------------------------------
struct PriorArgs {
    const double* E; int64_t lde; int S;
    const double* Qx[2]; const double* Qy[2];
    int rx[2], ry[2], off[2];              // per part (0 = lofi, 1 = hifi): orders and first row of its normals in E
    double sq[2];                          // sqrt(s_P)
    int first;                             // 0: both parts (multi-fidelity), 1: hifi only
    int kpad, R;
    double rho;
    double* CL;                            // [S][R] sqrt(s_L) Qx_L Xi_L Qy_L^T (lofi training rows), or null
    double* Cp;                            // [S][R] rho C_L + C_H
};
constexpr int PC_P = F_MAXR + 1;
constexpr int PC_SMEM = (2 * F_MAXR * PC_P + F_MAXR * F_MAXR) * 8;

__global__ void __launch_bounds__(256) prior_coef_kernel(PriorArgs a) {
    extern __shared__ double sm[];
    double* X = sm;                        // Xi[i][j]
    double* T = sm + F_MAXR * PC_P;        // (Qx Xi)[k][j]
    double* acc = sm + 2 * F_MAXR * PC_P;  // C_prior[l * kpad + k]
    const int s = blockIdx.x, tid = threadIdx.x;
    for (int e = tid; e < a.R; e += 256) acc[e] = 0.0;
    for (int P = a.first; P < 2; P++) {
        const int rx = a.rx[P], ry = a.ry[P];
        const double* Qx = a.Qx[P];
        const double* Qy = a.Qy[P];
        __syncthreads();
        for (int e = tid; e < rx * ry; e += 256) X[(e / ry) * PC_P + e % ry] = a.E[(int64_t)(a.off[P] + e) * a.lde + s];
        __syncthreads();
        for (int e = tid; e < rx * ry; e += 256) {
            const int k = e / ry, j = e % ry;
            double t = 0.0;
            for (int i = 0; i < rx; i++) t = fma(Qx[k * rx + i], X[i * PC_P + j], t);
            T[k * PC_P + j] = t;
        }
        __syncthreads();
        for (int e = tid; e < rx * ry; e += 256) {
            const int l = e / rx, k = e % rx;
            double c = 0.0;
            for (int j = 0; j < ry; j++) c = fma(T[k * PC_P + j], Qy[l * ry + j], c);
            c *= a.sq[P];
            const int o = l * a.kpad + k;
            if (P == 0) {
                a.CL[(int64_t)s * a.R + o] = c;
                acc[o] = a.rho * c;
            } else {
                acc[o] += c;
            }
        }
    }
    __syncthreads();
    for (int e = tid; e < a.R; e += 256) a.Cp[(int64_t)s * a.R + e] = acc[e];
}

// ---- Phi[n][l * kpad + k] = T_l(ty_n) T_k(tx_n) of the training points (zero for k >= rx, n >= N and columns >= R) -------------
__global__ void __launch_bounds__(256) train_basis_kernel(const double* __restrict__ Xt, int N, double xlo, double xhi, double ylo,
                                                          double yhi, int rx, int ry, int kpad, int ldp, double* __restrict__ Phi) {
    __shared__ double tb[2][F_MAXR];
    const int n = blockIdx.x;
    if (threadIdx.x < 2 && n < N) {        // the recurrence of cheb_basis_kernel
        const int ax = threadIdx.x;
        const double lo = ax ? ylo : xlo, hi = ax ? yhi : xhi;
        const int r = ax ? ry : rx;
        const double t = (2.0 * Xt[2 * n + ax] - (lo + hi)) / (hi - lo);
        double t0 = 1.0, t1 = t;
        for (int k = 0; k < r; k++) {
            tb[ax][k] = t0;
            const double t2 = 2.0 * t * t1 - t0;
            t0 = t1; t1 = t2;
        }
    }
    __syncthreads();
    for (int e = threadIdx.x; e < ldp; e += blockDim.x) {
        const int l = e / kpad, k = e % kpad;
        Phi[(int64_t)n * ldp + e] = (n < N && l < ry && k < rx) ? tb[1][l] * tb[0][k] : 0.0;
    }
}

// R[n][s] = y_n - m_n - f_s(X_n) - sd_n eta[n][s]  (zero in the padding rows / columns)
__global__ void residual_kernel(const double* __restrict__ y, const double* __restrict__ PL, const double* __restrict__ PH, int ldp,
                                const double* __restrict__ E, int64_t lde, int64_t row0, int N, int NL, int npad, int S, double mean_L,
                                double mean_H, double sd_L, double sd_H, double* __restrict__ R) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)npad * ldp) return;
    const int n = (int)(idx / ldp), s = (int)(idx % ldp);
    double v = 0.0;
    if (n < N && s < S) {
        const bool lo = n < NL;
        const double f = (lo ? PL : PH)[idx];
        v = y[n] - (lo ? mean_L : mean_H) - f - (lo ? sd_L : sd_H) * E[(row0 + n) * lde + s];
    }
    R[idx] = v;
}

// C[s][e] = Cp[s][e] + D[e][s]
__global__ void combine_kernel(const double* __restrict__ Cp, const double* __restrict__ D, int ldd, int R, int S,
                               double* __restrict__ C) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)S * R) return;
    const int s = (int)(idx / R), e = (int)(idx % R);
    C[idx] = Cp[idx] + (D ? D[(int64_t)e * ldd + s] : 0.0);
}

// ---- evaluation ------------------------------------------------------------------------------------------------------------
// One CTA per (grid column ix, tile of 64 draws, EV_TILES tiles of 64 rows iy), 4 warps 2 x 2, each 32 rows x 32 draws of F in
// registers (4 x 4 DMMA.8x8x4 tiles).  Hc[ix]'s 64 x ry slab is staged once; the Uy tiles stream through a cp.async double
// buffer.  Shared rows have a pitch P = 4 mod 16 doubles and ry <= P: the fragment loads of a half-warp (4 rows x 4 columns)
// hit 16 distinct bank pairs.  Lane (gq, tq) stores the pair of draws (2 tq, 2 tq + 1) of its row as one 16-byte store; the
// four lanes of a row write 64 contiguous bytes.
constexpr int EV_BM = 64, EV_BN = 64, EV_TILES = 4, EV_THREADS = 128;

struct EvalArgs {
    const double* Uy;                      // [ny][ry]
    const double* Hc; int64_t ldh;         // [ncols][S * ry]: Hc[ix][s * ry + l]
    double* F; int64_t ldf;
    int ny, S, ry, pitch, ytiles;
    double mean;
};

__global__ void __launch_bounds__(EV_THREADS) grid_sample_eval_kernel(EvalArgs a) {
    extern __shared__ __align__(16) double esm[];
    const int P = a.pitch;
    double* Bs = esm;                      // [64 draws][P]
    double* As = esm + EV_BN * P;          // [2][64 rows][P]
    const int ix = blockIdx.x, s0 = blockIdx.y * EV_BN;
    const int t0 = blockIdx.z * EV_TILES, t1 = min(t0 + EV_TILES, a.ytiles);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int gq = lane >> 2, tq = lane & 3;
    const int wm = (warp >> 1) * 32, wn = (warp & 1) * 32;
    const int ch = a.ry / 2;               // 16-byte chunks per row
    const double* hc = a.Hc + (int64_t)ix * a.ldh;
    for (int c = tid; c < EV_BN * ch; c += EV_THREADS) {
        const int r = c / ch, q = c % ch;
        const bool ok = s0 + r < a.S;
        cp_async16(Bs + r * P + 2 * q, hc + (ok ? (int64_t)(s0 + r) * a.ry + 2 * q : 0), ok);
    }
    auto stage = [&](int buf, int t) {
        double* dst = As + buf * EV_BM * P;
        for (int c = tid; c < EV_BM * ch; c += EV_THREADS) {
            const int r = c / ch, q = c % ch, iy = t * EV_BM + r;
            const bool ok = iy < a.ny;
            cp_async16(dst + r * P + 2 * q, a.Uy + (ok ? (int64_t)iy * a.ry + 2 * q : 0), ok);
        }
        cp_async_commit();
    };
    stage(0, t0);
    for (int t = t0; t < t1; t++) {
        const int buf = (t - t0) & 1;
        if (t + 1 < t1) {
            stage(buf ^ 1, t + 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        double acc[4][4][2];
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
            for (int j = 0; j < 4; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
        const double* sa = As + buf * EV_BM * P + (wm + gq) * P + tq;
        const double* sb = Bs + (wn + gq) * P + tq;
        for (int kk = 0; kk < a.ry; kk += 4) {
            double af[4], bf[4];
#pragma unroll
            for (int i = 0; i < 4; i++) af[i] = sa[i * 8 * P + kk];
#pragma unroll
            for (int j = 0; j < 4; j++) bf[j] = sb[j * 8 * P + kk];
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
        }
        __syncthreads();                   // the next iteration's stage overwrites this buffer
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int iy = t * EV_BM + wm + 8 * i + gq;
            if (iy >= a.ny) continue;
            double* row = a.F + ((int64_t)ix * a.ny + iy) * a.ldf;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int s = s0 + wn + 8 * j + 2 * tq;
                if (s + 1 < a.S)
                    *reinterpret_cast<double2*>(row + s) = make_double2(a.mean + acc[i][j][0], a.mean + acc[i][j][1]);
                else if (s < a.S)
                    row[s] = a.mean + acc[i][j][0];
            }
        }
    }
}

inline int64_t rup(int64_t v, int64_t m) { return (v + m - 1) / m * m; }
inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

struct CoefLayout {
    int64_t N, npad, rx, ry, kpad, R, Rp, Sw;
    int64_t doubles;
    double *Cp, *CL, *tabs, *big, *P1, *P2, *P3, *D;
};
// Workspace of the coefficient stage (doubles; every piece 16-byte aligned).  N = 0: the prior buffers only.
CoefLayout coef_layout(int64_t N, int64_t npad, int64_t rxL, int64_t ryL, int64_t rxH, int64_t ryH, int64_t S, void* work) {
    CoefLayout L{};
    L.N = N; L.npad = npad;
    L.rx = rxL > rxH ? rxL : rxH; L.ry = ryL > ryH ? ryL : ryH; L.kpad = rup(L.rx, 4);
    L.R = L.ry * L.kpad; L.Rp = rup(L.R, SG_RP); L.Sw = rup(S, 2);
    double* wp = static_cast<double*>(work);
    int64_t used = 0;
    auto carve = [&](int64_t n) { double* r = wp ? wp + used : nullptr; used += rup(n, 8); return r; };
    L.Cp = carve(L.Sw * L.R);
    L.CL = carve(L.Sw * L.R);
    if (N > 0) {
        L.tabs = carve((rxL + ryL + rxH + ryH) * npad);
        L.big = carve(npad * L.Rp);
        L.P1 = carve(npad * L.Sw);
        L.P2 = carve(npad * L.Sw);
        L.P3 = carve(npad * L.Sw);
        L.D = carve(L.Rp * L.Sw);
    }
    L.doubles = used;
    return L;
}

bool orders_ok(bool multi, int64_t rxL, int64_t ryL, int64_t rxH, int64_t ryH) {
    if (rxH <= 0 || ryH <= 0 || rxH > F_MAXR || ryH > F_MAXR || (ryH & 3)) return false;
    if (multi) return rxL > 0 && ryL > 0 && rxL <= F_MAXR && ryL <= F_MAXR && !(ryL & 3);
    return rxL == 0 && ryL == 0;
}

int64_t eval_doubles(int64_t ncols, int64_t ny, int64_t rx, int64_t ry, int64_t S) {
    return rup(rup(ncols, 64) * rup(rx, 4), 8) + rup(ny * ry, 8) + rup(rup(ncols, 64) * S * ry, 8);
}

}  // namespace mfgp

using namespace mfgp;

extern "C" int64_t mfgp_grid_sample_coef_workspace_bytes(int64_t N, int64_t rxL, int64_t ryL, int64_t rxH, int64_t ryH, int64_t S) {
    if (N < 0 || S <= 0) return 0;
    return coef_layout(N, N ? rup(N, MFGP_TILE) : 0, rxL, ryL, rxH, ryH, S, nullptr).doubles * 8 + 256;
}

extern "C" int mfgp_grid_sample_coef(const double* Xt, const double* y, int64_t NL, int64_t NH, const double* W, int64_t npad,
                                     int64_t ldw, const mfgp_params* p_host, int64_t rxL, int64_t ryL, int64_t rxH, int64_t ryH,
                                     double xlo, double xhi, double ylo, double yhi, const double* QxL, const double* QyL,
                                     const double* QxH, const double* QyH, const double* E, int64_t lde, int64_t S, double* C,
                                     void* work, int64_t work_bytes, void* stream) {
    if (!p_host || !E || !C || !work || !QxH || !QyH || NL < 0 || NH < 0 || S <= 0) return MFGP_ERR_INVALID;
    const bool multi = p_host->multi != 0;
    const int64_t N = NL + NH;
    if (!orders_ok(multi, rxL, ryL, rxH, ryH) || (multi && (!QxL || !QyL)) || (!multi && NL)) return MFGP_ERR_INVALID;
    if (!(xhi > xlo) || !(yhi > ylo) || !std::isfinite(xhi - xlo) || !std::isfinite(yhi - ylo)) return MFGP_ERR_INVALID;
    const int64_t d = rxL * ryL + rxH * ryH + N;
    if (!al16(E) || !al16(C) || (lde & 1) || lde < S || S >= (1LL << 24) || d >= (1LL << 31) / 2) return MFGP_ERR_INVALID;
    if (N > 0) {
        if (!Xt || !y || !W || !al16(W) || (ldw & 1) || npad != rup(N, MFGP_TILE) || ldw < npad || npad > (1 << 20))
            return MFGP_ERR_INVALID;
    }
    const CoefLayout chk = coef_layout(N, N ? npad : 0, rxL, ryL, rxH, ryH, S, nullptr);
    if (!al16(work) || work_bytes < chk.doubles * 8) return MFGP_ERR_INVALID;
    const CoefLayout L = coef_layout(N, N ? npad : 0, rxL, ryL, rxH, ryH, S, work);
    const DevParams dp = make_dev_params(*p_host);
    cudaStream_t st = static_cast<cudaStream_t>(stream);

    MFGP_CUDA_CHECK(cudaMemsetAsync(L.Cp, 0, sizeof(double) * (L.CL - L.Cp + L.Sw * L.R), st));     // Cp, CL (padding draw too)
    PriorArgs pa{};
    pa.E = E; pa.lde = lde; pa.S = (int)S;
    pa.Qx[0] = QxL; pa.Qy[0] = QyL; pa.Qx[1] = QxH; pa.Qy[1] = QyH;
    pa.rx[0] = (int)rxL; pa.ry[0] = (int)ryL; pa.rx[1] = (int)rxH; pa.ry[1] = (int)ryH;
    pa.off[0] = 0; pa.off[1] = (int)(rxL * ryL);
    pa.sq[0] = multi ? std::sqrt(p_host->s_L) : 0.0; pa.sq[1] = std::sqrt(p_host->s_H);
    pa.first = multi ? 0 : 1;
    pa.kpad = (int)L.kpad; pa.R = (int)L.R; pa.rho = dp.rho;
    pa.CL = L.CL; pa.Cp = L.Cp;
    MFGP_CUDA_CHECK(cudaFuncSetAttribute(prior_coef_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PC_SMEM));
    prior_coef_kernel<<<(unsigned)S, 256, PC_SMEM, st>>>(pa);
    MFGP_LAUNCH_CHECK();
    if (N == 0) {
        combine_kernel<<<(unsigned)((S * L.R + 255) / 256), 256, 0, st>>>(L.Cp, nullptr, 0, (int)L.R, (int)S, C);
        MFGP_LAUNCH_CHECK();
        return MFGP_OK;
    }
    const int Sw = (int)L.Sw;
    // the prior draws at the training points: f_L (lofi rows) and f_H (hifi rows), row tiles covering each range
    train_basis_kernel<<<(unsigned)npad, 256, 0, st>>>(Xt, (int)N, xlo, xhi, ylo, yhi, (int)L.rx, (int)L.ry, (int)L.kpad, (int)L.Rp, L.big);
    MFGP_LAUNCH_CHECK();
    GemmArgs g{};
    g.lda = L.Rp; g.ldb = L.R; g.ldc = Sw; g.N = Sw; g.K = (int)L.R; g.alpha = 1.0; g.mode = GEMM_GENERAL;
    if (NL > 0) {
        g.A = L.big; g.B = L.CL; g.C = L.P1; g.M = (int)rup(NL, 64);
        if (int rc = launch_gemm(g, true, 1, st)) return rc;
    }
    if (NH > 0) {
        const int64_t h0 = NL / 64 * 64;
        g.A = L.big + h0 * L.Rp; g.B = L.Cp; g.C = L.P2 + h0 * Sw; g.M = (int)(npad - h0);
        if (int rc = launch_gemm(g, true, 1, st)) return rc;
    }
    {
        const int64_t tot = npad * Sw;
        residual_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(y, L.P1, L.P2, Sw, E, lde, rxL * ryL + rxH * ryH, (int)N,
                                                                     (int)NL, (int)npad, (int)S, dp.mean_L, dp.mean_H,
                                                                     std::sqrt(dp.noise_L + dp.jitter), std::sqrt(dp.noise_H + dp.jitter), L.P3);
        MFGP_LAUNCH_CHECK();
    }
    // alpha = W^T (W R) = K^-1 R
    GemmArgs w{};
    w.A = W; w.lda = ldw; w.B = L.P3; w.ldb = Sw; w.C = L.P1; w.ldc = Sw;
    w.M = (int)npad; w.N = Sw; w.K = (int)npad; w.alpha = 1.0; w.mode = GEMM_A_LOWER;
    if (int rc = launch_gemm(w, false, 1, st)) return rc;
    w.B = L.P1; w.C = L.P2; w.mode = GEMM_AT_LOWER;
    if (int rc = launch_gemm_at(w, st)) return rc;
    // B: the cross-covariance's coefficients on the box (gp_factored.cu step 2, uniform layout), into the Phi buffer
    {
        double* tp = L.tabs;
        ChebJobs jobs = {};
        BTab bt[2] = {};
        int nt = 0;
        auto add = [&](int64_t rx, int64_t ry, double l, bool lofi) {
            double* Cx = tp; tp += rx * npad;
            double* Cy = tp; tp += ry * npad;
            jobs.j[2 * nt] = ChebJob{0, (int)rx, xlo, xhi, 1.0 / l, Cx};
            jobs.j[2 * nt + 1] = ChebJob{1, (int)ry, ylo, yhi, 1.0 / l, Cy};
            bt[nt] = BTab{Cx, Cy, (int)rx, (int)ry, lofi ? dp.rho * dp.s_L : 0.0, lofi ? dp.rho2 * dp.s_L : dp.s_H};
            nt++;
        };
        if (multi) add(rxL, ryL, p_host->l_L, true);
        add(rxH, ryH, p_host->l_H, false);
        dim3 cgrid((unsigned)((npad + CHEB_PTS - 1) / CHEB_PTS), (unsigned)(2 * nt));
        cheb_coef_kernel<<<cgrid, 256, 0, st>>>(Xt, (int)N, (int)npad, jobs);
        MFGP_LAUNCH_CHECK();
        FTrunc tr{};
        tr.ry = (int)L.ry;
        for (int l = 0; l <= F_MAXR; l++) tr.off[l] = (short)((l < L.ry ? l : L.ry) * L.kpad);
        for (int l = 0; l < F_MAXR; l++) tr.kx[l] = (short)(l < L.ry ? L.kpad : 0);
        tr.cols = (int)L.R;
        if (L.Rp > L.R) MFGP_CUDA_CHECK(cudaMemset2DAsync(L.big + L.R, L.Rp * 8, 0, (L.Rp - L.R) * 8, npad, st));
        dim3 bgrid((unsigned)((L.R + 127) / 128), (unsigned)npad);
        build_B_merged_kernel<<<bgrid, 128, 0, st>>>(bt[0], bt[1], nt, (int)npad, (int)N, (int)NL, tr, L.big, L.Rp);
        MFGP_LAUNCH_CHECK();
    }
    // D = B^T alpha, then C_s = C_prior,s + D_s
    GemmArgs b{};
    b.A = L.big; b.lda = L.Rp; b.B = L.P2; b.ldb = Sw; b.C = L.D; b.ldc = Sw;
    b.M = (int)L.Rp; b.N = Sw; b.K = (int)npad; b.alpha = 1.0; b.mode = GEMM_GENERAL;
    if (int rc = launch_gemm_at(b, st)) return rc;
    combine_kernel<<<(unsigned)((S * L.R + 255) / 256), 256, 0, st>>>(L.Cp, L.D, Sw, (int)L.R, (int)S, C);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

extern "C" int64_t mfgp_grid_sample_eval_workspace_bytes(int64_t ncols, int64_t ny, int64_t rx, int64_t ry, int64_t S) {
    if (ncols <= 0 || ny <= 0 || rx <= 0 || ry <= 0 || S <= 0) return 0;
    return eval_doubles(ncols, ny, rx, ry, S) * 8 + 256;
}

extern "C" int mfgp_grid_sample_eval(const double* ux, int64_t nx, const double* uy, int64_t ny, int64_t ix0, int64_t ncols,
                                     double xlo, double xhi, double ylo, double yhi, int64_t rx, int64_t ry, const double* C,
                                     int64_t S, double mean, double* F, int64_t ldf, void* work, int64_t work_bytes, void* stream) {
    if (!ux || !uy || !C || !F || !work || nx <= 0 || ny <= 0 || ix0 < 0 || ncols <= 0 || ix0 + ncols > nx || S <= 0)
        return MFGP_ERR_INVALID;
    if (rx <= 0 || rx > F_MAXR || ry <= 0 || ry > F_MAXR || (ry & 3)) return MFGP_ERR_INVALID;
    if (!(xhi > xlo) || !(yhi > ylo) || !std::isfinite(xhi - xlo) || !std::isfinite(yhi - ylo)) return MFGP_ERR_INVALID;
    if (!al16(C) || !al16(F) || !al16(work) || (ldf & 1) || ldf < S) return MFGP_ERR_INVALID;
    const int64_t kpad = rup(rx, 4), ncp = rup(ncols, 64);
    const int64_t ytiles = (ny + EV_BM - 1) / EV_BM, stiles = (S + EV_BN - 1) / EV_BN, zt = (ytiles + EV_TILES - 1) / EV_TILES;
    if (ncols >= (1LL << 31) || ny >= (1LL << 31) || stiles > 65535 || zt > 65535 || S * ry >= (1LL << 31)) return MFGP_ERR_INVALID;
    if (work_bytes < eval_doubles(ncols, ny, rx, ry, S) * 8) return MFGP_ERR_INVALID;
    double* wp = static_cast<double*>(work);
    double* Ux = wp;
    double* Uy = Ux + rup(ncp * kpad, 8);
    double* Hc = Uy + rup(ny * ry, 8);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MFGP_CUDA_CHECK(cudaMemsetAsync(Ux, 0, sizeof(double) * ncp * kpad, st));
    cheb_basis_kernel<<<(unsigned)((ncp + 127) / 128), 128, 0, st>>>(ux, (int)ix0, (int)ncols, (int)ncp, xlo, xhi, (int)rx, (int)kpad, 0, Ux);
    MFGP_LAUNCH_CHECK();
    cheb_basis_kernel<<<(unsigned)((ny + 127) / 128), 128, 0, st>>>(uy, 0, (int)ny, (int)ny, ylo, yhi, (int)ry, (int)ry, 0, Uy);
    MFGP_LAUNCH_CHECK();
    GemmArgs g{};           // Hc[ix][(s, l)] = sum_k Ux[ix][k] C[(s, l)][k]
    g.A = Ux; g.lda = kpad; g.B = C; g.ldb = kpad; g.C = Hc; g.ldc = S * ry;
    g.M = (int)ncp; g.N = (int)(S * ry); g.K = (int)kpad; g.alpha = 1.0; g.mode = GEMM_GENERAL;
    if (int rc = launch_gemm(g, true, 1, st)) return rc;
    EvalArgs a{};
    a.Uy = Uy; a.Hc = Hc; a.ldh = S * ry; a.F = F; a.ldf = ldf;
    a.ny = (int)ny; a.S = (int)S; a.ry = (int)ry; a.pitch = (int)((ry + 11) / 16 * 16 + 4); a.ytiles = (int)ytiles; a.mean = mean;
    const int smem = (int)(sizeof(double) * (EV_BN + 2 * EV_BM) * a.pitch);
    MFGP_CUDA_CHECK(cudaFuncSetAttribute(grid_sample_eval_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    grid_sample_eval_kernel<<<dim3((unsigned)ncols, (unsigned)stiles, (unsigned)zt), EV_THREADS, smem, st>>>(a);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}
