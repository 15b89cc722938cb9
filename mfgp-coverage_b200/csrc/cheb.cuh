// Chebyshev building blocks shared by the factored posterior (gp_factored.cu) and the pathwise grid sampler
// (gp_sample_grid.cu): coefficient tables of the training points' axis factors, basis tables of grid axes, and the merged
// coefficient matrix B of the cross-covariance.  `static`: each translation unit that includes this gets its own copy.
#pragma once
#include "common.cuh"

namespace mfgp {

constexpr int F_MAXR = 64;           // largest supported Chebyshev order per axis and part

// Column layout of the right-hand sides: term (l, k) -- T_l(ty) T_k(tx) -- sits in column off[l] + k, k < kx[l].  Uniform: kx[l] =
// kpad for every l.  Truncated: the caller keeps, per y term l, only the x terms whose coefficient bound a_y[l] a_x[k] is above
// its tolerance (the coefficients of an entire function decay super-exponentially in BOTH indices, so the tensor block's far
// corner is below rounding): ~1/3 fewer columns at the same entrywise accuracy.  Passed to kernels by value.
struct FTrunc {
    short off[F_MAXR + 1];
    short kx[F_MAXR];
    int ry, cols;
};

// ---- step 1a: Chebyshev coefficients c_k(n) of u -> exp(-0.5 ((u - U_n)/l)^2) on [lo, hi] --------------------------------------
// One launch for every (kernel part, axis) job (blockIdx.y); a CTA tabulates the job's r x r DCT matrix once in shared memory
// and then serves 32 training points, one warp per point at a time.
struct ChebJob { int axis, r; double lo, hi, inv_l; double* C; };
struct ChebJobs { ChebJob j[4]; };
constexpr int CHEB_PTS = 32;         // training points per CTA
static __global__ void __launch_bounds__(256) cheb_coef_kernel(const double* __restrict__ Xt, int N, int npad, ChebJobs jobs) {
    __shared__ double D[F_MAXR * (F_MAXR + 1)];     // D[k][j] = w_k cos(pi k (j + 1/2) / r), odd pitch: conflict-free over k
    __shared__ double node[F_MAXR];
    __shared__ double fv[8][F_MAXR];
    const ChebJob jb = jobs.j[blockIdx.y];
    const int r = jb.r, lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    double* __restrict__ C = jb.C;
    const double mid = 0.5 * (jb.lo + jb.hi), half = 0.5 * (jb.hi - jb.lo);
    for (int e = threadIdx.x; e < r * r; e += 256) {
        const int k = e / r, j = e % r;
        D[k * (F_MAXR + 1) + j] = cospi(k * (j + 0.5) / r) * (k == 0 ? 1.0 : 2.0) / r;
    }
    for (int j = threadIdx.x; j < r; j += 256) node[j] = mid + half * cospi((j + 0.5) / r);
    __syncthreads();
    for (int i = wib; i < CHEB_PTS; i += 8) {
        const int n = blockIdx.x * CHEB_PTS + i;
        if (n >= npad) break;
        if (n >= N) {                    // padding columns carry zeros
            for (int k = lane; k < r; k += 32) C[(int64_t)k * npad + n] = 0.0;
            continue;
        }
        const double U = Xt[2 * n + jb.axis];
        __syncwarp();
        for (int j = lane; j < r; j += 32) {
            const double d = (node[j] - U) * jb.inv_l;
            fv[wib][j] = exp(-0.5 * d * d);
        }
        __syncwarp();
        for (int k = lane; k < r; k += 32) {
            double s0 = 0.0;
            for (int j = 0; j < r; j++) s0 = fma(fv[wib][j], D[k * (F_MAXR + 1) + j], s0);
            C[(int64_t)k * npad + n] = s0;
        }
    }
}

// ---- step 1b: T_k(t(u)) for the grid axis values u[i], rows padded with zeros ------------------------------------------------
static __global__ void cheb_basis_kernel(const double* __restrict__ u, int i0, int count, int rows_pad, double lo, double hi, int r, int ld,
                                  int col0, double* __restrict__ T) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows_pad) return;
    double* row = T + (int64_t)i * ld + col0;
    if (i >= count) {
        for (int k = 0; k < r; k++) row[k] = 0.0;
        return;
    }
    const double t = (2.0 * u[i0 + i] - (lo + hi)) / (hi - lo);
    double t0 = 1.0, t1 = t;
    for (int k = 0; k < r; k++) {
        row[k] = t0;
        const double t2 = 2.0 * t * t1 - t0;
        t0 = t1; t1 = t2;
    }
}

// ---- step 2: B[n][l][k] = sum_P coef_P[n] Cy_P[l][n] Cx_P[k][n] ---------------------------------------------------------------
// Both kernel parts expand in the SAME Chebyshev basis T_l(ty) T_k(tx), so their coefficient tensors simply add: one B with
// rx = max(rxL, rxH), ry = max(ryL, ryH) instead of two (the lofi part's terms beyond its own orders are zero):
//   B[n][l][k] = cL[n] CyL[l][n] CxL[k][n] [l < ryL, k < rxL]  +  cH[n] CyH[l][n] CxH[k][n] [l < ryH, k < rxH]
struct BTab { const double* Cx; const double* Cy; int rx, ry; double coef_lo, coef_hi; };
static __global__ void build_B_merged_kernel(BTab t0, BTab t1, int ntab, int npad, int N, int NL, FTrunc tr, double* __restrict__ B,
                                      int64_t ldB) {
    const int n = blockIdx.y;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;       // column of term (l, k)
    if (e >= tr.cols) return;
    int l = 0;
    while (tr.off[l + 1] <= e) l++;
    const int k = e - tr.off[l];
    double v = 0.0;
    if (n < N) {
        if (l < t0.ry && k < t0.rx) v = (n < NL ? t0.coef_lo : t0.coef_hi) * t0.Cy[(int64_t)l * npad + n] * t0.Cx[(int64_t)k * npad + n];
        if (ntab > 1 && l < t1.ry && k < t1.rx)
            v += (n < NL ? t1.coef_lo : t1.coef_hi) * t1.Cy[(int64_t)l * npad + n] * t1.Cx[(int64_t)k * npad + n];
    }
    B[(int64_t)n * ldB + e] = v;
}

}  // namespace mfgp
