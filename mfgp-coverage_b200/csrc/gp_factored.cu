// Factored GP posterior on tensor-product grids (replaces SFGP.predict gaussian_process.py:121-148 / MFGP.predict :401-438,
// diagonal only, for the grids the reference actually uses: `[[x, y] for x in gx for y in gy]`, distribution.py:337-339).
//
// The cross-covariance of grid point (ix, iy) with training point n is separable per kernel part P in {lofi, hifi}:
//     psi[n] = sum_P coef_P[n] * ex_P(x_ix, X_n) * ey_P(y_iy, Y_n),      e(u, U) = exp(-0.5 ((u - U) / l_P)^2).
// As a function of the grid coordinate each factor is an entire function, so its Chebyshev interpolant on the grid's
// interval converges super-exponentially: with r ~ 20 (l = 0.58) / 36 (l = 0.2) terms the factor tables are reproduced to
// ~5e-15 ENTRYWISE (not a low-rank approximation of the training covariance -- nothing about K is truncated):
//     ex_P(x, X_n) = sum_k T_k(tx) Cx_P[k][n],    ey_P(y, Y_n) = sum_l T_l(ty) Cy_P[l][n].
// Then  v(ix, iy) = W psi = sum_{P,l} T_l(ty) * [ sum_k T_k(tx) * Y_P[:, l, k] ],   Y_P = W B_P,
//     B_P[n][l][k] = coef_P[n] Cy_P[l][n] Cx_P[k][n]                      (N x R_P, R_P = ry_P * kpad_P)
// and the whole grid costs ONE product W B (N^2 R / 2 MACs, R ~ 2.5k) instead of N^2 / 2 MACs PER GRID POINT:
//   step 1  Chebyshev coefficient tables of the training points, basis tables of the grid axes        (tiny)
//   step 2  B_P                                                                                         (84 MB at c4)
//   step 3  Y_P = W B_P                      DMMA tile GEMM, W lower triangular                         (2.1e10 MAC at c4)
//   step 4  Y'_P[ix][n][l] = sum_k Ux_P[ix][k] Y_P[n][l][k]      DMMA tile GEMM, per chunk of columns   (1.1e10 MAC)
//   step 5  G'(ix) = Y'(ix)^T Y'(ix)  (64 x 64),  h'(ix) = Y'(ix)^T z       one CTA per column, DMMA    (1.7e10 MAC)
//   step 6  var(ix, iy) = k0 - uy^T G'(ix) uy,  mu = mean + h'(ix) . uy      same CTA, G' in shared memory
// against 8.8e12 MAC for the dense path at c4 (1 M points, N = 4096).  Agreement with the dense path / the oracle:
// ~2e-14 k(0) (tests/test_gpu_factored.py).  Arbitrary point lists keep the dense path (gp_posterior.cu).
#include "common.cuh"
#include "gemm_f64.cuh"
#include <cstdlib>
#include <cstring>

namespace mfgp {

constexpr int F_LW = 64;             // padded number of y-expansion terms of the merged expansion (max(ryL, ryH) <= 64)
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

struct FPart {                       // one kernel part (lofi / hifi) of the factored expansion
    int rx, ry, kpad;                // x terms, y terms (multiple of 4), x terms padded to a multiple of 4
    int loff;                        // first column of this part inside the 64-wide y-term vector
    double inv_l;                    // 1 / length scale
    double* Cx; double* Cy;          // [r][npad] Chebyshev coefficients of the training points' axis factors
    double* B;  double* Y;           // [npad][ry * kpad]
    double* Ux;                      // [ncols_pad][kpad]  T_k(tx) of the grid columns
    double* Yp;                      // [chunk][npad][ry]  step-4 output of one chunk of columns
    double* Hz;                      // [ry][kpad]  z^T Y
};

// ---- step 1a: Chebyshev coefficients c_k(n) of u -> exp(-0.5 ((u - U_n)/l)^2) on [lo, hi] --------------------------------------
// One launch for every (kernel part, axis) job (blockIdx.y); a CTA tabulates the job's r x r DCT matrix once in shared memory
// and then serves 32 training points, one warp per point at a time.
struct ChebJob { int axis, r; double lo, hi, inv_l; double* C; };
struct ChebJobs { ChebJob j[4]; };
constexpr int CHEB_PTS = 32;         // training points per CTA
__global__ void __launch_bounds__(256) cheb_coef_kernel(const double* __restrict__ Xt, int N, int npad, ChebJobs jobs) {
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
__global__ void cheb_basis_kernel(const double* __restrict__ u, int i0, int count, int rows_pad, double lo, double hi, int r, int ld,
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
__global__ void build_B_merged_kernel(BTab t0, BTab t1, int ntab, int npad, int N, int NL, FTrunc tr, double* __restrict__ B,
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

// centred observations behind B: column 0 of the block = y - mean (gaussian_process.py:133, :419-424), the padding columns zero
__global__ void build_z_block_kernel(const double* __restrict__ y, int npad, int N, int NL, double mean_L, double mean_H,
                                     double* __restrict__ B, int64_t ldB) {
    const int n = blockIdx.x, c = threadIdx.x;
    double v = 0.0;
    if (c == 0 && n < N) v = y[n] - (n < NL ? mean_L : mean_H);
    B[(int64_t)n * ldB + c] = v;
}

// Y_all[n][off + e] -> contiguous Y_P[n][e] (step 4 views Y_P as a [(n, l)] x [k] matrix), and the solved z column
__global__ void unpack_Y_kernel(const double* __restrict__ Yall, int64_t ldY, int off, int cols, double* __restrict__ Yp) {
    const int n = blockIdx.y;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < cols) Yp[(int64_t)n * cols + e] = Yall[(int64_t)n * ldY + off + e];
}
// column block [zoff, zoff + blockDim.x) of Yall: the whitened observations, then zeros (the layout mfgp_cholesky_solve leaves)
__global__ void put_z_block_kernel(const double* __restrict__ z, int npad, double* __restrict__ Yall, int64_t ldY, int zoff) {
    const int n = blockIdx.x, c = threadIdx.x;
    Yall[(int64_t)n * ldY + zoff + c] = (c == 0) ? z[n] : 0.0;
}
__global__ void unpack_z_kernel(const double* __restrict__ Yall, int64_t ldY, int off, int npad, double* __restrict__ z) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n < npad) z[n] = Yall[(int64_t)n * ldY + off];
}

// Hz[e] = sum_n z[n] Y[n][e]: the mean needs z^T Y only contracted with T_k(tx) per column (h'(ix) = Ux(ix) . Hz).
// Two passes (fixed summation order): HZ_SPLIT row ranges per 32 columns, then one thread per column adds the partials.
constexpr int HZ_SPLIT = 16;
__global__ void __launch_bounds__(256) hz_partial_kernel(const double* __restrict__ Y, const double* __restrict__ z, int npad, int cols,
                                                         double* __restrict__ part) {
    __shared__ double red[8][32];
    const int e = blockIdx.x * 32 + (threadIdx.x & 31), w = threadIdx.x >> 5;
    const int rows = (npad + HZ_SPLIT - 1) / HZ_SPLIT;
    const int n0 = blockIdx.y * rows, n1 = min(npad, n0 + rows);
    double s = 0.0;
    if (e < cols) {
#pragma unroll 4
        for (int n = n0 + w; n < n1; n += 8) s = fma(z[n], Y[(int64_t)n * cols + e], s);
    }
    red[w][threadIdx.x & 31] = s;
    __syncthreads();
    if (w == 0 && e < cols) {
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < 8; k++) t += red[k][threadIdx.x & 31];
        part[(int64_t)blockIdx.y * cols + e] = t;
    }
}
__global__ void hz_reduce_kernel(const double* __restrict__ part, int cols, double* __restrict__ Hz, int accumulate) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= cols) return;
    double t = 0.0;
#pragma unroll
    for (int k = 0; k < HZ_SPLIT; k++) t += part[(int64_t)k * cols + e];
    Hz[e] = accumulate ? Hz[e] + t : t;
}

__global__ void zero_rows_kernel(double* __restrict__ Y, int64_t cols, int nrows) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < cols * nrows) Y[e] = 0.0;
}

// ---- steps 5 + 6: one CTA per grid column --------------------------------------------------------------------------------
constexpr int G_ROWS = 64;           // training rows per chunk

struct GramArgs {
    const double* YpL; const double* YpH; int ryL, ryH;        // step-4 outputs [cols][npad][ry]
    int npad;                                                  // rows of Y' held per column (all rows, or only the new ones)
    double* Gstore;                                            // optional [cols_total][F_LW][F_LW]: G'(ix) kept across calls
    int skip_eval;                                             // 1: stop behind the Gstore update (step 6 runs as geval_mma_kernel)
    int accumulate;                                            // 1: G' = Gstore + (the rows given); the store is updated
    const double* HzL; const double* HzH;                      // z^T Y_P, [ry][kpad]  (h'(ix) = Ux(ix) . Hz)
    const double* UxL; const double* UxH; int kL, kH;          // T_k(tx) of this launch's columns, [cols][kpad]
    const double* Uy;                                          // [ny][F_LW]
    int ny; int col_begin;                                     // first grid column (relative) of this launch
    double mean, k0;
    double* mu; double* var; double* qred;                     // flat outputs, index = col * ny + iy
    int pitch, nstage;                                         // shared-memory row pitch of a staged chunk (doubles), pipeline depth
    int poison;                                                // 1: NaN-fill the dynamic shared memory first (MFGP_DEBUG_POISON_SMEM)
};
constexpr int G_MAXSTAGE = 6;

// mbarrier / bulk-copy primitives (same PTX as gp_posterior.cu)
__device__ __forceinline__ uint32_t f_smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void f_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void f_mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void f_mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
            : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ void f_bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar) : "memory");
}

// G' is symmetric: only the lower 8x8 tiles are formed -- NT (NT + 1) / 2 of them for a padded width WM = 8 NT (15 for the
// usual WM = 40, 36 for WM = 64).  The four warps split the TRAINING ROWS of a chunk (warp w takes k-steps w, w+4, ...) and each
// accumulates ALL the tiles: A and B fragments of a tile pair are the same shared-memory words (A[m][k] = B[k][m] = Y'[k][m]),
// so a k-step costs NT fragment loads for NT (NT + 1) / 2 DMMAs; the four partial Gram matrices are added in fixed order.
// Staging: chunks of 64 training rows of Y'(ix) ride an nstage-deep ring of bulk copies (completion on mbarriers).  The
// shared row pitch is ry when ry = 4 (mod 8) -- fragment reads are then bank-conflict-free as they stand and the whole chunk is
// ONE contiguous 64 ry x 8-byte copy -- else ry + 4 with one copy per row.  Columns [ry, WM) of a staged row alias the next row
// (finite data, or the zero fill); they only ever meet the zero-padded entries of Uy -- but 0 * NaN is NaN, so the zero fill
// reaches past the ring through the last row's column WM - 1 (g_ring_slack).
__host__ __device__ constexpr int g_ring_slack(int wm, int pitch) { return wm - pitch > 8 ? wm - pitch : 8; }
template <int WM>
__global__ void __launch_bounds__(128) gram_eval_kernel(GramArgs a) {
    constexpr int NT = WM / 8, NTILES = NT * (NT + 1) / 2;
    constexpr int GP = WM + 2;
    extern __shared__ __align__(16) double gsm[];
    const int P = a.pitch, NST = a.nstage, ry = a.ryH;
    const int ring = NST * G_ROWS * P + g_ring_slack(WM, P);     // the last row's aliased columns stay inside the (zeroed) buffer
    double* Ts = gsm;                               // [NST][G_ROWS][P]  ring of chunks of Y'(ix)
    double* Gs = gsm + ring;                        // [WM][WM + 2]   (row pitch even: 16-byte loads)
    double* hs = Gs + WM * GP;                      // [F_LW]
    uint64_t* bars = reinterpret_cast<uint64_t*>(hs + 2 * F_LW);    // [NST] "chunk landed"
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int col = blockIdx.x;
    const int gq = lane >> 2, tq = lane & 3;
    const double* src = a.YpH + (int64_t)col * a.npad * ry;
    const uint32_t bar0 = f_smem_u32(bars);
    // zero ring; with `poison`, everything behind it up to the barriers reads NaN until written (a read of it shows in the output)
    const int fill = a.poison ? ring + WM * GP + 2 * F_LW : ring;
    for (int e = tid; e < fill; e += 128) Ts[e] = e < ring ? 0.0 : __longlong_as_double(-1ll);
    if (tid == 0) {
        for (int i = 0; i < NST; i++) f_mbar_init(bar0 + 8 * i, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncthreads();
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");        // generic-proxy zero fill before the async-proxy copies
    const uint32_t chunk_bytes = (uint32_t)(G_ROWS * ry * 8);
    const bool whole = P == ry;
    auto stage = [&](int buf, int n0) {
        if (tid == 0) f_mbar_arrive_expect_tx(bar0 + 8 * buf, chunk_bytes);
        double* dst = Ts + buf * G_ROWS * P;
        if (whole) {
            if (tid == 0) f_bulk_g2s(f_smem_u32(dst), src + (int64_t)n0 * ry, chunk_bytes, bar0 + 8 * buf);
        } else {
            __syncwarp();
            if (tid < G_ROWS) f_bulk_g2s(f_smem_u32(dst + tid * P), src + (int64_t)(n0 + tid) * ry, (uint32_t)(ry * 8), bar0 + 8 * buf);
        }
    };
    double acc[NTILES][2];
#pragma unroll
    for (int t = 0; t < NTILES; t++) acc[t][0] = acc[t][1] = 0.0;
    const int nchunk = a.npad / G_ROWS;
    for (int i = 0; i < NST - 1 && i < nchunk; i++) stage(i, i * G_ROWS);
    int buf = 0, par = 0;
    for (int ch = 0; ch < nchunk; ch++) {
        const int nx = ch + NST - 1;                                      // its buffer was released by the barrier of chunk ch - 1
        if (nx < nchunk) stage(nx % NST, nx * G_ROWS);
        f_mbar_wait(bar0 + 8 * buf, par);
        const double* T = Ts + buf * G_ROWS * P;
#pragma unroll
        for (int ks = 0; ks < G_ROWS / 16; ks++) {
            const double* row = T + (4 * (warp + 4 * ks) + tq) * P + gq;      // fragment word of tile index i: row[8 i]
            double f[NT];
#pragma unroll
            for (int i = 0; i < NT; i++) f[i] = row[8 * i];
#pragma unroll
            for (int i = 0; i < NT; i++)
#pragma unroll
                for (int j = 0; j <= i; j++) dmma884(acc[i * (i + 1) / 2 + j][0], acc[i * (i + 1) / 2 + j][1], f[i], f[j]);
        }
        __syncthreads();                                                  // everybody is done reading `buf`
        if (++buf == NST) { buf = 0; par ^= 1; }
    }
    // G' (both triangles) to shared memory: the warps add their partial sums one after the other
#pragma unroll 1
    for (int w = 0; w < 4; w++) {
        if (warp == w) {
#pragma unroll
            for (int i = 0; i < NT; i++)
#pragma unroll
                for (int j = 0; j <= i; j++) {
                    const int t = i * (i + 1) / 2 + j;
                    const int r = i * 8 + gq, c = j * 8 + tq * 2;           // C fragment: row gq, columns 2 tq, 2 tq + 1
                    double v0 = acc[t][0], v1 = acc[t][1];
                    if (w > 0) { v0 += Gs[r * GP + c]; v1 += Gs[r * GP + c + 1]; }
                    Gs[r * GP + c] = v0;
                    Gs[r * GP + c + 1] = v1;
                    if (i != j) {                                          // mirror (diagonal tiles hold both triangles)
                        Gs[c * GP + r] = v0;
                        Gs[(c + 1) * GP + r] = v1;
                    }
                }
        }
        __syncthreads();
    }
    if (a.Gstore) {          // keep / extend the column's Gram matrix for later row updates (incremental path)
        double* gst = a.Gstore + (int64_t)(a.col_begin + col) * F_LW * F_LW;
        for (int e = tid; e < WM * WM; e += 128) {
            const int r = e / WM, c = e % WM;
            double v = Gs[r * GP + c];
            if (a.accumulate) { v += gst[r * F_LW + c]; Gs[r * GP + c] = v; }
            gst[r * F_LW + c] = v;
        }
        if (a.skip_eval) return;
    }
    // h'(ix)[l] = sum_k Ux(ix)[k] Hz_P[l][k]     (Hz = z^T Y, computed once per posterior by hz_kernel)
    if (tid < F_LW) {
        double h = 0.0;
        if (tid < a.ryL) {
            const double* ux = a.UxL + (int64_t)col * a.kL;
            const double* hz = a.HzL + (int64_t)tid * a.kL;
            for (int k = 0; k < a.kL; k++) h = fma(ux[k], hz[k], h);
        } else if (tid < a.ryL + a.ryH) {
            const double* ux = a.UxH + (int64_t)col * a.kH;
            const double* hz = a.HzH + (int64_t)(tid - a.ryL) * a.kH;
            for (int k = 0; k < a.kH; k++) h = fma(ux[k], hz[k], h);
        }
        hs[tid] = h;
    }
    __syncthreads();
    // step 6: every grid point of the column;  q = sum_l u_l (G_ll u_l + 2 sum_{c<l} G_lc u_c)
    for (int iy = tid; iy < a.ny; iy += 128) {
        const double* up = a.Uy + (int64_t)iy * F_LW;
        double u[WM];
#pragma unroll
        for (int l = 0; l < WM; l += 2) {
            const double2 t = __ldg(reinterpret_cast<const double2*>(up + l));
            u[l] = t.x; u[l + 1] = t.y;
        }
        double q = 0.0, m = 0.0;
#pragma unroll
        for (int l = 0; l < WM; l += 2) {          // rows l, l+1 together: 16-byte loads of G
            const double* g0 = Gs + l * GP;
            const double* g1 = g0 + GP;
            double s0 = 0.0, s1 = 0.0;
#pragma unroll
            for (int c = 0; c < l; c += 2) {
                const double2 a0 = *reinterpret_cast<const double2*>(g0 + c);
                const double2 a1 = *reinterpret_cast<const double2*>(g1 + c);
                s0 = fma(a0.x, u[c], s0); s0 = fma(a0.y, u[c + 1], s0);
                s1 = fma(a1.x, u[c], s1); s1 = fma(a1.y, u[c + 1], s1);
            }
            const double2 d0 = *reinterpret_cast<const double2*>(g0 + l);
            const double2 d1 = *reinterpret_cast<const double2*>(g1 + l);
            s1 = fma(d1.x, u[l], s1);                                  // G[l+1][l] is below the diagonal of row l+1
            q = fma(u[l], fma(2.0, s0, d0.x * u[l]), q);
            q = fma(u[l + 1], fma(2.0, s1, d1.y * u[l + 1]), q);
            m = fma(hs[l], u[l], m);
            m = fma(hs[l + 1], u[l + 1], m);
        }
        const int64_t gidx = (int64_t)(a.col_begin + col) * a.ny + iy;
        a.var[gidx] = a.k0 - q;
        a.mu[gidx] = a.mean + m;
        if (a.qred) a.qred[gidx] = q;
    }
}

// ---- the Gram route ("M route") of steps 4 + 5 -------------------------------------------------------------------------------
// G'(ix)[l][l'] = sum_n Y'(ix)[n][l] Y'(ix)[n][l'],  Y'(ix)[n][l] = sum_k T_k(tx) Y[n][l][k]
//              = sum_{k,k'} T_k(tx) T_k'(tx) M[(l,k)][(l',k')],        M = Y^T Y   (R x R, independent of the column ix).
// So instead of contracting Y with T_k(tx) for every grid column (n_col N R MACs, a [n_col][N][ry] intermediate of 1.2 GB at
// c4) and forming n_col Gram matrices over the N training rows (n_col N w^2 / 2 MACs), ONE symmetric product M = Y^T Y
// (N R^2 / 2 MACs, split over K into a fixed number of partial sums added in order) is followed by ry (ry + 1) / 2 small
// quadratic forms per column -- 4.3e9 instead of 9.4e9 MACs at c4 and no intermediate beyond M (14 MB).  The row of M that
// belongs to the solved observation column z gives z^T Y (the mean's h'(ix)) for free.  Rounding: |Y|_F^2 = tr(B^T K^-1 B)
// is O(k(0)) even for near-singular K (B lives in the smooth subspace), so the R^2-term sum is as accurate as the direct
// Gram sum (measured: both 1e-14 k(0) against the oracle, well- and ill-conditioned hyper-parameters).
__global__ void syrk_reduce_lower_kernel(const double* __restrict__ part, int nsplit, int64_t stride, int n, double* __restrict__ M) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
    if (c >= n || (c >> 6) > (r >> 6)) return;          // tiles on or below the diagonal only
    double s = 0.0;
    for (int z = 0; z < nsplit; z++) s += part[(int64_t)z * stride + (int64_t)r * n + c];
    M[(int64_t)r * n + c] = s;
}

struct QformArgs {
    const double* M; int ldm;            // lower tiles of Y^T Y
    const double* Ux; int kpad;          // [ncols_pad][kpad]  T_k(tx)
    FTrunc tr;                           // block (l, l') of M: rows off[l] .. + kx[l], columns off[l'] .. + kx[l']
    int ry, ncols, pairs_per_cta;
    double* G;                           // [ncols][F_LW][F_LW], both triangles written
    int col_begin;
};
// CTA = 64 grid columns x a range of (l, l') pairs, l' <= l; warp w owns columns 16 w .. 16 w + 15 (two 8-row DMMA tiles).
// Per pair: T = U_blk (64 x kpad) * M_{l l'} (kpad x kpad) on DMMA, then the row-wise dot with U_blk straight off the
// accumulator fragments (two lane shuffles).  The A fragments (U) stay in registers for the whole CTA.
// STAGED (kpad <= 48): the kx[l] x kx[l'] block of M goes through shared memory -- fetched by the whole CTA with coalesced loads
// one pair AHEAD (into registers, parked in shared memory behind the current pair's barrier), so its L2 round trip hides behind
// the DMMA work; !STAGED: every thread loads its B fragments straight from M (four-fold redundant scattered loads: 134 us at
// c4 where the staged form needs 40).
template <int NT, bool STAGED>         // n tiles of 8: kpad <= 8 NT
__global__ void __launch_bounds__(128) qform_kernel(QformArgs a) {
    constexpr int KS = 2 * NT;                                   // k steps of 4
    constexpr int LD = STAGED ? (NT <= 4 ? 36 : 52) : 1;         // 2 LD = 8 (mod 32): conflict-free [k][n] fragment reads
    constexpr int PRE = STAGED ? 4 * NT : 1;                     // thread = (column n = tid & 63, rows (tid >> 6) + 2 i): no index division
    __shared__ double Us[64][8 * NT + 1];
    __shared__ double Bs[STAGED ? 8 * NT * LD : 1];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, gq = lane >> 2, tq = lane & 3;
    const int c0 = blockIdx.x * 64;
    for (int e = tid; e < 64 * 8 * NT; e += 128) {
        const int r = e / (8 * NT), k = e % (8 * NT);
        Us[r][k] = (k < a.kpad) ? a.Ux[(int64_t)(c0 + r) * a.kpad + k] : 0.0;      // Ux rows beyond ncols are zero-padded
    }
    __syncthreads();
    double af[2][KS];
#pragma unroll
    for (int rt = 0; rt < 2; rt++)
#pragma unroll
        for (int ks = 0; ks < KS; ks++) af[rt][ks] = Us[warp * 16 + rt * 8 + gq][ks * 4 + tq];
    const int npairs = a.ry * (a.ry + 1) / 2;
    int p = blockIdx.y * a.pairs_per_cta;
    const int pend = min(npairs, p + a.pairs_per_cta);
    int l = (int)((sqrt(8.0 * p + 1.0) - 1.0) * 0.5);
    while ((l + 1) * (l + 2) / 2 <= p) l++;
    while (l * (l + 1) / 2 > p) l--;
    int lp = p - l * (l + 1) / 2;
    double pre[PRE];
    auto fetch = [&](int fl, int flp) {              // this thread's share of block (fl, flp) of M -> registers
        const int ra = a.tr.off[fl], rb = a.tr.off[flp], ka = a.tr.kx[fl], kb = a.tr.kx[flp];
        const int n = tid & 63, c = rb + n;
#pragma unroll
        for (int i = 0; i < PRE; i++) {
            const int k = (tid >> 6) + 2 * i, r = ra + k;
            double v = 0.0;
            if (k < ka && n < kb)                                  // M is symmetric, stored for row tile >= column tile
                v = (r >= c) ? __ldg(a.M + (int64_t)r * a.ldm + c) : __ldg(a.M + (int64_t)c * a.ldm + r);
            pre[i] = v;
        }
    };
    auto stash = [&](int fl, int flp) {
        const int ka = a.tr.kx[fl], kb = a.tr.kx[flp], n = tid & 63;
#pragma unroll
        for (int i = 0; i < PRE; i++) {
            const int k = (tid >> 6) + 2 * i;
            if (k < ka && n < kb) Bs[k * LD + n] = pre[i];
        }
    };
    if (STAGED && p < pend) {
        fetch(l, lp);
        stash(l, lp);
        __syncthreads();
    }
    for (; p < pend; p++) {
        int nl = l, nlp = lp + 1;
        if (nlp > nl) { nl++; nlp = 0; }
        const bool more = p + 1 < pend;
        if (STAGED && more) fetch(nl, nlp);          // in flight while this pair is computed
        double acc[2][NT][2];
#pragma unroll
        for (int rt = 0; rt < 2; rt++)
#pragma unroll
            for (int j = 0; j < NT; j++) acc[rt][j][0] = acc[rt][j][1] = 0.0;
        const int ra = a.tr.off[l], rb = a.tr.off[lp], ka = a.tr.kx[l], kb = a.tr.kx[lp];
#pragma unroll
        for (int ks = 0; ks < KS; ks++) {
            if (ks * 4 >= ka) break;                               // (uniform) the block has only ka rows
            const int k = ks * 4 + tq;
            double b[NT];
#pragma unroll
            for (int j = 0; j < NT; j++) {
                const int n = j * 8 + gq;
                double v = 0.0;
                if (k < ka && n < kb) {
                    if (STAGED) {
                        v = Bs[k * LD + n];
                    } else {
                        const int r = ra + k, c = rb + n;
                        v = (r >= c) ? __ldg(a.M + (int64_t)r * a.ldm + c) : __ldg(a.M + (int64_t)c * a.ldm + r);
                    }
                }
                b[j] = v;
            }
#pragma unroll
            for (int rt = 0; rt < 2; rt++)
#pragma unroll
                for (int j = 0; j < NT; j++)
                    if (j * 8 < kb) dmma884(acc[rt][j][0], acc[rt][j][1], af[rt][ks], b[j]);       // (uniform) kb columns
        }
#pragma unroll
        for (int rt = 0; rt < 2; rt++) {
            const int row = warp * 16 + rt * 8 + gq;
            double q = 0.0;
#pragma unroll
            for (int j = 0; j < NT; j++) {                         // columns >= kb of the accumulators are zero
                q = fma(acc[rt][j][0], Us[row][j * 8 + 2 * tq], q);
                q = fma(acc[rt][j][1], Us[row][j * 8 + 2 * tq + 1], q);
            }
            q += __shfl_xor_sync(0xffffffffu, q, 1);
            q += __shfl_xor_sync(0xffffffffu, q, 2);
            if (tq == 0 && c0 + row < a.ncols) {
                double* g = a.G + (int64_t)(a.col_begin + c0 + row) * F_LW * F_LW;
                g[l * F_LW + lp] = q;
                g[lp * F_LW + l] = q;
            }
        }
        if (STAGED) {
            __syncthreads();                         // every warp is done with this pair's block
            if (more) {
                stash(nl, nlp);
                __syncthreads();
            }
        }
        l = nl; lp = nlp;
    }
}

// step 6 on its own (Gram route: G'(ix) is already complete in global memory): one CTA per grid column, 256 threads, each
// thread evaluates TWO grid points at a time (eight independent FMA chains), G' in shared memory (broadcast reads).
//   var = k0 - uy^T G' uy,   mu = mean + h'(ix) . uy,   h'(ix)[l] = sum_k Ux(ix)[k] Hz[l][k]
template <int WM, int NP>          // NP = 2: two points per thread (WM = 40), 1: one (WM = 64: the u vector alone takes 128 registers)
__global__ void __launch_bounds__(256) geval_kernel(const double* __restrict__ G, const double* __restrict__ Hz, const double* __restrict__ Ux,
                                                    int kpad, int ry, FTrunc tr, const double* __restrict__ Uy, int ny, double mean, double k0,
                                                    double* __restrict__ mu, double* __restrict__ var, double* __restrict__ qred) {
    constexpr int GP = WM + 2;
    __shared__ __align__(16) double Gs[WM * GP];
    __shared__ double hs[WM];
    const int tid = threadIdx.x, col = blockIdx.x;
    const double* g = G + (int64_t)col * F_LW * F_LW;
    for (int e = tid; e < WM * WM; e += 256) {
        const int r = e / WM, c = e % WM;
        Gs[r * GP + c] = (r < ry && c < ry) ? g[r * F_LW + c] : 0.0;
    }
    if (tid < WM) {
        double h = 0.0;
        if (tid < ry) {
            const double* ux = Ux + (int64_t)col * kpad;
            const double* hz = Hz + tr.off[tid];
            for (int k = 0; k < tr.kx[tid]; k++) h = fma(ux[k], hz[k], h);
        }
        hs[tid] = h;
    }
    __syncthreads();
    for (int iy0 = NP * tid; iy0 < ny; iy0 += NP * 256) {
        double u[NP][WM];
#pragma unroll
        for (int p = 0; p < NP; p++) {
            const double* up = Uy + (int64_t)min(iy0 + p, ny - 1) * F_LW;
#pragma unroll
            for (int l = 0; l < WM; l += 2) {
                const double2 a = __ldg(reinterpret_cast<const double2*>(up + l));
                u[p][l] = a.x; u[p][l + 1] = a.y;
            }
        }
        double q[NP], m[NP];
#pragma unroll
        for (int p = 0; p < NP; p++) q[p] = m[p] = 0.0;
#pragma unroll
        for (int l = 0; l < WM; l += 2) {          // rows l, l+1 together: 16-byte loads of G; the same sums as gram_eval_kernel
            const double* g0 = Gs + l * GP;
            const double* g1 = g0 + GP;
            double s0[NP], s1[NP];
#pragma unroll
            for (int p = 0; p < NP; p++) s0[p] = s1[p] = 0.0;
#pragma unroll
            for (int c = 0; c < l; c += 2) {
                const double2 a0 = *reinterpret_cast<const double2*>(g0 + c);
                const double2 a1 = *reinterpret_cast<const double2*>(g1 + c);
#pragma unroll
                for (int p = 0; p < NP; p++) {
                    s0[p] = fma(a0.x, u[p][c], s0[p]); s0[p] = fma(a0.y, u[p][c + 1], s0[p]);
                    s1[p] = fma(a1.x, u[p][c], s1[p]); s1[p] = fma(a1.y, u[p][c + 1], s1[p]);
                }
            }
            const double2 d0 = *reinterpret_cast<const double2*>(g0 + l);
            const double2 d1 = *reinterpret_cast<const double2*>(g1 + l);
#pragma unroll
            for (int p = 0; p < NP; p++) {
                s1[p] = fma(d1.x, u[p][l], s1[p]);                              // G[l+1][l] is below the diagonal of row l+1
                q[p] = fma(u[p][l], fma(2.0, s0[p], d0.x * u[p][l]), q[p]);
                q[p] = fma(u[p][l + 1], fma(2.0, s1[p], d1.y * u[p][l + 1]), q[p]);
                m[p] = fma(hs[l], u[p][l], m[p]);
                m[p] = fma(hs[l + 1], u[p][l + 1], m[p]);
            }
        }
#pragma unroll
        for (int p = 0; p < NP; p++) {
            if (iy0 + p >= ny) continue;
            const int64_t gidx = (int64_t)col * ny + iy0 + p;
            var[gidx] = k0 - q[p];
            mu[gidx] = mean + m[p];
            if (qred) qred[gidx] = q[p];
        }
    }
}

// The same step 6 on the tensor pipe: per grid column T' = Uy (ny x WM) B' (WM x WM) with B' the lower triangle of G'(ix), strictly
// lower entries doubled (u^T G' u = sum_{n <= k} B'[k][n] u_k u_n), then the row-wise dot with Uy straight off the accumulator
// fragments.  B' is lower triangular, so only the 8-column tiles j with 8 j <= 4 ks + 3 of k step ks are non-zero (30 of 50 at
// WM = 40); its fragments stay in registers for the whole column.  The FMA form above is fully unrolled over the triangle
// (~6000 FMAs of straight-line code per point pair, 224 registers, one CTA per SM) and reaches a quarter of the FP64 rate;
// this one is a 30-DMMA loop body: 177 -> ~70 us at c4.
template <int WM>
__global__ void __launch_bounds__(128) geval_mma_kernel(const double* __restrict__ G, const double* __restrict__ Hz,
                                                        const double* __restrict__ Ux, int kpad, int ry, FTrunc tr,
                                                        const double* __restrict__ Uy, int ny, double mean, double k0,
                                                        double* __restrict__ mu, double* __restrict__ var, double* __restrict__ qred) {
    constexpr int NT = WM / 8, KS = WM / 4, GP = WM + 1;
    __shared__ double Gs[WM * GP];
    __shared__ double hs[WM];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, gq = lane >> 2, tq = lane & 3;
    const int col = blockIdx.x;
    const double* g = G + (int64_t)col * F_LW * F_LW;
    for (int e = tid; e < WM * WM; e += 128) {
        const int k = e / WM, n = e % WM;
        double v = 0.0;
        if (k < ry && n <= k) v = (n < k) ? 2.0 * g[k * F_LW + n] : g[k * F_LW + k];
        Gs[k * GP + n] = v;
    }
    if (tid < WM) {
        double h = 0.0;
        if (tid < ry) {
            const double* ux = Ux + (int64_t)col * kpad;
            const double* hz = Hz + tr.off[tid];
            for (int k = 0; k < tr.kx[tid]; k++) h = fma(ux[k], hz[k], h);
        }
        hs[tid] = h;
    }
    __syncthreads();
    double bf[KS][NT];
#pragma unroll
    for (int ks = 0; ks < KS; ks++)
#pragma unroll
        for (int j = 0; j < NT; j++) bf[ks][j] = (8 * j <= 4 * ks + 3) ? Gs[(ks * 4 + tq) * GP + j * 8 + gq] : 0.0;
    double h0[NT], h1[NT];
#pragma unroll
    for (int j = 0; j < NT; j++) { h0[j] = hs[j * 8 + 2 * tq]; h1[j] = hs[j * 8 + 2 * tq + 1]; }
    for (int m0 = warp * 8; m0 < ny; m0 += 32) {
        const double* up = Uy + (int64_t)min(m0 + gq, ny - 1) * F_LW;
        double acc[NT][2];
#pragma unroll
        for (int j = 0; j < NT; j++) acc[j][0] = acc[j][1] = 0.0;
#pragma unroll
        for (int ks = 0; ks < KS; ks++) {
            const double av = __ldg(up + ks * 4 + tq);
#pragma unroll
            for (int j = 0; j < NT; j++)
                if (8 * j <= 4 * ks + 3) dmma884(acc[j][0], acc[j][1], av, bf[ks][j]);
        }
        double q = 0.0, m = 0.0;
#pragma unroll
        for (int j = 0; j < NT; j++) {
            const double2 u = __ldg(reinterpret_cast<const double2*>(up + j * 8 + 2 * tq));
            q = fma(acc[j][0], u.x, q); q = fma(acc[j][1], u.y, q);
            m = fma(h0[j], u.x, m); m = fma(h1[j], u.y, m);
        }
        q += __shfl_xor_sync(0xffffffffu, q, 1); m += __shfl_xor_sync(0xffffffffu, m, 1);
        q += __shfl_xor_sync(0xffffffffu, q, 2); m += __shfl_xor_sync(0xffffffffu, m, 2);
        if (tq == 0 && m0 + gq < ny) {
            const int64_t gidx = (int64_t)col * ny + m0 + gq;
            var[gidx] = k0 - q;
            mu[gidx] = mean + m;
            if (qred) qred[gidx] = q;
        }
    }
}

// rows / columns [ry, WM) of every G'(ix) must read as zero for gram_eval's padded quadratic form
__global__ void gpad_zero_kernel(double* __restrict__ G, int ry, int wm, int col_begin) {
    double* g = G + (int64_t)(col_begin + blockIdx.x) * F_LW * F_LW;
    for (int e = threadIdx.x; e < wm * wm; e += blockDim.x) {
        const int r = e / wm, c = e % wm;
        if (r >= ry || c >= ry) g[r * F_LW + c] = 0.0;
    }
}

// Hz[e] = M[zrow][e]  (z^T Y: the row of Y^T Y that belongs to the solved observation column)
__global__ void hz_from_M_kernel(const double* __restrict__ M, int ldm, int zrow, int cols, double* __restrict__ Hz) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < cols) Hz[e] = M[(int64_t)zrow * ldm + e];
}

}  // namespace mfgp

using namespace mfgp;

// ---- host side -------------------------------------------------------------------------------------------------------------
static inline int64_t round_up(int64_t v, int64_t m) { return (v + m - 1) / m * m; }

static inline int64_t imax(int64_t a, int64_t b) { return a > b ? a : b; }
constexpr int MR_MAXSPLIT = 8;       // most K ranges of the Y^T Y product

extern "C" int64_t mfgp_factored_workspace_bytes(int64_t npad, int64_t ncols, int64_t ny, int64_t rxL, int64_t ryL, int64_t rxH,
                                                 int64_t ryH, int64_t chunk_cols) {
    const int64_t rx = imax(rxL, rxH), ry = imax(ryL, ryH), kp = round_up(rx, 4);
    const int64_t ncp = round_up(ncols, 64), ch = round_up(chunk_cols, 64);
    int64_t d = 0;
    d += ny * 64 + npad + ry * kp;                             // Uy, solved z, Hz
    d += (rxL + ryL + rxH + ryH) * npad;                       // coefficient tables of both kernel parts
    const int64_t Rp = round_up(ry * kp + 1, 64);
    d += 2 * npad * Rp;                                        // B and Y (merged over the parts; room for the observation column)
    d += ncp * kp;                                             // Ux
    const int64_t direct = ch * npad * ry;                     // Y' of one chunk (direct route)
    const int64_t gram = (MR_MAXSPLIT + 1) * Rp * Rp + ncp * F_LW * F_LW;      // M = Y^T Y, its split-K partials, G'(ix)
    d += direct > gram ? direct : gram;
    return d * 8 + 4096;
}

// number of right-hand-side columns of the fused fit (mfgp_cholesky_solve): [B (ry * kpad columns) | y - mean | zero padding
// up to the next multiple of 64]
extern "C" int64_t mfgp_factored_rhs_cols(int64_t rxL, int64_t ryL, int64_t rxH, int64_t ryH) {
    return round_up(imax(ryL, ryH) * round_up(imax(rxL, rxH), 4) + 1, 64);
}

// Columns of the right-hand-side matrix for a truncated layout (kx[l] x terms kept for y term l, see FTrunc): sum kx + the
// observation column, padded to a multiple of 64.
extern "C" int64_t mfgp_factored_rhs_cols_trunc(int64_t ry, const int32_t* kx) {
    if (!kx || ry <= 0 || ry > F_MAXR) return 0;
    int64_t c = 0;
    for (int64_t l = 0; l < ry; l++) c += kx[l];
    return round_up(c + 1, 64);
}

namespace {
struct FGeom {
    const double* ux; int64_t nx; const double* uy; int64_t ny; int64_t ix0, ncols;
    const double* Xt; int64_t NL, NH, npad;
    const mfgp_params* p;
    int64_t rxL, ryL, rxH, ryH;
    double xlo, xhi, ylo, yhi;
    int64_t chunk;
};
struct FTab { int rx, ry; double inv_l; double* Cx; double* Cy; bool lofi; };
struct FLayout {
    FTab tabs[2]; int ntabs;         // coefficient tables per kernel part
    FPart parts[1]; int nparts;      // ONE merged expansion (rx = max, ry = max)
    double* Uy; double* zbuf; int64_t ncp, chunk; bool multi;
    FTrunc tr; bool truncated;       // column layout of the right-hand sides (uniform unless f_set_trunc was given a table)
};

// kx_host (optional, ry entries: x terms kept for y term l; multiples of 4 in [4, kpad]) -> column layout.  Returns false
// for an invalid table.
bool f_set_trunc(FLayout& L, const int32_t* kx_host) {
    const FPart& f = L.parts[0];
    FTrunc& t = L.tr;
    t.ry = f.ry;
    L.truncated = kx_host != nullptr;
    int o = 0;
    for (int l = 0; l < f.ry; l++) {
        const int k = kx_host ? kx_host[l] : f.kpad;
        if (k < 4 || k > f.kpad || (k & 3)) return false;
        t.off[l] = (short)o; t.kx[l] = (short)k;
        o += k;
    }
    for (int l = f.ry; l < F_MAXR; l++) { t.off[l] = (short)o; t.kx[l] = 0; }
    t.off[F_MAXR] = (short)o;
    t.cols = o;
    return true;
}

int f_validate(const FGeom& g, void* work, int64_t work_bytes) {
    if (!g.ux || !g.uy || !g.Xt || !g.p || !work) return MFGP_ERR_INVALID;
    const int64_t N = g.NL + g.NH;
    if (N <= 0 || g.npad < N || g.npad % MFGP_TILE || g.ncols <= 0 || g.ix0 < 0 || g.ix0 + g.ncols > g.nx || g.ny <= 0) return MFGP_ERR_INVALID;
    const bool multi = g.p->multi != 0;
    if (!multi && (g.rxL || g.ryL || g.NL)) return MFGP_ERR_INVALID;
    if (g.rxH <= 0 || g.ryH <= 0 || g.rxH > F_MAXR || g.ryH > F_MAXR || g.rxL > F_MAXR || g.ryL > F_MAXR || (g.ryL % 4) || (g.ryH % 4))
        return MFGP_ERR_INVALID;
    if (multi && (g.rxL <= 0 || g.ryL <= 0)) return MFGP_ERR_INVALID;
    if (!(g.xhi > g.xlo) || !(g.yhi > g.ylo) || g.chunk <= 0) return MFGP_ERR_INVALID;
    if (work_bytes < mfgp_factored_workspace_bytes(g.npad, g.ncols, g.ny, g.rxL, g.ryL, g.rxH, g.ryH, g.chunk)) return MFGP_ERR_INVALID;
    return MFGP_OK;
}

void f_carve(const FGeom& g, void* work, FLayout& L) {
    L.multi = g.p->multi != 0;
    L.ncp = round_up(g.ncols, 64); L.chunk = round_up(g.chunk, 64);
    double* wp = static_cast<double*>(work);
    auto carve = [&](int64_t n) { double* r = wp; wp += n; return r; };
    L.Uy = carve(g.ny * 64);
    L.zbuf = carve(g.npad);
    L.ntabs = 0;
    auto add_tab = [&](int rx, int ry, double l, bool lofi) {
        FTab& t = L.tabs[L.ntabs++];
        t.rx = rx; t.ry = ry; t.inv_l = 1.0 / l; t.lofi = lofi;
        t.Cx = carve((int64_t)rx * g.npad); t.Cy = carve((int64_t)ry * g.npad);
    };
    if (L.multi) add_tab((int)g.rxL, (int)g.ryL, g.p->l_L, true);
    add_tab((int)g.rxH, (int)g.ryH, g.p->l_H, false);
    FPart& f = L.parts[0];
    L.nparts = 1;
    f.rx = (int)imax(g.rxL, g.rxH); f.ry = (int)imax(g.ryL, g.ryH); f.kpad = (int)round_up(f.rx, 4); f.loff = 0; f.inv_l = 0.0;
    f.Cx = f.Cy = nullptr;
    {
        const int64_t Rp = round_up((int64_t)f.ry * f.kpad + 1, 64);         // [B | y - mean | 0 ...] / [Y | z | 0 ...] fit as well
        f.B = carve(g.npad * Rp); f.Y = carve(g.npad * Rp);
    }
    f.Ux = carve(L.ncp * f.kpad);
    {       // one region serves either route of steps 4 + 5: Y' of a chunk (direct) or M, its partials and G'(ix) (Gram route)
        const int64_t Rp = round_up((int64_t)f.ry * f.kpad + 1, 64);
        const int64_t direct = L.chunk * g.npad * f.ry;
        const int64_t gram = (MR_MAXSPLIT + 1) * Rp * Rp + L.ncp * F_LW * F_LW;
        f.Yp = carve(direct > gram ? direct : gram);
    }
    f.Hz = carve((int64_t)f.ry * f.kpad);
    f_set_trunc(L, nullptr);
}

// steps 1 + 2: tables of both kernel parts, basis tables, then the merged B either into the part's own buffer
// (Ball == nullptr) or into the leading columns of Ball
int f_tables_and_B(const FGeom& g, FLayout& L, double* Ball, int64_t ldB, cudaStream_t st) {
    const DevParams dp = make_dev_params(*g.p);
    const int64_t N = g.NL + g.NH, npad = g.npad;
    FPart& f = L.parts[0];
    MFGP_CUDA_CHECK(cudaMemsetAsync(L.Uy, 0, sizeof(double) * g.ny * 64, st));
    MFGP_CUDA_CHECK(cudaMemsetAsync(f.Ux, 0, sizeof(double) * L.ncp * f.kpad, st));
    cheb_basis_kernel<<<(unsigned)((L.ncp + 127) / 128), 128, 0, st>>>(g.ux, (int)g.ix0, (int)g.ncols, (int)L.ncp, g.xlo, g.xhi, f.rx, f.kpad,
                                                                    0, f.Ux);
    MFGP_LAUNCH_CHECK();
    cheb_basis_kernel<<<(unsigned)((g.ny + 127) / 128), 128, 0, st>>>(g.uy, 0, (int)g.ny, (int)g.ny, g.ylo, g.yhi, f.ry, 64, 0, L.Uy);
    MFGP_LAUNCH_CHECK();
    BTab bt[2] = {};
    ChebJobs jobs = {};
    for (int ti = 0; ti < L.ntabs; ti++) {
        FTab& t = L.tabs[ti];
        jobs.j[2 * ti] = ChebJob{0, t.rx, g.xlo, g.xhi, t.inv_l, t.Cx};
        jobs.j[2 * ti + 1] = ChebJob{1, t.ry, g.ylo, g.yhi, t.inv_l, t.Cy};
        // lofi part: rho s_L (lofi columns) / rho^2 s_L (hifi columns); hifi part: 0 / s_H  (gaussian_process.py:426-429)
        bt[ti] = BTab{t.Cx, t.Cy, t.rx, t.ry, t.lofi ? dp.rho * dp.s_L : 0.0, t.lofi ? dp.rho2 * dp.s_L : dp.s_H};
    }
    {
        dim3 cgrid((unsigned)((npad + CHEB_PTS - 1) / CHEB_PTS), (unsigned)(2 * L.ntabs));
        cheb_coef_kernel<<<cgrid, 256, 0, st>>>(g.Xt, (int)N, (int)npad, jobs);
        MFGP_LAUNCH_CHECK();
    }
    const int cols = L.tr.cols;                // ry * kpad, or fewer with a truncated layout (fused-fit form only)
    dim3 bgrid((unsigned)((cols + 127) / 128), (unsigned)npad);
    build_B_merged_kernel<<<bgrid, 128, 0, st>>>(bt[0], bt[1], L.ntabs, (int)npad, (int)N, (int)g.NL, L.tr, Ball ? Ball : f.B,
                                                Ball ? ldB : (int64_t)cols);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

// steps 4 - 6 from `rows` rows of Y_P (parts[].Y; all npad rows, or only the appended block) and their whitened
// observations z.  Gstore / Hz_store (optional) keep G'(ix) and z^T Y across calls; accumulate = 1 adds to them.
int f_tail(const FGeom& g, FLayout& L, const double* z, int64_t rows, double* Gstore, double* Hz_store, int accumulate,
           double* mu, double* var, double* qred, cudaStream_t st) {
    const DevParams dp = make_dev_params(*g.p);
    const int64_t npad = rows;
    const int ry0 = L.parts[0].ry;
    const bool narrow = ry0 <= 40;          // padded width of the y expansion: 40 (15 Gram tiles) or 64 (36)
    const int wm = narrow ? 40 : 64;
    const int pitch = (ry0 % 8 == 4) ? ry0 : ry0 + 4;
    int nstage = (int)(73728 / (G_ROWS * pitch * 8));
    nstage = nstage < 2 ? 2 : (nstage > G_MAXSTAGE ? G_MAXSTAGE : nstage);
    const size_t gsmem = sizeof(double) * ((size_t)nstage * G_ROWS * pitch + g_ring_slack(wm, pitch) + wm * (wm + 2) + 2 * F_LW) +
                         8 * G_MAXSTAGE + 64;
    const char* pe = getenv("MFGP_DEBUG_POISON_SMEM");          // read per call, as MFGP_GRAM: tests switch it inside one process
    const int poison = pe && std::strcmp(pe, "1") == 0;
    MFGP_CUDA_CHECK(cudaFuncSetAttribute(gram_eval_kernel<40>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gsmem));
    MFGP_CUDA_CHECK(cudaFuncSetAttribute(gram_eval_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gsmem));
    int64_t hoff = 0;
    for (int pi = 0; pi < L.nparts; pi++) {
        FPart& f = L.parts[pi];
        const int cols = f.ry * f.kpad;
        if (Hz_store) f.Hz = Hz_store + hoff;          // persistent across calls (incremental path)
        // partials go to the (not yet written) step-4 buffer: HZ_SPLIT x cols doubles << one column of Y'
        hz_partial_kernel<<<dim3((unsigned)((cols + 31) / 32), HZ_SPLIT), 256, 0, st>>>(f.Y, z, (int)npad, cols, f.Yp);
        MFGP_LAUNCH_CHECK();
        hz_reduce_kernel<<<(cols + 127) / 128, 128, 0, st>>>(f.Yp, cols, f.Hz, accumulate);
        MFGP_LAUNCH_CHECK();
        hoff += cols;
    }
    for (int64_t c0 = 0; c0 < g.ncols; c0 += L.chunk) {
        const int64_t cc = (g.ncols - c0 < L.chunk) ? g.ncols - c0 : L.chunk;
        const int64_t ccp = round_up(cc, 64);
        for (int pi = 0; pi < L.nparts; pi++) {
            FPart& f = L.parts[pi];
            GemmArgs gm{};          // step 4: Y'[col][(n, l)] = sum_k Ux[col][k] Y[(n, l)][k]
            gm.A = f.Ux + c0 * f.kpad; gm.lda = f.kpad; gm.B = f.Y; gm.ldb = f.kpad; gm.C = f.Yp; gm.ldc = npad * (int64_t)f.ry;
            gm.M = (int)ccp; gm.N = (int)(npad * f.ry); gm.K = f.kpad; gm.alpha = 1.0; gm.beta = 0.0; gm.mode = GEMM_GENERAL;
            int rc = launch_gemm(gm, true, 1, st);
            if (rc) return rc;
        }
        GramArgs ga;
        ga.YpL = nullptr; ga.YpH = L.parts[0].Yp;          // one merged expansion: the "L" slot of the kernel stays empty
        ga.ryL = 0; ga.ryH = L.parts[0].ry;
        ga.npad = (int)npad; ga.Uy = L.Uy; ga.ny = (int)g.ny; ga.col_begin = (int)c0;
        ga.Gstore = Gstore; ga.accumulate = accumulate;
        ga.skip_eval = Gstore != nullptr;              // with a store: the DMMA evaluation kernel below reads G'(ix) from it
        ga.HzL = nullptr; ga.HzH = L.parts[0].Hz;
        ga.UxL = nullptr; ga.UxH = L.parts[0].Ux + c0 * L.parts[0].kpad;
        ga.kL = 0; ga.kH = L.parts[0].kpad;
        ga.mean = dp.mean_H; ga.k0 = dp.k0; ga.mu = mu; ga.var = var; ga.qred = qred;
        ga.pitch = pitch; ga.nstage = nstage; ga.poison = poison;
        if (narrow) gram_eval_kernel<40><<<(unsigned)cc, 128, gsmem, st>>>(ga);
        else gram_eval_kernel<64><<<(unsigned)cc, 128, gsmem, st>>>(ga);
        MFGP_LAUNCH_CHECK();
    }
    if (Gstore) {            // step 6 for every column off the stored Gram matrices (tensor pipe; uniform column layout)
        FPart& f = L.parts[0];
        if (narrow)
            geval_mma_kernel<40><<<(unsigned)g.ncols, 128, 0, st>>>(Gstore, f.Hz, f.Ux, f.kpad, f.ry, L.tr, L.Uy, (int)g.ny, dp.mean_H, dp.k0, mu, var, qred);
        else
            geval_mma_kernel<64><<<(unsigned)g.ncols, 128, 0, st>>>(Gstore, f.Hz, f.Ux, f.kpad, f.ry, L.tr, L.Uy, (int)g.ny, dp.mean_H, dp.k0, mu, var, qred);
        MFGP_LAUNCH_CHECK();
    }
    return MFGP_OK;
}
// 0: cost model decides, 1: always the direct route (Y' + per-column Gram over the training rows), 2: always the Gram route
int gram_route_override() {          // read per call: tests and A/B timings switch it inside one process
    const char* e = getenv("MFGP_GRAM");
    if (!e) return 0;
    return std::strcmp(e, "direct") == 0 ? 1 : (std::strcmp(e, "m") == 0 ? 2 : 0);
}

// steps 4 - 6 by the Gram route from the solved right-hand sides Yall[npad][ldY] (columns [0, ry * kpad): Y, column
// ry * kpad: z, then zero padding up to ldY, a multiple of 64).  Returns MFGP_OK, or 1 when the direct route is cheaper.
// route of steps 4 + 5 for solved right-hand sides with row stride ldY: true = Gram route (cost model, MFGP_GRAM overrides)
bool f_gram_wanted(const FGeom& g, const FLayout& L, int64_t ldY) {
    const FPart& f = L.parts[0];
    const int64_t npad = g.npad, cols = L.tr.cols;
    const int wm = f.ry <= 40 ? 40 : 64;
    const int nt8 = (f.kpad + 7) / 8;
    if (ldY % 64 || ldY < cols + 1 || nt8 > 8) return false;
    const int ov = gram_route_override();
    if (L.truncated) return ov != 1;       // the truncated layout exists for this route only (MFGP_GRAM=direct: caller falls back)
    const double direct = (double)g.ncols * npad * cols + 0.6 * g.ncols * npad * wm * wm;
    const double gram = 0.5 * npad * (double)ldY * ldY + (double)round_up(g.ncols, 64) * (f.ry * (f.ry + 1) / 2) * 64.0 * nt8 * nt8;
    return !(ov == 1 || (ov == 0 && gram >= direct));
}

// Largest row stride of the solved right-hand sides: f_tail_gram keeps M, its split-K partials and G'(ix) at offsets 0, ldY^2 and
// (MR_MAXSPLIT + 1) ldY^2 of the step-4 region, which f_carve sizes for the uniform column count Rp.
int64_t f_max_ldY(const FLayout& L) { return round_up((int64_t)L.parts[0].ry * L.parts[0].kpad + 1, 64); }

// m_ready: M (f.Yp, row stride ldY) already holds Y^T Y (mfgp_cholesky_solve_gram wrote it)
int f_tail_gram(const FGeom& g, FLayout& L, const double* Yall, int64_t ldY, double* Gstore, double* Hz_store, double* mu,
                double* var, double* qred, bool m_ready, cudaStream_t st) {
    FPart& f = L.parts[0];
    const int64_t npad = g.npad, cols = L.tr.cols;
    const int wm = f.ry <= 40 ? 40 : 64;
    const int nt8 = (f.kpad + 7) / 8;
    if (!f_gram_wanted(g, L, ldY)) return (m_ready || L.truncated) ? MFGP_ERR_INVALID : 1;
    if (L.truncated && (Gstore || Hz_store)) return MFGP_ERR_INVALID;      // the incremental stores keep the uniform layout
    const DevParams dp = make_dev_params(*g.p);
    // M and its partial sums live where the direct route keeps Y'
    double* M = f.Yp;
    double* part = M + ldY * ldY;
    double* Gbuf = Gstore ? Gstore : part + (int64_t)MR_MAXSPLIT * ldY * ldY;
    if (!m_ready) {
        const int ntile = (int)(ldY / 64), tiles = ntile * (ntile + 1) / 2;
        int nsplit = 740 / tiles;                       // ~5 CTAs of the tile kernel per SM: one resident wave
        if (nsplit < 1) nsplit = 1;
        if (nsplit > MR_MAXSPLIT) nsplit = MR_MAXSPLIT;
        if (nsplit > npad / 128) nsplit = (int)imax(1, npad / 128);
        const int kchunk = (int)((npad / 64 + nsplit - 1) / nsplit) * 64;
        nsplit = (int)((npad + kchunk - 1) / kchunk);
        GemmArgs gm{};
        gm.A = Yall; gm.lda = ldY; gm.B = Yall; gm.ldb = ldY; gm.C = nsplit > 1 ? part : M; gm.ldc = ldY; gm.strideC = ldY * ldY;
        gm.M = (int)ldY; gm.N = (int)ldY; gm.K = (int)npad; gm.alpha = 1.0; gm.beta = 0.0; gm.mode = GEMM_SYRK_LOWER;
        gm.kchunk = nsplit > 1 ? kchunk : 0;
        int rc = launch_syrk_ata(gm, nsplit, st);
        if (rc) return rc;
        if (nsplit > 1) {
            syrk_reduce_lower_kernel<<<dim3((unsigned)((ldY + 127) / 128), (unsigned)ldY), 128, 0, st>>>(part, nsplit, ldY * ldY, (int)ldY, M);
            MFGP_LAUNCH_CHECK();
        }
    }
    if (Hz_store) f.Hz = Hz_store;
    hz_from_M_kernel<<<(unsigned)((cols + 127) / 128), 128, 0, st>>>(M, (int)ldY, (int)cols, (int)cols, f.Hz);
    MFGP_LAUNCH_CHECK();
    QformArgs qa;
    qa.M = M; qa.ldm = (int)ldY; qa.Ux = f.Ux; qa.kpad = f.kpad; qa.tr = L.tr; qa.ry = f.ry; qa.ncols = (int)g.ncols; qa.G = Gbuf; qa.col_begin = 0;
    const int npairs = f.ry * (f.ry + 1) / 2;
    const int cblocks = (int)((g.ncols + 63) / 64);
    int groups = (148 * 3) / cblocks;                            // 3 CTAs fit an SM (157 registers x 128 threads): one resident wave
    if (groups < 1) groups = 1;
    if (groups > npairs) groups = npairs;
    qa.pairs_per_cta = (npairs + groups - 1) / groups;
    groups = (npairs + qa.pairs_per_cta - 1) / qa.pairs_per_cta;
    const dim3 qgrid((unsigned)cblocks, (unsigned)groups);
    switch (nt8) {
        case 1: qform_kernel<1, true><<<qgrid, 128, 0, st>>>(qa); break;
        case 2: qform_kernel<2, true><<<qgrid, 128, 0, st>>>(qa); break;
        case 3: qform_kernel<3, true><<<qgrid, 128, 0, st>>>(qa); break;
        case 4: qform_kernel<4, true><<<qgrid, 128, 0, st>>>(qa); break;
        case 5: qform_kernel<5, true><<<qgrid, 128, 0, st>>>(qa); break;
        case 6: qform_kernel<6, true><<<qgrid, 128, 0, st>>>(qa); break;
        case 7: qform_kernel<7, false><<<qgrid, 128, 0, st>>>(qa); break;
        default: qform_kernel<8, false><<<qgrid, 128, 0, st>>>(qa); break;
    }
    MFGP_LAUNCH_CHECK();
    // step 6 (and h'(ix)): G' comes from the buffer, nothing else to add
    static const bool eval_fma = [] { const char* e = getenv("MFGP_GEVAL"); return e && std::strcmp(e, "fma") == 0; }();
    if (eval_fma) {
        if (wm == 40)
            geval_kernel<40, 2><<<(unsigned)g.ncols, 256, 0, st>>>(Gbuf, f.Hz, f.Ux, f.kpad, f.ry, L.tr, L.Uy, (int)g.ny, dp.mean_H, dp.k0, mu, var, qred);
        else
            geval_kernel<64, 1><<<(unsigned)g.ncols, 256, 0, st>>>(Gbuf, f.Hz, f.Ux, f.kpad, f.ry, L.tr, L.Uy, (int)g.ny, dp.mean_H, dp.k0, mu, var, qred);
    } else if (wm == 40) {
        geval_mma_kernel<40><<<(unsigned)g.ncols, 128, 0, st>>>(Gbuf, f.Hz, f.Ux, f.kpad, f.ry, L.tr, L.Uy, (int)g.ny, dp.mean_H, dp.k0, mu, var, qred);
    } else {
        geval_mma_kernel<64><<<(unsigned)g.ncols, 128, 0, st>>>(Gbuf, f.Hz, f.Ux, f.kpad, f.ry, L.tr, L.Uy, (int)g.ny, dp.mean_H, dp.k0, mu, var, qred);
    }
    MFGP_LAUNCH_CHECK();
    if (Gstore && f.ry < wm) {        // the incremental update adds into the padded wm x wm block of the store: its padding must be finite
        gpad_zero_kernel<<<(unsigned)g.ncols, 128, 0, st>>>(Gbuf, f.ry, wm, 0);
        MFGP_LAUNCH_CHECK();
    }
    return MFGP_OK;
}
}  // namespace

// Factored posterior for the whole columns [ix0, ix0 + ncols) of the tensor-product grid ux[nx] x uy[ny] (x-major); outputs
// are flat over those columns: index (ix - ix0) * ny + iy.  rx*/ry*: Chebyshev orders per axis and part (ryL, ryH multiples
// of 4, every order <= 64; rxL = ryL = 0 for a single-fidelity model) -- chosen by the caller so that the factor
// tables are reproduced to rounding (mfgp_coverage_b200/_engine.py: chebyshev_order).
// kx (optional, host): truncated column layout as in mfgp_factored_prepare_trunc; needs Gstore = Hz_store = NULL and takes the Gram
// route (MFGP_GRAM=direct falls back to the uniform layout).
extern "C" int mfgp_posterior_grid_factored_trunc(const double* ux, int64_t nx, const double* uy, int64_t ny, int64_t ix0, int64_t ncols,
                                                  const double* Xt, int64_t NL, int64_t NH, const double* W, int64_t npad, int64_t ldw,
                                                  const double* z, const mfgp_params* p_host, int64_t rxL, int64_t ryL, int64_t rxH,
                                                  int64_t ryH, double xlo, double xhi, double ylo, double yhi, int64_t chunk_cols,
                                                  const int32_t* kx, double* mu, double* var, double* qred, double* Gstore,
                                                  double* Hz_store, void* work, int64_t work_bytes, void* stream) {
    if (!W || !z || !mu || !var || ldw < npad) return MFGP_ERR_INVALID;
    FGeom g{ux, nx, uy, ny, ix0, ncols, Xt, NL, NH, npad, p_host, rxL, ryL, rxH, ryH, xlo, xhi, ylo, yhi, chunk_cols};
    int rc = f_validate(g, work, work_bytes);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    FLayout L;
    f_carve(g, work, L);
    FPart& f0 = L.parts[0];
    if (kx && !Gstore && !Hz_store && gram_route_override() != 1) {
        if (!f_set_trunc(L, kx)) return MFGP_ERR_INVALID;
    }
    const int64_t cols0 = L.tr.cols, Rp = round_up(cols0 + 1, 64);
    if (!Gstore && !Hz_store && f_gram_wanted(g, L, Rp)) {
        // Gram route with a standing factor: Yall = W [B | 0] in the padded layout of the fused form (row stride Rp), z into its
        // observation column, then M = Yall^T Yall as a launch of its own and the quadratic forms / evaluation of f_tail_gram
        rc = f_tables_and_B(g, L, f0.B, Rp, st);
        if (rc) return rc;
        put_z_block_kernel<<<(unsigned)npad, (int)(Rp - cols0), 0, st>>>(z, (int)npad, f0.B, Rp, (int)cols0);     // (zeros: W 0 = 0)
        MFGP_LAUNCH_CHECK();
        GemmArgs gm{};
        gm.A = W; gm.lda = ldw; gm.B = f0.B; gm.ldb = Rp; gm.C = f0.Y; gm.ldc = Rp;
        gm.M = (int)npad; gm.N = (int)Rp; gm.K = (int)npad; gm.alpha = 1.0; gm.beta = 0.0; gm.mode = GEMM_A_LOWER;
        rc = launch_gemm(gm, false, 1, st);
        if (rc) return rc;
        put_z_block_kernel<<<(unsigned)npad, (int)(Rp - cols0), 0, st>>>(z, (int)npad, f0.Y, Rp, (int)cols0);
        MFGP_LAUNCH_CHECK();
        return f_tail_gram(g, L, f0.Y, Rp, nullptr, nullptr, mu, var, qred, false, st);
    }
    rc = f_tables_and_B(g, L, nullptr, 0, st);
    if (rc) return rc;
    for (int pi = 0; pi < L.nparts; pi++) {       // step 3: Y = W B  (W lower triangular: k < m0 + 64)
        FPart& f = L.parts[pi];
        GemmArgs gm{};
        gm.A = W; gm.lda = ldw; gm.B = f.B; gm.ldb = (int64_t)f.ry * f.kpad; gm.C = f.Y; gm.ldc = (int64_t)f.ry * f.kpad;
        gm.M = (int)npad; gm.N = f.ry * f.kpad; gm.K = (int)npad; gm.alpha = 1.0; gm.beta = 0.0; gm.mode = GEMM_A_LOWER;
        rc = launch_gemm(gm, false, 1, st);
        if (rc) return rc;
    }
    return f_tail(g, L, z, npad, Gstore, Hz_store, 0, mu, var, qred, st);
}

extern "C" int mfgp_posterior_grid_factored(const double* ux, int64_t nx, const double* uy, int64_t ny, int64_t ix0, int64_t ncols,
                                            const double* Xt, int64_t NL, int64_t NH, const double* W, int64_t npad, int64_t ldw,
                                            const double* z, const mfgp_params* p_host, int64_t rxL, int64_t ryL, int64_t rxH,
                                            int64_t ryH, double xlo, double xhi, double ylo, double yhi, int64_t chunk_cols,
                                            double* mu, double* var, double* qred, double* Gstore, double* Hz_store, void* work,
                                            int64_t work_bytes, void* stream) {
    return mfgp_posterior_grid_factored_trunc(ux, nx, uy, ny, ix0, ncols, Xt, NL, NH, W, npad, ldw, z, p_host, rxL, ryL, rxH, ryH, xlo, xhi,
                                              ylo, yhi, chunk_cols, nullptr, mu, var, qred, Gstore, Hz_store, work, work_bytes, stream);
}

// kx (optional, host, max(ryL, ryH) entries): truncated column layout -- per y term l only the first kx[l] x terms are kept
// (multiples of 4 in [4, round_up(max(rxL, rxH), 4)]); Ball then has mfgp_factored_rhs_cols_trunc(ry, kx) columns.  Only the
// Gram route of steps 4 + 5 reads that layout: pair it with mfgp_factored_gram_target / mfgp_posterior_grid_factored_solved_gram
// called with the same kx.
extern "C" int mfgp_factored_prepare_trunc(const double* ux, int64_t nx, const double* uy, int64_t ny, int64_t ix0, int64_t ncols,
                                           const double* Xt, const double* y, int64_t NL, int64_t NH, int64_t npad,
                                           const mfgp_params* p_host, int64_t rxL, int64_t ryL, int64_t rxH, int64_t ryH, double xlo,
                                           double xhi, double ylo, double yhi, int64_t chunk_cols, const int32_t* kx, double* Ball,
                                           int64_t ldB, void* work, int64_t work_bytes, void* stream) {
    if (!y || !Ball) return MFGP_ERR_INVALID;
    FGeom g{ux, nx, uy, ny, ix0, ncols, Xt, NL, NH, npad, p_host, rxL, ryL, rxH, ryH, xlo, xhi, ylo, yhi, chunk_cols};
    int rc = f_validate(g, work, work_bytes);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    FLayout L;
    f_carve(g, work, L);
    if (!f_set_trunc(L, kx)) return MFGP_ERR_INVALID;
    const int64_t zoff = L.tr.cols;                                          // the column right behind B; the rest is zero padding
    const int64_t R = round_up(zoff + 1, 64);
    if (ldB < R) return MFGP_ERR_INVALID;
    rc = f_tables_and_B(g, L, Ball, ldB, st);
    if (rc) return rc;
    build_z_block_kernel<<<(unsigned)npad, (int)(R - zoff), 0, st>>>(y, (int)npad, (int)(NL + NH), (int)NL, p_host->mean_L, p_host->mean_H,
                                                                     Ball + zoff, ldB);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

extern "C" int mfgp_factored_prepare(const double* ux, int64_t nx, const double* uy, int64_t ny, int64_t ix0, int64_t ncols,
                                     const double* Xt, const double* y, int64_t NL, int64_t NH, int64_t npad,
                                     const mfgp_params* p_host, int64_t rxL, int64_t ryL, int64_t rxH, int64_t ryH, double xlo,
                                     double xhi, double ylo, double yhi, int64_t chunk_cols, double* Ball, int64_t ldB, void* work,
                                     int64_t work_bytes, void* stream) {
    return mfgp_factored_prepare_trunc(ux, nx, uy, ny, ix0, ncols, Xt, y, NL, NH, npad, p_host, rxL, ryL, rxH, ryH, xlo, xhi, ylo, yhi,
                                       chunk_cols, nullptr, Ball, ldB, work, work_bytes, stream);
}

// Fused-fit form, part 2: Yall = L^-1 Ball (mfgp_cholesky_solve) -> steps 4 - 6.  `work` must be the workspace that
// mfgp_factored_prepare filled (it holds the basis tables); z_out (optional) receives the whitened observations z[npad].
namespace {
int f_solved_impl(const FGeom& g, const int32_t* kx, const double* Yall, int64_t ldY, double* z_out, double* mu, double* var,
                  double* qred, double* Gstore, double* Hz_store, void* work, int64_t work_bytes, bool m_ready, cudaStream_t st) {
    if (!Yall || !mu || !var) return MFGP_ERR_INVALID;
    int rc = f_validate(g, work, work_bytes);
    if (rc) return rc;
    FLayout L;
    f_carve(g, work, L);
    if (!f_set_trunc(L, kx)) return MFGP_ERR_INVALID;
    const int64_t npad = g.npad;
    const int64_t zoff = L.tr.cols;
    if (ldY < round_up(zoff + 1, 64) || ldY > f_max_ldY(L)) return MFGP_ERR_INVALID;
    unpack_z_kernel<<<(unsigned)((npad + 255) / 256), 256, 0, st>>>(Yall, ldY, (int)zoff, (int)npad, L.zbuf);
    MFGP_LAUNCH_CHECK();
    if (z_out) MFGP_CUDA_CHECK(cudaMemcpyAsync(z_out, L.zbuf, sizeof(double) * npad, cudaMemcpyDeviceToDevice, st));
    rc = f_tail_gram(g, L, Yall, ldY, Gstore, Hz_store, mu, var, qred, m_ready, st);      // Gram route: M = Y^T Y, then quadratic forms
    if (rc <= 0) return rc;
    int64_t off = 0;                                                             // direct route (cheaper for few training rows)
    for (int pi = 0; pi < L.nparts; pi++) {
        FPart& f = L.parts[pi];
        const int cols = f.ry * f.kpad;
        dim3 ug((unsigned)((cols + 255) / 256), (unsigned)npad);
        unpack_Y_kernel<<<ug, 256, 0, st>>>(Yall, ldY, (int)off, cols, f.Y);
        MFGP_LAUNCH_CHECK();
        off += cols;
    }
    return f_tail(g, L, L.zbuf, npad, Gstore, Hz_store, 0, mu, var, qred, st);
}
}  // namespace

extern "C" int mfgp_posterior_grid_factored_solved(const double* ux, int64_t nx, const double* uy, int64_t ny, int64_t ix0,
                                                   int64_t ncols, const double* Xt, int64_t NL, int64_t NH, int64_t npad,
                                                   const mfgp_params* p_host, int64_t rxL, int64_t ryL, int64_t rxH, int64_t ryH,
                                                   double xlo, double xhi, double ylo, double yhi, int64_t chunk_cols,
                                                   const double* Yall, int64_t ldY, double* z_out, double* mu, double* var,
                                                   double* qred, double* Gstore, double* Hz_store, void* work,
                                                   int64_t work_bytes, void* stream) {
    FGeom g{ux, nx, uy, ny, ix0, ncols, Xt, NL, NH, npad, p_host, rxL, ryL, rxH, ryH, xlo, xhi, ylo, yhi, chunk_cols};
    return f_solved_impl(g, nullptr, Yall, ldY, z_out, mu, var, qred, Gstore, Hz_store, work, work_bytes, false,
                         static_cast<cudaStream_t>(stream));
}

// Where mfgp_cholesky_solve_gram must leave M = Yall^T Yall (row stride ldY) for the posterior call that follows: a pointer
// into `work` (the buffer of mfgp_factored_prepare), or NULL when steps 4 + 5 will take the direct route for this geometry
// (few training rows; MFGP_GRAM=direct) -- then call plain mfgp_cholesky_solve and mfgp_posterior_grid_factored_solved.
// kx: the truncated column layout given to mfgp_factored_prepare_trunc, or NULL (uniform).
extern "C" double* mfgp_factored_gram_target(int64_t nx, int64_t ny, int64_t ix0, int64_t ncols, int64_t NL, int64_t NH, int64_t npad,
                                             const mfgp_params* p_host, int64_t rxL, int64_t ryL, int64_t rxH, int64_t ryH,
                                             int64_t chunk_cols, const int32_t* kx, int64_t ldY, void* work, int64_t work_bytes) {
    if (!p_host || !work) return nullptr;
    if (work_bytes < mfgp_factored_workspace_bytes(npad, ncols, ny, rxL, ryL, rxH, ryH, chunk_cols)) return nullptr;
    FGeom g{nullptr, nx, nullptr, ny, ix0, ncols, nullptr, NL, NH, npad, p_host, rxL, ryL, rxH, ryH, 0.0, 1.0, 0.0, 1.0, chunk_cols};
    FLayout L;
    f_carve(g, work, L);
    if (!f_set_trunc(L, kx) || ldY < round_up((int64_t)L.tr.cols + 1, 64) || ldY > f_max_ldY(L)) return nullptr;
    return f_gram_wanted(g, L, ldY) ? L.parts[0].Yp : nullptr;
}

// mfgp_posterior_grid_factored_solved after mfgp_cholesky_solve_gram: M = Yall^T Yall is already standing at
// mfgp_factored_gram_target(...) inside `work`, so the symmetric product and its reduction are skipped.
extern "C" int mfgp_posterior_grid_factored_solved_gram(const double* ux, int64_t nx, const double* uy, int64_t ny, int64_t ix0,
                                                        int64_t ncols, const double* Xt, int64_t NL, int64_t NH, int64_t npad,
                                                        const mfgp_params* p_host, int64_t rxL, int64_t ryL, int64_t rxH,
                                                        int64_t ryH, double xlo, double xhi, double ylo, double yhi,
                                                        int64_t chunk_cols, const int32_t* kx, const double* Yall, int64_t ldY,
                                                        double* z_out, double* mu, double* var, double* qred, double* Gstore,
                                                        double* Hz_store, void* work, int64_t work_bytes, void* stream) {
    FGeom g{ux, nx, uy, ny, ix0, ncols, Xt, NL, NH, npad, p_host, rxL, ryL, rxH, ryH, xlo, xhi, ylo, yhi, chunk_cols};
    return f_solved_impl(g, kx, Yall, ldY, z_out, mu, var, qred, Gstore, Hz_store, work, work_bytes, true,
                         static_cast<cudaStream_t>(stream));
}

// Incremental form (after mfgp_cholesky_append): rows [row_lo, NL+NH) of the training set are new since Gstore / Hz_store
// (and mu / var) were last brought up to date by one of the full forms above with the same geometry and orders.  Only the
// new rows of Y = W B are formed (one split-K tile product over the 64-row blocks that hold them), contracted with T_k(tx),
// and added to the stored per-column Gram matrices; then every grid point is re-evaluated from G'(ix):
//   G'(ix) += Y'_new(ix)^T Y'_new(ix),   z^T Y += z_new^T Y_new,   var = k0 - uy^T G' uy,   mu = mean + (Ux(ix) . z^T Y) . uy.
// Cost at c4 with 64 new samples: ~7e8 MAC + the evaluation pass, against 4.2e10 MAC for the full factored form.
extern "C" int mfgp_posterior_grid_factored_update(const double* ux, int64_t nx, const double* uy, int64_t ny, int64_t ix0,
                                                   int64_t ncols, const double* Xt, int64_t NL, int64_t NH, int64_t row_lo,
                                                   const double* W, int64_t npad, int64_t ldw, const double* z,
                                                   const mfgp_params* p_host, int64_t rxL, int64_t ryL, int64_t rxH, int64_t ryH,
                                                   double xlo, double xhi, double ylo, double yhi, int64_t chunk_cols, double* mu,
                                                   double* var, double* qred, double* Gstore, double* Hz_store, void* work,
                                                   int64_t work_bytes, void* stream) {
    if (!W || !z || !mu || !var || !Gstore || !Hz_store || ldw < npad || row_lo <= 0 || row_lo >= NL + NH) return MFGP_ERR_INVALID;
    FGeom g{ux, nx, uy, ny, ix0, ncols, Xt, NL, NH, npad, p_host, rxL, ryL, rxH, ryH, xlo, xhi, ylo, yhi, chunk_cols};
    int rc = f_validate(g, work, work_bytes);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    FLayout L;
    f_carve(g, work, L);
    rc = f_tables_and_B(g, L, nullptr, 0, st);            // all rows of B: the new rows of Y contract over every training point
    if (rc) return rc;
    const int64_t rb = row_lo / 64 * 64;                  // first 64-row block that holds a new row
    const int64_t M = npad - rb;
    for (int pi = 0; pi < L.nparts; pi++) {
        FPart& f = L.parts[pi];
        const int64_t cols = (int64_t)f.ry * f.kpad;
        // Y_new = W[rb:npad, :] B, split over K; partial products parked in the (unused) tail of the part's Y buffer
        int nsplit = (int)(npad / 512);
        if (nsplit < 1) nsplit = 1;
        if (nsplit > 16) nsplit = 16;
        while (nsplit > 1 && (int64_t)(nsplit + 1) * M * cols > npad * cols) nsplit--;       // must fit behind Y_new in f.Y
        const int kchunk = (int)((npad / 64 + nsplit - 1) / nsplit) * 64;
        nsplit = (int)((npad + kchunk - 1) / kchunk);
        double* Ynew = f.Y;
        double* part = f.Y + M * cols;
        if (nsplit > 1) {
            GemmArgs gm{};
            gm.A = W + rb * ldw; gm.lda = ldw; gm.B = f.B; gm.ldb = cols; gm.C = part; gm.ldc = cols; gm.strideC = M * cols;
            gm.M = (int)M; gm.N = (int)cols; gm.K = (int)npad; gm.alpha = 1.0; gm.beta = 0.0; gm.mode = GEMM_GENERAL; gm.kchunk = kchunk;
            rc = launch_gemm(gm, false, nsplit, st);
            if (rc) return rc;
            dim3 rgrid((unsigned)((cols + 127) / 128), (unsigned)M);
            splitk_reduce_kernel<<<rgrid, 128, 0, st>>>(part, nsplit, M * cols, (int)cols, Ynew, cols, (int)M, (int)cols, 1.0, 0.0);
            MFGP_LAUNCH_CHECK();
        } else {
            GemmArgs gm{};
            gm.A = W + rb * ldw; gm.lda = ldw; gm.B = f.B; gm.ldb = cols; gm.C = Ynew; gm.ldc = cols;
            gm.M = (int)M; gm.N = (int)cols; gm.K = (int)npad; gm.alpha = 1.0; gm.beta = 0.0; gm.mode = GEMM_GENERAL;
            rc = launch_gemm(gm, false, 1, st);
            if (rc) return rc;
        }
        if (row_lo > rb) {        // rows [rb, row_lo) of the first block are old: already inside the stored G' and z^T Y
            const int64_t nz = (row_lo - rb) * cols;
            zero_rows_kernel<<<(unsigned)((nz + 255) / 256), 256, 0, st>>>(Ynew, cols, (int)(row_lo - rb));
            MFGP_LAUNCH_CHECK();
        }
    }
    // steps 4 - 6 on the M new rows only (g.npad stays the full size for the table shapes; f_tail takes the row count)
    return f_tail(g, L, z + rb, M, Gstore, Hz_store, 1, mu, var, qred, st);
}
