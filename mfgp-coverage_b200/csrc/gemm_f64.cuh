// Batched fp64 tile GEMM on DMMA for the factorisation kernels (Cholesky panel solve, SYRK trailing update,
// block-doubling triangular inverse) and the products of the factored posterior.  M is a multiple of 64 (buffers are padded
// to MFGP_TILE); N may end inside a tile (multiple of 2: loads zero-filled, stores predicated) and K inside a slab (multiple
// of 2: zero-filled).  C[M,N] = alpha * A[M,K] * op(B) + beta * C, row-major, one 64x64 C tile per 128-thread CTA
// (2x2 warps, 32x32 per warp = 4x4 DMMA 8x8 tiles), K streamed in 16-wide cp.async double-buffered slabs.
#pragma once
#include "common.cuh"

namespace mfgp {

enum GemmMode : int {
    GEMM_GENERAL = 0,
    GEMM_SYRK_LOWER = 1,   // only C tiles with row-tile >= col-tile are computed (B must be A, B_TRANS)
    GEMM_A_LOWER = 2,      // A[M,K=M] lower triangular: k < m0 + 64
    GEMM_B_LOWER = 3,      // B[K=N,N] (not transposed) lower triangular: k >= n0
    GEMM_BT_LOWER = 4,     // B[N,K=N] (transposed operand) lower triangular: k < n0 + 64
    GEMM_SYRK_LOWER_AUPPER = 5,  // C = A A^T lower tiles with A[M,K=M] UPPER triangular: k >= m0 (>= n0)
    GEMM_AT_LOWER = 6            // A_TRANS operand given as a lower triangular [K=M][M] matrix (op(A) upper): k >= m0
};

struct GemmArgs {
    const double* A; int64_t lda; int64_t strideA;
    const double* B; int64_t ldb; int64_t strideB;
    double* C; int64_t ldc; int64_t strideC;
    int M, N, K;
    double alpha, beta;
    int mode;
    int kchunk;            // > 0: split-K -- blockIdx.z selects the k range [z*kchunk, (z+1)*kchunk) (A, B not strided),
                           //      partial products go to C + z*strideC; reduce with splitk_reduce_kernel
};

constexpr int GT = 64;        // C tile
constexpr int GK = 16;        // K slab
constexpr int GLD = GK + 4;   // padded smem row (doubles): rows land on distinct 8-bank groups for the fragment reads
constexpr int GLDB = GT + 4;  // padded row for the non-transposed B slab [GK][GT]

// A_TRANS: the A operand is given as [k][m] (row-major, leading dimension lda), i.e. C = alpha * A^T * op(B) + beta * C
template <bool B_TRANS, bool A_TRANS = false>
__global__ void __launch_bounds__(128) gemm_f64_kernel(GemmArgs g) {
    const int m0 = blockIdx.y * GT, n0 = blockIdx.x * GT;
    if ((g.mode == GEMM_SYRK_LOWER || g.mode == GEMM_SYRK_LOWER_AUPPER) && n0 > m0) return;
    const bool splitk = g.kchunk > 0;
    const double* A = g.A + (splitk ? 0 : (int64_t)blockIdx.z * g.strideA);
    const double* B = g.B + (splitk ? 0 : (int64_t)blockIdx.z * g.strideB);
    double* C = g.C + (int64_t)blockIdx.z * g.strideC;

    __shared__ __align__(16) double As[2][A_TRANS ? GK * GLDB : GT * GLD];
    __shared__ __align__(16) double Bs[2][B_TRANS ? GT * GLD : GK * GLDB];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = (warp >> 1) * 32, wn = (warp & 1) * 32;
    const int gq = lane >> 2, tq = lane & 3;

    int kbeg = 0, kend = g.K;
    if (g.mode == GEMM_A_LOWER) kend = min(g.K, m0 + GT);
    if (g.mode == GEMM_B_LOWER) kbeg = n0;
    if (g.mode == GEMM_BT_LOWER) kend = min(g.K, n0 + GT);
    if (g.mode == GEMM_SYRK_LOWER_AUPPER || g.mode == GEMM_AT_LOWER) kbeg = m0;
    if (splitk) {
        kbeg = max(kbeg, (int)blockIdx.z * g.kchunk);
        kend = min(kend, ((int)blockIdx.z + 1) * g.kchunk);
    }

    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

    auto stage = [&](int buf, int k0) {
        // A slab: 64 rows x 16 doubles = 512 16-byte chunks (chunks at or beyond kend / N are zero-filled, never read)
        if (A_TRANS) {
#pragma unroll
            for (int c = tid; c < GK * (GT / 2); c += 128) {
                int r = c >> 5, q = c & 31;
                cp_async16(&As[buf][r * GLDB + q * 2], A + (int64_t)(k0 + r) * g.lda + m0 + q * 2, k0 + r < kend);
            }
        } else {
#pragma unroll
            for (int c = tid; c < GT * (GK / 2); c += 128) {
                int r = c >> 3, q = c & 7;
                cp_async16(&As[buf][r * GLD + q * 2], A + (int64_t)(m0 + r) * g.lda + k0 + q * 2, k0 + q * 2 < kend);
            }
        }
        if (B_TRANS) {
#pragma unroll
            for (int c = tid; c < GT * (GK / 2); c += 128) {
                int r = c >> 3, q = c & 7;
                cp_async16(&Bs[buf][r * GLD + q * 2], B + (int64_t)(n0 + r) * g.ldb + k0 + q * 2, k0 + q * 2 < kend && n0 + r < g.N);
            }
        } else {
#pragma unroll
            for (int c = tid; c < GK * (GT / 2); c += 128) {
                int r = c >> 5, q = c & 31;
                cp_async16(&Bs[buf][r * GLDB + q * 2], B + (int64_t)(k0 + r) * g.ldb + n0 + q * 2, k0 + r < kend && n0 + q * 2 < g.N);
            }
        }
        cp_async_commit();
    };

    const int nslab = (kend - kbeg + GK - 1) / GK;
    if (nslab > 0) stage(0, kbeg);
    for (int s = 0; s < nslab; s++) {
        const int buf = s & 1;
        if (s + 1 < nslab) {
            stage(buf ^ 1, kbeg + (s + 1) * GK);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < GK; kk += 4) {
            double a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; i++) a[i] = A_TRANS ? As[buf][(kk + tq) * GLDB + wm + i * 8 + gq] : As[buf][(wm + i * 8 + gq) * GLD + kk + tq];
#pragma unroll
            for (int j = 0; j < 4; j++)
                b[j] = B_TRANS ? Bs[buf][(wn + j * 8 + gq) * GLD + kk + tq] : Bs[buf][(kk + tq) * GLDB + wn + j * 8 + gq];
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
        __syncthreads();
    }

#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int64_t row = m0 + wm + i * 8 + gq;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (n0 + wn + j * 8 + tq * 2 >= g.N) continue;
            double2* p = reinterpret_cast<double2*>(C + row * g.ldc + n0 + wn + j * 8 + tq * 2);
            double2 out;
            if (g.beta != 0.0) {
                double2 old = *p;
                out.x = g.alpha * acc[i][j][0] + g.beta * old.x;
                out.y = g.alpha * acc[i][j][1] + g.beta * old.y;
            } else {
                out.x = g.alpha * acc[i][j][0];
                out.y = g.alpha * acc[i][j][1];
            }
            *p = out;
        }
    }
}

// out[r][c] = beta * out[r][c] + alpha * sum_z part[z][r][c]  (z in fixed order: deterministic)
static __global__ void splitk_reduce_kernel(const double* __restrict__ part, int nsplit, int64_t stride, int ldp, double* __restrict__ out,
                                            int64_t ldo, int rows, int cols, double alpha, double beta) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
    if (c >= cols || r >= rows) return;
    double s = 0.0;
    for (int z = 0; z < nsplit; z++) s += part[(int64_t)z * stride + (int64_t)r * ldp + c];
    double* o = out + (int64_t)r * ldo + c;
    *o = (beta != 0.0 ? beta * *o : 0.0) + alpha * s;
}

// C[M,N] (lower 64x64 tiles only: mode GEMM_SYRK_LOWER) = A^T A for A[K,M] row-major, optionally split over K (kchunk)
inline int launch_syrk_ata(const GemmArgs& g, int nsplit, cudaStream_t st) {
    if (g.M <= 0 || g.N <= 0 || nsplit <= 0) return MFGP_OK;
    dim3 grid((g.N + GT - 1) / GT, g.M / GT, nsplit);
    gemm_f64_kernel<false, true><<<grid, 128, 0, st>>>(g);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

// C[M,N] = alpha * A^T * B + beta * C for A[K,M] and B[K,N] row-major (modes GEMM_GENERAL, GEMM_AT_LOWER)
inline int launch_gemm_at(const GemmArgs& g, cudaStream_t st) {
    if (g.M <= 0 || g.N <= 0) return MFGP_OK;
    dim3 grid((g.N + GT - 1) / GT, g.M / GT, 1);
    gemm_f64_kernel<false, true><<<grid, 128, 0, st>>>(g);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

inline int launch_gemm(const GemmArgs& g, bool b_trans, int batch, cudaStream_t st) {
    if (g.M <= 0 || g.N <= 0 || batch <= 0) return MFGP_OK;
    dim3 grid((g.N + GT - 1) / GT, g.M / GT, batch);
    if (b_trans)
        gemm_f64_kernel<true><<<grid, 128, 0, st>>>(g);
    else
        gemm_f64_kernel<false><<<grid, 128, 0, st>>>(g);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

}  // namespace mfgp
