// Joint / cross posterior covariance (the cov[G,G] that SFGP.predict, reference gaussian_process.py:121-148, and
// MFGP.predict, :401-438, return; the default posterior of gp_posterior.cu keeps only its diagonal).
//
//   C[i][j] = k**(a_i, b_j) - sum_{n<N} V_A[n][i] V_B[n][j]          V = W psi^T, written by mfgp_posterior[_grid] (Vc)
//
// One CTA owns a 128 x 128 tile of C.  Warp-specialised, 384 threads:
//   * producer warp group: one lane of its first warp streams 32-row slabs of V_A and V_B with 2D TMA (cp.async.bulk.tensor, 128B swizzle, eight
//     16-column boxes per operand) into a 3-stage full/empty mbarrier ring.  Rows n >= N and columns past Ga / Gb read as
//     zeros (TMA out-of-bounds fill), so no size needs to be a multiple of the tile.
//   * 8 consumer warps, 2 x 4, each 64 x 32 of C in registers (8 x 4 DMMA.8x8x4 tiles), then the epilogue: k** from the
//     coordinates staged in shared memory (rbf_scaled, the reference's operation order; no noise, no jitter), minus the
//     accumulator, stored straight from registers.
// setmaxnreg moves registers from the producer group (40) to the consumers (232): 128 x 40 + 256 x 232 = 384 x 168, the
// CTA pool; with an even split the 128 accumulators per thread do not fit and spill.
// The k loop visits the slabs in order and DMMA's own order is fixed, so every element is bitwise reproducible.
// Symmetric form (B = A): only the tiles on or below the diagonal are launched, enumerated linearly; every value of a tile
// below the diagonal is stored twice, at (i, j) and (j, i), and a diagonal tile stores its lower half and mirrors it, so
// C == C^T bitwise without relying on DMMA giving equal values for (i, j) and (j, i).
#include <cmath>
#include <mutex>

#include "common.cuh"

namespace mfgp {

constexpr int CV_BM = 128;                 // tile of C (rows = points of A, columns = points of B)
constexpr int CV_BK = 32;                  // rows of V per slab
constexpr int CV_STAGES = 3;
constexpr int CV_CONSUMER_WARPS = 8;
constexpr int CV_THREADS = (CV_CONSUMER_WARPS + 4) * 32;   // + one producer warp group
constexpr int CV_MI = 8, CV_NI = 4;        // DMMA tiles per consumer warp (64 rows x 32 columns)
constexpr int CV_BOX_COLS = 16;            // one 128-byte swizzle row
constexpr int CV_BOX_BYTES = CV_BK * CV_BOX_COLS * 8;                     // 4096
constexpr int CV_OPERAND_BYTES = (CV_BM / CV_BOX_COLS) * CV_BOX_BYTES;    // 32768
constexpr int CV_STAGE_BYTES = 2 * CV_OPERAND_BYTES;
constexpr int CV_SMEM_BYTES = CV_STAGES * CV_STAGE_BYTES + 2 * CV_BM * 4 * 8 + 2 * CV_STAGES * 8 + 1024 /* alignment */;

struct CovArgs {
    const double* Xa; const double* Xb;    // points [G][2]; Xb == Xa in the symmetric form
    int64_t Ga, Gb;
    double* C; int64_t ldc;
    int nslab;                             // ceil(N / CV_BK); 0: C = k**
    int tiles_a;                           // row tiles of C
    int sym;
    DevParams p;
};

__device__ __forceinline__ void cv_coords(double* dst, const double* X, int64_t g0, int64_t G, const DevParams& p) {
    for (int e = threadIdx.x; e < CV_BM; e += CV_THREADS) {
        int64_t g = g0 + e;
        if (g >= G) g = G - 1;
        const double x = X[2 * g], y = X[2 * g + 1];
        dst[e * 4 + 0] = x / p.l_L;
        dst[e * 4 + 1] = y / p.l_L;
        dst[e * 4 + 2] = x / p.l_H;
        dst[e * 4 + 3] = y / p.l_H;
    }
}

// prior covariance k**(a, b): gaussian_process.py:146 (SF), :435-436 (MF: rho^2 k_L + k_H)
__device__ __forceinline__ double cv_prior(const double* a, const double* b, const DevParams& p) {
    const double kH = rbf_scaled(a[2], a[3], b[2], b[3], p.s_H);
    if (!p.multi) return kH;
    const double kL = rbf_scaled(a[0], a[1], b[0], b[1], p.s_L);
    return __dadd_rn(__dmul_rn(p.rho2, kL), kH);
}

__global__ void __launch_bounds__(CV_THREADS, 1)
posterior_cov_kernel(const __grid_constant__ CUtensorMap amap, const __grid_constant__ CUtensorMap bmap, CovArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // (keeps the shared address space: LDS)
    double* xa = reinterpret_cast<double*>(smem + CV_STAGES * CV_STAGE_BYTES);   // [128][4] scaled coordinates
    double* xb = xa + CV_BM * 4;
    uint64_t* bars = reinterpret_cast<uint64_t*>(xb + CV_BM * 4);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + CV_STAGES);

    // tile of this CTA: symmetric -> t = ti (ti + 1) / 2 + tj, tj <= ti; cross -> the row tiles of one column tile are
    // consecutive, so the CTAs in flight share their V_B slab and V_A stays in L2 when it is a block row
    int64_t ti, tj;
    const int64_t t = blockIdx.x;
    if (a.sym) {
        ti = (int64_t)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
        while ((ti + 1) * (ti + 2) / 2 <= t) ti++;
        while (ti * (ti + 1) / 2 > t) ti--;
        tj = t - ti * (ti + 1) / 2;
    } else {
        ti = t % a.tiles_a;
        tj = t / a.tiles_a;
    }
    const int64_t i0 = ti * CV_BM, j0 = tj * CV_BM;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const DevParams& p = a.p;

    if (tid == 0) {
        for (int s = 0; s < CV_STAGES; s++) {
            mbar_init(full0 + 8 * s, 1);                     // the producer's arrive.expect_tx
            mbar_init(empty0 + 8 * s, CV_CONSUMER_WARPS);    // one arrive per consumer warp per drain
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    cv_coords(xa, a.Xa, i0, a.Ga, p);
    cv_coords(xb, a.Xb, j0, a.Gb, p);
    __syncthreads();

    if (warp >= CV_CONSUMER_WARPS) {
        // =============================== PRODUCER ===============================
        reg_dealloc<40>();
        if (warp == CV_CONSUMER_WARPS && lane == 0) {
            for (int s = 0; s < a.nslab; s++) {
                const int stage = s % CV_STAGES;
                const uint32_t parity = (s / CV_STAGES) & 1;
                mbar_wait(empty0 + 8 * stage, parity ^ 1);
                mbar_arrive_expect_tx(full0 + 8 * stage, CV_STAGE_BYTES);     // out-of-bounds zeros count as well
                const uint32_t dst = smem_u32(smem + stage * CV_STAGE_BYTES);
#pragma unroll
                for (int q = 0; q < CV_BM / CV_BOX_COLS; q++) {
                    tma_load_2d(dst + q * CV_BOX_BYTES, &amap, (int)i0 + q * CV_BOX_COLS, s * CV_BK, full0 + 8 * stage);
                    tma_load_2d(dst + CV_OPERAND_BYTES + q * CV_BOX_BYTES, &bmap, (int)j0 + q * CV_BOX_COLS, s * CV_BK,
                                full0 + 8 * stage);
                }
            }
        }
        return;
    }

    // =============================== CONSUMERS ===============================
    reg_alloc<232>();
    const int gq = lane >> 2, tq = lane & 3;
    const int wm = warp & 1, wn = warp >> 1;          // rows 64 wm .. +64, columns 32 wn .. +32 of the tile
    // byte offset of this lane's element in a 16-column box for k-step parity kp and tile half h: slab row 4 kp + tq
    int off[2][2];
#pragma unroll
    for (int kp = 0; kp < 2; kp++)
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int c = cv_perm(gq, h), kr = 4 * kp + tq;
            off[kp][h] = kr * 128 + (((c >> 1) ^ kr) << 4) + ((c & 1) << 3);
        }
    double acc[CV_MI][CV_NI][2];
#pragma unroll
    for (int i = 0; i < CV_MI; i++)
#pragma unroll
        for (int j = 0; j < CV_NI; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

    for (int s = 0; s < a.nslab; s++) {
        const int stage = s % CV_STAGES;
        const uint32_t parity = (s / CV_STAGES) & 1;
        mbar_wait(full0 + 8 * stage, parity);
        const uint8_t* sa = smem + stage * CV_STAGE_BYTES + wm * 4 * CV_BOX_BYTES;                  // DMMA row tile i: box i/2
        const uint8_t* sb = smem + stage * CV_STAGE_BYTES + CV_OPERAND_BYTES + wn * 2 * CV_BOX_BYTES;   // column tile j: box j/2
#pragma unroll
        for (int ks = 0; ks < CV_BK / 4; ks++) {
            double af[CV_MI], bf[CV_NI];
#pragma unroll
            for (int i = 0; i < CV_MI; i++)
                af[i] = *reinterpret_cast<const double*>(sa + (i >> 1) * CV_BOX_BYTES + (ks >> 1) * 1024 + off[ks & 1][i & 1]);
#pragma unroll
            for (int j = 0; j < CV_NI; j++)
                bf[j] = *reinterpret_cast<const double*>(sb + (j >> 1) * CV_BOX_BYTES + (ks >> 1) * 1024 + off[ks & 1][j & 1]);
#pragma unroll
            for (int i = 0; i < CV_MI; i++)
#pragma unroll
                for (int j = 0; j < CV_NI; j++) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty0 + 8 * stage);
    }

    // =============================== EPILOGUE ===============================
    // lane (gq, tq) holds DMMA element (gq, 2 tq + c): tile row cv_perm(gq, i & 1), tile columns n0, n0 + 1 with
    // n0 = cv_perm(2 tq, j & 1) (even, so the pair is one 16-byte store when the row is aligned)
    const bool diag = a.sym && ti == tj;
#pragma unroll
    for (int i = 0; i < CV_MI; i++) {
        const int m = wm * 64 + (i >> 1) * 16 + cv_perm(gq, i & 1);
        const int64_t gi = i0 + m;
        if (gi >= a.Ga) continue;
        const double* pa = xa + m * 4;
#pragma unroll
        for (int j = 0; j < CV_NI; j++) {
            const int n = wn * 32 + (j >> 1) * 16 + cv_perm(2 * tq, j & 1);
            const int64_t gj = j0 + n;
            if (gj >= a.Gb) continue;
            const bool two = gj + 1 < a.Gb;
            double v[2];
            v[0] = cv_prior(pa, xb + n * 4, p) - acc[i][j][0];
            v[1] = two ? cv_prior(pa, xb + (n + 1) * 4, p) - acc[i][j][1] : 0.0;
            double* dst = a.C + gi * a.ldc + gj;
            if (diag) {
#pragma unroll
                for (int c = 0; c < 2; c++) {
                    if (c == 1 && !two) break;
                    if (gi >= gj + c) dst[c] = v[c];
                    if (gi > gj + c) a.C[(gj + c) * a.ldc + gi] = v[c];
                }
                continue;
            }
            if (two && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
                *reinterpret_cast<double2*>(dst) = make_double2(v[0], v[1]);
            } else {
                dst[0] = v[0];
                if (two) dst[1] = v[1];
            }
            if (a.sym) {
                a.C[gj * a.ldc + gi] = v[0];
                if (two) a.C[(gj + 1) * a.ldc + gi] = v[1];
            }
        }
    }
}

// tensor maps of V_A / V_B per device, reused while a caller passes the same buffers (common.cuh: cached_tensor_map)
struct CovMaps {
    std::mutex mu;
    CachedMap a, b;
};
CovMaps g_cov[16];

}  // namespace mfgp

using namespace mfgp;

extern "C" int mfgp_posterior_cov(const double* Xa, int64_t Ga, const double* Va, int64_t ldva, const double* Xb, int64_t Gb,
                                  const double* Vb, int64_t ldvb, int64_t N, const mfgp_params* p_host, double* C,
                                  int64_t ldc, void* stream) {
    const bool sym = Xb == nullptr;
    if (!p_host || !C || Ga < 0 || Gb < 0 || N < 0 || (Ga > 0 && !Xa)) return MFGP_ERR_INVALID;
    if (sym && (Vb != nullptr || Gb != Ga)) return MFGP_ERR_INVALID;
    if ((ldc & 1) || ldc < Gb || (reinterpret_cast<uintptr_t>(C) & 7)) return MFGP_ERR_INVALID;
    auto v_ok = [N](const double* V, int64_t ldv, int64_t G) {     // TMA: 16-byte aligned base and row pitch
        return N == 0 || (V != nullptr && (reinterpret_cast<uintptr_t>(V) & 15) == 0 && (ldv & 1) == 0 && ldv >= G);
    };
    if (!v_ok(Va, ldva, Ga) || (!sym && !v_ok(Vb, ldvb, Gb))) return MFGP_ERR_INVALID;
    if (N >= (1LL << 31) || Ga > (1LL << 31) - CV_BM || Gb > (1LL << 31) - CV_BM) return MFGP_ERR_INVALID;   // int TMA coordinates
    if (Ga == 0 || Gb == 0) return MFGP_OK;
    const int64_t ta = (Ga + CV_BM - 1) / CV_BM, tb = (Gb + CV_BM - 1) / CV_BM;
    const int64_t ntiles = sym ? ta * (ta + 1) / 2 : ta * tb;
    if (ntiles >= (1LL << 31)) return MFGP_ERR_INVALID;
    int dev = 0;
    MFGP_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 16) return MFGP_ERR_INVALID;

    CovArgs a{};
    a.Xa = Xa; a.Xb = sym ? Xa : Xb; a.Ga = Ga; a.Gb = Gb; a.C = C; a.ldc = ldc;
    a.nslab = (int)((N + CV_BK - 1) / CV_BK); a.tiles_a = (int)ta; a.sym = sym ? 1 : 0;
    a.p = make_dev_params(*p_host);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CovMaps& cm = g_cov[dev];
    std::lock_guard<std::mutex> lock(cm.mu);
    if (N > 0) {      // N = 0: C = k**, V is not read
        int rc = cached_tensor_map(cm.a, Va, N, Ga, ldva, CV_BOX_COLS, CV_BK, CU_TENSOR_MAP_SWIZZLE_128B);
        if (!rc && !sym) rc = cached_tensor_map(cm.b, Vb, N, Gb, ldvb, CV_BOX_COLS, CV_BK, CU_TENSOR_MAP_SWIZZLE_128B);
        if (rc) return rc;
    }
    MFGP_CUDA_CHECK(cudaFuncSetAttribute(posterior_cov_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CV_SMEM_BYTES));
    posterior_cov_kernel<<<(unsigned)ntiles, CV_THREADS, CV_SMEM_BYTES, st>>>(cm.a.map, sym ? cm.a.map : cm.b.map, a);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}
