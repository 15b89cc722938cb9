// Shared device helpers for libmfgp_b200 (sm_100a): FP64 tensor-core MMA, cp.async / TMA staging, error plumbing.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cuda.h>
#include <cuda_runtime.h>

#include "../../include/mfgp_b200.h"

namespace mfgp {

// ---- error plumbing -----------------------------------------------------------------------------------------------
void set_last_error(const char* what, cudaError_t e);

#define MFGP_CUDA_CHECK(expr)                                   \
    do {                                                        \
        cudaError_t _e = (expr);                                \
        if (_e != cudaSuccess) {                                \
            ::mfgp::set_last_error(#expr, _e);                  \
            return MFGP_ERR_CUDA;                               \
        }                                                       \
    } while (0)

void count_launch();
#define MFGP_LAUNCH_CHECK()                  \
    do {                                     \
        ::mfgp::count_launch();              \
        MFGP_CUDA_CHECK(cudaGetLastError()); \
    } while (0)

// ---- FP64 tensor-core MMA -----------------------------------------------------------------------------------------
// sm_100a executes every f64 mma.sync shape as DMMA.8x8x4 (profiles/r01_fp64_pipes.log: m8n8k4, m16n8k8 and
// m16n8k16 all issue at 64 MAC/clk/SM = 37.1 TFLOP/s), so the native 8x8x4 shape is used directly.
// Fragments (lane = 4*g + t, g = lane/4, t = lane%4):  A[g][t]   B[t][g]   C[g][2t], C[g][2t+1].
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// ---- cp.async (LDGSTS) 16-byte staging ----------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src, bool valid) {
    unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
    int bytes = valid ? 16 : 0;   // src-size 0 => destination zero-filled
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem_src), "r"(bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

// ---- mbarrier / TMA primitives (PTX) ----------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!done);
}
// box of a 2D tensor map at element coordinates (c0 = column, c1 = row) -> shared memory; completion in bytes on `bar`
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n" ::"r"(dst),
        "l"(map), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
}

// Row g (0..7) of DMMA tile half h inside a 16-column box of a [k][n] slab loaded with 128B swizzle (gp_cov.cu,
// gp_sample.cu).  The swizzle puts 16-byte chunk c of slab row k at chunk c ^ (k % 8); a half-warp loads rows k = 4p + t
// (t = 0..3) of the four g it holds, so the g must spread over both halves of the chunk range for the 16 loads to hit 16
// distinct bank pairs: g -> {0, 1, 8, 9, 2, 3, 10, 11} (+4 for h = 1).
__device__ __forceinline__ int cv_perm(int g, int h) { return (g & 1) | (((g >> 2) & 1) << 1) | (h << 2) | (((g >> 1) & 1) << 3); }

// register budget of a warpgroup after the role split of a warp-specialised kernel (every warp of the group executes it)
template <int R>
__device__ __forceinline__ void reg_alloc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;\n" ::"n"(R)); }
template <int R>
__device__ __forceinline__ void reg_dealloc() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" ::"n"(R)); }

// 2D tensor map of a row-major FP64 matrix (rows x cols, row stride ld elements) with a box of box_cols x box_rows;
// cuTensorMapEncodeTiled through the runtime's driver entry point query (no link-time dependency on libcuda).  The base
// must be 16-byte aligned and ld even; boxes reaching past the matrix read zeros.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline int make_tensor_map_2d(CUtensorMap* map, const double* base, int64_t rows, int64_t cols, int64_t ld, int box_cols,
                              int box_rows, CUtensorMapSwizzle swizzle) {
    static EncodeTiledFn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        MFGP_CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (qres != cudaDriverEntryPointSuccess || !fn) {
            set_last_error("cuTensorMapEncodeTiled entry point unavailable", cudaErrorUnknown);
            return MFGP_ERR_CUDA;
        }
        encode = reinterpret_cast<EncodeTiledFn>(fn);
    }
    const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};       // {columns (contiguous), rows}
    const cuuint64_t gstride[1] = {(cuuint64_t)ld * sizeof(double)};       // row pitch in bytes
    const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(base), gdim, gstride, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_last_error("cuTensorMapEncodeTiled failed", cudaErrorInvalidValue);
        return MFGP_ERR_CUDA;
    }
    return MFGP_OK;
}

// A tensor map kept while the next call passes the same buffer and shape (a step re-uses the same buffers, so the maps are
// encoded once).  Each cache slot serves one call site, whose box and swizzle are fixed.  The caller holds a mutex from the
// lookup through the launch that copies the map into its parameters: otherwise another host thread could re-encode the
// slot for its own buffers in between.
struct CachedMap {
    const double* base = nullptr;
    int64_t rows = 0, cols = 0, ld = 0;
    CUtensorMap map{};
};
inline int cached_tensor_map(CachedMap& m, const double* base, int64_t rows, int64_t cols, int64_t ld, int box_cols,
                             int box_rows, CUtensorMapSwizzle swizzle) {
    if (m.base == base && m.rows == rows && m.cols == cols && m.ld == ld) return MFGP_OK;
    m.base = nullptr;
    const int rc = make_tensor_map_2d(&m.map, base, rows, cols, ld, box_cols, box_rows, swizzle);
    if (rc) return rc;
    m.base = base; m.rows = rows; m.cols = cols; m.ld = ld;
    return MFGP_OK;
}

// ---- the RBF kernel with the reference's operation order (gaussian_process.py:75-79) -------------------------------
// inputs are coordinates ALREADY divided by the length scale
__device__ __forceinline__ double rbf_scaled(double ax, double ay, double bx, double by, double scale) {
    double d0 = ax - bx, d1 = ay - by;
    double q = __dadd_rn(__dmul_rn(d0, d0), __dmul_rn(d1, d1));
    return scale * exp(-0.5 * q);
}

struct DevParams {   // mfgp_params plus derived constants, passed by value to kernels
    double s_L, inv_unused, s_H, rho, rho2, noise_L, noise_H, mean_L, mean_H, jitter, l_L, l_H, k0;
    int multi;
};

inline DevParams make_dev_params(const mfgp_params& p) {
    DevParams d;
    d.s_L = p.multi ? p.s_L : 0.0;
    d.inv_unused = 0.0;
    d.s_H = p.s_H;
    d.rho = p.multi ? p.rho : 1.0;
    d.rho2 = d.rho * d.rho;   // "rho ** 2" in the reference
    d.noise_L = p.noise_L;
    d.noise_H = p.noise_H;
    d.mean_L = p.mean_L;
    d.mean_H = p.mean_H;
    d.jitter = p.jitter;
    d.l_L = p.multi ? p.l_L : 1.0;
    d.l_H = p.l_H;
    d.k0 = p.multi ? (d.rho2 * p.s_L + p.s_H) : p.s_H;   // gaussian_process.py:435-436 on the diagonal
    d.multi = p.multi;
    return d;
}

}  // namespace mfgp
