// Joint posterior draws at a point set from a Cholesky factor of its posterior covariance:
//
//   C = k**(X, X) - V^T V        (mfgp_posterior_cov, symmetric form)
//   L = chol(C + jitter I)       (mfgp_posterior_cov_factor: jitter and identity padding, then the fused tiled Cholesky)
//   F[g][s] = mu[g] + sum_{j<=g} L[g][j] E[j][s]          (mfgp_posterior_sample, posterior_sample_kernel)
//
// posterior_sample_kernel: one CTA owns a 64 x 64 tile of F (64 points x 64 draws).  Warp-specialised, 160 threads:
//   * producer warp: one lane streams 32-column slabs of L ([g][j] boxes, 16 columns x 64 rows) and 32-row slabs of E
//     ([j][s] boxes, 16 columns x 32 rows) with 2D TMA (128B swizzle) into a 3-stage full/empty mbarrier ring.  Rows of E
//     at or past G and columns past S read as zeros (TMA out-of-bounds fill).
//   * 4 consumer warps, 2 x 2, each 32 x 32 of F in registers (4 x 4 DMMA.8x8x4 tiles); mu is added in the epilogue.
// Row tile t reads L only up to its diagonal slab: about half of L is never touched.  In the slabs that reach past the
// tile's first row, elements with j > g are SELECTED to zero rather than multiplied by a zero: the strict upper part of L
// holds whatever the buffer held (C's mirrored half, W's blocks) and may be NaN or Inf.
// 64 x 64 tiles, two CTAs an SM: with S = 64 at G = 16384 there are 256 row tiles, and the longest (the bottom one, k = G)
// bounds the call; 128-row tiles would halve the parallelism and double that bound.  Tiles are launched bottom row first,
// so the long k loops start before the short ones.
// Split k: when the tiles cannot fill the SMs twice over (G = 2601, S = 64: 41 tiles), each tile is computed by a cluster of
// ksplit CTAs, rank r taking the r-th share of the tile's slabs.  The partial sums meet in distributed shared memory and
// are added in rank order, each rank finishing 1 / ksplit of the tile's elements.
// The k loop visits the slabs in order, DMMA's own order is fixed and ksplit depends only on G and S, so every element
// is bitwise reproducible.
#include <cmath>
#include <cooperative_groups.h>
#include <mutex>

#include "common.cuh"

namespace mfgp {

constexpr int PS_BM = 64;                  // rows of F (points) per tile
constexpr int PS_BN = 64;                  // columns of F (draws) per tile
constexpr int PS_BK = 32;                  // columns of L / rows of E per slab
constexpr int PS_STAGES = 3;
constexpr int PS_CONSUMER_WARPS = 4;
constexpr int PS_THREADS = (PS_CONSUMER_WARPS + 1) * 32;
constexpr int PS_MI = 4, PS_NI = 4;        // DMMA tiles per consumer warp (32 rows x 32 columns)
constexpr int PS_BOX_COLS = 16;            // one 128-byte swizzle row
constexpr int PS_A_BOX_BYTES = PS_BM * PS_BOX_COLS * 8;                   // 8192: 64 rows of L x 16 columns
constexpr int PS_B_BOX_BYTES = PS_BK * PS_BOX_COLS * 8;                   // 4096: 32 rows of E x 16 columns
constexpr int PS_A_BYTES = (PS_BK / PS_BOX_COLS) * PS_A_BOX_BYTES;        // 16384
constexpr int PS_B_BYTES = (PS_BN / PS_BOX_COLS) * PS_B_BOX_BYTES;        // 16384
constexpr int PS_STAGE_BYTES = PS_A_BYTES + PS_B_BYTES;
constexpr int PS_SMEM_BYTES = PS_STAGES * PS_STAGE_BYTES + 2 * PS_STAGES * 8 + 1024 /* alignment */;
constexpr int64_t PS_MAX_NPAD = 32768;     // largest factor mfgp_posterior_cov_factor accepts (tests/test_gpu_posterior_sample.py)

struct SampleArgs {
    const double* mu;
    double* F; int64_t ldf;
    int G, S;
    int tiles_n;                           // column tiles of F
    int tiles_m;                           // row tiles of F
    int ksplit;                            // CTAs (one cluster) per tile
};

__global__ void __launch_bounds__(PS_THREADS, 2)
posterior_sample_kernel(const __grid_constant__ CUtensorMap lmap, const __grid_constant__ CUtensorMap emap, SampleArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // 128B swizzle: 1024-byte aligned boxes
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + PS_STAGES * PS_STAGE_BYTES);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + PS_STAGES);

    const int tile = (int)(blockIdx.x / a.ksplit), rank = (int)(blockIdx.x % a.ksplit);
    const int ti = a.tiles_m - 1 - tile / a.tiles_n;                   // bottom row tiles (longest k loops) first
    const int tj = tile % a.tiles_n;
    const int i0 = ti * PS_BM, j0 = tj * PS_BN;
    const int kend = min(i0 + PS_BM, a.G);                             // L[g][j] = 0 for j > g: stop at the diagonal
    const int ntile_slabs = (kend + PS_BK - 1) / PS_BK;
    const int s0 = rank * ntile_slabs / a.ksplit, nslab = (rank + 1) * ntile_slabs / a.ksplit - s0;   // this rank's slabs
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    if (tid == 0) {
        for (int s = 0; s < PS_STAGES; s++) {
            mbar_init(full0 + 8 * s, 1);                     // the producer's arrive.expect_tx
            mbar_init(empty0 + 8 * s, PS_CONSUMER_WARPS);    // one arrive per consumer warp per drain
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncthreads();

    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    if (warp == PS_CONSUMER_WARPS) {
        // =============================== PRODUCER ===============================
        // (no early exit: the producer warp takes part in the cluster barriers of the reduction)
        if (lane == 0) {
            for (int it = 0; it < nslab; it++) {
                const int s = s0 + it;
                const int stage = it % PS_STAGES;
                const uint32_t parity = (it / PS_STAGES) & 1;
                mbar_wait(empty0 + 8 * stage, parity ^ 1);
                mbar_arrive_expect_tx(full0 + 8 * stage, PS_STAGE_BYTES);     // out-of-bounds zeros count as well
                const uint32_t dst = smem_u32(smem + stage * PS_STAGE_BYTES);
#pragma unroll
                for (int q = 0; q < PS_BK / PS_BOX_COLS; q++)
                    tma_load_2d(dst + q * PS_A_BOX_BYTES, &lmap, s * PS_BK + q * PS_BOX_COLS, i0, full0 + 8 * stage);
#pragma unroll
                for (int q = 0; q < PS_BN / PS_BOX_COLS; q++)
                    tma_load_2d(dst + PS_A_BYTES + q * PS_B_BOX_BYTES, &emap, j0 + q * PS_BOX_COLS, s * PS_BK, full0 + 8 * stage);
            }
        }
        cluster.sync();               // partials written (consumers, below)
        cluster.sync();               // every rank has read them
        return;
    }

    // =============================== CONSUMERS ===============================
    const int gq = lane >> 2, tq = lane & 3;
    const int wm = warp & 1, wn = warp >> 1;          // rows 32 wm .. +32, columns 32 wn .. +32 of the tile
    // L box ([g][j], 128-byte rows): this lane's A element (row gq of a DMMA row tile, column 4 (ks % 4) + tq of the box).
    // Row tiles start at multiples of 8 rows, so the swizzle row is gq: the 8 rows x 2 chunks of a half-warp's loads cover
    // all 32 banks, the minimum two wavefronts per warp.
    int offa[4];
#pragma unroll
    for (int q = 0; q < 4; q++) offa[q] = gq * 128 + (((2 * q + (tq >> 1)) ^ gq) << 4) + ((tq & 1) << 3);
    // E box ([j][s]): as gp_cov.cu's operands, rows 4 kp + tq, columns cv_perm(gq, h)
    int offb[2][2];
#pragma unroll
    for (int kp = 0; kp < 2; kp++)
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int c = cv_perm(gq, h), kr = 4 * kp + tq;
            offb[kp][h] = kr * 128 + (((c >> 1) ^ kr) << 4) + ((c & 1) << 3);
        }
    double acc[PS_MI][PS_NI][2];
#pragma unroll
    for (int i = 0; i < PS_MI; i++)
#pragma unroll
        for (int j = 0; j < PS_NI; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
    const int grow = i0 + wm * 32 + gq;               // this lane's row of DMMA row tile 0 (+ 8 i)

    for (int it = 0; it < nslab; it++) {
        const int s = s0 + it;
        const int stage = it % PS_STAGES;
        const uint32_t parity = (it / PS_STAGES) & 1;
        mbar_wait(full0 + 8 * stage, parity);
        const uint8_t* sa = smem + stage * PS_STAGE_BYTES + wm * 32 * 128;
        const uint8_t* sb = smem + stage * PS_STAGE_BYTES + PS_A_BYTES + wn * 2 * PS_B_BOX_BYTES;
        const bool masked = s * PS_BK + PS_BK - 1 > i0;    // the slab holds some j > g of this tile (warp-uniform)
#pragma unroll
        for (int ks = 0; ks < PS_BK / 4; ks++) {
            double af[PS_MI], bf[PS_NI];
#pragma unroll
            for (int i = 0; i < PS_MI; i++)
                af[i] = *reinterpret_cast<const double*>(sa + (ks >> 2) * PS_A_BOX_BYTES + i * 8 * 128 + offa[ks & 3]);
            if (masked) {
                const int k = s * PS_BK + 4 * ks + tq;
#pragma unroll
                for (int i = 0; i < PS_MI; i++) af[i] = k > grow + 8 * i ? 0.0 : af[i];     // select: NaN * 0 would be NaN
            }
#pragma unroll
            for (int j = 0; j < PS_NI; j++)
                bf[j] = *reinterpret_cast<const double*>(sb + (j >> 1) * PS_B_BOX_BYTES + (ks >> 1) * 1024 + offb[ks & 1][j & 1]);
#pragma unroll
            for (int i = 0; i < PS_MI; i++)
#pragma unroll
                for (int j = 0; j < PS_NI; j++) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty0 + 8 * stage);
    }

    // =============================== REDUCTION ===============================
    // partial sums -> this CTA's ring (free once every consumer warp is past its last slab), fragment-major:
    // part[(2 (4 i + j) + c) * 128 + thread].  Rank r finishes the fragment pairs v with v % ksplit == r, adding the
    // ranks' partials in rank order.
    asm volatile("bar.sync 1, %0;\n" ::"n"(PS_CONSUMER_WARPS * 32) : "memory");
    double* part = reinterpret_cast<double*>(smem);
#pragma unroll
    for (int i = 0; i < PS_MI; i++)
#pragma unroll
        for (int j = 0; j < PS_NI; j++) {
            part[(2 * (4 * i + j)) * 128 + tid] = acc[i][j][0];
            part[(2 * (4 * i + j) + 1) * 128 + tid] = acc[i][j][1];
        }
    cluster.sync();

    // =============================== EPILOGUE ===============================
    // lane (gq, tq) holds DMMA element (gq, 2 tq + c): tile row grow + 8 i, tile columns n0, n0 + 1 with
    // n0 = cv_perm(2 tq, j & 1) (even: the pair is one 16-byte store)
    for (int v = rank; v < PS_MI * PS_NI; v += a.ksplit) {
        const int i = v >> 2, j = v & 3;
        const int g = grow + 8 * i;
        const int n = j0 + wn * 32 + (j >> 1) * 16 + cv_perm(2 * tq, j & 1);
        double f0 = 0.0, f1 = 0.0;
        for (int q = 0; q < a.ksplit; q++) {
            const double* rp = cluster.map_shared_rank(part, q);
            f0 += rp[(2 * v) * 128 + tid];
            f1 += rp[(2 * v + 1) * 128 + tid];
        }
        if (g >= a.G || n >= a.S) continue;
        const double m = a.mu[g];
        double* row = a.F + (int64_t)g * a.ldf;
        if (n + 1 < a.S) *reinterpret_cast<double2*>(row + n) = make_double2(m + f0, m + f1);
        else row[n] = m + f0;
    }
    cluster.sync();                   // no CTA leaves while another still reads its partials
}

// C[npad, ld]: jitter on the first G diagonal entries, identity in rows / columns [G, npad).  Block y = row.
__global__ void cov_factor_prep_kernel(double* __restrict__ C, int64_t G, int64_t npad, int64_t ld, double jitter) {
    const int64_t r = blockIdx.y;
    double* row = C + r * ld;
    if (r < G) {
        if (threadIdx.x == 0) row[r] += jitter;
        for (int64_t c = G + threadIdx.x; c < npad; c += blockDim.x) row[c] = 0.0;
    } else {
        for (int64_t c = threadIdx.x; c < npad; c += blockDim.x) row[c] = c == r ? 1.0 : 0.0;
    }
}

// tensor maps of L / E per device, reused while a caller passes the same buffers (common.cuh: cached_tensor_map)
struct SampleMaps {
    std::mutex mu;
    CachedMap l, e;
    int sms = 0;
};
SampleMaps g_sample[16];

}  // namespace mfgp

using namespace mfgp;

extern "C" int mfgp_posterior_cov_factor(double* C, int64_t G, int64_t npad, int64_t ld, double jitter, double* W, int64_t ldw,
                                         int32_t* info, void* work, void* stream) {
    if (!C || !W || !info || !work || G < 0 || npad <= 0 || npad % MFGP_TILE || npad < G || npad > PS_MAX_NPAD)
        return MFGP_ERR_INVALID;
    if (!(jitter >= 0.0) || !std::isfinite(jitter)) return MFGP_ERR_INVALID;
    // the fused Cholesky's TMA operands (checked here too: nothing may be enqueued before a rejection)
    auto aligned = [](const void* p, int64_t l) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0 && (l & 1) == 0; };
    if (ld < npad || ldw < npad || !aligned(C, ld) || !aligned(W, ldw)) return MFGP_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cov_factor_prep_kernel<<<dim3(1, (unsigned)npad), 256, 0, st>>>(C, G, npad, ld, jitter);
    MFGP_LAUNCH_CHECK();
    return mfgp_cholesky(C, npad, ld, W, ldw, info, work, stream);
}

extern "C" int mfgp_posterior_sample(const double* L, int64_t G, int64_t ldl, const double* mu, const double* E, int64_t lde,
                                     int64_t S, double* F, int64_t ldf, void* stream) {
    if (G < 0 || S < 0) return MFGP_ERR_INVALID;
    if (G == 0 || S == 0) return MFGP_OK;
    if (!L || !mu || !E || !F || (reinterpret_cast<uintptr_t>(mu) & 7)) return MFGP_ERR_INVALID;
    auto aligned = [](const void* p, int64_t l) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0 && (l & 1) == 0; };
    if (!aligned(L, ldl) || !aligned(E, lde) || !aligned(F, ldf) || ldl < G || lde < S || ldf < S) return MFGP_ERR_INVALID;
    if (G > (1LL << 31) - PS_BM || S > (1LL << 31) - PS_BN) return MFGP_ERR_INVALID;      // int TMA coordinates
    const int64_t tm = (G + PS_BM - 1) / PS_BM, tn = (S + PS_BN - 1) / PS_BN;
    if (tm * tn >= (1LL << 31)) return MFGP_ERR_INVALID;
    int dev = 0;
    MFGP_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 16) return MFGP_ERR_INVALID;

    SampleArgs a{};
    a.mu = mu; a.F = F; a.ldf = ldf; a.G = (int)G; a.S = (int)S; a.tiles_m = (int)tm; a.tiles_n = (int)tn;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    SampleMaps& sm = g_sample[dev];
    std::lock_guard<std::mutex> lock(sm.mu);
    if (!sm.sms) MFGP_CUDA_CHECK(cudaDeviceGetAttribute(&sm.sms, cudaDevAttrMultiProcessorCount, dev));
    // split k (a power of two up to the portable cluster size 8) while the tiles fill fewer than two CTAs an SM and the
    // longest tile keeps at least four slabs per rank
    const int64_t max_slabs = (G + PS_BK - 1) / PS_BK;
    a.ksplit = 1;
    while (a.ksplit < 8 && tm * tn * a.ksplit < 2 * sm.sms && max_slabs >= 8 * a.ksplit) a.ksplit *= 2;
    int rc = cached_tensor_map(sm.l, L, G, G, ldl, PS_BOX_COLS, PS_BM, CU_TENSOR_MAP_SWIZZLE_128B);
    if (!rc) rc = cached_tensor_map(sm.e, E, G, S, lde, PS_BOX_COLS, PS_BK, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    MFGP_CUDA_CHECK(cudaFuncSetAttribute(posterior_sample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PS_SMEM_BYTES));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(tm * tn * a.ksplit));
    cfg.blockDim = dim3(PS_THREADS);
    cfg.dynamicSmemBytes = PS_SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)a.ksplit;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    MFGP_CUDA_CHECK(cudaLaunchKernelEx(&cfg, posterior_sample_kernel, sm.l.map, sm.e.map, a));
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}
