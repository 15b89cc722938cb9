// Fused GP posterior over a tile of grid points (replaces SFGP.predict, reference gaussian_process.py:121-148, and
// MFGP.predict, :401-438, diagonal only -- the reference's callers take np.diag of the covariance).
//
//   v = W psi(x*)          W = L^-1 (lower triangular, from mfgp_tri_inverse), psi = cross-covariance column
//   mu  = mean_H + v . z   z = W (y - mean)
//   var = k(0)  - v . v
//
// One CTA owns BN = 32 grid points and walks the 512-row blocks of W top to bottom; psi and V never reach HBM
// (unless the caller asks for the V cache of the Choi planner).  Warp-specialised, 384 threads:
//   * producer warp group (4 warps): one elected thread streams 512x16 tiles of W from L2/HBM with TMA
//     (cp.async.bulk.tensor, 128B swizzle) into a 3-stage shared-memory ring; all 128 producer threads GENERATE the
//     matching 16x32 tile of psi (fp64 exp) into the same stage.  mbarriers (full/empty per stage) carry the hand-off.
//   * consumer warp groups (8 warps): read A/B fragments from the ring and issue DMMA.8x8x4 into 128 KB of register
//     accumulators (512x32 fp64), then fold each finished row block of V into the two running column reductions.
// setmaxnreg moves registers from the producers (72) to the consumers (216); the two must balance exactly within the
// CTA pool of 384 x 168 registers, otherwise the consumers' setmaxnreg.inc never completes.
//
// Why the tile is tall: DMMA and DFMA share one datapath on sm_100a and an fp64 exp costs ~23 FP64 lane-slots
// (profiles/r01_fp64_pipes.log), so every regenerated psi element is paid in MMA time; with BM = 512 a psi element is
// reused 512 times per generation (exp ~ 9% of the MMA work at N = 4096).  v1 of this kernel (single-role CTA,
// cp.async double buffer) sat at 52% DMMA-pipe utilisation with the psi-generation load latency and the barrier
// phases exposed (profiles/r01_posterior_v1_ncu_summary.txt); the producer/consumer split hides both.
// Triangular structure: slabs right of the diagonal are never visited, and inside the diagonal square each warp
// skips the 8-row tiles that lie entirely above the diagonal (rows are interleaved over warps so this stays balanced).
#include <cuda.h>

#include "common.cuh"

namespace mfgp {

constexpr int P_BM = 512;            // rows of W per row block
constexpr int P_BN = 32;             // grid points per CTA
constexpr int P_BK = 16;             // K slab (16 doubles = one 128-byte swizzle row)
constexpr int P_STAGES = 3;
constexpr int P_CONSUMER_WARPS = 8;
constexpr int P_PRODUCER_WARPS = 4;
constexpr int P_THREADS = (P_CONSUMER_WARPS + P_PRODUCER_WARPS) * 32;
constexpr int P_MI = 8;              // 8-row tiles per consumer warp
constexpr int P_NI = 4;              // 8-column tiles per consumer warp
constexpr int P_PLD = P_BK + 4;      // padded psi row (doubles)
constexpr int P_W_STAGE_BYTES = P_BM * P_BK * 8;            // 65536
constexpr int P_PSI_STAGE_BYTES = P_BN * P_PLD * 8;         // 5120
constexpr int P_SMEM_BYTES = P_STAGES * (P_W_STAGE_BYTES + P_PSI_STAGE_BYTES) + P_BN * 4 * 8 +
                             P_CONSUMER_WARPS * P_BN * 2 * 8 + 2 * P_STAGES * 8 + 1024 /* alignment slack */;

struct PostArgs {
    const double* Xs; int64_t G;         // general mode: explicit points
    // grid mode (tensor-product grid, x-major): point g_lo + g <-> (ix, iy) = divmod(g_lo + g, ny); per-axis tables
    // TLx[nx][ldt], TLy[ny][ldt], THx[nx][ldt], THy[ny][ldt] with psi[g][n] = TLx[ix][n]*TLy[iy][n] + THx[ix][n]*THy[iy][n]
    const double* TLx; const double* TLy; const double* THx; const double* THy;
    int64_t ldt; int64_t g_lo; int ny;
    const double* Tt; int NL, NH;
    int npad;
    const double* z;
    double* mu; double* var; double* qout;   // qout (optional): sum of v^2, the variance reduction
    double* Vc; int64_t ldv;
    int remap_cols;      // > 0 (grid mode, whole columns): CTA b -> column b % remap_cols, y-band b / remap_cols, so the CTAs
                         // in flight share ONE band of the y-axis tables; the L2-resident set is W + a few MB instead of
                         // W + all y tables (which together exceed the 126 MB L2 at N = 4096)
    int row_lo;          // > 0: incremental update -- only rows >= row_lo of V are formed and ADDED to mu / var / qout
    DevParams p;
};

// ---- expect-tx primitive (PTX; mbarrier, TMA and setmaxnreg: common.cuh) --------------------------------------------------
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {   // adds to the tx-count, no arrival
    asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}

// MMA row slot g (0..7) of an 8-row tile <-> row of the tile.  With the TMA 128B swizzle (16-byte chunk index XOR
// row%8) a half-warp must touch rows whose row%8 differ in bits 1..2 to hit 16 distinct bank pairs: 0,2,4,6 | 1,3,5,7.
__device__ __forceinline__ int row_perm(int g) { return ((g & 3) << 1) | (g >> 2); }

template <bool GRID>
__global__ void __launch_bounds__(P_THREADS, 1)
posterior_kernel(const __grid_constant__ CUtensorMap wmap, PostArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* Wst = smem;                                                        // [S][512][16] doubles, swizzled
    double* Pst = reinterpret_cast<double*>(smem + P_STAGES * P_W_STAGE_BYTES); // [S][32][20]
    double* xs = Pst + P_STAGES * P_BN * P_PLD;                                 // [32][4]
    double* colacc = xs + P_BN * 4;                                             // [8][32][2]
    uint64_t* bars = reinterpret_cast<uint64_t*>(colacc + P_CONSUMER_WARPS * P_BN * 2);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + P_STAGES);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t g0 = (GRID && a.remap_cols > 0)
                           ? (int64_t)(blockIdx.x % a.remap_cols) * a.ny + (int64_t)(blockIdx.x / a.remap_cols) * P_BN
                           : (int64_t)blockIdx.x * P_BN;
    const int N = a.NL + a.NH;
    const DevParams& p = a.p;

    if (tid == 0) {
        for (int s = 0; s < P_STAGES; s++) {
            mbar_init(full0 + 8 * s, P_PRODUCER_WARPS * 32);     // every producer thread arrives once per fill
            mbar_init(empty0 + 8 * s, P_CONSUMER_WARPS);         // one arrive per consumer warp per drain
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (!GRID) {
        for (int e = tid; e < P_BN; e += P_THREADS) {
            int64_t g = g0 + e;
            if (g >= a.G) g = a.G - 1;
            const double x = a.Xs[2 * g], y = a.Xs[2 * g + 1];
            xs[e * 4 + 0] = x / p.l_L;
            xs[e * 4 + 1] = y / p.l_L;
            xs[e * 4 + 2] = x / p.l_H;
            xs[e * 4 + 3] = y / p.l_H;
        }
    }
    for (int e = tid; e < P_CONSUMER_WARPS * P_BN * 2; e += P_THREADS) colacc[e] = 0.0;
    __syncthreads();

    const int nrb = (a.npad + P_BM - 1) / P_BM;
    const int rb_begin = a.row_lo / P_BM;      // incremental update: row blocks below the first new row are not visited

    if (warp >= P_CONSUMER_WARPS) {
        // =============================== PRODUCERS ===============================
        reg_dealloc<72>();   // pool = 384 x 168: 128 x (168-72) freed == 256 x (216-168) claimed by the consumers
        const int pt = tid - P_CONSUMER_WARPS * 32;       // 0..127
        const int k = pt & 15;                            // column of the slab this thread generates
        const int gbase = pt >> 4;                        // grid points gbase, gbase+8, gbase+16, gbase+24
        // grid mode: table row offsets of this thread's four points (x-major flat index -> ix, iy)
        int offx[4], offy[4];          // element offsets (host checks (nx|ny) * ldt < 2^31)
        if (GRID) {
#pragma unroll
            for (int i = 0; i < 4; i++) {
                int64_t g = g0 + gbase + 8 * i;
                if (g >= a.G) g = a.G - 1;
                g += a.g_lo;
                offx[i] = (int)((g / a.ny) * a.ldt);
                offy[i] = (int)((g % a.ny) * a.ldt);
            }
        }
        int it = 0;
        for (int rb = rb_begin; rb < nrb; rb++) {
            const int row0 = rb * P_BM;
            const int nslab = min(a.npad, row0 + P_BM) / P_BK;
            for (int s = 0; s < nslab; s++, it++) {
                const int stage = it % P_STAGES;
                const uint32_t parity = (it / P_STAGES) & 1;
                const int n = s * P_BK + k;
                // operands of this slab are fetched BEFORE waiting for the ring slot: the L2 latency overlaps the wait
                double4 t = make_double4(0.0, 0.0, 0.0, 0.0);
                double lx[4], ly[4], hx[4], hy[4];
                if (GRID) {
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        lx[i] = __ldg(a.TLx + offx[i] + n);
                        ly[i] = __ldg(a.TLy + offy[i] + n);
                        hx[i] = __ldg(a.THx + offx[i] + n);
                        hy[i] = __ldg(a.THy + offy[i] + n);
                    }
                } else if (n < N) {
                    t = reinterpret_cast<const double4*>(a.Tt)[n];
                }
                mbar_wait(empty0 + 8 * stage, parity ^ 1);
                if (pt == 0) {
                    mbar_expect_tx(full0 + 8 * stage, P_W_STAGE_BYTES);
                    const uint32_t dst = smem_u32(Wst + stage * P_W_STAGE_BYTES);
                    tma_load_2d(dst, &wmap, s * P_BK, row0, full0 + 8 * stage);
                    tma_load_2d(dst + P_W_STAGE_BYTES / 2, &wmap, s * P_BK, row0 + P_BM / 2, full0 + 8 * stage);
                }
                // psi tile: element (point gi, training column n); gaussian_process.py:426-429 / :139
                double* pdst = Pst + stage * P_BN * P_PLD;
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const int gi = gbase + 8 * i;
                    double v = 0.0;
                    if (GRID) {
                        v = fma(hx[i], hy[i], lx[i] * ly[i]);      // scales, rho and padding zeros are folded into T?x
                    } else if (n < N) {
                        if (p.multi) {
                            const double kL = rbf_scaled(xs[gi * 4 + 0], xs[gi * 4 + 1], t.x, t.y, p.s_L);
                            if (n < a.NL) {
                                v = p.rho * kL;
                            } else {
                                const double kH = rbf_scaled(xs[gi * 4 + 2], xs[gi * 4 + 3], t.z, t.w, p.s_H);
                                v = __dadd_rn(__dmul_rn(p.rho2, kL), kH);
                            }
                        } else {
                            v = rbf_scaled(xs[gi * 4 + 2], xs[gi * 4 + 3], t.z, t.w, p.s_H);
                        }
                    }
                    pdst[gi * P_PLD + k] = v;
                }
                mbar_arrive(full0 + 8 * stage);      // release: this thread's psi stores are visible to the waiters
            }
        }
    } else {
        // =============================== CONSUMERS ===============================
        reg_alloc<216>();
        const int gq = lane >> 2, tq = lane & 3;
        const int pr = row_perm(gq);
        // byte offset of this lane's A element inside an 8-row tile for k-step kk: row pr, 16B-chunk ((kk+tq)/2)^pr
        int aoff[4];
#pragma unroll
        for (int j = 0; j < 4; j++) aoff[j] = pr * 128 + ((((j * 4 + tq) >> 1) ^ pr) << 4) + ((tq & 1) << 3);
        int it = 0;
        for (int rb = rb_begin; rb < nrb; rb++) {
            const int row0 = rb * P_BM;
            const int nslab = min(a.npad, row0 + P_BM) / P_BK;

            double acc[P_MI][P_NI][2];
#pragma unroll
            for (int i = 0; i < P_MI; i++)
#pragma unroll
                for (int j = 0; j < P_NI; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

            // last k (inclusive) at which 8-row tile i of this warp still has a non-zero W entry; -1 = tile unused
            int klim[P_MI];
#pragma unroll
            for (int i = 0; i < P_MI; i++) {
                const int r = row0 + (i * P_CONSUMER_WARPS + warp) * 8;
                klim[i] = (r < a.npad && r + 7 >= a.row_lo) ? r + 7 : -1;
            }

            for (int s = 0; s < nslab; s++, it++) {
                const int stage = it % P_STAGES;
                const uint32_t parity = (it / P_STAGES) & 1;
                const int k0 = s * P_BK;
                mbar_wait(full0 + 8 * stage, parity);
                const uint8_t* wsrc = Wst + stage * P_W_STAGE_BYTES + warp * 8 * 128;     // tile i adds i*8 warps*8 rows
                const double* psrc = Pst + stage * P_BN * P_PLD;
                const bool full = (k0 + P_BK <= row0) && (row0 + P_BM <= a.npad) && (row0 >= a.row_lo);
                if (full) {
                    double af[2][P_MI], bf[2][P_NI];
#pragma unroll
                    for (int i = 0; i < P_MI; i++)
                        af[0][i] = *reinterpret_cast<const double*>(wsrc + i * (P_CONSUMER_WARPS * 8 * 128) + aoff[0]);
#pragma unroll
                    for (int j = 0; j < P_NI; j++) bf[0][j] = psrc[(j * 8 + gq) * P_PLD + tq];
#pragma unroll
                    for (int ks = 0; ks < 4; ks++) {
                        const int cur = ks & 1, nxt = cur ^ 1;
                        if (ks < 3) {
#pragma unroll
                            for (int i = 0; i < P_MI; i++)
                                af[nxt][i] = *reinterpret_cast<const double*>(wsrc + i * (P_CONSUMER_WARPS * 8 * 128) + aoff[ks + 1]);
#pragma unroll
                            for (int j = 0; j < P_NI; j++) bf[nxt][j] = psrc[(j * 8 + gq) * P_PLD + (ks + 1) * 4 + tq];
                        }
#pragma unroll
                        for (int i = 0; i < P_MI; i++)
#pragma unroll
                            for (int j = 0; j < P_NI; j++) dmma884(acc[i][j][0], acc[i][j][1], af[cur][i], bf[cur][j]);
                    }
                } else {
#pragma unroll
                    for (int ks = 0; ks < 4; ks++) {
                        double bf[P_NI];
#pragma unroll
                        for (int j = 0; j < P_NI; j++) bf[j] = psrc[(j * 8 + gq) * P_PLD + ks * 4 + tq];
#pragma unroll
                        for (int i = 0; i < P_MI; i++) {
                            if (k0 + ks * 4 <= klim[i]) {   // warp-uniform
                                const double af =
                                    *reinterpret_cast<const double*>(wsrc + i * (P_CONSUMER_WARPS * 8 * 128) + aoff[ks]);
#pragma unroll
                                for (int j = 0; j < P_NI; j++) dmma884(acc[i][j][0], acc[i][j][1], af, bf[j]);
                            }
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(empty0 + 8 * stage);
            }

            // fold this row block of V into the column reductions (and the V cache if requested)
            double sq[P_NI][2], dt[P_NI][2];
#pragma unroll
            for (int j = 0; j < P_NI; j++) sq[j][0] = sq[j][1] = dt[j][0] = dt[j][1] = 0.0;
#pragma unroll
            for (int i = 0; i < P_MI; i++) {
                const int row = row0 + (i * P_CONSUMER_WARPS + warp) * 8 + pr;
                if (row < a.npad && row >= a.row_lo) {
                    const double zr = a.z[row];
#pragma unroll
                    for (int j = 0; j < P_NI; j++) {
                        const double v0 = acc[i][j][0], v1 = acc[i][j][1];
                        sq[j][0] += v0 * v0;
                        sq[j][1] += v1 * v1;
                        dt[j][0] += v0 * zr;
                        dt[j][1] += v1 * zr;
                        if (a.Vc != nullptr && row < N) {
                            const int64_t g = g0 + j * 8 + tq * 2;
                            double* dst = a.Vc + (int64_t)row * a.ldv + g;
                            if (g + 1 < a.G && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) {
                                *reinterpret_cast<double2*>(dst) = make_double2(v0, v1);
                            } else {
                                if (g < a.G) dst[0] = v0;
                                if (g + 1 < a.G) dst[1] = v1;
                            }
                        }
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < P_NI; j++)
#pragma unroll
                for (int c = 0; c < 2; c++) {
#pragma unroll
                    for (int o = 4; o < 32; o <<= 1) {
                        sq[j][c] += __shfl_xor_sync(0xffffffffu, sq[j][c], o);
                        dt[j][c] += __shfl_xor_sync(0xffffffffu, dt[j][c], o);
                    }
                }
            if (gq == 0) {
#pragma unroll
                for (int j = 0; j < P_NI; j++)
#pragma unroll
                    for (int c = 0; c < 2; c++) {
                        double* slot = colacc + (warp * P_BN + j * 8 + tq * 2 + c) * 2;
                        slot[0] += sq[j][c];
                        slot[1] += dt[j][c];
                    }
            }
        }
        // consumers only: named barrier 1 over the 256 consumer threads, then the final per-point results
        asm volatile("bar.sync 1, %0;\n" ::"n"(P_CONSUMER_WARPS * 32) : "memory");
        if (tid < P_BN) {
            const int64_t g = g0 + tid;
            if (g < a.G) {
                double s = 0.0, d = 0.0;
#pragma unroll
                for (int w = 0; w < P_CONSUMER_WARPS; w++) {
                    s += colacc[(w * P_BN + tid) * 2 + 0];
                    d += colacc[(w * P_BN + tid) * 2 + 1];
                }
                if (a.row_lo > 0) {      // incremental: the new rows' contributions are added to the standing posterior
                    a.var[g] -= s;
                    a.mu[g] += d;
                    if (a.qout) a.qout[g] += s;
                } else {
                    a.var[g] = p.k0 - s;
                    a.mu[g] = p.mean_H + d;
                    if (a.qout) a.qout[g] = s;
                }
            }
        }
    }
}

// ---- skinny incremental update ------------------------------------------------------------------------------------------
// After mfgp_cholesky_append only a few rows of V = W psi are new.  posterior_kernel's tile (512 rows x 32 points) would
// regenerate every psi element for 64 useful rows; here the CTA tile is 64 ROWS x 256 GRID POINTS instead: all eight
// consumer warps share the same 64 x 16 slab of W (one TMA box) and each owns 32 of the 256 points, so a psi element is
// still generated once per CTA and the register tile (8 x 4 DMMA tiles per warp) is the same.  Rows are processed in
// 64-row blocks [rb, rb+64) from the block that holds row_lo; each warp folds its own points -- no cross-warp reduction.
constexpr int U_BM = 64;
constexpr int U_BN = 256;
constexpr int U_W_STAGE_BYTES = U_BM * P_BK * 8;            // 8192
constexpr int U_PSI_STAGE_BYTES = U_BN * P_PLD * 8;         // 40960
constexpr int U_SMEM_BYTES = P_STAGES * (U_W_STAGE_BYTES + U_PSI_STAGE_BYTES) + U_BN * 4 * 8 + 2 * P_STAGES * 8 + 1024;

template <bool GRID>
__global__ void __launch_bounds__(P_THREADS, 1)
posterior_update_kernel(const __grid_constant__ CUtensorMap wmap, PostArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* Wst = smem;                                                        // [S][64][16] doubles, swizzled
    double* Pst = reinterpret_cast<double*>(smem + P_STAGES * U_W_STAGE_BYTES); // [S][256][20]
    double* xs = Pst + P_STAGES * U_BN * P_PLD;                                 // [256][4] scaled coordinates (general mode)
    int* offs = reinterpret_cast<int*>(xs);                                     // [256][2] table row offsets (grid mode)
    uint64_t* bars = reinterpret_cast<uint64_t*>(xs + U_BN * 4);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + P_STAGES);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t g0 = (GRID && a.remap_cols > 0)
                           ? (int64_t)(blockIdx.x % a.remap_cols) * a.ny + (int64_t)(blockIdx.x / a.remap_cols) * U_BN
                           : (int64_t)blockIdx.x * U_BN;
    const int N = a.NL + a.NH;
    const DevParams& p = a.p;

    if (tid == 0) {
        for (int s = 0; s < P_STAGES; s++) {
            mbar_init(full0 + 8 * s, P_PRODUCER_WARPS * 32);
            mbar_init(empty0 + 8 * s, P_CONSUMER_WARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    for (int e = tid; e < U_BN; e += P_THREADS) {
        int64_t g = g0 + e;
        if (g >= a.G) g = a.G - 1;
        if (GRID) {
            g += a.g_lo;
            offs[2 * e] = (int)((g / a.ny) * a.ldt);
            offs[2 * e + 1] = (int)((g % a.ny) * a.ldt);
        } else {
            const double x = a.Xs[2 * g], y = a.Xs[2 * g + 1];
            xs[e * 4 + 0] = x / p.l_L;
            xs[e * 4 + 1] = y / p.l_L;
            xs[e * 4 + 2] = x / p.l_H;
            xs[e * 4 + 3] = y / p.l_H;
        }
    }
    __syncthreads();

    const int rb0 = a.row_lo / U_BM * U_BM;

    if (warp >= P_CONSUMER_WARPS) {
        // =============================== PRODUCERS ===============================
        reg_dealloc<72>();
        const int pt = tid - P_CONSUMER_WARPS * 32;       // 0..127
        const int k = pt & 15;                            // column of the slab this thread generates
        const int gbase = pt >> 4;                        // points gbase + 8 i, i = 0..31
        // grid mode: the 256 consecutive x-major points of a CTA lie in at most two grid columns when ny >= 255; the
        // x-axis factors are then two values per training column (loaded once per slab) and only the y-axis factors
        // are fetched per element.  `second` marks this thread's points that lie in the second column.
        const int offx0 = GRID ? offs[0] : 0, offx1 = GRID ? offs[2 * (U_BN - 1)] : 0;
        bool two_col = GRID;
        unsigned second = 0;
        if (GRID) {
#pragma unroll 1
            for (int i = 0; i < U_BN / 8; i++) {
                const int ox = offs[2 * (gbase + 8 * i)];
                if (ox == offx1 && offx1 != offx0) second |= 1u << i;
                else if (ox != offx0) two_col = false;
            }
            two_col = __all_sync(0xffffffffu, two_col);      // (every producer thread reaches the same verdict per CTA
        }                                                     //  only if all see it: threads cover disjoint points)
        __shared__ int s_two_col;
        if (GRID) {
            if (pt == 0) s_two_col = 1;
            asm volatile("bar.sync 2, %0;\n" ::"n"(P_PRODUCER_WARPS * 32) : "memory");
            if (!two_col) s_two_col = 0;
            asm volatile("bar.sync 2, %0;\n" ::"n"(P_PRODUCER_WARPS * 32) : "memory");
            two_col = s_two_col != 0;
        }
        int it = 0;
        for (int rb = rb0; rb < a.npad; rb += U_BM) {
            const int nslab = (rb + U_BM) / P_BK;
            for (int s = 0; s < nslab; s++, it++) {
                const int stage = it % P_STAGES;
                const uint32_t parity = (it / P_STAGES) & 1;
                const int n = s * P_BK + k;
                double4 t = make_double4(0.0, 0.0, 0.0, 0.0);
                double lx0 = 0.0, hx0 = 0.0, lx1 = 0.0, hx1 = 0.0;
                if (GRID) {
                    if (two_col) {
                        lx0 = __ldg(a.TLx + offx0 + n); hx0 = __ldg(a.THx + offx0 + n);
                        lx1 = __ldg(a.TLx + offx1 + n); hx1 = __ldg(a.THx + offx1 + n);
                    }
                } else if (n < N) {
                    t = reinterpret_cast<const double4*>(a.Tt)[n];
                }
                mbar_wait(empty0 + 8 * stage, parity ^ 1);
                if (pt == 0) {
                    mbar_expect_tx(full0 + 8 * stage, U_W_STAGE_BYTES);
                    tma_load_2d(smem_u32(Wst + stage * U_W_STAGE_BYTES), &wmap, s * P_BK, rb, full0 + 8 * stage);
                }
                double* pdst = Pst + stage * U_BN * P_PLD;
                if (GRID && two_col) {
#pragma unroll 1
                    for (int i0 = 0; i0 < U_BN / 8; i0 += 8) {
                        double ly[8], hy[8];
#pragma unroll
                        for (int u = 0; u < 8; u++) {        // all loads of the batch first: their latencies overlap
                            const int oy = offs[2 * (gbase + 8 * (i0 + u)) + 1] + n;
                            ly[u] = __ldg(a.TLy + oy);
                            hy[u] = __ldg(a.THy + oy);
                        }
#pragma unroll
                        for (int u = 0; u < 8; u++) {
                            const bool sec = (second >> (i0 + u)) & 1u;
                            pdst[(gbase + 8 * (i0 + u)) * P_PLD + k] = fma(sec ? hx1 : hx0, hy[u], (sec ? lx1 : lx0) * ly[u]);
                        }
                    }
                } else {
#pragma unroll 2
                    for (int i = 0; i < U_BN / 8; i++) {
                        const int gi = gbase + 8 * i;
                        double v = 0.0;
                        if (GRID) {
                            const int ox = offs[2 * gi] + n, oy = offs[2 * gi + 1] + n;
                            v = fma(__ldg(a.THx + ox), __ldg(a.THy + oy), __ldg(a.TLx + ox) * __ldg(a.TLy + oy));
                        } else if (n < N) {
                            if (p.multi) {
                                const double kL = rbf_scaled(xs[gi * 4 + 0], xs[gi * 4 + 1], t.x, t.y, p.s_L);
                                if (n < a.NL) {
                                    v = p.rho * kL;
                                } else {
                                    const double kH = rbf_scaled(xs[gi * 4 + 2], xs[gi * 4 + 3], t.z, t.w, p.s_H);
                                    v = __dadd_rn(__dmul_rn(p.rho2, kL), kH);
                                }
                            } else {
                                v = rbf_scaled(xs[gi * 4 + 2], xs[gi * 4 + 3], t.z, t.w, p.s_H);
                            }
                        }
                        pdst[gi * P_PLD + k] = v;
                    }
                }
                mbar_arrive(full0 + 8 * stage);
            }
        }
    } else {
        // =============================== CONSUMERS ===============================
        reg_alloc<216>();
        const int gq = lane >> 2, tq = lane & 3;
        const int pr = row_perm(gq);
        int aoff[4];
#pragma unroll
        for (int j = 0; j < 4; j++) aoff[j] = pr * 128 + ((((j * 4 + tq) >> 1) ^ pr) << 4) + ((tq & 1) << 3);
        double sq[P_NI][2], dt[P_NI][2];
#pragma unroll
        for (int j = 0; j < P_NI; j++) sq[j][0] = sq[j][1] = dt[j][0] = dt[j][1] = 0.0;
        int it = 0;
        for (int rb = rb0; rb < a.npad; rb += U_BM) {
            const int nslab = (rb + U_BM) / P_BK;
            double acc[P_MI][P_NI][2];
#pragma unroll
            for (int i = 0; i < P_MI; i++)
#pragma unroll
                for (int j = 0; j < P_NI; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
            for (int s = 0; s < nslab; s++, it++) {
                const int stage = it % P_STAGES;
                const uint32_t parity = (it / P_STAGES) & 1;
                mbar_wait(full0 + 8 * stage, parity);
                const uint8_t* wsrc = Wst + stage * U_W_STAGE_BYTES;                     // tile i: rows 8 i .. 8 i + 7
                const double* psrc = Pst + stage * U_BN * P_PLD + warp * 32 * P_PLD;     // this warp's 32 points
                double af[2][P_MI], bf[2][P_NI];
#pragma unroll
                for (int i = 0; i < P_MI; i++) af[0][i] = *reinterpret_cast<const double*>(wsrc + i * (8 * 128) + aoff[0]);
#pragma unroll
                for (int j = 0; j < P_NI; j++) bf[0][j] = psrc[(j * 8 + gq) * P_PLD + tq];
#pragma unroll
                for (int ks = 0; ks < 4; ks++) {
                    const int cur = ks & 1, nxt = cur ^ 1;
                    if (ks < 3) {
#pragma unroll
                        for (int i = 0; i < P_MI; i++)
                            af[nxt][i] = *reinterpret_cast<const double*>(wsrc + i * (8 * 128) + aoff[ks + 1]);
#pragma unroll
                        for (int j = 0; j < P_NI; j++) bf[nxt][j] = psrc[(j * 8 + gq) * P_PLD + (ks + 1) * 4 + tq];
                    }
#pragma unroll
                    for (int i = 0; i < P_MI; i++)
#pragma unroll
                        for (int j = 0; j < P_NI; j++) dmma884(acc[i][j][0], acc[i][j][1], af[cur][i], bf[cur][j]);
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(empty0 + 8 * stage);
            }
            // fold the new rows of this block into the per-point sums
#pragma unroll
            for (int i = 0; i < P_MI; i++) {
                const int row = rb + i * 8 + pr;
                if (row >= a.row_lo && row < a.npad) {
                    const double zr = a.z[row];
#pragma unroll
                    for (int j = 0; j < P_NI; j++) {
                        const double v0 = acc[i][j][0], v1 = acc[i][j][1];
                        sq[j][0] += v0 * v0;
                        sq[j][1] += v1 * v1;
                        dt[j][0] += v0 * zr;
                        dt[j][1] += v1 * zr;
                    }
                }
            }
        }
#pragma unroll
        for (int j = 0; j < P_NI; j++)
#pragma unroll
            for (int c = 0; c < 2; c++) {
#pragma unroll
                for (int o = 4; o < 32; o <<= 1) {
                    sq[j][c] += __shfl_xor_sync(0xffffffffu, sq[j][c], o);
                    dt[j][c] += __shfl_xor_sync(0xffffffffu, dt[j][c], o);
                }
            }
        if (gq == 0) {
#pragma unroll
            for (int j = 0; j < P_NI; j++)
#pragma unroll
                for (int c = 0; c < 2; c++) {
                    const int64_t g = g0 + warp * 32 + j * 8 + tq * 2 + c;
                    if (g < a.G) {
                        a.var[g] -= sq[j][c];
                        a.mu[g] += dt[j][c];
                        if (a.qout) a.qout[g] += sq[j][c];
                    }
                }
        }
    }
}

__global__ void posterior_prior_kernel(int64_t G, double mean, double k0, double* __restrict__ mu, double* __restrict__ var,
                                       double* __restrict__ q) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g < G) {
        mu[g] = mean;
        var[g] = k0;
        if (q) q[g] = 0.0;
    }
}

// Per-axis factor tables of the separable RBF kernel on a tensor-product grid.  For axis value u and training point n:
//   TL[u][n] = cL[n] * exp(-0.5 (u/l_L - X_n/l_L)^2)  (x axis; the y-axis table carries no coefficient)
// with cL = rho*s_L for lofi columns, rho^2*s_L for hifi columns (MF), 0 for SF / padding; cH = s_H for hifi, else 0.
// exp(a)exp(b) replaces the reference's exp(a+b) (gaussian_process.py:79): a few ulp, far inside the 1e-9 tolerance.
__global__ void grid_tables_kernel(const double* __restrict__ u, int nu, int axis, const double* __restrict__ Tt, int NL, int NH,
                                   int npad, DevParams p, double* __restrict__ TL, double* __restrict__ TH, int64_t ldt) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    const int iu = blockIdx.y;
    if (n >= npad || iu >= nu) return;
    const int N = NL + NH;
    double vl = 0.0, vh = 0.0;
    if (n < N) {
        const double4 t = reinterpret_cast<const double4*>(Tt)[n];
        const double uv = u[iu];
        const double dl = uv / p.l_L - (axis == 0 ? t.x : t.y);
        const double dh = uv / p.l_H - (axis == 0 ? t.z : t.w);
        const bool lo = n < NL;
        if (p.multi) vl = exp(-0.5 * (dl * dl)) * (axis == 0 ? (lo ? p.rho * p.s_L : p.rho2 * p.s_L) : 1.0);
        if (!lo) vh = exp(-0.5 * (dh * dh)) * (axis == 0 ? p.s_H : 1.0);
    }
    TL[(int64_t)iu * ldt + n] = vl;
    TH[(int64_t)iu * ldt + n] = vh;
}

// 16 doubles (128 B) x 256 (or 64) rows of W per box; out-of-range rows read as zero
static int make_w_tensor_map(CUtensorMap* map, const double* W, int64_t npad, int64_t ldw, int box_rows = P_BM / 2) {
    return make_tensor_map_2d(map, W, npad, npad, ldw, P_BK, box_rows, CU_TENSOR_MAP_SWIZZLE_128B);
}

}  // namespace mfgp

using namespace mfgp;

static int posterior_common(PostArgs& a, bool grid, const double* W, int64_t npad, int64_t ldw, const mfgp_params* p_host,
                            cudaStream_t st) {
    const DevParams dp = make_dev_params(*p_host);
    a.p = dp;
    const int64_t N = (int64_t)a.NL + a.NH;
    if (N == 0) {   // empty model: constant mean and prior variance (gaussian_process.py:139-146 with no data)
        posterior_prior_kernel<<<(unsigned)((a.G + 255) / 256), 256, 0, st>>>(a.G, dp.mean_H, dp.k0, a.mu, a.var, a.qout);
        MFGP_LAUNCH_CHECK();
        return MFGP_OK;
    }
    if (!W || !a.z || npad < N || npad % MFGP_TILE || ldw < npad) return MFGP_ERR_INVALID;
    if ((reinterpret_cast<uintptr_t>(W) & 15) || (ldw & 1)) return MFGP_ERR_INVALID;     // TMA: 16-byte aligned rows
    if (!p_host->multi && a.NL != 0) return MFGP_ERR_INVALID;
    if (a.Vc && a.ldv < a.G) return MFGP_ERR_INVALID;
    if (a.row_lo < 0 || a.row_lo >= N) return MFGP_ERR_INVALID;
    CUtensorMap wmap;
    a.npad = (int)npad;
    const bool whole_cols = grid && a.ny > 0 && a.g_lo % a.ny == 0 && a.G % a.ny == 0;
    if (a.row_lo > 0 && a.Vc == nullptr && npad - a.row_lo / U_BM * U_BM <= 4 * U_BM) {
        a.remap_cols = (whole_cols && a.ny % U_BN == 0) ? (int)(a.G / a.ny) : 0;
        // few new rows: the 64-row x 256-point tiling keeps the psi regeneration amortised
        int rcu = make_w_tensor_map(&wmap, W, npad, ldw, U_BM);
        if (rcu) return rcu;
        const unsigned nb = (unsigned)((a.G + U_BN - 1) / U_BN);
        if (grid) {
            MFGP_CUDA_CHECK(cudaFuncSetAttribute(posterior_update_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, U_SMEM_BYTES));
            posterior_update_kernel<true><<<nb, P_THREADS, U_SMEM_BYTES, st>>>(wmap, a);
        } else {
            MFGP_CUDA_CHECK(cudaFuncSetAttribute(posterior_update_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, U_SMEM_BYTES));
            posterior_update_kernel<false><<<nb, P_THREADS, U_SMEM_BYTES, st>>>(wmap, a);
        }
        MFGP_LAUNCH_CHECK();
        return MFGP_OK;
    }
    int rc = make_w_tensor_map(&wmap, W, npad, ldw);
    if (rc) return rc;
    a.remap_cols = (whole_cols && a.ny % P_BN == 0) ? (int)(a.G / a.ny) : 0;
    const unsigned nblk = (unsigned)((a.G + P_BN - 1) / P_BN);
    if (grid) {
        MFGP_CUDA_CHECK(cudaFuncSetAttribute(posterior_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, P_SMEM_BYTES));
        posterior_kernel<true><<<nblk, P_THREADS, P_SMEM_BYTES, st>>>(wmap, a);
    } else {
        MFGP_CUDA_CHECK(cudaFuncSetAttribute(posterior_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, P_SMEM_BYTES));
        posterior_kernel<false><<<nblk, P_THREADS, P_SMEM_BYTES, st>>>(wmap, a);
    }
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

extern "C" int mfgp_posterior(const double* Xs, int64_t G, const double* Tt, int64_t NL, int64_t NH, const double* W,
                              int64_t npad, int64_t ldw, const double* z, const mfgp_params* p_host, double* mu,
                              double* var, double* qred, double* Vc, int64_t ldv, void* stream) {
    if (!p_host || !mu || !var || G < 0 || NL < 0 || NH < 0) return MFGP_ERR_INVALID;
    if (G == 0) return MFGP_OK;
    if (!Xs || (NL + NH > 0 && !Tt)) return MFGP_ERR_INVALID;
    PostArgs a{};
    a.Xs = Xs; a.G = G; a.Tt = Tt; a.NL = (int)NL; a.NH = (int)NH; a.z = z; a.mu = mu; a.var = var; a.qout = qred; a.Vc = Vc; a.ldv = ldv;
    return posterior_common(a, false, W, npad, ldw, p_host, static_cast<cudaStream_t>(stream));
}

extern "C" int mfgp_grid_tables(const double* ux, int64_t nx, const double* uy, int64_t ny, const double* Tt, int64_t NL,
                                int64_t NH, int64_t npad, const mfgp_params* p_host, double* TLx, double* TLy, double* THx,
                                double* THy, int64_t ldt, void* stream) {
    if (!ux || !uy || !Tt || !p_host || !TLx || !TLy || !THx || !THy || nx <= 0 || ny <= 0 || npad < NL + NH || ldt < npad)
        return MFGP_ERR_INVALID;
    if (nx * ldt >= (1LL << 31) || ny * ldt >= (1LL << 31)) return MFGP_ERR_INVALID;   // kernel uses 32-bit table offsets
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const DevParams dp = make_dev_params(*p_host);
    dim3 gx((unsigned)((npad + 127) / 128), (unsigned)nx), gy((unsigned)((npad + 127) / 128), (unsigned)ny);
    grid_tables_kernel<<<gx, 128, 0, st>>>(ux, (int)nx, 0, Tt, (int)NL, (int)NH, (int)npad, dp, TLx, THx, ldt);
    MFGP_LAUNCH_CHECK();
    grid_tables_kernel<<<gy, 128, 0, st>>>(uy, (int)ny, 1, Tt, (int)NL, (int)NH, (int)npad, dp, TLy, THy, ldt);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

extern "C" int mfgp_posterior_grid(int64_t ny, int64_t g_lo, int64_t G, const double* TLx, const double* TLy,
                                   const double* THx, const double* THy, int64_t ldt, int64_t NL, int64_t NH,
                                   const double* W, int64_t npad, int64_t ldw, const double* z, const mfgp_params* p_host,
                                   double* mu, double* var, double* qred, double* Vc, int64_t ldv, void* stream) {
    if (!p_host || !mu || !var || G < 0 || NL < 0 || NH < 0 || ny <= 0 || g_lo < 0) return MFGP_ERR_INVALID;
    if (G == 0) return MFGP_OK;
    if (NL + NH > 0 && (!TLx || !TLy || !THx || !THy || ldt < npad)) return MFGP_ERR_INVALID;
    PostArgs a{};
    a.G = G; a.TLx = TLx; a.TLy = TLy; a.THx = THx; a.THy = THy; a.ldt = ldt; a.g_lo = g_lo; a.ny = (int)ny;
    a.NL = (int)NL; a.NH = (int)NH; a.z = z; a.mu = mu; a.var = var; a.qout = qred; a.Vc = Vc; a.ldv = ldv;
    return posterior_common(a, true, W, npad, ldw, p_host, static_cast<cudaStream_t>(stream));
}

// Incremental forms: rows [row_lo, N) of V = W psi are new since mu / var (/ qred) were last computed -- samples appended
// by mfgp_cholesky_append -- and only their contributions are formed and added:  mu += v_new . z_new,  var -= |v_new|^2.
extern "C" int mfgp_posterior_update(const double* Xs, int64_t G, const double* Tt, int64_t NL, int64_t NH, const double* W,
                                     int64_t npad, int64_t ldw, const double* z, const mfgp_params* p_host, int64_t row_lo,
                                     double* mu, double* var, double* qred, double* Vc, int64_t ldv, void* stream) {
    if (!p_host || !mu || !var || G < 0 || NL < 0 || NH < 0 || row_lo <= 0 || row_lo >= NL + NH) return MFGP_ERR_INVALID;
    if (G == 0) return MFGP_OK;
    if (!Xs || !Tt) return MFGP_ERR_INVALID;
    PostArgs a{};
    a.Xs = Xs; a.G = G; a.Tt = Tt; a.NL = (int)NL; a.NH = (int)NH; a.z = z; a.mu = mu; a.var = var; a.qout = qred; a.Vc = Vc; a.ldv = ldv;
    a.row_lo = (int)row_lo;
    return posterior_common(a, false, W, npad, ldw, p_host, static_cast<cudaStream_t>(stream));
}

extern "C" int mfgp_posterior_grid_update(int64_t ny, int64_t g_lo, int64_t G, const double* TLx, const double* TLy,
                                          const double* THx, const double* THy, int64_t ldt, int64_t NL, int64_t NH,
                                          const double* W, int64_t npad, int64_t ldw, const double* z, const mfgp_params* p_host,
                                          int64_t row_lo, double* mu, double* var, double* qred, double* Vc, int64_t ldv,
                                          void* stream) {
    if (!p_host || !mu || !var || G < 0 || NL < 0 || NH < 0 || ny <= 0 || g_lo < 0 || row_lo <= 0 || row_lo >= NL + NH)
        return MFGP_ERR_INVALID;
    if (G == 0) return MFGP_OK;
    if (!TLx || !TLy || !THx || !THy || ldt < npad) return MFGP_ERR_INVALID;
    PostArgs a{};
    a.G = G; a.TLx = TLx; a.TLy = TLy; a.THx = THx; a.THy = THy; a.ldt = ldt; a.g_lo = g_lo; a.ny = (int)ny;
    a.NL = (int)NL; a.NH = (int)NH; a.z = z; a.mu = mu; a.var = var; a.qout = qred; a.Vc = Vc; a.ldv = ldv;
    a.row_lo = (int)row_lo;
    return posterior_common(a, true, W, npad, ldw, p_host, static_cast<cudaStream_t>(stream));
}
