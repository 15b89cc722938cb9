// GP fit on the device: training covariance, blocked Cholesky, triangular inverse, whitened observations.
// Replaces SFGP.updt_info (reference gaussian_process.py:229-255) and MFGP.updt_info (:493-529).
#include "common.cuh"
#include "gemm_f64.cuh"
#include <cstdlib>
#include <mutex>

namespace mfgp {

// ---- K assembly ------------------------------------------------------------------------------------------------------
// K_LL = k_L + noise_L I, K_LH = rho k_L, K_HH = rho^2 k_L + k_H + noise_H I, then + jitter I (gaussian_process.py:
// 523-529); SF: k + noise I + jitter I (:253-254).  Padding rows/cols [N, npad) carry the identity.  K is symmetric and
// the factorisation reads its lower triangle only, so tiles strictly above the diagonal are left untouched.
// Tt[i] = (x_i / l_L, y_i / l_L, x_i / l_H, y_i / l_H): the operands of rbf_scaled, divided ONCE per training point (the same
// IEEE divisions the reference performs per pair, gaussian_process.py:75-79) -- the covariance assembly then has no division left.
__global__ void scaled_coords_kernel(const double* __restrict__ Xt, int N, int npad, DevParams p, double* __restrict__ Tt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npad) return;
    double4 t = make_double4(0.0, 0.0, 0.0, 0.0);
    if (i < N) {
        const double xi = Xt[2 * i], yi = Xt[2 * i + 1];
        t = make_double4(xi / p.l_L, yi / p.l_L, xi / p.l_H, yi / p.l_H);
    }
    reinterpret_cast<double4*>(Tt)[i] = t;
}

// Tt != nullptr: the pre-divided coordinates (scaled_coords_kernel ran before); nullptr: divide here.
__global__ void build_train_cov_kernel(const double* __restrict__ Xt, int NL, int NH, DevParams p, double* __restrict__ K,
                                       int npad, int64_t ld, const double* __restrict__ Tt, int row_begin) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = row_begin + blockIdx.y * blockDim.y + threadIdx.y;
    const int N = NL + NH;
    if (i >= npad || j >= npad) return;
    if (j >= ((i >> 6) + 1) * 64) return;      // only the 64x64 tiles on or below the diagonal are ever read
    double v;
    if (i >= N || j >= N) {
        v = (i == j) ? 1.0 : 0.0;
    } else {
        double4 a, b;          // (x / l_L, y / l_L, x / l_H, y / l_H) of points i and j
        if (Tt != nullptr) {
            a = reinterpret_cast<const double4*>(Tt)[i];
            b = reinterpret_cast<const double4*>(Tt)[j];
        } else {
            const double xi = Xt[2 * i], yi = Xt[2 * i + 1], xj = Xt[2 * j], yj = Xt[2 * j + 1];
            a = make_double4(xi / p.l_L, yi / p.l_L, xi / p.l_H, yi / p.l_H);
            b = make_double4(xj / p.l_L, yj / p.l_L, xj / p.l_H, yj / p.l_H);
        }
        const bool iL = i < NL, jL = j < NL;
        if (p.multi) {
            const double kL = rbf_scaled(a.x, a.y, b.x, b.y, p.s_L);
            if (iL && jL) {
                v = kL;
                if (i == j) v = v + p.noise_L;
            } else if (iL != jL) {
                v = p.rho * kL;
            } else {
                const double kH = rbf_scaled(a.z, a.w, b.z, b.w, p.s_H);
                v = __dadd_rn(__dmul_rn(p.rho2, kL), kH);
                if (i == j) v = v + p.noise_H;
            }
        } else {
            v = rbf_scaled(a.z, a.w, b.z, b.w, p.s_H);
            if (i == j) v = v + p.noise_H;
        }
        if (i == j) v = v + p.jitter;
    }
    K[(int64_t)i * ld + j] = v;
}

// ---- 64x64 diagonal block: Cholesky + inverse in one CTA --------------------------------------------------------------
// 256 threads as a 16x16 grid; thread (ti, tc) keeps the 4x4 cyclic sub-blocks S[ti+16a][tc+16b] and M[ti+16a][tc+16b]
// in REGISTERS.  The sweep is bound by one serial chain per step (barrier -> read pivot -> reciprocal -> scale -> FMA ->
// publish, ~20-cycle FP64 latencies: profiles/r01_fp64_latency.log), so it eliminates TWO columns per step and keeps
// square roots off the chain altogether:
//   step k (columns j0 = 2k, j1 = j0+1): the owners publish the two UNSCALED columns U = [u1 u2] (as they stand after the
//   earlier steps); P = [[a, b], [b, c]] is their 2x2 pivot block; every thread forms P^-1 from ONE reciprocal
//   (1 / (ac - b^2)) and applies the rank-2 update S -= (U P^-1) U^T to its registers.
// Inverse: carried along in the same sweep -- M starts as the identity and, with rows j0, j1 of M published next to the
// columns, the rows below take M_i -= (U_i P^-1) [M_j0; M_j1].
// Afterwards, with C = chol(P) per pair (32 independent 2x2 factors, computed in parallel),
//   L[:, pair] = U C^-T     and     W[pair, :] = C^-1 M[pair, :]         (W = L^-1),
// i.e. even columns / rows are scaled by 1/sqrt(a), odd ones take (x_odd - (b/a) x_even) / sqrt(c - b^2/a); the even
// partner sits in the neighbouring lane (columns) or 16 lanes away (rows).  No divide or sqrt other than these.
// Pivot test as in LAPACK potrf (np.linalg.cholesky raises, gaussian_process.py:254 / :529): a > 0, then c - b^2/a > 0.
constexpr int PB = 64;
constexpr int PLD = PB + 1;

struct PotrfScratch {
    double2 colAB[2][PB], rowAB[2][PB];   // (.x, .y) = (column j0, column j1) of S / (row j0, row j1) of M
    double piv[3][PB / 2];                // a, b, c of every pivot block
    double fin[3][PB / 2];                // 1/sqrt(a), 1/sqrt(c - b^2/a), b/a
    int bad;
};

// BS = 64: the whole tile (s, m: 4x4 cyclic sub-blocks per thread); BS = 32: one half of the two-level form below (2x2).
// `col0`: global index of the block's first column (for the failing-pivot report).  Ls / Wsm (optional, shared memory, row
// stride lds_out): copies of L and of its inverse for the caller's next step.
// Barrier of the 256 threads that work on a tile: the whole CTA of potrf_diag_kernel and chol_dataflow_cpasync_kernel, the
// consumer warps of chol_dataflow_kernel (whose ninth warp, the producer, does not take part in the epilogue).
__device__ __forceinline__ void tile_bar() { asm volatile("bar.sync 1, 256;\n" ::: "memory"); }

template <int BS>
__device__ __forceinline__ void potrf_diag_body(const double* src, int64_t lds, double* A, int64_t ld,
                                                double* __restrict__ Winv, int64_t ldw, int32_t* __restrict__ info, int col0,
                                                PotrfScratch* sc, double* Lsm = nullptr, double* Wsm = nullptr, int lds_out = 0) {
    constexpr int NB = BS / 16;
    double2 (*colAB)[PB] = sc->colAB;
    double2 (*rowAB)[PB] = sc->rowAB;
    double (*piv)[PB / 2] = sc->piv;
    double (*fin)[PB / 2] = sc->fin;
    int& bad = sc->bad;
    const int tid = threadIdx.x;
    const int ti = tid >> 4, tc = tid & 15;
    if (tid == 0) bad = 0;
    double s[NB][NB], m[NB][NB];
#pragma unroll
    for (int a = 0; a < NB; a++)
#pragma unroll
        for (int b = 0; b < NB; b++) {
            const int r = ti + 16 * a, c = tc + 16 * b;
            s[a][b] = (c <= r) ? src[(int64_t)r * lds + c] : 0.0;
            m[a][b] = (r == c) ? 1.0 : 0.0;
        }
#pragma unroll
    for (int jb = 0; jb < NB; jb++) {
#pragma unroll 1
        for (int jp = 0; jp < 8; jp++) {
            const int k = jb * 8 + jp, j0 = 2 * k, j1 = j0 + 1, jj0 = 2 * jp, buf = k & 1;
            if ((tc & 14) == jj0) {          // owners of columns j0 (tc even) and j1 (tc odd); rows above are never read
                double* dst = reinterpret_cast<double*>(colAB[buf]) + (tc & 1);
#pragma unroll
                for (int a = 0; a < NB; a++) dst[2 * (ti + 16 * a)] = s[a][jb];
            }
            if ((ti & 14) == jj0) {          // owners of rows j0, j1 of M
                double* dst = reinterpret_cast<double*>(rowAB[buf]) + (ti & 1);
#pragma unroll
                for (int b = 0; b < NB; b++) dst[2 * (tc + 16 * b)] = m[jb][b];
            }
            tile_bar();
            const double2* col = colAB[buf];
            const double2* row = rowAB[buf];
            double pa = col[j0].x;
            const double2 p1 = col[j1];
            double pb = p1.x, pc = p1.y;
            double det = fma(pa, pc, -(pb * pb));
            if (!(pa > 0.0) || !(det > 0.0)) {          // uniform
                if (tid == 0 && !bad) {
                    bad = 1;
                    atomicCAS(info, 0, col0 + ((pa > 0.0) ? j1 : j0) + 1);
                }
                pa = 1.0; pb = 0.0; pc = 1.0; det = 1.0;
            }
            if (tid == 0) { piv[0][k] = pa; piv[1][k] = pb; piv[2][k] = pc; }
            const double idet = 1.0 / det;
            const double qa = pc * idet, qb = -pb * idet, qc = pa * idet;      // P^-1
            double t1[NB], t2[NB];
#pragma unroll
            for (int a = 0; a < NB; a++) {
                if (a < jb) continue;                       // rows of earlier 16-groups are final
                const double2 x = col[ti + 16 * a];
                t1[a] = fma(qa, x.x, qb * x.y);
                t2[a] = fma(qb, x.x, qc * x.y);
            }
#pragma unroll
            for (int b = 0; b < NB; b++) {
                if (b < jb) continue;                       // columns of earlier 16-groups are final
                const double2 y = col[tc + 16 * b];
                const bool live = tc + 16 * b > j1;         // only columns right of the pair change
#pragma unroll
                for (int a = 0; a < NB; a++) {
                    if (a < b) continue;                    // register groups strictly above the diagonal are never read
                    if (live) s[a][b] = fma(-t1[a], y.x, fma(-t2[a], y.y, s[a][b]));
                }
            }
#pragma unroll
            for (int b = 0; b < NB; b++) {
                if (b > jb) continue;                       // rows j0, j1 of M are zero right of column j1
                const double2 z = row[tc + 16 * b];
#pragma unroll
                for (int a = 0; a < NB; a++) {
                    if (a < jb) continue;                   // rows of earlier 16-groups are final
                    const bool live = ti + 16 * a > j1;     // only rows below the pair change
                    if (live) m[a][b] = fma(-t1[a], z.x, fma(-t2[a], z.y, m[a][b]));
                }
            }
        }
    }
    tile_bar();
    if (tid < BS / 2) {          // C = chol(P) of every pair
        const double a = piv[0][tid], b = piv[1][tid], c = piv[2][tid];
        const double r1 = rsqrt(a);
        const double g = b * r1 * r1;
        fin[0][tid] = r1;
        fin[1][tid] = rsqrt(fma(-g, b, c));
        fin[2][tid] = g;
    }
    tile_bar();
    const bool failed = bad != 0;
#pragma unroll
    for (int a = 0; a < NB; a++)
#pragma unroll
        for (int b = 0; b < NB; b++) {
            const int r = ti + 16 * a, c = tc + 16 * b;
            const double v = s[a][b], w = m[a][b];
            const double vp = __shfl_up_sync(0xffffffffu, v, 1);       // same row, column c-1
            const double wp = __shfl_up_sync(0xffffffffu, w, 16);      // row r-1, same column
            const int kc = c >> 1, kr = r >> 1;
            const double lv = (c & 1) ? (v - fin[2][kc] * vp) * fin[1][kc] : v * fin[0][kc];
            const double wv = (r & 1) ? (w - fin[2][kr] * wp) * fin[1][kr] : w * fin[0][kr];
            // on failure leave a harmless identity so later kernels stay finite; the host raises on `info`
            const double lo = failed ? ((r == c) ? 1.0 : 0.0) : ((c <= r) ? lv : 0.0);
            const double wo = failed ? ((r == c) ? 1.0 : 0.0) : ((c <= r) ? wv : 0.0);
            if (c <= r) A[(int64_t)r * ld + c] = lo;
            if (Winv != nullptr) Winv[(int64_t)r * ldw + c] = wo;
            if (Lsm != nullptr) Lsm[r * lds_out + c] = lo;
            if (Wsm != nullptr) Wsm[r * lds_out + c] = wo;
        }
}

__global__ void __launch_bounds__(256, 1) potrf_diag_kernel(double* __restrict__ A, int64_t ld, double* __restrict__ Winv,
                                                         int64_t ldw, int32_t* __restrict__ info, int jblk) {
    __shared__ __align__(16) PotrfScratch scratch;
    potrf_diag_body<PB>(A, ld, A, ld, Winv, ldw, info, jblk * PB, &scratch);
}

// ---- tiled Cholesky + forward substitution as ONE persistent dataflow kernel -----------------------------------------
// The launch-per-panel chain (potrf -> panel solve -> trailing update, three dependent kernels per 64 columns) is bound
// by launch and drain latency, not by flops.  Here every 64x64 tile of L (and of Y = L^-1 B) is one task; CTAs draw
// tasks from a ticket counter and synchronise through per-tile ready flags in global memory.  Left-looking: a task
// accumulates its sum over the earlier block columns k in registers AS the tiles L_*k become ready, so that when the
// diagonal block of its own column is finally factored only one 64^3 product remains:
//   L tile (i, c), i >= c+2:  L_ic = (A_ic - sum_{k<c} L_ik L_ck^T) W_cc^T
//   Y tile (c, r):            Y_cr = W_cc (B_cr - sum_{k<c} L_ck Y_kr)
//   chain task d (the critical path, ONE hop per block column): accumulates BOTH the sub-diagonal tile (d, d-1) and the
//                             diagonal tile (d, d) over k < d-1 (they share the A operand L_dk); when W_{d-1,d-1} is
//                             flagged it forms L_{d,d-1} = X W^T, subtracts L_{d,d-1} L_{d,d-1}^T from the diagonal tile
//                             out of shared memory, and factors + inverts it in place (two 32x32 halves, potrf_diag_body) -> W_dd.
//   Gram task (g, ti, tj) (optional, mfgp_cholesky_solve_gram): adds the block rows of group g of the SOLVED right-hand sides to
//                             tile (ti, tj) of M = Y^T Y, in place, groups in order; a second, low-priority ticket queue.
// Ticket order: chain 0; then per block column c: the chain tasks placed there (chain d sits d / chain_la columns ahead of
// column d - 1), the tiles (i, c) below the sub-diagonal, the Y tiles of block row c.
// A task other than an early chain task waits only on tasks with a SMALLER ticket, a CTA holds a ticket only while it is
// resident, and at most nb / chain_la + 2 CTAs can hold early chain tasks, so the scheme cannot deadlock; a Gram ticket is
// run only once every task its rows depend on has been drawn (oracle/tiled_cholesky.py restates both arguments and simulates
// them); a bounded spin (abort flag) guards against bugs all the same.
// Two CTAs share an SM; while one of them runs the latency-bound tail of a chain task it raises a per-SM pause flag and
// the other one idles between its k slabs (its DMMA traffic would otherwise stretch the chain by ~25%).
// Two forms of the kernel run the same task body (below) with different k loops.  chol_dataflow_cpasync_kernel: 256 threads
// stage each slab with cp.async and meet at one barrier per slab.  chol_dataflow_kernel, warp-specialised: 8 consumer warps
// run the DMMA loops and the epilogues; a ninth, producer warp draws the tickets, polls
// the tile flags and moves every slab with ONE 2D TMA copy per operand into a 3-slot ring (full / empty mbarriers), so the
// k loop has no CTA-wide barrier and no per-thread copy issue.  The TMA boxes are 4 doubles wider than the slab: the
// 4 columns past it land as the row padding that puts the 8 rows of a DMMA
// fragment read on distinct bank groups, so the slabs keep the padded layout the fragment reads are laid out for.  Those 4
// columns belong to the neighbouring k tile (Y tile, W block), whose flag has not been acquired and which another CTA may be
// writing at that moment: the copy may read in-flight data there.  That is intended -- no padding element is ever read.
constexpr int DF_K = 32;                 // K slab
constexpr int DF_LDA = DF_K + 4;         // [m][k] / [n][k] slabs: rows land on distinct 8-bank groups
constexpr int DF_LDT = PB + 4;           // [k][n] slabs and the 64x64 epilogue tiles
constexpr int DF_STAGE = PB * DF_LDA;    // doubles per operand per stage (64 x 36 = 2304 >= 32 x 68 = 2176)
constexpr int DF_TILE = PB * DF_LDT;     // one padded 64x64 tile
constexpr int DF_NSTAGE = 3;             // slabs in flight: one slab of compute (~0.5 us) does not cover an L2 round trip under load
constexpr int DF_SMEM_DOUBLES = DF_NSTAGE * 2 * DF_STAGE;     // 3 stages x (A, B) = 13824 doubles >= epilogue X, W, L tiles (13056)
constexpr int DF_SMEM_BYTES = DF_SMEM_DOUBLES * 8 + 128;      // + slack to align the TMA destinations to 128 bytes
constexpr int DF_THREADS = 256;                               // consumer threads
constexpr int DF_CTA_THREADS = DF_THREADS + 32;               // + the producer warp
constexpr uint32_t DF_MK_BYTES = PB * DF_LDA * 8;             // TMA box of an [m][k] / [n][k] slab (36 x 64 doubles)
constexpr uint32_t DF_KN_BYTES = DF_K * DF_LDT * 8;           // TMA box of a [k][n] slab (68 x 32 doubles)
constexpr uint32_t DF_TILE_BYTES = PB * DF_LDT * 8;           // TMA box of the epilogue's W_cc tile (68 x 64 doubles)
// Factorisations of fewer block columns (npad <= 2048: c2, c3) are bound by the chain of diagonal blocks and run the cp.async
// form of the kernel (chol_dataflow_cpasync_kernel).  Measured on a B200, cp.async vs TMA: N = 1024 0.298 vs 0.313 ms; N = 2048
// R = 0 0.610 vs 0.614 ms, R = 512 0.627 vs 0.621 ms; N = 4096 7-10 % faster with TMA
constexpr int DF_TMA_MIN_NB = 33;

struct DfArgs {
    double* K; int64_t ld;
    double* W; int64_t ldw;
    double* Bm; int64_t ldb;
    int nb, nr;
    int32_t* info;
    int* flagsL;        // [nb][nb]: tile (i, c) of L is final (diagonal: L_cc and W_cc)
    int* flagsY;        // [nb][nr]
    int* ctrl;          // [0] ticket counter, [1] abort, [2] Gram ticket counter, [3] diagonal blocks factored, [4] last column drawn
    int* pause;         // [number of SMs]
    int total;
    // optional Gram product M = Y^T Y of the SOLVED right-hand sides (lower 64x64 tiles), accumulated by low-priority tasks of
    // the same kernel: task (group of mg block rows, tile) adds the group's rows to the tile in place, groups in order
    double* M; int64_t ldm;
    int* flagsM;        // [groups][m_tiles]: the tile holds the sum over groups 0 .. g
    int mg, m_full, m_tiles, m_total, m_lead;      // m_full groups of mg block rows, then the rest in halving groups
    long long spin_limit;
    long long* trace;   // diagnostics (MFGP_DF_TRACE=1): 8 timestamps per chain task, else nullptr
    int chain_la;       // chain task d draws its ticket d / chain_la block columns early (0: with its own column)
};

// Block rows [kb, ke) of Gram group gi: m_full groups of mg rows, then the remaining rows (mg .. 2 mg - 1 of them) in groups that
// halve down to single rows -- ..., 4, 2, 1, 1 -- so that what is left of the Gram product when the chain of diagonal blocks
// ends is a two-slab task per tile instead of a 2 mg-slab one.  (Host twin: df_gram_groups.)
__host__ __device__ __forceinline__ void df_group_rows(int gi, int nb, int mg, int m_full, int& kb, int& ke) {
    if (gi < m_full) { kb = gi * mg; ke = kb + mg; return; }
    kb = m_full * mg;
    int left = nb - kb;
    for (int j = m_full; ; j++) {
        const int sz = left > 1 ? (left + 1) / 2 : left;
        if (j == gi) { ke = kb + sz; return; }
        kb += sz; left -= sz;
    }
}
__host__ __forceinline__ int df_gram_groups(int nb, int mg, int& m_full) {
    m_full = nb >= 2 * mg ? (nb - mg) / mg : 0;
    int left = nb - m_full * mg, n = m_full;
    while (left > 0) { left -= left > 1 ? (left + 1) / 2 : left; n++; }
    return n;
}

__device__ __forceinline__ void df_stamp(long long* trace, int task, int k) {
    if (trace != nullptr && threadIdx.x == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t));
        trace[task * 16 + k] = (long long)t;
        trace[task * 16 + 8 + k] = clock64();
    }
}

__device__ __forceinline__ int df_ld_acquire(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ int df_ld_relaxed(const int* p) {
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void df_st_release(int* p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}
// Publishes a tile: one thread releases its flag after a barrier that orders the CTA's stores of it.  kTma: the tiles are read
// by later tasks through the async proxy (TMA, chol_dataflow_kernel), so a proxy fence precedes the release (the reader adds
// one after its acquire); in one thread, after the barrier, because a fence in every thread would drain every thread's stores
// on the chain's path.  The cp.async form reads the tiles with generic loads and releases without the fence.
template <bool kTma>
__device__ __forceinline__ void df_publish(int* flag) {
    if constexpr (kTma) asm volatile("fence.proxy.async.global;\n" ::: "memory");
    df_st_release(flag, 1);
}
__device__ __forceinline__ void df_st_relaxed(int* p, int v) {
    asm volatile("st.relaxed.gpu.global.s32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}
// lane 0 of the calling warp spins until *f != 0 (or the abort flag is raised); every lane gets the verdict.  The spin uses
// relaxed loads (served by L2, no L1 invalidation per poll); ONE acquire load orders the tile reads behind the flag.
__device__ __forceinline__ bool df_wait(const int* f, int* ctrl, int32_t* info, long long limit) {
    int ok = 1;
    if ((threadIdx.x & 31) == 0) {
        if (!df_ld_relaxed(f)) {
            const long long t0 = clock64();
            while (!df_ld_relaxed(f)) {
                __nanosleep(32);
                if (clock64() - t0 > limit) { atomicExch(ctrl + 1, 1); atomicExch(info, -1); }
                if (*reinterpret_cast<volatile int*>(ctrl + 1)) { ok = 0; break; }
            }
        }
        (void)df_ld_acquire(f);
    }
    ok = __shfl_sync(0xffffffffu, ok, 0);
    __syncwarp();                 // shuffles carry no memory ordering: order lane 0's acquire before the other lanes' tile loads
    return ok != 0;
}

// The producer's flag check for the k tiles kt0, kt0 + 1, ... of a task: lane j < 16 reads the flag of the A tile of k tile
// kt0 + j, lane 16 + j that of its B tile (relaxed: one L2 round trip for up to 16 tiles).  Once a leading run of tiles is
// seen ready, every lane of the run takes ONE acquire load of its flag, and __syncwarp orders those acquires before lane 0's
// copies.  While tile kt0 is not ready only its two flags are polled (bounded spin, abort flag as in df_wait).  Returns the
// last tile of the run (>= kt0), or -1 once the abort flag is raised.
__device__ __forceinline__ int df_poll_tiles(const int* fa, int fas, const int* fb, int fbs, int kt0, int nk, int* ctrl, int32_t* info,
                                          long long limit) {
    const int lane = threadIdx.x & 31, j = lane & 15, kt = kt0 + j;
    const int* f = lane < 16 ? fa + (int64_t)kt * fas : fb + (int64_t)kt * fbs;
    long long t0 = 0;
    for (int spin = 0;; spin++) {
        const int v = (kt < nk && (spin == 0 || j == 0)) ? df_ld_relaxed(f) : 0;
        const unsigned m = __ballot_sync(0xffffffffu, v != 0);
        const unsigned both = m & (m >> 16) & 0xffffu;
        const int n = __ffs(~both) - 1;          // length of the leading run of ready tiles
        if (n > 0) {
            if (j < n) (void)df_ld_acquire(f);
            __syncwarp();
            return kt0 + n - 1;
        }
        int stop = 0;
        if (lane == 0) {
            if (spin == 0) t0 = clock64();
            else if (clock64() - t0 > limit) { atomicExch(ctrl + 1, 1); atomicExch(info, -1); }
            stop = *reinterpret_cast<volatile int*>(ctrl + 1);
        }
        if (__shfl_sync(0xffffffffu, stop, 0)) return -1;
        __nanosleep(32);
    }
}

// ---- the task body, shared by both forms of the kernel ----------------------------------------------------------------
// chol_dataflow_kernel (producer warp, TMA ring) and chol_dataflow_cpasync_kernel (256 threads, cp.async ring) differ in how the
// slabs and the W_cc tile reach shared memory and in how the CTA synchronises around them; they draw, decode, accumulate and
// finish their tasks through the functions below, which synchronise the 256 computing threads with tile_bar().

// Draws the CTA's next task into task[0..3] = kind (0: tile of L, 1: tile of Y, 2: chain task, 3: Gram task; -1: both queues
// are empty), column, index, aux.  Called by one thread of the CTA, whose state across calls is held_m (a Gram ticket claimed
// before it became runnable; initially -1) and the decoder's column, next chain task to place and that column's first ticket
// (dec_c, dec_dnext, dec_base; initially 0, 1, 1).
__device__ __forceinline__ void df_next_task(const DfArgs& g, int& held_m, int& dec_c, int& dec_dnext, int& dec_base, int* task) {
    int c = 0, kind = -1, idx = 0, aux = 0;
    int t = -1;
    if (g.M == nullptr) {
        t = atomicAdd(g.ctrl, 1);
    } else {
        // Two queues.  Critical = the factorisation and the substitution (ticket order as below); Gram = the tiles of
        // M = Y^T Y per group of block rows.  A CTA takes a Gram ticket only when (a) every task the group's rows depend on
        // has been DRAWN (a critical ticket of a later column was handed out), so that it cannot starve them of CTAs,
        // (b) the rows are factored (no waiting inside the task) and (c) the critical queue is at least m_lead block
        // columns ahead of the chain -- or when the critical queue is empty.  A ticket claimed too early (a race at a
        // group boundary) is HELD while the CTA goes on with critical tasks, so no CTA ever waits on an undrawn task.
        for (;;) {
            const int front = df_ld_relaxed(g.ctrl + 3), drawn = df_ld_relaxed(g.ctrl + 4);
            const bool crit_left = df_ld_relaxed(g.ctrl) < g.total;
            auto runnable = [&](int tm) {
                int kb_, ke_;
                df_group_rows(tm / g.m_tiles, g.nb, g.mg, g.m_full, kb_, ke_);
                const int last_row = ke_ - 1;
                return !crit_left || (drawn > last_row && last_row + 2 <= front);
            };
            if (held_m < 0) {
                const int tm = df_ld_relaxed(g.ctrl + 2);
                if (tm < g.m_total && runnable(tm) && (!crit_left || drawn - front >= g.m_lead)) {
                    const int got = atomicAdd(g.ctrl + 2, 1);
                    if (got < g.m_total) held_m = got;
                }
            }
            if (held_m >= 0 && runnable(held_m)) {
                kind = 3; c = held_m / g.m_tiles; idx = held_m % g.m_tiles;
                int ti = 0;
                while ((ti + 1) * (ti + 2) / 2 <= idx) ti++;
                aux = idx - ti * (ti + 1) / 2;        // tile (ti, aux), aux <= ti
                idx = ti;
                held_m = -1;
                break;
            }
            if (crit_left) {
                t = atomicAdd(g.ctrl, 1);
                if (t < g.total) break;
                t = -1;
                continue;
            }
            if (held_m < 0 && df_ld_relaxed(g.ctrl + 2) >= g.m_total) break;      // both queues are empty
        }
    }
    if (t == 0) {
        kind = 2; idx = 0;            // chain task 0: the first diagonal block
    } else if (t > 0 && t < g.total) {
        // Ticket order: per block column c -- the chain tasks PLACED there, the tiles (i, c) below the sub-diagonal, the
        // Y tiles of block row c.  Chain task d (k loop of d - 1 tile pairs: the longest task of its column) is placed
        // d / chain_la columns AHEAD of column d - 1, so that its accumulation is done by the time W_{d-1} arrives; it
        // then waits on a few tiles with later tickets, which the other CTAs go on drawing (at most nb / chain_la + 1
        // CTAs can ever be in that state).  Measured at N = 4096 with 1344 right-hand sides: 2.47 -> 2.12 ms.  Pulling
        // the near-diagonal tiles forward as well made it slower (2.14 .. 2.41 ms): they crowd out the bulk.
        // (a CTA's tickets only grow: the scan resumes at the column of its previous ticket -- dec_c, dec_dnext, dec_base)
        for (;;) {
            int nchain = 0;
            while (dec_dnext + nchain < g.nb) {
                const int d = dec_dnext + nchain;
                const int place = max(0, d - 1 - (g.chain_la > 0 ? d / g.chain_la : 0));
                if (place != dec_c) break;
                nchain++;
            }
            const int ntile = g.nb - dec_c - 2 > 0 ? g.nb - dec_c - 2 : 0;
            const int n = nchain + ntile + g.nr;
            if (t < dec_base + n) {
                const int tl = t - dec_base;
                c = dec_c;
                if (tl < nchain) { kind = 2; idx = dec_dnext + tl; }
                else if (tl < nchain + ntile) { kind = 0; idx = c + 2 + (tl - nchain); }
                else { kind = 1; idx = tl - nchain - ntile; }
                break;
            }
            dec_base += n; dec_c++; dec_dnext += nchain;
        }
        if (g.M != nullptr) atomicMax(g.ctrl + 4, c);
    }
    task[3] = aux;
    task[0] = kind; task[1] = c; task[2] = idx;
}

__device__ __forceinline__ unsigned df_smid() {
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;\n" : "=r"(smid));
    return smid;
}
// This SM's pause flag (re-derived where used: a pointer held across the k loop costs registers)
__device__ __forceinline__ int* df_pause_flag(const DfArgs& g) { return g.pause + df_smid(); }

// Per-CTA accounting (MFGP_DF_ACCOUNTING builds): SM clocks spent waiting (tile flags, slabs), in k loops and in total, the
// number of tasks, the exit time and the SM
__device__ __forceinline__ void df_exit_record(const DfArgs& g, long long t_wait, long long t_loop, long long t_begin, int n_tasks) {
    unsigned long long tg;
    asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(tg));
    long long* o = g.trace + 1024 * 16 + (int64_t)blockIdx.x * 8;
    o[0] = t_wait; o[1] = t_loop; o[2] = clock64() - t_begin; o[3] = n_tasks; o[4] = (long long)tg; o[5] = df_smid();
}

// Geometry of the task in task[].  c = block column whose diagonal inverse finishes the task; i = block row of the A operand /
// output tile (Gram task: task[1] = group gi of block rows [kb, kb + nk) of Y, tile (idx, tj) of M).  The k loop accumulates nk
// k tiles in nslab slabs; the A / B tiles of k tile kt are flagged ready at fa[kt * fas] / fb[kt * fbs].
struct DfTask {
    int kind, idx, c, i, gi, tj, kb, nk, nslab, fas, fbs;
    bool rhs, chain, gram, bkn;                  // bkn: B operand stored [k][n] (rows of Y)
    const int* fa;
    const int* fb;
};
__device__ __forceinline__ DfTask df_task(const DfArgs& g, const int* task) {
    DfTask t;
    t.kind = task[0]; t.idx = task[2]; t.tj = task[3];
    t.rhs = t.kind == 1; t.chain = t.kind == 2; t.gram = t.kind == 3; t.bkn = t.rhs || t.gram;
    t.c = t.chain ? t.idx - 1 : (t.gram ? 0 : task[1]);
    t.i = t.rhs ? t.c : t.idx;
    t.gi = t.gram ? task[1] : 0;
    int ke = 0;
    t.kb = 0;
    if (t.gram) df_group_rows(t.gi, g.nb, g.mg, g.m_full, t.kb, ke);
    t.nk = t.gram ? ke - t.kb : (t.chain ? (t.idx > 0 ? t.idx - 1 : 0) : t.c);
    t.nslab = t.nk * (PB / DF_K);
    t.fa = t.gram ? g.flagsY + (int64_t)t.kb * g.nr + t.idx : g.flagsL + (int64_t)t.i * g.nb;         // Y_k,idx or L_i,k
    t.fb = t.gram ? g.flagsY + (int64_t)t.kb * g.nr + t.tj
                  : (t.rhs ? g.flagsY + t.idx : g.flagsL + (int64_t)(t.c > 0 ? t.c : 0) * g.nb);   // Y_k,r (stride nr) or L_c,k
    t.fas = t.gram ? g.nr : 1;
    t.fbs = t.bkn ? g.nr : 1;
    return t;
}

// Output of the task in task[]: the tile the accumulators start from and the task writes (row stride ldc), the diagonal tile of
// a chain task, and the flag that publishes the tile.  Derived from the shared task[] where used: held in registers across the
// k loop, these pointers would spill.
struct DfOut {
    double* Ct; int64_t ldc;
    double* Cd;
    int* flag;
};
__device__ __forceinline__ DfOut df_out(const DfArgs& g, const int* task) {
    const int kind = task[0], idx = task[2], tj = task[3];
    const bool rhs = kind == 1, chain = kind == 2, gram = kind == 3;
    const int c = chain ? idx - 1 : (gram ? 0 : task[1]), cc = c > 0 ? c : 0;
    const int i = rhs ? c : idx;
    DfOut o;
    o.Ct = gram ? g.M + (int64_t)idx * PB * g.ldm + (int64_t)tj * PB
                : (rhs ? g.Bm + (int64_t)c * PB * g.ldb + (int64_t)idx * PB : g.K + (int64_t)i * PB * g.ld + (int64_t)cc * PB);
    o.ldc = gram ? g.ldm : (rhs ? g.ldb : g.ld);
    o.Cd = g.K + (int64_t)(chain ? idx : 0) * PB * (g.ld + 1);
    o.flag = gram ? g.flagsM + (int64_t)task[1] * g.m_tiles + idx * (idx + 1) / 2 + tj
                  : (rhs ? g.flagsY + (int64_t)c * g.nr + idx : g.flagsL + (int64_t)i * g.nb + cc);   // chain: tile (idx, idx - 1)
    return o;
}

// The 256 computing threads' share of a task's 64x64 tiles, as DMMA accumulator fragments: acc the output tile, acc2 the
// diagonal tile of a chain task.  8 warps as 4 x 2; a warp owns the 8x8 tiles (row tile (warp>>1) + 4x, column tile (warp&1) + 2y),
// x < 2, y < 4 -- interleaved, so that the triangular products of the chain task (W_cc lower, S symmetric) skip about the same
// share of DMMAs in every warp.  The epilogue's shared memory: X (later the diagonal tile S) at smem, W_cc at smem + DF_TILE,
// L_{i,c} of a chain task at smem + 2 DF_TILE, each [64][68].
struct DfTile {
    int wm, wn, gq, tq;
    double acc[2][4][2], acc2[2][4][2];

    // tid: the kernel's threadIdx.x, whose range the compiler knows from the kernel's launch bounds (the 256-thread kernel
    // then drops the DMMAs of the triangular products that no warp runs)
    __device__ __forceinline__ explicit DfTile(int tid) {
        const int lane = tid & 31, warp = tid >> 5;
        wm = (warp >> 1) * 8; wn = (warp & 1) * 8;
        gq = lane >> 2; tq = lane & 3;
    }

    // The accumulators START at minus the tile they will be subtracted from (A_ic or B_cr; chain tasks: also A_dd), so the
    // global reads of those tiles happen here, at the head of the task, instead of on the critical tail behind the flag.
    // (Gram task: at plus the tile's sum over the earlier groups, once that is flagged.)
    __device__ __forceinline__ void start(const DfArgs& g, const int* task, const DfTask& tk) {
        const bool has_tile = tk.gram ? tk.gi > 0 : !(tk.chain && tk.idx == 0);
        const DfOut in = df_out(g, task);
#pragma unroll
        for (int x = 0; x < 2; x++)
#pragma unroll
            for (int y = 0; y < 4; y++) {
                const int r = wm + x * 32 + gq, cc = wn + y * 16 + tq * 2;
                double2 v = make_double2(0.0, 0.0), d = make_double2(0.0, 0.0);
                if (has_tile) v = *reinterpret_cast<const double2*>(in.Ct + (int64_t)r * in.ldc + cc);
                if (tk.chain) d = *reinterpret_cast<const double2*>(in.Cd + (int64_t)r * g.ld + cc);
                acc[x][y][0] = tk.gram ? v.x : -v.x; acc[x][y][1] = tk.gram ? v.y : -v.y;
                acc2[x][y][0] = -d.x; acc2[x][y][1] = -d.y;
            }
    }

    // One 64 x 64 x 32 slab of the k loop out of shared memory (A at As, B at Bs)
    __device__ __forceinline__ void slab(const double* As, const double* Bs, const DfTask& tk) {
#pragma unroll
        for (int kk = 0; kk < DF_K; kk += 4) {
            double a[2], b[4];
#pragma unroll
            for (int x = 0; x < 2; x++)
                a[x] = tk.gram ? As[(kk + tq) * DF_LDT + wm + x * 32 + gq] : As[(wm + x * 32 + gq) * DF_LDA + kk + tq];
#pragma unroll
            for (int y = 0; y < 4; y++)
                b[y] = tk.bkn ? Bs[(kk + tq) * DF_LDT + wn + y * 16 + gq] : Bs[(wn + y * 16 + gq) * DF_LDA + kk + tq];
#pragma unroll
            for (int x = 0; x < 2; x++)
#pragma unroll
                for (int y = 0; y < 4; y++) dmma884(acc[x][y][0], acc[x][y][1], a[x], b[y]);
            if (tk.chain) {                           // diagonal tile (i, i): L_ik L_ik^T out of the same A slab, lower tiles only
#pragma unroll
                for (int y = 0; y < 4; y++) b[y] = As[(wn + y * 16 + gq) * DF_LDA + kk + tq];
#pragma unroll
                for (int x = 0; x < 2; x++)
#pragma unroll
                    for (int y = 0; y < 4; y++)
                        if (wn + y * 16 < wm + x * 32 + 8) dmma884(acc2[x][y][0], acc2[x][y][1], a[x], b[y]);
            }
        }
    }

    // Gram task: the tile's sum over groups 0 .. gi, back in place
    __device__ __forceinline__ void store(double* Ct, int64_t ldc) const {
#pragma unroll
        for (int x = 0; x < 2; x++)
#pragma unroll
            for (int y = 0; y < 4; y++) {
                const int r = wm + x * 32 + gq, cc = wn + y * 16 + tq * 2;
                double2 v;
                v.x = acc[x][y][0]; v.y = acc[x][y][1];
                *reinterpret_cast<double2*>(Ct + (int64_t)r * ldc + cc) = v;
            }
    }

    // X = C - sum into shared memory (the accumulator started at -C); the accumulator is free for the solve product
    __device__ __forceinline__ void stage_x(double* smem) {
        double* Xs = smem;
#pragma unroll
        for (int x = 0; x < 2; x++)
#pragma unroll
            for (int y = 0; y < 4; y++) {
                const int r = wm + x * 32 + gq, cc = wn + y * 16 + tq * 2;
                Xs[r * DF_LDT + cc] = -acc[x][y][0];
                Xs[r * DF_LDT + cc + 1] = -acc[x][y][1];
                acc[x][y][0] = acc[x][y][1] = 0.0;
            }
    }

    // With X and W_cc in shared memory: the output tile L_ic = X W_cc^T or Y_cr = W_cc X, stored in place (chain task: also
    // into the L region for the tail)
    __device__ __forceinline__ void solve(double* smem, const DfTask& tk, const DfOut& out) {
        const double* Xs = smem;
        const double* Ws = smem + DF_TILE;
        double* Ls = smem + 2 * DF_TILE;
#pragma unroll 4
        for (int kk = 0; kk < PB; kk += 4) {
            double a[2], b[4];
            if (!tk.rhs) {    // L_ic = X W_cc^T :  A = X [m][k],  B = W_cc [n][k] (lower triangular: k < n0 + 8)
#pragma unroll
                for (int x = 0; x < 2; x++) a[x] = Xs[(wm + x * 32 + gq) * DF_LDT + kk + tq];
#pragma unroll
                for (int y = 0; y < 4; y++) b[y] = (kk < wn + y * 16 + 8) ? Ws[(wn + y * 16 + gq) * DF_LDT + kk + tq] : 0.0;
#pragma unroll
                for (int x = 0; x < 2; x++)
#pragma unroll
                    for (int y = 0; y < 4; y++)
                        if (kk < wn + y * 16 + 8) dmma884(acc[x][y][0], acc[x][y][1], a[x], b[y]);
                continue;
            } else {          // Y_cr = W_cc X :    A = W_cc [m][k],  B = X [k][n]
#pragma unroll
                for (int x = 0; x < 2; x++) a[x] = Ws[(wm + x * 32 + gq) * DF_LDT + kk + tq];
#pragma unroll
                for (int y = 0; y < 4; y++) b[y] = Xs[(kk + tq) * DF_LDT + wn + y * 16 + gq];
            }
#pragma unroll
            for (int x = 0; x < 2; x++)
#pragma unroll
                for (int y = 0; y < 4; y++) dmma884(acc[x][y][0], acc[x][y][1], a[x], b[y]);
        }
#pragma unroll
        for (int x = 0; x < 2; x++)
#pragma unroll
            for (int y = 0; y < 4; y++) {
                const int r = wm + x * 32 + gq, cc = wn + y * 16 + tq * 2;
                double2 v;
                v.x = acc[x][y][0]; v.y = acc[x][y][1];
                *reinterpret_cast<double2*>(out.Ct + (int64_t)r * out.ldc + cc) = v;
                if (tk.chain) { Ls[r * DF_LDT + cc] = v.x; Ls[r * DF_LDT + cc + 1] = v.y; }
            }
    }

    // 32x32x32 product on DMMA, c = A B^T (b_nk) or A B, row stride DF_LDT: warp w owns row tile w >> 1 and the column tiles
    // 2 (w & 1), 2 (w & 1) + 1
    __device__ __forceinline__ void mm32(const double* A, const double* B, bool b_nk, double (&c)[2][2]) const {
        constexpr int H = PB / 2, LO = DF_LDT;
        const int m0 = wm, n0 = 2 * wn;
        c[0][0] = c[0][1] = c[1][0] = c[1][1] = 0.0;
#pragma unroll
        for (int kk = 0; kk < H; kk += 4) {
            const double av = A[(m0 + gq) * LO + kk + tq];
#pragma unroll
            for (int j = 0; j < 2; j++) {
                const double bv = b_nk ? B[(n0 + 8 * j + gq) * LO + kk + tq] : B[(kk + tq) * LO + n0 + 8 * j + gq];
                dmma884(c[j][0], c[j][1], av, bv);
            }
        }
    }

    // Chain task d = idx, after its solve product (if d > 0): S = A_dd - sum_k L_dk L_dk^T (acc2, finished with L_{d,d-1} out of
    // shared memory), the sub-diagonal tile published before the long factor step, then L_dd and W_dd = L_dd^-1 from S.
    // kTma: the tiles are read through the async proxy (df_publish).
    template <bool kTma>
    __device__ __forceinline__ void chain_tail(const DfArgs& g, int idx, double* smem, const DfOut& out) {
        double* Xs = smem;
        double* Ls = smem + 2 * DF_TILE;
        double* const Cd = out.Cd;
        double* Wd = g.W + (int64_t)idx * PB * (g.ldw + 1);
        df_stamp(g.trace, idx, 3);
        if (idx > 0) {
            tile_bar();                               // L_{i,c} complete in shared memory; X is free
#pragma unroll 4
            for (int kk = 0; kk < PB; kk += 4) {      // acc2 += L_ic L_ic^T
                double a[2], b[4];
#pragma unroll
                for (int x = 0; x < 2; x++) a[x] = Ls[(wm + x * 32 + gq) * DF_LDT + kk + tq];
#pragma unroll
                for (int y = 0; y < 4; y++) b[y] = Ls[(wn + y * 16 + gq) * DF_LDT + kk + tq];
#pragma unroll
                for (int x = 0; x < 2; x++)
#pragma unroll
                    for (int y = 0; y < 4; y++)
                        if (wn + y * 16 < wm + x * 32 + 8) dmma884(acc2[x][y][0], acc2[x][y][1], a[x], b[y]);
            }
        }
#pragma unroll
        for (int x = 0; x < 2; x++)
#pragma unroll
            for (int y = 0; y < 4; y++) {
                const int r = wm + x * 32 + gq, cc = wn + y * 16 + tq * 2;
                Xs[r * DF_LDT + cc] = -acc2[x][y][0];                 // S = A_dd - sum (acc2 started at -A_dd)
                Xs[r * DF_LDT + cc + 1] = -acc2[x][y][1];
            }
        tile_bar();                                   // (release by one thread after the barrier covers the CTA's writes)
        if (idx > 0 && threadIdx.x == 0) df_publish<kTma>(out.flag);      // the sub-diagonal tile, before the long factor step
        df_stamp(g.trace, idx, 4);
        // Two-level factor + inverse of the 64x64 diagonal tile S (in Xs): the pair-step sweep is latency-bound per step, and a
        // 32x32 block needs half the steps at half the work per step, so  [S11 .; S21 S22] -> L11, W11 = L11^-1 (sweep);
        // L21 = S21 W11^T; S22 -= L21 L21^T; L22, W22 (sweep); W21 = -W22 (L21 W11), the four small products on DMMA.
        PotrfScratch* sc = reinterpret_cast<PotrfScratch*>(smem + DF_TILE);      // W_cc is spent
        constexpr int H = PB / 2, LO = DF_LDT;
        double* L11s = Ls;                           // rows 0..31 of the Ls region: [L11 | W11]
        double* W11s = Ls + H;
        double* L21s = Ls + H * LO;                  // rows 32..63: [L21 | T = L21 W11]
        double* Tsm = Ls + H * LO + H;
        double* W22s = Xs;                           // S11 is consumed by then
        const int m0 = wm, n0 = 2 * wn;              // this thread's share of a 32x32 tile in mm32
        double c[2][2];
        potrf_diag_body<H>(Xs, LO, Cd, g.ld, Wd, g.ldw, g.info, idx * PB, sc, L11s, W11s, LO);
        tile_bar();
        mm32(Xs + H * LO, W11s, true, c);                            // L21 = S21 W11^T  (W11's upper part is stored as zeros)
#pragma unroll
        for (int j = 0; j < 2; j++) {
            const int r = m0 + gq, cc = n0 + 8 * j + tq * 2;
            *reinterpret_cast<double2*>(Cd + (int64_t)(H + r) * g.ld + cc) = make_double2(c[j][0], c[j][1]);
            L21s[r * LO + cc] = c[j][0]; L21s[r * LO + cc + 1] = c[j][1];
        }
        tile_bar();
        mm32(L21s, L21s, true, c);                                   // S22 -= L21 L21^T
#pragma unroll
        for (int j = 0; j < 2; j++) {
            const int r = m0 + gq, cc = n0 + 8 * j + tq * 2;
            Xs[(H + r) * LO + H + cc] -= c[j][0]; Xs[(H + r) * LO + H + cc + 1] -= c[j][1];
        }
        tile_bar();
        potrf_diag_body<H>(Xs + H * LO + H, LO, Cd + (int64_t)H * g.ld + H, g.ld, Wd + (int64_t)H * g.ldw + H, g.ldw, g.info,
                           idx * PB + H, sc, nullptr, W22s, LO);
        tile_bar();
        mm32(L21s, W11s, false, c);                                  // T = L21 W11
#pragma unroll
        for (int j = 0; j < 2; j++) {
            const int r = m0 + gq, cc = n0 + 8 * j + tq * 2;
            Tsm[r * LO + cc] = c[j][0]; Tsm[r * LO + cc + 1] = c[j][1];
        }
        tile_bar();
        mm32(W22s, Tsm, false, c);                                   // W21 = -W22 T;  W12 = 0
#pragma unroll
        for (int j = 0; j < 2; j++) {
            const int r = m0 + gq, cc = n0 + 8 * j + tq * 2;
            *reinterpret_cast<double2*>(Wd + (int64_t)(H + r) * g.ldw + cc) = make_double2(-c[j][0], -c[j][1]);
            *reinterpret_cast<double2*>(Wd + (int64_t)r * g.ldw + H + cc) = make_double2(0.0, 0.0);
        }
        df_stamp(g.trace, idx, 5);
    }
};

// The end of every task: once all computing threads have stored their share, one thread publishes the output tile (chain task:
// the diagonal block, L_dd and W_dd); a chain task also lowers the SM's pause flag and advances the Gram queue's gate.
template <bool kTma>
__device__ __forceinline__ void df_finish(const DfArgs& g, const DfTask& tk, int* flag) {
    tile_bar();
    if (threadIdx.x == 0) {
        df_publish<kTma>(tk.chain ? g.flagsL + (int64_t)tk.idx * g.nb + tk.idx : flag);   // covers the tile stores before the barrier
        if (tk.chain) {
            df_st_relaxed(df_pause_flag(g), 0);
            if (g.M != nullptr) atomicMax(g.ctrl + 3, tk.idx + 1);       // diagonal blocks factored (the Gram queue's gate)
        }
    }
    if (tk.chain) df_stamp(g.trace, tk.idx, 6);
}

__global__ void __maxnreg__(112)        // 2 CTAs of 288 threads per SM: 2 x 288 x 112 <= 65536 registers
chol_dataflow_kernel(const __grid_constant__ CUtensorMap kmap, const __grid_constant__ CUtensorMap bmap,
                     const __grid_constant__ CUtensorMap wmap, DfArgs g) {
    extern __shared__ __align__(128) uint8_t df_smem_raw[];
    // TMA destinations 128-byte aligned (offsetting the shared array keeps the compiler's shared-memory loads and stores)
    double* df_smem = reinterpret_cast<double*>(df_smem_raw + ((128u - (smem_u32(df_smem_raw) & 127u)) & 127u));
    __shared__ int task[6];                   // kind, column, index, aux; ring slabs moved before the task, W_cc tiles loaded before it
    __shared__ int ready_s[4];
    __shared__ int dec_s[6];                  // the producer's ticket and ring state (below)
    __shared__ int abort_s;                   // the producer met the abort flag in the k loop (read after the loop's barrier)
    __shared__ __align__(8) unsigned long long df_bars[2 * DF_NSTAGE + 1];     // full[slot], empty[slot], W_cc tile
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool producer = warp == DF_THREADS / 32;
    const uint32_t bar_full = smem_u32(&df_bars[0]), bar_empty = smem_u32(&df_bars[DF_NSTAGE]);
    const uint32_t bar_w = smem_u32(&df_bars[2 * DF_NSTAGE]);
    if (tid == 0) {
        for (int q = 0; q < DF_NSTAGE; q++) { mbar_init(bar_full + 8 * q, 1); mbar_init(bar_empty + 8 * q, DF_THREADS / 32); }
        mbar_init(bar_w, 1);
        abort_s = 0;
        dec_s[0] = -1; dec_s[1] = 0; dec_s[2] = 1; dec_s[3] = 1; dec_s[4] = 0; dec_s[5] = 0;
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    double* As0 = df_smem;
    double* Bs0 = df_smem + DF_NSTAGE * DF_STAGE;
    // diagnostics (MFGP_DF_TRACE=1): SM clocks this CTA's thread 0 spent waiting (tile flags, slabs), in k loops, and in total
#ifdef MFGP_DF_ACCOUNTING       // build with -DMFGP_DF_ACCOUNTING for profiles/tools/cta_account.py (costs ~10 registers)
    long long t_wait = 0, t_loop = 0, t_begin = clock64(), t_mark = 0;
    int n_tasks = 0;
    const bool tracing = g.trace != nullptr;
#else
    long long t_wait = 0, t_loop = 0, t_begin = 0, t_mark = 0;
    int n_tasks = 0;
    constexpr bool tracing = false;
#endif
    // producer lane 0's state, kept in shared memory (it is touched once per task; registers are the consumers' budget):
    // df_next_task's in dec_s[0..3]; the slabs this CTA has moved so far (ring slot = gs % 3, phase = gs / 3) and the W_cc
    // tiles (phase of bar_w) in dec_s[4], dec_s[5]

    for (;;) {
        if (!producer) asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");   // epilogue stores before the next TMA writes
        __syncthreads();                      // the previous task is done with shared memory and task[]
        if (producer && lane == 0) {
            df_next_task(g, dec_s[0], dec_s[1], dec_s[2], dec_s[3], task);
            task[4] = dec_s[4]; task[5] = dec_s[5];
        }
        __syncthreads();
        const DfTask tk = df_task(g, task);
        if (tk.kind < 0) {
            if (tracing && tid == 0) df_exit_record(g, t_wait, t_loop, t_begin, n_tasks);
            return;
        }
        n_tasks++;
        if (tk.gram && tk.gi > 0) {                   // the tile's sum over the earlier groups must be final
            if (tracing) t_mark = clock64();
            if (producer) {
                const bool w = df_wait(df_out(g, task).flag - g.m_tiles, g.ctrl, g.info, g.spin_limit);
                if (lane == 0) ready_s[2] = w ? 1 : 0;
            }
            __syncthreads();
            if (tracing) t_wait += clock64() - t_mark;
            if (ready_s[2] == 0) return;              // abort raised (uniform)
        }

        if (producer) {
            // ---- producer: flags -> one TMA copy per operand of slab s into ring slot (task[4] + s) % 3 ----------------------
            // operands of the k loop: A = L_i,k ([m][k]) or Y_k,ti ([k][m]);  B = L_c,k ([n][k], transposed product) or Y_k,r ([k][n])
            const CUtensorMap* amap = tk.gram ? &bmap : &kmap;
            const CUtensorMap* bsrc = tk.bkn ? &bmap : &kmap;
            const int a_col = tk.gram ? tk.idx * PB : 0, a_row = tk.gram ? tk.kb * PB : tk.i * PB;   // + s * DF_K on the k axis
            const int b_col = tk.gram ? tk.tj * PB : (tk.rhs ? tk.idx * PB : 0);
            const int b_row = tk.gram ? tk.kb * PB : (tk.rhs ? 0 : (tk.c > 0 ? tk.c : 0) * PB);
            const uint32_t bytes = (tk.gram ? DF_KN_BYTES : DF_MK_BYTES) + (tk.bkn ? DF_KN_BYTES : DF_MK_BYTES);
            int ready_kt = -1, paused = 0;
            for (int s = 0; s < tk.nslab; s++) {
                const bool fresh = (s >> 1) > ready_kt;           // tiles newly acquired for this slab
                if (fresh) {
                    const int r = df_poll_tiles(tk.fa, tk.fas, tk.fb, tk.fbs, s >> 1, tk.nk, g.ctrl, g.info, g.spin_limit);
                    if (r < 0) {                      // abort: keep the ring moving (the consumers must not be left waiting)
                        if (lane == 0) abort_s = 1;
                        ready_kt = tk.nk;
                    } else {
                        ready_kt = r;
                    }
                }
                if (lane == 0) {
                    const unsigned gs = (unsigned)task[4] + s;
                    const int slot = gs % DF_NSTAGE;
                    // the SM's other CTA is in a chain tail: the flag is cleared at the end of every chain task that set it, and the
                    // abort flag ends the wait as well (this thread feeds the consumers: a hang here would hang them on full[slot])
                    while (paused && df_ld_relaxed(df_pause_flag(g)) && !*reinterpret_cast<volatile int*>(g.ctrl + 1)) __nanosleep(200);
                    if (gs >= DF_NSTAGE) mbar_wait(bar_empty + 8 * slot, ((gs / DF_NSTAGE) + 1) & 1);
                    if (fresh) asm volatile("fence.proxy.async.global;\n" ::: "memory");   // acquired tiles -> reads by the TMA engine
                    const uint32_t fbar = bar_full + 8 * slot;
                    mbar_arrive_expect_tx(fbar, bytes);
                    const int k0 = s * DF_K;
                    tma_load_2d(smem_u32(As0 + slot * DF_STAGE), amap, tk.gram ? a_col : k0, tk.gram ? a_row + k0 : a_row, fbar);
                    tma_load_2d(smem_u32(Bs0 + slot * DF_STAGE), bsrc, tk.bkn ? b_col : k0, tk.bkn ? b_row + k0 : b_row, fbar);
                    paused = df_ld_relaxed(df_pause_flag(g));   // (sampled one slab ahead: the load is off the critical path)
                }
            }
            if (lane == 0) dec_s[4] += tk.nslab;
            __syncthreads();                          // the consumers are out of the last slab: the ring is free
            if (abort_s) return;
            if (tk.gram || (tk.chain && tk.idx == 0)) continue;
            // the epilogue's W_cc tile, into the W_cc region of the consumers' epilogue
            const bool w = df_wait(g.flagsL + (int64_t)tk.c * g.nb + tk.c, g.ctrl, g.info, g.spin_limit);
            if (lane == 0) {
                ready_s[3] = w ? 1 : 0;
                dec_s[5]++;
                if (w) {
                    if (tk.chain) df_st_relaxed(df_pause_flag(g), 1);
                    asm volatile("fence.proxy.async.global;\n" ::: "memory");
                    mbar_arrive_expect_tx(bar_w, DF_TILE_BYTES);
                    tma_load_2d(smem_u32(df_smem + DF_TILE), &wmap, tk.c * PB, tk.c * PB, bar_w);
                } else {
                    mbar_arrive(bar_w);               // release the consumers, who then see ready_s[3] == 0
                }
            }
            if (!w) return;
            continue;
        }

        // ---- consumers ----
        DfTile f(tid);
        f.start(g, task, tk);
        // k loop: wait for the slab, DMMA loop, hand the ring slot back -- no CTA-wide barrier
        const long long t_loop0 = tracing ? clock64() : 0;
        const unsigned gs0 = task[4];
        for (int s = 0; s < tk.nslab; s++) {
            const unsigned gs = gs0 + s;
            const int slot = gs % DF_NSTAGE;
            if (tracing) t_mark = clock64();
            mbar_wait(bar_full + 8 * slot, (gs / DF_NSTAGE) & 1);
            if (tracing) t_wait += clock64() - t_mark;
            f.slab(As0 + slot * DF_STAGE, Bs0 + slot * DF_STAGE, tk);
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_empty + 8 * slot);
        }
        __syncthreads();                              // every warp is out of the last slab: shared memory is free for the epilogue
        if (abort_s) return;                          // abort raised in the k loop (uniform: written before the barrier)

        // ---- epilogue (consumer warps only) ----
        if (tracing) t_loop += clock64() - t_loop0;
        if (tk.chain) df_stamp(g.trace, tk.idx, 0);
        const DfOut out = df_out(g, task);
        if (tk.gram) {
            f.store(out.Ct, out.ldc);
        } else if (!(tk.chain && tk.idx == 0)) {
            f.stage_x(df_smem);
            if (tracing) t_mark = clock64();
            tile_bar();                               // X is in shared memory
            if (tk.chain) df_stamp(g.trace, tk.idx, 1);
            mbar_wait(bar_w, task[5] & 1);            // W_cc is final (the producer acquired its flag) and in shared memory
            if (tracing) t_wait += clock64() - t_mark;
            if (ready_s[3] == 0) return;              // abort raised (uniform: written before the producer's arrival)
            if (tk.chain) df_stamp(g.trace, tk.idx, 2);
            f.solve(df_smem, tk, out);
        }
        if (tk.chain) f.chain_tail<true>(g, tk.idx, df_smem, out);
        df_finish<true>(g, tk, out.flag);
    }
}

// The same tasks with the k loop of the 256-thread form: every thread stages its share of each slab with 16-byte cp.async and
// the CTA meets at one barrier per slab.  Used below DF_TMA_MIN_NB block columns, where the chain of diagonal blocks sets the
// time: its per-column hop is ~0.9 us shorter here than in the producer-warp kernel (which runs at <= 112 registers), and that
// outweighs the k-loop throughput the TMA ring gains (profiles/r03_chol_tma_ab.txt).
__global__ void __launch_bounds__(DF_THREADS, 2) chol_dataflow_cpasync_kernel(DfArgs g) {
    extern __shared__ __align__(16) double df_smem[];
    __shared__ int task[4];
    __shared__ int ready_s[4];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double* As0 = df_smem;
    double* Bs0 = df_smem + DF_NSTAGE * DF_STAGE;
    int* const my_pause = df_pause_flag(g);
    // diagnostics (MFGP_DF_TRACE=1): SM clocks this CTA spent waiting for tile flags, in k loops, and in total
#ifdef MFGP_DF_ACCOUNTING       // build with -DMFGP_DF_ACCOUNTING for profiles/tools/cta_account.py (costs ~10 registers)
    long long t_wait = 0, t_loop = 0, t_begin = clock64(), t_mark = 0;
    int n_tasks = 0;
    const bool tracing = g.trace != nullptr;
#else
    long long t_wait = 0, t_loop = 0, t_begin = 0, t_mark = 0;
    int n_tasks = 0;
    constexpr bool tracing = false;
#endif
    int held_m = -1, dec_c = 0, dec_dnext = 1, dec_base = 1;      // thread 0: df_next_task's state

    for (;;) {
        __syncthreads();                      // the previous task is done with shared memory and task[]
        if (tid == 0) df_next_task(g, held_m, dec_c, dec_dnext, dec_base, task);
        __syncthreads();
        const DfTask tk = df_task(g, task);
        if (tk.kind < 0) {
            if (tracing && tid == 0) df_exit_record(g, t_wait, t_loop, t_begin, n_tasks);
            return;
        }
        n_tasks++;
        // operands of the k loop: A = L_i,k ([m][k]) or Y_k,ti ([k][m]);  B = L_c,k ([n][k], transposed product) or Y_k,r ([k][n])
        const double* Ag = tk.gram ? g.Bm + (int64_t)tk.kb * PB * g.ldb + (int64_t)tk.idx * PB : g.K + (int64_t)tk.i * PB * g.ld;
        const double* Bg = tk.gram ? g.Bm + (int64_t)tk.kb * PB * g.ldb + (int64_t)tk.tj * PB
                                   : (tk.rhs ? g.Bm + (int64_t)tk.idx * PB : g.K + (int64_t)(tk.c > 0 ? tk.c : 0) * PB * g.ld);
        bool ok = true;
        if (tk.gram && tk.gi > 0) {                   // the tile's sum over the earlier groups must be final
            if (tracing) t_mark = clock64();
            if (warp == 0) {
                const bool w = df_wait(df_out(g, task).flag - g.m_tiles, g.ctrl, g.info, g.spin_limit);
                if (lane == 0) ready_s[2] = w ? 1 : 0;
            }
            __syncthreads();
            if (tracing) t_wait += clock64() - t_mark;
            if (ready_s[2] == 0) return;              // abort raised (uniform)
        }
        DfTile f(tid);
        f.start(g, task, tk);

        // k loop: DF_NSTAGE slabs in flight.  A slab that opens a new k tile may only be staged once both operand tiles are
        // flagged ready; ONE thread samples those flags for the CTA every iteration (relaxed load, then one acquire when it
        // sees them set) and hands the verdict over through shared memory across the slab barriers.  If the next tile is not
        // ready, the slabs already in flight are computed first; the CTA only waits when nothing is left to compute.
        auto issue = [&](int s) {
            const int k0 = s * DF_K;
            double* As = As0 + (s % DF_NSTAGE) * DF_STAGE;
            double* Bs = Bs0 + (s % DF_NSTAGE) * DF_STAGE;
            if (!tk.gram) {
#pragma unroll
                for (int e = tid; e < PB * (DF_K / 2); e += DF_THREADS) {     // 64 rows x 16 chunks of 16 bytes
                    const int r = e >> 4, q = e & 15;
                    cp_async16(&As[r * DF_LDA + q * 2], Ag + (int64_t)r * g.ld + k0 + q * 2, true);
                }
            } else {
#pragma unroll
                for (int e = tid; e < DF_K * (PB / 2); e += DF_THREADS) {     // [k][m]: 32 rows x 32 chunks
                    const int r = e >> 5, q = e & 31;
                    cp_async16(&As[r * DF_LDT + q * 2], Ag + (int64_t)(k0 + r) * g.ldb + q * 2, true);
                }
            }
            if (!tk.bkn) {
#pragma unroll
                for (int e = tid; e < PB * (DF_K / 2); e += DF_THREADS) {
                    const int r = e >> 4, q = e & 15;
                    cp_async16(&Bs[r * DF_LDA + q * 2], Bg + (int64_t)r * g.ld + k0 + q * 2, true);
                }
            } else {
#pragma unroll
                for (int e = tid; e < DF_K * (PB / 2); e += DF_THREADS) { // 32 rows x 32 chunks
                    const int r = e >> 5, q = e & 31;
                    cp_async16(&Bs[r * DF_LDT + q * 2], Bg + (int64_t)(k0 + r) * g.ldb + q * 2, true);
                }
            }
            cp_async_commit();
        };
        auto sample = [&](int kt) -> int {            // both operand tiles of k tile kt flagged?  (thread 0 only)
            if (kt >= tk.nk) return 0;
            if (!(df_ld_relaxed(tk.fa + (int64_t)kt * tk.fas) & df_ld_relaxed(tk.fb + (int64_t)kt * tk.fbs))) return 0;
            return df_ld_acquire(tk.fa + (int64_t)kt * tk.fas) & df_ld_acquire(tk.fb + (int64_t)kt * tk.fbs);
        };
        // the same in two halves: the relaxed loads are ISSUED before a slab's DMMA loop and consumed after it, so their L2
        // round trip never sits between the CTA and its barrier; only a tile newly seen ready costs the acquire
        auto peek = [&](int kt) -> int {
            return kt < tk.nk ? (df_ld_relaxed(tk.fa + (int64_t)kt * tk.fas) & df_ld_relaxed(tk.fb + (int64_t)kt * tk.fbs)) : 0;
        };
        auto confirm = [&](int kt) -> int {
            return df_ld_acquire(tk.fa + (int64_t)kt * tk.fas) & df_ld_acquire(tk.fb + (int64_t)kt * tk.fbs);
        };
        const int nslab = tk.nslab;
        int paused = 0;
        const long long t_loop0 = tracing ? clock64() : 0;
        int staged = 0, ready_kt = -1;                // tiles 0 .. ready_kt are known to be ready (uniform)
        if (tid == 0) ready_s[0] = sample(0) ? 0 : -1;
        __syncthreads();
        ready_kt = ready_s[0];
        // ONE barrier per slab: slab s + 2 is staged right after the barrier of iteration s, into the ring slot that slab
        // s - 1 occupied -- every warp has left that slab's DMMA loop by then.  Thread 0's verdict on the next k tile travels
        // through ready_s[] across the same barrier (written after the DMMA loop of iteration s - 1, read after the barrier of s).
        while (staged < nslab && staged < DF_NSTAGE - 1 && (staged >> 1) <= ready_kt) { issue(staged); staged++; }
        for (int s = 0; s < nslab; s++) {
            if (staged <= s) {                        // slab s could not be staged ahead: its k tile was not ready
                const int kt = s >> 1;
                if (tracing) t_mark = clock64();
                if (warp == 0) {
                    bool w = df_wait(tk.fa + (int64_t)kt * tk.fas, g.ctrl, g.info, g.spin_limit);
                    w = df_wait(tk.fb + (int64_t)kt * tk.fbs, g.ctrl, g.info, g.spin_limit) && w;
                    if (lane == 0) ready_s[2] = w ? 1 : 0;
                }
                __syncthreads();                      // also orders warp 0's acquire before everybody's tile loads
                if (tracing) t_wait += clock64() - t_mark;
                ok = (ready_s[2] != 0) && ok;
                ready_kt = max(ready_kt, kt);
                issue(s);
                staged = s + 1;
                if (staged < nslab && (staged >> 1) <= ready_kt) { issue(staged); staged++; }
            }
            if (staged - 1 - s >= 1) cp_async_wait<1>(); else cp_async_wait<0>();
            if (lane == 0) {                          // the SM's other CTA is in the tail of a chain task: stand back
                while (paused && df_ld_relaxed(my_pause)) __nanosleep(200);
                paused = df_ld_relaxed(my_pause);     // (sampled one slab ahead: the load is off the critical path)
            }
            if (__syncthreads_or(!ok)) return;        // abort raised: every thread of the CTA leaves together
            ready_kt = max(ready_kt, ready_s[s & 1]);
            while (staged < nslab && staged <= s + DF_NSTAGE - 1 && (staged >> 1) <= ready_kt) { issue(staged); staged++; }
            const int seen = (tid == 0) ? peek(ready_kt + 1) : 0;
            f.slab(As0 + (s % DF_NSTAGE) * DF_STAGE, Bs0 + (s % DF_NSTAGE) * DF_STAGE, tk);
            if (tid == 0) ready_s[(s + 1) & 1] = (seen && confirm(ready_kt + 1)) ? ready_kt + 1 : ready_kt;
        }
        __syncthreads();                              // every warp is out of the last slab: shared memory is free for the epilogue

        // ---- epilogue ----
        if (tracing) t_loop += clock64() - t_loop0;
        if (tk.chain) df_stamp(g.trace, tk.idx, 0);
        const DfOut out = df_out(g, task);
        if (tk.gram) {
            f.store(out.Ct, out.ldc);
        } else if (!(tk.chain && tk.idx == 0)) {
            f.stage_x(df_smem);
            if (tracing) t_mark = clock64();
            if (warp == 0) {
                const bool w = df_wait(g.flagsL + (int64_t)tk.c * g.nb + tk.c, g.ctrl, g.info, g.spin_limit);
                if (lane == 0) ready_s[2] = w ? 1 : 0;
            }
            __syncthreads();                          // X is in shared memory, W_cc is final (warp 0 acquired its flag)
            if (tracing) t_wait += clock64() - t_mark;
            const bool okd = ready_s[2] != 0;
            if (tk.chain && tid == 0) df_st_relaxed(my_pause, 1);
            if (tk.chain) df_stamp(g.trace, tk.idx, 1);
            const double* Wcc = g.W + (int64_t)tk.c * PB * (g.ldw + 1);
            double* Ws = df_smem + DF_TILE;
#pragma unroll
            for (int e = tid; e < PB * (PB / 2); e += DF_THREADS) {
                const int r = e >> 5, q = e & 31;
                cp_async16(&Ws[r * DF_LDT + q * 2], Wcc + (int64_t)r * g.ldw + q * 2, okd);
            }
            cp_async_commit();
            cp_async_wait<0>();
            __syncthreads();
            if (!okd) {                               // abort raised (uniform: okd came through shared memory)
                if (tk.chain && tid == 0) df_st_relaxed(my_pause, 0);
                return;
            }
            if (tk.chain) df_stamp(g.trace, tk.idx, 2);
            f.solve(df_smem, tk, out);
        }
        if (tk.chain) f.chain_tail<false>(g, tk.idx, df_smem, out);
        df_finish<false>(g, tk, out.flag);
    }
}

__global__ void zero_offdiag_blocks_kernel(double* __restrict__ W, int npad, int64_t ldw) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = blockIdx.y;
    if (j >= npad) return;
    if ((i >> 6) != (j >> 6)) W[(int64_t)i * ldw + j] = 0.0;
}

__global__ void zero_cols_kernel(double* __restrict__ Wcol, int64_t ldw) { Wcol[(int64_t)blockIdx.y * ldw + threadIdx.x] = 0.0; }

// z = W (y - mean): one warp per row; W is lower triangular so only k <= row contributes
__global__ void whiten_kernel(const double* __restrict__ W, int npad, int64_t ldw, const double* __restrict__ y, int NL,
                              int NH, double mean_L, double mean_H, double* __restrict__ z, int row_begin) {
    const int row = row_begin + blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= npad) return;
    const int N = NL + NH;
    const int kmax = min(row + 1, N);
    double s = 0.0;
    for (int k = lane; k < kmax; k += 32) {
        const double yc = y[k] - (k < NL ? mean_L : mean_H);
        s += W[(int64_t)row * ldw + k] * yc;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) z[row] = s;
}

}  // namespace mfgp

using namespace mfgp;

extern "C" int64_t mfgp_npad(int64_t n) {
    if (n <= 0) return MFGP_TILE;
    return (n + MFGP_TILE - 1) / MFGP_TILE * MFGP_TILE;
}

// Synchronisation scratch of chol_dataflow_kernel: ticket counter + abort flag, per-SM pause flags, one ready flag per
// 64x64 tile of L and of Y.  It lives in CALLER-provided workspace (so two models may factorise concurrently on different
// streams of one device, and nothing is allocated inside the library).
constexpr int DF_CTRL_INTS = 16;         // ticket counters, abort flag, progress gauges (DfArgs::ctrl)
constexpr int DF_MIN_MG = 2;             // smallest group of block rows of a Gram task (sizes the flag array)
static int64_t df_scratch_ints(int64_t npad, int64_t R, bool gram = false) {
    const int64_t nb = npad / PB, nr = (R + PB - 1) / PB;
    int64_t n = DF_CTRL_INTS + 1024 + nb * nb + nb * nr;               // ctrl, per-SM pause flags, L tile flags, Y tile flags
    if (gram) n += ((nb + DF_MIN_MG - 1) / DF_MIN_MG + 16) * (nr * (nr + 1) / 2);   // Gram tile flags per group of block rows
    return n;
}
static int64_t df_scratch_bytes(int64_t npad, int64_t R, bool gram = false) {
    return (df_scratch_ints(npad, R, gram) * 4 + 255) / 256 * 256;
}

extern "C" int64_t mfgp_workspace_bytes(int64_t npad) {
    // T blocks of the inverse (npad^2/4 doubles) + one 64x64 block, then the tile flags of mfgp_cholesky
    return npad * npad * 2 + (int64_t)PB * PB * 8 + 256 + df_scratch_bytes(npad, 0);
}

extern "C" int64_t mfgp_cholesky_solve_workspace_bytes(int64_t npad, int64_t R) { return df_scratch_bytes(npad, R); }
extern "C" int64_t mfgp_cholesky_solve_gram_workspace_bytes(int64_t npad, int64_t R) { return df_scratch_bytes(npad, R, true); }

extern "C" int mfgp_build_train_cov(const double* Xt, int64_t NL, int64_t NH, const mfgp_params* p_host, double* K,
                                    int64_t npad, int64_t ld, double* Tt, void* stream) {
    if (!p_host || !K || NL < 0 || NH < 0 || npad < NL + NH || npad % MFGP_TILE || ld < npad) return MFGP_ERR_INVALID;
    if (NL + NH > 0 && !Xt) return MFGP_ERR_INVALID;
    if (!p_host->multi && NL != 0) return MFGP_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    dim3 block(32, 8), grid((unsigned)((npad + 31) / 32), (unsigned)((npad + 7) / 8));
    const DevParams dp = make_dev_params(*p_host);
    if (Tt) {
        scaled_coords_kernel<<<(unsigned)((npad + 255) / 256), 256, 0, st>>>(Xt, (int)(NL + NH), (int)npad, dp, Tt);
        MFGP_LAUNCH_CHECK();
    }
    build_train_cov_kernel<<<grid, block, 0, st>>>(Xt, (int)NL, (int)NH, dp, K, (int)npad, ld, Tt, 0);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

namespace {
// A tensor map of chol_dataflow_kernel, kept while the next call passes the same buffer and shape (a step refactors the same
// buffers, so the maps are encoded once).
struct DfMap {
    const double* base = nullptr;
    int64_t rows = 0, cols = 0, ld = 0;
    CUtensorMap map;
};
int df_cached_map(DfMap& m, const double* base, int64_t rows, int64_t cols, int64_t ld, int box_cols, int box_rows) {
    if (m.base == base && m.rows == rows && m.cols == cols && m.ld == ld) return MFGP_OK;
    m.base = nullptr;
    const int rc = make_tensor_map_2d(&m.map, base, rows, cols, ld, box_cols, box_rows, CU_TENSOR_MAP_SWIZZLE_NONE);
    if (rc) return rc;
    m.base = base; m.rows = rows; m.cols = cols; m.ld = ld;
    return MFGP_OK;
}

struct DfScratch {        // diagnostics (MFGP_DF_TRACE=1), the cached SM count and tensor maps; no data-path state
    long long* trace = nullptr;
    int trace_nb = 0;
    int trace_grid = 0;
    int sms = 0;
    std::mutex map_mu;    // held from the first map lookup through the launch that copies the maps into its parameters:
    DfMap kmap, bmap, wmap;   // otherwise another host thread could re-encode them for its own buffers in between
};
DfScratch g_df[16];

// One launch: K -> L (lower, in place), diagonal blocks of W -> inverses of L's diagonal blocks, Bm[npad, R] -> L^-1 Bm
// (R may be 0).  The ready flags live in `scratch` (df_scratch_bytes(npad, R) bytes of caller workspace), zeroed on `st`.
int chol_dataflow(double* K, int64_t npad, int64_t ld, double* W, int64_t ldw, int32_t* info, double* Bm, int64_t ldb, int64_t R,
                  double* M, int64_t ldm, int* scratch, cudaStream_t st) {
    int dev = 0;
    MFGP_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 16 || !scratch) return MFGP_ERR_INVALID;
    // TMA operands: boxes of [m][k] slabs of K / L (36 x 64), [k][n] slabs of B / Y (68 x 32) and the W_cc tile (68 x 64);
    // rows must start 16-byte aligned.  Checked before anything is enqueued, so a rejected call leaves info and the scratch alone
    auto aligned = [](const void* p, int64_t l) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0 && (l & 1) == 0; };
    // (the tiles of M are read and written as double2 by the Gram tasks of both forms)
    if (!aligned(K, ld) || !aligned(W, ldw) || (R > 0 && !aligned(Bm, ldb)) || (M && !aligned(M, ldm))) return MFGP_ERR_INVALID;
    DfScratch& sc = g_df[dev];
    const int nb = (int)(npad / PB), nr = (int)(R / PB);
    const int64_t need = df_scratch_ints(npad, R, M != nullptr);              // ctrl, per-SM pause flags, tile flags
    if (!sc.sms) MFGP_CUDA_CHECK(cudaDeviceGetAttribute(&sc.sms, cudaDevAttrMultiProcessorCount, dev));
    MFGP_CUDA_CHECK(cudaMemsetAsync(scratch, 0, need * sizeof(int), st));
    MFGP_CUDA_CHECK(cudaMemsetAsync(info, 0, sizeof(int32_t), st));
    DfArgs a{};
    a.K = K; a.ld = ld; a.W = W; a.ldw = ldw; a.Bm = Bm; a.ldb = ldb; a.nb = nb; a.nr = nr; a.info = info;
    a.ctrl = scratch; a.pause = scratch + DF_CTRL_INTS; a.flagsL = a.pause + 1024; a.flagsY = a.flagsL + (int64_t)nb * nb;
    a.total = nb + (nb - 1) * (nb - 2) / 2 + nb * nr;     // nb chain tasks, the tiles two or more below the diagonal, Y tiles
    if (M != nullptr && nr > 0) {
        // Gram tasks: groups of mg block rows (short tasks fill the chain-bound tail better; every task re-reads and re-writes
        // its 32 KB tile of M), drawn only while the critical queue is m_lead block columns ahead of the chain.  Measured
        // (N = 4096; 384 / 832 / 1344 right-hand sides): leads of 16 and more -- in effect "when the critical queue has run
        // dry", the chain-bound last block columns -- are best (1.53 / 1.79 / 2.19 ms against 1.56 / 1.87 / 2.25 ms at 8)
        static const int mg_env = [] { const char* e = getenv("MFGP_DF_MG"); return e ? atoi(e) : 8; }();
        static const int lead_env = [] { const char* e = getenv("MFGP_DF_MLEAD"); return e ? atoi(e) : 32; }();
        a.M = M; a.ldm = ldm; a.flagsM = a.flagsY + (int64_t)nb * nr;
        a.mg = mg_env < DF_MIN_MG ? DF_MIN_MG : mg_env;
        a.m_tiles = nr * (nr + 1) / 2;
        a.m_total = df_gram_groups(nb, a.mg, a.m_full) * a.m_tiles;
        a.m_lead = lead_env;
    }
    static const bool want_trace = [] { const char* e = getenv("MFGP_DF_TRACE"); return e && atoi(e) != 0; }();
    if (want_trace) {
        if (!sc.trace) MFGP_CUDA_CHECK(cudaMalloc(&sc.trace, 1024 * 24 * sizeof(long long)));
        MFGP_CUDA_CHECK(cudaMemsetAsync(sc.trace, 0, 1024 * 24 * sizeof(long long), st));
        a.trace = nb <= 1024 ? sc.trace : nullptr;
        sc.trace_nb = nb;
    }
    static const int chain_la = [] { const char* e = getenv("MFGP_DF_CHAIN_LA"); return e ? atoi(e) : 5; }();
    a.chain_la = chain_la;
    a.spin_limit = 4000000000LL;      // ~2 s of SM clocks: only a bug can get there
    static const int occ = [] { const char* e = getenv("MFGP_DF_OCC"); return e ? atoi(e) : 2; }();
    int grid = (occ < 1 ? 1 : occ) * sc.sms;
    if (grid > a.total + a.m_total) grid = a.total + a.m_total;
    sc.trace_grid = grid < 1024 ? grid : 1024;
    if (nb < DF_TMA_MIN_NB) {         // chain-bound: the cp.async kernel's shorter hop per block column wins
        constexpr int smem_c = DF_SMEM_DOUBLES * sizeof(double);
        MFGP_CUDA_CHECK(cudaFuncSetAttribute(chol_dataflow_cpasync_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_c));
        chol_dataflow_cpasync_kernel<<<grid, DF_THREADS, smem_c, st>>>(a);
        MFGP_LAUNCH_CHECK();
        return MFGP_OK;
    }
    std::lock_guard<std::mutex> lock(sc.map_mu);
    int rc = df_cached_map(sc.kmap, K, npad, npad, ld, DF_LDA, PB);
    if (!rc) rc = df_cached_map(sc.wmap, W, npad, npad, ldw, DF_LDT, PB);
    if (!rc && nr > 0) rc = df_cached_map(sc.bmap, Bm, npad, R, ldb, DF_LDT, DF_K);
    if (rc) return rc;
    constexpr int smem = DF_SMEM_BYTES;
    MFGP_CUDA_CHECK(cudaFuncSetAttribute(chol_dataflow_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    // (without right-hand sides no task reads the B / Y map)
    chol_dataflow_kernel<<<grid, DF_CTA_THREADS, smem, st>>>(sc.kmap.map, nr > 0 ? sc.bmap.map : sc.kmap.map, sc.wmap.map, a);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}
}  // namespace

// Diagnostics: with MFGP_DF_TRACE=1 in the environment the tiled Cholesky records 7 (globaltimer ns, SM clock) stamps per
// chain task; this copies them out ([task][16] int64).  Returns the number of chain tasks of the last call, or 0.
extern "C" int64_t mfgp_debug_chol_trace(int64_t* out, int64_t max_tasks) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) return 0;
    DfScratch& sc = g_df[dev];
    if (!sc.trace || !out) return 0;
    if (max_tasks < 0) {      // per-CTA accounting: out[1024][8] = {wait clocks, k-loop clocks, total clocks, tasks, exit time ns, SM}
        if (cudaMemcpy(out, sc.trace + 1024 * 16, 1024 * 8 * sizeof(long long), cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
        return sc.trace_grid;
    }
    int64_t n = sc.trace_nb < max_tasks ? sc.trace_nb : max_tasks;
    if (cudaMemcpy(out, sc.trace, n * 16 * sizeof(long long), cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
    return n;
}

extern "C" int mfgp_cholesky(double* K, int64_t npad, int64_t ld, double* W, int64_t ldw, int32_t* info, void* work,
                             void* stream) {
    if (!K || !info || npad <= 0 || npad % MFGP_TILE || ld < npad) return MFGP_ERR_INVALID;
    if (!W && !work) return MFGP_ERR_INVALID;
    if (W && ldw < npad) return MFGP_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (W) {
        if (!work) return MFGP_ERR_INVALID;
        // the tile flags sit behind the part of `work` that mfgp_tri_inverse uses (see mfgp_workspace_bytes)
        int* scratch = reinterpret_cast<int*>(static_cast<char*>(work) + npad * npad * 2 + (int64_t)PB * PB * 8 + 256);
        return chol_dataflow(K, npad, ld, W, ldw, info, nullptr, 0, 0, nullptr, 0, scratch, st);
    }
    MFGP_CUDA_CHECK(cudaMemsetAsync(info, 0, sizeof(int32_t), st));
    const int nb = (int)(npad / PB);
    constexpr int POTRF_SMEM = 0;   // the factor + inverse sweep lives in registers and static shared memory
    MFGP_CUDA_CHECK(cudaFuncSetAttribute(potrf_diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, POTRF_SMEM));
    for (int j = 0; j < nb; j++) {
        double* Ajj = K + (int64_t)j * PB * (ld + 1);
        double* Wjj = W ? W + (int64_t)j * PB * (ldw + 1) : static_cast<double*>(work);
        const int64_t ldi = W ? ldw : PB;
        potrf_diag_kernel<<<1, 256, POTRF_SMEM, st>>>(Ajj, ld, Wjj, ldi, info, j);
        MFGP_LAUNCH_CHECK();
        const int rem = (int)(npad - (int64_t)(j + 1) * PB);
        if (rem <= 0) break;
        double* A21 = K + (int64_t)(j + 1) * PB * ld + (int64_t)j * PB;
        GemmArgs t{};   // L21 = A21 * inv(L11)^T, in place
        t.A = A21; t.lda = ld; t.B = Wjj; t.ldb = ldi; t.C = A21; t.ldc = ld;
        t.M = rem; t.N = PB; t.K = PB; t.alpha = 1.0; t.beta = 0.0; t.mode = GEMM_GENERAL;
        int rc = launch_gemm(t, true, 1, st);
        if (rc) return rc;
        GemmArgs s{};   // A22 -= L21 L21^T (lower tiles)
        s.A = A21; s.lda = ld; s.B = A21; s.ldb = ld; s.C = K + (int64_t)(j + 1) * PB * (ld + 1); s.ldc = ld;
        s.M = rem; s.N = rem; s.K = PB; s.alpha = -1.0; s.beta = 1.0; s.mode = GEMM_SYRK_LOWER;
        rc = launch_gemm(s, true, 1, st);
        if (rc) return rc;
    }
    return MFGP_OK;
}

// Cholesky of K fused with the forward substitution of R right-hand sides: on return K holds L (lower), the diagonal
// blocks of W hold the inverses of L's diagonal blocks, and Bm[npad, R] holds L^-1 Bm; the explicit inverse
// (mfgp_tri_inverse) and the product W B are not needed by the factored posterior.  ONE launch of the tile-dataflow kernel
// (chol_dataflow, above).
extern "C" int mfgp_cholesky_solve(double* K, int64_t npad, int64_t ld, double* W, int64_t ldw, int32_t* info, double* Bm,
                                   int64_t ldb, int64_t R, void* work, int64_t work_bytes, void* stream) {
    if (!K || !W || !info || !Bm || npad <= 0 || npad % MFGP_TILE || ld < npad || ldw < npad || R <= 0 || R % GT || ldb < R)
        return MFGP_ERR_INVALID;
    if (!work || work_bytes < df_scratch_bytes(npad, R)) return MFGP_ERR_INVALID;
    return chol_dataflow(K, npad, ld, W, ldw, info, Bm, ldb, R, nullptr, 0, static_cast<int*>(work), static_cast<cudaStream_t>(stream));
}

// mfgp_cholesky_solve that ALSO leaves M = Y^T Y of the solved right-hand sides (R x R, row stride ldm >= R; the 64x64 tiles on
// and below the diagonal) -- the Gram route of the factored posterior needs exactly that product.  Its tiles are accumulated by
// low-priority tasks of the same tile-dataflow kernel, group of block rows by group of block rows in a fixed order (so M is
// deterministic), in the CTA slots the factorisation leaves idle while it waits on its chain of diagonal blocks.
extern "C" int mfgp_cholesky_solve_gram(double* K, int64_t npad, int64_t ld, double* W, int64_t ldw, int32_t* info, double* Bm,
                                        int64_t ldb, int64_t R, double* M, int64_t ldm, void* work, int64_t work_bytes,
                                        void* stream) {
    if (!M) return mfgp_cholesky_solve(K, npad, ld, W, ldw, info, Bm, ldb, R, work, work_bytes, stream);
    if (!K || !W || !info || !Bm || npad <= 0 || npad % MFGP_TILE || ld < npad || ldw < npad || R <= 0 || R % GT || ldb < R || ldm < R)
        return MFGP_ERR_INVALID;
    if (!work || work_bytes < df_scratch_bytes(npad, R, true)) return MFGP_ERR_INVALID;
    return chol_dataflow(K, npad, ld, W, ldw, info, Bm, ldb, R, M, ldm, static_cast<int*>(work), static_cast<cudaStream_t>(stream));
}

extern "C" int mfgp_tri_inverse(const double* L, int64_t npad, int64_t ld, double* W, int64_t ldw, void* work,
                                void* stream) {
    if (!L || !W || !work || npad <= 0 || npad % MFGP_TILE || ld < npad || ldw < npad) return MFGP_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    double* T = static_cast<double*>(work);
    {
        dim3 grid((unsigned)((npad + 255) / 256), (unsigned)npad);
        zero_offdiag_blocks_kernel<<<grid, 256, 0, st>>>(W, (int)npad, ldw);
        MFGP_LAUNCH_CHECK();
    }
    // block doubling: [[W11,0],[W21,W22]] with W21 = -W22 (L21 W11); all pairs of one level are independent
    for (int64_t b = PB; b < npad; b *= 2) {
        const int nfull = (int)(npad / (2 * b));
        const int64_t rem = npad - 2 * b * nfull;
        for (int pass = 0; pass < 2; pass++) {
            int batch;
            int64_t top, h;
            if (pass == 0) { batch = nfull; top = 0; h = b; }
            else { batch = (rem > b) ? 1 : 0; top = 2 * b * nfull; h = rem - b; }
            if (batch == 0) continue;
            GemmArgs g1{};   // T = L21 * W11   (W11 lower: k >= n0)
            g1.A = L + (top + b) * ld + top; g1.lda = ld; g1.strideA = 2 * b * (ld + 1);
            g1.B = W + top * (ldw + 1); g1.ldb = ldw; g1.strideB = 2 * b * (ldw + 1);
            g1.C = T; g1.ldc = b; g1.strideC = b * b;
            g1.M = (int)h; g1.N = (int)b; g1.K = (int)b; g1.alpha = 1.0; g1.beta = 0.0; g1.mode = GEMM_B_LOWER;
            int rc = launch_gemm(g1, false, batch, st);
            if (rc) return rc;
            GemmArgs g2{};   // W21 = -W22 * T  (W22 lower: k < m0 + 64)
            g2.A = W + (top + b) * (ldw + 1); g2.lda = ldw; g2.strideA = 2 * b * (ldw + 1);
            g2.B = T; g2.ldb = b; g2.strideB = b * b;
            g2.C = W + (top + b) * ldw + top; g2.ldc = ldw; g2.strideC = 2 * b * (ldw + 1);
            g2.M = (int)h; g2.N = (int)b; g2.K = (int)h; g2.alpha = -1.0; g2.beta = 0.0; g2.mode = GEMM_A_LOWER;
            rc = launch_gemm(g2, false, batch, st);
            if (rc) return rc;
        }
    }
    return MFGP_OK;
}

extern "C" int mfgp_whiten(const double* W, int64_t npad, int64_t ldw, const double* y, int64_t NL, int64_t NH,
                           const mfgp_params* p_host, double* z, void* stream) {
    if (!W || !z || !p_host || npad <= 0 || npad % MFGP_TILE || ldw < npad || NL + NH > npad) return MFGP_ERR_INVALID;
    if (NL + NH > 0 && !y) return MFGP_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int wpb = 8;
    whiten_kernel<<<(unsigned)((npad + wpb - 1) / wpb), wpb * 32, 0, st>>>(W, (int)npad, ldw, y, (int)NL, (int)NH,
                                                                          p_host->mean_L, p_host->mean_H, z, 0);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

// Bordered (append-only) update of the factor: the reference appends new samples at the END of [X_L; X_H]
// (gaussian_process.py:266-268, :540-542) and refactors from scratch; algebraically the leading block of L is unchanged,
// so only the block rows that hold new points are recomputed, one 64-row block at a time (left-looking):
//   K_b   = covariance rows of the block                       (build_train_cov_kernel, rows [rb, rb+64))
//   L_b,left = K_b[:, 0:rb] W11^T                              (W11 = inverse of the already-factored leading block)
//   S     = K_b[:, rb:rb+64] - L_b,left L_b,left^T ;  L_bb = chol(S), W_bb = L_bb^-1      (potrf_diag_kernel)
//   W_b,left = -W_bb (L_b,left W11)
//   z_b   = W_b,: (y - mean)
// The skinny products (64 rows, K up to N) are split over K so they fill the GPU; partial tiles are added in fixed order.
extern "C" int mfgp_cholesky_append(const double* Xt, int64_t NL, int64_t NH_old, int64_t NH_new, const mfgp_params* p_host,
                                    double* K, int64_t ld, double* W, int64_t ldw, const double* y, double* z, double* Tt,
                                    int32_t* info, void* work, int64_t work_bytes, void* stream) {
    if (!Xt || !p_host || !K || !W || !y || !z || !info || !work || NL < 0 || NH_old < 0 || NH_new < NH_old) return MFGP_ERR_INVALID;
    const int64_t N_old = NL + NH_old, N_new = NL + NH_new;
    if (N_new == N_old) return MFGP_OK;
    const int64_t npad = mfgp_npad(N_new);
    if (ld < npad || ldw < npad) return MFGP_ERR_INVALID;
    if (!p_host->multi && NL != 0) return MFGP_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const DevParams dp = make_dev_params(*p_host);
    MFGP_CUDA_CHECK(cudaMemsetAsync(info, 0, sizeof(int32_t), st));
    constexpr int POTRF_SMEM = 0;   // the factor + inverse sweep lives in registers and static shared memory
    MFGP_CUDA_CHECK(cudaFuncSetAttribute(potrf_diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, POTRF_SMEM));
    double* part = static_cast<double*>(work);
    if (Tt) {              // pre-divided coordinates of ALL rows (the blocks below read the old rows' as well)
        scaled_coords_kernel<<<(unsigned)((npad + 255) / 256), 256, 0, st>>>(Xt, (int)N_new, (int)npad, dp, Tt);
        MFGP_LAUNCH_CHECK();
    }
    for (int64_t rb = N_old / PB * PB; rb < npad; rb += PB) {
        {   // covariance rows of the block: columns [0, rb+64) are used, the rest of the row is rewritten too (harmless)
            dim3 block(32, 8), grid((unsigned)((rb + PB + 31) / 32), PB / 8);
            build_train_cov_kernel<<<grid, block, 0, st>>>(Xt, (int)NL, (int)NH_new, dp, K, (int)(rb + PB), ld, Tt, (int)rb);
            MFGP_LAUNCH_CHECK();
        }
        if (rb > 0) {     // the column block above the new diagonal block of W must read as zero (upper triangle)
            dim3 zgrid(1, (unsigned)rb);
            zero_cols_kernel<<<zgrid, PB, 0, st>>>(W + rb, ldw);
            MFGP_LAUNCH_CHECK();
        }
        double* Kb = K + rb * ld;              // block rows of K / L
        double* Wb = W + rb * ldw;
        double* Kbb = Kb + rb;
        double* Wbb = Wb + rb;
        if (rb > 0) {
            int nsplit = (int)(rb / 256);
            if (nsplit < 1) nsplit = 1;
            if (nsplit > 16) nsplit = 16;
            int kchunk = (int)((rb / PB + nsplit - 1) / nsplit) * PB;
            nsplit = (int)((rb + kchunk - 1) / kchunk);
            const int64_t pstride = (int64_t)PB * rb;
            if (work_bytes < (int64_t)nsplit * pstride * 8) return MFGP_ERR_INVALID;
            dim3 rgrid((unsigned)((rb + 127) / 128), PB);
            GemmArgs g1{};      // part[z] = K_b[:, 0:rb] * W11^T over the z-th k range (W11 lower: k < n0 + 64)
            g1.A = Kb; g1.lda = ld; g1.B = W; g1.ldb = ldw; g1.C = part; g1.ldc = rb; g1.strideC = pstride;
            g1.M = PB; g1.N = (int)rb; g1.K = (int)rb; g1.alpha = 1.0; g1.beta = 0.0; g1.mode = GEMM_BT_LOWER; g1.kchunk = kchunk;
            int rc = launch_gemm(g1, true, nsplit, st);
            if (rc) return rc;
            splitk_reduce_kernel<<<rgrid, 128, 0, st>>>(part, nsplit, pstride, (int)rb, Kb, ld, PB, (int)rb, 1.0, 0.0);   // L_b,left
            MFGP_LAUNCH_CHECK();
            GemmArgs g2{};      // part[z] = L_b,left L_b,left^T over the z-th k range
            g2.A = Kb; g2.lda = ld; g2.B = Kb; g2.ldb = ld; g2.C = part; g2.ldc = PB; g2.strideC = PB * PB;
            g2.M = PB; g2.N = PB; g2.K = (int)rb; g2.alpha = 1.0; g2.beta = 0.0; g2.mode = GEMM_GENERAL; g2.kchunk = kchunk;
            rc = launch_gemm(g2, true, nsplit, st);
            if (rc) return rc;
            splitk_reduce_kernel<<<dim3(1, PB), 64, 0, st>>>(part, nsplit, PB * PB, PB, Kbb, ld, PB, PB, -1.0, 1.0);        // S
            MFGP_LAUNCH_CHECK();
        }
        potrf_diag_kernel<<<1, 256, POTRF_SMEM, st>>>(Kbb, ld, Wbb, ldw, info, (int)(rb / PB));
        MFGP_LAUNCH_CHECK();
        if (rb > 0) {
            int nsplit = (int)(rb / 256);
            if (nsplit < 1) nsplit = 1;
            if (nsplit > 16) nsplit = 16;
            int kchunk = (int)((rb / PB + nsplit - 1) / nsplit) * PB;
            nsplit = (int)((rb + kchunk - 1) / kchunk);
            const int64_t pstride = (int64_t)PB * rb;
            double* T2 = part + (int64_t)nsplit * pstride;      // reduced L_b,left W11 lives behind the partials
            if (work_bytes < ((int64_t)nsplit + 1) * pstride * 8) return MFGP_ERR_INVALID;
            GemmArgs g3{};      // part[z] = L_b,left * W11 over the z-th k range (W11 lower: k >= n0)
            g3.A = Kb; g3.lda = ld; g3.B = W; g3.ldb = ldw; g3.C = part; g3.ldc = rb; g3.strideC = pstride;
            g3.M = PB; g3.N = (int)rb; g3.K = (int)rb; g3.alpha = 1.0; g3.beta = 0.0; g3.mode = GEMM_B_LOWER; g3.kchunk = kchunk;
            int rc = launch_gemm(g3, false, nsplit, st);
            if (rc) return rc;
            dim3 rgrid((unsigned)((rb + 127) / 128), PB);
            splitk_reduce_kernel<<<rgrid, 128, 0, st>>>(part, nsplit, pstride, (int)rb, T2, rb, PB, (int)rb, 1.0, 0.0);
            MFGP_LAUNCH_CHECK();
            GemmArgs g4{};      // W_b,left = -W_bb * T2
            g4.A = Wbb; g4.lda = ldw; g4.B = T2; g4.ldb = rb; g4.C = Wb; g4.ldc = ldw;
            g4.M = PB; g4.N = (int)rb; g4.K = PB; g4.alpha = -1.0; g4.beta = 0.0; g4.mode = GEMM_GENERAL;
            rc = launch_gemm(g4, false, 1, st);
            if (rc) return rc;
        }
        whiten_kernel<<<PB / 8, 256, 0, st>>>(W, (int)(rb + PB), ldw, y, (int)NL, (int)NH_new, p_host->mean_L, p_host->mean_H, z, (int)rb);
        MFGP_LAUNCH_CHECK();
    }
    return MFGP_OK;
}

extern "C" int64_t mfgp_append_workspace_bytes(int64_t npad) { return (int64_t)17 * PB * npad * 8 + 256; }
