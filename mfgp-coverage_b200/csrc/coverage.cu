// Coverage step on the device: bounded-Voronoi membership of every grid point + per-cell reductions, one pass.
// Replaces, in the reference's simulator.py: in_polygon :105-124, compute_loss :194-228, compute_centroids :231-283,
// compute_max_var :286-323, compute_sample_clusters :377-412 (the polygons themselves come from the caller).
//
// Membership rule.  The reference tests every point against every Qhull cell polygon with matplotlib's crossings
// test.  Away from cell borders that is the nearest-seed rule, so the fast path is an fp64 argmin over the seeds with
// the runner-up tracked; only when the two smallest squared distances are within `tie_tol` (the point is within
// ~tie_tol/(2*seed distance) of a bisector) is the reference's test evaluated literally -- same fp64 subtract /
// multiply / compare sequence, no FMA contraction -- against all cell polygons, and the point then lands in 0, 1 or
// several cells exactly as it does in the reference (SURVEY.md Appendix A.1/A.2).
//
// Reductions are deterministic: a fixed butterfly inside the warp per distinct cell, per-warp shared-memory slots,
// per-block partials in global memory, and a second kernel that adds the block partials in block order.
#include <cfloat>
#include <climits>
#include <cmath>

#include "common.cuh"
#include "argmax.cuh"
#include "cov_device.cuh"

namespace mfgp {

constexpr int COV_WARPS = COV_THREADS / 32;
constexpr int COV_MAX_CELLS = 256;
constexpr int C_SLOTS = 6;   // sum w, sum w x, sum w y, count, max var, argmax index (int64 bits)
constexpr int P_SLOTS = 2;   // sum d^2 f, count

struct CovPartition {
    const double* seeds; int A;
    const double* poly_xy; const int32_t* poly_off;
};

struct CovArgs {
    const double* xy; const double* w; const double* var; const double* f;
    int64_t G; int64_t base_index;
    CovPartition C, P;
    double tie_tol;
    TieRule amax_tol;     // tie rule of the per-cell arg-max (see argmax_combine)
    uint64_t* member_c;
    double* partials;     // [nblocks][C.A*C_SLOTS + P.A*P_SLOTS]
    const uint4* buckets_c; const uint4* buckets_p;   // candidate tables (cov_build_buckets_kernel)
    const double* geom_c; const double* geom_p;       // {x0, y0, 1/h} of each table
    int nb_c, nb_p;
    int* tie_count;       // optional: number of (point, partition) pairs whose membership the crossings test decided
};



__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

constexpr int CELL_NONE = -1, CELL_TIE = -2, CELL_TIE_HARD = -3;   // HARD: gap <= tie_tol / 10 (counted in tie_count)
constexpr int CA_THREADS = 128, CA_WARPS = CA_THREADS / 32, CA_BLOCKS_PER_SM = 6;   // assignment kernel CTA shape
constexpr int BK_MAX = 15;            // candidate ids per bucket entry (16 bytes: count + 15 ids)
constexpr unsigned BK_OVERFLOW = 255; // count byte: scan all seeds

// ---- candidate buckets -------------------------------------------------------------------------------------------------
// A coarse nb x nb bucket grid over the bounding box of the cell polygons; entry (ix, iy) lists every seed that can be
// the nearest one -- or within tie_tol of the nearest -- for ANY point of the bucket's box.  For a point p in the box
// best(p) <= M := min_c maxdist2(c, box), and a seed with dist2(p, c) <= best(p) + tie_tol has
// mindist2(c, box) <= M + tie_tol; boxes are inflated and the threshold carries relative slack, so the list is a superset
// and the per-point best / runner-up / gap decisions are IDENTICAL to a brute-force scan over all seeds.  Border buckets
// are unbounded outwards (points outside the polygons' box) and, like buckets with more than 15 candidates, are marked
// "scan all seeds".
struct BucketGrid {
    const uint4* table; int nb; double x0, y0, inv_h;   // bucket (ix, iy) = floor((p - origin) * inv_h), clamped
};

struct BucketBuild {
    const double* seeds; int A; const double* poly_xy; const int32_t* poly_off; int nb; uint4* table; double* geom;
};

// one warp per bucket (lanes stride the seeds); blockIdx.y selects the partition
__global__ void __launch_bounds__(256) cov_build_buckets_kernel(BucketBuild b0, BucketBuild b1, double tie_tol) {
    const BucketBuild& b = blockIdx.y == 0 ? b0 : b1;
    __shared__ unsigned char ids[8][16];
    __shared__ double s_box[8][4];
    const int tid = threadIdx.x, lane = tid & 31, wib = tid >> 5;
    const int A = b.A, nb = b.nb;
    if (A == 0 || blockIdx.x * 8 >= nb * nb) return;
    // bounding box of the polygon vertices (every CTA recomputes it: a few hundred vertices)
    const int nvert = b.poly_off[A];
    double x0 = DBL_MAX, x1 = -DBL_MAX, y0 = DBL_MAX, y1 = -DBL_MAX;
    for (int i = tid; i < nvert; i += 256) {
        const double2 v = reinterpret_cast<const double2*>(b.poly_xy)[i];
        x0 = fmin(x0, v.x); x1 = fmax(x1, v.x); y0 = fmin(y0, v.y); y1 = fmax(y1, v.y);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        x0 = fmin(x0, __shfl_xor_sync(0xffffffffu, x0, o)); x1 = fmax(x1, __shfl_xor_sync(0xffffffffu, x1, o));
        y0 = fmin(y0, __shfl_xor_sync(0xffffffffu, y0, o)); y1 = fmax(y1, __shfl_xor_sync(0xffffffffu, y1, o));
    }
    if (lane == 0) { s_box[wib][0] = x0; s_box[wib][1] = x1; s_box[wib][2] = y0; s_box[wib][3] = y1; }
    __syncthreads();
#pragma unroll
    for (int w = 0; w < 8; w++) {
        x0 = fmin(x0, s_box[w][0]); x1 = fmax(x1, s_box[w][1]);
        y0 = fmin(y0, s_box[w][2]); y1 = fmax(y1, s_box[w][3]);
    }
    const double h = fmax(x1 - x0, y1 - y0) / nb;
    const int bucket = blockIdx.x * 8 + wib;
    if (bucket == 0 && lane == 0) { b.geom[0] = x0; b.geom[1] = y0; b.geom[2] = 1.0 / h; }
    if (bucket >= nb * nb) return;
    const int ix = bucket % nb, iy = bucket / nb;
    uint4 e = make_uint4(BK_OVERFLOW, 0, 0, 0);
    const bool border = ix == 0 || iy == 0 || ix == nb - 1 || iy == nb - 1;
    if (!border && tie_tol < 1e300) {
        const double pad = 1e-6 * h;
        const double bx0 = x0 + ix * h - pad, bx1 = x0 + (ix + 1) * h + pad;
        const double by0 = y0 + iy * h - pad, by1 = y0 + (iy + 1) * h + pad;
        double M = DBL_MAX;
        for (int c = lane; c < A; c += 32) {
            const double sx = b.seeds[2 * c], sy = b.seeds[2 * c + 1];
            const double dxm = fmax(sx - bx0, bx1 - sx), dym = fmax(sy - by0, by1 - sy);
            M = fmin(M, dxm * dxm + dym * dym);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) M = fmin(M, __shfl_xor_sync(0xffffffffu, M, o));
        const double T = M * (1.0 + 1e-9) + tie_tol + 1e-300;
        int count = 0;
        for (int c0 = 0; c0 < A; c0 += 32) {      // ascending seed order, as the brute-force scan
            const int c = c0 + lane;
            bool is = false;
            if (c < A) {
                const double sx = b.seeds[2 * c], sy = b.seeds[2 * c + 1];
                const double dxn = fmax(fmax(bx0 - sx, sx - bx1), 0.0), dyn = fmax(fmax(by0 - sy, sy - by1), 0.0);
                is = dxn * dxn + dyn * dyn <= T;
            }
            const unsigned bal = __ballot_sync(0xffffffffu, is);
            const int posn = count + __popc(bal & ((1u << lane) - 1u));
            if (is && posn < BK_MAX) ids[wib][1 + posn] = (unsigned char)c;
            count += __popc(bal);
        }
        __syncwarp();
        if (count <= BK_MAX) {
            if (lane == 0) ids[wib][0] = (unsigned char)count;
            __syncwarp();
            const unsigned* w = reinterpret_cast<const unsigned*>(ids[wib]);
            // bytes beyond the count are stale: mask them so equal candidate sets give equal entries
            unsigned ww[4] = {w[0], w[1], w[2], w[3]};
            for (int k = count + 1; k < 16; k++) ww[k >> 2] &= ~(0xffu << (8 * (k & 3)));
            e = make_uint4(ww[0], ww[1], ww[2], ww[3]);
        }
    }
    if (lane == 0) b.table[bucket] = e;
}

// nearest-seed cell of one point: CELL_TIE when the runner-up is within tie_tol (the crossings test decides later)
__device__ __forceinline__ int classify_point(const BucketGrid& bg, const double* __restrict__ s_seeds, int A, double x,
                                              double y, double tie_tol) {
    int ix = (int)((x - bg.x0) * bg.inv_h), iy = (int)((y - bg.y0) * bg.inv_h);
    ix = min(max(ix, 0), bg.nb - 1);
    iy = min(max(iy, 0), bg.nb - 1);
    const uint4 e = __ldg(bg.table + iy * bg.nb + ix);
    const unsigned cnt = e.x & 0xffu;
    if (cnt == 1) return (e.x >> 8) & 0xffu;       // the bucket lies inside one cell (margin > tie_tol): no distances needed
    double best = DBL_MAX, second = DBL_MAX;
    int bi = CELL_NONE;
    if (cnt != BK_OVERFLOW) {
        for (unsigned k = 1; k <= cnt; k++) {
            const unsigned wsel = (k >> 2) == 0 ? e.x : ((k >> 2) == 1 ? e.y : ((k >> 2) == 2 ? e.z : e.w));
            const int c = (wsel >> (8 * (k & 3))) & 0xffu;
            const double dx = x - s_seeds[2 * c], dy = y - s_seeds[2 * c + 1];
            const double d = fma(dx, dx, dy * dy);
            if (d < best) { second = best; best = d; bi = c; }
            else if (d < second) second = d;
        }
    } else {
        for (int c = 0; c < A; c++) {
            const double dx = x - s_seeds[2 * c], dy = y - s_seeds[2 * c + 1];
            const double d = fma(dx, dx, dy * dy);
            if (d < best) { second = best; best = d; bi = c; }
            else if (d < second) second = d;
        }
    }
    const double gap = second - best;
    return (gap > tie_tol) ? bi : ((gap > 0.1 * tie_tol) ? CELL_TIE : CELL_TIE_HARD);
}

// membership words of one point (test / in_polygon output): the nearest cell, or the crossings test for tie points
template <int WORDS>
__device__ __noinline__ void write_members(uint64_t* __restrict__ dst, int cell, const double* __restrict__ s_poly,
                                           const int* __restrict__ s_off, int A, double x, double y) {
    uint64_t m[WORDS];
#pragma unroll
    for (int k = 0; k < WORDS; k++) m[k] = 0;
    if (cell >= 0) {
#pragma unroll
        for (int k = 0; k < WORDS; k++)
            if ((cell >> 6) == k) m[k] = 1ull << (cell & 63);
    } else {
        for (int c = 0; c < A; c++)
            if (crossings_inside(s_poly + 2 * s_off[c], s_off[c + 1] - s_off[c], x, y)) {
#pragma unroll
                for (int k = 0; k < WORDS; k++)
                    if ((c >> 6) == k) m[k] |= 1ull << (c & 63);
            }
    }
#pragma unroll
    for (int k = 0; k < WORDS; k++) dst[k] = m[k];
}

// Warp-level tie-aware arg-max of one (value, index) pair per lane (index < 0: lane has no entry): the exact maximum
// by butterfly, then the LOWEST index among the lanes within the tie band of that maximum (TieRule, argmax.cuh).
__device__ __forceinline__ ArgMax argmax_warp_band(ArgMax x, TieRule t) {
    double vmax = x.i >= 0 ? x.v : -DBL_MAX;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) vmax = fmax(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
    const double tol = t.rel > 0.0 ? fmax(t.rel * (t.k0 - vmax), 0.0) : 0.0;
    long long idx = (x.i >= 0 && vmax - x.v <= tol) ? x.i : LLONG_MAX;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const long long other = __shfl_xor_sync(0xffffffffu, idx, o);
        idx = other < idx ? other : idx;
    }
    return ArgMax{vmax, idx == LLONG_MAX ? -1LL : idx};
}

__device__ __forceinline__ void slot_add_c(double* __restrict__ slot, double s0, double s1, double s2, int cnt, ArgMax am,
                                           bool with_var, TieRule tol) {
    slot[0] += s0; slot[1] += s1; slot[2] += s2; slot[3] += (double)cnt;
    if (with_var) {
        long long* islot = reinterpret_cast<long long*>(slot);
        const ArgMax r = argmax_combine(ArgMax{slot[4], islot[5]}, am, tol);
        slot[4] = r.v; islot[5] = r.i;
    }
}

// the lane-local running sums of the cell a warp has been inside -> the warp's slot of that cell
__device__ __noinline__ void flush_c(double s0, double s1, double s2, int cnt, double amv, long long ami, double* __restrict__ slot,
                                     bool with_var, TieRule tol, int lane) {
    s0 = warp_sum(s0); s1 = warp_sum(s1); s2 = warp_sum(s2);
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    ArgMax am{amv, ami};
    if (with_var) am = argmax_warp_band(am, tol);
    if (lane == 0) slot_add_c(slot, s0, s1, s2, cnt, am, with_var, tol);
}
__device__ __noinline__ void flush_p(double s0, int cnt, double* __restrict__ slot, int lane) {
    s0 = warp_sum(s0);
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) { slot[0] += s0; slot[1] += (double)cnt; }
}

// Row straddles a cell border (or holds tie points): one fixed butterfly per distinct cell, straight into the slots.
// Tie points (within tie_tol of a bisector): the reference's crossings test against EVERY cell polygon decides --
// 0, 1 or several cells.
__device__ __noinline__ void mixed_c(int A, bool with_var, TieRule tol, const double* __restrict__ s_poly,
                                     const int* __restrict__ s_off, double* __restrict__ wacc, int cell, double x, double y,
                                     double wv, double vv, long long gidx, int lane, int* ties) {
    unsigned pending = __ballot_sync(0xffffffffu, cell >= 0);
    while (pending) {
        const int c = __shfl_sync(0xffffffffu, cell, __ffs(pending) - 1);
        const bool mine = cell == c;
        const unsigned who = __ballot_sync(0xffffffffu, mine);
        const double s0 = warp_sum(mine ? wv : 0.0), s1 = warp_sum(mine ? wv * x : 0.0), s2 = warp_sum(mine ? wv * y : 0.0);
        ArgMax am{vv, mine ? gidx : -1LL};
        if (with_var) am = argmax_warp_band(am, tol);
        if (lane == 0) slot_add_c(wacc + c * C_SLOTS, s0, s1, s2, __popc(who), am, with_var, tol);
        pending &= ~who;
    }
    const unsigned tied = __ballot_sync(0xffffffffu, cell == CELL_TIE);
    if (tied) {
        if (ties != nullptr && lane == 0) atomicAdd(ties, __popc(tied));
        for (int c = 0; c < A; c++) {
            const bool mine = cell == CELL_TIE && crossings_inside(s_poly + 2 * s_off[c], s_off[c + 1] - s_off[c], x, y);
            const unsigned who = __ballot_sync(0xffffffffu, mine);
            if (!who) continue;
            const double s0 = warp_sum(mine ? wv : 0.0), s1 = warp_sum(mine ? wv * x : 0.0), s2 = warp_sum(mine ? wv * y : 0.0);
            ArgMax am{vv, mine ? gidx : -1LL};
            if (with_var) am = argmax_warp_band(am, tol);
            if (lane == 0) slot_add_c(wacc + c * C_SLOTS, s0, s1, s2, __popc(who), am, with_var, tol);
        }
    }
}
__device__ __noinline__ void mixed_p(int A, const double* __restrict__ s_seeds, const double* __restrict__ s_poly,
                                     const int* __restrict__ s_off, double* __restrict__ wacc_p, int cell, double x, double y,
                                     double fv, int lane, int* ties) {
    unsigned pending = __ballot_sync(0xffffffffu, cell >= 0);
    while (pending) {
        const int c = __shfl_sync(0xffffffffu, cell, __ffs(pending) - 1);
        const bool mine = cell == c;
        const unsigned who = __ballot_sync(0xffffffffu, mine);
        const double dx = x - s_seeds[2 * c], dy = y - s_seeds[2 * c + 1];
        const double pl = __dmul_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), fv);     // simulator.py:215-216
        const double s0 = warp_sum(mine ? pl : 0.0);
        if (lane == 0) { wacc_p[c * P_SLOTS] += s0; wacc_p[c * P_SLOTS + 1] += (double)__popc(who); }
        pending &= ~who;
    }
    const unsigned tied = __ballot_sync(0xffffffffu, cell == CELL_TIE);
    if (tied) {
        if (ties != nullptr && lane == 0) atomicAdd(ties, __popc(tied));
        for (int c = 0; c < A; c++) {
            const bool mine = cell == CELL_TIE && crossings_inside(s_poly + 2 * s_off[c], s_off[c + 1] - s_off[c], x, y);
            const unsigned who = __ballot_sync(0xffffffffu, mine);
            if (!who) continue;
            const double dx = x - s_seeds[2 * c], dy = y - s_seeds[2 * c + 1];
            const double pl = __dmul_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), fv);
            const double s0 = warp_sum(mine ? pl : 0.0);
            if (lane == 0) { wacc_p[c * P_SLOTS] += s0; wacc_p[c * P_SLOTS + 1] += (double)__popc(who); }
        }
    }
}

// Each warp owns a contiguous range of 32-point rows (lane = point: coalesced 40 B/point streams, the next row's
// loads in flight while the current one is processed).  Per row and partition: bucket lookup -> a handful of candidate
// seeds -> nearest / runner-up cell.  While the whole warp stays inside ONE cell (the common case: consecutive grid
// points) every lane just adds into its own registers; the warp reduces only when it moves to another cell.  Rows
// that straddle a border or hold tie points take the butterfly-per-cell path.  Deterministic: fixed point -> lane ->
// warp -> block order.
template <int WORDS>
__global__ void __launch_bounds__(CA_THREADS, CA_BLOCKS_PER_SM) cov_assign_reduce_kernel(CovArgs a) {
    extern __shared__ __align__(16) double sm[];
    const int Ac = a.C.A, Ap = a.P.A;
    const int nvc = Ac ? a.C.poly_off[Ac] : 0, nvp = Ap ? a.P.poly_off[Ap] : 0;
    double* s_seed_c = sm;                       // [Ac*2]
    double* s_seed_p = s_seed_c + 2 * Ac;        // [Ap*2]
    double* s_poly_c = s_seed_p + 2 * Ap;        // [nvc*2]
    double* s_poly_p = s_poly_c + 2 * nvc;       // [nvp*2]
    double* s_acc = s_poly_p + 2 * nvp;          // [CA_WARPS][Ac*C_SLOTS + Ap*P_SLOTS]
    const int stride = Ac * C_SLOTS + Ap * P_SLOTS;
    int* s_off_c = reinterpret_cast<int*>(s_acc + CA_WARPS * stride);   // [Ac+1]
    int* s_off_p = s_off_c + (Ac + 1);                                    // [Ap+1]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < 2 * Ac; i += CA_THREADS) s_seed_c[i] = a.C.seeds[i];
    for (int i = tid; i < 2 * Ap; i += CA_THREADS) s_seed_p[i] = a.P.seeds[i];
    for (int i = tid; i < 2 * nvc; i += CA_THREADS) s_poly_c[i] = a.C.poly_xy[i];
    for (int i = tid; i < 2 * nvp; i += CA_THREADS) s_poly_p[i] = a.P.poly_xy[i];
    for (int i = tid; i <= Ac && Ac; i += CA_THREADS) s_off_c[i] = a.C.poly_off[i];
    for (int i = tid; i <= Ap && Ap; i += CA_THREADS) s_off_p[i] = a.P.poly_off[i];
    for (int i = tid; i < CA_WARPS * stride; i += CA_THREADS) s_acc[i] = 0.0;
    __syncthreads();
    double* wacc = s_acc + warp * stride;
    for (int c = lane; c < Ac; c += 32) {
        wacc[c * C_SLOTS + 4] = -DBL_MAX;
        reinterpret_cast<long long*>(wacc)[c * C_SLOTS + 5] = -1;
    }
    __syncwarp();
    const bool polygon_mode = !(a.tie_tol < 1e300);    // arbitrary polygons: the crossings test decides everywhere
    const bool with_var = a.var != nullptr;
    BucketGrid bgc{a.buckets_c, a.nb_c, 0.0, 0.0, 0.0}, bgp{a.buckets_p, a.nb_p, 0.0, 0.0, 0.0};
    if (Ac) { bgc.x0 = a.geom_c[0]; bgc.y0 = a.geom_c[1]; bgc.inv_h = a.geom_c[2]; }
    if (Ap) { bgp.x0 = a.geom_p[0]; bgp.y0 = a.geom_p[1]; bgp.inv_h = a.geom_p[2]; }

    // contiguous split of the 32-point rows over all warps of the grid
    const int64_t nrows = (a.G + 31) / 32;
    const int64_t nwarps = (int64_t)gridDim.x * CA_WARPS, gw = (int64_t)blockIdx.x * CA_WARPS + warp;
    const int64_t r0 = gw * nrows / nwarps, r1 = (gw + 1) * nrows / nwarps;

    double c_s0 = 0.0, c_s1 = 0.0, c_s2 = 0.0, p_s0 = 0.0;      // lane-local sums of the current cell (C / P partition)
    int c_cnt = 0, p_cnt = 0;
    ArgMax c_am{0.0, -1};
    double c_tol = 0.0;       // tie band of c_am (TieRule) -- refreshed when the index moves
    int cur_c = CELL_NONE, cur_p = CELL_NONE;
    const TieRule tol = a.amax_tol;
    const double tie_tol = a.tie_tol;
    const int64_t base_index = a.base_index;

    double2 nxy = make_double2(0.0, 0.0);
    double nw = 0.0, nv = 0.0, nf = 0.0;
    auto fetch = [&](int64_t row) {
        const int64_t g = row * 32 + lane;
        if (row < r1 && g < a.G) {
            nxy = __ldg(reinterpret_cast<const double2*>(a.xy) + g);
            if (a.w) nw = __ldg(a.w + g);
            if (with_var) nv = __ldg(a.var + g);
            if (a.f) nf = __ldg(a.f + g);
        }
    };
    fetch(r0);
#pragma unroll 1
    for (int64_t row = r0; row < r1; row++) {
        const int64_t g = row * 32 + lane;
        const bool valid = g < a.G;
        const double x = nxy.x, y = nxy.y, wv = nw, vv = nv, fv = nf;
        fetch(row + 1);
        if (Ac) {
            int cell = !valid ? CELL_NONE : (polygon_mode ? CELL_TIE : classify_point(bgc, s_seed_c, Ac, x, y, tie_tol));
            {
                const unsigned hm = __ballot_sync(0xffffffffu, cell == CELL_TIE_HARD);
                if (hm && a.tie_count != nullptr && lane == 0) atomicAdd(a.tie_count, __popc(hm));
                if (cell == CELL_TIE_HARD) cell = CELL_TIE;
            }
            if (a.member_c && valid) write_members<WORDS>(a.member_c + g * WORDS, cell, s_poly_c, s_off_c, Ac, x, y);
            const int c0 = __shfl_sync(0xffffffffu, cell, 0);       // lane 0 is valid whenever the row holds any point
            if (c0 >= 0 && __all_sync(0xffffffffu, cell == c0 || cell == CELL_NONE)) {
                if (c0 != cur_c) {
                    if (cur_c >= 0) flush_c(c_s0, c_s1, c_s2, c_cnt, c_am.v, c_am.i, wacc + cur_c * C_SLOTS, with_var, tol, lane);
                    c_s0 = c_s1 = c_s2 = 0.0; c_cnt = 0; c_am = ArgMax{0.0, -1};
                    cur_c = c0;
                }
                if (cell == c0) {
                    c_s0 += wv; c_s1 += wv * x; c_s2 += wv * y; c_cnt++;
                    if (with_var) {      // == argmax_combine(c_am, {vv, idx}) for an index above c_am.i, a few instructions
                        if (c_am.i < 0 || vv - c_am.v > c_tol) {
                            c_am = ArgMax{vv, (long long)(base_index + g)};
                            c_tol = tol.rel > 0.0 ? fmax(tol.rel * (tol.k0 - vv), 0.0) : 0.0;
                        } else if (vv > c_am.v) {
                            c_am.v = vv;
                        }
                    }
                }
            } else {
                mixed_c(Ac, with_var, tol, s_poly_c, s_off_c, wacc, cell, x, y, wv, vv, (long long)(base_index + g), lane, nullptr);
            }
        }
        if (Ap) {
            int cell = !valid ? CELL_NONE : (polygon_mode ? CELL_TIE : classify_point(bgp, s_seed_p, Ap, x, y, tie_tol));
            {
                const unsigned hm = __ballot_sync(0xffffffffu, cell == CELL_TIE_HARD);
                if (hm && a.tie_count != nullptr && lane == 0) atomicAdd(a.tie_count, __popc(hm));
                if (cell == CELL_TIE_HARD) cell = CELL_TIE;
            }
            const int c0 = __shfl_sync(0xffffffffu, cell, 0);
            if (c0 >= 0 && __all_sync(0xffffffffu, cell == c0 || cell == CELL_NONE)) {
                if (c0 != cur_p) {
                    if (cur_p >= 0) flush_p(p_s0, p_cnt, wacc + Ac * C_SLOTS + cur_p * P_SLOTS, lane);
                    p_s0 = 0.0; p_cnt = 0;
                    cur_p = c0;
                }
                if (cell == c0) {
                    const double dx = x - s_seed_p[2 * c0], dy = y - s_seed_p[2 * c0 + 1];
                    p_s0 += __dmul_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), fv);     // simulator.py:215-216
                    p_cnt++;
                }
            } else {
                mixed_p(Ap, s_seed_p, s_poly_p, s_off_p, wacc + Ac * C_SLOTS, cell, x, y, fv, lane, nullptr);
            }
        }
    }
    if (cur_c >= 0) flush_c(c_s0, c_s1, c_s2, c_cnt, c_am.v, c_am.i, wacc + cur_c * C_SLOTS, with_var, tol, lane);
    if (cur_p >= 0) flush_p(p_s0, p_cnt, wacc + Ac * C_SLOTS + cur_p * P_SLOTS, lane);
    __syncthreads();
    // block partial = warp slots combined in warp order
    // partials are laid out [slot][block] so the finalize kernel reads them coalesced
    double* out = a.partials + blockIdx.x;
    const int64_t pld = gridDim.x;
    for (int i = tid; i < Ac * C_SLOTS; i += CA_THREADS) {
        const int slot = i % C_SLOTS;
        if (slot < 4) {
            double s = 0.0;
            for (int w = 0; w < CA_WARPS; w++) s += s_acc[w * stride + i];
            out[i * pld] = s;
        } else if (slot == 4) {
            ArgMax best{0.0, -1};
            for (int w = 0; w < CA_WARPS; w++)
                best = argmax_combine(best, ArgMax{s_acc[w * stride + i], reinterpret_cast<const long long*>(s_acc)[w * stride + i + 1]},
                                      a.amax_tol);
            out[i * pld] = best.v;
            reinterpret_cast<long long*>(out)[(i + 1) * pld] = best.i;
        }
    }
    for (int i = tid; i < Ap * P_SLOTS; i += CA_THREADS) {
        double s = 0.0;
        for (int w = 0; w < CA_WARPS; w++) s += s_acc[w * stride + Ac * C_SLOTS + i];
        out[(Ac * C_SLOTS + i) * pld] = s;
    }
}

// ---- column-sweep variant for tensor-product grids --------------------------------------------------------------------
// Every grid of the reference is `[[x, y] for x in gx for y in gy]` (distribution.py:337-339): point g = ix*ny + iy.  Here a
// warp owns a BAND of 32 consecutive iy and walks a range of columns ix: lane l always looks at (ix, iy0 + l), so from one
// iteration to the next a lane moves by one grid step in x and stays inside the same Voronoi cell for ~100 iterations.
// Each lane therefore accumulates privately in registers, keyed by ITS OWN current cell, with no shuffles at all; when a
// lane's cell changes it parks its sums as one entry of a per-warp shared-memory queue (slot order: iteration, then lane
// -- deterministic), and lane 0 later adds the entries to the warp's per-cell slots in queue order.  Points within
// tie_tol of a bisector go to a second queue and are classified with the reference's crossings test, cooperatively.
// Loads are 32 consecutive points per warp per iteration (full sectors), the next column's in flight.
constexpr int SW_THREADS = 256, SW_WARPS = SW_THREADS / 32;
constexpr int SW_QCAP = 64;          // queue entries per warp and partition
constexpr int SW_DEPTH = 1;          // columns of loads in flight per lane
constexpr int SW_CW = 7;             // words per C entry: cell, s0, s1, s2, cnt, max var, arg-max index
constexpr int SW_PW = 3;             // words per P entry: cell, s0, cnt

struct SweepShape { int ny, ncols, nbands, nseg, cols_per_seg; };

__device__ __forceinline__ void sweep_drain_c(const double* __restrict__ q, int n, double* __restrict__ wacc, bool with_var,
                                              TieRule tol, int lane) {
    __syncwarp();
    if (lane == 0)
        for (int e = 0; e < n; e++) {
            const double* r = q + e * SW_CW;
            const int c = (int)__double_as_longlong(r[0]);
            slot_add_c(wacc + c * C_SLOTS, r[1], r[2], r[3], (int)__double_as_longlong(r[4]),
                       ArgMax{r[5], __double_as_longlong(r[6])}, with_var, tol);
        }
    __syncwarp();
}
__device__ __forceinline__ void sweep_drain_p(const double* __restrict__ q, int n, double* __restrict__ wacc_p, int lane) {
    __syncwarp();
    if (lane == 0)
        for (int e = 0; e < n; e++) {
            const double* r = q + e * SW_PW;
            const int c = (int)__double_as_longlong(r[0]);
            wacc_p[c * P_SLOTS] += r[1];
            wacc_p[c * P_SLOTS + 1] += (double)__double_as_longlong(r[2]);
        }
    __syncwarp();
}

// tie points of the queue, one at a time, all lanes cooperating: lane tests cells lane, lane+32, ... with the crossings test
__device__ __noinline__ void sweep_ties(const CovArgs& a, const long long* __restrict__ tq, int n, double* __restrict__ wacc,
                                        bool is_c, int lane) {
    const CovPartition& part = is_c ? a.C : a.P;
    const bool with_var = a.var != nullptr;
    for (int e = 0; e < n; e++) {
        const long long g = tq[e];
        const double2 p = reinterpret_cast<const double2*>(a.xy)[g];
        for (int c0 = 0; c0 < part.A; c0 += 32) {
            const int c = c0 + lane;
            bool in = false;
            if (c < part.A) {
                const int o = part.poly_off[c];
                in = crossings_inside(part.poly_xy + 2 * o, part.poly_off[c + 1] - o, p.x, p.y);
            }
            unsigned m = __ballot_sync(0xffffffffu, in);
            if (lane == 0)
                while (m) {
                    const int cc = c0 + __ffs(m) - 1;
                    m &= m - 1;
                    if (is_c) {
                        const double wv = a.w ? a.w[g] : 0.0;
                        slot_add_c(wacc + cc * C_SLOTS, wv, wv * p.x, wv * p.y, 1,
                                   ArgMax{with_var ? a.var[g] : 0.0, (long long)(a.base_index + g)}, with_var, a.amax_tol);
                    } else {
                        const double dx = p.x - part.seeds[2 * cc], dy = p.y - part.seeds[2 * cc + 1];
                        wacc[cc * P_SLOTS] += __dmul_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), a.f[g]);
                        wacc[cc * P_SLOTS + 1] += 1.0;
                    }
                }
        }
    }
    __syncwarp();
}

__global__ void __launch_bounds__(SW_THREADS, 2) cov_sweep_kernel(CovArgs a, SweepShape sh) {
    extern __shared__ __align__(16) double sm[];
    const int Ac = a.C.A, Ap = a.P.A;
    const int stride = Ac * C_SLOTS + Ap * P_SLOTS;
    double* s_seed_c = sm;                                   // [2 Ac]
    double* s_seed_p = s_seed_c + 2 * Ac;                    // [2 Ap]
    double* s_acc = s_seed_p + 2 * Ap;                       // [SW_WARPS][stride]
    double* s_qc = s_acc + SW_WARPS * stride;                // [SW_WARPS][SW_QCAP][SW_CW]
    double* s_qp = s_qc + SW_WARPS * SW_QCAP * SW_CW;        // [SW_WARPS][SW_QCAP][SW_PW]
    long long* s_tq = reinterpret_cast<long long*>(s_qp + SW_WARPS * SW_QCAP * SW_PW);   // [SW_WARPS][2][SW_QCAP]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < 2 * Ac; i += SW_THREADS) s_seed_c[i] = a.C.seeds[i];
    for (int i = tid; i < 2 * Ap; i += SW_THREADS) s_seed_p[i] = a.P.seeds[i];
    for (int i = tid; i < SW_WARPS * stride; i += SW_THREADS) s_acc[i] = 0.0;
    __syncthreads();
    double* wacc = s_acc + warp * stride;
    double* wacc_p = wacc + Ac * C_SLOTS;
    for (int c = lane; c < Ac; c += 32) {
        wacc[c * C_SLOTS + 4] = -DBL_MAX;
        reinterpret_cast<long long*>(wacc)[c * C_SLOTS + 5] = -1;
    }
    __syncwarp();
    double* qc = s_qc + warp * SW_QCAP * SW_CW;
    double* qp = s_qp + warp * SW_QCAP * SW_PW;
    long long* tqc = s_tq + warp * 2 * SW_QCAP;
    long long* tqp = tqc + SW_QCAP;
    const bool with_var = a.var != nullptr;
    const TieRule tol = a.amax_tol;
    const double tie_tol = a.tie_tol;
    BucketGrid bgc{a.buckets_c, a.nb_c, 0.0, 0.0, 0.0}, bgp{a.buckets_p, a.nb_p, 0.0, 0.0, 0.0};
    if (Ac) { bgc.x0 = a.geom_c[0]; bgc.y0 = a.geom_c[1]; bgc.inv_h = a.geom_c[2]; }
    if (Ap) { bgp.x0 = a.geom_p[0]; bgp.y0 = a.geom_p[1]; bgp.inv_h = a.geom_p[2]; }

    const int gw = blockIdx.x * SW_WARPS + warp;
    const int band = gw % sh.nbands, seg = gw / sh.nbands;
    const int iy = band * 32 + lane;
    const bool lane_ok = iy < sh.ny && seg < sh.nseg;
    const int col0 = seg * sh.cols_per_seg, col1 = min(sh.ncols, col0 + sh.cols_per_seg);
    const unsigned lt_mask = (1u << lane) - 1u;

    int cur_c = CELL_NONE, cur_p = CELL_NONE, c_cnt = 0, p_cnt = 0, qn_c = 0, qn_p = 0, tn_c = 0, tn_p = 0;
    double c_s0 = 0.0, c_s1 = 0.0, c_s2 = 0.0, p_s0 = 0.0, c_tol = 0.0;
    ArgMax c_am{0.0, -1};

    // software pipeline: the loads of the next SW_DEPTH columns are in flight while one column is processed
    // (16 warps x 32 lanes x 40 B x SW_DEPTH ~ 80 KB per SM outstanding: enough to cover the HBM latency)
    double2 nxy[SW_DEPTH];
    double nw[SW_DEPTH], nv[SW_DEPTH], nf[SW_DEPTH];
#pragma unroll
    for (int d = 0; d < SW_DEPTH; d++) { nxy[d] = make_double2(0.0, 0.0); nw[d] = nv[d] = nf[d] = 0.0; }
    auto fetch = [&](int col, double2& fxy, double& fw, double& fvv, double& ff) {
        if (lane_ok && col < col1) {
            const int64_t g = (int64_t)col * sh.ny + iy;
            fxy = __ldg(reinterpret_cast<const double2*>(a.xy) + g);
            if (a.w) fw = __ldg(a.w + g);
            if (with_var) fvv = __ldg(a.var + g);
            if (a.f) ff = __ldg(a.f + g);
        }
    };
#pragma unroll
    for (int d = 0; d < SW_DEPTH; d++) fetch(col0 + d, nxy[d], nw[d], nv[d], nf[d]);
#pragma unroll 1
    for (int colb = col0; colb < col1; colb += SW_DEPTH) {        // warp-uniform trip count (seg is uniform per warp)
#pragma unroll
      for (int d = 0; d < SW_DEPTH; d++) {
        const int col = colb + d;
        if (col >= col1) break;
        const int64_t g = (int64_t)col * sh.ny + iy;
        const double x = nxy[d].x, y = nxy[d].y, wv = nw[d], vv = nv[d], fv = nf[d];
        fetch(col + SW_DEPTH, nxy[d], nw[d], nv[d], nf[d]);
        if (Ac) {
            const int cell = lane_ok ? classify_point(bgc, s_seed_c, Ac, x, y, tie_tol) : CELL_NONE;
            const bool tie = cell == CELL_TIE || cell == CELL_TIE_HARD;
            const bool hard = cell == CELL_TIE_HARD;
            const int ncell = tie ? CELL_NONE : cell;
            const bool chg = ncell != cur_c;
            const bool psh = chg && cur_c >= 0;
            const unsigned pm = __ballot_sync(0xffffffffu, psh);
            if (pm) {
                if (qn_c + __popc(pm) > SW_QCAP) { sweep_drain_c(qc, qn_c, wacc, with_var, tol, lane); qn_c = 0; }
                if (psh) {
                    double* r = qc + (qn_c + __popc(pm & lt_mask)) * SW_CW;
                    r[0] = __longlong_as_double((long long)cur_c); r[1] = c_s0; r[2] = c_s1; r[3] = c_s2;
                    r[4] = __longlong_as_double((long long)c_cnt); r[5] = c_am.v; r[6] = __longlong_as_double(c_am.i);
                }
                qn_c += __popc(pm);
            }
            if (chg) { c_s0 = c_s1 = c_s2 = 0.0; c_cnt = 0; c_am = ArgMax{0.0, -1}; cur_c = ncell; }
            if (ncell >= 0) {
                c_s0 += wv; c_s1 += wv * x; c_s2 += wv * y; c_cnt++;
                if (with_var) {      // == argmax_combine(c_am, {vv, idx}) for an index above c_am.i
                    if (c_am.i < 0 || vv - c_am.v > c_tol) {
                        c_am = ArgMax{vv, (long long)(a.base_index + g)};
                        c_tol = tol.rel > 0.0 ? fmax(tol.rel * (tol.k0 - vv), 0.0) : 0.0;
                    } else if (vv > c_am.v) {
                        c_am.v = vv;
                    }
                }
            }
            const unsigned tm = __ballot_sync(0xffffffffu, tie);
            if (tm && a.tie_count != nullptr) {
                const unsigned hm = __ballot_sync(0xffffffffu, hard);
                if (hm && lane == 0) atomicAdd(a.tie_count, __popc(hm));
            }
            if (tm) {
                if (tn_c + __popc(tm) > SW_QCAP) {
                    sweep_drain_c(qc, qn_c, wacc, with_var, tol, lane); qn_c = 0;      // keep slot order: queue first
                    sweep_ties(a, tqc, tn_c, wacc, true, lane); tn_c = 0;
                }
                if (tie) tqc[tn_c + __popc(tm & lt_mask)] = g;
                tn_c += __popc(tm);
            }
        }
        if (Ap) {
            const int cell = lane_ok ? classify_point(bgp, s_seed_p, Ap, x, y, tie_tol) : CELL_NONE;
            const bool tie = cell == CELL_TIE || cell == CELL_TIE_HARD;
            const bool hard = cell == CELL_TIE_HARD;
            const int ncell = tie ? CELL_NONE : cell;
            const bool chg = ncell != cur_p;
            const bool psh = chg && cur_p >= 0;
            const unsigned pm = __ballot_sync(0xffffffffu, psh);
            if (pm) {
                if (qn_p + __popc(pm) > SW_QCAP) { sweep_drain_p(qp, qn_p, wacc_p, lane); qn_p = 0; }
                if (psh) {
                    double* r = qp + (qn_p + __popc(pm & lt_mask)) * SW_PW;
                    r[0] = __longlong_as_double((long long)cur_p); r[1] = p_s0; r[2] = __longlong_as_double((long long)p_cnt);
                }
                qn_p += __popc(pm);
            }
            if (chg) { p_s0 = 0.0; p_cnt = 0; cur_p = ncell; }
            if (ncell >= 0) {
                const double dx = x - s_seed_p[2 * ncell], dy = y - s_seed_p[2 * ncell + 1];
                p_s0 += __dmul_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), fv);     // simulator.py:215-216
                p_cnt++;
            }
            const unsigned tm = __ballot_sync(0xffffffffu, tie);
            if (tm && a.tie_count != nullptr) {
                const unsigned hm = __ballot_sync(0xffffffffu, hard);
                if (hm && lane == 0) atomicAdd(a.tie_count, __popc(hm));
            }
            if (tm) {
                if (tn_p + __popc(tm) > SW_QCAP) {
                    sweep_drain_p(qp, qn_p, wacc_p, lane); qn_p = 0;
                    sweep_ties(a, tqp, tn_p, wacc_p, false, lane); tn_p = 0;
                }
                if (tie) tqp[tn_p + __popc(tm & lt_mask)] = g;
                tn_p += __popc(tm);
            }
        }
      }
    }
    // end of the warp's range: parked entries first (queue order), then the lanes' live sums grouped by cell with fixed
    // butterflies, then the tie points
    if (Ac) {
        sweep_drain_c(qc, qn_c, wacc, with_var, tol, lane);
        unsigned pending = __ballot_sync(0xffffffffu, cur_c >= 0);
        while (pending) {
            const int c = __shfl_sync(0xffffffffu, cur_c, __ffs(pending) - 1);
            const bool mine = cur_c == c;
            const unsigned who = __ballot_sync(0xffffffffu, mine);
            const double s0 = warp_sum(mine ? c_s0 : 0.0), s1 = warp_sum(mine ? c_s1 : 0.0), s2 = warp_sum(mine ? c_s2 : 0.0);
            const int cnt = __reduce_add_sync(0xffffffffu, mine ? c_cnt : 0);
            ArgMax am = mine ? c_am : ArgMax{0.0, -1};
            if (with_var) am = argmax_warp_band(am, tol);
            if (lane == 0) slot_add_c(wacc + c * C_SLOTS, s0, s1, s2, cnt, am, with_var, tol);
            pending &= ~who;
        }
        if (tn_c) sweep_ties(a, tqc, tn_c, wacc, true, lane);
    }
    if (Ap) {
        sweep_drain_p(qp, qn_p, wacc_p, lane);
        unsigned pending = __ballot_sync(0xffffffffu, cur_p >= 0);
        while (pending) {
            const int c = __shfl_sync(0xffffffffu, cur_p, __ffs(pending) - 1);
            const bool mine = cur_p == c;
            const unsigned who = __ballot_sync(0xffffffffu, mine);
            const double s0 = warp_sum(mine ? p_s0 : 0.0);
            const int cnt = __reduce_add_sync(0xffffffffu, mine ? p_cnt : 0);
            if (lane == 0) { wacc_p[c * P_SLOTS] += s0; wacc_p[c * P_SLOTS + 1] += (double)cnt; }
            pending &= ~who;
        }
        if (tn_p) sweep_ties(a, tqp, tn_p, wacc_p, false, lane);
    }
    __syncthreads();
    double* out = a.partials + blockIdx.x;       // [slot][block], as cov_assign_reduce_kernel
    const int64_t pld = gridDim.x;
    for (int i = tid; i < Ac * C_SLOTS; i += SW_THREADS) {
        const int slot = i % C_SLOTS;
        if (slot < 4) {
            double s = 0.0;
            for (int w = 0; w < SW_WARPS; w++) s += s_acc[w * stride + i];
            out[i * pld] = s;
        } else if (slot == 4) {
            ArgMax best{0.0, -1};
            for (int w = 0; w < SW_WARPS; w++)
                best = argmax_combine(best, ArgMax{s_acc[w * stride + i], reinterpret_cast<const long long*>(s_acc)[w * stride + i + 1]}, tol);
            out[i * pld] = best.v;
            reinterpret_cast<long long*>(out)[(i + 1) * pld] = best.i;
        }
    }
    for (int i = tid; i < Ap * P_SLOTS; i += SW_THREADS) {
        double s = 0.0;
        for (int w = 0; w < SW_WARPS; w++) s += s_acc[w * stride + Ac * C_SLOTS + i];
        out[(Ac * C_SLOTS + i) * pld] = s;
    }
}

// One warp per output: lanes stride over the block partials in block order, then a fixed butterfly.
__global__ void __launch_bounds__(256) cov_finalize_kernel(const double* __restrict__ partials, int nblocks, int Ac, int Ap,
                                                           TieRule amax_tol, double* __restrict__ cent, double* __restrict__ amax_val,
                                                           int64_t* __restrict__ amax_idx, double* __restrict__ lossp) {
    const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    const int64_t pld = nblocks;
    if (i < Ac * 4) {
        const int c = i / 4, s = i % 4;
        const double* src = partials + (int64_t)(c * C_SLOTS + s) * pld;
        double acc = 0.0;
#pragma unroll 4
        for (int b = lane; b < nblocks; b += 32) acc += src[b];
        acc = warp_sum(acc);
        if (cent && lane == 0) cent[i] = acc;
    } else if (i < Ac * 5) {
        const int c = i - Ac * 4;
        const double* sv = partials + (int64_t)(c * C_SLOTS + 4) * pld;
        const long long* si = reinterpret_cast<const long long*>(partials) + (int64_t)(c * C_SLOTS + 5) * pld;
        ArgMax best{0.0, -1};
#pragma unroll 4
        for (int b = lane; b < nblocks; b += 32) best = argmax_combine(best, ArgMax{sv[b], si[b]}, amax_tol);
        best = argmax_warp(best, amax_tol);
        if (lane == 0) {
            if (amax_val) amax_val[c] = best.v;
            if (amax_idx) amax_idx[c] = best.i;
        }
    } else if (i < Ac * 5 + Ap * 2) {
        const int j = i - Ac * 5;
        const double* src = partials + (int64_t)(Ac * C_SLOTS + j) * pld;
        double acc = 0.0;
#pragma unroll 4
        for (int b = lane; b < nblocks; b += 32) acc += src[b];
        acc = warp_sum(acc);
        if (lossp && lane == 0) lossp[j] = acc;
    }
}

constexpr int COV_BUCKETS_MAX = 128;
constexpr int COV_MAX_BLOCKS = 148 * 6;     // upper bound of the CTA count of any assignment kernel (sizes the partials)
// bucket grid side: about eight buckets per mean cell spacing, so most buckets lie inside ONE cell
inline int cov_bucket_side(int64_t A) {
    int nb = 16;
    while (nb < COV_BUCKETS_MAX && (int64_t)nb * nb < 64 * A) nb *= 2;
    return nb;
}

// number of CTAs of the assignment kernel: every warp gets at least one whole chunk
inline int cov_chunk_blocks(int64_t G) {
    const int64_t nrows = (G + 31) / 32;
    int64_t b = (nrows + 4 * CA_WARPS - 1) / (4 * CA_WARPS);     // at least ~4 rows per warp
    const int64_t cap = 148 * CA_BLOCKS_PER_SM;      // one resident wave; warps grid-stride over the chunks
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (int)b;
}

}  // namespace mfgp

using namespace mfgp;

extern "C" int64_t cov_workspace_bytes(int64_t G, int64_t Ac, int64_t Ap) {
    const int64_t stride = Ac * C_SLOTS + Ap * P_SLOTS;
    const int64_t nb = COV_MAX_BLOCKS;
    int64_t a = nb * stride * 8;
    int64_t b = nb * 16;
    return (a > b ? a : b) + 256 + 2 * ((int64_t)COV_BUCKETS_MAX * COV_BUCKETS_MAX * 16 + 64);
}

static int cov_assign_reduce_impl(const double* xy, const double* w, const double* var, const double* f, int64_t G,
                                 int64_t base_index, const double* seeds_c, int64_t Ac, const double* poly_xy_c,
                                 const int32_t* poly_off_c, int64_t nvert_c, const double* seeds_p, int64_t Ap,
                                 const double* poly_xy_p, const int32_t* poly_off_p, int64_t nvert_p, double tie_tol, double amax_k0, double amax_rel, double* cent, double* amax_val,
                                 int64_t* amax_idx, double* lossp, uint64_t* member_c, int32_t* tie_count, void* work,
                                 int64_t work_bytes, void* stream, int64_t ny) {
    if (!xy || G <= 0 || Ac < 0 || Ap < 0 || Ac + Ap == 0 || Ac > COV_MAX_CELLS || Ap > COV_MAX_CELLS) return MFGP_ERR_INVALID;
    if (Ac && (!seeds_c || !poly_xy_c || !poly_off_c)) return MFGP_ERR_INVALID;
    if (Ap && (!seeds_p || !poly_xy_p || !poly_off_p || !f)) return MFGP_ERR_INVALID;
    if (!work || work_bytes < cov_workspace_bytes(G, Ac, Ap)) return MFGP_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (nvert_c < 0 || nvert_p < 0) return MFGP_ERR_INVALID;
    const int64_t nvc = Ac ? nvert_c : 0, nvp = Ap ? nvert_p : 0;   // == poly_off[A], passed by the host to size shared memory
    CovArgs a;
    a.xy = xy; a.w = w; a.var = var; a.f = f; a.G = G; a.base_index = base_index;
    a.C = {seeds_c, (int)Ac, poly_xy_c, poly_off_c};
    a.P = {seeds_p, (int)Ap, poly_xy_p, poly_off_p};
    a.tie_tol = tie_tol; a.amax_tol = TieRule{amax_k0, amax_rel > 0.0 ? amax_rel : 0.0}; a.member_c = member_c; a.partials = static_cast<double*>(work);
    a.tie_count = tie_count;
    if (tie_count) MFGP_CUDA_CHECK(cudaMemsetAsync(tie_count, 0, sizeof(int32_t), st));
    const int stride = (int)(Ac * C_SLOTS + Ap * P_SLOTS);
    {   // candidate bucket tables live behind the block partials in the workspace
        const int64_t nbmax = COV_MAX_BLOCKS;
        const int64_t pa = nbmax * stride * 8, pb = nbmax * 16;
        char* base = static_cast<char*>(work) + (((pa > pb ? pa : pb) + 255) / 256) * 256;
        const int64_t tbytes = (int64_t)COV_BUCKETS_MAX * COV_BUCKETS_MAX * 16;
        a.buckets_c = reinterpret_cast<const uint4*>(base);
        a.geom_c = reinterpret_cast<const double*>(base + tbytes);
        a.buckets_p = reinterpret_cast<const uint4*>(base + tbytes + 64);
        a.geom_p = reinterpret_cast<const double*>(base + 2 * tbytes + 64);
        a.nb_c = cov_bucket_side(Ac);
        a.nb_p = cov_bucket_side(Ap);
        BucketBuild bc{seeds_c, (int)Ac, poly_xy_c, poly_off_c, a.nb_c, const_cast<uint4*>(a.buckets_c), const_cast<double*>(a.geom_c)};
        BucketBuild bp{seeds_p, (int)Ap, poly_xy_p, poly_off_p, a.nb_p, const_cast<uint4*>(a.buckets_p), const_cast<double*>(a.geom_p)};
        const int nbm = a.nb_c > a.nb_p ? a.nb_c : a.nb_p;
        cov_build_buckets_kernel<<<dim3((unsigned)((nbm * nbm + 7) / 8), 2), 256, 0, st>>>(bc, bp, tie_tol);
        MFGP_LAUNCH_CHECK();
    }
    const int nfin = (int)(Ac * 5 + Ap * 2);
    if (ny > 0 && G % ny == 0 && member_c == nullptr && tie_tol < 1e300 && G / ny < (1 << 30)) {
        // tensor-product grid, nearest-seed cells: column sweep (lane-private accumulation, no shuffles in the loop)
        SweepShape sh;
        sh.ny = (int)ny; sh.ncols = (int)(G / ny); sh.nbands = (int)((ny + 31) / 32);
        int nseg = (148 * 16 + sh.nbands - 1) / sh.nbands;                  // ~16 warps per SM: one resident wave
        if (nseg > sh.ncols) nseg = sh.ncols;
        sh.cols_per_seg = (sh.ncols + nseg - 1) / nseg;
        sh.nseg = (sh.ncols + sh.cols_per_seg - 1) / sh.cols_per_seg;
        const int64_t nwarps = (int64_t)sh.nbands * sh.nseg;
        const int sblocks = (int)((nwarps + SW_WARPS - 1) / SW_WARPS);
        const size_t ssmem = sizeof(double) * (2 * Ac + 2 * Ap + (size_t)SW_WARPS * stride + (size_t)SW_WARPS * SW_QCAP * (SW_CW + SW_PW)) +
                             sizeof(long long) * SW_WARPS * 2 * SW_QCAP;
        if (ssmem <= 200 * 1024 && sblocks <= COV_MAX_BLOCKS && sh.nbands <= 148 * 16) {
            MFGP_CUDA_CHECK(cudaFuncSetAttribute(cov_sweep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssmem));
            cov_sweep_kernel<<<sblocks, SW_THREADS, ssmem, st>>>(a, sh);
            MFGP_LAUNCH_CHECK();
            cov_finalize_kernel<<<(nfin + 7) / 8, 256, 0, st>>>(a.partials, sblocks, (int)Ac, (int)Ap, a.amax_tol, cent, amax_val, amax_idx, lossp);
            MFGP_LAUNCH_CHECK();
            return MFGP_OK;
        }
    }
    const size_t smem = sizeof(double) * (2 * Ac + 2 * Ap + 2 * (size_t)nvc + 2 * (size_t)nvp + (size_t)CA_WARPS * stride) +
                        sizeof(int) * (Ac + Ap + 2);
    if (smem > 200 * 1024) return MFGP_ERR_INVALID;
    const int nblocks = cov_chunk_blocks(G);
    const int words = (int)((Ac > Ap ? Ac : Ap) + 63) / 64;
    auto launch = [&](auto kern) -> int {
        MFGP_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<nblocks, CA_THREADS, smem, st>>>(a);
        MFGP_LAUNCH_CHECK();
        return MFGP_OK;
    };
    int rc;
    if (words <= 1) rc = launch(cov_assign_reduce_kernel<1>);
    else if (words == 2) rc = launch(cov_assign_reduce_kernel<2>);
    else rc = launch(cov_assign_reduce_kernel<4>);
    if (rc) return rc;
    cov_finalize_kernel<<<(nfin + 7) / 8, 256, 0, st>>>(a.partials, nblocks, (int)Ac, (int)Ap, a.amax_tol, cent, amax_val, amax_idx, lossp);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

extern "C" int cov_assign_reduce(const double* xy, const double* w, const double* var, const double* f, int64_t G,
                                 int64_t base_index, const double* seeds_c, int64_t Ac, const double* poly_xy_c,
                                 const int32_t* poly_off_c, int64_t nvert_c, const double* seeds_p, int64_t Ap,
                                 const double* poly_xy_p, const int32_t* poly_off_p, int64_t nvert_p, double tie_tol, double amax_k0,
                                 double amax_rel, double* cent, double* amax_val, int64_t* amax_idx, double* lossp,
                                 uint64_t* member_c, int32_t* tie_count, void* work, int64_t work_bytes, void* stream) {
    return cov_assign_reduce_impl(xy, w, var, f, G, base_index, seeds_c, Ac, poly_xy_c, poly_off_c, nvert_c, seeds_p, Ap, poly_xy_p,
                                  poly_off_p, nvert_p, tie_tol, amax_k0, amax_rel, cent, amax_val, amax_idx, lossp, member_c,
                                  tie_count, work, work_bytes, stream, 0);
}

extern "C" int cov_assign_reduce_grid(const double* xy, const double* w, const double* var, const double* f, int64_t G, int64_t ny,
                                      int64_t base_index, const double* seeds_c, int64_t Ac, const double* poly_xy_c,
                                      const int32_t* poly_off_c, int64_t nvert_c, const double* seeds_p, int64_t Ap,
                                      const double* poly_xy_p, const int32_t* poly_off_p, int64_t nvert_p, double tie_tol,
                                      double amax_k0, double amax_rel, double* cent, double* amax_val, int64_t* amax_idx,
                                      double* lossp, int32_t* tie_count, void* work, int64_t work_bytes, void* stream) {
    if (ny <= 0 || G % ny) return MFGP_ERR_INVALID;
    return cov_assign_reduce_impl(xy, w, var, f, G, base_index, seeds_c, Ac, poly_xy_c, poly_off_c, nvert_c, seeds_p, Ap, poly_xy_p,
                                  poly_off_p, nvert_p, tie_tol, amax_k0, amax_rel, cent, amax_val, amax_idx, lossp, nullptr,
                                  tie_count, work, work_bytes, stream, ny);
}

extern "C" int cov_argmax(const double* v, int64_t G, int64_t base_index, double k0, double rel, double* out_val,
                          int64_t* out_idx, void* work, int64_t work_bytes, void* stream) {
    const TieRule tol{k0, rel > 0.0 ? rel : 0.0};
    if (!v || G <= 0 || !out_val || !out_idx || !work) return MFGP_ERR_INVALID;
    const int nblocks = cov_blocks(G);
    if (work_bytes < (int64_t)nblocks * 16) return MFGP_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    double* pv = static_cast<double*>(work);
    long long* pi = reinterpret_cast<long long*>(pv + nblocks);
    argmax_partial_kernel<<<nblocks, 256, 0, st>>>(v, G, base_index, tol, pv, pi);
    MFGP_LAUNCH_CHECK();
    argmax_final_kernel<<<1, 32, 0, st>>>(pv, pi, nblocks, tol, out_val, out_idx);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

// ---- bounded Voronoi cells by half-plane clipping (SURVEY.md section 8f rank 2) -----------------------------------------
// The reference mirrors the seeds across the four sides of the box cushioned by eps and asks Qhull for the diagram of
// the 5A points (simulator.py:154-191).  The first A cells of that diagram are exactly the cells of the A seeds clipped
// to the box inflated by eps/2 (the bisector of a seed and its own mirror image; mirror images of OTHER seeds never cut
// closer than the seeds themselves), so each cell is the inflated box clipped by the A-1 bisector half-planes
// (Sutherland-Hodgman).  Agrees with Qhull's vertices to ~1e-13 (areas to ~1e-12); only grid points lying EXACTLY on a
// bisector can be classified differently, which is why the Qhull path stays the default for parity runs.
// One thread per cell; polygons are packed into poly_xy / poly_off in cell order; areas by the shoelace formula
// (simulator.py:127-136).  flag[0] != 0: a polygon outgrew VC_MAXV or the packed capacity.
namespace mfgp {
// Two launches per partition: (1) a warp per cell, VC_WARPS cells per CTA, as many CTAs as it takes -- vertices into a
// fixed-stride scratch, vertex count and shoelace area per cell; (2) one CTA packs the cells back to back (prefix sum of the
// counts -> poly_off) for the coverage kernels.
__global__ void __launch_bounds__(VC_WARPS * 32) cov_voronoi_clip_kernel(const double* __restrict__ seeds, int A, double x0, double x1,
                                                                         double y0, double y1, double* __restrict__ scratch,
                                                                         int32_t* __restrict__ counts, double* __restrict__ areas,
                                                                         int32_t* __restrict__ flag) {
    __shared__ double s_seeds[2 * COV_MAX_CELLS];
    __shared__ double s_buf[VC_WARPS][256];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int e = tid; e < 2 * A; e += blockDim.x) s_seeds[e] = seeds[e];
    __syncthreads();
    const int i = blockIdx.x * VC_WARPS + warp;
    if (i >= A) return;
    bool overflow = false;
    int which = 0;
    const int n = vc_clip_cell(s_seeds, A, i, x0, x1, y0, y1, s_buf[warp], lane, overflow, which);
    const double* px = s_buf[warp] + 128 * which;
    const double* py = px + 64;
    double* dst = scratch + (int64_t)i * 2 * VC_MAXV;
    for (int v = lane; v < n; v += 32) { dst[2 * v] = px[v]; dst[2 * v + 1] = py[v]; }
    if (lane == 0) {
        // shoelace: 0.5 |x . roll(y,1) - y . roll(x,1)|, summed in vertex order
        double s1 = 0.0, s2 = 0.0;
        for (int v = 0; v < n; v++) {
            const int u = (v + n - 1) % n;
            s1 += px[v] * py[u];
            s2 += py[v] * px[u];
        }
        counts[i] = n;
        areas[i] = overflow ? __longlong_as_double(0x7ff8000000000000LL) : 0.5 * fabs(s1 - s2);   // NaN poisons loss / centroid
        if (overflow) atomicExch(flag, 1);
    }
}

__global__ void __launch_bounds__(256) cov_voronoi_pack_kernel(const double* __restrict__ scratch, const int32_t* __restrict__ counts, int A,
                                                               double* __restrict__ poly_xy, int32_t* __restrict__ poly_off,
                                                               int cap_vertices, double* __restrict__ areas, int32_t* __restrict__ flag) {
    __shared__ int off[COV_MAX_CELLS + 1];
    const int tid = threadIdx.x;
    if (tid == 0) {
        off[0] = 0;
        for (int c = 0; c < A; c++) off[c + 1] = off[c] + counts[c];
    }
    __syncthreads();
    for (int e = tid; e <= A; e += blockDim.x) poly_off[e] = off[e];
    if (off[A] > cap_vertices) {                                  // uniform
        if (tid == 0) atomicExch(flag, 1);
        for (int e = tid; e < A; e += blockDim.x) areas[e] = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    const int lane = tid & 31, warp = tid >> 5;
    for (int c = warp; c < A; c += 8) {
        const double* src = scratch + (int64_t)c * 2 * VC_MAXV;
        double* dst = poly_xy + 2 * (int64_t)off[c];
        const int n2 = 2 * (off[c + 1] - off[c]);
        for (int e = lane; e < n2; e += 32) dst[e] = src[e];
    }
}

// O(A) finishing of the per-cell partial sums with the reference's arithmetic (simulator.py:215-219, :256-271):
// out[0] = loss, out[1 + 2i], out[2 + 2i] = centroid i (clamped to the grid's extent), out[1 + 2A + i] = max variance of
// cell i, out[1 + 3A + i] = its arg-max grid index (as a double; exact below 2^53, -1 = empty cell).
__global__ void cov_finish_kernel(const double* __restrict__ cent, const double* __restrict__ areas_c, int Ac,
                                  const double* __restrict__ lossp, const double* __restrict__ areas_p, int Ap,
                                  const double* __restrict__ amax_val, const int64_t* __restrict__ amax_idx, double xmin,
                                  double xmax, double ymin, double ymax, const int32_t* __restrict__ flag0,
                                  const int32_t* __restrict__ flag1, const int32_t* __restrict__ flag2,
                                  const int32_t* __restrict__ flag3, double* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) {
        out[1 + 4 * Ac] = flag0 ? (double)*flag0 : 0.0;      // e.g. the Cholesky `info` and the clip-capacity flags: the
        out[2 + 4 * Ac] = flag1 ? (double)*flag1 : 0.0;      // host learns about a failure without an extra sync
        out[3 + 4 * Ac] = flag2 ? (double)*flag2 : 0.0;
        out[4 + 4 * Ac] = flag3 ? (double)*flag3 : 0.0;      // e.g. cov_assign_reduce's tie counter
        double loss = 0.0;
        for (int c = 0; c < Ap; c++) loss += (lossp[2 * c] / lossp[2 * c + 1]) * areas_p[c];     // cell order, like :215-219
        out[0] = Ap ? loss : 0.0;
    }
    if (i < Ac) {
        const double n = cent[4 * i + 3], a = areas_c[i];
        const double f_int = (cent[4 * i] / n) * a;
        double cx = ((cent[4 * i + 1] / n) * a) / f_int, cy = ((cent[4 * i + 2] / n) * a) / f_int;
        if (cx < xmin) cx = xmin;
        if (cx > xmax) cx = xmax;
        if (cy < ymin) cy = ymin;
        if (cy > ymax) cy = ymax;
        out[1 + 2 * i] = cx;
        out[2 + 2 * i] = cy;
        out[1 + 2 * Ac + i] = amax_val ? amax_val[i] : 0.0;
        out[1 + 3 * Ac + i] = amax_idx ? (double)amax_idx[i] : -1.0;
    }
}
}  // namespace mfgp

extern "C" int64_t cov_voronoi_clip_workspace_bytes(int64_t A) { return A * (2 * VC_MAXV * 8 + 4) + 256; }

extern "C" int cov_voronoi_clip(const double* seeds, int64_t A, double xmin, double xmax, double ymin, double ymax, double eps,
                                double* poly_xy, int32_t* poly_off, int64_t cap_vertices, double* areas, int32_t* flag,
                                void* work, int64_t work_bytes, void* stream) {
    if (!seeds || A <= 0 || A > COV_MAX_CELLS || !poly_xy || !poly_off || !areas || !flag || cap_vertices < 4) return MFGP_ERR_INVALID;
    if (!work || work_bytes < cov_voronoi_clip_workspace_bytes(A)) return MFGP_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MFGP_CUDA_CHECK(cudaMemsetAsync(flag, 0, sizeof(int32_t), st));
    const double h = 0.5 * eps;
    double* scratch = static_cast<double*>(work);
    int32_t* counts = reinterpret_cast<int32_t*>(scratch + A * 2 * VC_MAXV);
    cov_voronoi_clip_kernel<<<(unsigned)((A + VC_WARPS - 1) / VC_WARPS), VC_WARPS * 32, 0, st>>>(seeds, (int)A, xmin - h, xmax + h, ymin - h,
                                                                                         ymax + h, scratch, counts, areas, flag);
    MFGP_LAUNCH_CHECK();
    cov_voronoi_pack_kernel<<<1, 256, 0, st>>>(scratch, counts, (int)A, poly_xy, poly_off, (int)cap_vertices, areas, flag);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

namespace mfgp {

// ---- per-cell centroids of posterior draws, reduced in Chebyshev coefficient space ------------------------------------------
// A draw over a tensor-product grid is F_s(ix, iy) = mean + sum_l sum_k Uy[iy][l] Ux[ix][k] C_s[l][k] (mfgp_grid_sample_coef's
// coefficients, basis T_l(ty) T_k(tx) on the sampler's box).  The Lloyd partials of cell i are linear in the draw:
//   sum_{p in cell i} w(p) F_s(p) = <C'_s, Mom_i^w>,   Mom_i^w[l][k] = sum_ix Ux[ix][k] sum_{iy in cell i, column ix} w Uy[iy][l]
// with w in {1, x, y} and C' = C + mean on term (0, 0) (T_0 = 1).  So the moments are formed once per partition and every draw
// costs 3 dot products of length ry kpad per cell; no draw is evaluated.
//   cov_moment_basis_kernel    Ux[ix][k] (zero for k >= rx), Uy[iy][l] from the grid's own coordinates
//   cov_moment_columns_kernel  one CTA per column: membership as cov_assign_reduce_grid (nearest seed + runner-up, the
//                              crossings test for ties), then Sy[i][ix][0][l] = sum Uy[iy][l], Sy[i][ix][1][l] = sum y Uy[iy][l]
//                              over the column's points of cell i; thread (m, l) owns those sums and adds in row order
//   cov_moment_reduce_kernel   one CTA per cell over the columns it touches: Mom_i^{1,x,y} = Ux^T Sy_i (x weights per column)
//   cov_moment_centroid_kernel one CTA per (cell, 32 draws): the three dot products, then cov_finish's centroid arithmetic
// Every sum runs in a fixed order (no floating-point atomics): the same inputs give the same bits.
constexpr int CM_MAXR = 64;            // largest Chebyshev order per axis (the sampler's limit)
constexpr int CM_THREADS = 2 * CM_MAXR; // column kernel: thread (m, l) owns moment m of y term l
constexpr int CM_ROWS = 512;           // rows of a column classified per pass
constexpr int CM_WORDS = COV_MAX_CELLS / 64;
constexpr int CR_COLS = 16;            // columns staged per step of the reduction kernel
constexpr int CC_WARPS = 8, CC_DRAWS = 32;   // centroid kernel: draws per CTA (CC_DRAWS / CC_WARPS per warp)

struct MomArgs {
    const double* xy; int64_t nx, ny;
    const double* seeds; int A; const double* poly_xy; const int32_t* poly_off;
    double tie_tol;
    const uint4* buckets; const double* geom; int nb;
    const double* Uy; int ry;
    double* Sy;             // [A][nx][2][ry]
    int* colr;              // [A][2]: first and last column that holds a point of the cell
    int* tie_count;
};

__global__ void cov_moment_basis_kernel(const double* __restrict__ xy, int64_t nx, int64_t ny, double xlo, double xhi, double ylo,
                                        double yhi, int rx, int kpad, int ry, double* __restrict__ Ux, double* __restrict__ Xc,
                                        double* __restrict__ Uy) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nx + ny) return;
    const bool isx = i < nx;
    const double u = isx ? xy[2 * (i * ny)] : xy[2 * (i - nx) + 1];
    const double lo = isx ? xlo : ylo, hi = isx ? xhi : yhi;
    const int r = isx ? rx : ry, w = isx ? kpad : ry;
    double* row = isx ? Ux + i * kpad : Uy + (i - nx) * ry;
    if (isx) Xc[i] = u;
    const double t = (2.0 * u - (lo + hi)) / (hi - lo);      // the recurrence of cheb_basis_kernel (cheb.cuh)
    double t0 = 1.0, t1 = t;
    for (int k = 0; k < w; k++) {
        row[k] = k < r ? t0 : 0.0;
        const double t2 = 2.0 * t * t1 - t0;
        t0 = t1; t1 = t2;
    }
}

__global__ void __launch_bounds__(CM_THREADS) cov_moment_columns_kernel(MomArgs a) {
    __shared__ double s_seeds[2 * COV_MAX_CELLS];
    __shared__ int s_cell[CM_ROWS];
    __shared__ double s_y[CM_ROWS];
    __shared__ unsigned long long s_mask[CM_ROWS][CM_WORDS];
    const int tid = threadIdx.x, lane = tid & 31;
    const int64_t ix = blockIdx.x;
    for (int i = tid; i < 2 * a.A; i += CM_THREADS) s_seeds[i] = a.seeds[i];
    const BucketGrid bg{a.buckets, a.nb, a.geom[0], a.geom[1], a.geom[2]};
    const bool polygon_mode = !(a.tie_tol < 1e300);
    const int ry = a.ry;
    const bool owner = tid < 2 * ry;
    const int m = tid < ry ? 0 : 1, l = tid < ry ? tid : tid - ry;
    const bool ranges = tid == 0;          // thread (0, 0) sees every run of every cell: it keeps the column ranges
    double* __restrict__ sy = a.Sy + (ix * 2 + m) * ry + l;           // + cell * nx * 2 * ry
    const int64_t cstride = a.nx * 2 * ry;
    double acc = 0.0;
    int cur = CELL_NONE;
    auto flush = [&]() {
        if (cur >= 0) {
            sy[cur * cstride] += acc;
            if (ranges) { atomicMin(a.colr + 2 * cur, (int)ix); atomicMax(a.colr + 2 * cur + 1, (int)ix); }
        }
        acc = 0.0;
        cur = CELL_NONE;
    };
    for (int64_t r0 = 0; r0 < a.ny; r0 += CM_ROWS) {
        const int nr = (int)min((int64_t)CM_ROWS, a.ny - r0);
        __syncthreads();                   // the previous pass's rows are consumed (and the seeds are in)
        for (int rb = 0; rb < CM_ROWS; rb += CM_THREADS) {
            const int r = rb + tid;
            const bool valid = r < nr;
            int cell = CELL_NONE;
            double x = 0.0, y = 0.0;
            if (valid) {
                const double2 p = __ldg(reinterpret_cast<const double2*>(a.xy) + ix * a.ny + r0 + r);
                x = p.x; y = p.y;
                cell = polygon_mode ? CELL_TIE : classify_point(bg, s_seeds, a.A, x, y, a.tie_tol);
            }
            const unsigned hm = __ballot_sync(0xffffffffu, cell == CELL_TIE_HARD);
            if (hm && a.tie_count != nullptr && lane == 0) atomicAdd(a.tie_count, __popc(hm));
            if (cell == CELL_TIE_HARD) cell = CELL_TIE;
            if (cell == CELL_TIE) {        // the reference's crossings test against every cell polygon: 0, 1 or several cells
                unsigned long long k0 = 0ull, k1 = 0ull, k2 = 0ull, k3 = 0ull;
                for (int c = 0; c < a.A; c++) {
                    const int o = a.poly_off[c];
                    if (crossings_inside(a.poly_xy + 2 * o, a.poly_off[c + 1] - o, x, y)) {
                        const unsigned long long bit = 1ull << (c & 63);
                        const int w = c >> 6;
                        k0 |= w == 0 ? bit : 0ull; k1 |= w == 1 ? bit : 0ull; k2 |= w == 2 ? bit : 0ull; k3 |= w == 3 ? bit : 0ull;
                    }
                }
                s_mask[r][0] = k0; s_mask[r][1] = k1; s_mask[r][2] = k2; s_mask[r][3] = k3;
            }
            if (valid) { s_cell[r] = cell; s_y[r] = y; }
        }
        __syncthreads();
        if (owner) {
            const double* __restrict__ uy = a.Uy + r0 * ry + l;
            for (int r = 0; r < nr; r++) {
                const int c = s_cell[r];
                const double u = __ldg(uy + (int64_t)r * ry);
                const double v = m ? s_y[r] * u : u;
                if (c >= 0) {
                    if (c != cur) { flush(); cur = c; }
                    acc += v;
                } else {
                    flush();
#pragma unroll
                    for (int w = 0; w < CM_WORDS; w++) {
                        unsigned long long mk = s_mask[r][w];
                        while (mk) {
                            const int cc = 64 * w + __ffsll((long long)mk) - 1;
                            mk &= mk - 1;
                            sy[cc * cstride] += v;
                            if (ranges) { atomicMin(a.colr + 2 * cc, (int)ix); atomicMax(a.colr + 2 * cc + 1, (int)ix); }
                        }
                    }
                }
            }
        }
    }
    if (owner) flush();
}

__global__ void cov_moment_init_kernel(int* __restrict__ colr, int A) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < A) { colr[2 * i] = INT_MAX; colr[2 * i + 1] = -1; }
}

// Mom[i][0] = Ux^T Sy_i[., 0], Mom[i][1] = (x Ux)^T Sy_i[., 0], Mom[i][2] = Ux^T Sy_i[., 1] over the columns cell i touches.
// Thread (tl, tk) owns the terms l = tl + 16 a, k = tk + 16 b (a, b < 4): 48 accumulators in registers, columns in order.
__global__ void __launch_bounds__(256) cov_moment_reduce_kernel(const double* __restrict__ Sy, const int* __restrict__ colr,
                                                                const double* __restrict__ Ux, const double* __restrict__ Xc,
                                                                int64_t nx, int ry, int kpad, double* __restrict__ mom) {
    __shared__ double s_sy[CR_COLS][2][CM_MAXR];
    __shared__ double s_ux[CR_COLS][CM_MAXR];
    __shared__ double s_x[CR_COLS];
    const int c = blockIdx.x, tid = threadIdx.x;
    const int tl = tid >> 4, tk = tid & 15;
    const int c0 = colr[2 * c], c1 = colr[2 * c + 1];
    double acc[3][4][4];
#pragma unroll
    for (int q = 0; q < 3; q++)
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
            for (int j = 0; j < 4; j++) acc[q][i][j] = 0.0;
    const double* syc = Sy + (int64_t)c * nx * 2 * ry;
    for (int64_t b0 = c0; b0 <= c1; b0 += CR_COLS) {      // empty cell: c1 = -1 < c0, no iteration
        const int nc = (int)min((int64_t)CR_COLS, (int64_t)c1 + 1 - b0);
        __syncthreads();
        for (int e = tid; e < nc * 2 * ry; e += 256) {
            const int q = e / (2 * ry), rem = e % (2 * ry);
            s_sy[q][rem / ry][rem % ry] = syc[(b0 + q) * 2 * ry + rem];
        }
        for (int e = tid; e < nc * kpad; e += 256) s_ux[e / kpad][e % kpad] = Ux[(b0 + e / kpad) * kpad + e % kpad];
        if (tid < nc) s_x[tid] = Xc[b0 + tid];
        __syncthreads();
        for (int q = 0; q < nc; q++) {
            double a0[4], a1[4], u[4], ux[4];
            const double xq = s_x[q];
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int ll = tl + 16 * i;
                a0[i] = ll < ry ? s_sy[q][0][ll] : 0.0;
                a1[i] = ll < ry ? s_sy[q][1][ll] : 0.0;
            }
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int k = tk + 16 * j;
                u[j] = k < kpad ? s_ux[q][k] : 0.0;
                ux[j] = xq * u[j];
            }
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    acc[0][i][j] = fma(a0[i], u[j], acc[0][i][j]);
                    acc[1][i][j] = fma(a0[i], ux[j], acc[1][i][j]);
                    acc[2][i][j] = fma(a1[i], u[j], acc[2][i][j]);
                }
        }
    }
    const int64_t R = (int64_t)ry * kpad;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int ll = tl + 16 * i;
        if (ll >= ry) continue;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int k = tk + 16 * j;
            if (k >= kpad) continue;
#pragma unroll
            for (int q = 0; q < 3; q++) mom[((int64_t)c * 3 + q) * R + ll * kpad + k] = acc[q][i][j];
        }
    }
}

// cent[s][i] = (sum F_s, sum F_s x, sum F_s y, n) of cell i = <C'_s, Mom_i^{1,x,y}>, n = Mom_i^1[0][0] (an exact count: T_0 = 1);
// centroids[s][i] with cov_finish's arithmetic: ((m/n) area) / ((m0/n) area), then the one-sided clamps (NaN stays NaN).
__global__ void __launch_bounds__(CC_WARPS * 32) cov_moment_centroid_kernel(const double* __restrict__ mom, int A, int R,
                                                                            const double* __restrict__ C, int S, double mean,
                                                                            const double* __restrict__ areas, double xmin,
                                                                            double xmax, double ymin, double ymax,
                                                                            double* __restrict__ cent, double* __restrict__ cen) {
    extern __shared__ __align__(16) double s_mom[];     // [3][R]
    const int c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int e = tid; e < 3 * R; e += CC_WARPS * 32) s_mom[e] = mom[(int64_t)c * 3 * R + e];
    __syncthreads();
    const double n = s_mom[0], area = areas[c];
    for (int si = warp; si < CC_DRAWS; si += CC_WARPS) {
        const int s = blockIdx.y * CC_DRAWS + si;
        if (s >= S) break;
        const double* cs = C + (int64_t)s * R;
        double m0 = 0.0, m1 = 0.0, m2 = 0.0;
        for (int e = lane; e < R; e += 32) {
            const double v = e == 0 ? cs[0] + mean : cs[e];
            m0 = fma(v, s_mom[e], m0);
            m1 = fma(v, s_mom[R + e], m1);
            m2 = fma(v, s_mom[2 * R + e], m2);
        }
        m0 = warp_sum(m0); m1 = warp_sum(m1); m2 = warp_sum(m2);
        if (lane == 0) {
            double* o = cent + ((int64_t)s * A + c) * 4;
            o[0] = m0; o[1] = m1; o[2] = m2; o[3] = n;
            const double f_int = __dmul_rn(__ddiv_rn(m0, n), area);
            double cx = __ddiv_rn(__dmul_rn(__ddiv_rn(m1, n), area), f_int);
            double cy = __ddiv_rn(__dmul_rn(__ddiv_rn(m2, n), area), f_int);
            if (cx < xmin) cx = xmin;
            if (cx > xmax) cx = xmax;
            if (cy < ymin) cy = ymin;
            if (cy > ymax) cy = ymax;
            cen[((int64_t)s * A + c) * 2] = cx;
            cen[((int64_t)s * A + c) * 2 + 1] = cy;
        }
    }
}

struct MomLayout { double *Sy, *Ux, *Xc, *Uy; int* colr; uint4* buckets; double* geom; int64_t bytes; };
inline int64_t cm_rup(int64_t v) { return (v + 255) / 256 * 256; }
inline MomLayout cm_layout(int64_t nx, int64_t ny, int64_t A, int64_t rx, int64_t ry, void* work) {
    const int64_t kpad = (rx + 3) / 4 * 4;
    char* base = static_cast<char*>(work);
    int64_t used = 0;
    auto carve = [&](int64_t bytes) { char* p = base ? base + used : nullptr; used += cm_rup(bytes); return p; };
    MomLayout L{};
    L.Sy = reinterpret_cast<double*>(carve(A * nx * 2 * ry * 8));
    L.Ux = reinterpret_cast<double*>(carve(nx * kpad * 8));
    L.Xc = reinterpret_cast<double*>(carve(nx * 8));
    L.Uy = reinterpret_cast<double*>(carve(ny * ry * 8));
    L.colr = reinterpret_cast<int*>(carve(A * 2 * 4));
    L.buckets = reinterpret_cast<uint4*>(carve((int64_t)COV_BUCKETS_MAX * COV_BUCKETS_MAX * 16));
    L.geom = reinterpret_cast<double*>(carve(64));
    L.bytes = used;
    return L;
}
inline bool cm_al(const void* p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }
inline bool cm_box_ok(double lo, double hi) { return hi > lo && std::isfinite(hi - lo); }
}  // namespace mfgp

extern "C" int64_t cov_cell_moments_workspace_bytes(int64_t nx, int64_t ny, int64_t A, int64_t rx, int64_t ry) {
    if (nx <= 0 || ny <= 0 || A <= 0 || A > COV_MAX_CELLS || rx <= 0 || rx > CM_MAXR || ry <= 0 || ry > CM_MAXR) return 0;
    return cm_layout(nx, ny, A, rx, ry, nullptr).bytes;
}

extern "C" int cov_cell_moments(const double* xy, int64_t nx, int64_t ny, const double* seeds, int64_t A, const double* poly_xy,
                                const int32_t* poly_off, double tie_tol, double xlo, double xhi, double ylo, double yhi, int64_t rx,
                                int64_t ry, double* mom, int32_t* tie_count, void* work, int64_t work_bytes, void* stream) {
    if (!xy || !seeds || !poly_xy || !poly_off || !mom || !work) return MFGP_ERR_INVALID;
    if (nx <= 0 || ny <= 0 || nx >= (1LL << 31) - 1 || ny >= (1LL << 40) / nx || A <= 0 || A > COV_MAX_CELLS) return MFGP_ERR_INVALID;
    if (rx <= 0 || rx > CM_MAXR || ry <= 0 || ry > CM_MAXR || tie_tol != tie_tol || tie_tol < 0.0) return MFGP_ERR_INVALID;
    if (!cm_box_ok(xlo, xhi) || !cm_box_ok(ylo, yhi)) return MFGP_ERR_INVALID;
    if (!cm_al(xy, 16) || !cm_al(poly_xy, 16) || !cm_al(seeds, 8) || !cm_al(poly_off, 4) || !cm_al(mom, 16) || !cm_al(work, 16) ||
        !cm_al(tie_count, 4))
        return MFGP_ERR_INVALID;
    if (work_bytes < cm_layout(nx, ny, A, rx, ry, nullptr).bytes) return MFGP_ERR_INVALID;
    const MomLayout L = cm_layout(nx, ny, A, rx, ry, work);
    const int kpad = (int)((rx + 3) / 4 * 4);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (tie_count) MFGP_CUDA_CHECK(cudaMemsetAsync(tie_count, 0, sizeof(int32_t), st));
    MFGP_CUDA_CHECK(cudaMemsetAsync(L.Sy, 0, sizeof(double) * A * nx * 2 * ry, st));
    cov_moment_init_kernel<<<(unsigned)((A + 255) / 256), 256, 0, st>>>(L.colr, (int)A);
    MFGP_LAUNCH_CHECK();
    const int nb = cov_bucket_side(A);
    BucketBuild bb{seeds, (int)A, poly_xy, poly_off, nb, L.buckets, L.geom};
    cov_build_buckets_kernel<<<dim3((unsigned)((nb * nb + 7) / 8), 1), 256, 0, st>>>(bb, bb, tie_tol);
    MFGP_LAUNCH_CHECK();
    cov_moment_basis_kernel<<<(unsigned)((nx + ny + 127) / 128), 128, 0, st>>>(xy, nx, ny, xlo, xhi, ylo, yhi, (int)rx, kpad, (int)ry,
                                                                              L.Ux, L.Xc, L.Uy);
    MFGP_LAUNCH_CHECK();
    MomArgs a{xy, nx, ny, seeds, (int)A, poly_xy, poly_off, tie_tol, L.buckets, L.geom, nb, L.Uy, (int)ry, L.Sy, L.colr, tie_count};
    cov_moment_columns_kernel<<<(unsigned)nx, CM_THREADS, 0, st>>>(a);
    MFGP_LAUNCH_CHECK();
    cov_moment_reduce_kernel<<<(unsigned)A, 256, 0, st>>>(L.Sy, L.colr, L.Ux, L.Xc, nx, (int)ry, kpad, mom);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

extern "C" int64_t cov_cell_moments_centroids_workspace_bytes(int64_t A, int64_t rx, int64_t ry, int64_t S) {
    (void)A; (void)rx; (void)ry; (void)S;
    return 0;
}

extern "C" int cov_cell_moments_centroids(const double* mom, int64_t A, int64_t rx, int64_t ry, const double* C, int64_t S, double mean,
                                          const double* areas, double xmin, double xmax, double ymin, double ymax, double* cent,
                                          double* centroids, void* work, int64_t work_bytes, void* stream) {
    (void)work;
    if (!mom || !C || !areas || !cent || !centroids || work_bytes < 0) return MFGP_ERR_INVALID;
    if (A <= 0 || A > COV_MAX_CELLS || rx <= 0 || rx > CM_MAXR || ry <= 0 || ry > CM_MAXR || S <= 0 || S >= (1LL << 21))
        return MFGP_ERR_INVALID;
    if (!cm_al(mom, 16) || !cm_al(C, 16) || !cm_al(areas, 8) || !cm_al(cent, 16) || !cm_al(centroids, 16)) return MFGP_ERR_INVALID;
    const int R = (int)(ry * ((rx + 3) / 4 * 4));
    const int smem = 3 * R * (int)sizeof(double);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MFGP_CUDA_CHECK(cudaFuncSetAttribute(cov_moment_centroid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    cov_moment_centroid_kernel<<<dim3((unsigned)A, (unsigned)((S + CC_DRAWS - 1) / CC_DRAWS)), CC_WARPS * 32, smem, st>>>(
        mom, (int)A, R, C, (int)S, mean, areas, xmin, xmax, ymin, ymax, cent, centroids);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

extern "C" int cov_finish(const double* cent, const double* areas_c, int64_t Ac, const double* lossp, const double* areas_p,
                          int64_t Ap, const double* amax_val, const int64_t* amax_idx, double xmin, double xmax, double ymin,
                          double ymax, const int32_t* flag0, const int32_t* flag1, const int32_t* flag2, const int32_t* flag3,
                          double* out, void* stream) {
    if (!out || Ac < 0 || Ap < 0 || (Ac && (!cent || !areas_c)) || (Ap && (!lossp || !areas_p))) return MFGP_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int n = (int)(Ac > 1 ? Ac : 1);
    cov_finish_kernel<<<(n + 127) / 128, 128, 0, st>>>(cent, areas_c, (int)Ac, lossp, areas_p, (int)Ap, amax_val, amax_idx, xmin, xmax,
                                                      ymin, ymax, flag0, flag1, flag2, flag3, out);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}
