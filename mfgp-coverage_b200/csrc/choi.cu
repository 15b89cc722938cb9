// Choi greedy sample planner on the cached V = L^-1 Psi^T (replaces compute_sample_points, reference
// simulator.py:326-374, which refits and re-predicts the whole grid for every pick).
//
// Every candidate is a grid point, so appending pick j to the training set is a bordered Cholesky step whose new
// factor row is the cached column l = V[:, j]:  d = sqrt(k(0) + noise_H + jitter - l.l),
// v[g] = (k_HH(x_g, x_j) - sum_n l[n] V[n, g]) / d,  var[g] -= v[g]^2.  The pseudo-observation equals the current
// mean, so the posterior mean does not change (SURVEY.md section 7 step 5).  One pick = one pass over V: 8*n*G bytes,
// HBM-bound.  The same kernel produces the block-level candidates of the next first-index argmax.
#include <cfloat>

#include "common.cuh"
#include "argmax.cuh"

namespace mfgp {

constexpr int CH_THREADS = 128;
constexpr int CH_COLS = CH_THREADS * 2;

// Device-resident loop state: the host launches a BATCH of (append, arg-max) pairs without synchronising; each pair
// checks `done` / the threshold on the device, so the greedy loop costs one host round trip per batch, not per pick.
struct ChoiState {
    long long n;          // valid rows of the V cache
    long long picks;      // picks recorded so far (all batches)
    long long done;       // 1: max var <= threshold or a limit was reached -> remaining launches of the batch are no-ops
    long long pick;       // grid index to append next (the current first-index arg-max)
    double val;           // its variance
};

struct ChoiArgs {
    const double* Xs; int64_t G;
    double* Vc; int64_t ldv;                 // rows [0, state->n) valid; row state->n is written
    double* var;
    ChoiState* state;
    DevParams p;
    TieRule tol;                             // arg-max tie rule
    double* q;                               // running sum of v^2 per grid point (variance reduction)
    double* pv; long long* pi;               // per-block argmax candidates of the updated variance
    double threshold; long long cap; long long max_picks;
    long long* picks_dev;                    // [max_picks] grid indices in selection order
};

// The append pass over one cache.  The picked point's column l = V[0:n, j] is read from `lcol` with row stride `lstride`
// and its coordinates from `xyj`: the own cache and Xs on one GPU, the staged winner slot on a grid shard.  `base` is the
// global grid index of local point 0, so the block candidates carry global indices.
__device__ __forceinline__ void choi_append_body(const ChoiArgs& a, const double* lcol, int64_t lstride, const double* xyj,
                                                 int64_t base) {
    extern __shared__ __align__(16) double l[];   // [n]
    __shared__ double red[CH_THREADS / 32];
    __shared__ double sv[CH_THREADS / 32];
    __shared__ long long si[CH_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int an = (int)a.state->n;
    double part = 0.0;
    for (int n = tid; n < an; n += CH_THREADS) {
        const double v = lcol[(int64_t)n * lstride];
        l[n] = v;
        part += v * v;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (lane == 0) red[warp] = part;
    __syncthreads();
    double ll = 0.0;
#pragma unroll
    for (int w = 0; w < CH_THREADS / 32; w++) ll += red[w];
    const DevParams& p = a.p;
    const double d = sqrt(p.k0 + p.noise_H + p.jitter - ll);
    const double xj = xyj[0], yj = xyj[1];

    const int64_t g = (int64_t)blockIdx.x * CH_COLS + tid * 2;
    ArgMax best{0.0, -1};
    if (g < a.G) {
        const bool pair = (g + 1 < a.G) && ((a.ldv & 1) == 0);
        double s0 = 0.0, s1 = 0.0;
        if (pair) {
            const double* col = a.Vc + g;
            int n = 0;
            for (; n + 16 <= an; n += 16) {       // 16 x 16 B in flight per thread: the pass over V is HBM-bound
                double2 v[16];
#pragma unroll
                for (int u = 0; u < 16; u++) v[u] = __ldcs(reinterpret_cast<const double2*>(col + (int64_t)(n + u) * a.ldv));
#pragma unroll
                for (int u = 0; u < 16; u++) { s0 += l[n + u] * v[u].x; s1 += l[n + u] * v[u].y; }
            }
            for (; n < an; n++) {
                const double2 v = *reinterpret_cast<const double2*>(col + (int64_t)n * a.ldv);
                s0 += l[n] * v.x; s1 += l[n] * v.y;
            }
        } else {
            for (int n = 0; n < an; n++) {
                s0 += l[n] * a.Vc[(int64_t)n * a.ldv + g];
                if (g + 1 < a.G) s1 += l[n] * a.Vc[(int64_t)n * a.ldv + g + 1];
            }
        }
#pragma unroll
        for (int c = 0; c < 2; c++) {
            const int64_t gg = g + c;
            if (gg < a.G) {
                const double x = a.Xs[2 * gg], y = a.Xs[2 * gg + 1];
                double k;
                const double kH = rbf_scaled(xj / p.l_H, yj / p.l_H, x / p.l_H, y / p.l_H, p.s_H);
                if (p.multi) {
                    const double kL = rbf_scaled(xj / p.l_L, yj / p.l_L, x / p.l_L, y / p.l_L, p.s_L);
                    k = __dadd_rn(__dmul_rn(p.rho2, kL), kH);
                } else {
                    k = kH;
                }
                const double v = (k - (c ? s1 : s0)) / d;
                a.Vc[(int64_t)an * a.ldv + gg] = v;
                const double nq = a.q[gg] + v * v;         // var is recomputed from the accumulated reduction, as the
                a.q[gg] = nq;                              // reference's full predict does (k** - psi beta), never decremented
                const double nv = p.k0 - nq;
                a.var[gg] = nv;
                best = argmax_combine(best, ArgMax{nv, (long long)(base + gg)}, a.tol);
            }
        }
    }
    best = argmax_warp(best, a.tol);
    if (lane == 0) { sv[warp] = best.v; si[warp] = best.i; }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < CH_THREADS / 32; w++) best = argmax_combine(best, ArgMax{sv[w], si[w]}, a.tol);
        a.pv[blockIdx.x] = best.v; a.pi[blockIdx.x] = best.i;
    }
}

__global__ void __launch_bounds__(CH_THREADS) choi_append_kernel(ChoiArgs a) {
    if (a.state->done) return;                    // uniform for the whole grid
    const int64_t j = a.state->pick;
    choi_append_body(a, a.Vc + j, a.ldv, a.Xs + 2 * j, 0);
}

// One warp: the row just written becomes valid, the block candidates give the next arg-max, and the loop condition of
// simulator.py:345 (`while max_var > threshold`) is evaluated on the device.
__global__ void choi_advance_kernel(ChoiArgs a, int nblocks, int first) {
    ChoiState* st = a.state;
    if (st->done) return;
    ArgMax best{0.0, -1};
    if (first) {            // the arg-max of the incoming variance was computed by cov_argmax into (val, pick)
        best = ArgMax{st->val, st->pick};
    } else {
        for (int i = threadIdx.x; i < nblocks; i += 32) best = argmax_combine(best, ArgMax{a.pv[i], a.pi[i]}, a.tol);
        best = argmax_warp(best, a.tol);
    }
    if (threadIdx.x == 0) {
        if (!first) st->n += 1;
        st->val = best.v;
        st->pick = best.i;
        if (!(best.v > a.threshold) || st->picks >= a.max_picks || st->n >= a.cap) st->done = 1;
        else a.picks_dev[st->picks++] = best.i;
    }
}

// ---- grid-sharded planner -------------------------------------------------------------------------------------------
// Each rank owns the whole-column slice [base, base + G) of the grid and the V cache, q and var of that slice.  One pick:
//   append  (choi_shard_append_kernel): the pass above over the local slice, l and (x_j, y_j) from the staged winner slot;
//   propose (choi_shard_propose_kernel): the shard's candidate into a send slot of cap + 4 doubles
//            [value, index bits, x_j, y_j, V[0:n, j_local]], index -1 when the shard has none or the plan is done;
//   the host all-gathers the slots of every rank (rank order);
//   select  (choi_shard_select_kernel): fold the slots in rank order with argmax_combine (a tie goes to the lowest
//            global index, as on one GPU), apply the loop condition of choi_advance_kernel, record the pick and stage the
//            winner's slot for the next append.
// The select is deterministic and sees the same slots on every rank, so every rank holds the same state.

struct ShardState {
    ChoiState c;
    long long fresh;      // 1 between begin and the first select: (val, pick) is the slice's cov_argmax, no row was appended
};

struct ShardLayout {
    ShardState* st;
    long long* picks;     // [cap + 1] global grid indices in selection order
    double* stage;        // [cap + 4] the winner's slot of the last select
    double* pv; long long* pi;
    void* awork; int64_t awork_bytes;
    int nblocks;
};

// work: ShardState (128 B), picks, stage, block candidates, cov_argmax workspace (256-byte aligned).
inline int64_t shard_layout(int64_t G, int64_t cap, void* work, int64_t work_bytes, ShardLayout* L) {
    const int nblocks = (int)((G + CH_COLS - 1) / CH_COLS);
    const int64_t head = 128 + (cap + 1) * 8 + (cap + 4) * 8 + (int64_t)nblocks * 16;
    const int64_t aoff = (head + 255) / 256 * 256;
    const int64_t need = aoff + cov_workspace_bytes(G, 1, 0);
    if (L) {
        char* w = static_cast<char*>(work);
        L->st = reinterpret_cast<ShardState*>(w);
        L->picks = reinterpret_cast<long long*>(w + 128);
        L->stage = reinterpret_cast<double*>(L->picks + cap + 1);
        L->pv = L->stage + cap + 4;
        L->pi = reinterpret_cast<long long*>(L->pv + nblocks);
        L->awork = w + aoff;
        L->awork_bytes = work_bytes - aoff;
        L->nblocks = nblocks;
    }
    return need;
}

__global__ void __launch_bounds__(CH_THREADS) choi_shard_append_kernel(ChoiArgs a, const double* stage, int64_t base) {
    if (a.state->done) return;                    // uniform for the whole grid
    choi_append_body(a, stage + 4, 1, stage + 2, base);
}

// One block: warp 0 folds the block candidates (or takes the slice's cov_argmax after begin), the block copies the column.
__global__ void __launch_bounds__(CH_THREADS) choi_shard_propose_kernel(ChoiArgs a, ShardState* ss, int nblocks, int64_t base,
                                                                        double* send) {
    __shared__ long long win;
    const ChoiState* st = &ss->c;
    if (threadIdx.x < 32) {
        ArgMax best{0.0, -1};
        if (!st->done) {
            if (ss->fresh) {
                best = ArgMax{st->val, st->pick};
            } else {
                for (int i = threadIdx.x; i < nblocks; i += 32) best = argmax_combine(best, ArgMax{a.pv[i], a.pi[i]}, a.tol);
                best = argmax_warp(best, a.tol);
            }
        }
        if (threadIdx.x == 0) {
            send[0] = best.v;
            send[1] = __longlong_as_double(best.i);
            if (best.i >= 0) {
                send[2] = a.Xs[2 * (best.i - base)];
                send[3] = a.Xs[2 * (best.i - base) + 1];
            }
            win = best.i;
        }
    }
    __syncthreads();
    if (win < 0) return;
    const int64_t jl = win - base;
    const int64_t rows = st->n + (ss->fresh ? 0 : 1);       // the append's row is valid from here on
    for (int64_t r = threadIdx.x; r < rows; r += blockDim.x) send[4 + r] = a.Vc[r * a.ldv + jl];
}

// One block: thread 0 folds the `world` slots in rank order and advances the state, the block stages the winner's slot.
__global__ void __launch_bounds__(CH_THREADS) choi_shard_select_kernel(ChoiArgs a, ShardState* ss, const double* recv, int world,
                                                                       int64_t width, double* stage) {
    __shared__ int win;
    __shared__ long long rows;
    ChoiState* st = &ss->c;
    if (threadIdx.x == 0) {
        win = -1;
        rows = 0;
    }
    if (threadIdx.x == 0 && !st->done) {         // only thread 0 reads or writes the state
        ArgMax best{0.0, -1};
        for (int r = 0; r < world; r++)
            best = argmax_combine(best, ArgMax{recv[r * width], __double_as_longlong(recv[r * width + 1])}, a.tol);
        if (!ss->fresh) st->n += 1;
        ss->fresh = 0;
        st->val = best.v;
        st->pick = best.i;
        if (best.i < 0 || !(best.v > a.threshold) || st->picks >= a.max_picks || st->n >= a.cap) {
            st->done = 1;
        } else {
            a.picks_dev[st->picks++] = best.i;
            for (int r = 0; r < world; r++)
                if (__double_as_longlong(recv[r * width + 1]) == best.i) { win = r; break; }
        }
        rows = st->n;
    }
    __syncthreads();
    if (win < 0) return;
    const double* s = recv + (int64_t)win * width;
    for (int64_t k = threadIdx.x; k < rows + 4; k += blockDim.x) stage[k] = s[k];
}

}  // namespace mfgp

using namespace mfgp;

extern "C" int64_t choi_greedy(const double* Xs, int64_t G, double* Vc, int64_t ldv, int64_t n0, int64_t cap, double* var,
                               double* q, const mfgp_params* p_host, double threshold, double tie_rel, int64_t max_picks,
                               int64_t* picks_host,
                               void* work, int64_t work_bytes, void* stream) {
    if (!Xs || !Vc || !var || !q || !p_host || !picks_host || !work || G <= 0 || ldv < G || n0 < 0 || cap < n0) return MFGP_ERR_INVALID;
    if (max_picks > cap - n0) max_picks = cap - n0;           // the V cache holds cap rows: the caller grows it and resumes
    const int nblocks = (int)((G + CH_COLS - 1) / CH_COLS);
    const int64_t need = (int64_t)nblocks * 16 + 128 + (max_picks + 1) * 8 + cov_workspace_bytes(G, 1, 0);
    if (work_bytes < need) return MFGP_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    double* pv = static_cast<double*>(work);
    long long* pi = reinterpret_cast<long long*>(pv + nblocks);
    ChoiState* state = reinterpret_cast<ChoiState*>(pi + nblocks);
    long long* picks_dev = reinterpret_cast<long long*>(state + 2);
    void* awork = picks_dev + max_picks + 1;
    const int64_t awork_bytes = work_bytes - ((char*)awork - (char*)work);
    const DevParams dp = make_dev_params(*p_host);
    const TieRule tol{dp.k0, tie_rel > 0.0 ? tie_rel : 0.0};
    ChoiState h{n0, 0, 0, -1, 0.0};
    MFGP_CUDA_CHECK(cudaMemcpyAsync(state, &h, sizeof(h), cudaMemcpyHostToDevice, st));
    int rc = cov_argmax(var, G, 0, tol.k0, tol.rel, &state->val, reinterpret_cast<int64_t*>(&state->pick), awork, awork_bytes, st);
    if (rc) return rc;
    ChoiArgs a;
    a.Xs = Xs; a.G = G; a.Vc = Vc; a.ldv = ldv; a.var = var; a.state = state; a.p = dp; a.tol = tol; a.q = q; a.pv = pv; a.pi = pi;
    a.threshold = threshold; a.cap = cap; a.max_picks = max_picks; a.picks_dev = picks_dev;
    choi_advance_kernel<<<1, 32, 0, st>>>(a, nblocks, 1);
    MFGP_LAUNCH_CHECK();
    constexpr int BATCH = 16;
    int64_t n_hi = n0;                // upper bound of state->n known to the host (sizes the shared-memory column)
    while (true) {
        for (int b = 0; b < BATCH; b++) {
            n_hi++;
            const size_t smem = sizeof(double) * (size_t)n_hi;
            if (smem > 48 * 1024)
                MFGP_CUDA_CHECK(cudaFuncSetAttribute(choi_append_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            choi_append_kernel<<<nblocks, CH_THREADS, smem, st>>>(a);
            MFGP_LAUNCH_CHECK();
            choi_advance_kernel<<<1, 32, 0, st>>>(a, nblocks, 0);
            MFGP_LAUNCH_CHECK();
        }
        MFGP_CUDA_CHECK(cudaMemcpyAsync(&h, state, sizeof(h), cudaMemcpyDeviceToHost, st));
        MFGP_CUDA_CHECK(cudaStreamSynchronize(st));
        if (h.done) break;
        n_hi = h.n;
    }
    if (h.picks > 0) {
        MFGP_CUDA_CHECK(cudaMemcpyAsync(picks_host, picks_dev, sizeof(long long) * h.picks, cudaMemcpyDeviceToHost, st));
        MFGP_CUDA_CHECK(cudaStreamSynchronize(st));
    }
    return h.picks;
}

extern "C" int64_t choi_shard_workspace_bytes(int64_t G, int64_t cap) {
    if (G <= 0 || cap < 0) return MFGP_ERR_INVALID;
    return shard_layout(G, cap, nullptr, 0, nullptr);
}

static ChoiArgs shard_args(const ShardLayout& L, const double* Xs, int64_t G, const double* Vc, int64_t ldv, double* var, double* q,
                           const mfgp_params* p_host, double tie_rel) {
    ChoiArgs a{};
    a.Xs = Xs; a.G = G; a.Vc = const_cast<double*>(Vc); a.ldv = ldv; a.var = var; a.q = q; a.state = &L.st->c;
    a.p = make_dev_params(*p_host);
    a.tol = TieRule{a.p.k0, tie_rel > 0.0 ? tie_rel : 0.0};
    a.pv = L.pv; a.pi = L.pi; a.picks_dev = L.picks;
    return a;
}

extern "C" int choi_shard_begin(const double* Xs, int64_t G, int64_t base, const double* Vc, int64_t ldv, int64_t n0, int64_t cap,
                                const double* var, const mfgp_params* p_host, double tie_rel, double* send, void* work,
                                int64_t work_bytes, void* stream) {
    if (!Xs || !Vc || !var || !p_host || !send || !work || G <= 0 || base < 0 || ldv < G || n0 < 0 || cap < n0)
        return MFGP_ERR_INVALID;
    ShardLayout L;
    if (work_bytes < shard_layout(G, cap, work, work_bytes, &L)) return MFGP_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const ChoiArgs a = shard_args(L, Xs, G, Vc, ldv, nullptr, nullptr, p_host, tie_rel);
    const ShardState h{{n0, 0, 0, -1, 0.0}, 1};
    MFGP_CUDA_CHECK(cudaMemcpyAsync(L.st, &h, sizeof(h), cudaMemcpyHostToDevice, st));
    int rc = cov_argmax(var, G, base, a.tol.k0, a.tol.rel, &L.st->c.val, reinterpret_cast<int64_t*>(&L.st->c.pick), L.awork,
                        L.awork_bytes, st);
    if (rc) return rc;
    choi_shard_propose_kernel<<<1, CH_THREADS, 0, st>>>(a, L.st, 0, base, send);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

extern "C" int choi_shard_append(const double* Xs, int64_t G, int64_t base, double* Vc, int64_t ldv, int64_t cap, double* var,
                                 double* q, const mfgp_params* p_host, double tie_rel, void* work, int64_t work_bytes,
                                 void* stream) {
    if (!Xs || !Vc || !var || !q || !p_host || !work || G <= 0 || base < 0 || ldv < G || cap < 0) return MFGP_ERR_INVALID;
    ShardLayout L;
    if (work_bytes < shard_layout(G, cap, work, work_bytes, &L)) return MFGP_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const ChoiArgs a = shard_args(L, Xs, G, Vc, ldv, var, q, p_host, tie_rel);
    const size_t smem = sizeof(double) * (size_t)(cap > 0 ? cap : 1);     // the column l: n < cap rows while planning
    if (smem > 48 * 1024)
        MFGP_CUDA_CHECK(cudaFuncSetAttribute(choi_shard_append_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    choi_shard_append_kernel<<<L.nblocks, CH_THREADS, smem, st>>>(a, L.stage, base);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

extern "C" int choi_shard_propose(const double* Xs, int64_t G, int64_t base, const double* Vc, int64_t ldv, int64_t cap,
                                  const mfgp_params* p_host, double tie_rel, double* send, void* work, int64_t work_bytes,
                                  void* stream) {
    if (!Xs || !Vc || !p_host || !send || !work || G <= 0 || base < 0 || ldv < G || cap < 0) return MFGP_ERR_INVALID;
    ShardLayout L;
    if (work_bytes < shard_layout(G, cap, work, work_bytes, &L)) return MFGP_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const ChoiArgs a = shard_args(L, Xs, G, Vc, ldv, nullptr, nullptr, p_host, tie_rel);
    choi_shard_propose_kernel<<<1, CH_THREADS, 0, st>>>(a, L.st, L.nblocks, base, send);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

extern "C" int choi_shard_select(const double* recv, int64_t world, int64_t G, int64_t cap, const mfgp_params* p_host,
                                 double threshold, double tie_rel, int64_t max_picks, void* work, int64_t work_bytes,
                                 void* stream) {
    if (!recv || !p_host || !work || world <= 0 || world > (1 << 20) || G <= 0 || cap < 0 || max_picks < 0) return MFGP_ERR_INVALID;
    ShardLayout L;
    if (work_bytes < shard_layout(G, cap, work, work_bytes, &L)) return MFGP_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ChoiArgs a = shard_args(L, nullptr, G, nullptr, 0, nullptr, nullptr, p_host, tie_rel);
    a.threshold = threshold; a.cap = cap; a.max_picks = max_picks < cap ? max_picks : cap;
    choi_shard_select_kernel<<<1, CH_THREADS, 0, st>>>(a, L.st, recv, (int)world, cap + 4, L.stage);
    MFGP_LAUNCH_CHECK();
    return MFGP_OK;
}

extern "C" int choi_shard_status(int64_t G, int64_t cap, const void* work, int64_t work_bytes, int64_t* status_host,
                                 int64_t* picks_host, void* stream) {
    if (!work || !status_host || G <= 0 || cap < 0) return MFGP_ERR_INVALID;
    ShardLayout L;
    if (work_bytes < shard_layout(G, cap, const_cast<void*>(work), work_bytes, &L)) return MFGP_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ChoiState h;
    MFGP_CUDA_CHECK(cudaMemcpyAsync(&h, &L.st->c, sizeof(h), cudaMemcpyDeviceToHost, st));
    MFGP_CUDA_CHECK(cudaStreamSynchronize(st));
    status_host[0] = h.n; status_host[1] = h.picks; status_host[2] = h.done;
    if (picks_host && h.picks > 0) {
        MFGP_CUDA_CHECK(cudaMemcpyAsync(picks_host, L.picks, sizeof(long long) * h.picks, cudaMemcpyDeviceToHost, st));
        MFGP_CUDA_CHECK(cudaStreamSynchronize(st));
    }
    return MFGP_OK;
}
