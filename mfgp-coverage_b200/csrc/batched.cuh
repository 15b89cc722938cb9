// Argument block and small helpers of the batched replicate stepper, shared by its step kernels (batched.cu) and the
// Thompson draw stage (batched_thompson.cu).
#pragma once
#include "common.cuh"

namespace mfgp {

constexpr int BT_THREADS = 256;
constexpr int BT_MAXA = 16;          // agents per run
constexpr int BT_LOGC = 11;          // X, Y, XMax, YMax, VarMax, Var0, XCentroid, YCentroid, ProbExplore, Explore, Distance

struct BatchArgs {
    int runs, G, nx, ny, A, NL, cap, algo, iterations, max_samples;      // algo: 0 lloyd, 1 periodic, 2 todescato, 3 choi, 4 thompson
    double xmin, xmax, ymin, ymax, eps, tie_tol, amax_rel;
    DevParams p;
    const double* xy; const double* f; const double* ux; const double* uy;
    double* Xt; double* y; double* W; double* z;                         // [runs][cap(,2 | ,cap)]
    double* TxL; double* TyL; double* TxH; double* TyH;                  // [runs][cap][nx | ny]
    double* mu; double* var;                                             // [runs][G]
    double* pos; double* prev; double* cen;                              // [runs][A][2]
    long long* pos_idx;                                                  // [runs][A] grid index of the position, or -1
    double* prob; int* explore;                                          // [runs][A]
    int* Ncur; int* knew; int* status; int* noise_used; int* nsamples;   // [runs]
    int* ties;                                                           // [runs][iterations]
    const double* noise; const double* unif;                             // [runs][max_samples], [runs][iterations][A]
    double* log_loss; double* log_agent; double* log_sample;             // [runs][it], [runs][it][A][BT_LOGC], [runs][max_samples][5]
    double* q; long long* picks; int* nplan; int* plan_state;            // Choi planner: [runs][G], [runs][cap], [runs], [runs]
    int* pmask; int* ccount; int* cties;                                 // Choi clusters: [runs][cap], [runs][A], [runs]
    int* tour_off; int* tour_cur; long long* tour;                       // Choi tours: [runs*A+1], [runs*A], [tour_off[runs*A]]
    const long long* seed; unsigned short* cmask; double* ccell; int* rowidx;   // Thompson: [runs], [runs][G], [runs][A][2], [runs][cap]
};

bool batch_valid(const mfgp_batch* b, const mfgp_params* p_host);
BatchArgs batch_args(const mfgp_batch* b, const mfgp_params* p_host);

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// cross-covariance of training row n of run r with grid point (ix, iy), from the axis tables (batch_posterior_kernel)
__device__ __forceinline__ double bt_psi(const BatchArgs& a, int r, int n, int ix, int iy) {
    const int64_t t = (int64_t)r * a.cap + n;
    double psi = 0.0;
    if (n >= a.NL) psi = a.p.s_H * (a.TxH[t * a.nx + ix] * a.TyH[t * a.ny + iy]);
    if (a.p.multi) psi = fma(n < a.NL ? a.p.rho * a.p.s_L : a.p.rho2 * a.p.s_L, a.TxL[t * a.nx + ix] * a.TyL[t * a.ny + iy], psi);
    return psi;
}

}  // namespace mfgp
