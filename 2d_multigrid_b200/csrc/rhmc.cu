// rhmc.cu -- the vector updates of the multi-shift CG (Jegerlehner, hep-lat/9612014) for (M + sigma_k) x_k = phi, M = D^dag D,
// all shifts at once, on complex128 two-component level-0 fields (the solver of one-flavour RHMC).
//
// The base system is A = M + sigma_0 with the smallest shift; shift k runs on A + s_k, s_k = sigma_k - sigma_0 >= 0, with the
// base residual times zeta_k.  One iteration, with the host driving the operator through the existing entry points
// (t = D p_0 with the fused |t|^2 = <p_0, M p_0>, u = gamma5 t, w = D u, so M p_0 = gamma5 w):
//   mg2d_msc_pass_a  alpha = |r|^2 / (|t|^2 + sigma_0 |p_0|^2) (every CTA, from the device scalars);
//                    r -= alpha (gamma5 w + sigma_0 p_0), |r|^2 reduced in the kernel; the last CTA then runs the scalar
//                    recurrences in fp64 (beta, zeta_k, a_k = alpha zeta_k' / zeta_k, b_k = beta (zeta_k' / zeta_k)^2), records
//                    (alpha, beta) for the Lanczos tridiagonal and the number of shifts that stay active.
//   mg2d_msc_pass_b  for the active shifts k < n_active: x_k += a_k p_k, p_k = zeta_k r + b_k p_k; accumulate mode (X == NULL)
//                    keeps one y instead of the x_k: y += sum_k w_k a_k p_k.  |p_0|^2 is reduced in the kernel when sigma_0 != 0.
// Shift dropping: a shift whose residual |zeta_k| |r| is below the threshold stops being updated.  The shifts are sorted
// ascending, so |zeta_k| decreases with k and the active set is the range [0, n_active): n_active = 1 + the last k above it.
//
// HBM roofline (complex128, 32 B per site and vector): pass A reads r, w [, p_0] and writes r: 96 B/site (128 with sigma_0 != 0);
// pass B reads r once and each active x_k, p_k once and writes them once: 32 + 128 N_active B/site; accumulate mode
// 32 + 64 (y) + 64 N_active B/site.  Shift vectors are laid out [N][S][2].  Grid-stride loops over sites.
#include "common.cuh"

namespace {

using C = double2;
constexpr int MS_THREADS = 256;

inline int ms_grid(mg2d_ctx* ctx, long long n) {
    long long nb = (n + MS_THREADS - 1) / MS_THREADS;
    const long long cap = (long long)ctx->num_sms * 8;
    if (nb > cap) nb = cap;
    if (nb > MG2D_MAX_PARTIALS) nb = MG2D_MAX_PARTIALS;
    return nb < 1 ? 1 : (int)nb;
}

// Sum of one double over the grid in a fixed order (as grid_reduce); returns true in the last CTA to finish, where *total holds
// the sum for all its threads.
__device__ __forceinline__ bool grid_sum_last(double v, double* __restrict__ partials, unsigned int* __restrict__ counter,
                                              double* total) {
    __shared__ double s_red[MS_THREADS / 32];
    __shared__ double s_tot;
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
    if (lane == 0) s_red[warp] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double x = 0.0;
        for (int w = 0; w < MS_THREADS / 32; ++w) x += s_red[w];
        partials[blockIdx.x] = x;
        __threadfence();
        s_last = (atomicAdd(counter, 1u) == gridDim.x - 1u);
    }
    __syncthreads();
    if (!s_last) return false;
    __threadfence();
    if (warp == 0) {
        double x = 0.0;
        for (int c = lane; c < (int)gridDim.x; c += 32) x += __ldcg(&partials[c]);
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) x += __shfl_xor_sync(0xffffffffu, x, m);
        if (lane == 0) { s_tot = x; *counter = 0u; }
    }
    __syncthreads();
    *total = s_tot;
    return true;
}

__device__ __forceinline__ double alpha_of(const double* __restrict__ sc, const double* __restrict__ dots, double sigma0) {
    return sc[MG2D_MSC_RR] / (dots[MG2D_DOT_OUT2] + sigma0 * sc[MG2D_MSC_PP]);
}

template <bool SIG>
__global__ void __launch_bounds__(MS_THREADS)
msc_pass_a_kernel(C* __restrict__ r, const C* __restrict__ w, const C* __restrict__ p0, const double* __restrict__ dots,
                  double* __restrict__ sc, double sigma0, int nshift, long long S, double* __restrict__ partials,
                  unsigned int* __restrict__ counter) {
    const double alpha = alpha_of(sc, dots, sigma0);
    double rr = 0.0;
    for (long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x; s < S; s += (long long)gridDim.x * blockDim.x) {
        C r0 = r[2 * s], r1 = r[2 * s + 1];
        C w0 = __ldg(w + 2 * s), w1 = __ldg(w + 2 * s + 1);
        w1 = make_double2(-w1.x, -w1.y);                                        // gamma5 w
        if (SIG) {
            const C q0 = __ldg(p0 + 2 * s), q1 = __ldg(p0 + 2 * s + 1);
            w0 = make_double2(fma(sigma0, q0.x, w0.x), fma(sigma0, q0.y, w0.y));
            w1 = make_double2(fma(sigma0, q1.x, w1.x), fma(sigma0, q1.y, w1.y));
        }
        r0 = make_double2(fma(-alpha, w0.x, r0.x), fma(-alpha, w0.y, r0.y));
        r1 = make_double2(fma(-alpha, w1.x, r1.x), fma(-alpha, w1.y, r1.y));
        r[2 * s] = r0;
        r[2 * s + 1] = r1;
        rr += r0.x * r0.x + r0.y * r0.y + r1.x * r1.x + r1.y * r1.y;
    }
    double rr_new;
    if (!grid_sum_last(rr, partials, counter, &rr_new)) return;
    if (threadIdx.x != 0) return;
    // the scalar recurrences of the iteration, in fp64, by one thread
    const double beta = rr_new / sc[MG2D_MSC_RR];
    const double alpha_prev = sc[MG2D_MSC_ALPHA_PREV], beta_prev = sc[MG2D_MSC_BETA_PREV];
    const int it = (int)sc[MG2D_MSC_ITER];
    double* sig = sc + MG2D_MSC_SHIFTS;
    double* zeta = sig + nshift;
    double* zeta_prev = zeta + nshift;
    double* a = zeta_prev + nshift;
    double* b = a + nshift;
    const int nact = (int)sc[MG2D_MSC_NACT_NEXT];
    int nact_next = 0;
    for (int k = 0; k < nact; ++k) {
        const double z = zeta[k], zp = zeta_prev[k];
        const double zn = z * zp * alpha_prev / (alpha * beta_prev * (zp - z) + zp * alpha_prev * (1.0 + sig[k] * alpha));
        const double q = zn / z;
        a[k] = alpha * q;
        b[k] = beta * q * q;
        zeta_prev[k] = z;
        zeta[k] = zn;
        if (zn * zn * rr_new > sc[MG2D_MSC_THRESH]) nact_next = k + 1;
    }
    double* hist = b + 2 * nshift;                                               // after the weights w[N]
    hist[2 * it] = alpha;
    hist[2 * it + 1] = beta;
    sc[MG2D_MSC_RR] = rr_new;
    sc[MG2D_MSC_ALPHA_PREV] = alpha;
    sc[MG2D_MSC_BETA_PREV] = beta;
    sc[MG2D_MSC_NACT] = nact;
    sc[MG2D_MSC_NACT_NEXT] = nact_next;
    sc[MG2D_MSC_ITER] = it + 1;
}

// x_k += a_k p_k ; p_k = zeta_k r + b_k p_k  (ACC: y += sum_k w_k a_k p_k instead of the x_k update)
template <bool ACC, bool SIG>
__global__ void __launch_bounds__(MS_THREADS)
msc_pass_b_kernel(C* __restrict__ X, C* __restrict__ Pk, C* __restrict__ y, const C* __restrict__ r, double* __restrict__ sc,
                  int nshift, long long S, double* __restrict__ partials, unsigned int* __restrict__ counter) {
    const int nact = (int)sc[MG2D_MSC_NACT];
    const double* zeta = sc + MG2D_MSC_SHIFTS + nshift;
    const double* a = zeta + 2 * nshift;
    const double* b = a + nshift;
    const double* wt = b + nshift;
    double pp = 0.0;
    const long long vs = 2 * S;
    for (long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x; s < S; s += (long long)gridDim.x * blockDim.x) {
        const C r0 = __ldg(r + 2 * s), r1 = __ldg(r + 2 * s + 1);
        C y0 = make_double2(0.0, 0.0), y1 = y0;
#pragma unroll 4
        for (int k = 0; k < nact; ++k) {
            C* pk = Pk + k * vs + 2 * s;
            const C q0 = pk[0], q1 = pk[1];
            const double ak = a[k], bk = b[k], zk = zeta[k];
            if (ACC) {
                const double c = wt[k] * ak;
                y0 = make_double2(fma(c, q0.x, y0.x), fma(c, q0.y, y0.y));
                y1 = make_double2(fma(c, q1.x, y1.x), fma(c, q1.y, y1.y));
            } else {
                C* xk = X + k * vs + 2 * s;
                const C x0 = xk[0], x1 = xk[1];
                xk[0] = make_double2(fma(ak, q0.x, x0.x), fma(ak, q0.y, x0.y));
                xk[1] = make_double2(fma(ak, q1.x, x1.x), fma(ak, q1.y, x1.y));
            }
            const C n0 = make_double2(fma(zk, r0.x, bk * q0.x), fma(zk, r0.y, bk * q0.y));
            const C n1 = make_double2(fma(zk, r1.x, bk * q1.x), fma(zk, r1.y, bk * q1.y));
            pk[0] = n0;
            pk[1] = n1;
            if (SIG && k == 0) pp += n0.x * n0.x + n0.y * n0.y + n1.x * n1.x + n1.y * n1.y;
        }
        if (ACC && nact > 0) {
            const C v0 = y[2 * s], v1 = y[2 * s + 1];
            y[2 * s] = make_double2(v0.x + y0.x, v0.y + y0.y);
            y[2 * s + 1] = make_double2(v1.x + y1.x, v1.y + y1.y);
        }
    }
    if (SIG) {
        double v[1] = {pp};
        grid_reduce<1, MS_THREADS>(v, partials, counter, sc + MG2D_MSC_PP, blockIdx.x, gridDim.x);
    }
}

}  // namespace

extern "C" int mg2d_msc_pass_a(mg2d_ctx* ctx, void* r, const void* w, const void* p0, const double* dots, double* sc,
                               double sigma0, int nshift, long long nsites, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!r || !w || !dots || !sc || nsites < 1 || nshift < 1 || nshift > MG2D_MSC_MAX_SHIFTS || !(sigma0 >= 0.0) ||
        (sigma0 != 0.0 && !p0))
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_msc_pass_a: bad argument");
    const int grid = ms_grid(ctx, nsites);
    cudaStream_t st = (cudaStream_t)stream;
    if (sigma0 != 0.0)
        msc_pass_a_kernel<true><<<grid, MS_THREADS, 0, st>>>((C*)r, (const C*)w, (const C*)p0, dots, sc, sigma0, nshift, nsites,
                                                            ctx->partials, ctx->counter);
    else
        msc_pass_a_kernel<false><<<grid, MS_THREADS, 0, st>>>((C*)r, (const C*)w, nullptr, dots, sc, 0.0, nshift, nsites,
                                                             ctx->partials, ctx->counter);
    return mg2d_check_launch(ctx, "mg2d_msc_pass_a");
}

extern "C" int mg2d_msc_pass_b(mg2d_ctx* ctx, void* X, void* P, void* y, const void* r, double* sc, double sigma0, int nshift,
                               long long nsites, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!P || !r || !sc || nsites < 1 || nshift < 1 || nshift > MG2D_MSC_MAX_SHIFTS || (X == nullptr) == (y == nullptr) ||
        !(sigma0 >= 0.0))
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_msc_pass_b: bad argument (exactly one of X and y is set)");
    const int grid = ms_grid(ctx, nsites);
    cudaStream_t st = (cudaStream_t)stream;
#define MSB(ACC, SIG) msc_pass_b_kernel<ACC, SIG><<<grid, MS_THREADS, 0, st>>>((C*)X, (C*)P, (C*)y, (const C*)r, sc, nshift, nsites, \
                                                                               ctx->partials, ctx->counter)
    if (y) { if (sigma0 != 0.0) MSB(true, true); else MSB(true, false); }
    else   { if (sigma0 != 0.0) MSB(false, true); else MSB(false, false); }
#undef MSB
    return mg2d_check_launch(ctx, "mg2d_msc_pass_b");
}
