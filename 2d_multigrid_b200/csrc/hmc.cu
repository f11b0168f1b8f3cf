// hmc.cu -- the molecular-dynamics updates of two-flavour Wilson Hybrid Monte Carlo on U(1) links theta[s][2], U = e^{i theta}.
//
//   mg2d_hmc_momentum  P_mu(s) -= eps (F^g_mu(s) + F^f_mu(s)), both directions in one pass:
//     gauge force of S_g = beta sum_P (1 - cos theta_P), sin theta_P = Im U_P (the plaquette of mg2d_plaquette):
//       F^g_x(s) = beta [sin theta_P(s) - sin theta_P(s-y)],   F^g_y(s) = beta [sin theta_P(s-x) - sin theta_P(s)]
//     fermion force of S_f = phi^dag (D^dag D)^-1 phi with X = (D^dag D)^-1 phi, Y = D X, and the hopping terms of wilson.cu
//     (D(s, s+mu) = U_mu(s) 1/2(1-s_mu), D(s+mu, s) = conj(U_mu(s)) 1/2(1+s_mu)):
//       F^f_mu(s) = dS_f/dtheta_mu(s) = -2 Re[Y^dag dD/dtheta_mu(s) X]
//                 = Im[U_mu(s) conj(h-_mu Y(s)) h-_mu X(s+mu)] - Im[conj(U_mu(s)) conj(h+_mu Y(s+mu)) h+_mu X(s)]
//     with the half-spinor projections of wilson.cu, v^dag 1/2(1 -+ s_mu) w = 1/2 conj(h-+ v) h-+ w:
//       h-_x v = v0 - v1,  h+_x v = v0 + v1,  h-_y v = v0 + i v1,  h+_y v = v0 - i v1
//     X = Y = NULL: gauge force only (pure-gauge HMC).
//   mg2d_hmc_links     theta += eps P; U = e^{i theta} (complex128) and optionally its complex64 copy, in place
//   mg2d_gamma5        out = gamma5 in = sigma3 in (the pseudofermion algebra of D^dag = gamma5 D gamma5)
//
// HBM roofline (complex128 fields and links, fp64 momenta): the momentum update moves P in + out (32 B/site), U (32), X and Y
// (32 + 32) = 128 B/site (64 without fermions); the link update theta in + out (32), P (16), U out (32) [+ 16 complex64] =
// 80 [96] B/site.  Neighbour rows are re-read from L1/L2, not HBM.  Grid-stride loops over sites.
#include "common.cuh"

namespace {

using C = double2;

__device__ __forceinline__ int wrap(int i, int n) { return i < 0 ? i + n : (i >= n ? i - n : i); }

// Im of the anticlockwise plaquette with base (x, y): U_x(b) U_y(b+x) conj(U_x(b+y)) conj(U_y(b)), as mg2d_plaquette
__device__ __forceinline__ double im_plaq(const C* __restrict__ U, int x, int y, int L) {
    const size_t b = (size_t)y * L + x, bx = (size_t)y * L + wrap(x + 1, L), by = (size_t)wrap(y + 1, L) * L + x;
    const C a = cmul(__ldg(U + 2 * b), __ldg(U + 2 * bx + 1)), c = cmul(__ldg(U + 2 * by), __ldg(U + 2 * b + 1));
    return cmulc(c, a).y;
}

__device__ __forceinline__ C hx_m(C v0, C v1) { return make_double2(v0.x - v1.x, v0.y - v1.y); }
__device__ __forceinline__ C hx_p(C v0, C v1) { return make_double2(v0.x + v1.x, v0.y + v1.y); }
__device__ __forceinline__ C hy_m(C v0, C v1) { return make_double2(v0.x - v1.y, v0.y + v1.x); }   // v0 + i v1
__device__ __forceinline__ C hy_p(C v0, C v1) { return make_double2(v0.x + v1.y, v0.y - v1.x); }   // v0 - i v1

// Im[u conj(a) b]
__device__ __forceinline__ double im_ucab(C u, C a, C b) { return cmul(u, cmulc(a, b)).y; }

__global__ void __launch_bounds__(256)
hmc_momentum_kernel(double* __restrict__ P, const C* __restrict__ U, const C* __restrict__ X, const C* __restrict__ Y,
                    double beta, double eps, int L) {
    const long long S = (long long)L * L;
    for (long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x; s < S; s += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(s / L), x = (int)(s - (long long)y * L);
        const double p0 = im_plaq(U, x, y, L);
        double fx = beta * (p0 - im_plaq(U, x, wrap(y - 1, L), L));
        double fy = beta * (im_plaq(U, wrap(x - 1, L), y, L) - p0);
        if (X != nullptr) {
            const long long sx = (long long)y * L + wrap(x + 1, L), sy = (long long)wrap(y + 1, L) * L + x;
            const C x0 = __ldg(X + 2 * s), x1 = __ldg(X + 2 * s + 1), y0 = __ldg(Y + 2 * s), y1 = __ldg(Y + 2 * s + 1);
            const C xx0 = __ldg(X + 2 * sx), xx1 = __ldg(X + 2 * sx + 1), yx0 = __ldg(Y + 2 * sx), yx1 = __ldg(Y + 2 * sx + 1);
            const C xy0 = __ldg(X + 2 * sy), xy1 = __ldg(X + 2 * sy + 1), yy0 = __ldg(Y + 2 * sy), yy1 = __ldg(Y + 2 * sy + 1);
            const C ux = __ldg(U + 2 * s), uy = __ldg(U + 2 * s + 1);
            fx += im_ucab(ux, hx_m(y0, y1), hx_m(xx0, xx1)) - im_ucab(cconj(ux), hx_p(yx0, yx1), hx_p(x0, x1));
            fy += im_ucab(uy, hy_m(y0, y1), hy_m(xy0, xy1)) - im_ucab(cconj(uy), hy_p(yy0, yy1), hy_p(x0, x1));
        }
        const double2 p = reinterpret_cast<const double2*>(P)[s];
        reinterpret_cast<double2*>(P)[s] = make_double2(p.x - eps * fx, p.y - eps * fy);
    }
}

// theta += eps P (no FMA contraction: equals the fp64 torch restatement bit for bit); U = polar(1, theta) as mg2d_phases_to_links
__global__ void __launch_bounds__(256)
hmc_links_kernel(double* __restrict__ theta, const double* __restrict__ P, double eps, C* __restrict__ U, float2* __restrict__ U32,
                 long long n) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const double t = __dadd_rn(theta[e], __dmul_rn(eps, P[e]));
        theta[e] = t;
        double sn, cs;
        sincos(t, &sn, &cs);
        U[e] = make_double2(cs, sn);
        if (U32 != nullptr) U32[e] = make_float2((float)cs, (float)sn);
    }
}

__global__ void gamma5_kernel(C* __restrict__ out, const C* __restrict__ in, long long S) {
    for (long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x; s < S; s += (long long)gridDim.x * blockDim.x) {
        const C v1 = in[2 * s + 1];
        out[2 * s] = in[2 * s];
        out[2 * s + 1] = make_double2(-v1.x, -v1.y);
    }
}

inline int grid_for(mg2d_ctx* ctx, long long n) {
    long long nb = (n + 255) / 256;
    const long long cap = (long long)ctx->num_sms * 8;
    if (nb > cap) nb = cap;
    return nb < 1 ? 1 : (int)nb;
}

}  // namespace

extern "C" int mg2d_hmc_momentum(mg2d_ctx* ctx, double* P, const void* U, const void* X, const void* Y, double beta, double eps,
                                 int L, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!P || !U || L < 2 || (X == nullptr) != (Y == nullptr))
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_hmc_momentum: bad argument (X and Y are both set or both NULL)");
    hmc_momentum_kernel<<<grid_for(ctx, (long long)L * L), 256, 0, (cudaStream_t)stream>>>(P, (const C*)U, (const C*)X, (const C*)Y,
                                                                                           beta, eps, L);
    return mg2d_check_launch(ctx, "mg2d_hmc_momentum");
}

extern "C" int mg2d_hmc_links(mg2d_ctx* ctx, double* theta, const double* P, double eps, void* U, void* U32, long long nelem,
                              void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!theta || !P || !U || nelem < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_hmc_links: bad argument");
    hmc_links_kernel<<<grid_for(ctx, nelem), 256, 0, (cudaStream_t)stream>>>(theta, P, eps, (C*)U, (float2*)U32, nelem);
    return mg2d_check_launch(ctx, "mg2d_hmc_links");
}

extern "C" int mg2d_gamma5(mg2d_ctx* ctx, void* out, const void* in, long long nsites, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!out || !in || nsites < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_gamma5: bad argument");
    gamma5_kernel<<<grid_for(ctx, nsites), 256, 0, (cudaStream_t)stream>>>((C*)out, (const C*)in, nsites);
    return mg2d_check_launch(ctx, "mg2d_gamma5");
}
