// gauge.cu -- inputs of the hot path generated on the device: counter-based random fields and quenched U(1) links.
//
//   mg2d_fill_uniform      f_init_near_null_vector / f_init_vectors (S6/modules_indiv.h:16-68) for lattices too large
//                          for the reference's sequential std::mt19937 stream: a COUNTER-based generator keyed on
//                          (seed, stream, global element index), so that a strip of a domain-decomposed field holds
//                          exactly the numbers the single-GPU field holds at the same global sites
//   mg2d_fill_gaussian     normal deviates by Box-Muller on the same counter generator (HMC momenta and pseudofermion sources)
//   mg2d_gauge_metropolis  one checkerboard half-update of the compact-U(1) Wilson action (the reference only reads
//                          such configurations, S6/gauge.h:44,88-110, beta in {6, 32}); mirrored draw-for-draw by
//                          oracle gauge_quenched_phases_counter
//   mg2d_plaquette         Gauge::f_plaquette, S6/gauge.h:50-63
//   mg2d_clover_field      the real site field f(s) = (c_sw/8) sum_{P corner s} Im U_P of the clover self term (2+m) 1 + f s3
//   mg2d_phases_to_links   U = polar(1, theta), S6/gauge.h:106
#include "common.cuh"

namespace {

// splitmix64 finaliser over (seed, stream, index); 53 mantissa bits -> [0,1).  oracle/mg_oracle.py: counter_uniform
__device__ __forceinline__ double counter_u01(unsigned long long seed, unsigned long long stream, unsigned long long idx) {
    unsigned long long z = seed * 0x9E3779B97F4A7C15ull + stream * 0xD1B54A32D192ED03ull + (idx + 1ull) * 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z = z ^ (z >> 31);
    return (double)(z >> 11) * (1.0 / 9007199254740992.0);
}

template <typename T>
__global__ void fill_uniform_kernel(cplx<T>* __restrict__ out, long long n, unsigned long long offset, unsigned long long seed,
                                    unsigned long long stream, double lo, double hi) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const double u = counter_u01(seed, stream, offset + (unsigned long long)e);
        out[e] = mk<T>((T)__dadd_rn(lo, __dmul_rn(hi - lo, u)), (T)0);     // no FMA contraction: equals the numpy oracle bit for bit
    }
}

// out[e] = sd sqrt(-2 ln(1 - u1)) cos(2 pi u2), u1 / u2 = counter numbers at index 2(offset+e) / 2(offset+e)+1 (Box-Muller,
// cosine branch): one real N(0, sd^2) deviate per element, so a sub-range of the field is drawn independently.
// oracle mirror: tests/test_hmc.py counter_gaussian
__global__ void fill_gaussian_kernel(double* __restrict__ out, long long n, unsigned long long offset, unsigned long long seed,
                                     unsigned long long stream, double sd) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const unsigned long long k = 2ull * (offset + (unsigned long long)e);
        const double u1 = counter_u01(seed, stream, k), u2 = counter_u01(seed, stream, k + 1ull);
        out[e] = sd * sqrt(-2.0 * log(1.0 - u1)) * cospi(2.0 * u2);
    }
}

// theta[s][2], s = x + y*L.  Updates theta[s][mu] on the sites with (x + y) % 2 == parity.
__global__ void __launch_bounds__(256)
gauge_metropolis_kernel(double* __restrict__ theta, int L, double beta, double delta, int mu, int parity,
                        unsigned long long seed, unsigned long long tag) {
    const int Lh = L / 2;
    const long long n = (long long)Lh * L;
    const int nu = 1 - mu;
    for (long long h = blockIdx.x * (long long)blockDim.x + threadIdx.x; h < n; h += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(h / Lh);
        const int x = 2 * (int)(h - (long long)y * Lh) + ((y + parity) & 1);
        const int xp = (x + 1 == L) ? 0 : x + 1, xm = (x == 0) ? L - 1 : x - 1;
        const int yp = (y + 1 == L) ? 0 : y + 1, ym = (y == 0) ? L - 1 : y - 1;
        const long long s = x + (long long)y * L;
        // neighbours along mu and nu
        const long long s_pmu = (mu == 0) ? xp + (long long)y * L : x + (long long)yp * L;
        const long long s_pnu = (nu == 0) ? xp + (long long)y * L : x + (long long)yp * L;
        const long long s_mnu = (nu == 0) ? xm + (long long)y * L : x + (long long)ym * L;
        const long long s_mnu_pmu = (mu == 0) ? (xp + (long long)ym * L) : (xm + (long long)yp * L);
        const double old = theta[2 * s + mu];
        const double t_nu = theta[2 * s + nu], t_nu_pmu = theta[2 * s_pmu + nu], o_mu_pnu = theta[2 * s_pnu + mu];
        const double t_nu_mnu = theta[2 * s_mnu + nu], t_nu_mnu_pmu = theta[2 * s_mnu_pmu + nu], o_mu_mnu = theta[2 * s_mnu + mu];
        const double u1 = counter_u01(seed, 2ull * tag, (unsigned long long)s);
        const double u2 = counter_u01(seed, 2ull * tag + 1ull, (unsigned long long)s);
        const double trial = __dadd_rn(old, __dmul_rn(2.0 * u1 - 1.0, delta));   // no FMA contraction (oracle parity)
        // S(t) = -beta (cos(t + t_nu(x+mu) - mu(x+nu) - t_nu(x)) + cos(t_nu(x-nu) + t - t_nu(x-nu+mu) - mu(x-nu)))
        // (same association order as the oracle, so both see identical arguments)
        const double s_new = -beta * (cos(trial + t_nu_pmu - o_mu_pnu - t_nu) + cos(t_nu_mnu + trial - t_nu_mnu_pmu - o_mu_mnu));
        const double s_old = -beta * (cos(old + t_nu_pmu - o_mu_pnu - t_nu) + cos(t_nu_mnu + old - t_nu_mnu_pmu - o_mu_mnu));
        if (u2 < exp(-(s_new - s_old))) theta[2 * s + mu] = trial;
    }
}

template <typename T>
__global__ void __launch_bounds__(256)
plaquette_kernel(const cplx<T>* __restrict__ U, int L, double* __restrict__ partials, unsigned int* __restrict__ counter,
                 double* __restrict__ out) {
    using C = cplx<T>;
    const long long S = (long long)L * L;
    double red[2] = {0.0, 0.0};
    for (long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x; s < S; s += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(s / L), x = (int)(s - (long long)y * L);
        const long long sx = ((x + 1 == L) ? 0 : x + 1) + (long long)y * L, sy = x + (long long)((y + 1 == L) ? 0 : y + 1) * L;
        const C ux = __ldg(U + 2 * s), uy = __ldg(U + 2 * s + 1), uy_x = __ldg(U + 2 * sx + 1), ux_y = __ldg(U + 2 * sy);
        // U_x(s) U_y(s+x) conj(U_x(s+y)) conj(U_y(s))   (S6/gauge.h:58-61)
        const C a = cmul(ux, uy_x), b = cmul(ux_y, uy);
        const C p = cmulc(b, a);
        red[0] += (double)p.x; red[1] += (double)p.y;
    }
    grid_reduce<2, 256>(red, partials, counter, out, blockIdx.x, gridDim.x);
}

// Im of the anticlockwise plaquette with base (x, y), y in [-1, Ly-1]: link rows -1 and Ly come from U_lo / U_hi
template <typename T>
__device__ __forceinline__ T im_plaquette(const cplx<T>* __restrict__ U, const cplx<T>* __restrict__ U_lo,
                                          const cplx<T>* __restrict__ U_hi, int x, int y, int Lx, int Ly) {
    using C = cplx<T>;
    const int xp = (x + 1 == Lx) ? 0 : x + 1;
    const C* r0 = (y < 0) ? U_lo : U + 2 * (size_t)y * Lx;                         // links of row y
    const C* r1 = (y + 1 == Ly) ? U_hi : U + 2 * (size_t)(y + 1) * Lx;             // links of row y+1
    const C ux = __ldg(r0 + 2 * x), uy = __ldg(r0 + 2 * x + 1), uy_x = __ldg(r0 + 2 * xp + 1), ux_y = __ldg(r1 + 2 * x);
    // U_x(b) U_y(b+x) conj(U_x(b+y)) conj(U_y(b)), as in plaquette_kernel
    const C a = cmul(ux, uy_x), b = cmul(ux_y, uy);
    return cmulc(b, a).y;
}

// F[s] = (c_sw/8) (P(s) + P(s-x) + P(s-y) + P(s-x-y)), P(b) = Im U_P(b): the four plaquettes with a corner at s.  The same
// operations in the same order at every site, so a strip gives its rows of the whole-lattice field bit for bit.
template <typename T>
__global__ void clover_field_kernel(T* __restrict__ F, const cplx<T>* __restrict__ U, const cplx<T>* __restrict__ U_lo,
                                    const cplx<T>* __restrict__ U_hi, T c8, int Lx, int Ly) {
    const long long S = (long long)Lx * Ly;
    for (long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x; s < S; s += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(s / Lx), x = (int)(s - (long long)y * Lx);
        const int xm = (x == 0) ? Lx - 1 : x - 1;
        const T p = im_plaquette<T>(U, U_lo, U_hi, x, y, Lx, Ly) + im_plaquette<T>(U, U_lo, U_hi, xm, y, Lx, Ly)
                  + im_plaquette<T>(U, U_lo, U_hi, x, y - 1, Lx, Ly) + im_plaquette<T>(U, U_lo, U_hi, xm, y - 1, Lx, Ly);
        F[s] = c8 * p;
    }
}

template <typename T>
__global__ void phases_to_links_kernel(cplx<T>* __restrict__ U, const double* __restrict__ theta, long long n) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        double sn, cs;
        sincos(theta[e], &sn, &cs);
        U[e] = mk<T>((T)cs, (T)sn);
    }
}

inline int grid_for(mg2d_ctx* ctx, long long n) {
    long long nb = (n + 255) / 256;
    const long long cap = (long long)ctx->num_sms * 8;
    if (nb > cap) nb = cap;
    if (nb > MG2D_MAX_PARTIALS) nb = MG2D_MAX_PARTIALS;
    return nb < 1 ? 1 : (int)nb;
}

}  // namespace

extern "C" int mg2d_fill_uniform(mg2d_ctx* ctx, void* out, long long nelem, long long offset, unsigned long long seed,
                                 unsigned long long stream_id, double lo, double hi, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!out || nelem < 1 || offset < 0) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_fill_uniform: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = grid_for(ctx, nelem);
    if (dtype == MG2D_C128) fill_uniform_kernel<double><<<grid, 256, 0, st>>>((double2*)out, nelem, (unsigned long long)offset, seed, stream_id, lo, hi);
    else if (dtype == MG2D_C64) fill_uniform_kernel<float><<<grid, 256, 0, st>>>((float2*)out, nelem, (unsigned long long)offset, seed, stream_id, lo, hi);
    else return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_fill_uniform: bad dtype");
    return mg2d_check_launch(ctx, "mg2d_fill_uniform");
}

extern "C" int mg2d_fill_gaussian(mg2d_ctx* ctx, double* out, long long nelem, long long offset, unsigned long long seed,
                                  unsigned long long stream_id, double variance, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!out || nelem < 1 || offset < 0 || !(variance >= 0.0)) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_fill_gaussian: bad argument");
    fill_gaussian_kernel<<<grid_for(ctx, nelem), 256, 0, (cudaStream_t)stream>>>(out, nelem, (unsigned long long)offset, seed,
                                                                                  stream_id, sqrt(variance));
    return mg2d_check_launch(ctx, "mg2d_fill_gaussian");
}

extern "C" int mg2d_gauge_metropolis(mg2d_ctx* ctx, double* theta, int L, double beta, double delta, int mu, int parity,
                                     unsigned long long seed, unsigned long long tag, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!theta || L < 2 || (L & 1) || (mu != 0 && mu != 1) || (parity != 0 && parity != 1))
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_gauge_metropolis: bad argument (L must be even)");
    gauge_metropolis_kernel<<<grid_for(ctx, (long long)L * L / 2), 256, 0, (cudaStream_t)stream>>>(theta, L, beta, delta, mu, parity, seed, tag);
    return mg2d_check_launch(ctx, "mg2d_gauge_metropolis");
}

extern "C" int mg2d_plaquette(mg2d_ctx* ctx, const void* U, int L, int dtype, double* out, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!U || !out || L < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_plaquette: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = grid_for(ctx, (long long)L * L);
    if (dtype == MG2D_C128) plaquette_kernel<double><<<grid, 256, 0, st>>>((const double2*)U, L, ctx->partials, ctx->counter, out);
    else if (dtype == MG2D_C64) plaquette_kernel<float><<<grid, 256, 0, st>>>((const float2*)U, L, ctx->partials, ctx->counter, out);
    else return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_plaquette: bad dtype");
    return mg2d_check_launch(ctx, "mg2d_plaquette");
}

extern "C" int mg2d_clover_field(mg2d_ctx* ctx, void* F, const void* U, const void* U_lo, const void* U_hi, double csw, int Lx,
                                 int Ly, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!F || !U || !U_lo || !U_hi || Lx < 1 || Ly < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_clover_field: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = grid_for(ctx, (long long)Lx * Ly);
    const double c8 = csw / 8.0;
    if (dtype == MG2D_C128) clover_field_kernel<double><<<grid, 256, 0, st>>>((double*)F, (const double2*)U, (const double2*)U_lo, (const double2*)U_hi, c8, Lx, Ly);
    else if (dtype == MG2D_C64) clover_field_kernel<float><<<grid, 256, 0, st>>>((float*)F, (const float2*)U, (const float2*)U_lo, (const float2*)U_hi, (float)c8, Lx, Ly);
    else return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_clover_field: bad dtype");
    return mg2d_check_launch(ctx, "mg2d_clover_field");
}

extern "C" int mg2d_phases_to_links(mg2d_ctx* ctx, void* U, const double* theta, long long nelem, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!U || !theta || nelem < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_phases_to_links: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = grid_for(ctx, nelem);
    if (dtype == MG2D_C128) phases_to_links_kernel<double><<<grid, 256, 0, st>>>((double2*)U, theta, nelem);
    else if (dtype == MG2D_C64) phases_to_links_kernel<float><<<grid, 256, 0, st>>>((float2*)U, theta, nelem);
    else return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_phases_to_links: bad dtype");
    return mg2d_check_launch(ctx, "mg2d_phases_to_links");
}
