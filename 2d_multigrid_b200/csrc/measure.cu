// measure.cu -- observables of a gauge ensemble on U(1) links U[s][2] (complex128, whole lattice L x L, s = x + y L).
//
//   mg2d_meson_contract  out[y][a][b] = G_ab(y) = sum_x tr[s_a S(x,y) s_b s3 S(x,y)^dag s3], S_{al,be} = psi_be(s)_al, from the
//                        two propagator columns psi_be = D^-1 e_{s0,be}; s0 = 1, s1..s3 the Pauli matrices (gamma_x, gamma_y,
//                        gamma5).  -G_ab is the connected correlator of the bilinears s_a, s_b (gamma5-hermiticity gives the
//                        backward propagator).  One CTA per row: the ten independent products M_pq = sum_x v_p conj(v_q),
//                        v = (S00, S01, S10, S11), are reduced in a fixed order and the basis is changed at the end.
//                        HBM: 64 B/site read (both columns), 256 B/row written -> bytes-bound.
//   mg2d_topo_charge     out[0] = sum_P arg U_P, arg in (-pi, pi], U_P oriented as in mg2d_plaquette (Q = out[0] / 2 pi).
//                        HBM: 32 B/site (neighbour links re-read from L1/L2) -> bytes-bound.
//   mg2d_wilson_loops    out[(T-1) r_max + R-1] = sum_s W_RT(s) (re, im), the anticlockwise R x T loop with base s.  With
//                        U(1) links the loop is h_R(x,y) conj(h_R(x,y+T)) prod_{j<T} c_R(x,y+j), h_R = the product of the
//                        R x-links from (x,y), c_R(x,y) = U_y(x+R,y) conj(U_y(x,y)) (one rung of the two y-sides).  A CTA
//                        takes one R (blockIdx.y) and a 32-column tile of bases; it builds h_R and c_R for the tile rows and
//                        the t_max halo rows in shared memory, and every thread marches T = 1..t_max from its base with one
//                        running product (2 complex products per (s, R, T)).  Reading the links is 32 B/site per R from
//                        L2/HBM; the r_max t_max complex products per site read from shared memory bound the kernel
//                        (compute- and shared-memory-bound, not bytes-bound).
//
// Every reduction is in a fixed order for a fixed launch shape (the sums of the last two finish in the last CTA), so results
// are bit-identical from run to run.  No float atomics.
#include <math_constants.h>
#include "common.cuh"

namespace {

using C = double2;

__device__ __forceinline__ int wrap_hi(int i, int n) { return i >= n ? i - n : i; }

inline int grid_for(mg2d_ctx* ctx, long long n) {
    long long nb = (n + 255) / 256;
    const long long cap = (long long)ctx->num_sms * 8;
    if (nb > cap) nb = cap;
    if (nb > MG2D_MAX_PARTIALS) nb = MG2D_MAX_PARTIALS;
    return nb < 1 ? 1 : (int)nb;
}

// ---- meson contraction ---------------------------------------------------------------------------------------------
// reduced slots: 0..3 = M_pp (real), then the upper triangle p < q as (re, im): (0,1) (0,2) (0,3) (1,2) (1,3) (2,3)
constexpr int MESON_NR = 16;
constexpr int MESON_THREADS = 256;

__device__ __forceinline__ void meson_accumulate(double (&m)[MESON_NR], C v0, C v1, C v2, C v3) {
    const C v[4] = {v0, v1, v2, v3};
#pragma unroll
    for (int p = 0; p < 4; ++p) m[p] = fma(v[p].x, v[p].x, fma(v[p].y, v[p].y, m[p]));
    int k = 4;
#pragma unroll
    for (int p = 0; p < 4; ++p) {
#pragma unroll
        for (int q = p + 1; q < 4; ++q) {
            // v_p conj(v_q)
            m[k] = fma(v[p].x, v[q].x, fma(v[p].y, v[q].y, m[k]));
            m[k + 1] = fma(v[p].y, v[q].x, fma(-v[p].x, v[q].y, m[k + 1]));
            k += 2;
        }
    }
}

// (sigma_a)_{ij}, a = 0..3
__device__ __forceinline__ C pauli(int a, int i, int j) {
    switch (a) {
        case 0: return make_double2(i == j ? 1.0 : 0.0, 0.0);
        case 1: return make_double2(i != j ? 1.0 : 0.0, 0.0);
        case 2: return make_double2(0.0, i == j ? 0.0 : (i == 0 ? -1.0 : 1.0));
        default: return make_double2(i == j ? (i == 0 ? 1.0 : -1.0) : 0.0, 0.0);
    }
}

__global__ void __launch_bounds__(MESON_THREADS)
meson_contract_kernel(const C* __restrict__ psi0, const C* __restrict__ psi1, int L, double* __restrict__ out) {
    __shared__ double s_red[MESON_NR][MESON_THREADS / 32];
    __shared__ double s_m[MESON_NR];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int y = blockIdx.x; y < L; y += gridDim.x) {
        double m[MESON_NR];
#pragma unroll
        for (int r = 0; r < MESON_NR; ++r) m[r] = 0.0;
        const C* r0 = psi0 + 2 * (size_t)y * L;
        const C* r1 = psi1 + 2 * (size_t)y * L;
        for (int x = threadIdx.x; x < L; x += MESON_THREADS) {
            C a0, a1, b0, b1;               // psi0(s) = (S00, S10), psi1(s) = (S01, S11)
            ld256(r0 + 2 * x, a0, a1);
            ld256(r1 + 2 * x, b0, b1);
            meson_accumulate(m, a0, b0, a1, b1);
        }
#pragma unroll
        for (int r = 0; r < MESON_NR; ++r) {
            double v = m[r];
#pragma unroll
            for (int k = 16; k > 0; k >>= 1) v += __shfl_xor_sync(0xffffffffu, v, k);
            if (lane == 0) s_red[r][warp] = v;
        }
        __syncthreads();
        if (threadIdx.x < MESON_NR) {
            double v = 0.0;
            for (int w = 0; w < MESON_THREADS / 32; ++w) v += s_red[threadIdx.x][w];
            s_m[threadIdx.x] = v;
        }
        __syncthreads();
        if (threadIdx.x < 16) {
            // G_ab = sum_{ijkl} (s_a)_{ij} s3_{ii} (s_b s3)_{kl} M[(j,k)][(i,l)],  M[p][q] = sum_x v_p conj(v_q), p = 2 row + col
            const int a = threadIdx.x >> 2, b = threadIdx.x & 3;
            C g = make_double2(0.0, 0.0);
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 2; ++j)
#pragma unroll
                    for (int k = 0; k < 2; ++k)
#pragma unroll
                        for (int l = 0; l < 2; ++l) {
                            const int p = 2 * j + k, q = 2 * i + l;
                            C mpq;
                            if (p == q) mpq = make_double2(s_m[p], 0.0);
                            else {
                                const int lo = p < q ? p : q, hi = p < q ? q : p;
                                const int slot = 4 + 2 * (lo == 0 ? hi - 1 : (lo == 1 ? hi + 1 : 5));
                                mpq = make_double2(s_m[slot], p < q ? s_m[slot + 1] : -s_m[slot + 1]);
                            }
                            C coef = cmul(pauli(a, i, j), pauli(b, k, l));
                            const double sgn = (i == 0 ? 1.0 : -1.0) * (l == 0 ? 1.0 : -1.0);   // s3_{ii} and the s3 of s_b s3
                            coef = cscale(coef, sgn);
                            g = cadd(g, cmul(coef, mpq));
                        }
            reinterpret_cast<C*>(out)[(size_t)y * 16 + threadIdx.x] = g;
        }
        __syncthreads();
    }
}

// ---- topological charge --------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
topo_charge_kernel(const C* __restrict__ U, int L, double* __restrict__ partials, unsigned int* __restrict__ counter,
                   double* __restrict__ out) {
    const long long S = (long long)L * L;
    double red[1] = {0.0};
    for (long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x; s < S; s += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(s / L), x = (int)(s - (long long)y * L);
        const long long sx = wrap_hi(x + 1, L) + (long long)y * L, sy = x + (long long)wrap_hi(y + 1, L) * L;
        const C ux = __ldg(U + 2 * s), uy = __ldg(U + 2 * s + 1), uy_x = __ldg(U + 2 * sx + 1), ux_y = __ldg(U + 2 * sy);
        // U_x(s) U_y(s+x) conj(U_x(s+y)) conj(U_y(s)), as plaquette_kernel (gauge.cu)
        const C p = cmulc(cmul(ux_y, uy), cmul(ux, uy_x));
        double a = atan2(p.y, p.x);
        if (a == -CUDART_PI) a = CUDART_PI;             // (-pi, pi]
        red[0] += a;
    }
    grid_reduce<1, 256>(red, partials, counter, out, blockIdx.x, gridDim.x);
}

// ---- Wilson loops --------------------------------------------------------------------------------------------------
constexpr int WL_TX = 32;              // base columns of a tile (one per lane)
constexpr int WL_TY = 32;              // base rows of a tile
constexpr int WL_THREADS = 256;        // 8 warps: warp w takes base rows w, w + 8, ...
constexpr int WL_MAX = 32;             // r_max, t_max <= WL_MAX

__global__ void __launch_bounds__(WL_THREADS)
wilson_loops_kernel(const C* __restrict__ U, int L, int r_max, int t_max, double* __restrict__ partials,
                    unsigned int* __restrict__ counter, double* __restrict__ out) {
    extern __shared__ C s_hc[];                              // h_R then c_R, (WL_TY + t_max) rows of WL_TX each
    __shared__ double s_red[2 * WL_MAX][WL_THREADS / 32];
    __shared__ bool s_last;
    const int R = blockIdx.y + 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ntx = (L + WL_TX - 1) / WL_TX, nty = (L + WL_TY - 1) / WL_TY;
    const int nrows = WL_TY + t_max;
    C (*s_h)[WL_TX] = reinterpret_cast<C (*)[WL_TX]>(s_hc);
    C (*s_c)[WL_TX] = reinterpret_cast<C (*)[WL_TX]>(s_hc + (size_t)nrows * WL_TX);
    C acc[WL_MAX];
#pragma unroll
    for (int t = 0; t < WL_MAX; ++t) acc[t] = make_double2(0.0, 0.0);

    for (int tile = blockIdx.x; tile < ntx * nty; tile += gridDim.x) {
        const int x0 = (tile % ntx) * WL_TX, y0 = (tile / ntx) * WL_TY;
        __syncthreads();                                      // the previous tile's readers are done with s_h / s_c
        for (int e = threadIdx.x; e < nrows * WL_TX; e += WL_THREADS) {
            const int r = e / WL_TX, cx = e - r * WL_TX;
            const int x = (x0 + cx) % L, y = (y0 + r) % L;       // a small lattice wraps more than once
            const C* row = U + 2 * (size_t)y * L;
            C h = __ldg(row + 2 * x);
            for (int i = 1; i < R; ++i) h = cmul(h, __ldg(row + 2 * wrap_hi(x + i, L)));
            s_h[r][cx] = h;
            s_c[r][cx] = cmulc(__ldg(row + 2 * x + 1), __ldg(row + 2 * wrap_hi(x + R, L) + 1));
        }
        __syncthreads();
        if (x0 + lane < L) {
            for (int r = warp; r < WL_TY && y0 + r < L; r += WL_THREADS / 32) {
                const C hb = s_h[r][lane];
                C P = make_double2(1.0, 0.0);
#pragma unroll
                for (int t = 0; t < WL_MAX; ++t) {
                    if (t < t_max) {
                        P = cmul(P, s_c[r + t][lane]);
                        acc[t] = cadd(acc[t], cmul(cmulc(s_h[r + t + 1][lane], hb), P));
                    }
                }
            }
        }
    }

    // per-CTA sums of acc[0..t_max) -> partials[(blockIdx.y gridDim.x + blockIdx.x)][2 t + (re, im)]
#pragma unroll
    for (int t = 0; t < WL_MAX; ++t) {
        if (t < t_max) {
            double re = acc[t].x, im = acc[t].y;
#pragma unroll
            for (int k = 16; k > 0; k >>= 1) {
                re += __shfl_xor_sync(0xffffffffu, re, k);
                im += __shfl_xor_sync(0xffffffffu, im, k);
            }
            if (lane == 0) { s_red[2 * t][warp] = re; s_red[2 * t + 1][warp] = im; }
        }
    }
    __syncthreads();
    const size_t cta = (size_t)blockIdx.y * gridDim.x + blockIdx.x;
    if (threadIdx.x < 2 * t_max) {
        double v = 0.0;
        for (int w = 0; w < WL_THREADS / 32; ++w) v += s_red[threadIdx.x][w];
        partials[cta * MG2D_MAX_RED + threadIdx.x] = v;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int t = atomicAdd(counter, 1u);
        s_last = (t == gridDim.x * gridDim.y - 1u);
    }
    __syncthreads();
    if (s_last) {
        __threadfence();
        // out[(T-1) r_max + (R-1)]: a fixed-order sum over the gridDim.x CTAs of that R
        for (int o = threadIdx.x; o < 2 * r_max * t_max; o += WL_THREADS) {
            const int c = o & 1, k = o >> 1, t = k / r_max, rr = k - t * r_max;
            double v = 0.0;
            for (int b = 0; b < (int)gridDim.x; ++b) v += __ldcg(&partials[((size_t)rr * gridDim.x + b) * MG2D_MAX_RED + 2 * t + c]);
            out[o] = v;
        }
        if (threadIdx.x == 0) *counter = 0u;
    }
}

}  // namespace

extern "C" int mg2d_meson_contract(mg2d_ctx* ctx, const void* psi0, const void* psi1, int L, double* out, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!psi0 || !psi1 || !out || L < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_meson_contract: bad argument");
    if (((uintptr_t)psi0 | (uintptr_t)psi1) & 31u)
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_meson_contract: the propagator columns must be 32-byte aligned");
    const int grid = L < MG2D_MAX_PARTIALS ? L : MG2D_MAX_PARTIALS;
    meson_contract_kernel<<<grid, MESON_THREADS, 0, (cudaStream_t)stream>>>((const C*)psi0, (const C*)psi1, L, out);
    return mg2d_check_launch(ctx, "mg2d_meson_contract");
}

extern "C" int mg2d_topo_charge(mg2d_ctx* ctx, const void* U, int L, double* out, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!U || !out || L < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_topo_charge: bad argument");
    topo_charge_kernel<<<grid_for(ctx, (long long)L * L), 256, 0, (cudaStream_t)stream>>>((const C*)U, L, ctx->partials,
                                                                                           ctx->counter, out);
    return mg2d_check_launch(ctx, "mg2d_topo_charge");
}

extern "C" int mg2d_wilson_loops(mg2d_ctx* ctx, const void* U, int L, int r_max, int t_max, double* out, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!U || !out || L < 2) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_wilson_loops: bad argument");
    if (r_max < 1 || t_max < 1 || r_max > WL_MAX || t_max > WL_MAX || r_max >= L || t_max >= L)
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_wilson_loops: need 1 <= r_max, t_max <= 32 and r_max, t_max < L");
    const long long tiles = (long long)((L + WL_TX - 1) / WL_TX) * ((L + WL_TY - 1) / WL_TY);
    long long gx = (long long)ctx->num_sms * 4 / r_max;          // about 4 waves over all R (167 registers: one CTA per SM)
    if (gx > MG2D_MAX_PARTIALS / r_max) gx = MG2D_MAX_PARTIALS / r_max;
    if (gx > tiles) gx = tiles;
    if (gx < 1) gx = 1;
    const size_t smem = (size_t)2 * (WL_TY + t_max) * WL_TX * sizeof(C);       // up to 64 KB
    if (cudaFuncSetAttribute(wilson_loops_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)(2 * (WL_TY + WL_MAX) * WL_TX * sizeof(C))) != cudaSuccess)
        return mg2d_check_launch(ctx, "mg2d_wilson_loops: shared-memory opt-in");
    wilson_loops_kernel<<<dim3((unsigned)gx, (unsigned)r_max), WL_THREADS, smem, (cudaStream_t)stream>>>(
        (const C*)U, L, r_max, t_max, ctx->partials, ctx->counter, out);
    return mg2d_check_launch(ctx, "mg2d_wilson_loops");
}
