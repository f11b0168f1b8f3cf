// wilson.cu -- matrix-free U(1) Wilson-Dirac stencil on the fine lattice (n = 2 spin components).
//
// Replaces Level::f_compute_lvl0_matrix (wilson branch, S6/level.h:155-172) fused into Level::f_apply_D
// (S6/level.h:251-265), f_residue (:61-77) and the two norms of f_get_residue_mag (:79-98):
//
//   (D psi)(s) = (2+m) psi(s) + U_x(s) 1/2(1-s1) psi(s+x) + conj(U_x(s-x)) 1/2(1+s1) psi(s-x)
//                             + U_y(s) 1/2(1-s2) psi(s+y) + conj(U_y(s-y)) 1/2(1+s2) psi(s-y)
//   1/2(1-s1)psi = 1/2 (a,-a),  a = psi0-psi1      1/2(1+s1)psi = 1/2 (b, b),  b = psi0+psi1
//   1/2(1-s2)psi = 1/2 (c,-ic), c = psi0+i psi1    1/2(1+s2)psi = 1/2 (d, id), d = psi0-i psi1
//
// Clover (Sheikholeslami-Wohlert) variant, template flag SW: the self term becomes (2+m) 1 + f(s) s3 with the real site field
// f of mg2d_clover_field (csrc/gauge.cu), i.e. (2+m+f) on component 0 and (2+m-f) on component 1.
//
// Twisted-mass variant, template flag TM (with or without SW): + i mu gamma5 = i mu s3 on the self term, i.e. (2+m+f+i mu) on
// component 0 and (2+m-f-i mu) on component 1.  mu is one constant per launch, so the bytes are those of the Wilson / SW kernel.
//
// HBM roofline: algorithmic traffic 96 B/site in complex128 (psi in 32 + links 32 + out 32), +32 with b; SW adds f: 104 B/site
// (c64: 48 -> 52).
//
// Kernel design (v1, "column march"): a CTA owns a strip of WX consecutive x and marches over RY rows in y.
// Each thread keeps the three rows psi(x,y-1), psi(x,y), psi(x,y+1) and U_y(x,y-1) in registers, so every
// psi/U element is loaded from global memory exactly once per CTA (plus the two halo rows of the march and
// two halo columns); x-neighbour data is exchanged as projected half-spinors (one complex each way) through
// warp shuffles, with the warp-edge lanes falling back to a global load.
#include <cmath>
#include "common.cuh"
#include "spinor.cuh"

namespace {

constexpr int WX = 128;       // threads per CTA = x-extent of a CTA column strip
constexpr int RY_MAX = 32;    // rows marched per work item (fewer on small lattices, to keep every SM busy)

// "<entry point>: <what>" (the Wilson and clover entry points share their argument checks)
inline int mg2d_fail2(mg2d_ctx* ctx, const char* name, const char* what) {
    snprintf(ctx->err, sizeof(ctx->err), "%s: %s", name, what);
    return MG2D_EINVAL;
}

// MODE 0: out = D in ; MODE 1: out = b - D in.  DOTS: also reduce |out|^2, <out,in>, |b|^2.  SW: clover self term from F.
// TM: twisted-mass self term i mu s3.
// (the clover and twisted variants with DOTS ask for 5 CTAs per SM: left to its own heuristic ptxas spills the loop bound of
// the complex128 residual-norm variant.  The twisted variants without DOTS ask for the occupancy the Wilson kernel reaches,
// 7 CTAs per SM in complex128 (72 registers) and 10 in complex64 (48): left alone, ptxas gives the complex128 twisted apply
// 78 registers, 6 CTAs per SM, and it runs 24% slower than the Wilson apply.  The Wilson instantiations keep the plain bound
// and their code)
template <typename T, int MODE, bool DOTS, bool SW, bool TM>
__global__ void __launch_bounds__(WX, ((SW || TM) && DOTS) ? 5 : (TM ? (sizeof(T) == 8 ? 7 : 10) : 0))
wilson_march_kernel(cplx<T>* __restrict__ out, const cplx<T>* __restrict__ in,
                    const cplx<T>* __restrict__ in_lo, const cplx<T>* __restrict__ in_hi,
                    const cplx<T>* __restrict__ U, const cplx<T>* __restrict__ U_lo,
                    const cplx<T>* __restrict__ b, T diag, int Lx, int Ly, int RY,
                    double* __restrict__ partials, unsigned int* __restrict__ counter,
                    double* __restrict__ dots, XComm* xc, const T* __restrict__ F, T mu) {
    using C = cplx<T>;
    const int nsx = (Lx + WX - 1) / WX;
    const int nsy = (Ly + RY - 1) / RY;
    const int nwork = nsx * nsy;
    const int lane = threadIdx.x & 31;
    double red[4] = {0.0, 0.0, 0.0, 0.0};
    const T half = (T)0.5;

    for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
        const int wy = w / nsx, wx = w - wy * nsx;
        const int x = wx * WX + threadIdx.x;
        const bool active = x < Lx;
        const int xc = active ? x : Lx - 1;                  // clamp so that every lane takes part in shuffles
        const int xp = (xc + 1 == Lx) ? 0 : xc + 1;
        const int xm = (xc == 0) ? Lx - 1 : xc - 1;
        const int y0 = wy * RY;
        const int y1 = min(y0 + RY, Ly);

        // rolling rows: prev = row y-1, cur = row y, next = row y+1
        Spinor<T> prev = (y0 == 0) ? load_spinor<T>(in_lo, xc) : load_spinor<T>(in, (size_t)(y0 - 1) * Lx + xc);
        Spinor<T> cur = load_spinor<T>(in, (size_t)y0 * Lx + xc);
        C uy_prev = (y0 == 0) ? __ldg(U_lo + 2 * (size_t)xc + 1) : __ldg(U + 2 * ((size_t)(y0 - 1) * Lx + xc) + 1);

        for (int y = y0; y < y1; ++y) {
            const size_t s = (size_t)y * Lx + xc;
            Spinor<T> next = (y + 1 == Ly) ? load_spinor<T>(in_hi, xc) : load_spinor<T>(in, s + Lx);
            const Spinor<T> lk = load_spinor<T>(U, s);            // (U_x(s), U_y(s)) share the spinor layout
            const C ux = lk.c0, uy = lk.c1;

            // x-direction half spinors of THIS site, to be handed to the neighbours
            C a_here = csub(cur.c0, cur.c1);                      // needed by site x-1  (their +x hop)
            C wb_here = cmulc(ux, cadd(cur.c0, cur.c1));          // conj(U_x(s)) b(s): needed by site x+1
            C a_xp = shfl_c(a_here, lane + 1);                    // a(s+x)
            C wb_xm = shfl_c(wb_here, lane - 1);                  // conj(U_x(s-x)) b(s-x)
            if (lane == 31 || xc + 1 == Lx) {                     // warp edge / periodic wrap: global load
                Spinor<T> q = load_spinor<T>(in, (size_t)y * Lx + xp);
                a_xp = csub(q.c0, q.c1);
            }
            if (lane == 0) {
                Spinor<T> q = load_spinor<T>(in, (size_t)y * Lx + xm);
                C uxm = __ldg(U + 2 * ((size_t)y * Lx + xm));
                wb_xm = cmulc(uxm, cadd(q.c0, q.c1));
            }
            const C A = cmul(ux, a_xp);
            const C B = wb_xm;
            const C Cc = cmul(uy, cadd(next.c0, cmul_i(next.c1)));        // U_y(s) c(s+y)
            const C Dd = cmulc(uy_prev, csub(prev.c0, cmul_i(prev.c1)));  // conj(U_y(s-y)) d(s-y)

            Spinor<T> o;
            C h0 = cadd(cadd(A, B), cadd(Cc, Dd));
            C h1 = cadd(csub(B, A), cmul_i(csub(Dd, Cc)));
            o.c0.x = fma(diag, cur.c0.x, half * h0.x); o.c0.y = fma(diag, cur.c0.y, half * h0.y);
            o.c1.x = fma(diag, cur.c1.x, half * h1.x); o.c1.y = fma(diag, cur.c1.y, half * h1.y);
            if (SW) {                                             // + f s3 psi(s)
                const T f = __ldg(F + s);
                o.c0.x = fma(f, cur.c0.x, o.c0.x); o.c0.y = fma(f, cur.c0.y, o.c0.y);
                o.c1.x = fma(-f, cur.c1.x, o.c1.x); o.c1.y = fma(-f, cur.c1.y, o.c1.y);
            }
            if (TM) {                                             // + i mu s3 psi(s)
                o.c0.x = fma(-mu, cur.c0.y, o.c0.x); o.c0.y = fma(mu, cur.c0.x, o.c0.y);
                o.c1.x = fma(mu, cur.c1.y, o.c1.x); o.c1.y = fma(-mu, cur.c1.x, o.c1.y);
            }
            if (MODE == 1) {
                Spinor<T> bb = load_spinor<T>(b, s);
                if (DOTS && active) red[3] += (double)bb.c0.x * bb.c0.x + (double)bb.c0.y * bb.c0.y
                                            + (double)bb.c1.x * bb.c1.x + (double)bb.c1.y * bb.c1.y;
                o.c0 = csub(bb.c0, o.c0); o.c1 = csub(bb.c1, o.c1);
            }
            if (active) {
                store_spinor<T>(out, s, o);
                if (DOTS) {
                    red[0] += (double)o.c0.x * o.c0.x + (double)o.c0.y * o.c0.y
                            + (double)o.c1.x * o.c1.x + (double)o.c1.y * o.c1.y;
                    // <out, in> = conj(out) * in
                    red[1] += (double)o.c0.x * cur.c0.x + (double)o.c0.y * cur.c0.y
                            + (double)o.c1.x * cur.c1.x + (double)o.c1.y * cur.c1.y;
                    red[2] += (double)o.c0.x * cur.c0.y - (double)o.c0.y * cur.c0.x
                            + (double)o.c1.x * cur.c1.y - (double)o.c1.y * cur.c1.x;
                }
            }
            prev = cur; cur = next; uy_prev = uy;
        }
    }
    if (DOTS) grid_reduce<4, WX>(red, partials, counter, dots, blockIdx.x, gridDim.x, xc);
}

// red-black Gauss-Seidel half sweep, matrix-free: phi(s) = (r(s) - hop(s)) / (2+m) on the sites with
// (x + y + yoff) % 2 == colour (f_relax's update, S6/level.h:116-121, with D0 = (2+m) 1).  One thread per
// updated site; a warp covers 64 consecutive x.  Traffic per full sweep (c128): phi 32+32, r 32, links 2x32; SW: + f 8.
// SW: D0 = diag(d+f, d-f), d = 2+m, inverted from one reciprocal 1/((d+f)(d-f)); a site with f == 0 uses inv_diag itself,
// so c_sw = 0 reproduces the Wilson sweep bit for bit.
// TM: D0 = diag(d+f+i mu, d-f-i mu) (f = 0 without SW), inverted by tm_self_inverse (spinor.cuh), tz = 1/(d+i mu).
template <typename T, bool SW, bool TM>
__global__ void __launch_bounds__(256)
wilson_rb_kernel(cplx<T>* phi, const cplx<T>* lo, const cplx<T>* hi, const cplx<T>* __restrict__ U,
                 const cplx<T>* __restrict__ U_lo, const cplx<T>* __restrict__ r, T inv_diag, int Lx, int Ly,
                 int colour, int yoff, const T* __restrict__ F, T diag, T mu, cplx<T> tz) {
    using C = cplx<T>;
    const int Lh = Lx / 2;
    const long long S2 = (long long)Lh * Ly;
    const T half = (T)0.5;
    for (long long h = blockIdx.x * (long long)blockDim.x + threadIdx.x; h < S2; h += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(h / Lh);
        const int x = 2 * (int)(h - (long long)y * Lh) + ((y + yoff + colour) & 1);
        const size_t row = (size_t)y * Lx, s = row + x;
        const int xp = (x + 1 == Lx) ? 0 : x + 1, xm = (x == 0) ? Lx - 1 : x - 1;
        const Spinor<T> qxp = load_spinor_c<T>(phi, row + xp), qxm = load_spinor_c<T>(phi, row + xm);
        const Spinor<T> qyp = (y + 1 == Ly) ? load_spinor_c<T>(hi, x) : load_spinor_c<T>(phi, s + Lx);
        const Spinor<T> qym = (y == 0) ? load_spinor_c<T>(lo, x) : load_spinor_c<T>(phi, s - Lx);
        const Spinor<T> lk = load_spinor<T>(U, s);
        const C uxm = __ldg(U + 2 * (row + xm));
        const C uym = (y == 0) ? __ldg(U_lo + 2 * (size_t)x + 1) : __ldg(U + 2 * (s - Lx) + 1);
        const C A = cmul(lk.c0, csub(qxp.c0, qxp.c1));
        const C B = cmulc(uxm, cadd(qxm.c0, qxm.c1));
        const C Cc = cmul(lk.c1, cadd(qyp.c0, cmul_i(qyp.c1)));
        const C Dd = cmulc(uym, csub(qym.c0, cmul_i(qym.c1)));
        const C h0 = cadd(cadd(A, B), cadd(Cc, Dd));
        const C h1 = cadd(csub(B, A), cmul_i(csub(Dd, Cc)));
        T i0 = inv_diag, i1 = inv_diag;
        if (SW && !TM) {
            const T f = __ldg(F + s);
            if (f != (T)0) { const T q = (T)1 / ((diag + f) * (diag - f)); i0 = (diag - f) * q; i1 = (diag + f) * q; }
        }
        Spinor<T> o;
        if (TM) {
            C z0, z1;
            tm_self_inverse<T>(SW ? __ldg(F + s) : (T)0, diag, mu, tz, z0, z1);
            C t0 = mk<T>(-half * h0.x, -half * h0.y), t1 = mk<T>(-half * h1.x, -half * h1.y);
            if (r) { const Spinor<T> rr = load_spinor<T>(r, s); t0 = cadd(rr.c0, t0); t1 = cadd(rr.c1, t1); }
            o.c0 = cmul(t0, z0); o.c1 = cmul(t1, z1);
        } else if (r) {
            const Spinor<T> rr = load_spinor<T>(r, s);
            o.c0.x = (rr.c0.x - half * h0.x) * i0; o.c0.y = (rr.c0.y - half * h0.y) * i0;
            o.c1.x = (rr.c1.x - half * h1.x) * i1; o.c1.y = (rr.c1.y - half * h1.y) * i1;
        } else {
            o.c0.x = -half * h0.x * i0; o.c0.y = -half * h0.y * i0;
            o.c1.x = -half * h1.x * i1; o.c1.y = -half * h1.y * i1;
        }
        store_spinor<T>(phi, s, o);
    }
}

// materialise D[s][5][n][n] (column-major blocks) for the level-0 operator
template <typename T>
__global__ void lvl0_matrix_kernel(cplx<T>* __restrict__ D, const cplx<T>* __restrict__ U,
                                   const cplx<T>* __restrict__ U_lo, T diag, int wilson, int Lx, int Ly) {
    using C = cplx<T>;
    const size_t S = (size_t)Lx * Ly;
    for (size_t s = blockIdx.x * (size_t)blockDim.x + threadIdx.x; s < S; s += (size_t)gridDim.x * blockDim.x) {
        const int y = (int)(s / Lx), x = (int)(s - (size_t)y * Lx);
        const int xm = (x == 0) ? Lx - 1 : x - 1;
        const C ux = U[2 * s], uy = U[2 * s + 1];
        const C uxm = cconj(U[2 * ((size_t)y * Lx + xm)]);
        const C uym = cconj(y == 0 ? U_lo[2 * (size_t)x + 1] : U[2 * ((size_t)(y - 1) * Lx + x) + 1]);
        const C zero = mk<T>(0, 0);
        if (!wilson) {   // gauged Laplace, S6/level.h:139-153: D0 = -(4+m) (diag carries the sign)
            C* d = D + s * 5;
            d[0] = mk<T>(diag, 0); d[1] = ux; d[2] = uxm; d[3] = uy; d[4] = uym;
        } else {         // S6/level.h:155-172; block (i,j) stored at j*2+i
            C* d = D + s * 20;
            const T h = (T)0.5;
            d[0] = mk<T>(diag, 0); d[1] = zero; d[2] = zero; d[3] = mk<T>(diag, 0);
            // 1/2 (1 - s1) = 1/2 [[1,-1],[-1,1]]
            C p = cscale(ux, h), mneg = cscale(ux, -h);
            d[4] = p; d[5] = mneg; d[6] = mneg; d[7] = p;
            // 1/2 (1 + s1) = 1/2 [[1,1],[1,1]]
            p = cscale(uxm, h);
            d[8] = p; d[9] = p; d[10] = p; d[11] = p;
            // 1/2 (1 - s2) = 1/2 [[1, i],[-i, 1]]  -> (0,0)=1,(1,0)=-i,(0,1)=i,(1,1)=1 (column-major order)
            p = cscale(uy, h);
            d[12] = p; d[13] = cmul_mi(p); d[14] = cmul_i(p); d[15] = p;
            // 1/2 (1 + s2) = 1/2 [[1,-i],[i,1]]
            p = cscale(uym, h);
            d[16] = p; d[17] = cmul_i(p); d[18] = cmul_mi(p); d[19] = p;
        }
    }
}

// clover term of the stored level-0 Wilson operator: D[s][0] += diag(F[s], -F[s])  (column-major: (0,0) at 0, (1,1) at 3)
template <typename T>
__global__ void clover_add_kernel(cplx<T>* __restrict__ D, const T* __restrict__ F, long long S) {
    for (long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x; s < S; s += (long long)gridDim.x * blockDim.x) {
        const T f = F[s];
        D[20 * s].x += f;
        D[20 * s + 3].x -= f;
    }
}

// twisted-mass term of the stored level-0 Wilson operator: D[s][0] += diag(i mu, -i mu)
template <typename T>
__global__ void twist_add_kernel(cplx<T>* __restrict__ D, T mu, long long S) {
    for (long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x; s < S; s += (long long)gridDim.x * blockDim.x) {
        D[20 * s].y += mu;
        D[20 * s + 3].y -= mu;
    }
}

// a stored operator's twist set in place: Im D[s][0](i,i) = base[s][i] + delta Gamma5_c(i,i), Gamma5_c = diag(+1 x n/2, -1 x n/2),
// summed in fp64 and rounded once to T (delta = 0 writes back the fp64 copy of the imaginary parts exactly)
template <typename T>
__global__ void twist_set_kernel(cplx<T>* __restrict__ D, const double* __restrict__ base, double delta, int n, long long S) {
    const long long nel = S * n;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < nel; e += (long long)gridDim.x * blockDim.x) {
        const long long s = e / n;
        const int i = (int)(e - s * n);
        const double v = base[e] + (2 * i < n ? delta : -delta);
        D[(size_t)s * 5 * n * n + (size_t)i * n + i].y = (T)v;
    }
}

template <typename T>
int launch_wilson(mg2d_ctx* ctx, void* out, const void* in, const void* in_lo, const void* in_hi, const void* U,
                  const void* U_lo, const void* F, const void* b, double mass, bool tm, double mu, int Lx, int Ly, int mode,
                  double* dots, cudaStream_t st, const char* name) {
    using C = cplx<T>;
    // rows per work item: as many as possible (each item re-reads 2 halo rows) while >= 6 CTAs per SM exist
    int RY = RY_MAX;
    while (RY > 4 && ((Lx + WX - 1) / WX) * ((Ly + RY - 1) / RY) < ctx->num_sms * 6) RY >>= 1;
    const int nwork = ((Lx + WX - 1) / WX) * ((Ly + RY - 1) / RY);
    int grid = nwork < MG2D_MAX_PARTIALS ? nwork : MG2D_MAX_PARTIALS;
    const T diag = (T)(2.0 + mass);
#define WL(MODE, DOTS, SW, TM)                                                                              \
    wilson_march_kernel<T, MODE, DOTS, SW, TM><<<grid, WX, 0, st>>>((C*)out, (const C*)in, (const C*)in_lo,  \
        (const C*)in_hi, (const C*)U, (const C*)U_lo, (const C*)b, diag, Lx, Ly, RY, ctx->partials, ctx->counter, dots, \
        ctx->xreduce ? ctx->xcomm : nullptr, (const T*)F, (T)mu)
#define WL_MODES(SW, TM)                                                                                    \
    if (mode == MG2D_MODE_APPLY) { if (dots) WL(0, true, SW, TM); else WL(0, false, SW, TM); }              \
    else                         { if (dots) WL(1, true, SW, TM); else WL(1, false, SW, TM); }
    if (tm) {
        if (F) { WL_MODES(true, true) } else { WL_MODES(false, true) }
    } else {
        if (F) { WL_MODES(true, false) } else { WL_MODES(false, false) }
    }
#undef WL_MODES
#undef WL
    return mg2d_check_launch(ctx, name);
}

int wilson_apply(mg2d_ctx* ctx, void* out, const void* in, const void* in_lo, const void* in_hi, const void* U, const void* U_lo,
                 const void* F, const void* b, double mass, bool tm, double mu, int Lx, int Ly, int mode, int dtype, double* dots,
                 void* stream, const char* name) {
    if (!ctx) return MG2D_EINVAL;
    if (!out || !in || !in_lo || !in_hi || !U || !U_lo || Lx < 2 || Ly < 1) return mg2d_fail2(ctx, name, "bad argument");
    if (mode == MG2D_MODE_RESID && !b) return mg2d_fail2(ctx, name, "MODE_RESID needs b");
    if (mode != MG2D_MODE_APPLY && mode != MG2D_MODE_RESID) return mg2d_fail2(ctx, name, "bad mode");
    if (out == in) return mg2d_fail2(ctx, name, "out must not alias in");
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MG2D_C128) return launch_wilson<double>(ctx, out, in, in_lo, in_hi, U, U_lo, F, b, mass, tm, mu, Lx, Ly, mode, dots, st, name);
    if (dtype == MG2D_C64)  return launch_wilson<float>(ctx, out, in, in_lo, in_hi, U, U_lo, F, b, mass, tm, mu, Lx, Ly, mode, dots, st, name);
    return mg2d_fail2(ctx, name, "bad dtype");
}

int wilson_relax_rb(mg2d_ctx* ctx, void* phi, const void* phi_lo, const void* phi_hi, const void* U, const void* U_lo,
                    const void* F, const void* r, double mass, bool tm, double mu, int Lx, int Ly, int colour, int yoff, int dtype,
                    void* stream, const char* name) {
    if (!ctx) return MG2D_EINVAL;
    if (!phi || !phi_lo || !phi_hi || !U || !U_lo || Lx < 2 || (Lx & 1) || Ly < 1 || (colour != 0 && colour != 1))
        return mg2d_fail2(ctx, name, "bad argument (Lx must be even)");
    cudaStream_t st = (cudaStream_t)stream;
    const long long S2 = (long long)(Lx / 2) * Ly;
    long long nb = (S2 + 255) / 256; if (nb > (long long)ctx->num_sms * 32) nb = (long long)ctx->num_sms * 32;
    const double inv = 1.0 / (2.0 + mass);
#define RB(T, SW, TM) wilson_rb_kernel<T, SW, TM><<<(int)nb, 256, 0, st>>>((cplx<T>*)phi, (const cplx<T>*)phi_lo,   \
        (const cplx<T>*)phi_hi, (const cplx<T>*)U, (const cplx<T>*)U_lo, (const cplx<T>*)r, (T)inv, Lx, Ly, colour, yoff,  \
        (const T*)F, (T)(2.0 + mass), (T)mu, tm_tz<T>(2.0 + mass, mu))
#define RB_SW(T, TM) { if (F) RB(T, true, TM); else RB(T, false, TM); }
    if (dtype == MG2D_C128) { if (tm) RB_SW(double, true) else RB_SW(double, false) }
    else if (dtype == MG2D_C64) { if (tm) RB_SW(float, true) else RB_SW(float, false) }
    else return mg2d_fail2(ctx, name, "bad dtype");
#undef RB_SW
#undef RB
    return mg2d_check_launch(ctx, name);
}

}  // namespace

extern "C" int mg2d_wilson_apply(mg2d_ctx* ctx, void* out, const void* in, const void* in_lo, const void* in_hi,
                                 const void* U, const void* U_lo, const void* b, double mass, int Lx, int Ly,
                                 int mode, int dtype, double* dots, void* stream) {
    return wilson_apply(ctx, out, in, in_lo, in_hi, U, U_lo, nullptr, b, mass, false, 0.0, Lx, Ly, mode, dtype, dots, stream,
                        "mg2d_wilson_apply");
}

extern "C" int mg2d_wilson_sw_apply(mg2d_ctx* ctx, void* out, const void* in, const void* in_lo, const void* in_hi,
                                    const void* U, const void* U_lo, const void* F, const void* b, double mass, int Lx, int Ly,
                                    int mode, int dtype, double* dots, void* stream) {
    if (ctx && !F) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_wilson_sw_apply: F is NULL");
    return wilson_apply(ctx, out, in, in_lo, in_hi, U, U_lo, F, b, mass, false, 0.0, Lx, Ly, mode, dtype, dots, stream,
                        "mg2d_wilson_sw_apply");
}

extern "C" int mg2d_wilson_tm_apply(mg2d_ctx* ctx, void* out, const void* in, const void* in_lo, const void* in_hi,
                                    const void* U, const void* U_lo, const void* F, const void* b, double mass, double mu, int Lx,
                                    int Ly, int mode, int dtype, double* dots, void* stream) {
    if (ctx && !std::isfinite(mu)) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_wilson_tm_apply: mu is not finite");
    return wilson_apply(ctx, out, in, in_lo, in_hi, U, U_lo, F, b, mass, true, mu, Lx, Ly, mode, dtype, dots, stream,
                        "mg2d_wilson_tm_apply");
}

extern "C" int mg2d_lvl0_matrix(mg2d_ctx* ctx, void* D, const void* U, const void* U_lo, double mass, int stencil,
                                int Lx, int Ly, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!D || !U || !U_lo || Lx < 1 || Ly < 1 || (stencil != 0 && stencil != 1)) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_lvl0_matrix: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t S = (size_t)Lx * Ly;
    int grid = (int)((S + 255) / 256); if (grid > ctx->num_sms * 8) grid = ctx->num_sms * 8;
    const int wilson = stencil == 0;
    const double diag = wilson ? (2.0 + mass) : -(4.0 + mass);
    if (dtype == MG2D_C128) lvl0_matrix_kernel<double><<<grid, 256, 0, st>>>((double2*)D, (const double2*)U, (const double2*)U_lo, diag, wilson, Lx, Ly);
    else if (dtype == MG2D_C64) lvl0_matrix_kernel<float><<<grid, 256, 0, st>>>((float2*)D, (const float2*)U, (const float2*)U_lo, (float)diag, wilson, Lx, Ly);
    else return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_lvl0_matrix: bad dtype");
    return mg2d_check_launch(ctx, "mg2d_lvl0_matrix");
}

extern "C" int mg2d_clover_add(mg2d_ctx* ctx, void* D, const void* F, long long nsites, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!D || !F || nsites < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_clover_add: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    long long grid = (nsites + 255) / 256; if (grid > (long long)ctx->num_sms * 8) grid = (long long)ctx->num_sms * 8;
    if (dtype == MG2D_C128) clover_add_kernel<double><<<(int)grid, 256, 0, st>>>((double2*)D, (const double*)F, nsites);
    else if (dtype == MG2D_C64) clover_add_kernel<float><<<(int)grid, 256, 0, st>>>((float2*)D, (const float*)F, nsites);
    else return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_clover_add: bad dtype");
    return mg2d_check_launch(ctx, "mg2d_clover_add");
}

extern "C" int mg2d_twist_add(mg2d_ctx* ctx, void* D, double mu, long long nsites, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!D || nsites < 1 || !std::isfinite(mu)) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_twist_add: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    long long grid = (nsites + 255) / 256; if (grid > (long long)ctx->num_sms * 8) grid = (long long)ctx->num_sms * 8;
    if (dtype == MG2D_C128) twist_add_kernel<double><<<(int)grid, 256, 0, st>>>((double2*)D, mu, nsites);
    else if (dtype == MG2D_C64) twist_add_kernel<float><<<(int)grid, 256, 0, st>>>((float2*)D, (float)mu, nsites);
    else return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_twist_add: bad dtype");
    return mg2d_check_launch(ctx, "mg2d_twist_add");
}

extern "C" int mg2d_twist_set(mg2d_ctx* ctx, void* D, const double* base, double delta, int n, long long nsites, int dtype,
                              void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!D || !base || nsites < 1 || !std::isfinite(delta)) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_twist_set: bad argument");
    if (n != 2 && n != 4 && n != 8 && n != 16 && n != 32)
        return mg2d_fail(ctx, MG2D_EUNSUPPORTED, "mg2d_twist_set: n_dof must be one of 2,4,8,16,32");
    cudaStream_t st = (cudaStream_t)stream;
    const long long nel = nsites * n;
    long long grid = (nel + 255) / 256; if (grid > (long long)ctx->num_sms * 8) grid = (long long)ctx->num_sms * 8;
    if (dtype == MG2D_C128) twist_set_kernel<double><<<(int)grid, 256, 0, st>>>((double2*)D, base, delta, n, nsites);
    else if (dtype == MG2D_C64) twist_set_kernel<float><<<(int)grid, 256, 0, st>>>((float2*)D, base, delta, n, nsites);
    else return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_twist_set: bad dtype");
    return mg2d_check_launch(ctx, "mg2d_twist_set");
}

extern "C" int mg2d_wilson_relax_rb(mg2d_ctx* ctx, void* phi, const void* phi_lo, const void* phi_hi, const void* U,
                                    const void* U_lo, const void* r, double mass, int Lx, int Ly, int colour, int yoff,
                                    int dtype, void* stream) {
    return wilson_relax_rb(ctx, phi, phi_lo, phi_hi, U, U_lo, nullptr, r, mass, false, 0.0, Lx, Ly, colour, yoff, dtype, stream,
                           "mg2d_wilson_relax_rb");
}

extern "C" int mg2d_wilson_sw_relax_rb(mg2d_ctx* ctx, void* phi, const void* phi_lo, const void* phi_hi, const void* U,
                                       const void* U_lo, const void* F, const void* r, double mass, int Lx, int Ly, int colour,
                                       int yoff, int dtype, void* stream) {
    if (ctx && !F) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_wilson_sw_relax_rb: F is NULL");
    return wilson_relax_rb(ctx, phi, phi_lo, phi_hi, U, U_lo, F, r, mass, false, 0.0, Lx, Ly, colour, yoff, dtype, stream,
                           "mg2d_wilson_sw_relax_rb");
}

extern "C" int mg2d_wilson_tm_relax_rb(mg2d_ctx* ctx, void* phi, const void* phi_lo, const void* phi_hi, const void* U,
                                       const void* U_lo, const void* F, const void* r, double mass, double mu, int Lx, int Ly,
                                       int colour, int yoff, int dtype, void* stream) {
    if (ctx && !std::isfinite(mu)) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_wilson_tm_relax_rb: mu is not finite");
    return wilson_relax_rb(ctx, phi, phi_lo, phi_hi, U, U_lo, F, r, mass, true, mu, Lx, Ly, colour, yoff, dtype, stream,
                           "mg2d_wilson_tm_relax_rb");
}
