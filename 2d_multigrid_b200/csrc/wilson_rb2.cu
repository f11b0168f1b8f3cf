// wilson_rb2.cu -- matrix-free red-black Gauss-Seidel sweep of the U(1) Wilson operator, BOTH colours in one pass.
//
// Update rule of Level::f_relax (S6/level.h:116-121) with the level-0 Wilson stencil of f_compute_lvl0_matrix
// (S6/level.h:155-172, D0 = (2+m) 1), in the two-colour ordering (colour (x+y+yoff)%2 == 0 first, then colour 1;
// mirrored by oracle Level.relax_rb):   phi(s) <- (r(s) - hop(s)) / (2+m).
//
// Why one pass: the half-sweep kernel (wilson_rb_kernel) touches one 32-byte spinor out of every 64 bytes of phi and
// r, so DRAM moves ~1.4x the algorithmic bytes (ncu, round 1: 105 MB for 67 MB) and each field is streamed twice per
// sweep.  Here a warp owns a tile of 64 consecutive columns (two per lane) and marches in y with a one-row lag
// between the colours:
//     step rho:   stage R(rho)   : red site of row rho     from the OLD black values of rows rho-1, rho, rho+1
//                 stage B(rho-1) : black site of row rho-1 from the NEW red values of rows rho-2, rho-1, rho
// All intermediate values live in registers (3 black + 3 red spinors per lane); x-neighbours arrive as projected
// half-spinors through one warp shuffle per stage.  The new red values a black update needs from outside the tile
// are recomputed: the two outer columns of a tile and the rows y0-1 / y1 of a chunk are halo (computed, not stored),
// which needs OLD data two rows / two columns deep -- hence the sweep is out of place (out != in) and strips take
// two-row halos `in_lo2` / `in_hi2`.  Old red values are never read.
// Traffic per site and sweep (c128): phi 32 (read) + 32 (write) + links 32 + r 32 = 128 B, every byte of every
// fetched line used (the half-sweep kernel: 160 B algorithmic, ~224 B moved).
//
// Clover variant (template flag SW): D0 = diag(d+f, d-f) with d = 2+m and the real site field f of mg2d_clover_field; every
// update (halo rows and columns included) loads its site's f once and inverts D0 from one reciprocal 1/((d+f)(d-f)).  The red stage recomputes rows -1 and Ly, so strips pass f there as F_lo / F_hi.
// Traffic: + f 8 B/site = 136 B (c64: 68 B).
//
// Twisted-mass variant (template flag TM, with or without SW): D0 = diag(d+f+i mu, d-f-i mu), f = 0 without SW, inverted by
// tm_self_inverse (spinor.cuh): the launch constants tz = 1/(d+i mu) and conj(tz) without clover, one reciprocal per site
// with it.  mu has no halo; the bytes are those of the Wilson / SW sweep.
#include <cmath>
#include "common.cuh"
#include "spinor.cuh"

namespace {

constexpr int RB2_THREADS = 128;
constexpr int RB2_W = 62;        // inner (stored) columns per warp tile; lanes hold columns X0-1 .. X0+62

template <typename T>
struct Rb2Args {
    cplx<T>* out;
    const cplx<T>* in; const cplx<T>* in_lo2; const cplx<T>* in_hi2;
    const cplx<T>* U; const cplx<T>* U_lo2; const cplx<T>* U_hi;
    const cplx<T>* r; const cplx<T>* r_lo; const cplx<T>* r_hi;
    T inv_diag;
    int Lx, Ly, RY, yoff;
    HaloLinkDev link;      // strips: fused neighbour push / wait (mine == NULL: none)
    const T* F; const T* F_lo; const T* F_hi;    // SW: clover field of the local rows, rows -1 and Ly
    T diag;                                      // SW: 2+m
    T mu;                                        // TM: twisted mass
    T tz_re, tz_im;                              // TM: 1/(2+m + i mu) (two reals: a complex member would realign the struct)
};

// a * b and conj(a) * b with the rounding written out: each component is fma(first product, second product rounded).  Left
// to the compiler, which of the two products is fused follows the instruction schedule, and it differed between the LINKED
// and the unlinked instantiation: a strip relaxed to last-bit different values than the same rows on one GPU.
template <typename C> __device__ __forceinline__ C rb2_mul(C a, C b) {
    C r; r.x = fma(a.x, b.x, -(a.y * b.y)); r.y = fma(a.x, b.y, a.y * b.x); return r;
}
template <typename C> __device__ __forceinline__ C rb2_mulc(C a, C b) {
    C r; r.x = fma(a.x, b.x, a.y * b.y); r.y = fma(a.x, b.y, -(a.y * b.x)); return r;
}

template <typename T>
__device__ __forceinline__ const cplx<T>* rb2_row(const cplx<T>* f, const cplx<T>* lo2, const cplx<T>* hi, int y, int Lx, int Ly) {
    if (y < 0) return lo2 + (size_t)(y + 2) * Lx * 2;
    if (y >= Ly) return hi + (size_t)(y - Ly) * Lx * 2;
    return f + (size_t)y * Lx * 2;
}

// phi of row y, column x: rows outside [0, Ly) come from the halo buffers, which on linked strips a neighbour kernel has
// just written over NVLink (read them with system-scope loads, never through the non-coherent path)
template <typename T>
__device__ __forceinline__ Spinor<T> rb2_phi(const Rb2Args<T>& a, int y, int x, bool linked) {
    const cplx<T>* row = rb2_row<T>(a.in, a.in_lo2, a.in_hi2, y, a.Lx, a.Ly);
    if (linked && (y < 0 || y >= a.Ly)) return load_spinor_sys<T>(row, (size_t)x);
    return load_spinor<T>(row, (size_t)x);
}

// clover field at (y, x), y in [-1, Ly]
template <typename T>
__device__ __forceinline__ T rb2_f(const Rb2Args<T>& a, int y, int x) {
    const T* row = (y < 0) ? a.F_lo : (y >= a.Ly ? a.F_hi : a.F + (size_t)y * a.Lx);
    return __ldg(row + x);
}

// phi(s) <- (r(s) - 1/2 hop(s)) / (2+m);  a_xp = (psi0 - psi1)(s+x), wb_xm = conj(U_x(s-x)) (psi0 + psi1)(s-x)
// SW: component 0 divided by d+f, component 1 by d-f (f == 0: inv_diag itself, as in wilson_rb_kernel)
// TM: component 0 divided by d+f+i mu, component 1 by d-f-i mu
template <typename T, bool HAS_R, bool SW, bool TM>
__device__ __forceinline__ Spinor<T> rb2_update(cplx<T> ux, cplx<T> a_xp, cplx<T> wb_xm, cplx<T> uy, const Spinor<T>& qyp,
                                                cplx<T> uym, const Spinor<T>& qym, const cplx<T>* __restrict__ r_row, int x,
                                                T inv_diag, const Rb2Args<T>& a, int y) {
    using C = cplx<T>;
    const T half = (T)0.5;
    const C A = rb2_mul(ux, a_xp);
    const C B = wb_xm;
    const C Cc = rb2_mul(uy, cadd(qyp.c0, cmul_i(qyp.c1)));
    const C Dd = rb2_mulc(uym, csub(qym.c0, cmul_i(qym.c1)));
    const C h0 = cadd(cadd(A, B), cadd(Cc, Dd));
    const C h1 = cadd(csub(B, A), cmul_i(csub(Dd, Cc)));
    T i0 = inv_diag, i1 = inv_diag;
    if (SW && !TM) {
        const T f = rb2_f<T>(a, y, x), d = a.diag;
        if (f != (T)0) { const T q = (T)1 / ((d + f) * (d - f)); i0 = (d - f) * q; i1 = (d + f) * q; }
    }
    Spinor<T> o;
    if (TM) {
        C z0, z1;
        tm_self_inverse<T>(SW ? rb2_f<T>(a, y, x) : (T)0, a.diag, a.mu, mk<T>(a.tz_re, a.tz_im), z0, z1);
        C t0 = mk<T>(-half * h0.x, -half * h0.y), t1 = mk<T>(-half * h1.x, -half * h1.y);
        if (HAS_R) { const Spinor<T> rr = load_spinor<T>(r_row, (size_t)x); t0 = cadd(rr.c0, t0); t1 = cadd(rr.c1, t1); }
        o.c0 = rb2_mul(t0, z0); o.c1 = rb2_mul(t1, z1);
    } else if (HAS_R) {
        const Spinor<T> rr = load_spinor<T>(r_row, (size_t)x);
        o.c0.x = (rr.c0.x - half * h0.x) * i0; o.c0.y = (rr.c0.y - half * h0.y) * i0;
        o.c1.x = (rr.c1.x - half * h1.x) * i1; o.c1.y = (rr.c1.y - half * h1.y) * i1;
    } else {
        o.c0.x = -half * h0.x * i0; o.c0.y = -half * h0.y * i0;
        o.c1.x = -half * h1.x * i1; o.c1.y = -half * h1.y * i1;
    }
    return o;
}

// row y of the result: the lane's two columns; boundary rows also go to the strip neighbours' halo buffers
// (rows 0,1 -> prev's hi2 buffer, rows Ly-2,Ly-1 -> next's lo2 buffer)
template <typename T>
__device__ __forceinline__ void rb2_store(const Rb2Args<T>& a, int y, int x0, int x1, bool act0, bool act1, const Spinor<T>& v0,
                                          const Spinor<T>& v1, cplx<T>* push_lo, cplx<T>* push_hi) {
    cplx<T>* orow = a.out + (size_t)y * a.Lx * 2;
    if (act0) store_spinor<T>(orow, (size_t)x0, v0);
    if (act1) store_spinor<T>(orow, (size_t)x1, v1);
    if (push_lo) {
        if (y < 2) {
            cplx<T>* prow = push_hi + (size_t)y * a.Lx * 2;
            if (act0) store_spinor<T>(prow, (size_t)x0, v0);
            if (act1) store_spinor<T>(prow, (size_t)x1, v1);
        }
        if (y + 2 >= a.Ly) {
            cplx<T>* prow = push_lo + (size_t)(y + 2 - a.Ly) * a.Lx * 2;
            if (act0) store_spinor<T>(prow, (size_t)x0, v0);
            if (act1) store_spinor<T>(prow, (size_t)x1, v1);
        }
    }
}

template <typename T, bool HAS_R, bool LINKED, bool SW, bool TM>
__global__ void __launch_bounds__(RB2_THREADS, 4)
wilson_rb2_kernel(Rb2Args<T> a) {
    using C = cplx<T>;
    const int Lx = a.Lx, Ly = a.Ly, RY = a.RY;
    const int lane = threadIdx.x & 31;
    const int ntx = (Lx + RB2_W - 1) / RB2_W;
    const int nchunks = (Ly + RY - 1) / RY;
    const long long nitems = (long long)ntx * nchunks;
    const long long wstride = (long long)gridDim.x * (RB2_THREADS / 32);
    // strips: chunks that touch the halo rows wait for the neighbours' rows (flags >= local epoch) before their first halo
    // read and store the boundary rows they produce into the neighbours' two-row halo buffers (mg2d_halo_link, include/mg2d.h)
    constexpr bool linked = LINKED;
    unsigned long long epoch = 0ull;
    bool waited = false, ticketed = false;
    C* push_lo = nullptr; C* push_hi = nullptr;
    // chunks whose rows touch the halo (chunk 0 and the last one or two: y1 + 2 > Ly) come FIRST, in item order
    // 0, nchunks-1, (nchunks-2), then the interior ascending; the warps that own them report as soon as their last boundary
    // item is stored, and the last of them publishes while the interior of this launch is still streaming
    int ntail = 0;
    if (linked) {
        push_lo = (C*)a.link.push_next_lo; push_hi = (C*)a.link.push_prev_hi;
        if (nchunks >= 2) ntail = 1;
        if (nchunks >= 3 && (long long)(nchunks - 1) * RY + 2 > Ly) ntail = 2;
    }
    const long long nbi = (long long)ntx * (1 + ntail);         // boundary items (they are the first nbi items)
    for (long long item = (long long)blockIdx.x * (RB2_THREADS / 32) + (threadIdx.x >> 5); item < nitems; item += wstride) {
        int chunk = (int)(item / ntx);
        const int tile = (int)(item - (long long)chunk * ntx);
        if (linked) chunk = (chunk == 0) ? 0 : (chunk <= ntail ? nchunks - chunk : chunk - ntail);
        const int X0 = tile * RB2_W;
        const int y0 = chunk * RY, y1 = min(y0 + RY, Ly);
        // the lane's two columns: c0 = X0 + 2*lane - 1 (odd), c1 = X0 + 2*lane (even), periodic
        const int j0 = 2 * lane - 1, j1 = 2 * lane;
        int x0 = (X0 + j0) % Lx; if (x0 < 0) x0 += Lx;
        const int x1 = (X0 + j1) % Lx;
        const bool act0 = j0 >= 0 && X0 + j0 < Lx;                 // j0 < RB2_W always
        const bool act1 = j1 < RB2_W && X0 + j1 < Lx;
        const int xm_out = (x0 == 0) ? Lx - 1 : x0 - 1;            // lane 0: column left of the tile
        const int xp_out = (x1 + 1 == Lx) ? 0 : x1 + 1;            // lane 31: column right of the tile

        if (linked && !waited && item < nbi) {                                        // warp-uniform: first boundary item
            // (the epoch only advances after every boundary warp has taken its ticket, i.e. after this read)
            epoch = a.link.mine->epoch;
            if (a.link.wait && lane == 0 && !(spin_until(&a.link.mine->flag_lo, epoch) && spin_until(&a.link.mine->flag_hi, epoch)))
                atomicExch(&a.link.mine->error, 1ull);
            __syncwarp();
            waited = true;
        }
        // rho = row of the red stage.  Black column of row y: c0 when (y + yoff) is even (then c1 is red), else c1.
        int rho = y0 - 1;
        Spinor<T> bk_m, bk_0, bk_p, rd_mm, rd_m, rd_0;
        C um_ux0, um_uy0, um_ux1, um_uy1;          // links of row rho-1, both columns
        C umm_uy0, umm_uy1;                        // U_y of row rho-2
        {
            const bool c1_red_m = ((rho - 1 + 2 + a.yoff) & 1) == 0;     // row rho-1
            bk_m = rb2_phi<T>(a, rho - 1, c1_red_m ? x0 : x1, linked);
            bk_0 = rb2_phi<T>(a, rho, c1_red_m ? x1 : x0, linked);
            const C* ur = rb2_row<T>(a.U, a.U_lo2, a.U_hi, rho - 1, Lx, Ly);
            const Spinor<T> l0 = load_spinor<T>(ur, (size_t)x0), l1 = load_spinor<T>(ur, (size_t)x1);
            um_ux0 = l0.c0; um_uy0 = l0.c1; um_ux1 = l1.c0; um_uy1 = l1.c1;
            umm_uy0 = um_uy0; umm_uy1 = um_uy1;                         // not used before the first shift
            rd_mm = bk_m; rd_m = bk_m; rd_0 = bk_m;                      // placeholders until the red stages fill them
        }
        for (; rho <= y1; ++rho) {
            const bool c1_red = ((rho + 2 + a.yoff) & 1) == 0;          // warp-uniform
            const C* urow = rb2_row<T>(a.U, a.U_lo2, a.U_hi, rho, Lx, Ly);
            const Spinor<T> l0 = load_spinor<T>(urow, (size_t)x0), l1 = load_spinor<T>(urow, (size_t)x1);
            const C u0_ux0 = l0.c0, u0_uy0 = l0.c1, u0_ux1 = l1.c0, u0_uy1 = l1.c1;
            // black value of row rho+1 sits in the column that is red in row rho
            bk_p = rb2_phi<T>(a, rho + 1, c1_red ? x1 : x0, linked);
            const bool do_black = (rho - 1 >= y0);                       // rho - 1 < y1 always
            const C* rrow = HAS_R ? rb2_row<T>(a.r, a.r_lo - (size_t)Lx * 2, a.r_hi, rho, Lx, Ly) : nullptr;
            const C* rrow_m = HAS_R ? rb2_row<T>(a.r, a.r_lo - (size_t)Lx * 2, a.r_hi, rho - 1, Lx, Ly) : nullptr;
            if (c1_red) {
                // ---- stage R(rho): target c1; -x source = own c0 (bk_0), +x source = lane+1's c0
                C a_here = csub(bk_0.c0, bk_0.c1);
                C a_xp = shfl_c(a_here, lane + 1);
                if (lane == 31) { const Spinor<T> q = rb2_phi<T>(a, rho, xp_out, linked); a_xp = csub(q.c0, q.c1); }
                const C wb = rb2_mulc(u0_ux0, cadd(bk_0.c0, bk_0.c1));
                rd_0 = rb2_update<T, HAS_R, SW, TM>(u0_ux1, a_xp, wb, u0_uy1, bk_p, um_uy1, bk_m, rrow, x1, a.inv_diag, a, rho);
                if (do_black) {
                    // ---- stage B(rho-1): target c1 of row rho-1; red sources of that row sit in c0 (rd_m)
                    a_here = csub(rd_m.c0, rd_m.c1);
                    a_xp = shfl_c(a_here, lane + 1);
                    const C wbm = rb2_mulc(um_ux0, cadd(rd_m.c0, rd_m.c1));
                    const Spinor<T> nb = rb2_update<T, HAS_R, SW, TM>(um_ux1, a_xp, wbm, um_uy1, rd_0, umm_uy1, rd_mm, rrow_m, x1, a.inv_diag, a, rho - 1);
                    rb2_store<T>(a, rho - 1, x0, x1, act0, act1, rd_m, nb, push_lo, push_hi);
                }
            } else {
                // ---- stage R(rho): target c0; +x source = own c1 (bk_0), -x source = lane-1's c1
                C wb_here = rb2_mulc(u0_ux1, cadd(bk_0.c0, bk_0.c1));
                C wb_xm = shfl_c(wb_here, lane - 1);
                if (lane == 0) {
                    const Spinor<T> q = rb2_phi<T>(a, rho, xm_out, linked);
                    wb_xm = rb2_mulc(__ldg(urow + 2 * (size_t)xm_out), cadd(q.c0, q.c1));
                }
                const C ap = csub(bk_0.c0, bk_0.c1);
                rd_0 = rb2_update<T, HAS_R, SW, TM>(u0_ux0, ap, wb_xm, u0_uy0, bk_p, um_uy0, bk_m, rrow, x0, a.inv_diag, a, rho);
                if (do_black) {
                    // ---- stage B(rho-1): target c0 of row rho-1; red sources of that row sit in c1 (rd_m)
                    wb_here = rb2_mulc(um_ux1, cadd(rd_m.c0, rd_m.c1));
                    wb_xm = shfl_c(wb_here, lane - 1);
                    const C apm = csub(rd_m.c0, rd_m.c1);
                    const Spinor<T> nb = rb2_update<T, HAS_R, SW, TM>(um_ux0, apm, wb_xm, um_uy0, rd_0, umm_uy0, rd_mm, rrow_m, x0, a.inv_diag, a, rho - 1);
                    rb2_store<T>(a, rho - 1, x0, x1, act0, act1, nb, rd_m, push_lo, push_hi);
                }
            }
            bk_m = bk_0; bk_0 = bk_p;
            rd_mm = rd_m; rd_m = rd_0;
            umm_uy0 = um_uy0; umm_uy1 = um_uy1;
            um_ux0 = u0_ux0; um_uy0 = u0_uy0; um_ux1 = u0_ux1; um_uy1 = u0_uy1;
        }
        if (linked && push_lo && waited && !ticketed && item + wstride >= nbi) {
            // this warp's last boundary item is stored (only boundary warps have peer stores in flight, only they are counted)
            ticketed = true;
            __threadfence_system();
            __syncwarp();
            if (lane == 0) {
                const unsigned long long nbw = (unsigned long long)(nbi < wstride ? nbi : wstride);     // warps that own boundary items
                const unsigned long long t = atomicAdd(&a.link.mine->ticket, 1ull);
                if (t == nbw - 1ull) {
                    __threadfence_system();
                    a.link.mine->ticket = 0ull;
                    publish2(&a.link.next->flag_lo, &a.link.prev->flag_hi, epoch + 1ull, a.link.relaxed);
                    a.link.mine->epoch = epoch + 1ull;
                }
            }
        }
    }
}

template <typename T>
int launch_rb2(mg2d_ctx* ctx, void* out, const void* in, const void* in_lo2, const void* in_hi2, const void* U,
               const void* U_lo2, const void* U_hi, const void* F, const void* F_lo, const void* F_hi, const void* r,
               const void* r_lo, const void* r_hi, double mass, bool tm, double mu, int Lx, int Ly, int yoff,
               const mg2d_halo_link* link, cudaStream_t st, const char* name) {
    using C = cplx<T>;
    Rb2Args<T> a;
    memset(&a.link, 0, sizeof(a.link));
    if (link) {
        a.link.mine = (HaloSlot*)link->slot_mine; a.link.prev = (HaloSlot*)link->slot_prev; a.link.next = (HaloSlot*)link->slot_next;
        a.link.push_next_lo = link->push_next_lo; a.link.push_prev_hi = link->push_prev_hi; a.link.wait = link->wait; a.link.relaxed = mg2d_publish_relaxed();
    }
    a.out = (C*)out; a.in = (const C*)in; a.in_lo2 = (const C*)in_lo2; a.in_hi2 = (const C*)in_hi2;
    a.U = (const C*)U; a.U_lo2 = (const C*)U_lo2; a.U_hi = (const C*)U_hi;
    a.r = (const C*)r; a.r_lo = (const C*)r_lo; a.r_hi = (const C*)r_hi;
    a.inv_diag = (T)(1.0 / (2.0 + mass));
    a.F = (const T*)F; a.F_lo = (const T*)F_lo; a.F_hi = (const T*)F_hi;
    a.diag = (T)(2.0 + mass);
    a.mu = (T)mu;
    { const cplx<T> tz = tm_tz<T>(2.0 + mass, mu); a.tz_re = tz.x; a.tz_im = tz.y; }
    a.Lx = Lx; a.Ly = Ly; a.yoff = yoff;
    // rows per chunk: every chunk re-reads 3 rows of phi and 2 of the links, so as long as possible while the
    // machine stays full (>= 12 warps per SM)
    const int ntx = (Lx + RB2_W - 1) / RB2_W;
    const long long want = (long long)ctx->num_sms * 12;
    int RY = 128;
    while (RY > 8 && (long long)ntx * ((Ly + RY - 1) / RY) < want) RY >>= 1;
    a.RY = RY;
    const long long nitems = (long long)ntx * ((Ly + RY - 1) / RY);
    long long grid = (nitems + RB2_THREADS / 32 - 1) / (RB2_THREADS / 32);
    const long long cap = (long long)ctx->num_sms * 4;
    if (grid > cap) grid = cap;
#define RB2(SW, TM)                                                                                         \
    if (link) {                                                                                             \
        if (r) wilson_rb2_kernel<T, true, true, SW, TM><<<(int)grid, RB2_THREADS, 0, st>>>(a);              \
        else   wilson_rb2_kernel<T, false, true, SW, TM><<<(int)grid, RB2_THREADS, 0, st>>>(a);             \
    } else {                                                                                                \
        if (r) wilson_rb2_kernel<T, true, false, SW, TM><<<(int)grid, RB2_THREADS, 0, st>>>(a);             \
        else   wilson_rb2_kernel<T, false, false, SW, TM><<<(int)grid, RB2_THREADS, 0, st>>>(a);            \
    }
    if (tm) {
        if (F) { RB2(true, true) } else { RB2(false, true) }
    } else {
        if (F) { RB2(true, false) } else { RB2(false, false) }
    }
#undef RB2
    return mg2d_check_launch(ctx, name);
}

int wilson_relax_rb2(mg2d_ctx* ctx, void* out, const void* in, const void* in_lo2, const void* in_hi2, const void* U,
                     const void* U_lo2, const void* U_hi, const void* F, const void* F_lo, const void* F_hi, const void* r,
                     const void* r_lo, const void* r_hi, double mass, bool tm, double mu, int Lx, int Ly, int yoff, int dtype,
                     const mg2d_halo_link* link, void* stream, const char* name) {
    if (!ctx) return MG2D_EINVAL;
    if (!out || !in || !in_lo2 || !in_hi2 || !U || !U_lo2 || !U_hi || Lx < 2 || (Lx & 1) || Ly < 2 || (r && (!r_lo || !r_hi)) ||
        (link && (!link->slot_mine || !link->slot_prev || !link->slot_next || ((link->push_next_lo == nullptr) != (link->push_prev_hi == nullptr))))) {
        snprintf(ctx->err, sizeof(ctx->err), "%s: bad argument (Lx even, Ly >= 2)", name);
        return MG2D_EINVAL;
    }
    if (out == in) { snprintf(ctx->err, sizeof(ctx->err), "%s: out must not alias in", name); return MG2D_EINVAL; }
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MG2D_C128) return launch_rb2<double>(ctx, out, in, in_lo2, in_hi2, U, U_lo2, U_hi, F, F_lo, F_hi, r, r_lo, r_hi, mass, tm, mu, Lx, Ly, yoff, link, st, name);
    if (dtype == MG2D_C64)  return launch_rb2<float>(ctx, out, in, in_lo2, in_hi2, U, U_lo2, U_hi, F, F_lo, F_hi, r, r_lo, r_hi, mass, tm, mu, Lx, Ly, yoff, link, st, name);
    snprintf(ctx->err, sizeof(ctx->err), "%s: bad dtype", name);
    return MG2D_EINVAL;
}

}  // namespace

extern "C" int mg2d_wilson_relax_rb2(mg2d_ctx* ctx, void* out, const void* in, const void* in_lo2, const void* in_hi2,
                                     const void* U, const void* U_lo2, const void* U_hi, const void* r, const void* r_lo,
                                     const void* r_hi, double mass, int Lx, int Ly, int yoff, int dtype,
                                     const mg2d_halo_link* link, void* stream) {
    return wilson_relax_rb2(ctx, out, in, in_lo2, in_hi2, U, U_lo2, U_hi, nullptr, nullptr, nullptr, r, r_lo, r_hi, mass, false, 0.0,
                            Lx, Ly, yoff, dtype, link, stream, "mg2d_wilson_relax_rb2");
}

extern "C" int mg2d_wilson_sw_relax_rb2(mg2d_ctx* ctx, void* out, const void* in, const void* in_lo2, const void* in_hi2,
                                        const void* U, const void* U_lo2, const void* U_hi, const void* F, const void* F_lo,
                                        const void* F_hi, const void* r, const void* r_lo, const void* r_hi, double mass, int Lx,
                                        int Ly, int yoff, int dtype, const mg2d_halo_link* link, void* stream) {
    if (ctx && (!F || !F_lo || !F_hi)) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_wilson_sw_relax_rb2: F, F_lo and F_hi are required");
    return wilson_relax_rb2(ctx, out, in, in_lo2, in_hi2, U, U_lo2, U_hi, F, F_lo, F_hi, r, r_lo, r_hi, mass, false, 0.0, Lx, Ly,
                            yoff, dtype, link, stream, "mg2d_wilson_sw_relax_rb2");
}

extern "C" int mg2d_wilson_tm_relax_rb2(mg2d_ctx* ctx, void* out, const void* in, const void* in_lo2, const void* in_hi2,
                                        const void* U, const void* U_lo2, const void* U_hi, const void* F, const void* F_lo,
                                        const void* F_hi, const void* r, const void* r_lo, const void* r_hi, double mass,
                                        double mu, int Lx, int Ly, int yoff, int dtype, const mg2d_halo_link* link, void* stream) {
    if (ctx && F && (!F_lo || !F_hi)) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_wilson_tm_relax_rb2: F needs F_lo and F_hi");
    if (ctx && !std::isfinite(mu)) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_wilson_tm_relax_rb2: mu is not finite");
    return wilson_relax_rb2(ctx, out, in, in_lo2, in_hi2, U, U_lo2, U_hi, F, F_lo, F_hi, r, r_lo, r_hi, mass, true, mu, Lx, Ly,
                            yoff, dtype, link, stream, "mg2d_wilson_tm_relax_rb2");
}
