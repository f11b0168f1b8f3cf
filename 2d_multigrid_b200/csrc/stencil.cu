// stencil.cu -- generic 5-point block stencil with n x n complex blocks per site and slot.
//
// Replaces, for every level whose operator is stored (all coarse levels; level 0 in reference-compat mode):
//   Level::f_apply_D   S6/level.h:251-265     v'(s) = D1 v(s+x) + D2 v(s-x) + D3 v(s+y) + D4 v(s-y) + D0 v(s)
//   Level::f_residue   S6/level.h:61-77       r' = r - D phi           (+ norms of f_get_residue_mag :79-98)
//   Level::f_relax     S6/level.h:100-128     phi(s) = -D0(s)^-1 (sum_{k>=1} D_k phi(s+d_k) - r(s))
//                                             gs_flag=0 Jacobi ; gs_flag=1 lexicographic GS (x outer, y inner)
//
// Layout: D[s][k][j][i] (column-major blocks).  A group of G lanes owns one site and streams its 5*n*n
// elements with stride G (element e = g + G*t), so a warp always reads 32 consecutive 16-byte elements:
// lane g keeps row i = g % n and column-part jp = g / n; partial sums are combined with log2(G/n) butterfly
// shuffles.  Algorithmic traffic per site (c128): apply (5n^2+2n)*16 B, relax (5n^2+3n)*16 B (+n^2*16 D0inv).
#include "common.cuh"
#include <cooperative_groups.h>
#include <cuda_fp16.h>
namespace cg = cooperative_groups;

namespace {

template <int N> struct GroupOf { static constexpr int G = (N == 1) ? 1 : (N == 2) ? 4 : (N == 4) ? 16 : 32; };

// neighbour row pointer + site for slot k (1..4) of site (x,y) of an Lx x Ly strip with halo rows lo/hi
template <typename C>
__device__ __forceinline__ const C* nbr_ptr(const C* in, const C* lo, const C* hi, int k, int x, int y, int Lx, int Ly, int N) {
    switch (k) {
        case 0: return in + ((size_t)y * Lx + x) * N;
        case 1: return in + ((size_t)y * Lx + ((x + 1 == Lx) ? 0 : x + 1)) * N;
        case 2: return in + ((size_t)y * Lx + ((x == 0) ? Lx - 1 : x - 1)) * N;
        case 3: return (y + 1 == Ly) ? hi + (size_t)x * N : in + ((size_t)(y + 1) * Lx + x) * N;
        default: return (y == 0) ? lo + (size_t)x * N : in + ((size_t)(y - 1) * Lx + x) * N;
    }
}

// sum_{k=K0..4} D_k(s) v(s+d_k), row i of the result valid in every lane of the group.
// LD selects the load used for the field (ldcg for in-place Gauss-Seidel, ldg otherwise).
template <typename T, int N, int G, int K0, bool COHERENT>
__device__ __forceinline__ cplx<T> stencil_row(const cplx<T>* __restrict__ Ds, const cplx<T>* in, const cplx<T>* lo,
                                               const cplx<T>* hi, int x, int y, int Lx, int Ly, int g) {
    using C = cplx<T>;
    constexpr int JP = G / N;                 // column parts per group
    constexpr int ITERS = (5 * N) / JP;       // (k,j) pairs per lane
    constexpr int T0 = (K0 * N) / JP;
    const int jp = g / N;
    C acc = mk<T>(0, 0);
#pragma unroll
    for (int t = T0; t < ITERS; ++t) {
        const int k = (JP * t) / N;                 // compile-time after unrolling (jp < JP, JP | N)
        const int j = jp + (JP * t) % N;
        const C d = __ldg(Ds + g + G * t);
        const C* p = nbr_ptr<C>(in, lo, hi, k, x, y, Lx, Ly, N) + j;
        C v;
        if (COHERENT) { v = __ldcg(p); } else { v = __ldg(p); }
        cfma(acc, d, v);
    }
#pragma unroll
    for (int m = N; m < G; m <<= 1) acc = cadd(acc, shfl_xor_c(acc, m));
    return acc;
}

// out_i = - sum_j Dinv[j*N+i] w_j, w distributed one row per lane (lane i of the group holds w_i)
template <typename T, int N, int G>
__device__ __forceinline__ cplx<T> apply_minus_inv(const cplx<T>* __restrict__ Dinv_s, cplx<T> w, int g) {
    using C = cplx<T>;
    constexpr int JP = G / N;
    const int i = g % N, jp = g / N;
    C acc = mk<T>(0, 0);
#pragma unroll
    for (int u = 0; u < N / JP + (N % JP ? 1 : 0); ++u) {
        const int j = jp + JP * u;
        C wj = shfl_c(w, (j < N) ? j : 0, G);
        if (j < N) { const C d = __ldg(Dinv_s + j * N + i); cfma(acc, d, wj); }
    }
#pragma unroll
    for (int m = N; m < G; m <<= 1) acc = cadd(acc, shfl_xor_c(acc, m));
    acc.x = -acc.x; acc.y = -acc.y;
    return acc;
}

constexpr int ST_THREADS = 256;

// MODE 0 apply, 1 residual, 2 Jacobi sweep
template <typename T, int N, int MODE, bool DOTS>
__global__ void __launch_bounds__(ST_THREADS)
stencil_kernel(cplx<T>* __restrict__ out, const cplx<T>* __restrict__ in, const cplx<T>* __restrict__ in_lo,
               const cplx<T>* __restrict__ in_hi, const cplx<T>* __restrict__ D, const cplx<T>* __restrict__ Dinv,
               const cplx<T>* __restrict__ b, int Lx, int Ly, long long vstride, long long hstride,
               double* __restrict__ partials, unsigned int* __restrict__ counter, double* __restrict__ dots, XComm* xc) {
    using C = cplx<T>;
    constexpr int G = GroupOf<N>::G;
    constexpr int GPB = ST_THREADS / G;
    const int g = threadIdx.x % G, grp = threadIdx.x / G;
    const int i = g % N, jp = g / N;
    const int v = blockIdx.y;
    out += (size_t)v * vstride; in += (size_t)v * vstride;
    in_lo += (size_t)v * hstride; in_hi += (size_t)v * hstride;
    if (b) b += (size_t)v * vstride;
    const long long S = (long long)Lx * Ly;
    double red[4] = {0.0, 0.0, 0.0, 0.0};
    const long long nsteps = (S + GPB - 1) / GPB;
    for (long long step = blockIdx.x; step < nsteps; step += gridDim.x) {
        long long s = step * GPB + grp;
        const bool active = s < S;
        if (!active) s = S - 1;
        const int y = (int)(s / Lx), x = (int)(s - (long long)y * Lx);
        const C* Ds = D + (size_t)s * 5 * N * N;
        C o;
        if (MODE == 2) {
            C acc = stencil_row<T, N, G, 1, false>(Ds, in, in_lo, in_hi, x, y, Lx, Ly, g);
            if (b) acc = csub(acc, __ldg(b + (size_t)s * N + i));
            o = apply_minus_inv<T, N, G>(Dinv + (size_t)s * N * N, acc, g);
        } else {
            o = stencil_row<T, N, G, 0, false>(Ds, in, in_lo, in_hi, x, y, Lx, Ly, g);
            if (MODE == 1) {
                const C bb = __ldg(b + (size_t)s * N + i);
                if (DOTS && active && jp == 0) red[3] += (double)bb.x * bb.x + (double)bb.y * bb.y;
                o = csub(bb, o);
            }
        }
        if (active && jp == 0) {
            out[(size_t)s * N + i] = o;
            if (DOTS) {
                const C vi = __ldg(in + (size_t)s * N + i);
                red[0] += (double)o.x * o.x + (double)o.y * o.y;
                red[1] += (double)o.x * vi.x + (double)o.y * vi.y;
                red[2] += (double)o.x * vi.y - (double)o.y * vi.x;
            }
        }
    }
    if (DOTS) grid_reduce<4, ST_THREADS>(red, partials + (size_t)v * MG2D_MAX_PARTIALS * 4, counter + v,
                                         dots + 4 * v, blockIdx.x, gridDim.x, xc);
}

// red-black Gauss-Seidel half sweep: sites with (x + y + yoff) % 2 == colour are updated in place from the
// other colour (f_relax's update rule in the two-colour ordering).  Lx must be even.
template <typename T, int N>
__global__ void __launch_bounds__(ST_THREADS)
stencil_rb_kernel(cplx<T>* phi, const cplx<T>* lo, const cplx<T>* hi, const cplx<T>* __restrict__ D,
                  const cplx<T>* __restrict__ Dinv, const cplx<T>* __restrict__ r, int Lx, int Ly, int colour, int yoff,
                  long long vstride, long long hstride) {
    using C = cplx<T>;
    constexpr int G = GroupOf<N>::G;
    constexpr int GPB = ST_THREADS / G;
    const int g = threadIdx.x % G, grp = threadIdx.x / G;
    const int i = g % N, jp = g / N;
    const int v = blockIdx.y;
    phi += (size_t)v * vstride; lo += (size_t)v * hstride; hi += (size_t)v * hstride;
    if (r) r += (size_t)v * vstride;
    const int Lh = Lx / 2;
    const long long S2 = (long long)Lh * Ly;
    const long long nsteps = (S2 + GPB - 1) / GPB;
    for (long long step = blockIdx.x; step < nsteps; step += gridDim.x) {
        long long h = step * GPB + grp;
        const bool active = h < S2;
        if (!active) h = S2 - 1;
        const int y = (int)(h / Lh);
        const int x = 2 * (int)(h - (long long)y * Lh) + ((y + yoff + colour) & 1);
        const size_t s = (size_t)y * Lx + x;
        C acc = stencil_row<T, N, G, 1, true>(D + s * 5 * N * N, phi, lo, hi, x, y, Lx, Ly, g);
        if (r) acc = csub(acc, __ldg(r + s * N + i));
        C o = apply_minus_inv<T, N, G>(Dinv + s * N * N, acc, g);
        if (active && jp == 0) phi[s * N + i] = o;
    }
}

// Batched red-black half sweep: NV vectors per pass share one stream of the operator blocks (near-null generation
// relaxes nc/2 vectors with the same operator, S6/level.h:224-233; with blockIdx.y = vector the 16x16-block operator
// would be re-streamed once per vector).  blockIdx.y selects the batch of NV vectors.
template <typename T, int N, int NV>
__global__ void __launch_bounds__(ST_THREADS)
stencil_rb_batch_kernel(cplx<T>* phi, const cplx<T>* lo, const cplx<T>* hi, const cplx<T>* __restrict__ D,
                        const cplx<T>* __restrict__ Dinv, const cplx<T>* __restrict__ r, int Lx, int Ly, int colour, int yoff,
                        long long vstride, long long hstride) {
    using C = cplx<T>;
    constexpr int G = GroupOf<N>::G;
    constexpr int GPB = ST_THREADS / G;
    constexpr int JP = G / N;
    constexpr int ITERS = (5 * N) / JP, T0 = N / JP;
    const int g = threadIdx.x % G, grp = threadIdx.x / G;
    const int i = g % N, jp = g / N;
    const size_t v0 = (size_t)blockIdx.y * NV;
    phi += v0 * vstride; lo += v0 * hstride; hi += v0 * hstride;
    if (r) r += v0 * vstride;
    const int Lh = Lx / 2;
    const long long S2 = (long long)Lh * Ly;
    const long long nsteps = (S2 + GPB - 1) / GPB;
    for (long long step = blockIdx.x; step < nsteps; step += gridDim.x) {
        long long h = step * GPB + grp;
        const bool active = h < S2;
        if (!active) h = S2 - 1;
        const int y = (int)(h / Lh);
        const int x = 2 * (int)(h - (long long)y * Lh) + ((y + yoff + colour) & 1);
        const size_t s = (size_t)y * Lx + x;
        const C* Ds = D + s * 5 * N * N;
        C acc[NV];
#pragma unroll
        for (int v = 0; v < NV; ++v) acc[v] = mk<T>(0, 0);
#pragma unroll
        for (int t = T0; t < ITERS; ++t) {
            const int k = (JP * t) / N;
            const int j = jp + (JP * t) % N;
            const C d = __ldg(Ds + g + G * t);
            const bool in_hi = (k == 3 && y + 1 == Ly), in_lo = (k == 4 && y == 0);
            const C* p = nbr_ptr<C>(phi, lo, hi, k, x, y, Lx, Ly, N) + j;
            const long long st = (in_hi || in_lo) ? hstride : vstride;
#pragma unroll
            for (int v = 0; v < NV; ++v) cfma(acc[v], d, __ldcg(p + (size_t)v * st));
        }
#pragma unroll
        for (int v = 0; v < NV; ++v) {
#pragma unroll
            for (int m = N; m < G; m <<= 1) acc[v] = cadd(acc[v], shfl_xor_c(acc[v], m));
            if (r) acc[v] = csub(acc[v], __ldg(r + (size_t)v * vstride + s * N + i));
        }
        C out[NV];
#pragma unroll
        for (int v = 0; v < NV; ++v) out[v] = mk<T>(0, 0);
        const C* Is = Dinv + s * N * N;
#pragma unroll
        for (int u = 0; u < N / JP; ++u) {
            const int j = jp + JP * u;
            const C d = __ldg(Is + j * N + i);
#pragma unroll
            for (int v = 0; v < NV; ++v) cfma(out[v], d, shfl_c(acc[v], j, G));
        }
#pragma unroll
        for (int v = 0; v < NV; ++v) {
#pragma unroll
            for (int m = N; m < G; m <<= 1) out[v] = cadd(out[v], shfl_xor_c(out[v], m));
            if (active && jp == 0) phi[(size_t)v * vstride + s * N + i] = mk<T>(-out[v].x, -out[v].y);
        }
    }
}

// Red-black half sweep on PRE-MULTIPLIED hopping blocks  M_k(s) = -D0(s)^-1 D_k(s), k = 1..4  (layout M[s][k-1][j][i]):
//     phi(s) <- sum_k M_k(s) phi(s+d_k) + c(s),   c(s) = D0(s)^-1 r(s)
// which is f_relax's update (S6/level.h:116-121) with the inverse folded into the blocks: 4 n x n blocks per updated
// site instead of 5 (the level-1 sweep of the bench sits at the HBM roofline, so only fewer bytes make it faster),
// and no second dependent mat-vec phase (shorter critical path on the small, latency-bound levels).
// CMODE 0: r = 0 (near-null relaxation); 1: first sweep of a relax call, c = D0^-1 r is computed here and stored in
// cbuf; 2: c read from cbuf.  NV vectors per pass share one stream of the blocks (blockIdx.y = batch of NV).
// LINK (strips): boundary rows are processed FIRST; before its first step on them a CTA waits for the neighbours' halo rows
// (flags >= local epoch), every updated boundary value is also stored into the neighbour's halo buffer over NVLink, and
// the last boundary CTA to finish publishes epoch + 1 (see mg2d_halo_link in include/mg2d.h) while the interior streams.
template <typename T, int N, int NV, int CMODE, bool LINK>
__global__ void __launch_bounds__(ST_THREADS)
stencil_rb_pm_kernel(cplx<T>* phi, const cplx<T>* lo, const cplx<T>* hi, const cplx<T>* __restrict__ M,
                     const cplx<T>* __restrict__ Dinv, const cplx<T>* __restrict__ r, cplx<T>* cbuf, int Lx, int Ly,
                     int colour, int yoff, long long vstride, long long hstride, HaloLinkDev link) {
    using C = cplx<T>;
    constexpr int G = GroupOf<N>::G;
    constexpr int GPB = ST_THREADS / G;
    constexpr int JP = G / N;
    constexpr int ITERS = (4 * N) / JP;
    const int g = threadIdx.x % G, grp = threadIdx.x / G;
    const int i = g % N, jp = g / N;
    const size_t v0 = (size_t)blockIdx.y * NV;
    phi += v0 * vstride; lo += v0 * hstride; hi += v0 * hstride;
    if (CMODE == 1) r += v0 * vstride;
    if (CMODE != 0) cbuf += v0 * vstride;
    C* push_lo = nullptr; C* push_hi = nullptr;     // neighbours' buffers: next's lo halo <- my last row, prev's hi halo <- my row 0
    __shared__ unsigned long long s_epoch;
    bool waited = false;                            // this CTA works on boundary rows: it has read the epoch (and waited)
    bool ticketed = false;                          // ... and has reported the end of its boundary work
    if (LINK) {
        // (no epoch read here: a dependent load + barrier in front of every CTA's first loads costs ~20 % of a half sweep when
        // each CTA lives for one step; only the CTAs that reach the boundary rows need the epoch)
        if (link.push_next_lo) { push_lo = (C*)link.push_next_lo + v0 * hstride; push_hi = (C*)link.push_prev_hi + v0 * hstride; }
    }
    const int Lh = Lx / 2;
    const long long S2 = (long long)Lh * Ly;
    const long long nsteps = (S2 + GPB - 1) / GPB;
    // strips: the two boundary rows come FIRST (row order 0, Ly-1, 1, 2, .., Ly-2): their CTAs wait for the neighbours' rows of
    // the previous launch (published early in that launch for the same reason), push what they produce and publish the new
    // epoch while the interior of this launch is still streaming -- neither the fence + flag round trips at the end of the
    // boundary work nor the neighbours' wait sit on the critical path
    const long long nb_half = (long long)(Ly >= 2 ? 2 : 1) * Lh;                     // half-row sites of the boundary rows
    for (long long step = blockIdx.x; step < nsteps; step += gridDim.x) {
        long long h = step * GPB + grp;
        const bool active = h < S2;
        if (!active) h = S2 - 1;
        int y = (int)(h / Lh);
        const int xh = (int)(h - (long long)y * Lh);
        if (LINK) {
            y = (y == 0) ? 0 : (y == 1 ? Ly - 1 : y - 1);                          // rows 0, Ly-1, then 1 .. Ly-2
            if (!waited && step * GPB < nb_half) {                                   // CTA-uniform: first boundary step
                if (threadIdx.x == 0) {
                    const unsigned long long e = link.mine->epoch;      // advanced only after every boundary CTA has taken its ticket
                    s_epoch = e;
                    if ((link.wait & 1) && !(spin_until(&link.mine->flag_lo, e) && spin_until(&link.mine->flag_hi, e)))
                        atomicExch(&link.mine->error, 1ull);
                }
                __syncthreads();
                waited = true;
            }
        }
        const int x = 2 * xh + ((y + yoff + colour) & 1);
        const size_t s = (size_t)y * Lx + x;
        const C* Ms = M + s * 4 * N * N;
        C acc[NV];
#pragma unroll
        for (int v = 0; v < NV; ++v) acc[v] = mk<T>(0, 0);
        // The loads are issued in explicit batches of CH block elements + their field values before any of them is consumed:
        // left to itself the compiler interleaves load / FMA pairs to save registers, and an in-order warp then has only 2-5
        // loads in flight (ncu, round 2: the sweep then depends on occupancy and loses 20-40 % on small strips).
        // (halo rows are peer-written: ld.cg reads them from L2, the coherence point of NVLink-incoming stores; no
        // inline-asm loads here -- their compiler barrier would serialise the independent loads)
        constexpr int CH = (ITERS < 8 / NV) ? ITERS : ((8 / NV) < 2 ? 2 : 8 / NV);
        static_assert(ITERS % CH == 0, "chunking");
#pragma unroll
        for (int t0 = 0; t0 < ITERS; t0 += CH) {
            C d[CH], pv[CH][NV];
#pragma unroll
            for (int u = 0; u < CH; ++u) {
                const int t = t0 + u;
                const int k = 1 + (JP * t) / N;
                const int j = jp + (JP * t) % N;
                d[u] = __ldg(Ms + g + G * t);
                const bool in_hi = (k == 3 && y + 1 == Ly), in_lo = (k == 4 && y == 0);
                const C* p = nbr_ptr<C>(phi, lo, hi, k, x, y, Lx, Ly, N) + j;
                const long long st = (in_hi || in_lo) ? hstride : vstride;
#pragma unroll
                for (int v = 0; v < NV; ++v) pv[u][v] = __ldcg(p + (size_t)v * st);
            }
            if constexpr (NV == 1 && CH == 8) {
                C (&pf)[CH] = *reinterpret_cast<C(*)[CH]>(&pv[0][0]);
                keep_all(d); keep_all(pf);
            }
#pragma unroll
            for (int u = 0; u < CH; ++u)
#pragma unroll
                for (int v = 0; v < NV; ++v) cfma(acc[v], d[u], pv[u][v]);
        }
#pragma unroll
        for (int v = 0; v < NV; ++v) {
#pragma unroll
            for (int m = N; m < G; m <<= 1) acc[v] = cadd(acc[v], shfl_xor_c(acc[v], m));
            if (CMODE == 1) {
                const C w = __ldg(r + (size_t)v * vstride + s * N + i);
                const C c = apply_minus_inv<T, N, G>(Dinv + s * N * N, w, g);       // = -D0^-1 r
                acc[v] = csub(acc[v], c);
                if (active && jp == 0) cbuf[(size_t)v * vstride + s * N + i] = mk<T>(-c.x, -c.y);
            } else if (CMODE == 2) {
                acc[v] = cadd(acc[v], __ldg(cbuf + (size_t)v * vstride + s * N + i));
            }
            if (active && jp == 0) {
                phi[(size_t)v * vstride + s * N + i] = acc[v];
                if (LINK && push_lo) {
                    if (y == 0) push_hi[(size_t)v * hstride + (size_t)x * N + i] = acc[v];
                    if (y + 1 == Ly) push_lo[(size_t)v * hstride + (size_t)x * N + i] = acc[v];
                }
            }
        }
        if (LINK && push_lo && waited && !ticketed && (step + gridDim.x) * GPB >= nb_half) {
            // this CTA's last boundary step is done: only the CTAs that worked on boundary rows have peer stores in flight and
            // only they are counted (the neighbours read nothing else of this launch); the last of them publishes
            ticketed = true;
            __threadfence_system();
            __syncthreads();
            if (threadIdx.x == 0) {
                const long long nbs = (nb_half + GPB - 1) / GPB;             // steps that touch the boundary rows
                const unsigned long long nbound = (unsigned long long)(nbs < (long long)gridDim.x ? nbs : (long long)gridDim.x) * gridDim.y;
                const unsigned long long t = atomicAdd(&link.mine->ticket, 1ull);
                if (t == nbound - 1ull) {
                    __threadfence_system();
                    link.mine->ticket = 0ull;
                    publish2(&link.next->flag_lo, &link.prev->flag_hi, s_epoch + 1ull, link.relaxed);
                    link.mine->epoch = s_epoch + 1ull;
                }
            }
        }
    }
}

// ALL sweeps of one relax call on a small level in ONE cooperative launch: the half sweeps are separated by grid-wide
// barriers instead of kernel boundaries.  On the levels that fit in L2 (<= a few thousand sites of 16x16 blocks) a half
// sweep is a ~10 us launch that moves a few MB: pure latency, 16 of them per level and cycle, and on strips every rank pays
// it in full because these levels are replicated.  Whole periodic lattice on this GPU, one vector.
template <typename T, int N>
__global__ void __launch_bounds__(ST_THREADS)
stencil_rb_pm_sweeps_kernel(cplx<T>* phi, const cplx<T>* __restrict__ M, const cplx<T>* __restrict__ Dinv,
                            const cplx<T>* __restrict__ r, cplx<T>* cbuf, int L, int nsweeps) {
    using C = cplx<T>;
    constexpr int G = GroupOf<N>::G;
    constexpr int GPB = ST_THREADS / G;
    constexpr int JP = G / N;
    constexpr int ITERS = (4 * N) / JP;
    cg::grid_group grid = cg::this_grid();
    const int g = threadIdx.x % G, grp = threadIdx.x / G;
    const int i = g % N, jp = g / N;
    const int Lh = L / 2;
    const long long S2 = (long long)Lh * L;
    const long long nsteps = (S2 + GPB - 1) / GPB;
    const C* lo = phi + (size_t)(L - 1) * L * N;
    for (int it = 0; it < nsweeps; ++it) {
        for (int colour = 0; colour < 2; ++colour) {
            for (long long step = blockIdx.x; step < nsteps; step += gridDim.x) {
                long long h = step * GPB + grp;
                const bool active = h < S2;
                if (!active) h = S2 - 1;
                const int y = (int)(h / Lh);
                const int x = 2 * (int)(h - (long long)y * Lh) + ((y + colour) & 1);
                const size_t s = (size_t)y * L + x;
                const C* Ms = M + s * 4 * N * N;
                C acc = mk<T>(0, 0);
                // latency-bound (a few CTAs, L2-resident operator): every load of a batch is in flight before the first FMA
                constexpr int CH = ITERS < 16 ? ITERS : 16;
#pragma unroll
                for (int t0 = 0; t0 < ITERS; t0 += CH) {
                    C d[CH], pv[CH];
#pragma unroll
                    for (int u = 0; u < CH; ++u) {
                        const int t = t0 + u;
                        const int k = 1 + (JP * t) / N;
                        const int j = jp + (JP * t) % N;
                        d[u] = __ldg(Ms + g + G * t);
                        pv[u] = __ldcg(nbr_ptr<C>(phi, lo, phi, k, x, y, L, L, N) + j);
                    }
                    keep_all(d); keep_all(pv);
#pragma unroll
                    for (int u = 0; u < CH; ++u) cfma(acc, d[u], pv[u]);
                }
#pragma unroll
                for (int m = N; m < G; m <<= 1) acc = cadd(acc, shfl_xor_c(acc, m));
                if (r) {
                    if (it == 0) {
                        const C c = apply_minus_inv<T, N, G>(Dinv + s * N * N, __ldg(r + s * N + i), g);     // = -D0^-1 r
                        acc = csub(acc, c);
                        if (active && jp == 0) cbuf[s * N + i] = mk<T>(-c.x, -c.y);
                    } else {
                        acc = cadd(acc, __ldcg(cbuf + s * N + i));
                    }
                }
                if (active && jp == 0) phi[s * N + i] = acc;
            }
            grid.sync();
        }
    }
}

// ---- low-rank hopping blocks ------------------------------------------------------------------------------------
// On the first coarse level the hopping block towards direction k is a sum over the R = block fine links that cross the
// aggregate face, and each fine hopping term has rank one (the spin projector (1 -+ sigma_mu)/2 of the Wilson operator,
// S6/level.h:155-172; a scalar for the Laplacian): D_k(X) = sum_b a_b b_b^dagger has rank <= R, and so has the
// pre-multiplied block M_k = -D0^-1 D_k = sum_b (-D0^-1 a_b) b_b^dagger.  For R < N/2 the factors are fewer bytes than the
// block: 2*4*R*N numbers per site instead of 4*N*N -- half for the 16-dof level over 4x4 aggregates, the level whose
// sweep dominates the cycle and already runs at the HBM roofline.
//     t_q  = sum_j conj(b_q)_j phi(s+d_k(q))_j          q = (k-1)*R + b   (stage 1: Q = 4R dot products of length N)
//     phi(s)_i <- sum_q ma_q,i t_q + c(s)_i             ma_q = -D0^-1 a_q (stage 2)
// One warp per site.  Storage per site: [Bc: IT x 32][MA: IT x 32] complex, IT = N*R/8, already in lane order:
//     Bc[t][g] = conj(b_q)_j   with q = g / LP, j = (g % LP)*IT + t,  LP = 32/Q lanes share one dot product
//     MA[t][g] = ma_q,i        with i = g % N,  q = t*H + g / N,      H = 32/N pair classes
// so every load is 32 consecutive elements.  (built by mg2d_lowrank_pack from the factors of mg2d_hop_factors)
template <int N, int R> struct LowRank {
    static constexpr int Q = 4 * R, IT = N * R / 8, LP = 32 / Q, H = 32 / N, SITE = 64 * IT;
    static_assert(Q <= 32 && (32 % Q) == 0 && (32 % N) == 0 && N >= 8 && (N * R) % 8 == 0 && LP * IT == N, "unsupported (N, R)");
};

// NV vectors per pass share one stream of the factors (blockIdx.y = batch of NV; near-null generation).
template <typename T, int N, int R, int NV, int CMODE, bool LINK>
__global__ void __launch_bounds__(ST_THREADS)
stencil_rb_lr_kernel(cplx<T>* phi, const cplx<T>* lo, const cplx<T>* hi, const cplx<T>* __restrict__ F,
                     const cplx<T>* __restrict__ Dinv, const cplx<T>* __restrict__ r, cplx<T>* cbuf, int Lx, int Ly,
                     int colour, int yoff, long long vstride, long long hstride, HaloLinkDev link) {
    using C = cplx<T>;
    using LR = LowRank<N, R>;
    constexpr int G = 32, GPB = ST_THREADS / G, IT = LR::IT;
    __shared__ C s_t[GPB][NV][LR::Q];
    const int g = threadIdx.x % G, grp = threadIdx.x / G;
    const int i = g % N;
    const int q1 = g / LR::LP, k1 = 1 + q1 / R, j0 = (g % LR::LP) * IT;
    const size_t v0 = (size_t)blockIdx.y * NV;
    phi += v0 * vstride; lo += v0 * hstride; hi += v0 * hstride;
    if (CMODE == 1) r += v0 * vstride;
    if (CMODE != 0) cbuf += v0 * vstride;
    C* push_lo = nullptr; C* push_hi = nullptr;
    __shared__ unsigned long long s_epoch;
    bool waited = false;                            // this CTA works on boundary rows (see stencil_rb_pm_kernel)
    bool ticketed = false;
    if (LINK) {
        if (link.push_next_lo) { push_lo = (C*)link.push_next_lo + v0 * hstride; push_hi = (C*)link.push_prev_hi + v0 * hstride; }
    }
    const int Lh = Lx / 2;
    const long long S2 = (long long)Lh * Ly;
    const long long nsteps = (S2 + GPB - 1) / GPB;
    // strips: the two boundary rows come FIRST (row order 0, Ly-1, 1, 2, .., Ly-2): their CTAs wait for the neighbours' rows of
    // the previous launch (published early in that launch for the same reason), push what they produce and publish the new
    // epoch while the interior of this launch is still streaming -- neither the fence + flag round trips at the end of the
    // boundary work nor the neighbours' wait sit on the critical path
    const long long nb_half = (long long)(Ly >= 2 ? 2 : 1) * Lh;                     // half-row sites of the boundary rows
    for (long long step = blockIdx.x; step < nsteps; step += gridDim.x) {
        long long h = step * GPB + grp;
        const bool active = h < S2;
        if (!active) h = S2 - 1;
        int y = (int)(h / Lh);
        const int xh = (int)(h - (long long)y * Lh);
        if (LINK) {
            y = (y == 0) ? 0 : (y == 1 ? Ly - 1 : y - 1);                          // rows 0, Ly-1, then 1 .. Ly-2
            if (!waited && step * GPB < nb_half) {                                   // CTA-uniform: first boundary step
                if (threadIdx.x == 0) {
                    const unsigned long long e = link.mine->epoch;      // advanced only after every boundary CTA has taken its ticket
                    s_epoch = e;
                    if (link.wait && !(spin_until(&link.mine->flag_lo, e) && spin_until(&link.mine->flag_hi, e)))
                        atomicExch(&link.mine->error, 1ull);
                }
                __syncthreads();
                waited = true;
            }
        }
        const int x = 2 * xh + ((y + yoff + colour) & 1);
        const size_t s = (size_t)y * Lx + x;
        const C* Fs = F + s * LR::SITE;
        C bc[IT], ma[IT];
#pragma unroll
        for (int t = 0; t < IT; ++t) bc[t] = __ldg(Fs + 32 * t + g);
#pragma unroll
        for (int t = 0; t < IT; ++t) ma[t] = __ldg(Fs + 32 * IT + 32 * t + g);
        const C* pn = nbr_ptr<C>(phi, lo, hi, k1, x, y, Lx, Ly, N) + j0;
        const bool halo_row = (k1 == 3 && y + 1 == Ly) || (k1 == 4 && y == 0);
        const long long st = halo_row ? hstride : vstride;
#pragma unroll
        for (int v = 0; v < NV; ++v) {
            C tq = mk<T>(0, 0);
#pragma unroll
            for (int t = 0; t < IT; ++t) cfma(tq, bc[t], __ldcg(pn + (size_t)v * st + t));
#pragma unroll
            for (int m = 1; m < LR::LP; m <<= 1) tq = cadd(tq, shfl_xor_c(tq, m));
            if ((g % LR::LP) == 0) s_t[grp][v][q1] = tq;
        }
        __syncwarp();
#pragma unroll
        for (int v = 0; v < NV; ++v) {
            C acc = mk<T>(0, 0);
#pragma unroll
            for (int t = 0; t < IT; ++t) cfma(acc, ma[t], s_t[grp][v][t * LR::H + g / N]);
#pragma unroll
            for (int m = N; m < G; m <<= 1) acc = cadd(acc, shfl_xor_c(acc, m));
            if (CMODE == 1) {
                const C w = __ldg(r + (size_t)v * vstride + s * N + i);
                const C c = apply_minus_inv<T, N, G>(Dinv + s * N * N, w, g);       // = -D0^-1 r
                acc = csub(acc, c);
                if (active && g < N) cbuf[(size_t)v * vstride + s * N + i] = mk<T>(-c.x, -c.y);
            } else if (CMODE == 2) {
                acc = cadd(acc, __ldg(cbuf + (size_t)v * vstride + s * N + i));
            }
            if (active && g < N) {
                phi[(size_t)v * vstride + s * N + i] = acc;
                if (LINK && push_lo) {
                    if (y == 0) push_hi[(size_t)v * hstride + (size_t)x * N + i] = acc;
                    if (y + 1 == Ly) push_lo[(size_t)v * hstride + (size_t)x * N + i] = acc;
                }
            }
        }
        __syncwarp();
        if (LINK && push_lo && waited && !ticketed && (step + gridDim.x) * GPB >= nb_half) {       // (see stencil_rb_pm_kernel)
            ticketed = true;
            __threadfence_system();
            __syncthreads();
            if (threadIdx.x == 0) {
                const long long nbs = (nb_half + GPB - 1) / GPB;
                const unsigned long long nbound = (unsigned long long)(nbs < (long long)gridDim.x ? nbs : (long long)gridDim.x) * gridDim.y;
                const unsigned long long t = atomicAdd(&link.mine->ticket, 1ull);
                if (t == nbound - 1ull) {
                    __threadfence_system();
                    link.mine->ticket = 0ull;
                    publish2(&link.next->flag_lo, &link.prev->flag_hi, s_epoch + 1ull, link.relaxed);
                    link.mine->epoch = s_epoch + 1ull;
                }
            }
        }
    }
}

// Factors of the hopping blocks of the first coarse level (see above).  One warp per coarse site; for pair q = (k-1)*R + b
// the fine link (s -> s' = s + d_k) crossing face k at boundary position b has the hopping block D_k(s) = a v^dagger
// (rank one: a = the column of largest norm, v^dagger = a^dagger D / |a|^2, checked to 1e-13 -> status bit 4 otherwise);
//     A[X][q][i] = sum_j P(s)[i][j] a_j ,   B[X][q][i] = sum_j P(s')[i][j] v_j     =>  D_k(X) = sum_b A_q B_q^dagger
template <typename T>
__global__ void __launch_bounds__(256)
hop_factors_kernel(cplx<T>* __restrict__ A, cplx<T>* __restrict__ B, const cplx<T>* __restrict__ Df,
                   const cplx<T>* __restrict__ P, const cplx<T>* __restrict__ P_lo, const cplx<T>* __restrict__ P_hi,
                   int nf, int nc, int Lxf, int Lyf, int blk, int* status) {
    using C = cplx<T>;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const int Lxc = Lxf / blk, Lyc = Lyf / blk;
    const long long nagg = (long long)Lxc * Lyc;
    const int Q = 4 * blk, E = nf * nc;
    for (long long X = (long long)blockIdx.x * wpb + warp; X < nagg; X += (long long)gridDim.x * wpb) {
        const int yc = (int)(X / Lxc), xc = (int)(X - (long long)yc * Lxc);
        for (int q = 0; q < Q; ++q) {
            const int k = 1 + q / blk, b = q % blk;
            // boundary site of face k: x1 = blk-1 (k=1), 0 (k=2), y1 = blk-1 (k=3), 0 (k=4); b runs along the face
            const int x1 = (k == 1) ? blk - 1 : (k == 2) ? 0 : b;
            const int y1 = (k == 3) ? blk - 1 : (k == 4) ? 0 : b;
            const int xf = blk * xc + x1, yf = blk * yc + y1;
            const size_t s = (size_t)yf * Lxf + xf;
            const C* Ps = P + s * E;
            const C* Pn;
            if (k == 1) Pn = P + ((size_t)yf * Lxf + (xf + 1 == Lxf ? 0 : xf + 1)) * E;
            else if (k == 2) Pn = P + ((size_t)yf * Lxf + (xf == 0 ? Lxf - 1 : xf - 1)) * E;
            else if (k == 3) Pn = (yf + 1 == Lyf) ? P_hi + (size_t)xf * E : P + ((size_t)(yf + 1) * Lxf + xf) * E;
            else Pn = (yf == 0) ? P_lo + (size_t)xf * E : P + ((size_t)(yf - 1) * Lxf + xf) * E;
            const C* Dk = Df + (s * 5 + k) * nf * nf;          // Dk[j*nf + i] = D(i,j)
            // column of largest norm (every lane computes the same small thing; nf <= 2)
            int jbest = 0; double best = -1.0;
            for (int j = 0; j < nf; ++j) {
                double n2 = 0.0;
                for (int ii = 0; ii < nf; ++ii) { const C d = Dk[j * nf + ii]; n2 += (double)d.x * d.x + (double)d.y * d.y; }
                if (n2 > best) { best = n2; jbest = j; }
            }
            C a[2], v[2];
            for (int ii = 0; ii < nf; ++ii) a[ii] = Dk[jbest * nf + ii];
            double err = 0.0, tot = 0.0;
            for (int j = 0; j < nf; ++j) {
                C w = mk<T>(0, 0);                               // a^dagger D[:, j]
                for (int ii = 0; ii < nf; ++ii) cfmac(w, a[ii], Dk[j * nf + ii]);
                if (best > 0.0) { w.x = (T)(w.x / best); w.y = (T)(w.y / best); }
                v[j] = cconj(w);                                 // D(i,j) = a_i conj(v_j)
                for (int ii = 0; ii < nf; ++ii) {
                    const C d = Dk[j * nf + ii];
                    const C rec = cmul(a[ii], w);
                    err += (double)(d.x - rec.x) * (d.x - rec.x) + (double)(d.y - rec.y) * (d.y - rec.y);
                    tot += (double)d.x * d.x + (double)d.y * d.y;
                }
            }
            if (lane == 0 && status && err > 1e-26 * tot) atomicOr(status, 4);
            for (int ic = lane; ic < nc; ic += 32) {
                C sa = mk<T>(0, 0), sb = mk<T>(0, 0);
                for (int j = 0; j < nf; ++j) { cfma(sa, Ps[ic * nf + j], a[j]); cfma(sb, Pn[ic * nf + j], v[j]); }
                A[((size_t)X * Q + q) * nc + ic] = sa;
                B[((size_t)X * Q + q) * nc + ic] = sb;
            }
        }
    }
}

// F (lane-ordered factors for stencil_rb_lr_kernel) from A, B and D0^-1:  ma_q = -D0^-1 a_q,  Bc = conj(B).
// WITH_B = false rewrites only the -D0^-1 A half (B unread), with the same operations as the full pack.
template <typename T, int N, int R, bool WITH_B = true>
__global__ void __launch_bounds__(256)
lowrank_pack_kernel(cplx<T>* __restrict__ F, const cplx<T>* __restrict__ A, const cplx<T>* __restrict__ B,
                    const cplx<T>* __restrict__ Dinv, long long S) {
    using C = cplx<T>;
    using LR = LowRank<N, R>;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    for (long long s = (long long)blockIdx.x * wpb + warp; s < S; s += (long long)gridDim.x * wpb) {
        const C* As = A + (size_t)s * LR::Q * N;
        const C* Bs = B + (size_t)s * LR::Q * N;
        const C* inv = Dinv + (size_t)s * N * N;
        C* Fs = F + (size_t)s * LR::SITE;
        for (int t = 0; t < LR::IT; ++t) {
            if (WITH_B) {
                const int q = lane / LR::LP, j = (lane % LR::LP) * LR::IT + t;
                Fs[32 * t + lane] = cconj(Bs[q * N + j]);
            }
            const int i = lane % N, q2 = t * LR::H + lane / N;
            C acc = mk<T>(0, 0);
            for (int l = 0; l < N; ++l) cfma(acc, inv[l * N + i], As[q2 * N + l]);
            Fs[32 * LR::IT + 32 * t + lane] = mk<T>(-acc.x, -acc.y);
        }
    }
}

// M[s][k-1] = -D0inv[s] D[s][k], k = 1..4 (column-major blocks).  One CTA walks over sites; the site's D0^-1 and
// the four hopping blocks are staged in shared memory.
template <typename T, int N>
__global__ void __launch_bounds__(256)
premultiply_kernel(cplx<T>* __restrict__ M, const cplx<T>* __restrict__ D, const cplx<T>* __restrict__ Dinv, long long S) {
    using C = cplx<T>;
    __shared__ C s_inv[N * N];
    __shared__ C s_d[4 * N * N];
    for (long long s = blockIdx.x; s < S; s += gridDim.x) {
        for (int e = threadIdx.x; e < N * N; e += blockDim.x) s_inv[e] = __ldg(Dinv + (size_t)s * N * N + e);
        for (int e = threadIdx.x; e < 4 * N * N; e += blockDim.x) s_d[e] = __ldg(D + (size_t)s * 5 * N * N + N * N + e);
        __syncthreads();
        for (int e = threadIdx.x; e < 4 * N * N; e += blockDim.x) {
            const int k = e / (N * N), j = (e / N) % N, i = e % N;
            C a = mk<T>(0, 0);
#pragma unroll 4
            for (int l = 0; l < N; ++l) cfma(a, s_inv[l * N + i], s_d[k * N * N + j * N + l]);
            M[(size_t)s * 4 * N * N + e] = mk<T>(-a.x, -a.y);
        }
        __syncthreads();
    }
}

// Red-black half sweep for the complex64 preconditioner hierarchy with the operator blocks stored in HALF precision
// (`__half2` = (re,im), same [s][k][j][i] order; arithmetic and fields stay fp32).  The stored operator is the dominant
// HBM traffic of a cycle (4 hop blocks + D0inv per updated site), so halving its bytes again is the remaining lever once the
// fp32 kernel sits at the roofline.  One warp per site; every lane loads 16 bytes = 4 consecutive rows i of one column j,
// keeps 4 accumulators, partial sums meet in log2(128/N) butterfly steps; the intermediate vector goes through 128 B of
// shared memory for the D0inv product.  N in {8, 16, 32}.
template <int N>
__global__ void __launch_bounds__(ST_THREADS)
stencil_rb_h_kernel(float2* phi, const float2* lo, const float2* hi, const __half2* __restrict__ Dh,
                    const __half2* __restrict__ Dinvh, const float2* __restrict__ r, int Lx, int Ly, int colour, int yoff) {
    constexpr int WPB = ST_THREADS / 32;
    constexpr int HOP_CHUNKS = 4 * N * N / 4, INV_CHUNKS = N * N / 4;      // 16-byte chunks (4 elements) per site
    constexpr int KJ_STEP = 128 / N;                                        // (k,j) advance per 32-lane step
    __shared__ float2 s_w[WPB][N];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int i0 = (4 * lane) % N, kj0 = (4 * lane) / N;
    const int Lh = Lx / 2;
    const long long S2 = (long long)Lh * Ly;
    for (long long h = (long long)blockIdx.x * WPB + warp; h < S2; h += (long long)gridDim.x * WPB) {
        const int y = (int)(h / Lh);
        const int x = 2 * (int)(h - (long long)y * Lh) + ((y + yoff + colour) & 1);
        const size_t s = (size_t)y * Lx + x;
        const uint4* Hs = reinterpret_cast<const uint4*>(Dh + s * 5 * N * N + N * N);   // hop blocks k = 1..4
        float2 acc[4] = {{0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}};
#pragma unroll
        for (int t = 0; t < HOP_CHUNKS / 32; ++t) {
            const int kj = kj0 + KJ_STEP * t;
            const int k = 1 + kj / N, j = kj % N;
            const uint4 raw = __ldg(Hs + lane + 32 * t);
            const float2 v = __ldcg(nbr_ptr<float2>(phi, lo, hi, k, x, y, Lx, Ly, N) + j);
            const __half2* hp = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
            for (int q = 0; q < 4; ++q) cfma(acc[q], __half22float2(hp[q]), v);
        }
#pragma unroll
        for (int m = N / 4; m < 32; m <<= 1)
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[q] = cadd(acc[q], shfl_xor_c(acc[q], m));
        if (lane < N / 4) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                float2 w = acc[q];
                if (r) w = csub(w, __ldg(r + s * N + i0 + q));
                s_w[warp][i0 + q] = w;
            }
        }
        __syncwarp();
        const uint4* Is = reinterpret_cast<const uint4*>(Dinvh + s * N * N);
        float2 out[4] = {{0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}};
#pragma unroll
        for (int t = 0; t < (INV_CHUNKS + 31) / 32; ++t) {
            const int c = lane + 32 * t;
            if (c < INV_CHUNKS) {
                const int j = kj0 + KJ_STEP * t;
                const uint4 raw = __ldg(Is + c);
                const float2 wj = s_w[warp][j];
                const __half2* hp = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
                for (int q = 0; q < 4; ++q) cfma(out[q], __half22float2(hp[q]), wj);
            }
        }
#pragma unroll
        for (int m = N / 4; m < 32; m <<= 1)
#pragma unroll
            for (int q = 0; q < 4; ++q) out[q] = cadd(out[q], shfl_xor_c(out[q], m));
        if (lane < N / 4) {
            float4* dst = reinterpret_cast<float4*>(phi + s * N + i0);
            dst[0] = make_float4(-out[0].x, -out[0].y, -out[1].x, -out[1].y);
            dst[1] = make_float4(-out[2].x, -out[2].y, -out[3].x, -out[3].y);
        }
        __syncwarp();
    }
}

// (re,im) fp32 pairs -> __half2, elementwise (builds the half-precision copy of D / D0inv)
__global__ void to_half_kernel(__half2* __restrict__ dst, const float2* __restrict__ src, long long n) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
        dst[e] = __float22half2_rn(__ldg(src + e));
}

// lexicographic Gauss-Seidel by anti-diagonal wavefronts (cooperative launch, grid.sync between fronts)
template <typename T, int N>
__global__ void __launch_bounds__(ST_THREADS)
gs_wavefront_kernel(cplx<T>* phi, const cplx<T>* __restrict__ D, const cplx<T>* __restrict__ Dinv,
                    const cplx<T>* __restrict__ r, int L, int num_iter, int nvec, long long vstride) {
    using C = cplx<T>;
    constexpr int G = GroupOf<N>::G;
    constexpr int GPB = ST_THREADS / G;
    cg::grid_group grid = cg::this_grid();
    const int g = threadIdx.x % G, grp = threadIdx.x / G;
    const int i = g % N, jp = g / N;
    const long long ngroups = (long long)gridDim.x * GPB;
    const long long gid = (long long)blockIdx.x * GPB + grp;
    for (int it = 0; it < num_iter; ++it) {
        for (int c = 0; c <= 2 * L - 2; ++c) {
            const int x0 = max(0, c - L + 1), x1 = min(c, L - 1);
            const int cnt = x1 - x0 + 1;
            const long long total = (long long)cnt * nvec;
            const long long rounds = (total + ngroups - 1) / ngroups;
            for (long long rd = 0; rd < rounds; ++rd) {
                long long idx = rd * ngroups + gid;
                const bool active = idx < total;
                if (!active) idx = total - 1;
                const int v = (int)(idx / cnt);
                const int x = x0 + (int)(idx - (long long)v * cnt), y = c - x;
                const size_t s = (size_t)y * L + x;
                C* ph = phi + (size_t)v * vstride;
                C acc = stencil_row<T, N, G, 1, true>(D + s * 5 * N * N, ph, ph + (size_t)(L - 1) * L * N, ph,
                                                      x, y, L, L, g);
                if (r) acc = csub(acc, __ldg(r + (size_t)v * vstride + s * N + i));
                C o = apply_minus_inv<T, N, G>(Dinv + s * N * N, acc, g);
                if (active && jp == 0) __stcg(ph + s * N + i, o);
            }
            grid.sync();
        }
    }
}

// The same sweep on a STRIP of rows [y0, y0+Ly) of the global L x Lg lattice (multi-GPU): the anti-diagonal fronts x + y = c are
// global, every rank updates the part of front c that lies in its rows.  What a front needs from the neighbours
// (lexicographic order, x outer / y inner, S6/level.h:104-123):
//   * first local row reads phi(x, y0-1): the value the previous rank produced on front c-1 (NEW), except on rank 0 where it is
//     the periodic wrap row Lg-1, still OLD when column x starts -> `lo` halo, filled by an exchange before the sweep, and on
//     ranks > 0 overwritten entry by entry by the previous rank as it goes;
//   * last local row reads phi(x, y0+Ly): OLD (the next rank updates it one front later, in ITS memory) -> `hi` halo from the
//     exchange; except on the last rank, where it is row 0 of rank 0, already NEW -> rank 0 stores its row-0 results into the
//     last rank's `hi` halo.
// Progress is published through a dedicated halo slot: flag_lo = 1 + last front whose last-row value the previous rank has
// delivered, flag_hi = 1 + last column rank 0 has delivered (both offset by the sweep count, slot epoch * 4L); a front is
// entered only when the value it needs has arrived.  One sweep per launch (the caller exchanges OLD rows in between).
// Latency-bound by construction (2L-1 dependent fronts + a flag hop per front): parity mode, like the single-GPU kernel.
struct GsStripLinks {
    HaloSlot* mine; HaloSlot* next; HaloSlot* last;     // the GS progress slots (mine, next rank's, last rank's)
    void* push_next_lo;                                 // next rank's lo halo (NULL on the last rank)
    void* push_last_hi;                                 // last rank's hi halo (non-NULL on rank 0 only)
    int first, is_last;
};

template <typename T, int N>
__global__ void __launch_bounds__(ST_THREADS)
gs_wavefront_strip_kernel(cplx<T>* phi, const cplx<T>* lo, const cplx<T>* hi, const cplx<T>* __restrict__ D,
                          const cplx<T>* __restrict__ Dinv, const cplx<T>* __restrict__ r, int L, int Ly, int y0, int Lg,
                          GsStripLinks a) {
    using C = cplx<T>;
    constexpr int G = GroupOf<N>::G;
    constexpr int GPB = ST_THREADS / G;
    cg::grid_group grid = cg::this_grid();
    const int g = threadIdx.x % G, grp = threadIdx.x / G;
    const int i = g % N, jp = g / N;
    const long long ngroups = (long long)gridDim.x * GPB;
    const long long gid = (long long)blockIdx.x * GPB + grp;
    __shared__ unsigned long long s_base;
    __shared__ int s_ok;
    if (threadIdx.x == 0) { s_base = a.mine->epoch * 4ull * (unsigned long long)(L + Lg); s_ok = 1; }
    __syncthreads();
    const unsigned long long base = s_base;
    C* push_lo = (C*)a.push_next_lo;
    C* push_hi = (C*)a.push_last_hi;
    for (int c = y0; c <= y0 + Ly - 1 + L - 1; ++c) {
        const int x0 = max(0, c - (y0 + Ly - 1)), x1 = min(c - y0, L - 1);     // my sites of front c: x in [x0, x1], y = c - x
        const int cnt = x1 - x0 + 1;
        const bool has_first = (c - y0 <= L - 1);              // site (c - y0, y0) exists
        const bool has_last = (c - (y0 + Ly - 1) >= 0);        // site (c - (y0+Ly-1), y0+Ly-1) exists
        if (threadIdx.x == 0) {
            bool ok = true;
            if (has_first && !a.first) ok = spin_until(&a.mine->flag_lo, base + (unsigned long long)c);
            if (ok && has_last && a.is_last)       // (one rank: it is its own "rank 0" and has delivered column x on front x)
                ok = spin_until(&a.mine->flag_hi, base + (unsigned long long)(c - (y0 + Ly - 1)) + 1ull);
            if (!ok) { s_ok = 0; atomicExch(&a.mine->error, 1ull); }
        }
        __syncthreads();
        const long long rounds = (cnt + ngroups - 1) / ngroups;
        for (long long rd = 0; rd < rounds; ++rd) {
            long long idx = rd * ngroups + gid;
            const bool active = idx < cnt;
            if (!active) idx = cnt - 1;
            const int x = x0 + (int)idx, yl = c - x - y0;                      // local row
            const size_t s = (size_t)yl * L + x;
            C acc = stencil_row<T, N, G, 1, true>(D + s * 5 * N * N, phi, lo, hi, x, yl, L, Ly, g);
            if (r) acc = csub(acc, __ldg(r + s * N + i));
            C o = apply_minus_inv<T, N, G>(Dinv + s * N * N, acc, g);
            if (active && jp == 0) {
                __stcg(phi + s * N + i, o);
                if (push_lo && yl == Ly - 1) push_lo[(size_t)x * N + i] = o;
                if (push_hi && yl == 0) push_hi[(size_t)x * N + i] = o;
            }
            if ((push_lo && yl == Ly - 1) || (push_hi && yl == 0)) __threadfence_system();
        }
        grid.sync();
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            __threadfence_system();
            if (push_lo && has_last) st_relaxed_sys(&a.next->flag_lo, base + (unsigned long long)c + 1ull);
            if (push_hi && has_first) st_relaxed_sys(&a.last->flag_hi, base + (unsigned long long)c + 1ull);   // y0 = 0: c = column
        }
    }
    grid.sync();
    if (blockIdx.x == 0 && threadIdx.x == 0) a.mine->epoch = a.mine->epoch + 1ull;
}

// D0inv[s] = inverse(D[s][0]); one warp per site, Gauss-Jordan with partial pivoting in shared memory
template <typename T, int N>
__global__ void block_inverse_kernel(cplx<T>* __restrict__ Dinv, const cplx<T>* __restrict__ D, long long S) {
    using C = cplx<T>;
    extern __shared__ unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    C* A = reinterpret_cast<C*>(smem_raw) + (size_t)warp * 2 * N * N;   // A[i][j] row-major
    C* B = A + N * N;
    for (long long s = (long long)blockIdx.x * nwarps + warp; s < S; s += (long long)gridDim.x * nwarps) {
        const C* src = D + (size_t)s * 5 * N * N;
        for (int e = lane; e < N * N; e += 32) {
            const int j = e / N, i = e - j * N;
            A[i * N + j] = src[e];
            B[i * N + j] = mk<T>(i == j ? (T)1 : (T)0, (T)0);
        }
        __syncwarp();
        for (int c = 0; c < N; ++c) {
            // pivot: largest |A[r][c]|, r >= c (ties -> smallest r)
            T best = (T)-1; int br = c;
            for (int r = c + lane; r < N; r += 32) {
                const C a = A[r * N + c];
                const T m = a.x * a.x + a.y * a.y;
                if (m > best) { best = m; br = r; }
            }
#pragma unroll
            for (int m = 16; m > 0; m >>= 1) {
                const T ob = __shfl_xor_sync(0xffffffffu, best, m);
                const int orr = __shfl_xor_sync(0xffffffffu, br, m);
                if (ob > best || (ob == best && orr < br)) { best = ob; br = orr; }
            }
            if (br != c) {
                for (int j = lane; j < N; j += 32) {
                    C t = A[c * N + j]; A[c * N + j] = A[br * N + j]; A[br * N + j] = t;
                    t = B[c * N + j]; B[c * N + j] = B[br * N + j]; B[br * N + j] = t;
                }
            }
            __syncwarp();
            const C pv = A[c * N + c];
            const T den = pv.x * pv.x + pv.y * pv.y;
            const C pinv = mk<T>(pv.x / den, -pv.y / den);
            __syncwarp();
            for (int j = lane; j < N; j += 32) {
                A[c * N + j] = cmul(A[c * N + j], pinv);
                B[c * N + j] = cmul(B[c * N + j], pinv);
            }
            __syncwarp();
            for (int rr = 0; rr < N; ++rr) {
                if (rr == c) continue;
                const C f = A[rr * N + c];
                __syncwarp();
                for (int j = lane; j < N; j += 32) {
                    C a = A[rr * N + j]; C t = cmul(f, A[c * N + j]); A[rr * N + j] = csub(a, t);
                    C bb = B[rr * N + j]; t = cmul(f, B[c * N + j]); B[rr * N + j] = csub(bb, t);
                }
                __syncwarp();
            }
        }
        C* dst = Dinv + (size_t)s * N * N;
        for (int e = lane; e < N * N; e += 32) {
            const int j = e / N, i = e - j * N;
            dst[e] = B[i * N + j];
        }
        __syncwarp();
    }
}

template <typename T, int N>
int launch_stencil(mg2d_ctx* ctx, void* out, const void* in, const void* lo, const void* hi, const void* D,
                   const void* Dinv, const void* b, int Lx, int Ly, int mode, int nvec, long long vstride,
                   long long hstride, double* dots, cudaStream_t st) {
    using C = cplx<T>;
    constexpr int GPB = ST_THREADS / GroupOf<N>::G;
    const long long S = (long long)Lx * Ly;
    long long nsteps = (S + GPB - 1) / GPB;
    int gx = (int)(nsteps < MG2D_MAX_PARTIALS ? nsteps : MG2D_MAX_PARTIALS);
    dim3 grid(gx, nvec);
#define SL(MODE, DOTS)                                                                                         \
    stencil_kernel<T, N, MODE, DOTS><<<grid, ST_THREADS, 0, st>>>((C*)out, (const C*)in, (const C*)lo, (const C*)hi, \
        (const C*)D, (const C*)Dinv, (const C*)b, Lx, Ly, vstride, hstride, ctx->partials, ctx->counter, dots, (ctx->xreduce && nvec == 1) ? ctx->xcomm : nullptr)
    if (mode == 0) { if (dots) SL(0, true); else SL(0, false); }
    else if (mode == 1) { if (dots) SL(1, true); else SL(1, false); }
    else SL(2, false);
#undef SL
    return mg2d_check_launch(ctx, "mg2d_stencil");
}

template <typename T>
int dispatch_stencil(mg2d_ctx* ctx, int n, void* out, const void* in, const void* lo, const void* hi, const void* D,
                     const void* Dinv, const void* b, int Lx, int Ly, int mode, int nvec, long long vstride,
                     long long hstride, double* dots, cudaStream_t st) {
    switch (n) {
#define CASE(N) case N: return launch_stencil<T, N>(ctx, out, in, lo, hi, D, Dinv, b, Lx, Ly, mode, nvec, vstride, hstride, dots, st)
        CASE(1); CASE(2); CASE(4); CASE(8); CASE(16); CASE(32);
#undef CASE
        default: return mg2d_fail(ctx, MG2D_EUNSUPPORTED, "mg2d_stencil: n_dof must be one of 1,2,4,8,16,32");
    }
}

template <typename T, int N>
int launch_gs(mg2d_ctx* ctx, void* phi, const void* D, const void* Dinv, const void* r, int L, int num_iter,
              int nvec, long long vstride, cudaStream_t st) {
    using C = cplx<T>;
    constexpr int GPB = ST_THREADS / GroupOf<N>::G;
    int per_sm = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, gs_wavefront_kernel<T, N>, ST_THREADS, 0);
    if (e != cudaSuccess || per_sm < 1) return mg2d_fail(ctx, MG2D_ECUDA, "mg2d_relax_gs: occupancy query failed");
    long long need = ((long long)L * nvec + GPB - 1) / GPB;
    long long cap = (long long)per_sm * ctx->num_sms;
    int grid = (int)(need < cap ? need : cap);
    if (grid < 1) grid = 1;
    C* phi_ = (C*)phi; const C* D_ = (const C*)D; const C* Dinv_ = (const C*)Dinv; const C* r_ = (const C*)r;
    void* args[] = {&phi_, &D_, &Dinv_, &r_, &L, &num_iter, &nvec, &vstride};
    e = cudaLaunchCooperativeKernel((const void*)gs_wavefront_kernel<T, N>, dim3(grid), dim3(ST_THREADS), args, 0, st);
    if (e != cudaSuccess) { snprintf(ctx->err, sizeof(ctx->err), "mg2d_relax_gs: %s", cudaGetErrorString(e)); return MG2D_ECUDA; }
    return mg2d_check_launch(ctx, "mg2d_relax_gs");
}

template <typename T, int N>
int launch_gs_strip(mg2d_ctx* ctx, void* phi, const void* lo, const void* hi, const void* D, const void* Dinv, const void* r,
                    int L, int Ly, int y0, int Lg, GsStripLinks a, cudaStream_t st) {
    using C = cplx<T>;
    constexpr int GPB = ST_THREADS / GroupOf<N>::G;
    int per_sm = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, gs_wavefront_strip_kernel<T, N>, ST_THREADS, 0);
    if (e != cudaSuccess || per_sm < 1) return mg2d_fail(ctx, MG2D_ECUDA, "mg2d_relax_gs_strip: occupancy query failed");
    const int front = L < Ly ? L : Ly;
    long long need = ((long long)front + GPB - 1) / GPB;
    long long cap = (long long)per_sm * ctx->num_sms;
    int grid = (int)(need < cap ? need : cap);
    if (grid < 1) grid = 1;
    C* phi_ = (C*)phi; const C* lo_ = (const C*)lo; const C* hi_ = (const C*)hi; const C* D_ = (const C*)D;
    const C* Dinv_ = (const C*)Dinv; const C* r_ = (const C*)r;
    void* args[] = {&phi_, &lo_, &hi_, &D_, &Dinv_, &r_, &L, &Ly, &y0, &Lg, &a};
    e = cudaLaunchCooperativeKernel((const void*)gs_wavefront_strip_kernel<T, N>, dim3(grid), dim3(ST_THREADS), args, 0, st);
    if (e != cudaSuccess) { snprintf(ctx->err, sizeof(ctx->err), "mg2d_relax_gs_strip: %s", cudaGetErrorString(e)); return MG2D_ECUDA; }
    return mg2d_check_launch(ctx, "mg2d_relax_gs_strip");
}

template <typename T>
int dispatch_gs(mg2d_ctx* ctx, int n, void* phi, const void* D, const void* Dinv, const void* r, int L, int num_iter,
                int nvec, long long vstride, cudaStream_t st) {
    switch (n) {
#define CASE(N) case N: return launch_gs<T, N>(ctx, phi, D, Dinv, r, L, num_iter, nvec, vstride, st)
        CASE(1); CASE(2); CASE(4); CASE(8); CASE(16); CASE(32);
#undef CASE
        default: return mg2d_fail(ctx, MG2D_EUNSUPPORTED, "mg2d_relax_gs: n_dof must be one of 1,2,4,8,16,32");
    }
}

template <typename T, int N>
int launch_rb(mg2d_ctx* ctx, void* phi, const void* lo, const void* hi, const void* D, const void* Dinv, const void* r,
              int Lx, int Ly, int colour, int yoff, int nvec, long long vstride, long long hstride, cudaStream_t st) {
    using C = cplx<T>;
    constexpr int GPB = ST_THREADS / GroupOf<N>::G;
    const long long S2 = (long long)(Lx / 2) * Ly;
    long long nsteps = (S2 + GPB - 1) / GPB;
    long long cap = (long long)ctx->num_sms * 32;
    if (N >= 4 && nvec % 4 == 0) {     // stream the operator once per 4 vectors
        dim3 gridb((int)(nsteps < cap ? nsteps : cap), nvec / 4);
        stencil_rb_batch_kernel<T, N, 4><<<gridb, ST_THREADS, 0, st>>>((C*)phi, (const C*)lo, (const C*)hi, (const C*)D, (const C*)Dinv,
                                                                     (const C*)r, Lx, Ly, colour, yoff, vstride, hstride);
        return mg2d_check_launch(ctx, "mg2d_relax_rb");
    }
    dim3 grid((int)(nsteps < cap ? nsteps : cap), nvec);
    stencil_rb_kernel<T, N><<<grid, ST_THREADS, 0, st>>>((C*)phi, (const C*)lo, (const C*)hi, (const C*)D, (const C*)Dinv,
                                                      (const C*)r, Lx, Ly, colour, yoff, vstride, hstride);
    return mg2d_check_launch(ctx, "mg2d_relax_rb");
}

template <typename T>
int dispatch_rb(mg2d_ctx* ctx, int n, void* phi, const void* lo, const void* hi, const void* D, const void* Dinv,
                const void* r, int Lx, int Ly, int colour, int yoff, int nvec, long long vstride, long long hstride,
                cudaStream_t st) {
    switch (n) {
#define CASE(N) case N: return launch_rb<T, N>(ctx, phi, lo, hi, D, Dinv, r, Lx, Ly, colour, yoff, nvec, vstride, hstride, st)
        CASE(1); CASE(2); CASE(4); CASE(8); CASE(16); CASE(32);
#undef CASE
        default: return mg2d_fail(ctx, MG2D_EUNSUPPORTED, "mg2d_relax_rb: n_dof must be one of 1,2,4,8,16,32");
    }
}

inline HaloLinkDev make_link(const mg2d_halo_link* l) {
    HaloLinkDev d;
    memset(&d, 0, sizeof(d));
    if (l) {
        d.mine = (HaloSlot*)l->slot_mine; d.prev = (HaloSlot*)l->slot_prev; d.next = (HaloSlot*)l->slot_next;
        d.push_next_lo = l->push_next_lo; d.push_prev_hi = l->push_prev_hi; d.wait = l->wait; d.relaxed = mg2d_publish_relaxed();
    }
    return d;
}

template <typename T, int N>
int launch_rb_pm(mg2d_ctx* ctx, void* phi, const void* lo, const void* hi, const void* M, const void* Dinv, const void* r,
                 void* cbuf, int cmode, int Lx, int Ly, int colour, int yoff, int nvec, long long vstride, long long hstride,
                 const mg2d_halo_link* link, cudaStream_t st) {
    using C = cplx<T>;
    constexpr int GPB = ST_THREADS / GroupOf<N>::G;
    const long long S2 = (long long)(Lx / 2) * Ly;
    long long nsteps = (S2 + GPB - 1) / GPB;
    long long cap = (long long)ctx->num_sms * 32;
    const int gx = (int)(nsteps < cap ? nsteps : cap);
    const HaloLinkDev ld = make_link(link);
    // resident CTAs per SM are capped at 5 through (unused) dynamic shared memory.  Measured on B200 (tools/link_probe.py, 16-dof
    // blocks): a halo-linked half sweep on a 256 x 32 strip takes 18.2 us with 5 CTAs of 256 threads per SM and 20.4 us with the 6
    // the register count would allow; whole-lattice sweeps do not care (15.0 us / 92 us either way).  MG2D_PM_CTAS overrides.
    // (Also measured and rejected: programmatic dependent launch for this kernel -- -0.5 us on a whole lattice, +2 us on strips.)
    static int pm_ctas = -1;
    if (pm_ctas < 0) { const char* e = getenv("MG2D_PM_CTAS"); pm_ctas = e ? atoi(e) : 5; if (pm_ctas < 1 || pm_ctas > 8) pm_ctas = 5; }
    const size_t dsm = (N >= 8) ? (size_t)(200 * 1024 / pm_ctas / 1024) * 1024 - 2048 : 0;     // <= 48 KB for >= 5 CTAs (no attribute needed)
#define PM(NV, CM, LK) (dsm > 48 * 1024 ? (void)cudaFuncSetAttribute(stencil_rb_pm_kernel<T, N, NV, CM, LK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dsm) : (void)0), \
    stencil_rb_pm_kernel<T, N, NV, CM, LK><<<dim3(gx, nvec / NV), ST_THREADS, dsm, st>>>((C*)phi, (const C*)lo, (const C*)hi, \
        (const C*)M, (const C*)Dinv, (const C*)r, (C*)cbuf, Lx, Ly, colour, yoff, vstride, hstride, ld)
#define PMC(NV, LK) do { if (cmode == 0) PM(NV, 0, LK); else if (cmode == 1) PM(NV, 1, LK); else PM(NV, 2, LK); } while (0)
    if (N >= 4 && nvec % 4 == 0) { if (link) PMC(4, true); else PMC(4, false); }
    else                         { if (link) PMC(1, true); else PMC(1, false); }
#undef PMC
#undef PM
    return mg2d_check_launch(ctx, "mg2d_relax_rb_pm");
}

template <typename T>
int dispatch_rb_pm(mg2d_ctx* ctx, int n, void* phi, const void* lo, const void* hi, const void* M, const void* Dinv,
                   const void* r, void* cbuf, int cmode, int Lx, int Ly, int colour, int yoff, int nvec, long long vstride,
                   long long hstride, const mg2d_halo_link* link, cudaStream_t st) {
    switch (n) {
#define CASE(N) case N: return launch_rb_pm<T, N>(ctx, phi, lo, hi, M, Dinv, r, cbuf, cmode, Lx, Ly, colour, yoff, nvec, vstride, hstride, link, st)
        CASE(1); CASE(2); CASE(4); CASE(8); CASE(16); CASE(32);
#undef CASE
        default: return mg2d_fail(ctx, MG2D_EUNSUPPORTED, "mg2d_relax_rb_pm: n_dof must be one of 1,2,4,8,16,32");
    }
}

template <typename T, int N>
int launch_rb_pm_sweeps(mg2d_ctx* ctx, void* phi, const void* M, const void* Dinv, const void* r, void* cbuf, int L, int nsweeps,
                        cudaStream_t st) {
    using C = cplx<T>;
    constexpr int GPB = ST_THREADS / GroupOf<N>::G;
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, stencil_rb_pm_sweeps_kernel<T, N>, ST_THREADS, 0) != cudaSuccess || per_sm < 1)
        return mg2d_fail(ctx, MG2D_ECUDA, "mg2d_relax_rb_pm_sweeps: occupancy query failed");
    const long long nsteps = ((long long)(L / 2) * L + GPB - 1) / GPB;
    long long cap = (long long)(per_sm < 2 ? per_sm : 2) * ctx->num_sms;        // a small grid keeps the barrier cheap
    int grid = (int)(nsteps < cap ? nsteps : cap);
    C* phi_ = (C*)phi; const C* M_ = (const C*)M; const C* Dinv_ = (const C*)Dinv; const C* r_ = (const C*)r; C* cbuf_ = (C*)cbuf;
    void* args[] = {&phi_, &M_, &Dinv_, &r_, &cbuf_, &L, &nsweeps};
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(ST_THREADS); cfg.dynamicSmemBytes = 0; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelExC(&cfg, (const void*)stencil_rb_pm_sweeps_kernel<T, N>, args);
    if (e != cudaSuccess) { snprintf(ctx->err, sizeof(ctx->err), "mg2d_relax_rb_pm_sweeps: %s", cudaGetErrorString(e)); cudaGetLastError(); return MG2D_ECUDA; }
    return mg2d_check_launch(ctx, "mg2d_relax_rb_pm_sweeps");
}

template <typename T>
int dispatch_rb_pm_sweeps(mg2d_ctx* ctx, int n, void* phi, const void* M, const void* Dinv, const void* r, void* cbuf, int L,
                          int nsweeps, cudaStream_t st) {
    switch (n) {
#define CASE(N) case N: return launch_rb_pm_sweeps<T, N>(ctx, phi, M, Dinv, r, cbuf, L, nsweeps, st)
        CASE(1); CASE(2); CASE(4); CASE(8); CASE(16);
#undef CASE
        default: return mg2d_fail(ctx, MG2D_EUNSUPPORTED, "mg2d_relax_rb_pm_sweeps: n_dof must be one of 1,2,4,8,16");
    }
}

template <typename T, int N, int R>
int launch_rb_lr(mg2d_ctx* ctx, void* phi, const void* lo, const void* hi, const void* F, const void* Dinv, const void* r,
                 void* cbuf, int cmode, int Lx, int Ly, int colour, int yoff, int nvec, long long vstride, long long hstride,
                 const mg2d_halo_link* link, cudaStream_t st) {
    using C = cplx<T>;
    constexpr int GPB = ST_THREADS / 32;
    const long long S2 = (long long)(Lx / 2) * Ly;
    long long nsteps = (S2 + GPB - 1) / GPB;
    long long cap = (long long)ctx->num_sms * 32;
    const int gx = (int)(nsteps < cap ? nsteps : cap);
    const HaloLinkDev ld = make_link(link);
#define LRK(NV, CM, LK) stencil_rb_lr_kernel<T, N, R, NV, CM, LK><<<dim3(gx, nvec / NV), ST_THREADS, 0, st>>>((C*)phi, (const C*)lo, (const C*)hi, \
        (const C*)F, (const C*)Dinv, (const C*)r, (C*)cbuf, Lx, Ly, colour, yoff, vstride, hstride, ld)
#define LRC(NV, LK) do { if (cmode == 0) LRK(NV, 0, LK); else if (cmode == 1) LRK(NV, 1, LK); else LRK(NV, 2, LK); } while (0)
    if (nvec % 4 == 0) { if (link) LRC(4, true); else LRC(4, false); }
    else               { if (link) LRC(1, true); else LRC(1, false); }
#undef LRC
#undef LRK
    return mg2d_check_launch(ctx, "mg2d_relax_rb_lr");
}

template <typename T>
int dispatch_premul(mg2d_ctx* ctx, int n, void* M, const void* D, const void* Dinv, long long S, cudaStream_t st) {
    using C = cplx<T>;
    long long nb = S; if (nb > (long long)ctx->num_sms * 16) nb = (long long)ctx->num_sms * 16;
    switch (n) {
#define CASE(N) case N: premultiply_kernel<T, N><<<(int)nb, 256, 0, st>>>((C*)M, (const C*)D, (const C*)Dinv, S); break
        CASE(1); CASE(2); CASE(4); CASE(8); CASE(16);
#undef CASE
        default: return mg2d_fail(ctx, MG2D_EUNSUPPORTED, "mg2d_premultiply: n_dof must be one of 1,2,4,8,16");
    }
    return mg2d_check_launch(ctx, "mg2d_premultiply");
}

template <typename T, int N>
int launch_inverse(mg2d_ctx* ctx, void* Dinv, const void* D, long long S, cudaStream_t st) {
    using C = cplx<T>;
    const size_t per_warp = 2 * (size_t)N * N * sizeof(C);
    int warps = (int)(48 * 1024 / per_warp); if (warps > 8) warps = 8; if (warps < 1) warps = 1;
    long long nb = (S + warps - 1) / warps; if (nb > ctx->num_sms * 16) nb = ctx->num_sms * 16;
    block_inverse_kernel<T, N><<<(int)nb, warps * 32, warps * per_warp, st>>>((C*)Dinv, (const C*)D, S);
    return mg2d_check_launch(ctx, "mg2d_block_inverse");
}

template <typename T>
int dispatch_inverse(mg2d_ctx* ctx, int n, void* Dinv, const void* D, long long S, cudaStream_t st) {
    switch (n) {
#define CASE(N) case N: return launch_inverse<T, N>(ctx, Dinv, D, S, st)
        CASE(1); CASE(2); CASE(4); CASE(8); CASE(16); CASE(32);
#undef CASE
        default: return mg2d_fail(ctx, MG2D_EUNSUPPORTED, "mg2d_block_inverse: n_dof must be one of 1,2,4,8,16,32");
    }
}

}  // namespace

extern "C" int mg2d_stencil_apply(mg2d_ctx* ctx, void* out, const void* in, const void* in_lo, const void* in_hi,
                                  const void* D, const void* b, int n, int Lx, int Ly, int mode, int dtype,
                                  int nvec, long long vstride, long long hstride, double* dots, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!out || !in || !in_lo || !in_hi || !D || Lx < 1 || Ly < 1 || nvec < 1 || nvec > 64)
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_stencil_apply: bad argument");
    if (mode != MG2D_MODE_APPLY && mode != MG2D_MODE_RESID) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_stencil_apply: bad mode");
    if (mode == MG2D_MODE_RESID && !b) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_stencil_apply: MODE_RESID needs b");
    if (out == in) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_stencil_apply: out must not alias in");
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MG2D_C128) return dispatch_stencil<double>(ctx, n, out, in, in_lo, in_hi, D, nullptr, b, Lx, Ly, mode, nvec, vstride, hstride, dots, st);
    if (dtype == MG2D_C64)  return dispatch_stencil<float>(ctx, n, out, in, in_lo, in_hi, D, nullptr, b, Lx, Ly, mode, nvec, vstride, hstride, dots, st);
    return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_stencil_apply: bad dtype");
}

extern "C" int mg2d_relax_jacobi(mg2d_ctx* ctx, void* out, const void* in, const void* in_lo, const void* in_hi,
                                 const void* D, const void* D0inv, const void* r, int n, int Lx, int Ly, int dtype,
                                 int nvec, long long vstride, long long hstride, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!out || !in || !in_lo || !in_hi || !D || !D0inv || Lx < 1 || Ly < 1 || nvec < 1 || nvec > 64)
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_relax_jacobi: bad argument");
    if (out == in) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_relax_jacobi: out must not alias in");
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MG2D_C128) return dispatch_stencil<double>(ctx, n, out, in, in_lo, in_hi, D, D0inv, r, Lx, Ly, 2, nvec, vstride, hstride, nullptr, st);
    if (dtype == MG2D_C64)  return dispatch_stencil<float>(ctx, n, out, in, in_lo, in_hi, D, D0inv, r, Lx, Ly, 2, nvec, vstride, hstride, nullptr, st);
    return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_relax_jacobi: bad dtype");
}

extern "C" int mg2d_relax_gs(mg2d_ctx* ctx, void* phi, const void* D, const void* D0inv, const void* r, int n, int L,
                             int num_iter, int dtype, int nvec, long long vstride, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!phi || !D || !D0inv || L < 2 || num_iter < 0 || nvec < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_relax_gs: bad argument");
    if (num_iter == 0) return MG2D_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MG2D_C128) return dispatch_gs<double>(ctx, n, phi, D, D0inv, r, L, num_iter, nvec, vstride, st);
    if (dtype == MG2D_C64)  return dispatch_gs<float>(ctx, n, phi, D, D0inv, r, L, num_iter, nvec, vstride, st);
    return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_relax_gs: bad dtype");
}

extern "C" int mg2d_block_inverse(mg2d_ctx* ctx, void* D0inv, const void* D, int n, long long nsites, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!D0inv || !D || nsites < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_block_inverse: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MG2D_C128) return dispatch_inverse<double>(ctx, n, D0inv, D, nsites, st);
    if (dtype == MG2D_C64)  return dispatch_inverse<float>(ctx, n, D0inv, D, nsites, st);
    return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_block_inverse: bad dtype");
}

extern "C" int mg2d_relax_rb(mg2d_ctx* ctx, void* phi, const void* phi_lo, const void* phi_hi, const void* D,
                             const void* D0inv, const void* r, int n, int Lx, int Ly, int colour, int yoff, int dtype,
                             int nvec, long long vstride, long long hstride, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!phi || !phi_lo || !phi_hi || !D || !D0inv || Lx < 2 || (Lx & 1) || Ly < 1 || nvec < 1 || (colour != 0 && colour != 1))
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_relax_rb: bad argument (Lx must be even)");
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MG2D_C128) return dispatch_rb<double>(ctx, n, phi, phi_lo, phi_hi, D, D0inv, r, Lx, Ly, colour, yoff, nvec, vstride, hstride, st);
    if (dtype == MG2D_C64)  return dispatch_rb<float>(ctx, n, phi, phi_lo, phi_hi, D, D0inv, r, Lx, Ly, colour, yoff, nvec, vstride, hstride, st);
    return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_relax_rb: bad dtype");
}

extern "C" int mg2d_to_half(mg2d_ctx* ctx, void* dst_half2, const void* src_c64, long long nelem, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!dst_half2 || !src_c64 || nelem < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_to_half: bad argument");
    long long nb = (nelem + 255) / 256; if (nb > (long long)ctx->num_sms * 16) nb = (long long)ctx->num_sms * 16;
    to_half_kernel<<<(int)nb, 256, 0, (cudaStream_t)stream>>>((__half2*)dst_half2, (const float2*)src_c64, nelem);
    return mg2d_check_launch(ctx, "mg2d_to_half");
}

extern "C" int mg2d_relax_rb_half(mg2d_ctx* ctx, void* phi, const void* phi_lo, const void* phi_hi, const void* Dh,
                                  const void* D0invh, const void* r, int n, int Lx, int Ly, int colour, int yoff, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!phi || !phi_lo || !phi_hi || !Dh || !D0invh || Lx < 2 || (Lx & 1) || Ly < 1 || (colour != 0 && colour != 1))
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_relax_rb_half: bad argument (Lx must be even)");
    cudaStream_t st = (cudaStream_t)stream;
    const long long S2 = (long long)(Lx / 2) * Ly;
    long long nb = (S2 + ST_THREADS / 32 - 1) / (ST_THREADS / 32);
    if (nb > (long long)ctx->num_sms * 32) nb = (long long)ctx->num_sms * 32;
#define RBH(N) stencil_rb_h_kernel<N><<<(int)nb, ST_THREADS, 0, st>>>((float2*)phi, (const float2*)phi_lo, (const float2*)phi_hi, \
        (const __half2*)Dh, (const __half2*)D0invh, (const float2*)r, Lx, Ly, colour, yoff)
    switch (n) {
        case 8: RBH(8); break;
        case 16: RBH(16); break;
        case 32: RBH(32); break;
        default: return mg2d_fail(ctx, MG2D_EUNSUPPORTED, "mg2d_relax_rb_half: n_dof must be 8, 16 or 32");
    }
#undef RBH
    return mg2d_check_launch(ctx, "mg2d_relax_rb_half");
}

extern "C" int mg2d_premultiply(mg2d_ctx* ctx, void* M, const void* D, const void* D0inv, int n, long long nsites, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!M || !D || !D0inv || nsites < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_premultiply: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MG2D_C128) return dispatch_premul<double>(ctx, n, M, D, D0inv, nsites, st);
    if (dtype == MG2D_C64)  return dispatch_premul<float>(ctx, n, M, D, D0inv, nsites, st);
    return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_premultiply: bad dtype");
}

extern "C" int mg2d_relax_rb_pm(mg2d_ctx* ctx, void* phi, const void* phi_lo, const void* phi_hi, const void* M, const void* D0inv,
                                const void* r, void* cbuf, int cmode, int n, int Lx, int Ly, int colour, int yoff, int dtype,
                                int nvec, long long vstride, long long hstride, const mg2d_halo_link* link, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!phi || !phi_lo || !phi_hi || !M || Lx < 2 || (Lx & 1) || Ly < 1 || nvec < 1 || (colour != 0 && colour != 1) ||
        cmode < 0 || cmode > 2 || (cmode == 1 && (!r || !D0inv || !cbuf)) || (cmode == 2 && !cbuf) ||
        (link && (!link->slot_mine || !link->slot_prev || !link->slot_next || ((link->push_next_lo == nullptr) != (link->push_prev_hi == nullptr)))))
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_relax_rb_pm: bad argument (Lx must be even)");
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MG2D_C128) return dispatch_rb_pm<double>(ctx, n, phi, phi_lo, phi_hi, M, D0inv, r, cbuf, cmode, Lx, Ly, colour, yoff, nvec, vstride, hstride, link, st);
    if (dtype == MG2D_C64)  return dispatch_rb_pm<float>(ctx, n, phi, phi_lo, phi_hi, M, D0inv, r, cbuf, cmode, Lx, Ly, colour, yoff, nvec, vstride, hstride, link, st);
    return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_relax_rb_pm: bad dtype");
}

extern "C" int mg2d_relax_rb_pm_sweeps(mg2d_ctx* ctx, void* phi, const void* M, const void* D0inv, const void* r, void* cbuf,
                                       int n, int L, int nsweeps, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!phi || !M || L < 2 || (L & 1) || nsweeps < 1 || (r && (!D0inv || !cbuf)))
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_relax_rb_pm_sweeps: bad argument (L must be even)");
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MG2D_C128) return dispatch_rb_pm_sweeps<double>(ctx, n, phi, M, D0inv, r, cbuf, L, nsweeps, st);
    if (dtype == MG2D_C64)  return dispatch_rb_pm_sweeps<float>(ctx, n, phi, M, D0inv, r, cbuf, L, nsweeps, st);
    return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_relax_rb_pm_sweeps: bad dtype");
}

#define MG2D_LR_CASES(CALL) \
    if (n == 16 && rank == 4) { CALL(16, 4); } \
    else if (n == 8 && rank == 2) { CALL(8, 2); }

extern "C" int mg2d_lowrank_supported(int n, int rank) {
    return (n == 16 && rank == 4) || (n == 8 && rank == 2);
}

extern "C" int mg2d_relax_rb_lr(mg2d_ctx* ctx, void* phi, const void* phi_lo, const void* phi_hi, const void* F, const void* D0inv,
                                const void* r, void* cbuf, int cmode, int n, int rank, int Lx, int Ly, int colour, int yoff,
                                int dtype, int nvec, long long vstride, long long hstride, const struct mg2d_halo_link* link,
                                void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!phi || !phi_lo || !phi_hi || !F || Lx < 2 || (Lx & 1) || Ly < 1 || cmode < 0 || cmode > 2 || (cmode == 1 && (!r || !D0inv)) ||
        (cmode != 0 && !cbuf) || nvec < 1)
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_relax_rb_lr: bad argument (Lx must be even)");
    cudaStream_t st = (cudaStream_t)stream;
#define CALL_D(N, R) return launch_rb_lr<double, N, R>(ctx, phi, phi_lo, phi_hi, F, D0inv, r, cbuf, cmode, Lx, Ly, colour, yoff, nvec, vstride, hstride, link, st)
#define CALL_F(N, R) return launch_rb_lr<float, N, R>(ctx, phi, phi_lo, phi_hi, F, D0inv, r, cbuf, cmode, Lx, Ly, colour, yoff, nvec, vstride, hstride, link, st)
    if (dtype == MG2D_C128) { MG2D_LR_CASES(CALL_D) }
    else if (dtype == MG2D_C64) { MG2D_LR_CASES(CALL_F) }
    else return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_relax_rb_lr: bad dtype");
#undef CALL_D
#undef CALL_F
    return mg2d_fail(ctx, MG2D_EUNSUPPORTED, "mg2d_relax_rb_lr: (n, rank) must be (16,4) or (8,2)");
}

extern "C" int mg2d_hop_factors(mg2d_ctx* ctx, void* A, void* B, const void* Df, const void* P, const void* P_lo, const void* P_hi,
                                int nf, int nc, int Lxf, int Lyf, int block, int dtype, int* status, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!A || !B || !Df || !P || !P_lo || !P_hi || nf < 1 || nf > 2 || nc < 1 || block < 1 || Lxf % block || Lyf % block)
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_hop_factors: bad argument (fine n_dof must be 1 or 2)");
    cudaStream_t st = (cudaStream_t)stream;
    const long long nagg = (long long)(Lxf / block) * (Lyf / block);
    long long nb = (nagg + 7) / 8;
    if (nb > (long long)ctx->num_sms * 16) nb = (long long)ctx->num_sms * 16;
    if (dtype == MG2D_C128)
        hop_factors_kernel<double><<<(int)nb, 256, 0, st>>>((cplx<double>*)A, (cplx<double>*)B, (const cplx<double>*)Df, (const cplx<double>*)P,
                                                            (const cplx<double>*)P_lo, (const cplx<double>*)P_hi, nf, nc, Lxf, Lyf, block, status);
    else if (dtype == MG2D_C64)
        hop_factors_kernel<float><<<(int)nb, 256, 0, st>>>((cplx<float>*)A, (cplx<float>*)B, (const cplx<float>*)Df, (const cplx<float>*)P,
                                                           (const cplx<float>*)P_lo, (const cplx<float>*)P_hi, nf, nc, Lxf, Lyf, block, status);
    else return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_hop_factors: bad dtype");
    return mg2d_check_launch(ctx, "mg2d_hop_factors");
}

extern "C" int mg2d_lowrank_pack(mg2d_ctx* ctx, void* F, const void* A, const void* B, const void* D0inv, int n, int rank,
                                 long long S, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!F || !A || !B || !D0inv || S < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_lowrank_pack: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    long long nb = (S + 7) / 8;
    if (nb > (long long)ctx->num_sms * 16) nb = (long long)ctx->num_sms * 16;
#define CALL_D(N, R) { lowrank_pack_kernel<double, N, R><<<(int)nb, 256, 0, st>>>((cplx<double>*)F, (const cplx<double>*)A, (const cplx<double>*)B, (const cplx<double>*)D0inv, S); return mg2d_check_launch(ctx, "mg2d_lowrank_pack"); }
#define CALL_F(N, R) { lowrank_pack_kernel<float, N, R><<<(int)nb, 256, 0, st>>>((cplx<float>*)F, (const cplx<float>*)A, (const cplx<float>*)B, (const cplx<float>*)D0inv, S); return mg2d_check_launch(ctx, "mg2d_lowrank_pack"); }
    if (dtype == MG2D_C128) { MG2D_LR_CASES(CALL_D) }
    else if (dtype == MG2D_C64) { MG2D_LR_CASES(CALL_F) }
    else return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_lowrank_pack: bad dtype");
#undef CALL_D
#undef CALL_F
    return mg2d_fail(ctx, MG2D_EUNSUPPORTED, "mg2d_lowrank_pack: (n, rank) must be (16,4) or (8,2)");
}

extern "C" int mg2d_lowrank_pack_a(mg2d_ctx* ctx, void* F, const void* A, const void* D0inv, int n, int rank, long long S, int dtype,
                                   void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!F || !A || !D0inv || S < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_lowrank_pack_a: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    long long nb = (S + 7) / 8;
    if (nb > (long long)ctx->num_sms * 16) nb = (long long)ctx->num_sms * 16;
#define CALL_D(N, R) { lowrank_pack_kernel<double, N, R, false><<<(int)nb, 256, 0, st>>>((cplx<double>*)F, (const cplx<double>*)A, nullptr, (const cplx<double>*)D0inv, S); return mg2d_check_launch(ctx, "mg2d_lowrank_pack_a"); }
#define CALL_F(N, R) { lowrank_pack_kernel<float, N, R, false><<<(int)nb, 256, 0, st>>>((cplx<float>*)F, (const cplx<float>*)A, nullptr, (const cplx<float>*)D0inv, S); return mg2d_check_launch(ctx, "mg2d_lowrank_pack_a"); }
    if (dtype == MG2D_C128) { MG2D_LR_CASES(CALL_D) }
    else if (dtype == MG2D_C64) { MG2D_LR_CASES(CALL_F) }
    else return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_lowrank_pack_a: bad dtype");
#undef CALL_D
#undef CALL_F
    return mg2d_fail(ctx, MG2D_EUNSUPPORTED, "mg2d_lowrank_pack_a: (n, rank) must be (16,4) or (8,2)");
}

extern "C" int mg2d_relax_gs_strip(mg2d_ctx* ctx, void* phi, const void* phi_lo, const void* phi_hi, const void* D, const void* D0inv,
                                   const void* r, int n, int Lx, int Ly, int y0, int Lglobal, int dtype, void* slot_mine,
                                   void* slot_next, void* slot_last, void* push_next_lo, void* push_last_hi, int first_rank,
                                   int last_rank, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!phi || !phi_lo || !phi_hi || !D || !D0inv || Lx < 2 || Ly < 1 || y0 < 0 || y0 + Ly > Lglobal || !slot_mine || !slot_next || !slot_last)
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_relax_gs_strip: bad argument");
    GsStripLinks a;
    a.mine = (HaloSlot*)slot_mine; a.next = (HaloSlot*)slot_next; a.last = (HaloSlot*)slot_last;
    a.push_next_lo = push_next_lo; a.push_last_hi = push_last_hi; a.first = first_rank; a.is_last = last_rank;
    cudaStream_t st = (cudaStream_t)stream;
#define CASE(TT, N) case N: return launch_gs_strip<TT, N>(ctx, phi, phi_lo, phi_hi, D, D0inv, r, Lx, Ly, y0, Lglobal, a, st)
    if (dtype == MG2D_C128) { switch (n) { CASE(double, 1); CASE(double, 2); CASE(double, 4); CASE(double, 8); CASE(double, 16); CASE(double, 32); default: break; } }
    else if (dtype == MG2D_C64) { switch (n) { CASE(float, 1); CASE(float, 2); CASE(float, 4); CASE(float, 8); CASE(float, 16); CASE(float, 32); default: break; } }
    else return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_relax_gs_strip: bad dtype");
#undef CASE
    return mg2d_fail(ctx, MG2D_EUNSUPPORTED, "mg2d_relax_gs_strip: n_dof must be one of 1,2,4,8,16,32");
}
