// transfer.cu -- block-aggregation kernels: restriction / prolongation over near-null vectors, per-aggregate
// orthonormalisation, and the Galerkin coarse operator  D_c = P D_f P^dagger.
//
//   mg2d_restrict       Near_null::f_restriction   S6/near_null.h:217-240
//   mg2d_prolong_add    Near_null::f_prolongation  S6/near_null.h:242-264 (+ zeroing of f_prolongate_phi,
//                                                  S6/modules_main.h:243-252)
//   mg2d_pack_null      tail of Level::f_near_null S6/level.h:217-246
//   mg2d_norm_nn        Near_null::f_norm_nn       S6/near_null.h:24-48 (f_block_norm, S6/modules_indiv.h:94-135)
//   mg2d_ortho          Near_null::f_ortho         S6/near_null.h:97-173
//   mg2d_check_ortho    Near_null::f_check_ortho   S6/near_null.h:175-214
//   mg2d_coarse_matrix  f_compute_coarse_matrix    S6/modules_main.h:81-185
//
// Aggregates follow f_get_base_site (S6/modules_indiv.h:6-14): coarse site (xc,yc) owns the fine sites
// ((bx+x1)%Lx, (by+y1)%Ly), x1,y1 < block, base shifted by (0,0),(1,0),(1,1),(0,1) for quad 1..4.
// One lane group (restrict/prolong), one warp (norm/ortho) or one CTA (Galerkin) per aggregate.
// P layout: P[s][ic][jf] (nc x nf row-major per fine site) -- the group streams it with stride G, coalesced.
#include "common.cuh"

namespace {

struct AggGeom { int Lxf, Lyf, Lxc, Lyc, block, dx, dy; };

__host__ __device__ inline AggGeom make_geom(int Lxf, int Lyf, int block, int quad) {
    AggGeom g; g.Lxf = Lxf; g.Lyf = Lyf; g.Lxc = Lxf / block; g.Lyc = Lyf / block; g.block = block;
    g.dx = (quad == 2 || quad == 3) ? 1 : 0; g.dy = (quad == 3 || quad == 4) ? 1 : 0;
    return g;
}
// fine site b = x1*block + y1 (x1 outer, y1 inner as in the reference loops) of aggregate X
__device__ __forceinline__ size_t agg_site(const AggGeom& g, int xc, int yc, int b) {
    const int x1 = b / g.block, y1 = b - x1 * g.block;
    int xf = g.block * xc - g.dx + x1; if (xf < 0) xf += g.Lxf; if (xf >= g.Lxf) xf -= g.Lxf;
    int yf = g.block * yc - g.dy + y1; if (yf < 0) yf += g.Lyf; if (yf >= g.Lyf) yf -= g.Lyf;
    return (size_t)yf * g.Lxf + xf;
}

constexpr int TR_THREADS = 256;
template <int NF, int NC> struct TrGroup {
    static constexpr int E = NF * NC;
    static constexpr int G = E < 32 ? E : 32;
    static constexpr int ACC = E / G;
};

template <typename T, int NF, int NC>
__global__ void __launch_bounds__(TR_THREADS)
restrict_kernel(cplx<T>* __restrict__ vc, const cplx<T>* __restrict__ vf, const cplx<T>* __restrict__ P, AggGeom geo) {
    using C = cplx<T>;
    constexpr int E = TrGroup<NF, NC>::E, G = TrGroup<NF, NC>::G, ACC = TrGroup<NF, NC>::ACC, GPB = TR_THREADS / G;
    const int g = threadIdx.x % G, grp = threadIdx.x / G;
    const long long nagg = (long long)geo.Lxc * geo.Lyc;
    const long long nsteps = (nagg + GPB - 1) / GPB;
    const int nb = geo.block * geo.block;
    for (long long step = blockIdx.x; step < nsteps; step += gridDim.x) {
        long long X = step * GPB + grp;
        const bool active = X < nagg;
        if (!active) X = nagg - 1;
        const int yc = (int)(X / geo.Lxc), xc = (int)(X - (long long)yc * geo.Lxc);
        C acc[ACC];
#pragma unroll
        for (int t = 0; t < ACC; ++t) acc[t] = mk<T>(0, 0);
#pragma unroll 4
        for (int b = 0; b < nb; ++b) {
            const size_t s = agg_site(geo, xc, yc, b);
            const C v = __ldg(vf + s * NF + (g % NF));
            const C* Ps = P + s * E;
#pragma unroll
            for (int t = 0; t < ACC; ++t) cfma(acc[t], __ldg(Ps + g + G * t), v);
        }
#pragma unroll
        for (int t = 0; t < ACC; ++t) {
            C a = acc[t];
#pragma unroll
            for (int m = 1; m < NF; m <<= 1) a = cadd(a, shfl_xor_c(a, m));
            if (active && (g % NF) == 0) vc[(size_t)X * NC + (g + G * t) / NF] = a;
        }
    }
}

template <typename T, int NF, int NC>
__global__ void __launch_bounds__(TR_THREADS)
prolong_kernel(cplx<T>* __restrict__ vf, cplx<T>* __restrict__ vc, const cplx<T>* __restrict__ P, AggGeom geo, int zero_vc) {
    using C = cplx<T>;
    constexpr int E = TrGroup<NF, NC>::E, G = TrGroup<NF, NC>::G, ACC = TrGroup<NF, NC>::ACC, GPB = TR_THREADS / G;
    const int g = threadIdx.x % G, grp = threadIdx.x / G;
    const long long nagg = (long long)geo.Lxc * geo.Lyc;
    const long long nsteps = (nagg + GPB - 1) / GPB;
    const int nb = geo.block * geo.block;
    for (long long step = blockIdx.x; step < nsteps; step += gridDim.x) {
        long long X = step * GPB + grp;
        const bool active = X < nagg;
        if (!active) X = nagg - 1;
        const int yc = (int)(X / geo.Lxc), xc = (int)(X - (long long)yc * geo.Lxc);
        C w[ACC];
#pragma unroll
        for (int t = 0; t < ACC; ++t) w[t] = vc[(size_t)X * NC + (g + G * t) / NF];
#pragma unroll 4
        for (int b = 0; b < nb; ++b) {
            const size_t s = agg_site(geo, xc, yc, b);
            const C* Ps = P + s * E;
            C a = mk<T>(0, 0);
#pragma unroll
            for (int t = 0; t < ACC; ++t) cfmac(a, __ldg(Ps + g + G * t), w[t]);   // conj(P) * vc
#pragma unroll
            for (int m = NF; m < G; m <<= 1) a = cadd(a, shfl_xor_c(a, m));
            if (active && g < NF) { C* o = vf + s * NF + g; *o = cadd(*o, a); }
        }
        if (zero_vc) {
            __syncwarp();
            if (active) for (int i = g; i < NC; i += G) vc[(size_t)X * NC + i] = mk<T>(0, 0);
        }
    }
}

// ---- chirality-compacted projector (Wilson levels) -----------------------------------------------------------
// f_near_null stores row d < nc/2 with only its first nf/2 columns non-zero and row d >= nc/2 with only the last nf/2
// (S6/level.h:236-245); block normalisation and Gram-Schmidt keep that structure (rows of opposite chirality have
// an exactly zero dot product).  Pc[s][i][j'] (nc x nf/2) keeps the non-zero half of every row, halving the bytes
// streamed by restriction and prolongation.  Results equal the dense kernels (the dropped terms are x*0).
template <int NF, int NC> struct TrGroupC {
    static constexpr int HF = NF / 2;
    static constexpr int E = HF * NC;
    static constexpr int G = E < 32 ? E : 32;
    static constexpr int ACC = E / G;
};

template <typename T, int NF, int NC>
__global__ void __launch_bounds__(TR_THREADS)
restrict_chiral_kernel(cplx<T>* __restrict__ vc, const cplx<T>* __restrict__ vf, const cplx<T>* __restrict__ Pc, AggGeom geo) {
    using C = cplx<T>;
    using TG = TrGroupC<NF, NC>;
    constexpr int HF = TG::HF, E = TG::E, G = TG::G, ACC = TG::ACC, GPB = TR_THREADS / G;
    const int g = threadIdx.x % G, grp = threadIdx.x / G;
    const long long nagg = (long long)geo.Lxc * geo.Lyc;
    const long long nsteps = (nagg + GPB - 1) / GPB;
    const int nb = geo.block * geo.block;
    for (long long step = blockIdx.x; step < nsteps; step += gridDim.x) {
        long long X = step * GPB + grp;
        const bool active = X < nagg;
        if (!active) X = nagg - 1;
        const int yc = (int)(X / geo.Lxc), xc = (int)(X - (long long)yc * geo.Lxc);
        C acc[ACC];
#pragma unroll
        for (int t = 0; t < ACC; ++t) acc[t] = mk<T>(0, 0);
#pragma unroll 4
        for (int b = 0; b < nb; ++b) {
            const size_t s = agg_site(geo, xc, yc, b);
            const C* Ps = Pc + s * E;
            const C v0 = __ldg(vf + s * NF + (g % HF)), v1 = __ldg(vf + s * NF + HF + (g % HF));
#pragma unroll
            for (int t = 0; t < ACC; ++t) {
                const int i = (g + G * t) / HF;
                cfma(acc[t], __ldg(Ps + g + G * t), (i >= NC / 2) ? v1 : v0);
            }
        }
#pragma unroll
        for (int t = 0; t < ACC; ++t) {
            C a = acc[t];
#pragma unroll
            for (int m = 1; m < HF; m <<= 1) a = cadd(a, shfl_xor_c(a, m));
            if (active && (g % HF) == 0) vc[(size_t)X * NC + (g + G * t) / HF] = a;
        }
    }
}

// Level 0 -> 1 of the headline workload (2-component spinors, 16 coarse dof, 4x4 aggregates): 16 lanes per aggregate, lane i
// owns coarse row i.  The 16 projector elements a lane needs (one per fine site) are all requested before the first FMA
// (fully unrolled, known trip count), and the fine spinors are loaded ONCE per group -- lane b fetches site b with one
// 32-byte load and the group broadcasts it by shuffle -- instead of every lane re-loading both components of every site
// (the generic kernel: 48 load instructions per lane, at most 12 in flight; ncu round 2: 5.3 TB/s).
template <typename T>
__global__ void __launch_bounds__(TR_THREADS)
restrict_chiral_nf2_nc16_blk4_kernel(cplx<T>* __restrict__ vc, const cplx<T>* __restrict__ vf, const cplx<T>* __restrict__ Pc, AggGeom geo) {
    using C = cplx<T>;
    constexpr int G = 16, GPB = TR_THREADS / G, NB = 16;
    const int g = threadIdx.x % G, grp = threadIdx.x / G;
    const long long nagg = (long long)geo.Lxc * geo.Lyc;
    const long long nsteps = (nagg + GPB - 1) / GPB;
    for (long long step = blockIdx.x; step < nsteps; step += gridDim.x) {
        long long X = step * GPB + grp;
        const bool active = X < nagg;
        if (!active) X = nagg - 1;
        const int yc = (int)(X / geo.Lxc), xc = (int)(X - (long long)yc * geo.Lxc);
        const size_t smine = agg_site(geo, xc, yc, g);                  // lane g fetches fine site g of the aggregate
        const C w0 = __ldg(vf + smine * 2), w1 = __ldg(vf + smine * 2 + 1);
        C p[NB];
#pragma unroll
        for (int b = 0; b < NB; ++b) p[b] = __ldg(Pc + agg_site(geo, xc, yc, b) * 16 + g);
        C acc = mk<T>(0, 0);
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            const C v0 = shfl_c(w0, b, G), v1 = shfl_c(w1, b, G);
            cfma(acc, p[b], (g >= 8) ? v1 : v0);                        // rows 8..15 are the second chirality
        }
        if (active) vc[(size_t)X * 16 + g] = acc;
    }
}

// accumulate != 0: vf += P^dagger vc ; accumulate == 0: vf = P^dagger vc (every fine site belongs to one aggregate)
template <typename T, int NF, int NC>
__global__ void __launch_bounds__(TR_THREADS)
prolong_chiral_kernel(cplx<T>* __restrict__ vf, cplx<T>* __restrict__ vc, const cplx<T>* __restrict__ Pc, AggGeom geo,
                      int zero_vc, int accumulate) {
    using C = cplx<T>;
    using TG = TrGroupC<NF, NC>;
    constexpr int HF = TG::HF, E = TG::E, G = TG::G, ACC = TG::ACC, GPB = TR_THREADS / G;
    const int g = threadIdx.x % G, grp = threadIdx.x / G;
    const long long nagg = (long long)geo.Lxc * geo.Lyc;
    const long long nsteps = (nagg + GPB - 1) / GPB;
    const int nb = geo.block * geo.block;
    for (long long step = blockIdx.x; step < nsteps; step += gridDim.x) {
        long long X = step * GPB + grp;
        const bool active = X < nagg;
        if (!active) X = nagg - 1;
        const int yc = (int)(X / geo.Lxc), xc = (int)(X - (long long)yc * geo.Lxc);
        C w[ACC];
#pragma unroll
        for (int t = 0; t < ACC; ++t) w[t] = vc[(size_t)X * NC + (g + G * t) / HF];
#pragma unroll 4
        for (int b = 0; b < nb; ++b) {
            const size_t s = agg_site(geo, xc, yc, b);
            const C* Ps = Pc + s * E;
            C a0 = mk<T>(0, 0), a1 = mk<T>(0, 0);
#pragma unroll
            for (int t = 0; t < ACC; ++t) {
                const int i = (g + G * t) / HF;
                const C pv = __ldg(Ps + g + G * t);
                if (i >= NC / 2) cfmac(a1, pv, w[t]); else cfmac(a0, pv, w[t]);
            }
#pragma unroll
            for (int m = HF; m < G; m <<= 1) { a0 = cadd(a0, shfl_xor_c(a0, m)); a1 = cadd(a1, shfl_xor_c(a1, m)); }
            if (active && g < HF) {
                C* o0 = vf + s * NF + g; C* o1 = vf + s * NF + HF + g;
                if (accumulate) { *o0 = cadd(*o0, a0); *o1 = cadd(*o1, a1); } else { *o0 = a0; *o1 = a1; }
            }
        }
        if (zero_vc) {
            __syncwarp();
            if (active) for (int i = g; i < NC; i += G) vc[(size_t)X * NC + i] = mk<T>(0, 0);
        }
    }
}

// Level 0 -> Wilson spinors (NF = 2) with 4x4 aggregates and NC coarse dof: the generic lane mapping needs a
// log2(NC)-step butterfly per fine site (shuffle-bound: 32 SHFL per 512 B streamed).  Here a warp owns one aggregate,
// streams Pc coalesced exactly as before, parks the products conj(Pc[s][i]) * vc[i] in a padded shared-memory tile
// [16 sites][NC] and then lane (site b, chirality c) adds its NC/2 terms: no shuffles, 2 x 4 KB of shared traffic
// per 4 KB of DRAM traffic.
template <typename T, int NC>
__global__ void __launch_bounds__(TR_THREADS)
prolong_chiral_nf2_blk4_kernel(cplx<T>* __restrict__ vf, cplx<T>* __restrict__ vc, const cplx<T>* __restrict__ Pc, AggGeom geo,
                               int zero_vc, int accumulate) {
    using C = cplx<T>;
    constexpr int NB = 16, PAD = NC + 1, WPB = TR_THREADS / 32, SPP = 32 / NC;   // SPP sites per pass of the warp
    static_assert(NC == 16 || NC == 8, "NC");
    __shared__ C tile[WPB][NB * PAD];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    C* tl = tile[warp];
    const long long nagg = (long long)geo.Lxc * geo.Lyc;
    const int i = lane % NC, sub = lane / NC;
    for (long long X = (long long)blockIdx.x * WPB + warp; X < nagg; X += (long long)gridDim.x * WPB) {
        const int yc = (int)(X / geo.Lxc), xc = (int)(X - (long long)yc * geo.Lxc);
        const C w = vc[(size_t)X * NC + i];
#pragma unroll
        for (int b0 = 0; b0 < NB; b0 += SPP) {
            const int b = b0 + sub;
            const size_t s = agg_site(geo, xc, yc, b);
            tl[b * PAD + i] = cmulc(__ldg(Pc + s * NC + i), w);      // conj(P) * vc
        }
        __syncwarp();
        {   // lane = (site b, chirality c)
            const int b = lane >> 1, c = lane & 1;
            C a = mk<T>(0, 0);
#pragma unroll
            for (int k = 0; k < NC / 2; ++k) a = cadd(a, tl[b * PAD + c * (NC / 2) + k]);
            const size_t s = agg_site(geo, xc, yc, b);
            C* o = vf + s * 2 + c;
            if (accumulate) *o = cadd(*o, a); else *o = a;
        }
        __syncwarp();
        if (zero_vc && lane < NC) vc[(size_t)X * NC + lane] = mk<T>(0, 0);
    }
}

// ---- setup kernels (runtime nf, nc) -------------------------------------------------------------------
template <typename T>
__global__ void pack_null_kernel(cplx<T>* __restrict__ P, const cplx<T>* __restrict__ V, int nvec, long long vstride,
                                 int nf, int nc, long long S, int wilson) {
    using C = cplx<T>;
    const long long total = S * nc * nf;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int j = (int)(e % nf);
        const int row = (int)((e / nf) % nc);
        const long long s = e / ((long long)nf * nc);
        C val = mk<T>(0, 0);
        if (!wilson) {
            if (row < nvec) val = cconj(V[(size_t)row * vstride + s * nf + j]);
            else val = P[e];
        } else {
            const int h = nf / 2, v = row % (nc / 2);
            const bool upper_row = row < nc / 2;
            if (v < nvec) { if (upper_row == (j < h)) val = cconj(V[(size_t)v * vstride + s * nf + j]); }
            else val = P[e];
        }
        P[e] = val;
    }
}

// sum over the aggregate's (b, j) entries of row d; lanes stride, butterfly -> all lanes
template <typename T>
__device__ __forceinline__ void row_norm_dot(const cplx<T>* P, const AggGeom& geo, int xc, int yc, int nf, int nc,
                                             int d_u, int d_t, int lane, double& nrm2, double& dre, double& dim_) {
    const int nb = geo.block * geo.block, len = nb * nf;
    nrm2 = 0.0; dre = 0.0; dim_ = 0.0;
    for (int e = lane; e < len; e += 32) {
        const int b = e / nf, j = e - b * nf;
        const size_t s = agg_site(geo, xc, yc, b);
        const cplx<T> u = P[(s * nc + d_u) * nf + j];
        nrm2 += (double)u.x * u.x + (double)u.y * u.y;
        if (d_t >= 0) {
            const cplx<T> t = P[(s * nc + d_t) * nf + j];
            dre += (double)u.x * t.x + (double)u.y * t.y;
            dim_ += (double)u.x * t.y - (double)u.y * t.x;
        }
    }
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) {
        nrm2 += __shfl_xor_sync(0xffffffffu, nrm2, m);
        dre += __shfl_xor_sync(0xffffffffu, dre, m);
        dim_ += __shfl_xor_sync(0xffffffffu, dim_, m);
    }
}

template <typename T>
__device__ __forceinline__ void row_block_normalise(cplx<T>* P, const AggGeom& geo, int xc, int yc, int nf, int nc,
                                                    int d, int lane, int* status) {
    double n2, a, b;
    row_norm_dot<T>(P, geo, xc, yc, nf, nc, d, -1, lane, n2, a, b);
    const double nrm = sqrt(n2);
    if (status && lane == 0 && (isnan(nrm) || nrm < 1e-40)) atomicOr(status, 1);   // S6/modules_indiv.h:119-126
    const int len = geo.block * geo.block * nf;
    for (int e = lane; e < len; e += 32) {
        const int bb = e / nf, j = e - bb * nf;
        const size_t s = agg_site(geo, xc, yc, bb);
        cplx<T>* p = P + (s * nc + d) * nf + j;
        cplx<T> v = *p; v.x = (T)(v.x / nrm); v.y = (T)(v.y / nrm); *p = v;
    }
    __syncwarp();
}

// MODE 0: norm_nn ; 1: ortho ; 2: check_ortho (max |<d1,d2>| -> out via atomicMax on the bit pattern)
template <typename T, int MODE>
__global__ void __launch_bounds__(128)
aggregate_rows_kernel(cplx<T>* P, AggGeom geo, int nf, int nc, int* status, unsigned long long* out_max) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const long long nagg = (long long)geo.Lxc * geo.Lyc;
    const int len = geo.block * geo.block * nf;
    double worst = 0.0;
    for (long long X = (long long)blockIdx.x * wpb + warp; X < nagg; X += (long long)gridDim.x * wpb) {
        const int yc = (int)(X / geo.Lxc), xc = (int)(X - (long long)yc * geo.Lxc);
        if (MODE == 0) {
            for (int d = 0; d < nc; ++d) row_block_normalise<T>(P, geo, xc, yc, nf, nc, d, lane, status);
        } else if (MODE == 1) {
            for (int d1 = 0; d1 < nc; ++d1) {
                for (int d2 = 0; d2 < d1; ++d2) {
                    double n2, dre, dim_;
                    row_norm_dot<T>(P, geo, xc, yc, nf, nc, d2, d1, lane, n2, dre, dim_);
                    const double nrm = sqrt(n2);
                    if (status && lane == 0 && (isnan(nrm) || nrm < 1e-8 || isnan(dre) || isnan(dim_))) atomicOr(status, 2);
                    const double cr = dre / nrm, ci = dim_ / nrm;     // (dot/norm), S6/near_null.h:165
                    for (int e = lane; e < len; e += 32) {
                        const int b = e / nf, j = e - b * nf;
                        const size_t s = agg_site(geo, xc, yc, b);
                        const cplx<T> u = P[(s * nc + d2) * nf + j];
                        cplx<T>* tp = P + (s * nc + d1) * nf + j;
                        cplx<T> t = *tp;
                        t.x = (T)(t.x - (cr * u.x - ci * u.y));
                        t.y = (T)(t.y - (cr * u.y + ci * u.x));
                        *tp = t;
                    }
                    __syncwarp();
                }
                row_block_normalise<T>(P, geo, xc, yc, nf, nc, d1, lane, status);
            }
        } else {
            for (int d1 = 0; d1 < nc; ++d1)
                for (int d2 = 0; d2 < d1; ++d2) {
                    double n2, dre, dim_;
                    row_norm_dot<T>(P, geo, xc, yc, nf, nc, d1, d2, lane, n2, dre, dim_);
                    worst = fmax(worst, sqrt(dre * dre + dim_ * dim_));
                }
        }
    }
    if (MODE == 2 && lane == 0) atomicMax(out_max, (unsigned long long)__double_as_longlong(worst));
}

// Galerkin: one CTA per coarse site.  Shared: acc[5][nc*nc] + T[nf*nc].
template <typename T>
__global__ void __launch_bounds__(256)
coarse_matrix_kernel(cplx<T>* __restrict__ Dc, const cplx<T>* __restrict__ Df, const cplx<T>* __restrict__ P,
                     const cplx<T>* __restrict__ P_lo, const cplx<T>* __restrict__ P_hi, AggGeom geo, int nf, int nc) {
    using C = cplx<T>;
    extern __shared__ unsigned char smem_raw[];
    C* acc = reinterpret_cast<C*>(smem_raw);          // [5][nc*nc], element (i,i') at i'*nc+i (column-major)
    C* Tm = acc + 5 * nc * nc;                        // [nf][nc]: T[j][i'] = sum_j' Df_k(j,j') conj(P(s')[i'][j'])
    const long long nagg = (long long)geo.Lxc * geo.Lyc;
    const int nb = geo.block * geo.block, blk = geo.block;
    const int E = nf * nc;
    for (long long X = blockIdx.x; X < nagg; X += gridDim.x) {
        const int yc = (int)(X / geo.Lxc), xc = (int)(X - (long long)yc * geo.Lxc);
        for (int o = threadIdx.x; o < 5 * nc * nc; o += blockDim.x) acc[o] = mk<T>(0, 0);
        __syncthreads();
        for (int b = 0; b < nb; ++b) {
            const int x1 = b / blk, y1 = b - x1 * blk;
            const size_t s = agg_site(geo, xc, yc, b);
            const int yf = (int)(s / geo.Lxf), xf = (int)(s - (size_t)yf * geo.Lxf);
            const C* Ps = P + s * E;
            for (int k = 0; k < 5; ++k) {
                // neighbour projector block and destination slot (S6/modules_main.h:130-155)
                const C* Pn; int slot;
                if (k == 0) { Pn = Ps; slot = 0; }
                else if (k == 1) { Pn = P + ((size_t)yf * geo.Lxf + (xf + 1 == geo.Lxf ? 0 : xf + 1)) * E; slot = (x1 != blk - 1) ? 0 : 1; }
                else if (k == 2) { Pn = P + ((size_t)yf * geo.Lxf + (xf == 0 ? geo.Lxf - 1 : xf - 1)) * E; slot = (x1 != 0) ? 0 : 2; }
                else if (k == 3) { Pn = (yf + 1 == geo.Lyf) ? P_hi + (size_t)xf * E : P + ((size_t)(yf + 1) * geo.Lxf + xf) * E; slot = (y1 != blk - 1) ? 0 : 3; }
                else { Pn = (yf == 0) ? P_lo + (size_t)xf * E : P + ((size_t)(yf - 1) * geo.Lxf + xf) * E; slot = (y1 != 0) ? 0 : 4; }
                const C* Dk = Df + (s * 5 + k) * nf * nf;
                for (int e = threadIdx.x; e < E; e += blockDim.x) {
                    const int j = e / nc, ip = e - j * nc;
                    C t = mk<T>(0, 0);
                    for (int jp = 0; jp < nf; ++jp) {
                        const C d = __ldg(Dk + jp * nf + j);
                        const C p = __ldg(Pn + ip * nf + jp);
                        // d * conj(p)
                        t.x = fma(d.x, p.x, t.x); t.x = fma(d.y, p.y, t.x);
                        t.y = fma(d.y, p.x, t.y); t.y = fma(-d.x, p.y, t.y);
                    }
                    Tm[e] = t;
                }
                __syncthreads();
                C* dst = acc + slot * nc * nc;
                for (int o = threadIdx.x; o < nc * nc; o += blockDim.x) {
                    const int ip = o / nc, i = o - ip * nc;
                    C a = dst[o];
                    for (int j = 0; j < nf; ++j) cfma(a, __ldg(Ps + i * nf + j), Tm[j * nc + ip]);
                    dst[o] = a;
                }
                __syncthreads();
            }
        }
        C* out = Dc + (size_t)X * 5 * nc * nc;
        for (int o = threadIdx.x; o < 5 * nc * nc; o += blockDim.x) out[o] = acc[o];
        __syncthreads();
    }
}

template <typename T, int NF, int NC>
int launch_transfer(mg2d_ctx* ctx, int which, void* vc, void* vf, const void* P, AggGeom geo, int zero_vc, cudaStream_t st) {
    using C = cplx<T>;
    constexpr int GPB = TR_THREADS / TrGroup<NF, NC>::G;
    const long long nagg = (long long)geo.Lxc * geo.Lyc;
    long long nb = (nagg + GPB - 1) / GPB;
    if (nb > (long long)ctx->num_sms * 32) nb = (long long)ctx->num_sms * 32;
    if (which == 0) restrict_kernel<T, NF, NC><<<(int)nb, TR_THREADS, 0, st>>>((C*)vc, (const C*)vf, (const C*)P, geo);
    else prolong_kernel<T, NF, NC><<<(int)nb, TR_THREADS, 0, st>>>((C*)vf, (C*)vc, (const C*)P, geo, zero_vc);
    return mg2d_check_launch(ctx, which == 0 ? "mg2d_restrict" : "mg2d_prolong_add");
}

template <typename T>
int dispatch_transfer(mg2d_ctx* ctx, int which, void* vc, void* vf, const void* P, int nf, int nc, AggGeom geo,
                      int zero_vc, cudaStream_t st) {
#define PAIR(NF, NC) if (nf == NF && nc == NC) return launch_transfer<T, NF, NC>(ctx, which, vc, vf, P, geo, zero_vc, st)
    PAIR(1, 1); PAIR(1, 2); PAIR(1, 4); PAIR(1, 8); PAIR(1, 16); PAIR(1, 32);
    PAIR(2, 2); PAIR(2, 4); PAIR(2, 8); PAIR(2, 16); PAIR(2, 32);
    PAIR(4, 4); PAIR(8, 8); PAIR(16, 16); PAIR(32, 32);
    PAIR(4, 8); PAIR(4, 16); PAIR(8, 16); PAIR(4, 2);
#undef PAIR
    return mg2d_fail(ctx, MG2D_EUNSUPPORTED, "mg2d_restrict/prolong: unsupported (nf, nc) pair");
}

template <typename T, int NF, int NC>
int launch_transfer_c(mg2d_ctx* ctx, int which, void* vc, void* vf, const void* P, AggGeom geo, int zero_vc, int accumulate, cudaStream_t st) {
    using C = cplx<T>;
    constexpr int GPB = TR_THREADS / TrGroupC<NF, NC>::G;
    const long long nagg = (long long)geo.Lxc * geo.Lyc;
    long long nb = (nagg + GPB - 1) / GPB;
    if (nb > (long long)ctx->num_sms * 32) nb = (long long)ctx->num_sms * 32;
    if (which == 0) {
        if constexpr (NF == 2 && NC == 16) {
            if (geo.block == 4) {
                restrict_chiral_nf2_nc16_blk4_kernel<T><<<(int)nb, TR_THREADS, 0, st>>>((C*)vc, (const C*)vf, (const C*)P, geo);
                return mg2d_check_launch(ctx, "mg2d_restrict_chiral");
            }
        }
        restrict_chiral_kernel<T, NF, NC><<<(int)nb, TR_THREADS, 0, st>>>((C*)vc, (const C*)vf, (const C*)P, geo);
    } else {
        if constexpr (NF == 2 && (NC == 8 || NC == 16)) {
            if (geo.block == 4) {
                long long nw = (nagg + TR_THREADS / 32 - 1) / (TR_THREADS / 32);
                if (nw > (long long)ctx->num_sms * 32) nw = (long long)ctx->num_sms * 32;
                prolong_chiral_nf2_blk4_kernel<T, NC><<<(int)nw, TR_THREADS, 0, st>>>((C*)vf, (C*)vc, (const C*)P, geo, zero_vc, accumulate);
                return mg2d_check_launch(ctx, "mg2d_prolong_chiral");
            }
        }
        prolong_chiral_kernel<T, NF, NC><<<(int)nb, TR_THREADS, 0, st>>>((C*)vf, (C*)vc, (const C*)P, geo, zero_vc, accumulate);
    }
    return mg2d_check_launch(ctx, which == 0 ? "mg2d_restrict_chiral" : "mg2d_prolong_chiral");
}

template <typename T>
int dispatch_transfer_c(mg2d_ctx* ctx, int which, void* vc, void* vf, const void* P, int nf, int nc, AggGeom geo,
                        int zero_vc, int accumulate, cudaStream_t st) {
#define PAIR(NF, NC) if (nf == NF && nc == NC) return launch_transfer_c<T, NF, NC>(ctx, which, vc, vf, P, geo, zero_vc, accumulate, st)
    PAIR(2, 4); PAIR(2, 8); PAIR(2, 16); PAIR(2, 32);
    PAIR(4, 4); PAIR(8, 8); PAIR(16, 16); PAIR(32, 32);
    PAIR(4, 8); PAIR(4, 16); PAIR(8, 16);
#undef PAIR
    return mg2d_fail(ctx, MG2D_EUNSUPPORTED, "mg2d_restrict/prolong_chiral: unsupported (nf, nc) pair");
}

inline int check_geom(mg2d_ctx* ctx, int Lxf, int Lyf, int block, int quad, const char* name) {
    if (Lxf < 1 || Lyf < 1 || block < 1 || quad < 1 || quad > 4 || Lxf % block || Lyf % block) {
        snprintf(ctx->err, sizeof(ctx->err), "%s: bad geometry (Lx=%d Ly=%d block=%d quad=%d)", name, Lxf, Lyf, block, quad);
        return MG2D_EINVAL;
    }
    return MG2D_OK;
}

}  // namespace

extern "C" int mg2d_restrict(mg2d_ctx* ctx, void* vc, const void* vf, const void* P, int nf, int nc, int Lxf, int Lyf,
                             int block, int quad, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!vc || !vf || !P) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_restrict: null pointer");
    if (int rc = check_geom(ctx, Lxf, Lyf, block, quad, "mg2d_restrict")) return rc;
    AggGeom geo = make_geom(Lxf, Lyf, block, quad);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MG2D_C128) return dispatch_transfer<double>(ctx, 0, vc, (void*)vf, P, nf, nc, geo, 0, st);
    if (dtype == MG2D_C64)  return dispatch_transfer<float>(ctx, 0, vc, (void*)vf, P, nf, nc, geo, 0, st);
    return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_restrict: bad dtype");
}

extern "C" int mg2d_prolong_add(mg2d_ctx* ctx, void* vf, void* vc, const void* P, int nf, int nc, int Lxf, int Lyf,
                                int block, int quad, int zero_vc, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!vc || !vf || !P) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_prolong_add: null pointer");
    if (int rc = check_geom(ctx, Lxf, Lyf, block, quad, "mg2d_prolong_add")) return rc;
    AggGeom geo = make_geom(Lxf, Lyf, block, quad);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MG2D_C128) return dispatch_transfer<double>(ctx, 1, vc, vf, P, nf, nc, geo, zero_vc, st);
    if (dtype == MG2D_C64)  return dispatch_transfer<float>(ctx, 1, vc, vf, P, nf, nc, geo, zero_vc, st);
    return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_prolong_add: bad dtype");
}

extern "C" int mg2d_pack_null(mg2d_ctx* ctx, void* P, const void* V, int nvec, long long vstride, int nf, int nc,
                              long long nsites, int wilson, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!P || !V || nvec < 1 || nf < 1 || nc < 1 || nsites < 1 || (wilson && ((nf & 1) || (nc & 1) || nvec > nc / 2)) || (!wilson && nvec > nc))
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_pack_null: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    long long total = nsites * nc * nf;
    long long nb = (total + 255) / 256; if (nb > (long long)ctx->num_sms * 16) nb = (long long)ctx->num_sms * 16;
    if (dtype == MG2D_C128) pack_null_kernel<double><<<(int)nb, 256, 0, st>>>((double2*)P, (const double2*)V, nvec, vstride, nf, nc, nsites, wilson);
    else if (dtype == MG2D_C64) pack_null_kernel<float><<<(int)nb, 256, 0, st>>>((float2*)P, (const float2*)V, nvec, vstride, nf, nc, nsites, wilson);
    else return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_pack_null: bad dtype");
    return mg2d_check_launch(ctx, "mg2d_pack_null");
}

template <int MODE>
static int launch_rows(mg2d_ctx* ctx, void* P, int nf, int nc, int Lxf, int Lyf, int block, int quad, int dtype,
                       int* status, double* out, void* stream, const char* name) {
    if (!ctx) return MG2D_EINVAL;
    if (!P || nf < 1 || nc < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d aggregate rows: bad argument");
    if (int rc = check_geom(ctx, Lxf, Lyf, block, quad, name)) return rc;
    AggGeom geo = make_geom(Lxf, Lyf, block, quad);
    cudaStream_t st = (cudaStream_t)stream;
    const long long nagg = (long long)geo.Lxc * geo.Lyc;
    long long nb = (nagg + 3) / 4; if (nb > (long long)ctx->num_sms * 32) nb = (long long)ctx->num_sms * 32;
    if (MODE == 2) { if (cudaMemsetAsync(out, 0, sizeof(double), st) != cudaSuccess) return mg2d_fail(ctx, MG2D_ECUDA, "memset failed"); }
    if (dtype == MG2D_C128) aggregate_rows_kernel<double, MODE><<<(int)nb, 128, 0, st>>>((double2*)P, geo, nf, nc, status, (unsigned long long*)out);
    else if (dtype == MG2D_C64) aggregate_rows_kernel<float, MODE><<<(int)nb, 128, 0, st>>>((float2*)P, geo, nf, nc, status, (unsigned long long*)out);
    else return mg2d_fail(ctx, MG2D_EINVAL, "mg2d aggregate rows: bad dtype");
    return mg2d_check_launch(ctx, name);
}

extern "C" int mg2d_norm_nn(mg2d_ctx* ctx, void* P, int nf, int nc, int Lxf, int Lyf, int block, int quad, int dtype,
                            int* status, void* stream) {
    return launch_rows<0>(ctx, P, nf, nc, Lxf, Lyf, block, quad, dtype, status, nullptr, stream, "mg2d_norm_nn");
}
extern "C" int mg2d_ortho(mg2d_ctx* ctx, void* P, int nf, int nc, int Lxf, int Lyf, int block, int quad, int dtype,
                          int* status, void* stream) {
    return launch_rows<1>(ctx, P, nf, nc, Lxf, Lyf, block, quad, dtype, status, nullptr, stream, "mg2d_ortho");
}
extern "C" int mg2d_check_ortho(mg2d_ctx* ctx, const void* P, int nf, int nc, int Lxf, int Lyf, int block, int quad,
                                int dtype, double* out, void* stream) {
    if (!out) return ctx ? mg2d_fail(ctx, MG2D_EINVAL, "mg2d_check_ortho: null out") : MG2D_EINVAL;
    return launch_rows<2>(ctx, (void*)P, nf, nc, Lxf, Lyf, block, quad, dtype, nullptr, out, stream, "mg2d_check_ortho");
}

extern "C" int mg2d_coarse_matrix(mg2d_ctx* ctx, void* Dc, const void* Df, const void* P, const void* P_lo, const void* P_hi,
                                  int nf, int nc, int Lxf, int Lyf, int block, int quad, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!Dc || !Df || !P || !P_lo || !P_hi || nf < 1 || nc < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_coarse_matrix: bad argument");
    if (int rc = check_geom(ctx, Lxf, Lyf, block, quad, "mg2d_coarse_matrix")) return rc;
    AggGeom geo = make_geom(Lxf, Lyf, block, quad);
    cudaStream_t st = (cudaStream_t)stream;
    const long long nagg = (long long)geo.Lxc * geo.Lyc;
    long long nb = nagg; if (nb > (long long)ctx->num_sms * 8) nb = (long long)ctx->num_sms * 8;
    const size_t csz = dtype == MG2D_C128 ? sizeof(double2) : sizeof(float2);
    const size_t smem = (size_t)(5 * nc * nc + nf * nc) * csz;
    if (smem > 200 * 1024) return mg2d_fail(ctx, MG2D_EUNSUPPORTED, "mg2d_coarse_matrix: nc too large for shared memory");
    cudaError_t e;
    if (dtype == MG2D_C128) {
        e = cudaFuncSetAttribute(coarse_matrix_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return mg2d_fail(ctx, MG2D_ECUDA, "mg2d_coarse_matrix: cannot set shared memory size");
        coarse_matrix_kernel<double><<<(int)nb, 256, smem, st>>>((double2*)Dc, (const double2*)Df, (const double2*)P, (const double2*)P_lo, (const double2*)P_hi, geo, nf, nc);
    } else if (dtype == MG2D_C64) {
        e = cudaFuncSetAttribute(coarse_matrix_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return mg2d_fail(ctx, MG2D_ECUDA, "mg2d_coarse_matrix: cannot set shared memory size");
        coarse_matrix_kernel<float><<<(int)nb, 256, smem, st>>>((float2*)Dc, (const float2*)Df, (const float2*)P, (const float2*)P_lo, (const float2*)P_hi, geo, nf, nc);
    } else return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_coarse_matrix: bad dtype");
    return mg2d_check_launch(ctx, "mg2d_coarse_matrix");
}

extern "C" int mg2d_restrict_chiral(mg2d_ctx* ctx, void* vc, const void* vf, const void* Pc, int nf, int nc, int Lxf, int Lyf,
                                    int block, int quad, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!vc || !vf || !Pc) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_restrict_chiral: null pointer");
    if (int rc = check_geom(ctx, Lxf, Lyf, block, quad, "mg2d_restrict_chiral")) return rc;
    AggGeom geo = make_geom(Lxf, Lyf, block, quad);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MG2D_C128) return dispatch_transfer_c<double>(ctx, 0, vc, (void*)vf, Pc, nf, nc, geo, 0, 1, st);
    if (dtype == MG2D_C64)  return dispatch_transfer_c<float>(ctx, 0, vc, (void*)vf, Pc, nf, nc, geo, 0, 1, st);
    return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_restrict_chiral: bad dtype");
}

extern "C" int mg2d_prolong_chiral(mg2d_ctx* ctx, void* vf, void* vc, const void* Pc, int nf, int nc, int Lxf, int Lyf,
                                   int block, int quad, int zero_vc, int accumulate, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!vc || !vf || !Pc) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_prolong_chiral: null pointer");
    if (int rc = check_geom(ctx, Lxf, Lyf, block, quad, "mg2d_prolong_chiral")) return rc;
    AggGeom geo = make_geom(Lxf, Lyf, block, quad);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MG2D_C128) return dispatch_transfer_c<double>(ctx, 1, vc, vf, Pc, nf, nc, geo, zero_vc, accumulate, st);
    if (dtype == MG2D_C64)  return dispatch_transfer_c<float>(ctx, 1, vc, vf, Pc, nf, nc, geo, zero_vc, accumulate, st);
    return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_prolong_chiral: bad dtype");
}
