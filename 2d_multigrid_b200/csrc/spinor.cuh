// spinor.cuh -- 2-component spinor loads/stores shared by the matrix-free Wilson kernels (wilson.cu, wilson_rb2.cu).
#pragma once
#include "common.cuh"

namespace {

template <typename T> struct Spinor { cplx<T> c0, c1; };

template <typename T>
__device__ __forceinline__ Spinor<T> load_spinor(const cplx<T>* __restrict__ p, size_t s) {
    Spinor<T> r;
    if constexpr (sizeof(T) == 8) {
        ld256(p + 2 * s, r.c0, r.c1);       // one LDG.E.256 per spinor (sm_100a)
    } else {
        float4 v = __ldg(reinterpret_cast<const float4*>(p) + s);
        r.c0 = make_float2(v.x, v.y); r.c1 = make_float2(v.z, v.w);
    }
    return r;
}
// coherent variant (ld.global, no .nc) for kernels that update the field they read
template <typename T>
__device__ __forceinline__ Spinor<T> load_spinor_c(const cplx<T>* p, size_t s) {
    Spinor<T> r;
    if constexpr (sizeof(T) == 8) {
        asm volatile("ld.global.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(r.c0.x), "=d"(r.c0.y), "=d"(r.c1.x), "=d"(r.c1.y) : "l"(p + 2 * s));
    } else {
        float4 v = *(reinterpret_cast<const float4*>(p) + s);
        r.c0 = make_float2(v.x, v.y); r.c1 = make_float2(v.z, v.w);
    }
    return r;
}
// halo rows a strip neighbour wrote over NVLink: read from L2 (ld.cg), the coherence point of peer stores -- never through
// the non-coherent path.  Plain intrinsics, no inline asm, so the compiler keeps scheduling loads across it.
template <typename T>
__device__ __forceinline__ Spinor<T> load_spinor_sys(const cplx<T>* p, size_t s) {
    Spinor<T> r;
    if constexpr (sizeof(T) == 8) {
        r.c0 = __ldcg(p + 2 * s); r.c1 = __ldcg(p + 2 * s + 1);
    } else {
        const float4 v = __ldcg(reinterpret_cast<const float4*>(p) + s);
        r.c0 = make_float2(v.x, v.y); r.c1 = make_float2(v.z, v.w);
    }
    return r;
}
template <typename T>
__device__ __forceinline__ void store_spinor(cplx<T>* __restrict__ p, size_t s, const Spinor<T>& v) {
    if constexpr (sizeof(T) == 8) {
        st256(p + 2 * s, v.c0, v.c1);
    } else {
        reinterpret_cast<float4*>(p)[s] = make_float4(v.c0.x, v.c0.y, v.c1.x, v.c1.y);
    }
}

// Twisted mass (template flag TM of the Wilson kernels): self block diag(d+f+i mu, d-f-i mu), d = 2+m, f the clover field
// (0 without clover).  A sweep multiplies component 0 by z0 = 1/(d+f+i mu) and component 1 by z1 = 1/(d-f-i mu).  Where
// f == 0 these are the launch constants tz = 1/(d+i mu) and conj(tz); a clover site takes both from one reciprocal
// 1/(|d+f+i mu|^2 |d-f-i mu|^2).
template <typename T>
__device__ __forceinline__ void tm_self_inverse(T f, T d, T mu, cplx<T> tz, cplx<T>& z0, cplx<T>& z1) {
    z0 = tz; z1 = cconj(tz);
    if (f != (T)0) {
        const T a = d + f, b = d - f, mu2 = mu * mu;
        const T na = fma(a, a, mu2), nb = fma(b, b, mu2);
        const T q = (T)1 / (na * nb);
        const T ia = nb * q, ib = na * q;                   // 1/|a+i mu|^2, 1/|b-i mu|^2
        z0 = mk<T>(a * ia, -mu * ia);
        z1 = mk<T>(b * ib, mu * ib);
    }
}
// the launch constant tz = 1/(d + i mu) of tm_self_inverse, formed in double on the host
template <typename T>
inline cplx<T> tm_tz(double d, double mu) {
    const double den = d * d + mu * mu;
    cplx<T> z; z.x = (T)(d / den); z.y = (T)(-mu / den);
    return z;
}

}  // namespace
