// common.cuh -- shared device helpers for libmg2d_sm100.so (sm_100a only).
#pragma once
#include <cstdlib>
#include <cstring>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include "../../include/mg2d.h"

#define MG2D_MAX_PARTIALS 4096   // max CTAs contributing to one reduction
#define MG2D_MAX_RED 64          // max doubles per reduction (batched dots)

// ---- multi-GPU records living in the CUDA-IPC slabs (identical offsets on every rank) ---------------------------
#define MG2D_MAX_RANKS 8
#define MG2D_XRED_MAX 64         // doubles per cross-GPU reduction

struct HaloSlot {            // one per exchanged field (level, width, depth); 64 bytes
    unsigned long long flag_lo, flag_hi;     // written by prev / next: epoch of the rows now in my lo / hi halo buffer
    unsigned long long ack_prev, ack_next;   // written by prev / next: last epoch of MY rows they have consumed
    unsigned long long epoch;                // local: number of publishes done
    unsigned long long error;                // local: a neighbour did not answer within the spin bound
    unsigned long long ticket;               // local: CTAs of the running kernel that finished
    unsigned long long pad;
};

struct XRedArea {            // all-reduce mailbox: every rank writes its partial sums into every peer's area
    unsigned long long flag[2][MG2D_MAX_RANKS];              // [parity][source rank] = epoch of buf[parity][source]
    double buf[2][MG2D_MAX_RANKS][MG2D_XRED_MAX];
};

struct XComm {               // local descriptor (plain device memory) of the rank's place among its peers
    int world, rank;
    unsigned long long epoch;                // all-reduces completed
    unsigned long long error;
    int relaxed;                             // flags published with relaxed stores behind the one fence (mg2d_publish_relaxed)
    XRedArea* area[MG2D_MAX_RANKS];          // area[q] = rank q's mailbox (peer-mapped; area[rank] is local)
};

// what a stencil kernel needs to push its boundary rows to the strip neighbours and to wait for theirs (host struct
// mg2d_halo_link of include/mg2d.h, resolved to typed pointers)
struct HaloLinkDev {
    HaloSlot* mine; HaloSlot* prev; HaloSlot* next;
    void* push_next_lo; void* push_prev_hi;
    int wait;
    int relaxed;     // publish flags with relaxed system-scope stores behind ONE fence (default) instead of two release stores
};

// MG2D_PUBLISH=release restores the two st.release.sys per publication (each carries its own system-scope fence: three
// sequential NVLink round trips at the tail of every halo-linked kernel); default: __threadfence_system() once, then relaxed stores
inline int mg2d_publish_relaxed() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("MG2D_PUBLISH"); v = (e && !strcmp(e, "release")) ? 0 : 1; }
    return v;
}

struct mg2d_ctx {
    int device;
    int launches;
    double* partials;        // [MG2D_MAX_PARTIALS][MG2D_MAX_RED]
    unsigned int* counter;   // last-block-done tickets, one per reduction "channel"
    int num_sms;
    XComm* xcomm;            // multi-GPU: descriptor for reductions fused into the kernels (NULL on one GPU)
    int xreduce;             // 1: reductions of the following calls are summed over all ranks inside the kernel
    char err[512];
};

static inline int mg2d_fail(mg2d_ctx* c, int code, const char* msg) {
    if (c) snprintf(c->err, sizeof(c->err), "%s", msg);
    return code;
}
static inline int mg2d_check_launch(mg2d_ctx* c, const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        if (c) snprintf(c->err, sizeof(c->err), "%s: %s", what, cudaGetErrorString(e));
        return MG2D_ECUDA;
    }
    if (c) c->launches++;
    return MG2D_OK;
}

// ---- complex arithmetic on (re,im) pairs ------------------------------------------------------------
template <typename T> struct cplx_of;
template <> struct cplx_of<double> { using type = double2; };
template <> struct cplx_of<float>  { using type = float2; };
template <typename T> using cplx = typename cplx_of<T>::type;

template <typename T> __device__ __forceinline__ cplx<T> mk(T re, T im) { cplx<T> r; r.x = re; r.y = im; return r; }
template <typename C> __device__ __forceinline__ C cadd(C a, C b) { a.x += b.x; a.y += b.y; return a; }
template <typename C> __device__ __forceinline__ C csub(C a, C b) { a.x -= b.x; a.y -= b.y; return a; }
template <typename C> __device__ __forceinline__ C cmul(C a, C b) { C r; r.x = a.x * b.x - a.y * b.y; r.y = a.x * b.y + a.y * b.x; return r; }
// conj(a) * b
template <typename C> __device__ __forceinline__ C cmulc(C a, C b) { C r; r.x = a.x * b.x + a.y * b.y; r.y = a.x * b.y - a.y * b.x; return r; }
// acc += a * b
template <typename C> __device__ __forceinline__ void cfma(C& acc, C a, C b) {
    acc.x = fma(a.x, b.x, acc.x); acc.x = fma(-a.y, b.y, acc.x);
    acc.y = fma(a.x, b.y, acc.y); acc.y = fma(a.y, b.x, acc.y);
}
// acc += conj(a) * b
template <typename C> __device__ __forceinline__ void cfmac(C& acc, C a, C b) {
    acc.x = fma(a.x, b.x, acc.x); acc.x = fma(a.y, b.y, acc.x);
    acc.y = fma(a.x, b.y, acc.y); acc.y = fma(-a.y, b.x, acc.y);
}
template <typename C> __device__ __forceinline__ C cconj(C a) { a.y = -a.y; return a; }
template <typename C> __device__ __forceinline__ C cmul_i(C a) { C r; r.x = -a.y; r.y = a.x; return r; }   // i*a
template <typename C> __device__ __forceinline__ C cmul_mi(C a) { C r; r.x = a.y; r.y = -a.x; return r; }  // -i*a
template <typename C, typename T> __device__ __forceinline__ C cscale(C a, T s) { a.x *= s; a.y *= s; return a; }

// read-only 8/16-byte loads
__device__ __forceinline__ double2 ldg(const double2* p) { return __ldg(p); }
__device__ __forceinline__ float2  ldg(const float2* p)  { return __ldg(p); }

// 256-bit global accesses (sm_100a: LDG.E.256 / STG.E.256); p must be 32-byte aligned
__device__ __forceinline__ void ld256(const double2* p, double2& a, double2& b) {
    asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a.x), "=d"(a.y), "=d"(b.x), "=d"(b.y) : "l"(p));
}
__device__ __forceinline__ void st256(double2* p, const double2& a, const double2& b) {
    asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" :: "l"(p), "d"(a.x), "d"(a.y), "d"(b.x), "d"(b.y) : "memory");
}

__device__ __forceinline__ double shfl_xor_d(double v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
template <typename C> __device__ __forceinline__ C shfl_xor_c(C v, int m) {
    v.x = __shfl_xor_sync(0xffffffffu, v.x, m); v.y = __shfl_xor_sync(0xffffffffu, v.y, m); return v;
}
template <typename C> __device__ __forceinline__ C shfl_c(C v, int src, int width = 32) {
    v.x = __shfl_sync(0xffffffffu, v.x, src, width); v.y = __shfl_sync(0xffffffffu, v.y, src, width); return v;
}

// Scheduling fence for a batch of loaded values: one empty asm that "modifies" all of them, so every load of the batch must
// have been ISSUED before the first consumer can be scheduled (the compiler otherwise sinks each load next to its FMA to
// save registers, leaving an in-order warp with 2-5 loads in flight instead of the whole batch).  No instruction is emitted.
__device__ __forceinline__ void keep8(double2 (&v)[8]) {
    asm volatile("" : "+d"(v[0].x), "+d"(v[0].y), "+d"(v[1].x), "+d"(v[1].y), "+d"(v[2].x), "+d"(v[2].y), "+d"(v[3].x), "+d"(v[3].y),
                      "+d"(v[4].x), "+d"(v[4].y), "+d"(v[5].x), "+d"(v[5].y), "+d"(v[6].x), "+d"(v[6].y), "+d"(v[7].x), "+d"(v[7].y));
}
__device__ __forceinline__ void keep8(float2 (&v)[8]) {
    asm volatile("" : "+f"(v[0].x), "+f"(v[0].y), "+f"(v[1].x), "+f"(v[1].y), "+f"(v[2].x), "+f"(v[2].y), "+f"(v[3].x), "+f"(v[3].y),
                      "+f"(v[4].x), "+f"(v[4].y), "+f"(v[5].x), "+f"(v[5].y), "+f"(v[6].x), "+f"(v[6].y), "+f"(v[7].x), "+f"(v[7].y));
}
template <typename C, int K> __device__ __forceinline__ void keep_all(C (&v)[K]) {
    if constexpr (K % 8 == 0) {
#pragma unroll
        for (int b = 0; b < K; b += 8) keep8(*reinterpret_cast<C(*)[8]>(&v[b]));
    }
}

// ---- system-scope flag accesses (peer memory over NVLink) ---------------------------------------------
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}
// two flags of the same value; the caller has already executed __threadfence_system() after the data they guard
__device__ __forceinline__ void publish2(unsigned long long* a, unsigned long long* b, unsigned long long v, int relaxed) {
    if (relaxed) { st_relaxed_sys(a, v); st_relaxed_sys(b, v); }
    else { st_release_sys(a, v); st_release_sys(b, v); }
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ double ld_relaxed_sys_f64(const double* p) {
    double v;
    asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}
// bounded spin (~20 s): a lost peer becomes an error flag, never a hang
__device__ __forceinline__ bool spin_until(const unsigned long long* p, unsigned long long want) {
    for (long long it = 0; it < (1ll << 27); ++it) {
        if (ld_acquire_sys(p) >= want) return true;
        __nanosleep(it < 64 ? 20 : 150);
    }
    return false;
}

// Sum `vals[0..nr)` (shared memory, block-uniform) over all ranks: every rank stores its numbers into every peer's
// mailbox, raises the peer's flag, waits for all flags of its own mailbox and adds the contributions in rank order, so
// all ranks obtain bit-identical results.  Called by ONE CTA (all its threads).  Two mailbox halves alternate: a rank
// can only be one reduction ahead of its slowest peer (it needs that peer's contribution to finish the current one).
__device__ __forceinline__ void xcomm_allreduce(XComm* xc, const double* vals, int nr, double* out) {
    const int world = xc->world, rank = xc->rank;
    const unsigned long long e = xc->epoch + 1ull;
    const int par = (int)(e & 1ull);
    __shared__ int s_ok;
    if (threadIdx.x == 0) s_ok = 1;
    __syncthreads();
    for (int t = threadIdx.x; t < world * nr; t += blockDim.x) {
        const int q = t / nr, k = t - q * nr;
        xc->area[q]->buf[par][rank][k] = vals[k];
    }
    __threadfence_system();
    __syncthreads();
    if ((int)threadIdx.x < world) {
        if (xc->relaxed) st_relaxed_sys(&xc->area[threadIdx.x]->flag[par][rank], e);
        else st_release_sys(&xc->area[threadIdx.x]->flag[par][rank], e);
        if (!spin_until(&xc->area[rank]->flag[par][threadIdx.x], e)) s_ok = 0;
    }
    __syncthreads();
    if ((int)threadIdx.x < nr) {
        double x = 0.0;
        for (int q = 0; q < world; ++q) x += ld_relaxed_sys_f64(&xc->area[rank]->buf[par][q][threadIdx.x]);
        out[threadIdx.x] = x;
    }
    __syncthreads();
    if (threadIdx.x == 0) { xc->epoch = e; if (!s_ok) xc->error = 1ull; }
}

// ---- deterministic grid-wide reduction of NR doubles -------------------------------------------------
// Every CTA calls this with its per-thread values; the warp/CTA tree and the final pass over the per-CTA
// partials run in a fixed order, so results are bit-reproducible for a fixed launch configuration.
// `out[r]` is written by the last CTA to finish.  All threads of the CTA must call it.
// xc != NULL: the result is additionally summed over all ranks (xcomm_allreduce) by the last CTA.
template <int NR, int NTHREADS>
__device__ __forceinline__ void grid_reduce(double (&v)[NR], double* __restrict__ partials,
                                            unsigned int* __restrict__ counter, double* __restrict__ out,
                                            int cta_linear, int num_ctas, XComm* xc = nullptr) {
    __shared__ double s_red[NR][NTHREADS / 32];
    __shared__ double s_tot[NR];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int r = 0; r < NR; ++r) {
        double x = v[r];
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) x += __shfl_xor_sync(0xffffffffu, x, m);
        if (lane == 0) s_red[r][warp] = x;
    }
    __syncthreads();
    if (threadIdx.x < NR) {
        double x = 0.0;
        for (int w = 0; w < NTHREADS / 32; ++w) x += s_red[threadIdx.x][w];
        partials[(size_t)cta_linear * NR + threadIdx.x] = x;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int t = atomicAdd(counter, 1u);
        s_last = (t == (unsigned int)num_ctas - 1u);
    }
    __syncthreads();
    if (s_last) {
        __threadfence();
        // fixed-order sum over CTAs: warp r handles slot r (strided, then shuffle tree)
        for (int r = warp; r < NR; r += NTHREADS / 32) {
            double x = 0.0;
            for (int c = lane; c < num_ctas; c += 32) x += __ldcg(&partials[(size_t)c * NR + r]);
#pragma unroll
            for (int m = 16; m > 0; m >>= 1) x += __shfl_xor_sync(0xffffffffu, x, m);
            if (lane == 0) { if (xc) s_tot[r] = x; else out[r] = x; }
        }
        if (threadIdx.x == 0) *counter = 0u;
        if (xc) {                       // block-uniform: s_last and xc are
            __syncthreads();
            xcomm_allreduce(xc, s_tot, NR, out);
        }
    }
}
