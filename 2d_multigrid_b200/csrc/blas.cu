// blas.cu -- handle management and the fused vector updates of the MR smoother / V-cycle driver.
//   mg2d_mr_update       MR smoother step (ours; BASELINE.json north_star)
//   mg2d_norm2 / scale   f_g_norm, S6/modules_indiv.h:70-92
//   mg2d_cdot_batch      Gram matrix + source of f_min_res, S6/modules_main.h:324-366
//   mg2d_scale_phi       f_scale_phi, S6/modules_main.h:375-384
//   mg2d_minres_solve    A.colPivHouseholderQr().solve(src), S6/modules_main.h:371
// All are pure streaming kernels: HBM-bound, 16-byte (c128) / 8-byte (c64) vector accesses, grid-stride.
#include "common.cuh"

namespace {

constexpr int BL_THREADS = 256;

inline int stream_grid(mg2d_ctx* ctx, long long n, int per_thread = 1) {
    long long nb = (n + (long long)BL_THREADS * per_thread - 1) / ((long long)BL_THREADS * per_thread);
    long long cap = (long long)ctx->num_sms * 8;
    if (nb > cap) nb = cap;
    if (nb > MG2D_MAX_PARTIALS) nb = MG2D_MAX_PARTIALS;
    if (nb < 1) nb = 1;
    return (int)nb;
}

template <typename T>
__global__ void __launch_bounds__(BL_THREADS)
mr_update_kernel(cplx<T>* __restrict__ phi, cplx<T>* __restrict__ res, const cplx<T>* __restrict__ t,
                 const double* __restrict__ dots, double omega, long long n, long long vstride) {
    using C = cplx<T>;
    const int v = blockIdx.y;
    const double tt = dots[4 * v + MG2D_DOT_OUT2];
    // alpha = omega * <t,res>/<t,t>
    const double ar = tt > 0.0 ? omega * dots[4 * v + MG2D_DOT_OUTIN_RE] / tt : 0.0;
    const double ai = tt > 0.0 ? omega * dots[4 * v + MG2D_DOT_OUTIN_IM] / tt : 0.0;
    const C alpha = mk<T>((T)ar, (T)ai), nalpha = mk<T>((T)-ar, (T)-ai);
    phi += (size_t)v * vstride; res += (size_t)v * vstride; t += (size_t)v * vstride;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        C p = phi[e], r = res[e];
        const C tv = __ldg(t + e);
        cfma(p, alpha, r);
        cfma(r, nalpha, tv);
        phi[e] = p; res[e] = r;
    }
}

template <typename T>
__global__ void __launch_bounds__(BL_THREADS)
axpy_kernel(cplx<T>* __restrict__ y, const cplx<T>* __restrict__ x, double a_re, double a_im,
            const double* __restrict__ a_dev, long long n) {
    using C = cplx<T>;
    if (a_dev) { a_re = a_dev[0]; a_im = a_dev[1]; }
    const C a = mk<T>((T)a_re, (T)a_im);
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        C yv = y[e];
        cfma(yv, a, __ldg(x + e));
        y[e] = yv;
    }
}

// y += sign * (num/den) * x  [and y2 += sign * (num/den) * x2], coefficients on the device (GCR updates)
template <typename T>
__global__ void __launch_bounds__(BL_THREADS)
axpy_ratio2_kernel(cplx<T>* __restrict__ y, const cplx<T>* __restrict__ x, cplx<T>* __restrict__ y2,
                   const cplx<T>* __restrict__ x2, const double* __restrict__ num, const double* __restrict__ den,
                   double sign, long long n) {
    using C = cplx<T>;
    const double d = den[0];
    const C a = d > 0.0 ? mk<T>((T)(sign * num[0] / d), (T)(sign * num[1] / d)) : mk<T>(0, 0);
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        C yv = y[e];
        cfma(yv, a, __ldg(x + e));
        y[e] = yv;
        if (y2) { C y2v = y2[e]; cfma(y2v, a, __ldg(x2 + e)); y2[e] = y2v; }
    }
}

template <typename T>
__global__ void __launch_bounds__(BL_THREADS) zero_kernel(cplx<T>* __restrict__ x, long long n) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
        x[e] = mk<T>(0, 0);
}

template <typename TD, typename TS>
__global__ void __launch_bounds__(BL_THREADS) convert_kernel(cplx<TD>* __restrict__ dst, const cplx<TS>* __restrict__ src, long long n) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const cplx<TS> s = __ldg(src + e);
        dst[e] = mk<TD>((TD)s.x, (TD)s.y);
    }
}

template <typename T>
__global__ void __launch_bounds__(BL_THREADS)
norm2_kernel(const cplx<T>* __restrict__ x, long long n, double* __restrict__ partials, unsigned int* __restrict__ counter,
             double* __restrict__ out, XComm* xc) {
    double red[1] = {0.0};
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const cplx<T> v = __ldg(x + e);
        red[0] += (double)v.x * v.x + (double)v.y * v.y;
    }
    grid_reduce<1, BL_THREADS>(red, partials, counter, out, blockIdx.x, gridDim.x, xc);
}

// one (i,j) pair per blockIdx.y; out[2*(i*ny+j)] = sum conj(x_i) y_j
template <typename T>
__global__ void __launch_bounds__(BL_THREADS)
cdot_kernel(const cplx<T>* __restrict__ x, long long xstride, const cplx<T>* __restrict__ y, long long ystride, int ny,
            long long n, double* __restrict__ partials, unsigned int* __restrict__ counter, double* __restrict__ out) {
    const int pair = blockIdx.y;
    const int i = pair / ny, j = pair - i * ny;
    const cplx<T>* xi = x + (size_t)i * xstride;
    const cplx<T>* yj = y + (size_t)j * ystride;
    double red[2] = {0.0, 0.0};
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const cplx<T> a = __ldg(xi + e), b = __ldg(yj + e);
        red[0] += (double)a.x * b.x + (double)a.y * b.y;
        red[1] += (double)a.x * b.y - (double)a.y * b.x;
    }
    grid_reduce<2, BL_THREADS>(red, partials + (size_t)pair * MG2D_MAX_PARTIALS * 2, counter + pair, out + 2 * pair,
                               blockIdx.x, gridDim.x);
}

template <typename T>
__global__ void __launch_bounds__(BL_THREADS)
scale_inv_norm_kernel(cplx<T>* __restrict__ x, const double* __restrict__ norm2, long long n) {
    const double inv = 1.0 / sqrt(norm2[0]);
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        cplx<T> v = x[e];
        // the reference divides (vec /= g_norm, S6/modules_indiv.h:89); keep a true division in fp64
        if constexpr (sizeof(T) == 8) { const double nrm = sqrt(norm2[0]); v.x /= nrm; v.y /= nrm; }
        else { v.x = (T)(v.x * inv); v.y = (T)(v.y * inv); }
        x[e] = v;
    }
}

template <typename T>
__global__ void __launch_bounds__(BL_THREADS)
scale_phi_kernel(cplx<T>* __restrict__ phi, cplx<T>* __restrict__ e, long long estride, const double* __restrict__ a,
                 int ncopies, long long n) {
    using C = cplx<T>;
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        C p = phi[k];
        for (int q = 0; q < ncopies; ++q) {
            C* eq = e + (size_t)q * estride;
            cfma(p, mk<T>((T)a[2 * q], (T)a[2 * q + 1]), eq[k]);
            eq[k] = mk<T>(0, 0);
        }
        phi[k] = p;
    }
}

// column-pivoted Householder QR solve of an n x n (n <= 4) complex system, one thread.
__global__ void minres_solve_kernel(const double* __restrict__ gram, const double* __restrict__ src, int n,
                                    double* __restrict__ a) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double2 A[4][4], c[4], y[4];
    int perm[4];
    double diag[4];
    for (int i = 0; i < n; ++i) {
        perm[i] = i; c[i] = make_double2(src[2 * i], src[2 * i + 1]);
        for (int j = 0; j < n; ++j) A[i][j] = make_double2(gram[2 * (i * n + j)], gram[2 * (i * n + j) + 1]);
    }
    for (int k = 0; k < n; ++k) {
        int best = k; double bn = -1.0;
        for (int j = k; j < n; ++j) {
            double s = 0.0;
            for (int i = k; i < n; ++i) s += A[i][j].x * A[i][j].x + A[i][j].y * A[i][j].y;
            if (s > bn) { bn = s; best = j; }
        }
        if (best != k) {
            for (int i = 0; i < n; ++i) { double2 t = A[i][k]; A[i][k] = A[i][best]; A[i][best] = t; }
            int t = perm[k]; perm[k] = perm[best]; perm[best] = t;
        }
        double alpha = 0.0;
        for (int i = k; i < n; ++i) alpha += A[i][k].x * A[i][k].x + A[i][k].y * A[i][k].y;
        alpha = sqrt(alpha);
        if (alpha == 0.0) { diag[k] = 0.0; continue; }
        double2 v[4];
        for (int i = k; i < n; ++i) v[i] = A[i][k];
        const double a0 = sqrt(v[k].x * v[k].x + v[k].y * v[k].y);
        double2 ph = a0 != 0.0 ? make_double2(v[k].x / a0, v[k].y / a0) : make_double2(1.0, 0.0);
        v[k].x += ph.x * alpha; v[k].y += ph.y * alpha;
        double vn = 0.0;
        for (int i = k; i < n; ++i) vn += v[i].x * v[i].x + v[i].y * v[i].y;
        vn = sqrt(vn);
        for (int i = k; i < n; ++i) { v[i].x /= vn; v[i].y /= vn; }
        for (int j = k; j < n; ++j) {            // A[k:,j] -= 2 v (v^H A[k:,j])
            double2 d = make_double2(0.0, 0.0);
            for (int i = k; i < n; ++i) cfmac(d, v[i], A[i][j]);
            for (int i = k; i < n; ++i) { double2 t = cmul(v[i], d); A[i][j].x -= 2.0 * t.x; A[i][j].y -= 2.0 * t.y; }
        }
        double2 d = make_double2(0.0, 0.0);
        for (int i = k; i < n; ++i) cfmac(d, v[i], c[i]);
        for (int i = k; i < n; ++i) { double2 t = cmul(v[i], d); c[i].x -= 2.0 * t.x; c[i].y -= 2.0 * t.y; }
        diag[k] = sqrt(A[k][k].x * A[k][k].x + A[k][k].y * A[k][k].y);
    }
    double dmax = 0.0;
    for (int k = 0; k < n; ++k) dmax = fmax(dmax, diag[k]);
    const double thresh = 2.220446049250313e-16 * n * dmax;
    int rank = 0;
    for (int k = 0; k < n; ++k) rank += diag[k] > thresh ? 1 : 0;
    for (int i = 0; i < n; ++i) y[i] = make_double2(0.0, 0.0);
    for (int i = rank - 1; i >= 0; --i) {
        double2 s = c[i];
        for (int j = i + 1; j < rank; ++j) { double2 t = cmul(A[i][j], y[j]); s.x -= t.x; s.y -= t.y; }
        const double den = A[i][i].x * A[i][i].x + A[i][i].y * A[i][i].y;
        y[i] = make_double2((s.x * A[i][i].x + s.y * A[i][i].y) / den, (s.y * A[i][i].x - s.x * A[i][i].y) / den);
    }
    for (int i = 0; i < n; ++i) { a[2 * perm[i]] = y[i].x; a[2 * perm[i] + 1] = y[i].y; }
}

}  // namespace

// ---- handle ----------------------------------------------------------------------------------------------
extern "C" int mg2d_version(void) { return 100; }

extern "C" int mg2d_create(mg2d_ctx** out, int device) {
    if (!out) return MG2D_EINVAL;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return MG2D_ECUDA;
    if (cudaSetDevice(device) != cudaSuccess) return MG2D_ECUDA;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return MG2D_ECUDA;
    if (prop.major != 10) return MG2D_EUNSUPPORTED;   // sm_100a only: no fallback path exists
    mg2d_ctx* c = new mg2d_ctx();
    c->device = device; c->launches = 0; c->num_sms = prop.multiProcessorCount; c->err[0] = 0;
    c->partials = nullptr; c->counter = nullptr; c->xcomm = nullptr; c->xreduce = 0;
    if (cudaMalloc(&c->partials, sizeof(double) * MG2D_MAX_PARTIALS * 4 * 64) != cudaSuccess ||
        cudaMalloc(&c->counter, sizeof(unsigned int) * 256) != cudaSuccess ||
        cudaMemset(c->counter, 0, sizeof(unsigned int) * 256) != cudaSuccess) {
        cudaFree(c->partials); cudaFree(c->counter); delete c;
        return MG2D_ECUDA;
    }
    *out = c;
    return MG2D_OK;
}

extern "C" int mg2d_destroy(mg2d_ctx* c) {
    if (!c) return MG2D_EINVAL;
    cudaSetDevice(c->device);
    cudaFree(c->partials); cudaFree(c->counter);
    delete c;
    return MG2D_OK;
}

extern "C" const char* mg2d_last_error(mg2d_ctx* c) { return c ? c->err : "mg2d: null handle"; }
extern "C" int mg2d_launch_count(mg2d_ctx* c) { return c ? c->launches : -1; }

#define DISPATCH_T(dtype, CALL_D, CALL_F, NAME)                                         \
    if (dtype == MG2D_C128) { CALL_D; } else if (dtype == MG2D_C64) { CALL_F; }         \
    else return mg2d_fail(ctx, MG2D_EINVAL, NAME ": bad dtype");                        \
    return mg2d_check_launch(ctx, NAME)

extern "C" int mg2d_mr_update(mg2d_ctx* ctx, void* phi, void* res, const void* t, const double* dots, double omega,
                              long long nelem, int dtype, int nvec, long long vstride, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!phi || !res || !t || !dots || nelem < 1 || nvec < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_mr_update: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid(stream_grid(ctx, nelem), nvec);
    DISPATCH_T(dtype,
        (mr_update_kernel<double><<<grid, BL_THREADS, 0, st>>>((double2*)phi, (double2*)res, (const double2*)t, dots, omega, nelem, vstride)),
        (mr_update_kernel<float><<<grid, BL_THREADS, 0, st>>>((float2*)phi, (float2*)res, (const float2*)t, dots, omega, nelem, vstride)),
        "mg2d_mr_update");
}

extern "C" int mg2d_axpy(mg2d_ctx* ctx, void* y, const void* x, double a_re, double a_im, const double* a_dev,
                         long long nelem, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!y || !x || nelem < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_axpy: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = stream_grid(ctx, nelem);
    DISPATCH_T(dtype,
        (axpy_kernel<double><<<grid, BL_THREADS, 0, st>>>((double2*)y, (const double2*)x, a_re, a_im, a_dev, nelem)),
        (axpy_kernel<float><<<grid, BL_THREADS, 0, st>>>((float2*)y, (const float2*)x, a_re, a_im, a_dev, nelem)),
        "mg2d_axpy");
}

extern "C" int mg2d_zero(mg2d_ctx* ctx, void* x, long long nelem, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!x || nelem < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_zero: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = stream_grid(ctx, nelem);
    DISPATCH_T(dtype,
        (zero_kernel<double><<<grid, BL_THREADS, 0, st>>>((double2*)x, nelem)),
        (zero_kernel<float><<<grid, BL_THREADS, 0, st>>>((float2*)x, nelem)),
        "mg2d_zero");
}

extern "C" int mg2d_copy(mg2d_ctx* ctx, void* dst, const void* src, long long nelem, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!dst || !src || nelem < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_copy: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = stream_grid(ctx, nelem);
    DISPATCH_T(dtype,
        (convert_kernel<double, double><<<grid, BL_THREADS, 0, st>>>((double2*)dst, (const double2*)src, nelem)),
        (convert_kernel<float, float><<<grid, BL_THREADS, 0, st>>>((float2*)dst, (const float2*)src, nelem)),
        "mg2d_copy");
}

extern "C" int mg2d_convert(mg2d_ctx* ctx, void* dst, int dst_dtype, const void* src, int src_dtype, long long nelem, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!dst || !src || nelem < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_convert: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = stream_grid(ctx, nelem);
    if (dst_dtype == MG2D_C128 && src_dtype == MG2D_C64) convert_kernel<double, float><<<grid, BL_THREADS, 0, st>>>((double2*)dst, (const float2*)src, nelem);
    else if (dst_dtype == MG2D_C64 && src_dtype == MG2D_C128) convert_kernel<float, double><<<grid, BL_THREADS, 0, st>>>((float2*)dst, (const double2*)src, nelem);
    else if (dst_dtype == src_dtype) return mg2d_copy(ctx, dst, src, nelem, dst_dtype, stream);
    else return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_convert: bad dtype");
    return mg2d_check_launch(ctx, "mg2d_convert");
}

extern "C" int mg2d_norm2(mg2d_ctx* ctx, const void* x, long long nelem, int dtype, double* out, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!x || !out || nelem < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_norm2: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = stream_grid(ctx, nelem);
    XComm* xc = ctx->xreduce ? ctx->xcomm : nullptr;
    DISPATCH_T(dtype,
        (norm2_kernel<double><<<grid, BL_THREADS, 0, st>>>((const double2*)x, nelem, ctx->partials, ctx->counter, out, xc)),
        (norm2_kernel<float><<<grid, BL_THREADS, 0, st>>>((const float2*)x, nelem, ctx->partials, ctx->counter, out, xc)),
        "mg2d_norm2");
}

extern "C" int mg2d_cdot_batch(mg2d_ctx* ctx, const void* x, long long xstride, int nx, const void* y, long long ystride,
                               int ny, long long nelem, int dtype, double* out, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!x || !y || !out || nelem < 1 || nx < 1 || ny < 1 || nx * ny > 64) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_cdot_batch: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid(stream_grid(ctx, nelem), nx * ny);
    DISPATCH_T(dtype,
        (cdot_kernel<double><<<grid, BL_THREADS, 0, st>>>((const double2*)x, xstride, (const double2*)y, ystride, ny, nelem, ctx->partials, ctx->counter, out)),
        (cdot_kernel<float><<<grid, BL_THREADS, 0, st>>>((const float2*)x, xstride, (const float2*)y, ystride, ny, nelem, ctx->partials, ctx->counter, out)),
        "mg2d_cdot_batch");
}

extern "C" int mg2d_scale_inv_norm(mg2d_ctx* ctx, void* x, const double* norm2, long long nelem, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!x || !norm2 || nelem < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_scale_inv_norm: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = stream_grid(ctx, nelem);
    DISPATCH_T(dtype,
        (scale_inv_norm_kernel<double><<<grid, BL_THREADS, 0, st>>>((double2*)x, norm2, nelem)),
        (scale_inv_norm_kernel<float><<<grid, BL_THREADS, 0, st>>>((float2*)x, norm2, nelem)),
        "mg2d_scale_inv_norm");
}

extern "C" int mg2d_minres_solve(mg2d_ctx* ctx, const double* gram, const double* src, int ncopies, double* a, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!gram || !src || !a || ncopies < 1 || ncopies > 4) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_minres_solve: bad argument");
    minres_solve_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(gram, src, ncopies, a);
    return mg2d_check_launch(ctx, "mg2d_minres_solve");
}

extern "C" int mg2d_scale_phi(mg2d_ctx* ctx, void* phi, void* e, long long estride, const double* a, int ncopies,
                              long long nelem, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!phi || !e || !a || ncopies < 1 || ncopies > 4 || nelem < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_scale_phi: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = stream_grid(ctx, nelem);
    DISPATCH_T(dtype,
        (scale_phi_kernel<double><<<grid, BL_THREADS, 0, st>>>((double2*)phi, (double2*)e, estride, a, ncopies, nelem)),
        (scale_phi_kernel<float><<<grid, BL_THREADS, 0, st>>>((float2*)phi, (float2*)e, estride, a, ncopies, nelem)),
        "mg2d_scale_phi");
}

extern "C" int mg2d_axpy_ratio2(mg2d_ctx* ctx, void* y, const void* x, void* y2, const void* x2, const double* num,
                                const double* den, double sign, long long nelem, int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!y || !x || !num || !den || nelem < 1 || ((y2 == nullptr) != (x2 == nullptr))) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_axpy_ratio2: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = stream_grid(ctx, nelem);
    DISPATCH_T(dtype,
        (axpy_ratio2_kernel<double><<<grid, BL_THREADS, 0, st>>>((double2*)y, (const double2*)x, (double2*)y2, (const double2*)x2, num, den, sign, nelem)),
        (axpy_ratio2_kernel<float><<<grid, BL_THREADS, 0, st>>>((float2*)y, (const float2*)x, (float2*)y2, (const float2*)x2, num, den, sign, nelem)),
        "mg2d_axpy_ratio2");
}

// ---- fused updates of the outer flexible GCR (classical Gram-Schmidt against the stored directions) -------------
// One pass each instead of 2 launches per stored direction: K1 all projections <W_j, w>; K2 w -= sum b_j W_j,
// z -= sum b_j Z_j with |w|^2 and <w, r> of the NEW w accumulated on the fly; K3 x += a z, r -= a w with |r|^2.
namespace {
constexpr int GCR_MAXJ = 8;

// the projections, specialised on the number of stored directions like gcr_ortho_w_kernel (registers follow NJ; U independent
// elements per thread keep (NJ+1)*U loads in flight)
template <typename T, int NJ, int U>
__global__ void __launch_bounds__(BL_THREADS)
gcr_dots_nj_kernel(const cplx<T>* __restrict__ W, long long stride, const cplx<T>* __restrict__ w, long long n,
                   double* __restrict__ partials, unsigned int* __restrict__ counter, double* __restrict__ out, XComm* xc) {
    using C = cplx<T>;
    double red[2 * GCR_MAXJ];
#pragma unroll
    for (int k = 0; k < 2 * GCR_MAXJ; ++k) red[k] = 0.0;
    const long long nthreads = (long long)gridDim.x * blockDim.x;
    for (long long e0 = blockIdx.x * (long long)blockDim.x + threadIdx.x; e0 < n; e0 += nthreads * U) {
        C b[U], a[U][NJ];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long e = e0 + u * nthreads;
            if (e < n) {
                b[u] = __ldg(w + e);
#pragma unroll
                for (int j = 0; j < NJ; ++j) a[u][j] = __ldg(W + (size_t)j * stride + e);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (e0 + u * nthreads < n) {
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    red[2 * j] += (double)a[u][j].x * b[u].x + (double)a[u][j].y * b[u].y;
                    red[2 * j + 1] += (double)a[u][j].x * b[u].y - (double)a[u][j].y * b[u].x;
                }
            }
        }
    }
    grid_reduce<2 * GCR_MAXJ, BL_THREADS>(red, partials, counter, out, blockIdx.x, gridDim.x, xc);
}

template <typename T>
int launch_dots_nj(mg2d_ctx* ctx, const void* W, long long stride, int nj, const void* w, long long nelem, double* out, cudaStream_t st) {
    using C = cplx<T>;
    XComm* xc = ctx->xreduce ? ctx->xcomm : nullptr;
#define DK(NJ, U) gcr_dots_nj_kernel<T, NJ, U><<<stream_grid(ctx, nelem, U), BL_THREADS, 0, st>>>((const C*)W, stride, (const C*)w, nelem, ctx->partials, ctx->counter, out, xc)
    switch (nj) {
        case 1: DK(1, 4); break;
        case 2: DK(2, 4); break;
        case 3: DK(3, 2); break;
        case 4: DK(4, 2); break;
        case 5: DK(5, 2); break;
        case 6: DK(6, 1); break;
        case 7: DK(7, 1); break;
        default: DK(8, 1); break;
    }
#undef DK
    return mg2d_check_launch(ctx, "mg2d_gcr_dots");
}

template <typename T>
__global__ void __launch_bounds__(BL_THREADS)
gcr_ortho_kernel(cplx<T>* __restrict__ w, cplx<T>* __restrict__ z, const cplx<T>* __restrict__ r,
                 const cplx<T>* __restrict__ W, const cplx<T>* __restrict__ Z, long long stride, int nj,
                 const double* __restrict__ dots, const double* __restrict__ wn2, long long n,
                 double* __restrict__ partials, unsigned int* __restrict__ counter, double* __restrict__ out, XComm* xc) {
    using C = cplx<T>;
    C beta[GCR_MAXJ];
#pragma unroll
    for (int j = 0; j < GCR_MAXJ; ++j) {
        const double d = (j < nj) ? wn2[j] : 0.0;
        beta[j] = (j < nj && d > 0.0) ? mk<T>((T)(-dots[2 * j] / d), (T)(-dots[2 * j + 1] / d)) : mk<T>(0, 0);
    }
    double red[4] = {0.0, 0.0, 0.0, 0.0};
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        C wv = w[e];
        if (z) {
            C zv = z[e];
#pragma unroll
            for (int j = 0; j < GCR_MAXJ; ++j) {
                if (j < nj) {
                    cfma(wv, beta[j], __ldg(W + (size_t)j * stride + e));
                    cfma(zv, beta[j], __ldg(Z + (size_t)j * stride + e));
                }
            }
            z[e] = zv;
        } else {                                   // lazy variant: the preconditioned directions stay raw (see gcr_step_lazy_kernel)
#pragma unroll
            for (int j = 0; j < GCR_MAXJ; ++j)
                if (j < nj) cfma(wv, beta[j], __ldg(W + (size_t)j * stride + e));
        }
        w[e] = wv;
        const C rv = __ldg(r + e);
        red[0] += (double)wv.x * wv.x + (double)wv.y * wv.y;
        red[1] += (double)wv.x * rv.x + (double)wv.y * rv.y;       // <w, r> = conj(w) r
        red[2] += (double)wv.x * rv.y - (double)wv.y * rv.x;
    }
    grid_reduce<4, BL_THREADS>(red, partials, counter, out, blockIdx.x, gridDim.x, xc);
}

// The lazy variant's orthogonalisation (w only), specialised on the number of stored directions: registers (and with them
// the resident warps) follow NJ instead of the worst case, and U independent elements per thread keep enough bytes in flight
// when only a few streams are read (NJ = 0: w and r only).
template <typename T, int NJ, int U>
__global__ void __launch_bounds__(BL_THREADS)
gcr_ortho_w_kernel(cplx<T>* __restrict__ w, const cplx<T>* __restrict__ r, const cplx<T>* __restrict__ W, long long stride,
                   const double* __restrict__ dots, const double* __restrict__ wn2, long long n,
                   double* __restrict__ partials, unsigned int* __restrict__ counter, double* __restrict__ out, XComm* xc) {
    using C = cplx<T>;
    __shared__ C s_beta[NJ > 0 ? NJ : 1];
    if ((int)threadIdx.x < NJ) {
        const double d = wn2[threadIdx.x];
        s_beta[threadIdx.x] = d > 0.0 ? mk<T>((T)(-dots[2 * threadIdx.x] / d), (T)(-dots[2 * threadIdx.x + 1] / d)) : mk<T>(0, 0);
    }
    __syncthreads();
    double red[4] = {0.0, 0.0, 0.0, 0.0};
    const long long nthreads = (long long)gridDim.x * blockDim.x;
    for (long long e0 = blockIdx.x * (long long)blockDim.x + threadIdx.x; e0 < n; e0 += nthreads * U) {
        C wv[U], rv[U], Wv[U][NJ > 0 ? NJ : 1];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long e = e0 + u * nthreads;
            if (e < n) {
                wv[u] = w[e]; rv[u] = __ldg(r + e);
#pragma unroll
                for (int j = 0; j < NJ; ++j) Wv[u][j] = __ldg(W + (size_t)j * stride + e);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long e = e0 + u * nthreads;
            if (e < n) {
#pragma unroll
                for (int j = 0; j < NJ; ++j) cfma(wv[u], s_beta[j], Wv[u][j]);
                w[e] = wv[u];
                red[0] += (double)wv[u].x * wv[u].x + (double)wv[u].y * wv[u].y;
                red[1] += (double)wv[u].x * rv[u].x + (double)wv[u].y * rv[u].y;       // <w, r> = conj(w) r
                red[2] += (double)wv[u].x * rv[u].y - (double)wv[u].y * rv[u].x;
            }
        }
    }
    grid_reduce<4, BL_THREADS>(red, partials, counter, out, blockIdx.x, gridDim.x, xc);
}

template <typename T>
int launch_ortho_w(mg2d_ctx* ctx, void* w, const void* r, const void* W, long long stride, int nj, const double* dots,
                   const double* wn2, long long nelem, double* out, cudaStream_t st) {
    using C = cplx<T>;
    XComm* xc = ctx->xreduce ? ctx->xcomm : nullptr;
#define OW(NJ, U) gcr_ortho_w_kernel<T, NJ, U><<<stream_grid(ctx, nelem, U), BL_THREADS, 0, st>>>((C*)w, (const C*)r, (const C*)W, stride, dots, wn2, nelem, ctx->partials, ctx->counter, out, xc)
    switch (nj) {
        case 0: OW(0, 4); break;
        case 1: OW(1, 4); break;
        case 2: OW(2, 2); break;
        case 3: OW(3, 2); break;
        case 4: OW(4, 2); break;
        case 5: OW(5, 1); break;
        case 6: OW(6, 1); break;
        case 7: OW(7, 1); break;
        default: OW(8, 1); break;
    }
#undef OW
    return mg2d_check_launch(ctx, "mg2d_gcr_ortho");
}

template <typename T>
__global__ void __launch_bounds__(BL_THREADS)
gcr_step_kernel(cplx<T>* __restrict__ x, cplx<T>* __restrict__ r, const cplx<T>* __restrict__ z, const cplx<T>* __restrict__ w,
                const double* __restrict__ wr, double* __restrict__ wn2_slot, long long n, double* __restrict__ partials,
                unsigned int* __restrict__ counter, double* __restrict__ out, XComm* xc) {
    using C = cplx<T>;
    const double d = wr[0];                       // wr = { |w|^2, Re<w,r>, Im<w,r> } as written by gcr_ortho_kernel
    const C a = d > 0.0 ? mk<T>((T)(wr[1] / d), (T)(wr[2] / d)) : mk<T>(0, 0);
    const C na = mk<T>(-a.x, -a.y);
    if (wn2_slot && blockIdx.x == 0 && threadIdx.x == 0) *wn2_slot = d;      // |w_slot|^2 for the projections of later iterations
    double red[1] = {0.0};
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        C xv = x[e], rv = r[e];
        cfma(xv, a, __ldg(z + e));
        cfma(rv, na, __ldg(w + e));
        x[e] = xv; r[e] = rv;
        red[0] += (double)rv.x * rv.x + (double)rv.y * rv.y;
    }
    grid_reduce<1, BL_THREADS>(red, partials, counter, out, blockIdx.x, gridDim.x, xc);
}
// Lazy solution update.  With zh_j = z_j - sum_{i<j} b_ij zh_i (what gcr_ortho_kernel does to z when it is given one) the
// orthogonalised direction is a combination zh_j = sum_{i<=j} c_ij z_i of the RAW preconditioned residuals, c_.j = e_j -
// sum_{i<j} b_ij c_.i, and the solution after the cycle is x + sum_i g_i z_i with g_i = sum_j a_j c_ij.  The 8 x 8
// recursion runs in one thread; the vectors z_i are then never rewritten and x is touched once per restart cycle
// (gcr_xupdate_kernel) instead of every iteration: (2j+9) instead of (3j+14) vector passes in iteration j of a cycle.
// coef (doubles): c[i][j] at 2*(8*i+j), g[i] at 128 + 2*i.
template <typename T>
__global__ void __launch_bounds__(BL_THREADS)
gcr_step_lazy_kernel(cplx<T>* __restrict__ r, const cplx<T>* __restrict__ w, const double* __restrict__ wr,
                     double* __restrict__ wn2_slot, const double* __restrict__ dots, const double* __restrict__ wn2, int nj,
                     double* __restrict__ coef, long long n, double* __restrict__ partials, unsigned int* __restrict__ counter,
                     double* __restrict__ out, XComm* xc) {
    using C = cplx<T>;
    const double d = wr[0];
    const double ar = d > 0.0 ? wr[1] / d : 0.0, ai = d > 0.0 ? wr[2] / d : 0.0;
    const C na = mk<T>((T)-ar, (T)-ai);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        *wn2_slot = d;
        double cr[GCR_MAXJ], ci[GCR_MAXJ];
        for (int i = 0; i < GCR_MAXJ; ++i) { cr[i] = (i == nj) ? 1.0 : 0.0; ci[i] = 0.0; }
        for (int i = 0; i < nj; ++i) {
            const double di = wn2[i];
            const double br = di > 0.0 ? dots[2 * i] / di : 0.0, bi = di > 0.0 ? dots[2 * i + 1] / di : 0.0;
            for (int l = 0; l <= i; ++l) {                       // c_.j -= b_ij c_.i  (column i has entries l <= i)
                const double xr = coef[2 * (8 * l + i)], xi = coef[2 * (8 * l + i) + 1];
                cr[l] -= br * xr - bi * xi;
                ci[l] -= br * xi + bi * xr;
            }
        }
        for (int l = 0; l < GCR_MAXJ; ++l) {
            coef[2 * (8 * l + nj)] = cr[l]; coef[2 * (8 * l + nj) + 1] = ci[l];
            const double gr = (nj == 0) ? 0.0 : coef[128 + 2 * l], gi = (nj == 0) ? 0.0 : coef[128 + 2 * l + 1];
            coef[128 + 2 * l] = gr + (ar * cr[l] - ai * ci[l]);
            coef[128 + 2 * l + 1] = gi + (ar * ci[l] + ai * cr[l]);
        }
    }
    double red[1] = {0.0};
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        C rv = r[e];
        cfma(rv, na, __ldg(w + e));
        r[e] = rv;
        red[0] += (double)rv.x * rv.x + (double)rv.y * rv.y;
    }
    grid_reduce<1, BL_THREADS>(red, partials, counter, out, blockIdx.x, gridDim.x, xc);
}

template <typename T>
__global__ void __launch_bounds__(BL_THREADS)
gcr_xupdate_kernel(cplx<T>* __restrict__ x, const cplx<T>* __restrict__ Z, long long stride, int nj,
                   const double* __restrict__ coef, long long n) {
    using C = cplx<T>;
    C g[GCR_MAXJ];
#pragma unroll
    for (int j = 0; j < GCR_MAXJ; ++j) g[j] = (j < nj) ? mk<T>((T)coef[128 + 2 * j], (T)coef[128 + 2 * j + 1]) : mk<T>(0, 0);
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        C xv = x[e];
#pragma unroll
        for (int j = 0; j < GCR_MAXJ; ++j)
            if (j < nj) cfma(xv, g[j], __ldg(Z + (size_t)j * stride + e));
        x[e] = xv;
    }
}
}  // namespace

extern "C" int mg2d_gcr_step_lazy(mg2d_ctx* ctx, void* r, const void* w, const double* wr, double* wn2_slot, const double* dots,
                                  const double* wn2, int nj, double* coef, long long nelem, int dtype, double* out, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!r || !w || !wr || !wn2_slot || !coef || !out || nelem < 1 || nj < 0 || nj >= GCR_MAXJ || (nj > 0 && (!dots || !wn2)))
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_gcr_step_lazy: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = stream_grid(ctx, nelem);
    XComm* xc = ctx->xreduce ? ctx->xcomm : nullptr;
    DISPATCH_T(dtype,
        (gcr_step_lazy_kernel<double><<<grid, BL_THREADS, 0, st>>>((double2*)r, (const double2*)w, wr, wn2_slot, dots, wn2, nj, coef, nelem, ctx->partials, ctx->counter, out, xc)),
        (gcr_step_lazy_kernel<float><<<grid, BL_THREADS, 0, st>>>((float2*)r, (const float2*)w, wr, wn2_slot, dots, wn2, nj, coef, nelem, ctx->partials, ctx->counter, out, xc)),
        "mg2d_gcr_step_lazy");
}

extern "C" int mg2d_gcr_xupdate(mg2d_ctx* ctx, void* x, const void* Z, long long stride, int nj, const double* coef, long long nelem,
                                int dtype, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!x || !Z || !coef || nelem < 1 || nj < 1 || nj > GCR_MAXJ) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_gcr_xupdate: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = stream_grid(ctx, nelem);
    DISPATCH_T(dtype,
        (gcr_xupdate_kernel<double><<<grid, BL_THREADS, 0, st>>>((double2*)x, (const double2*)Z, stride, nj, coef, nelem)),
        (gcr_xupdate_kernel<float><<<grid, BL_THREADS, 0, st>>>((float2*)x, (const float2*)Z, stride, nj, coef, nelem)),
        "mg2d_gcr_xupdate");
}

extern "C" int mg2d_gcr_dots(mg2d_ctx* ctx, const void* W, long long stride, int nj, const void* w, long long nelem, int dtype,
                             double* out, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!W || !w || !out || nj < 1 || nj > GCR_MAXJ || nelem < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_gcr_dots: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MG2D_C128) return launch_dots_nj<double>(ctx, W, stride, nj, w, nelem, out, st);
    if (dtype == MG2D_C64) return launch_dots_nj<float>(ctx, W, stride, nj, w, nelem, out, st);
    return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_gcr_dots: bad dtype");
}

extern "C" int mg2d_gcr_ortho(mg2d_ctx* ctx, void* w, void* z, const void* r, const void* W, const void* Z, long long stride, int nj,
                              const double* dots, const double* wn2, long long nelem, int dtype, double* out, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!w || !r || !out || nj < 0 || nj > GCR_MAXJ || nelem < 1 || (nj > 0 && (!W || (z && !Z) || !dots || !wn2)))
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_gcr_ortho: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = stream_grid(ctx, nelem);
    if (!z) {
        if (dtype == MG2D_C128) return launch_ortho_w<double>(ctx, w, r, W, stride, nj, dots, wn2, nelem, out, st);
        if (dtype == MG2D_C64) return launch_ortho_w<float>(ctx, w, r, W, stride, nj, dots, wn2, nelem, out, st);
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_gcr_ortho: bad dtype");
    }
    XComm* xc = ctx->xreduce ? ctx->xcomm : nullptr;
    DISPATCH_T(dtype,
        (gcr_ortho_kernel<double><<<grid, BL_THREADS, 0, st>>>((double2*)w, (double2*)z, (const double2*)r, (const double2*)W, (const double2*)Z, stride, nj, dots, wn2, nelem, ctx->partials, ctx->counter, out, xc)),
        (gcr_ortho_kernel<float><<<grid, BL_THREADS, 0, st>>>((float2*)w, (float2*)z, (const float2*)r, (const float2*)W, (const float2*)Z, stride, nj, dots, wn2, nelem, ctx->partials, ctx->counter, out, xc)),
        "mg2d_gcr_ortho");
}

extern "C" int mg2d_gcr_step(mg2d_ctx* ctx, void* x, void* r, const void* z, const void* w, const double* wr, double* wn2_slot,
                             long long nelem, int dtype, double* out, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!x || !r || !z || !w || !wr || !out || nelem < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_gcr_step: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = stream_grid(ctx, nelem);
    XComm* xc = ctx->xreduce ? ctx->xcomm : nullptr;
    DISPATCH_T(dtype,
        (gcr_step_kernel<double><<<grid, BL_THREADS, 0, st>>>((double2*)x, (double2*)r, (const double2*)z, (const double2*)w, wr, wn2_slot, nelem, ctx->partials, ctx->counter, out, xc)),
        (gcr_step_kernel<float><<<grid, BL_THREADS, 0, st>>>((float2*)x, (float2*)r, (const float2*)z, (const float2*)w, wr, wn2_slot, nelem, ctx->partials, ctx->counter, out, xc)),
        "mg2d_gcr_step");
}

// =========================================================================================================
// Peer-to-peer halo exchange over NVLink (multi-GPU strips): ONE kernel per exchange that (1) tells both
// neighbours their previous rows were consumed, (2) waits for the neighbours' acknowledgements, (3) stores
// this rank's boundary rows straight into the neighbours' halo buffers (mapped peer memory, CUDA IPC),
// (4) publishes the new epoch with a system-scope release and (5) waits for both neighbours' rows.
// No NCCL call, no host involvement; the epoch counter lives in device memory so the kernel can be replayed
// from a CUDA graph.  A bounded spin turns a lost peer into an error flag instead of a hang.
// =========================================================================================================
namespace {

// first/last: this rank's boundary rows (nvec pieces of row16 16-byte words, src_stride16 apart);
// next_lo / prev_hi: the neighbours' halo buffers; slots: mine and the two neighbours'.
// HX_CTAS CTAs share the copy; none depends on another one being resident (each spins on remote-written flags
// only), the last CTA to finish its stores publishes the epoch and waits for the incoming rows.
constexpr int HX_CTAS = 8;
constexpr int HX_THREADS = 512;

__global__ void __launch_bounds__(HX_THREADS)
halo_exchange_kernel(const uint4* __restrict__ first, const uint4* __restrict__ last, long long src_stride16,
                     long long row16, int nvec, uint4* __restrict__ next_lo, uint4* __restrict__ prev_hi,
                     HaloSlot* mine, HaloSlot* prev, HaloSlot* next, int relaxed) {
    __shared__ unsigned long long s_epoch;
    __shared__ int s_ok, s_last;
    if (threadIdx.x == 0) {
        const unsigned long long e = mine->epoch;     // only advanced after every CTA of this launch has arrived
        s_epoch = e;
        if (blockIdx.x == 0) {
            // I am prev's "next": its rows of epoch e (my lo_buf) are consumed (by kernels that completed before this launch)
            publish2(&prev->ack_next, &next->ack_prev, e, relaxed);
        }
        s_ok = spin_until(&mine->ack_next, e) && spin_until(&mine->ack_prev, e);
    }
    __syncthreads();
    const unsigned long long e = s_epoch;
    if (s_ok) {
        const long long total = (long long)nvec * row16;
        for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
            const long long v = k / row16, c = k - v * row16;
            next_lo[k] = last[v * src_stride16 + c];
            prev_hi[k] = first[v * src_stride16 + c];
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        if (!s_ok) atomicExch(&mine->error, 1ull);
        const unsigned long long t = atomicAdd(&mine->ticket, 1ull);
        s_last = (t == (unsigned long long)gridDim.x - 1);
    }
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        __threadfence_system();
        mine->ticket = 0;
        // a time-out anywhere in this launch poisons the exchange: the neighbours get an epoch they can recognise
        // (all-ones) instead of stale rows published as fresh, and the error word stays set for the host to raise on
        const bool failed = ld_acquire_sys(&mine->error) != 0ull;
        if (failed) {
            st_release_sys(&next->flag_lo, ~0ull);
            st_release_sys(&prev->flag_hi, ~0ull);
        } else {
            publish2(&next->flag_lo, &prev->flag_hi, e + 1, relaxed);
            const bool ok = spin_until(&mine->flag_lo, e + 1) && spin_until(&mine->flag_hi, e + 1);
            if (!ok || ld_acquire_sys(&mine->flag_lo) == ~0ull || ld_acquire_sys(&mine->flag_hi) == ~0ull) mine->error = 1;
        }
        mine->epoch = e + 1;
    }
}

// standalone all-reduce of n <= MG2D_XRED_MAX doubles in place (batched reductions that are not fused into their kernel)
__global__ void __launch_bounds__(128) xcomm_allreduce_kernel(XComm* xc, double* buf, int n) {
    __shared__ double s_v[MG2D_XRED_MAX];
    if ((int)threadIdx.x < n) s_v[threadIdx.x] = buf[threadIdx.x];
    __syncthreads();
    xcomm_allreduce(xc, s_v, n, buf);
}

}  // namespace

extern "C" int mg2d_ipc_alloc(mg2d_ctx* ctx, long long bytes, void** ptr, void* handle64) {
    if (!ctx) return MG2D_EINVAL;
    if (!ptr || !handle64 || bytes < 1) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_ipc_alloc: bad argument");
    cudaIpcMemHandle_t h;
    if (cudaMalloc(ptr, (size_t)bytes) != cudaSuccess || cudaMemset(*ptr, 0, (size_t)bytes) != cudaSuccess ||
        cudaIpcGetMemHandle(&h, *ptr) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) {
        snprintf(ctx->err, sizeof(ctx->err), "mg2d_ipc_alloc: %s", cudaGetErrorString(cudaGetLastError()));
        return MG2D_ECUDA;
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "ipc handle size");
    memcpy(handle64, &h, 64);
    return MG2D_OK;
}

extern "C" int mg2d_ipc_open(mg2d_ctx* ctx, const void* handle64, void** ptr) {
    if (!ctx) return MG2D_EINVAL;
    if (!ptr || !handle64) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_ipc_open: bad argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    cudaError_t e = cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { snprintf(ctx->err, sizeof(ctx->err), "mg2d_ipc_open: %s", cudaGetErrorString(e)); cudaGetLastError(); return MG2D_ECUDA; }
    return MG2D_OK;
}

extern "C" int mg2d_halo_exchange(mg2d_ctx* ctx, const void* first, const void* last, long long src_stride_bytes,
                                  long long row_bytes, int nvec, void* next_lo, void* prev_hi, void* slot_mine,
                                  void* slot_prev, void* slot_next, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!first || !last || !next_lo || !prev_hi || !slot_mine || !slot_prev || !slot_next || nvec < 1 || row_bytes < 16 ||
        (row_bytes & 15) || (src_stride_bytes & 15))
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_halo_exchange: bad argument (rows must be multiples of 16 bytes)");
    halo_exchange_kernel<<<(nvec * (row_bytes / 16) > 4096 ? HX_CTAS : 1), HX_THREADS, 0, (cudaStream_t)stream>>>((const uint4*)first, (const uint4*)last, src_stride_bytes / 16,
        row_bytes / 16, nvec, (uint4*)next_lo, (uint4*)prev_hi, (HaloSlot*)slot_mine, (HaloSlot*)slot_prev, (HaloSlot*)slot_next, mg2d_publish_relaxed());
    return mg2d_check_launch(ctx, "mg2d_halo_exchange");
}

// ---- cross-GPU reductions fused into the kernels -------------------------------------------------------------------
extern "C" int mg2d_comm_create(mg2d_ctx* ctx, int world, int rank, void* const* area_ptrs, void** desc_out) {
    if (!ctx) return MG2D_EINVAL;
    if (world < 1 || world > MG2D_MAX_RANKS || rank < 0 || rank >= world || !area_ptrs || !desc_out)
        return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_comm_create: bad argument (at most 8 ranks)");
    XComm h;
    memset(&h, 0, sizeof(h));
    h.world = world; h.rank = rank; h.relaxed = mg2d_publish_relaxed();
    for (int q = 0; q < world; ++q) {
        if (!area_ptrs[q]) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_comm_create: null mailbox pointer");
        h.area[q] = (XRedArea*)area_ptrs[q];
    }
    XComm* d = nullptr;
    if (cudaMalloc(&d, sizeof(XComm)) != cudaSuccess || cudaMemcpy(d, &h, sizeof(XComm), cudaMemcpyHostToDevice) != cudaSuccess)
        return mg2d_fail(ctx, MG2D_ECUDA, "mg2d_comm_create: allocation failed");
    *desc_out = d;
    ctx->xcomm = d;
    return MG2D_OK;
}

extern "C" int mg2d_comm_attach(mg2d_ctx* ctx, void* desc) {
    if (!ctx) return MG2D_EINVAL;
    ctx->xcomm = (XComm*)desc;
    if (!desc) ctx->xreduce = 0;
    return MG2D_OK;
}

extern "C" int mg2d_comm_reduce(mg2d_ctx* ctx, int on) {
    if (!ctx) return MG2D_EINVAL;
    if (on && !ctx->xcomm) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_comm_reduce: no communicator attached");
    ctx->xreduce = on ? 1 : 0;
    return MG2D_OK;
}

extern "C" int mg2d_comm_mailbox_bytes(void) { return (int)sizeof(XRedArea); }

extern "C" int mg2d_comm_error(mg2d_ctx* ctx, void* desc, long long* out) {
    if (!ctx) return MG2D_EINVAL;
    if (!desc || !out) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_comm_error: bad argument");
    XComm h;
    if (cudaMemcpy(&h, desc, sizeof(XComm), cudaMemcpyDeviceToHost) != cudaSuccess) return mg2d_fail(ctx, MG2D_ECUDA, "mg2d_comm_error: copy failed");
    *out = (long long)h.error;
    return MG2D_OK;
}

extern "C" int mg2d_allreduce(mg2d_ctx* ctx, double* buf, int n, void* stream) {
    if (!ctx) return MG2D_EINVAL;
    if (!buf || n < 1 || n > MG2D_XRED_MAX || !ctx->xcomm) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_allreduce: bad argument / no communicator");
    xcomm_allreduce_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(ctx->xcomm, buf, n);
    return mg2d_check_launch(ctx, "mg2d_allreduce");
}

// sum of the error words of `nslots` halo slots (64-byte records starting at `slots`)
extern "C" int mg2d_halo_errors(mg2d_ctx* ctx, const void* slots, int nslots, long long* out) {
    if (!ctx) return MG2D_EINVAL;
    if (!slots || nslots < 0 || !out) return mg2d_fail(ctx, MG2D_EINVAL, "mg2d_halo_errors: bad argument");
    long long tot = 0;
    if (nslots > 0) {
        HaloSlot* h = new HaloSlot[nslots];
        if (cudaMemcpy(h, slots, (size_t)nslots * sizeof(HaloSlot), cudaMemcpyDeviceToHost) != cudaSuccess) {
            delete[] h;
            return mg2d_fail(ctx, MG2D_ECUDA, "mg2d_halo_errors: copy failed");
        }
        for (int i = 0; i < nslots; ++i) tot += (long long)h[i].error;
        delete[] h;
    }
    *out = tot;
    return MG2D_OK;
}
