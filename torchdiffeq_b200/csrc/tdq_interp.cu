// tdq_interp.cu -- dense output of an accepted step and the initial-step probe.
//
//   k_fit_eval     y_mid, the quartic's coefficients and the requested outputs   rk_common.py:363-369, interp.py:1-48
//   k_interp_eval  p((t - t0)/(t1 - t0)) from STORED coefficients                interp.py:25-48 (events, dense closures)
//   k_poly_eval    p(x) for a caller-supplied abscissa                           odeint.py:111-157
//   k_probe        y0 + h0*f0                                                    misc.py:66
//
// The fit is LAZY.  The reference fits an interpolant after every accepted step (rk_common.py:341) and uses it
// only when an output time falls inside the step.  Here the controller kernel knows, before the fit would
// run, whether any t[j] lies in (t0, t1] (or whether the caller keeps dense output / handles events); only
// then does k_fit_eval do anything: it reads the step's eight operands once, forms the coefficients in
// registers and writes the output rows directly -- coefficients go to memory only when the caller asked
// for them.  The arithmetic, and hence every output bit, is that of interp.py:17-22, :39-46.
#include "tdq_common.cuh"
#include "tdq_shape.cuh"

namespace {

constexpr int kThreads = 256;

// x = T((t - t0)/(t1 - t0)) in float64 then cast (interp.py:39-40); running powers, not Horner (interp.py:42-46).
template <typename T> __device__ __forceinline__ T eval_poly(T e, T d, T cq, T b, T a, T x) {
    using A = Ar<T>;
    T total = A::add(e, A::mul(x, d));
    T xp = A::mul(x, x);
    total = A::add(total, A::mul(xp, cq));
    xp = A::mul(xp, x);
    total = A::add(total, A::mul(xp, b));
    xp = A::mul(xp, x);
    total = A::add(total, A::mul(xp, a));
    return total;
}

template <typename T, int NK, bool VECTOR, bool STORE>
__global__ void __launch_bounds__(kThreads)
k_fit_eval(const TdqCtrl *__restrict__ c, const T *__restrict__ y1p, const T *__restrict__ kSp, KPtrs kmid,
           T *__restrict__ ce, T *__restrict__ cd, T *__restrict__ cc, T *__restrict__ cb, T *__restrict__ ca,
           T *__restrict__ solution, size_t n) {
    if (!c->fit_now) return;
    using A = Ar<T>;
    const T *y0p = reinterpret_cast<const T *>(c->y0_prev);
    const T *k0p = reinterpret_cast<const T *>(c->k0_prev);
    T mf[NK];
    const T *km[NK];
#pragma unroll
    for (int m = 0; m < NK; ++m) {
        mf[m] = (T)c->fit_mcoef[m];
        km[m] = reinterpret_cast<const T *>(kmid.p[m] ? kmid.p[m] : (const void *)k0p);
    }
    const T sdt = (T)c->fit_sdt;
    const T two_sdt = A::mul((T)2, sdt);                    // 2 * dt (exact)
    const int lo = c->emit_lo, hi = c->emit_hi;
    const double t0 = c->t0, t1 = c->t1;

    auto fit = [&](T y0v, T y1v, T f0, T f1, const T *kv, T &e, T &d, T &cq, T &b, T &a) {
        T acc = A::mul(kv[0], mf[0]);
#pragma unroll
        for (int m = 1; m < NK; ++m) acc = A::add(acc, A::mul(kv[m], mf[m]));
        const T ymid = A::add(y0v, acc);
        // a = 2*dt*(f1 - f0) - 8*(y1 + y0) + 16*y_mid
        a = A::add(A::sub(A::mul(two_sdt, A::sub(f1, f0)), A::mul((T)8, A::add(y1v, y0v))), A::mul((T)16, ymid));
        // b = dt*(5*f0 - 3*f1) + 18*y0 + 14*y1 - 32*y_mid
        b = A::sub(A::add(A::add(A::mul(sdt, A::sub(A::mul((T)5, f0), A::mul((T)3, f1))), A::mul((T)18, y0v)),
                          A::mul((T)14, y1v)),
                   A::mul((T)32, ymid));
        // c = dt*(f1 - 4*f0) - 11*y0 - 5*y1 + 16*y_mid
        cq = A::add(A::sub(A::sub(A::mul(sdt, A::sub(f1, A::mul((T)4, f0))), A::mul((T)11, y0v)), A::mul((T)5, y1v)),
                    A::mul((T)16, ymid));
        d = A::mul(sdt, f0);
        e = y0v;
    };
    auto xof = [&](int j) -> T { return (T)((c->t_out[j] - t0) / (t1 - t0)); };

    if (VECTOR) {
        using V = Vec<T>;
        const size_t nvec = n / V::N;
        for (size_t v = (size_t)blockIdx.x * kThreads + threadIdx.x; v < nvec; v += (size_t)gridDim.x * kThreads) {
            const size_t i0 = v * V::N;
            V a0 = ld_stream<T>(y0p + i0), a1 = ld_stream<T>(y1p + i0);
            V f0 = ld_stream<T>(k0p + i0), f1 = ld_stream<T>(kSp + i0);
            V kv[NK];
#pragma unroll
            for (int m = 0; m < NK; ++m) kv[m] = ld_stream<T>(km[m] + i0);
            V re, rd, rc, rb, ra;
#pragma unroll
            for (int e = 0; e < V::N; ++e) {
                T ke[NK];
#pragma unroll
                for (int m = 0; m < NK; ++m) ke[m] = kv[m].v[e];
                fit(a0.v[e], a1.v[e], f0.v[e], f1.v[e], ke, re.v[e], rd.v[e], rc.v[e], rb.v[e], ra.v[e]);
            }
            if (STORE) {
                st_vec<T>(ce + i0, re); st_vec<T>(cd + i0, rd); st_vec<T>(cc + i0, rc);
                st_vec<T>(cb + i0, rb); st_vec<T>(ca + i0, ra);
            }
            for (int j = lo; j < hi; ++j) {
                const T x = xof(j);
                V r;
#pragma unroll
                for (int l = 0; l < V::N; ++l) r.v[l] = eval_poly<T>(re.v[l], rd.v[l], rc.v[l], rb.v[l], ra.v[l], x);
                st_vec<T>(solution + (size_t)j * n + i0, r);
            }
        }
        if (blockIdx.x == gridDim.x - 1) {
            const size_t i = nvec * V::N + threadIdx.x;
            if (i < n) {
                T ke[NK];
#pragma unroll
                for (int m = 0; m < NK; ++m) ke[m] = km[m][i];
                T e, d, cq, b, a;
                fit(y0p[i], y1p[i], k0p[i], kSp[i], ke, e, d, cq, b, a);
                if (STORE) { ce[i] = e; cd[i] = d; cc[i] = cq; cb[i] = b; ca[i] = a; }
                for (int j = lo; j < hi; ++j) solution[(size_t)j * n + i] = eval_poly<T>(e, d, cq, b, a, xof(j));
            }
        }
    } else {
        for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (size_t)gridDim.x * kThreads) {
            T ke[NK];
#pragma unroll
            for (int m = 0; m < NK; ++m) ke[m] = km[m][i];
            T e, d, cq, b, a;
            fit(y0p[i], y1p[i], k0p[i], kSp[i], ke, e, d, cq, b, a);
            if (STORE) { ce[i] = e; cd[i] = d; cc[i] = cq; cb[i] = b; ca[i] = a; }
            for (int j = lo; j < hi; ++j) solution[(size_t)j * n + i] = eval_poly<T>(e, d, cq, b, a, xof(j));
        }
    }
}

template <typename T, int NK>
int launch_fit(const TdqCtrl *c, const void *y1, const void *kS, const KPtrs &kmid, void *const *coeff, void *solution,
               size_t n, bool vec, cudaStream_t st) {
    size_t blocks = ((vec ? n / Vec<T>::N : n) + kThreads - 1) / kThreads;
    // persistent, two blocks per SM: 64 KB of loads in flight per SM saturate HBM when the fit runs, and the usual no-op
    // launch (73 of 74 attempts of configs[1]) costs a few hundred blocks' worth of scheduling less
    const size_t cap = (size_t)tdq_sm_count() * 2;
    if (blocks > cap) blocks = cap;
    if (blocks == 0) blocks = 1;
    T *co[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    if (coeff) for (int i = 0; i < 5; ++i) co[i] = (T *)coeff[i];
#define TDQ_L(V_, S_) k_fit_eval<T, NK, V_, S_><<<(unsigned)blocks, kThreads, 0, st>>>( \
        c, (const T *)y1, (const T *)kS, kmid, co[0], co[1], co[2], co[3], co[4], (T *)solution, n)
    if (vec) { if (coeff) TDQ_L(true, true); else TDQ_L(true, false); }
    else     { if (coeff) TDQ_L(false, true); else TDQ_L(false, false); }
#undef TDQ_L
    return 0;
}

template <typename T>
int dispatch_fit(int nk, const TdqCtrl *c, const void *y1, const void *kS, const KPtrs &kmid, void *const *coeff,
                 void *solution, size_t n, bool vec, cudaStream_t st) {
    switch (nk) {
#define TDQ_CASE(N) case N: return launch_fit<T, N>(c, y1, kS, kmid, coeff, solution, n, vec, st);
        TDQ_CASE(1) TDQ_CASE(2) TDQ_CASE(3) TDQ_CASE(4) TDQ_CASE(5) TDQ_CASE(6) TDQ_CASE(7) TDQ_CASE(8)
        TDQ_CASE(9) TDQ_CASE(10) TDQ_CASE(11) TDQ_CASE(12) TDQ_CASE(13) TDQ_CASE(14) TDQ_CASE(15)
        TDQ_CASE(16) TDQ_CASE(17)
#undef TDQ_CASE
    }
    return -1;
}

// p(x) for a caller-supplied abscissa x (float64, cast to T like interp.py:39-40); used by dense-output
// closures that keep their own (t0, t1, coefficients) per accepted step (odeint.py:111-157).
template <typename T>
__global__ void __launch_bounds__(kThreads)
k_poly_eval(const T *__restrict__ ce, const T *__restrict__ cd, const T *__restrict__ cc, const T *__restrict__ cb,
            const T *__restrict__ ca, T *__restrict__ out, double x64, size_t n) {
    const T x = (T)x64;
    for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (size_t)gridDim.x * kThreads)
        out[i] = eval_poly<T>(ce[i], cd[i], cc[i], cb[i], ca[i], x);
}

// The stored interpolant of the last accepted step at a device-resident time (event bisection).
template <typename T>
__global__ void __launch_bounds__(kThreads)
k_interp_eval_at(const TdqCtrl *__restrict__ c, const T *__restrict__ ce, const T *__restrict__ cd,
                 const T *__restrict__ cc, const T *__restrict__ cb, const T *__restrict__ ca, T *__restrict__ out,
                 const double *__restrict__ t_at, size_t n) {
    const double t0 = c->t0, t1 = c->t1;
    const T x = (T)((*t_at - t0) / (t1 - t0));
    for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (size_t)gridDim.x * kThreads)
        out[i] = eval_poly<T>(ce[i], cd[i], cc[i], cb[i], ca[i], x);
}

// y_probe = y0 + h0*f0 with f0 = s*k0 (misc.py:66)
template <typename T>
__global__ void __launch_bounds__(kThreads)
k_probe(const TdqCtrl *__restrict__ c, T *__restrict__ out, const T *y0, const T *f0, size_t n) {
    using A = Ar<T>;
    if (y0 == nullptr) y0 = reinterpret_cast<const T *>(c->y0_cur);
    if (f0 == nullptr) f0 = reinterpret_cast<const T *>(c->k0_cur);
    const T h = A::mul((T)c->t_sign, (T)c->h0);
    for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (size_t)gridDim.x * kThreads)
        out[i] = A::add(y0[i], A::mul(h, f0[i]));
}

}  // namespace

extern "C" {

int tdq_initial_step_probe(void *ctrl_dev, int32_t dtype, void *y_probe, const void *y0, const void *f0, size_t n,
                           void *stream) {
    TDQ_REQUIRE(ctrl_dev && y_probe, "null argument");
    TDQ_REAL_VIEW(dtype, n);
    if (n == 0) return TDQ_OK;
    size_t blocks = (n + kThreads - 1) / kThreads;
    if (blocks > (size_t)tdq_sm_count() * 16) blocks = (size_t)tdq_sm_count() * 16;
    TDQ_DISPATCH_T(dtype, (k_probe<T><<<(unsigned)blocks, kThreads, 0, (cudaStream_t)stream>>>(
                               (const TdqCtrl *)ctrl_dev, (T *)y_probe, (const T *)y0, (const T *)f0, n)));
    TDQ_CHECK_CUDA(cudaGetLastError());
    return TDQ_OK;
}

int tdq_interp_fit_eval(void *ctrl_dev, const tdq_tableau *tab, int32_t dtype, const void *y1, const void *const *k,
                        void *const *coeff, void *solution, size_t n, void *stream) {
    TDQ_REQUIRE(ctrl_dev && tab && y1 && k && solution, "null argument");
    TDQ_REAL_VIEW(dtype, n);
    TdqHostShape hs;
    tdq_shape_from_tableau(tab, &hs);
    const int S = hs.n_stages;
    const int nk = hs.mid_nnz;
    TDQ_REQUIRE(nk >= 1, "tableau has no mid-point weights");
    TDQ_REQUIRE(k[S] != nullptr, "k_S is required");
    KPtrs kmid;
    memset(&kmid, 0, sizeof(kmid));
    bool vec = tdq_aligned16(y1) && tdq_aligned16(k[S]) && tdq_aligned16(solution) &&
               ((n * (dtype == TDQ_F32 ? 4 : 8)) % 16 == 0);
    for (int m = 0; m < nk; ++m) {
        const int j = hs.mid_idx[m];
        kmid.p[m] = k[j];
        TDQ_REQUIRE(kmid.p[m] != nullptr || j == 0, "missing stage slot for a non-zero mid-point weight");
        vec = vec && tdq_aligned16(kmid.p[m]);
    }
    if (coeff)
        for (int i = 0; i < 5; ++i) {
            TDQ_REQUIRE(coeff[i] != nullptr, "five coefficient buffers are required");
            vec = vec && tdq_aligned16(coeff[i]);
        }
    if (n == 0) return TDQ_OK;
    int rc = -1;
    TDQ_DISPATCH_T(dtype, rc = dispatch_fit<T>(nk, (const TdqCtrl *)ctrl_dev, y1, k[S], kmid, coeff, solution, n, vec,
                                               (cudaStream_t)stream));
    TDQ_REQUIRE(rc == 0, "unsupported number of mid-point terms");
    TDQ_CHECK_CUDA(cudaGetLastError());
    return TDQ_OK;
}

int tdq_poly_eval(int32_t dtype, const void *const *coeff, double x, void *out, size_t n, void *stream) {
    TDQ_REQUIRE(coeff && out, "null argument");
    TDQ_REAL_VIEW(dtype, n);
    for (int i = 0; i < 5; ++i) TDQ_REQUIRE(coeff[i] != nullptr, "five coefficient buffers are required");
    if (n == 0) return TDQ_OK;
    size_t blocks = (n + kThreads - 1) / kThreads;
    if (blocks > (size_t)tdq_sm_count() * 8) blocks = (size_t)tdq_sm_count() * 8;
    TDQ_DISPATCH_T(dtype, (k_poly_eval<T><<<(unsigned)blocks, kThreads, 0, (cudaStream_t)stream>>>(
                               (const T *)coeff[0], (const T *)coeff[1], (const T *)coeff[2], (const T *)coeff[3],
                               (const T *)coeff[4], (T *)out, x, n)));
    TDQ_CHECK_CUDA(cudaGetLastError());
    return TDQ_OK;
}

int tdq_interp_eval_at(void *ctrl_dev, int32_t dtype, const void *const *coeff, const double *t_dev, void *out,
                       size_t n, void *stream) {
    TDQ_REQUIRE(ctrl_dev && coeff && out && t_dev, "null argument");
    TDQ_REAL_VIEW(dtype, n);
    for (int i = 0; i < 5; ++i) TDQ_REQUIRE(coeff[i] != nullptr, "five coefficient buffers are required");
    if (n == 0) return TDQ_OK;
    size_t blocks = (n + kThreads - 1) / kThreads;
    if (blocks > (size_t)tdq_sm_count() * 8) blocks = (size_t)tdq_sm_count() * 8;
    TDQ_DISPATCH_T(dtype, (k_interp_eval_at<T><<<(unsigned)blocks, kThreads, 0, (cudaStream_t)stream>>>(
                               (const TdqCtrl *)ctrl_dev, (const T *)coeff[0], (const T *)coeff[1], (const T *)coeff[2],
                               (const T *)coeff[3], (const T *)coeff[4], (T *)out, t_dev, n)));
    TDQ_CHECK_CUDA(cudaGetLastError());
    return TDQ_OK;
}

}  // extern "C"
