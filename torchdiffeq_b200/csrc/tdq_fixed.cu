// tdq_fixed.cu -- fixed-grid RK4 (3/8 rule) and the augmented-state pack.
//
//   k_rk4        stage values and the final update of rk4_alt_step_func   rk_common.py:110-118, fixed_grid.py:24-29, solvers.py:115
//   k_fixed_emit outputs of one grid step by linear interpolation         solvers.py:117-125, :175-181
//   k_pack       concat + per-segment scale of the augmented dynamics     misc.py:137-145, :158-165, adjoint.py:94-105
//
// The step size comes from a device array indexed by a device step counter so that one captured
// step graph serves the whole grid.
#include "tdq_common.cuh"
#include "tdq_shape.cuh"

namespace {

constexpr int kThreads = 256;

// 1/3 as Python computes it (rk_common.py:94 `_one_third = 1 / 3`), then cast to T by torch when it
// multiplies a T tensor.
template <typename T, int WHICH>
__device__ __forceinline__ T rk_expr(T dt, T y, T a, T b, T c_, T d) {
    using A = Ar<T>;
    const T third = (T)(1.0 / 3.0);
    {
        if (WHICH == 1) return A::add(y, A::mul(A::mul(dt, a), third));                 // y0 + dt*k1*_one_third
        if (WHICH == 2) return A::add(y, A::mul(dt, A::sub(b, A::mul(a, third))));      // y0 + dt*(k2 - k1*_one_third)
        if (WHICH == 3) return A::add(y, A::mul(dt, A::add(A::sub(a, b), c_)));         // y0 + dt*(k1 - k2 + k3)
        if (WHICH == 4) {                                                               // y0 + (k1 + 3*(k2 + k3) + k4)*dt*0.125
            const T s = A::add(A::add(a, A::mul((T)3, A::add(b, c_))), d);
            return A::add(y, A::mul(A::mul(s, dt), (T)0.125));
        }
        // the other fixed-grid methods of fixed_grid.py:6-60 (rk_common.py:121-158)
        if (WHICH == 5) return A::add(y, A::mul(dt, a));                                // euler / midpoint final / heun2 stage: y0 + dt*k
        if (WHICH == 6) return A::add(y, A::mul(a, A::mul((T)0.5, dt)));                // midpoint stage: y0 + f0*half_dt
        if (WHICH == 7) return A::add(y, A::mul(dt, A::add(A::mul(a, (T)0.5), A::mul(b, (T)0.5))));   // heun2: y0 + dt*(k1/2 + k2/2)
        if (WHICH == 8) return A::add(y, A::mul(dt, A::mul(b, (T)(2.0 / 3.0))));        // heun3 stage 3: y0 + dt*(k1*0 + k2*2/3)
        // heun3 final: y0 + dt*(k1*1/4 + k2*0 + k3*3/4)
        return A::add(y, A::mul(dt, A::add(A::mul(a, (T)0.25), A::mul(c_, (T)0.75))));
    }
}

template <typename T, int WHICH, bool VECTOR>
__global__ void __launch_bounds__(kThreads)
k_rk4(T *__restrict__ out, const T *__restrict__ y0, const T *__restrict__ k1, const T *__restrict__ k2,
      const T *__restrict__ k3, const T *__restrict__ k4, const T *__restrict__ dt_arr,
      const int64_t *__restrict__ step, size_t n) {
    // which operands the expression reads (k1,k2,k3,k4)
    constexpr bool kA = WHICH != 8;
    constexpr bool kB = WHICH == 2 || WHICH == 3 || WHICH == 4 || WHICH == 7 || WHICH == 8;
    constexpr bool kC = WHICH == 3 || WHICH == 4 || WHICH == 9;
    constexpr bool kD = WHICH == 4;
    const T dt = dt_arr[step ? *step : 0];
    auto f = [&](T y, T a, T b, T c_, T d) -> T { return rk_expr<T, WHICH>(dt, y, a, b, c_, d); };
    if (VECTOR) {
        using V = Vec<T>;
        const size_t nvec = n / V::N;
        const size_t v = (size_t)blockIdx.x * kThreads + threadIdx.x;
        if (v < nvec) {
            const size_t i0 = v * V::N;
            V y = ld_stream<T>(y0 + i0), a, b, c_, d;
            if (kA) a = ld_stream<T>(k1 + i0);
            if (kB) b = ld_stream<T>(k2 + i0);
            if (kC) c_ = ld_stream<T>(k3 + i0);
            if (kD) d = ld_stream<T>(k4 + i0);
            V r;
#pragma unroll
            for (int e = 0; e < V::N; ++e)
                r.v[e] = f(y.v[e], kA ? a.v[e] : (T)0, kB ? b.v[e] : (T)0, kC ? c_.v[e] : (T)0, kD ? d.v[e] : (T)0);
            st_vec<T>(out + i0, r);
        }
        if (blockIdx.x == gridDim.x - 1) {
            const size_t i = nvec * V::N + threadIdx.x;
            if (i < n)
                out[i] = f(y0[i], kA ? k1[i] : (T)0, kB ? k2[i] : (T)0, kC ? k3[i] : (T)0, kD ? k4[i] : (T)0);
        }
    } else {
        for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (size_t)gridDim.x * kThreads)
            out[i] = f(y0[i], kA ? k1[i] : (T)0, kB ? k2[i] : (T)0, kC ? k3[i] : (T)0, kD ? k4[i] : (T)0);
    }
}

template <typename T, int WHICH>
void launch_rk4(void *out, const void *y0, const void *k1, const void *k2, const void *k3, const void *k4,
                const void *dt, const int64_t *step, size_t n, bool vec, cudaStream_t st) {
    if (vec) {
        const size_t nvec = n / Vec<T>::N;
        size_t blocks = (nvec + kThreads - 1) / kThreads;
        if (blocks == 0) blocks = 1;
        k_rk4<T, WHICH, true><<<(unsigned)blocks, kThreads, 0, st>>>((T *)out, (const T *)y0, (const T *)k1,
                                                                      (const T *)k2, (const T *)k3, (const T *)k4,
                                                                      (const T *)dt, step, n);
    } else {
        size_t blocks = (n + kThreads - 1) / kThreads;
        if (blocks == 0) blocks = 1;
        if (blocks > 148 * 16) blocks = 148 * 16;
        k_rk4<T, WHICH, false><<<(unsigned)blocks, kThreads, 0, st>>>((T *)out, (const T *)y0, (const T *)k1,
                                                                       (const T *)k2, (const T *)k3, (const T *)k4,
                                                                       (const T *)dt, step, n);
    }
}

// Linear-interpolation outputs of the step that just finished, then the carry y0 <- y1.
// mode 0: y0 (t == t0), 1: y1 (t == t1), 2: y0 + slope*(y1 - y0) (solvers.py:175-181).
// The last block to finish (ticket in step[1]) advances the device step counter and stages the next step's four
// func times -- every block has read step[0] by then, so no second launch is needed.
template <typename T>
__global__ void __launch_bounds__(kThreads)
k_fixed_emit(T *__restrict__ y0, const T *__restrict__ y1, T *__restrict__ solution,
             const int32_t *__restrict__ rec_begin, const int32_t *__restrict__ out_idx,
             const int32_t *__restrict__ mode, const T *__restrict__ slope, int64_t *step,
             const unsigned char *__restrict__ tst_all, unsigned char *__restrict__ tcur, int64_t n_steps, size_t n) {
    using A = Ar<T>;
    const int64_t s = step[0];
    const int lo = rec_begin[s], hi = rec_begin[s + 1];
    for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (size_t)gridDim.x * kThreads) {
        const T a = y0[i], b = y1[i];
        for (int r = lo; r < hi; ++r) {
            const int md = mode[r];
            solution[(size_t)out_idx[r] * n + i] = (md == 0) ? a : (md == 1) ? b : A::add(a, A::mul(slope[r], A::sub(b, a)));
        }
        y0[i] = b;                                            // solvers.py:126  y0 = y1
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        unsigned long long *ticket = reinterpret_cast<unsigned long long *>(step + 1);
        const unsigned long long t = atomicAdd(ticket, 1ull);
        if (t == gridDim.x - 1) {
            *ticket = 0ull;
            const int64_t nxt = s + 1;
            step[0] = nxt;
            if (nxt < n_steps)
                for (int b = 0; b < 4 * (int)sizeof(T); ++b) tcur[b] = tst_all[nxt * 4 * sizeof(T) + b];
        }
    }
}

// The LAST expression of a step (y1 = y0 + dy) fused with k_fixed_emit: y1 never goes to memory as a separate
// array -- it is formed in registers, the step's linear-interpolation outputs are written, and it replaces y0.
template <typename T, int WHICH>
__global__ void __launch_bounds__(kThreads)
k_final_emit(T *__restrict__ y0, const T *__restrict__ k1, const T *__restrict__ k2, const T *__restrict__ k3,
             const T *__restrict__ k4, const T *__restrict__ dt_arr, T *__restrict__ solution,
             const int32_t *__restrict__ rec_begin, const int32_t *__restrict__ out_idx,
             const int32_t *__restrict__ mode, const T *__restrict__ slope, int64_t *step,
             const unsigned char *__restrict__ tst_all, unsigned char *__restrict__ tcur, int64_t n_steps, size_t n) {
    using A = Ar<T>;
    constexpr bool kA = WHICH != 8;
    constexpr bool kB = WHICH == 4 || WHICH == 7;
    constexpr bool kC = WHICH == 4 || WHICH == 9;
    constexpr bool kD = WHICH == 4;
    const int64_t s = step[0];
    const T dt = dt_arr[s];
    const int lo = rec_begin[s], hi = rec_begin[s + 1];
    for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (size_t)gridDim.x * kThreads) {
        const T a = y0[i];
        const T b = rk_expr<T, WHICH>(dt, a, kA ? k1[i] : (T)0, kB ? k2[i] : (T)0, kC ? k3[i] : (T)0, kD ? k4[i] : (T)0);
        for (int r = lo; r < hi; ++r) {
            const int md = mode[r];
            solution[(size_t)out_idx[r] * n + i] = (md == 0) ? a : (md == 1) ? b : A::add(a, A::mul(slope[r], A::sub(b, a)));
        }
        y0[i] = b;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        unsigned long long *ticket = reinterpret_cast<unsigned long long *>(step + 1);
        const unsigned long long t = atomicAdd(ticket, 1ull);
        if (t == gridDim.x - 1) {
            *ticket = 0ull;
            const int64_t nxt = s + 1;
            step[0] = nxt;
            if (nxt < n_steps)
                for (int b = 0; b < 4 * (int)sizeof(T); ++b) tcur[b] = tst_all[nxt * 4 * sizeof(T) + b];
        }
    }
}

// Cubic Hermite outputs of one step (solvers.py:120-125, :166-173): for records r in [lo, hi)
//   solution[out_idx[r]] = ((c0*y0 + c1*f0) + c2*y1) + c3*f1,  c = (h00, h10*dt, h01, h11*dt) cast to T
// f0 / f1 are RAW func outputs; the reverse-time sign is already inside c1 and c3.
template <typename T>
__global__ void __launch_bounds__(kThreads)
k_fixed_emit_cubic(const T *__restrict__ y0, const T *__restrict__ y1, const T *__restrict__ f0,
                   const T *__restrict__ f1, T *__restrict__ solution, const int32_t *__restrict__ out_idx,
                   const T *__restrict__ coef, int lo, int hi, size_t n) {
    using A = Ar<T>;
    for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (size_t)gridDim.x * kThreads) {
        const T a = y0[i], b = y1[i], fa = f0[i], fb = f1[i];
        for (int r = lo; r < hi; ++r) {
            const T *c = coef + 4 * (size_t)r;
            const T v = A::add(A::add(A::add(A::mul(c[0], a), A::mul(c[1], fa)), A::mul(c[2], b)), A::mul(c[3], fb));
            solution[(size_t)out_idx[r] * n + i] = v;
        }
    }
}

// Generic linear combination for the multistep (Adams) predictor / corrector of fixed_adams.py:198-215:
//   out = [base +] ((x_0*c_0 + x_1*c_1) + x_2*c_2) + ...      products and sums rounded separately, ascending order,
// the first product initialises the sum (Python's sum() starts from 0 + x_0*c_0 = x_0*c_0 exactly).
struct LinArgs {
    const void *x[TDQ_MAX_K];
    double c[TDQ_MAX_K];
};

template <typename T>
__global__ void __launch_bounds__(kThreads)
k_lincomb(T *__restrict__ out, const T *base, LinArgs a, int n_terms, size_t n) {
    using A = Ar<T>;
    for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (size_t)gridDim.x * kThreads) {
        T acc = A::mul(reinterpret_cast<const T *>(a.x[0])[i], (T)a.c[0]);
        for (int m = 1; m < n_terms; ++m) acc = A::add(acc, A::mul(reinterpret_cast<const T *>(a.x[m])[i], (T)a.c[m]));
        out[i] = base ? A::add(base[i], acc) : acc;
    }
}

struct PackArgs {
    const void *src[TDQ_MAX_SEGS];
    int64_t off[TDQ_MAX_SEGS];
    int64_t len[TDQ_MAX_SEGS];
    double scale[TDQ_MAX_SEGS];
};

template <typename T>
__global__ void __launch_bounds__(kThreads) k_pack(T *__restrict__ dst, PackArgs a, int n_src) {
    using A = Ar<T>;
    const int s = blockIdx.y;
    if (s >= n_src) return;
    const T *src = reinterpret_cast<const T *>(a.src[s]);
    T *d = dst + a.off[s];
    const int64_t len = a.len[s];
    const T sc = (T)a.scale[s];
    const bool plain = (sc == (T)1);
    const bool neg = (sc == (T)-1);
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < len; i += (int64_t)gridDim.x * kThreads) {
        T v = src ? src[i] : (T)0;
        if (!plain) v = neg ? -v : A::mul(sc, v);
        d[i] = v;
    }
}

}  // namespace

extern "C" {

int tdq_rk4_stage(int32_t dtype, int32_t which, void *y_out, const void *y0, const void *k1, const void *k2,
                  const void *k3, const void *k4, const void *dt_dev, const int64_t *step_dev, size_t n,
                  void *stream) {
    TDQ_REQUIRE(y_out && y0 && dt_dev, "null argument");
    TDQ_REAL_VIEW(dtype, n);
    TDQ_REQUIRE(which >= 1 && which <= 9, "which must be 1..9");
    const bool nA = which != 8, nB = which == 2 || which == 3 || which == 4 || which == 7 || which == 8,
               nC = which == 3 || which == 4 || which == 9, nD = which == 4;
    TDQ_REQUIRE(!nA || k1, "k1 required");
    TDQ_REQUIRE(!nB || k2, "k2 required");
    TDQ_REQUIRE(!nC || k3, "k3 required");
    TDQ_REQUIRE(!nD || k4, "k4 required");
    if (n == 0) return TDQ_OK;
    bool vec = tdq_aligned16(y_out) && tdq_aligned16(y0) && (!nA || tdq_aligned16(k1)) && (!nB || tdq_aligned16(k2)) &&
               (!nC || tdq_aligned16(k3)) && (!nD || tdq_aligned16(k4));
    cudaStream_t st = (cudaStream_t)stream;
    switch (which) {
        case 1: TDQ_DISPATCH_T(dtype, (launch_rk4<T, 1>(y_out, y0, k1, k2, k3, k4, dt_dev, step_dev, n, vec, st))); break;
        case 2: TDQ_DISPATCH_T(dtype, (launch_rk4<T, 2>(y_out, y0, k1, k2, k3, k4, dt_dev, step_dev, n, vec, st))); break;
        case 3: TDQ_DISPATCH_T(dtype, (launch_rk4<T, 3>(y_out, y0, k1, k2, k3, k4, dt_dev, step_dev, n, vec, st))); break;
        case 4: TDQ_DISPATCH_T(dtype, (launch_rk4<T, 4>(y_out, y0, k1, k2, k3, k4, dt_dev, step_dev, n, vec, st))); break;
        case 5: TDQ_DISPATCH_T(dtype, (launch_rk4<T, 5>(y_out, y0, k1, k2, k3, k4, dt_dev, step_dev, n, vec, st))); break;
        case 6: TDQ_DISPATCH_T(dtype, (launch_rk4<T, 6>(y_out, y0, k1, k2, k3, k4, dt_dev, step_dev, n, vec, st))); break;
        case 7: TDQ_DISPATCH_T(dtype, (launch_rk4<T, 7>(y_out, y0, k1, k2, k3, k4, dt_dev, step_dev, n, vec, st))); break;
        case 8: TDQ_DISPATCH_T(dtype, (launch_rk4<T, 8>(y_out, y0, k1, k2, k3, k4, dt_dev, step_dev, n, vec, st))); break;
        default: TDQ_DISPATCH_T(dtype, (launch_rk4<T, 9>(y_out, y0, k1, k2, k3, k4, dt_dev, step_dev, n, vec, st))); break;
    }
    TDQ_CHECK_CUDA(cudaGetLastError());
    return TDQ_OK;
}

int tdq_fixed_emit(int32_t dtype, void *y0, const void *y1, void *solution, const int32_t *rec_begin_dev,
                   const int32_t *out_idx_dev, const int32_t *mode_dev, const void *slope_dev, int64_t *step_dev,
                   const void *tstage_all_dev, void *tstage_cur_dev, int64_t n_steps, size_t n, void *stream) {
    TDQ_REQUIRE(y0 && y1 && solution && rec_begin_dev && out_idx_dev && mode_dev && slope_dev && step_dev &&
                    tstage_all_dev && tstage_cur_dev,
                "null argument");
    TDQ_REAL_VIEW(dtype, n);
    cudaStream_t st = (cudaStream_t)stream;
    size_t blocks = (n + kThreads - 1) / kThreads;
    if (blocks == 0) blocks = 1;
    if (blocks > 148 * 8) blocks = 148 * 8;
    TDQ_DISPATCH_T(dtype, (k_fixed_emit<T><<<(unsigned)blocks, kThreads, 0, st>>>(
                               (T *)y0, (const T *)y1, (T *)solution, rec_begin_dev, out_idx_dev, mode_dev,
                               (const T *)slope_dev, step_dev, (const unsigned char *)tstage_all_dev,
                               (unsigned char *)tstage_cur_dev, n_steps, n)));
    TDQ_CHECK_CUDA(cudaGetLastError());
    return TDQ_OK;
}

int tdq_fixed_final_emit(int32_t dtype, int32_t which, void *y0, const void *k1, const void *k2, const void *k3,
                         const void *k4, const void *dt_dev, void *solution, const int32_t *rec_begin_dev,
                         const int32_t *out_idx_dev, const int32_t *mode_dev, const void *slope_dev, int64_t *step_dev,
                         const void *tstage_all_dev, void *tstage_cur_dev, int64_t n_steps, size_t n, void *stream) {
    TDQ_REQUIRE(y0 && dt_dev && solution && rec_begin_dev && out_idx_dev && mode_dev && slope_dev && step_dev &&
                    tstage_all_dev && tstage_cur_dev,
                "null argument");
    TDQ_REQUIRE(which == 4 || which == 5 || which == 7 || which == 9, "which must be a final expression (4, 5, 7, 9)");
    TDQ_REQUIRE(k1 && (which == 5 || which == 9 || k2) && (which != 4 && which != 9 || k3) && (which != 4 || k4),
                "missing stage slot");
    TDQ_REAL_VIEW(dtype, n);
    cudaStream_t st = (cudaStream_t)stream;
    size_t blocks = (n + kThreads - 1) / kThreads;
    if (blocks == 0) blocks = 1;
    if (blocks > 148 * 8) blocks = 148 * 8;
#define TDQ_FE(W) TDQ_DISPATCH_T(dtype, (k_final_emit<T, W><<<(unsigned)blocks, kThreads, 0, st>>>(                    \
        (T *)y0, (const T *)k1, (const T *)k2, (const T *)k3, (const T *)k4, (const T *)dt_dev, (T *)solution,              \
        rec_begin_dev, out_idx_dev, mode_dev, (const T *)slope_dev, step_dev, (const unsigned char *)tstage_all_dev,        \
        (unsigned char *)tstage_cur_dev, n_steps, n)))
    if (which == 4) TDQ_FE(4);
    else if (which == 5) TDQ_FE(5);
    else if (which == 7) TDQ_FE(7);
    else TDQ_FE(9);
#undef TDQ_FE
    TDQ_CHECK_CUDA(cudaGetLastError());
    return TDQ_OK;
}

int tdq_lincomb(int32_t dtype, void *out, const void *base, const void *const *x, const double *coefs, int32_t n_terms,
                size_t n, void *stream) {
    TDQ_REQUIRE(out && x && coefs, "null argument");
    TDQ_REAL_VIEW(dtype, n);
    TDQ_REQUIRE(n_terms >= 1 && n_terms <= TDQ_MAX_K, "n_terms out of range");
    LinArgs a;
    memset(&a, 0, sizeof(a));
    for (int m = 0; m < n_terms; ++m) {
        TDQ_REQUIRE(x[m] != nullptr, "null term");
        a.x[m] = x[m];
        a.c[m] = coefs[m];
    }
    if (n == 0) return TDQ_OK;
    size_t blocks = (n + kThreads - 1) / kThreads;
    if (blocks > 148 * 8) blocks = 148 * 8;
    TDQ_DISPATCH_T(dtype, (k_lincomb<T><<<(unsigned)blocks, kThreads, 0, (cudaStream_t)stream>>>(
                               (T *)out, (const T *)base, a, n_terms, n)));
    TDQ_CHECK_CUDA(cudaGetLastError());
    return TDQ_OK;
}

int tdq_fixed_emit_cubic(int32_t dtype, const void *y0, const void *y1, const void *f0, const void *f1, void *solution,
                         const int32_t *out_idx_dev, const void *coef_dev, int32_t rec_lo, int32_t rec_hi, size_t n,
                         void *stream) {
    TDQ_REQUIRE(y0 && y1 && f0 && f1 && solution && out_idx_dev && coef_dev, "null argument");
    TDQ_REAL_VIEW(dtype, n);
    TDQ_REQUIRE(rec_lo >= 0 && rec_hi >= rec_lo, "bad record range");
    if (n == 0 || rec_hi == rec_lo) return TDQ_OK;
    size_t blocks = (n + kThreads - 1) / kThreads;
    if (blocks > 148 * 8) blocks = 148 * 8;
    TDQ_DISPATCH_T(dtype, (k_fixed_emit_cubic<T><<<(unsigned)blocks, kThreads, 0, (cudaStream_t)stream>>>(
                               (const T *)y0, (const T *)y1, (const T *)f0, (const T *)f1, (T *)solution, out_idx_dev,
                               (const T *)coef_dev, rec_lo, rec_hi, n)));
    TDQ_CHECK_CUDA(cudaGetLastError());
    return TDQ_OK;
}

int tdq_pack_segments(int32_t dtype, void *dst, const void *const *src, const int64_t *offsets, const int64_t *lens,
                      const double *scales, int32_t n_src, void *stream) {
    TDQ_REQUIRE(dst && src && offsets && lens && scales, "null argument");
    TDQ_REQUIRE(n_src >= 1 && n_src <= TDQ_MAX_SEGS, "n_src out of range");
    size_t w = 1;                                   // components per element
    TDQ_REAL_VIEW(dtype, w);
    PackArgs a;
    memset(&a, 0, sizeof(a));
    int64_t max_len = 0;
    for (int i = 0; i < n_src; ++i) {
        TDQ_REQUIRE(lens[i] >= 0 && offsets[i] >= 0, "negative segment");
        a.src[i] = src[i];
        a.off[i] = offsets[i] * (int64_t)w;
        a.len[i] = lens[i] * (int64_t)w;
        a.scale[i] = scales[i];
        if (a.len[i] > max_len) max_len = a.len[i];
    }
    if (max_len == 0) return TDQ_OK;
    size_t bx = (size_t)((max_len + kThreads * 4 - 1) / (kThreads * 4));
    if (bx == 0) bx = 1;
    if (bx > 148 * 8) bx = 148 * 8;
    dim3 grid((unsigned)bx, (unsigned)n_src);
    TDQ_DISPATCH_T(dtype, (k_pack<T><<<grid, kThreads, 0, (cudaStream_t)stream>>>((T *)dst, a, n_src)));
    TDQ_CHECK_CUDA(cudaGetLastError());
    return TDQ_OK;
}

}  // extern "C"
