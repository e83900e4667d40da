// tdq_common.cuh -- device control block, rounding-exact arithmetic helpers and 128-bit vector access
// shared by every kernel of libtdq.  sm_100a only.
#pragma once

#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>
#include <string.h>

#include "tdq.h"

#define TDQ_ROWS (TDQ_MAX_STAGES + 1)   // stage rows 0..S-1 plus the c_sol row S

// ------------------------------------------------------------------------------------------------
// Control block.  Lives in device memory (caller-allocated, tdq_ctrl_size() bytes).  Every scalar
// the reference keeps as a 0-dim tensor or Python float in RKAdaptiveStepsizeODESolver
// (rk_common.py:161-369) lives here so that no decision needs the host.
// "T-valued" doubles hold a value that is exactly representable in the state dtype T.
// ------------------------------------------------------------------------------------------------
struct TdqCtrl {
    // ---- static: method -------------------------------------------------------------------
    int32_t dtype, n_stages, order, fsal;
    int32_t ratio_f64, n_out, n_step_t, next_step_index;
    int32_t row_nnz[TDQ_ROWS];               // non-zero entries per combine row
    int32_t row_idx[TDQ_ROWS][TDQ_MAX_K];    // their stage-slot indices, ascending
    int32_t err_nnz, mid_nnz;
    int32_t err_idx[TDQ_MAX_K], mid_idx[TDQ_MAX_K];
    double alpha[TDQ_MAX_STAGES];            // T-valued (rk_common.py:201)
    double beta[TDQ_ROWS][TDQ_MAX_K];        // T-valued, compacted like row_idx; row S = c_sol
    double c_err[TDQ_MAX_K], c_mid[TDQ_MAX_K]; // T-valued, compacted
    // ---- static: options ------------------------------------------------------------------
    double rtol, atol;                       // float64 as given (rk_common.py:186-187)
    double min_step, max_step, safety, ifactor, dfactor, t_sign;
    int64_t max_num_steps, n_global;
    const double *t_out;                     // ascending output times, float64, device
    const double *step_t;                    // optional sorted grid, float64, device
    const double *jump_t;                    // optional sorted discontinuity points, float64, device
    int32_t n_jump_t, next_jump_index, on_jump_t, pad_jump;
    tdq_mailbox *mbox;                       // mapped host memory (device view) or NULL
    // ---- sharded solves: peer exchange of the norm partials (tdq_ctrl_set_exchange) ----------
    void *xpeer[TDQ_MAX_RANKS];              // rank r's TdqXBuf as mapped in this process
    unsigned long long xepoch;               // solve number, identical on all ranks
    int32_t xrank, xworld;
    // ---- dynamic: rk_state (rk_common.py:18) ----------------------------------------------
    double t0, t1, dt;                       // last accepted interval [t0,t1]; dt = NEXT step size
    double att_t0, att_dt, att_t1;           // the attempt in flight
    double ratio, h0;
    int32_t on_step_t, accept, status, done;
    int32_t halt, out_cursor, emit_lo, emit_hi;
    int64_t n_accept, n_reject, n_steps_interval;
    uint64_t seq;
    // ---- state pointer table (tdq_ctrl_init from tdq_options.ybuf/kbuf) -----------------------
    // The accepted state y0 and its derivative f0 = k_0 live in ybuf[par] / kbuf[par].  Every attempt
    // the error-norm kernel writes the candidate (y1, k_S) into the OTHER pair; accepting is `par ^= 1`
    // in the controller -- no copy kernel (rk_common.py:341, :352 y_next = y1, f_next = f1).
    void *ybuf[2], *kbuf[2];
    const void *y0_cur, *k0_cur;             // = ybuf[par], kbuf[par]
    const void *y0_prev, *k0_prev;           // the pair of the step just accepted (interpolant fit)
    int32_t par, always_fit, fit_now, y0_bad;
    unsigned long long loop_handle;          // cudaGraphConditionalHandle of the device-side while, or 0
    // ---- per-attempt constants (T-valued), written by prepare / controller -----------------
    double coef[TDQ_ROWS][TDQ_MAX_K];        // t_sign * fl_T(beta_ij * T(dt))   (rk_common.py:79)
    double ecoef[TDQ_MAX_K];                 // t_sign * fl_T(T(dt) * e_j)       (rk_common.py:89)
    double fit_mcoef[TDQ_MAX_K];             // t_sign * fl_T(T(dt) * mid_j) of the ACCEPTED attempt
    double fit_sdt;                          // t_sign * T(dt) of the accepted attempt
    double att_dtT;                          // T(dt) of the attempt in flight
    // ---- state-dtype scalars torch views alias (func's time argument) ----------------------
    alignas(16) unsigned char tstage[8 * TDQ_MAX_K];
    alignas(16) unsigned char taux[8 * 4];
};

// Exchange buffer of one rank.  Four slots: (solve epoch parity, attempt parity).  Within a solve a rank can be at
// most one attempt ahead of a peer (its next controller needs that peer's next flag), hence the attempt parity;
// across solves a fast rank may start solve e+1 while a slow peer is still SUMMING the last attempt of solve e
// out of its own buffer (ADVICE r1), hence the epoch parity -- it cannot get two solves ahead, because the first
// attempt of solve e+1 needs every peer's flag of that solve.
struct TdqXBuf {
    double vals[4][TDQ_MAX_RANKS][TDQ_MAX_SEGS + 2];
    unsigned long long flags[4][TDQ_MAX_RANKS];
};

// ------------------------------------------------------------------------------------------------
// Contraction-free arithmetic: the reference rounds after every product and every sum
// (torch elementwise ops), so no FMA may be formed.
// ------------------------------------------------------------------------------------------------
template <typename T> struct Ar;
template <> struct Ar<float> {
    static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
    static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
    static __device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
    static __device__ __forceinline__ float div(float a, float b) { return __fdiv_rn(a, b); }
    static __device__ __forceinline__ float abs(float a) { return fabsf(a); }
    static __device__ __forceinline__ float max_nan(float a, float b) {   // torch.max propagates NaN
        return (a != a || b != b) ? CUDART_NAN_F : fmaxf(a, b);
    }
    static __device__ __forceinline__ bool finite(float a) { return isfinite(a); }
    static __device__ __forceinline__ float cabs(float re, float im) { return hypotf(re, im); }   // torch's complex abs
};
template <> struct Ar<double> {
    static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
    static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
    static __device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
    static __device__ __forceinline__ double div(double a, double b) { return __ddiv_rn(a, b); }
    static __device__ __forceinline__ double abs(double a) { return fabs(a); }
    static __device__ __forceinline__ double max_nan(double a, double b) {
        return (a != a || b != b) ? CUDART_NAN : fmax(a, b);
    }
    static __device__ __forceinline__ bool finite(double a) { return isfinite(a); }
    static __device__ __forceinline__ double cabs(double re, double im) { return hypot(re, im); }
};

// ------------------------------------------------------------------------------------------------
// 128-bit access.  Vec<T>::N elements per 16-byte transaction (4 x f32, 2 x f64).
// Streaming loads skip L1 allocation: every element is touched once per kernel.
// ------------------------------------------------------------------------------------------------
template <typename T> struct Vec;
template <> struct alignas(16) Vec<float> {
    static constexpr int N = 4;
    float v[4];
};
template <> struct alignas(16) Vec<double> {
    static constexpr int N = 2;
    double v[2];
};

template <typename T> __device__ __forceinline__ Vec<T> ld_stream(const T *p);
template <> __device__ __forceinline__ Vec<float> ld_stream<float>(const float *p) {
    Vec<float> r;
    asm volatile("ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]) : "l"(p));
    return r;
}
template <> __device__ __forceinline__ Vec<double> ld_stream<double>(const double *p) {
    Vec<double> r;
    asm volatile("ld.global.L1::no_allocate.v2.f64 {%0,%1}, [%2];"
                 : "=d"(r.v[0]), "=d"(r.v[1]) : "l"(p));
    return r;
}
template <typename T> __device__ __forceinline__ void st_vec(T *p, const Vec<T> &x);
template <> __device__ __forceinline__ void st_vec<float>(float *p, const Vec<float> &x) {
    asm volatile("st.global.v4.f32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "f"(x.v[0]), "f"(x.v[1]), "f"(x.v[2]), "f"(x.v[3]) : "memory");
}
template <> __device__ __forceinline__ void st_vec<double>(double *p, const Vec<double> &x) {
    asm volatile("st.global.v2.f64 [%0], {%1,%2};" :: "l"(p), "d"(x.v[0]), "d"(x.v[1]) : "memory");
}

// A pointer that comes straight out of a global load (the control block's pointer table: y0_cur, k0_cur, ybuf[], kbuf[])
// carries that load's SCOREBOARD into every address computation that uses it.  ptxas counts a loop's own loads on the
// same scoreboard, so "wait for the pointer" becomes "wait for every load issued so far": the second group of loads of an
// iteration is not issued before the first has returned (seen with ncu as long-scoreboard stalls on IADD3; it cost the
// fused linear stage 55 us instead of 39 us).  One integer add with a run-time zero the compiler cannot fold turns the
// pointer into an ALU result.  `n` is any size_t kernel argument below 2^63.
template <typename P>
__device__ __forceinline__ P *tdq_detach(P *p, size_t n) {
    return reinterpret_cast<P *>(reinterpret_cast<uintptr_t>(p) + (n >> 63));
}

// Stage-slot pointer bundle passed by value.
struct KPtrs {
    const void *p[TDQ_MAX_K];
};
struct KPtrsMut {
    void *p[TDQ_MAX_K];
};

// Warp + block sum of doubles (deterministic order).  Result valid in thread 0.
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}
template <int THREADS> __device__ __forceinline__ double block_sum(double v, double *smem /* THREADS/32 */) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    v = warp_sum(v);
    __syncthreads();          // protect smem reuse across calls
    if (lane == 0) smem[w] = v;
    __syncthreads();
    double r = 0.0;
    if (w == 0) {
        r = (lane < THREADS / 32) ? smem[lane] : 0.0;
        r = warp_sum(r);
    }
    return r;
}

// Host-side helpers (tdq_api.cu)
void tdq_set_error(const char *fmt, ...);
#define TDQ_CHECK_CUDA(expr)                                                              \
    do {                                                                                  \
        cudaError_t _e = (expr);                                                          \
        if (_e != cudaSuccess) {                                                          \
            tdq_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return TDQ_ERR_CUDA;                                                          \
        }                                                                                 \
    } while (0)
#define TDQ_REQUIRE(cond, msg)                                                            \
    do {                                                                                  \
        if (!(cond)) {                                                                    \
            tdq_set_error("%s: %s", __func__, msg);                                       \
            return TDQ_ERR_INVALID;                                                       \
        }                                                                                 \
    } while (0)

static inline bool tdq_aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
