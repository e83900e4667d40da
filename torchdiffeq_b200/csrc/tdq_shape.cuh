// tdq_shape.cuh -- host-side helpers shared by the launchers of libtdq's translation units.
#pragma once

#include "tdq_common.cuh"

#define TDQ_ROWS_H (TDQ_MAX_STAGES + 1)

// Host mirror of the tableau sparsity (so launchers can pick template arguments without reading device
// memory).  It is a function of the tableau only; launchers recompute it from the tdq_tableau the
// caller passes (cheap) instead of caching it per control block.
struct TdqHostShape {
    int valid;
    int n_stages, fsal;
    int row_nnz[TDQ_ROWS_H];
    int row_idx[TDQ_ROWS_H][TDQ_MAX_K];
    int err_nnz, mid_nnz;
    int err_idx[TDQ_MAX_K], mid_idx[TDQ_MAX_K];
};

void tdq_shape_from_tableau(const tdq_tableau *tab, TdqHostShape *h);   // tdq_stream.cu
int tdq_sm_count();                                                     // tdq_stream.cu

#define TDQ_DISPATCH_T(dtype, ...)                                         \
    do {                                                                   \
        if ((dtype) == TDQ_F32) { using T = float; __VA_ARGS__; }          \
        else if ((dtype) == TDQ_F64) { using T = double; __VA_ARGS__; }    \
        else { tdq_set_error("unsupported dtype %d", (int)(dtype)); return TDQ_ERR_INVALID; } \
    } while (0)

// Components per element of a state dtype: 1 (real), 2 (complex: interleaved re, im), 0 (not a dtype code).
static inline int tdq_dtype_width(int32_t dtype) {
    return (dtype == TDQ_F32 || dtype == TDQ_F64) ? 1 : (dtype == TDQ_C64 || dtype == TDQ_C128) ? 2 : 0;
}
// The component dtype of a state dtype (itself for real codes).
static inline int32_t tdq_real_code(int32_t dtype) {
    return dtype == TDQ_C64 ? TDQ_F32 : dtype == TDQ_C128 ? TDQ_F64 : dtype;
}

// The one place that knows what a complex state is to a launcher whose arithmetic only applies REAL coefficients
// (stage combines, the probe, the interpolant, fixed-grid steps, Adams sums, the pack, copies): z * (c + 0i) is
// (re * c, im * c) bit for bit, so such a launcher runs its real kernel on the 2n components of n complex elements.
// Rewrites (dtype, n) to (component dtype, components); refuses unknown codes.
#define TDQ_REAL_VIEW(dtype, n)                                                               \
    do {                                                                                      \
        const int w_ = tdq_dtype_width(dtype);                                                \
        if (w_ == 0) { tdq_set_error("%s: unsupported dtype %d", __func__, (int)(dtype)); return TDQ_ERR_INVALID; } \
        (n) *= w_;                                                                            \
        (dtype) = tdq_real_code(dtype);                                                       \
    } while (0)
