// tdq_norm.cu -- scaled squared norms with a deterministic two-level reduction, fused with the state commit.
//
//   MODE 0  error ratio of an attempt (rk_common.py:89 tail, misc.py:80-82, :22-23, :30-33, adjoint.py:247-271):
//               err = err_pre (+ k_S * fl(dt*e_S) for FSAL tableaus)      the prefix comes from k_combine_final
//               tol = atol + rtol * max(|y0|, |y1|)
//               out[s] = sum over norm segment s of (err/tol)^2 ; out[n_seg] = # non-finite y1 elements
//           and, in the same pass over y1 and k_S, the CANDIDATE commit: y1 -> ybuf[par^1], k_S -> kbuf[par^1]
//           (the controller accepts by flipping `par`; rk_common.py:338-352 without a copy kernel).
//   MODE 1  out[s] = sum (x / scale)^2,         scale = atol + |y0| * rtol          misc.py:55-58
//   MODE 2  out[s] = sum ((x - x2) / scale)^2                                       misc.py:69
//
// Complex states (CPX): T is the component dtype and an element is an interleaved (re, im) pair.  |.| is the modulus
// (hypot, what torch's complex abs computes), tol and scale stay real, x/tol is x * fl(1/tol) componentwise (torch's
// complex-by-real division), and an element adds |x/tol|^2 = fl(fl(hypot(q))^2) once (.abs().pow(2)); it is non-finite
// when either part is.  Indices, segments and chunk lengths count elements; a chunk holds at most kChunk components.
//
// Work decomposition.  Single segment covering [0, n): a persistent grid of at most kMaxGrid blocks,
// thread-local float64 accumulation over a fixed block-strided assignment, one partial per block.
// Several segments (tuple states, the adjoint's augmented state, any number of them): a CHUNK TABLE in
// device memory (tdq_norm_table_fill) cuts [0, n) into pieces of at most kChunk elements, each inside
// one segment or inside a gap (padding / elements no norm looks at: still committed, still checked for
// non-finite values); one partial per chunk.  In both cases the last block to finish (ticket) adds the
// partials in index order, so a result depends on n and the segment list only -- not on the schedule.
#include "tdq_common.cuh"
#include "tdq_shape.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kChunk = 2048;            // elements per chunk of the multi-segment path
constexpr int kMaxGrid = 148 * 4;       // persistent grid of the single-segment path (B200: 148 SMs); a constant,
                                        // so that partial sums do not depend on the device the library runs on

template <typename T, bool VTOL> struct TolT { using type = T; };
template <typename T> struct TolT<T, true> { using type = double; };

// components per element
template <bool CPX> constexpr int kWidth = CPX ? 2 : 1;

struct NormArgs {
    const void *x;          // MODE 0: err_pre          MODE 1/2: x
    const void *x2;         // MODE 0: k_S              MODE 2: x2
    const void *y0;         // NULL: the control block's current y0
    const void *y1;         // MODE 0 only
    const double *rtol_v, *atol_v;
    const int64_t *table;   // chunk table (MULTI) or NULL
    double *partials;       // [0..1]: ticket word; then sums[P], then bad[P]
    double *out;            // [n_seg + 1]
    void *q_out;            // WRITEQ: err/tol per element (a pair per complex element)
    size_t n;               // elements
    int n_parts;            // P: blocks (single) or chunks (multi)
    int n_seg;
};

template <typename T, bool CPX, int MODE, bool VECTOR, bool VTOL, bool MULTI, bool WRITEQ>
__global__ void __launch_bounds__(kThreads)
k_norm(const TdqCtrl *__restrict__ c, NormArgs a) {
    if (c->halt) return;
    using A = Ar<T>;
    using Q = typename TolT<T, VTOL>::type;     // dtype of tol and of err/tol (float64 with vector tolerances)
    using V = Vec<T>;
    constexpr int VN = VECTOR ? V::N : 1;
    constexpr int EW = kWidth<CPX>;             // components per element
    constexpr int VE = V::N / EW;               // elements per 16-byte vector
    __shared__ double red[kThreads / 32];
    __shared__ bool is_last;

    const T *x = reinterpret_cast<const T *>(a.x);
    const T *x2 = reinterpret_cast<const T *>(a.x2);
    const T *y0 = tdq_detach(reinterpret_cast<const T *>(a.y0 ? a.y0 : c->y0_cur), a.n);
    const T *y1 = reinterpret_cast<const T *>(a.y1);
    const T rtolT = (T)c->rtol, atolT = (T)c->atol;   // 0-dim float64 tensors act as scalars of T (misc.py:81)
    // MODE 0: the last error weight, when it belongs to k_S of an FSAL tableau, is not in the prefix
    const bool ek = MODE == 0 && c->fsal && c->err_nnz > 0 && c->err_idx[c->err_nnz - 1] == c->n_stages;
    const T ecS = ek ? (T)c->ecoef[c->err_nnz - 1] : (T)0;
    T *ycand = nullptr, *kcand = nullptr;
    if (MODE == 0 && c->ybuf[0] != nullptr) {
        ycand = tdq_detach(reinterpret_cast<T *>(c->ybuf[c->par ^ 1]), a.n);
        kcand = tdq_detach(reinterpret_cast<T *>(c->kbuf[c->par ^ 1]), a.n);
    }
    double *p_sum = a.partials + 2, *p_bad = p_sum + a.n_parts;

    double acc = 0.0, bad = 0.0;
    // one element: returns nothing, accumulates into acc/bad.  v0 = y0[i]; xa = x[i]; xb = x2[i]; v1 = y1[i]
    auto element = [&](size_t i, T v0, T v1, T xa, T xb, bool in_seg) {
        if (MODE == 0 && !A::finite(v1)) bad += 1.0;
        if (MODE == 1 && !A::finite(v0)) bad += 1.0;      // d0's pass over y0 doubles as rk_common.py:287's check
        if (!in_seg) return;
        T num;
        if (MODE == 0) num = ek ? A::add(xa, A::mul(xb, ecS)) : xa;
        else num = (MODE == 2) ? A::sub(xa, xb) : xa;
        Q q;
        if (VTOL) {
            const double rt = a.rtol_v[i], at = a.atol_v[i];
            double tol;
            if (MODE == 0) tol = at + rt * (double)A::max_nan(A::abs(v0), A::abs(v1));
            else tol = at + (double)A::abs(v0) * rt;
            q = (Q)((double)num / tol);
        } else {
            T tol;
            if (MODE == 0) tol = A::add(atolT, A::mul(rtolT, A::max_nan(A::abs(v0), A::abs(v1))));
            else tol = A::add(atolT, A::mul(A::abs(v0), rtolT));
            q = (Q)A::div(num, tol);
        }
        if (WRITEQ) reinterpret_cast<Q *>(a.q_out)[i] = q;
        const Q q2 = Ar<Q>::mul(q, q);                 // .abs().pow(2)
        acc += (double)q2;
    };
    // one complex element: v0 = y0[i], v1 = y1[i], xa = x[i], xb = x2[i] as (re, im) pairs
    auto celement = [&](size_t i, const T *v0, const T *v1, const T *xa, const T *xb, bool in_seg) {
        if (MODE == 0 && !(A::finite(v1[0]) && A::finite(v1[1]))) bad += 1.0;
        if (MODE == 1 && !(A::finite(v0[0]) && A::finite(v0[1]))) bad += 1.0;
        if (!in_seg) return;
        T num[2];
#pragma unroll
        for (int p = 0; p < 2; ++p) {
            if (MODE == 0) num[p] = ek ? A::add(xa[p], A::mul(xb[p], ecS)) : xa[p];
            else num[p] = (MODE == 2) ? A::sub(xa[p], xb[p]) : xa[p];
        }
        const T m0 = A::cabs(v0[0], v0[1]);
        Q q[2];
        if (VTOL) {
            const double rt = a.rtol_v[i], at = a.atol_v[i];
            double tol;
            if (MODE == 0) tol = at + rt * (double)A::max_nan(m0, A::cabs(v1[0], v1[1]));
            else tol = at + (double)m0 * rt;
            const double r = 1.0 / tol;
            q[0] = (Q)((double)num[0] * r);
            q[1] = (Q)((double)num[1] * r);
        } else {
            T tol;
            if (MODE == 0) tol = A::add(atolT, A::mul(rtolT, A::max_nan(m0, A::cabs(v1[0], v1[1]))));
            else tol = A::add(atolT, A::mul(m0, rtolT));
            const T r = A::div((T)1, tol);
            q[0] = (Q)A::mul(num[0], r);
            q[1] = (Q)A::mul(num[1], r);
        }
        if (WRITEQ) {
            reinterpret_cast<Q *>(a.q_out)[2 * i] = q[0];
            reinterpret_cast<Q *>(a.q_out)[2 * i + 1] = q[1];
        }
        const Q m = Ar<Q>::cabs(q[0], q[1]);
        acc += (double)Ar<Q>::mul(m, m);               // .abs().pow(2)
    };
    auto scalar_at = [&](size_t i, bool in_seg) {
        if constexpr (CPX) {
            const size_t j = 2 * i;
            const T v0[2] = {y0[j], y0[j + 1]};
            const T xa[2] = {x[j], x[j + 1]};
            const T v1[2] = {(MODE == 0) ? y1[j] : (T)0, (MODE == 0) ? y1[j + 1] : (T)0};
            const T xb[2] = {(MODE != 1) ? x2[j] : (T)0, (MODE != 1) ? x2[j + 1] : (T)0};
            celement(i, v0, v1, xa, xb, in_seg);
            if (MODE == 0 && ycand) {
                ycand[j] = v1[0]; ycand[j + 1] = v1[1];
                kcand[j] = xb[0]; kcand[j + 1] = xb[1];
            }
        } else {
            const T v1 = (MODE == 0) ? y1[i] : (T)0;
            const T xb = (MODE != 1) ? x2[i] : (T)0;
            element(i, y0[i], v1, x[i], xb, in_seg);
            if (MODE == 0 && ycand) { ycand[i] = v1; kcand[i] = xb; }
        }
    };
    // the VE elements of one 16-byte vector, the first of which is element i
    auto vector_at = [&](size_t i, const V &a0, const V &a1, const V &xa, const V &xb, bool in_seg) {
#pragma unroll
        for (int e = 0; e < VE; ++e) {
            if constexpr (CPX)
                celement(i + e, &a0.v[2 * e], &a1.v[2 * e], &xa.v[2 * e], &xb.v[2 * e], in_seg);
            else
                element(i + e, a0.v[e], (MODE == 0) ? a1.v[e] : (T)0, xa.v[e], (MODE != 1) ? xb.v[e] : (T)0,
                        in_seg);
        }
    };

    if (!MULTI) {
        // ---- one segment = [0, n): persistent blocks, fixed block-strided assignment -------------------
        constexpr int U = 2;
        if (VECTOR) {
            const size_t nvec = a.n / VE;
            const size_t stride = (size_t)gridDim.x * (kThreads * U);
            for (size_t base = (size_t)blockIdx.x * (kThreads * U) + threadIdx.x; base < nvec; base += stride) {
                V a0[U], a1[U], xa[U], xb[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const size_t v = base + (size_t)u * kThreads;
                    if (v < nvec) {
                        const size_t i0 = v * V::N;
                        a0[u] = ld_stream<T>(y0 + i0);
                        xa[u] = ld_stream<T>(x + i0);
                        if (MODE == 0) a1[u] = ld_stream<T>(y1 + i0);
                        if (MODE != 1) xb[u] = ld_stream<T>(x2 + i0);
                    }
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const size_t v = base + (size_t)u * kThreads;
                    if (v < nvec) {
                        const size_t i0 = v * V::N;
                        vector_at(v * VE, a0[u], a1[u], xa[u], xb[u], true);
                        if (MODE == 0 && ycand) {
                            st_vec<T>(ycand + i0, a1[u]);
                            st_vec<T>(kcand + i0, xb[u]);
                        }
                    }
                }
            }
            if (blockIdx.x == 0) {
                const size_t i = nvec * VE + threadIdx.x;
                if (i < a.n) scalar_at(i, true);
            }
        } else {
            for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < a.n; i += (size_t)gridDim.x * kThreads)
                scalar_at(i, true);
        }
        const double tsum = block_sum<kThreads>(acc, red);
        const double tbad = block_sum<kThreads>(bad, red);
        if (threadIdx.x == 0) {
            p_sum[blockIdx.x] = tsum;
            p_bad[blockIdx.x] = tbad;
        }
    } else {
        // ---- chunk table -----------------------------------------------------------------------------
        const int64_t *tb = a.table;
        const int n_seg = (int)tb[0], n_chunks = (int)tb[1];
        const int64_t *chunk_start = tb + 4 + 2 * (int64_t)n_seg;
        const int64_t *chunk_meta = chunk_start + n_chunks;
        // slots per thread: a chunk holds at most kChunk components, i.e. kChunk / V::N vectors or kChunk / EW elements
        constexpr int U = kChunk / (kThreads * (VECTOR ? VN : EW));
        for (int ch = blockIdx.x; ch < n_chunks; ch += gridDim.x) {
            const int64_t start = chunk_start[ch], meta = chunk_meta[ch];
            const int len = (int)(meta & 0xffffffffll);
            const bool in_seg = (meta >> 32) != 0;
            acc = 0.0;
            bad = 0.0;
            if (in_seg || MODE == 0) {
                if (VECTOR) {
                    const int nvec = len / VE;
                    V a0[U], a1[U], xa[U], xb[U];
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const int v = threadIdx.x + u * kThreads;
                        if (v < nvec) {
                            const size_t i0 = ((size_t)start + (size_t)v * VE) * EW;
                            a0[u] = ld_stream<T>(y0 + i0);
                            xa[u] = ld_stream<T>(x + i0);
                            if (MODE == 0) a1[u] = ld_stream<T>(y1 + i0);
                            if (MODE != 1) xb[u] = ld_stream<T>(x2 + i0);
                        }
                    }
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const int v = threadIdx.x + u * kThreads;
                        if (v < nvec) {
                            const size_t i0 = ((size_t)start + (size_t)v * VE) * EW;
                            vector_at((size_t)start + (size_t)v * VE, a0[u], a1[u], xa[u], xb[u], in_seg);
                            if (MODE == 0 && ycand) {
                                st_vec<T>(ycand + i0, a1[u]);
                                st_vec<T>(kcand + i0, xb[u]);
                            }
                        }
                    }
                    const int i = nvec * VE + threadIdx.x;
                    if (i < len) scalar_at((size_t)start + i, in_seg);
                } else {
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const int i = threadIdx.x + u * kThreads;
                        if (i < len) scalar_at((size_t)start + i, in_seg);
                    }
                }
            }
            const double tsum = block_sum<kThreads>(acc, red);
            const double tbad = block_sum<kThreads>(bad, red);
            if (threadIdx.x == 0) {
                p_sum[ch] = tsum;
                p_bad[ch] = tbad;
            }
        }
    }

    // ---- ticket: the last block to finish adds the partials in index order -------------------------
    unsigned int *ticket = reinterpret_cast<unsigned int *>(a.partials);
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned int t = atomicAdd(ticket, 1u);
        is_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    const int P = a.n_parts;
    {
        double b = 0.0;
        for (int i = threadIdx.x; i < P; i += kThreads) b += __ldcg(&p_bad[i]);
        const double sb = block_sum<kThreads>(b, red);
        if (threadIdx.x == 0) a.out[a.n_seg] = sb;
    }
    if (!MULTI) {
        double s = 0.0;
        for (int i = threadIdx.x; i < P; i += kThreads) s += __ldcg(&p_sum[i]);
        const double ss = block_sum<kThreads>(s, red);
        if (threadIdx.x == 0) a.out[0] = ss;
    } else {
        const int64_t *tb = a.table;
        const int n_seg = (int)tb[0];
        const int64_t *seg_first = tb + 4, *seg_nch = seg_first + n_seg;
        // small segments: one thread each, sequential over its few chunks
        for (int s = threadIdx.x; s < n_seg; s += kThreads) {
            const int nch = (int)seg_nch[s];
            if (nch > 4) continue;
            const int f = (int)seg_first[s];
            double v = 0.0;
            for (int i = 0; i < nch; ++i) v += __ldcg(&p_sum[f + i]);
            a.out[s] = v;
        }
        // large segments: one warp each, lanes strided, fixed shuffle tree
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
        int big = 0;
        for (int s = 0; s < n_seg; ++s) {
            const int nch = (int)seg_nch[s];
            if (nch <= 4) continue;
            if ((big++ % (kThreads / 32)) != w) continue;
            const int f = (int)seg_first[s];
            double v = 0.0;
            for (int i = lane; i < nch; i += 32) v += __ldcg(&p_sum[f + i]);
            v = warp_sum(v);
            if (lane == 0) a.out[s] = v;
        }
    }
    if (threadIdx.x == 0) *ticket = 0;                      // self-reset for the next launch
}

// Candidate commit on its own (callers with a custom norm callable, whose error pass does not commit).
template <typename T>
__global__ void __launch_bounds__(kThreads)
k_commit(const TdqCtrl *__restrict__ c, const T *__restrict__ y1, const T *__restrict__ kS, size_t n) {
    if (c->halt || c->ybuf[0] == nullptr) return;
    T *ycand = reinterpret_cast<T *>(c->ybuf[c->par ^ 1]);
    T *kcand = reinterpret_cast<T *>(c->kbuf[c->par ^ 1]);
    for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (size_t)gridDim.x * kThreads) {
        ycand[i] = y1[i];
        kcand[i] = kS[i];
    }
}

template <typename T, bool CPX, int MODE>
int launch_norm(const TdqCtrl *c, NormArgs &a, bool vec, cudaStream_t st) {
    const bool vtol = a.rtol_v != nullptr;
    const bool multi = a.table != nullptr;
    const bool wq = a.q_out != nullptr;
    unsigned grid;
    if (multi) {
        grid = (unsigned)a.n_parts;
        const unsigned cap = (unsigned)tdq_sm_count() * 8;
        if (grid > cap) grid = cap;
    } else {
        grid = (unsigned)a.n_parts;
    }
    if (grid == 0) grid = 1;
#define TDQ_L(V_, VT_, M_, WQ_) k_norm<T, CPX, MODE, V_, VT_, M_, WQ_><<<grid, kThreads, 0, st>>>(c, a)
#define TDQ_L3(V_, VT_, M_) do { if (wq && MODE == 0) TDQ_L(V_, VT_, M_, (MODE == 0)); else TDQ_L(V_, VT_, M_, false); } while (0)
#define TDQ_L2(V_, VT_) do { if (multi) TDQ_L3(V_, VT_, true); else TDQ_L3(V_, VT_, false); } while (0)
    if (vec) { if (vtol) TDQ_L2(true, true); else TDQ_L2(true, false); }
    else     { if (vtol) TDQ_L2(false, true); else TDQ_L2(false, false); }
#undef TDQ_L2
#undef TDQ_L3
#undef TDQ_L
    return 0;
}

// k_norm for a state dtype code; -1 for a code that is not one
template <int MODE>
int dispatch_norm(int32_t dtype, const TdqCtrl *c, NormArgs &a, bool vec, cudaStream_t st) {
    switch (dtype) {
        case TDQ_F32: return launch_norm<float, false, MODE>(c, a, vec, st);
        case TDQ_F64: return launch_norm<double, false, MODE>(c, a, vec, st);
        case TDQ_C64: return launch_norm<float, true, MODE>(c, a, vec, st);
        case TDQ_C128: return launch_norm<double, true, MODE>(c, a, vec, st);
        default: return -1;
    }
}

// elements per 16-byte vector of a state dtype (4 float32, 2 float64 or complex64, 1 complex128)
inline int vec_elems(int32_t dtype) { return 16 / (tdq_dtype_width(dtype) * (tdq_real_code(dtype) == TDQ_F32 ? 4 : 8)); }

// number of partials (= blocks) of the single-segment path for n elements
inline int single_parts(size_t n, bool vec, int vn) {
    const size_t units = vec ? n / vn : n;                              // vectors or scalars to distribute
    const size_t per_block = vec ? (size_t)kThreads * 2 : (size_t)kThreads;
    size_t blocks = (units + per_block - 1) / per_block;
    if (blocks > (size_t)kMaxGrid) blocks = kMaxGrid;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

}  // namespace

extern "C" {

size_t tdq_norm_partials_len(size_t n, int64_t n_chunks) {
    // two planes (sums, non-finite counts) of one double per part + the ticket word (8 bytes, 2 doubles reserved)
    size_t parts = (size_t)kMaxGrid;
    if (n_chunks > 0 && (size_t)n_chunks > parts) parts = (size_t)n_chunks;
    (void)n;
    return 2 * parts + 2;
}

int64_t tdq_norm_table_fill(const int64_t *seg_offsets, const int64_t *seg_lens, int32_t n_seg, int64_t n,
                            int32_t dtype, int64_t *table_host, int64_t capacity_words) {
    // Returns the number of int64 words the table needs (fills table_host when capacity suffices), or -1.
    // Layout: [n_seg, n_chunks, kChunk, aligned] seg_first[n_seg] seg_nchunks[n_seg] chunk_start[n_chunks]
    // chunk_meta[n_chunks] (len | (segment+1) << 32; 0 = gap).  Gaps are cut so that every chunk of at least
    // one 16-byte vector starts on a 16-byte boundary; `aligned` says whether every SEGMENT does too.
    if (!seg_offsets || !seg_lens || n_seg < 1 || n < 0 || tdq_dtype_width(dtype) == 0) {
        tdq_set_error("tdq_norm_table_fill: bad argument");
        return -1;
    }
    const int64_t vn = vec_elems(dtype);
    const int64_t kChunk = ::kChunk / tdq_dtype_width(dtype);   // elements per chunk: at most kChunk components
    int64_t ch = 0;
    int64_t *seg_first = nullptr, *seg_nch = nullptr, *chunk_start = nullptr, *chunk_meta = nullptr;
    bool write = false;
    auto emit = [&](int64_t lo, int64_t hi, int64_t seg_plus1) {
        if (seg_plus1 == 0 && lo < hi && (lo % vn) != 0) {                // unaligned head of a gap: scalar chunk
            int64_t mid = (lo + vn - 1) / vn * vn;
            if (mid > hi) mid = hi;
            if (write) { chunk_start[ch] = lo; chunk_meta[ch] = (mid - lo); }
            ++ch;
            lo = mid;
        }
        for (int64_t b = lo; b < hi; b += kChunk) {
            const int64_t len = (hi - b < kChunk) ? hi - b : kChunk;
            if (write) { chunk_start[ch] = b; chunk_meta[ch] = len | (seg_plus1 << 32); }
            ++ch;
        }
    };
    int64_t aligned = 1;
    for (int pass = 0; pass < 2; ++pass) {
        int64_t pos = 0;
        ch = 0;
        for (int s = 0; s < n_seg; ++s) {
            if (seg_offsets[s] < pos || seg_lens[s] < 0 || seg_offsets[s] + seg_lens[s] > n) {
                tdq_set_error("tdq_norm_table_fill: segments must be ascending, disjoint and inside [0, n)");
                return -1;
            }
            if (seg_offsets[s] % vn != 0) aligned = 0;
            emit(pos, seg_offsets[s], 0);
            if (write) seg_first[s] = ch;
            const int64_t first = ch;
            emit(seg_offsets[s], seg_offsets[s] + seg_lens[s], (int64_t)s + 1);
            if (write) seg_nch[s] = ch - first;
            pos = seg_offsets[s] + seg_lens[s];
        }
        emit(pos, n, 0);
        if (pass == 1) break;
        const int64_t n_chunks = ch;
        const int64_t words = 4 + 2 * (int64_t)n_seg + 2 * n_chunks;
        if (!table_host || capacity_words < words) return words;
        seg_first = table_host + 4;
        seg_nch = seg_first + n_seg;
        chunk_start = seg_nch + n_seg;
        chunk_meta = chunk_start + n_chunks;
        table_host[0] = n_seg;
        table_host[1] = n_chunks;
        table_host[2] = kChunk;
        table_host[3] = aligned;
        write = true;
    }
    return 4 + 2 * (int64_t)n_seg + 2 * ch;
}

static int norm_common(NormArgs &a, const int64_t *table_dev, int64_t n_chunks, int32_t n_seg, int32_t dtype,
                       bool table_aligned, bool *vec) {
    const int vn = vec_elems(dtype);
    a.table = table_dev;
    a.n_seg = n_seg;
    if (table_dev) {
        if (n_chunks < 1) return -1;
        a.n_parts = (int)n_chunks;
        *vec = *vec && table_aligned;
    } else {
        if (n_seg != 1) return -1;
        a.n_parts = single_parts(a.n, *vec, vn);
    }
    return 0;
}

int tdq_error_norm_commit(void *ctrl_dev, int32_t dtype, const void *err_pre, const void *k_last, const void *y0,
                          const void *y1, const double *rtol_vec, const double *atol_vec, const int64_t *table_dev,
                          int64_t n_chunks, int32_t table_aligned, int32_t n_seg, size_t n, double *partials,
                          double *out, void *err_over_tol_out, void *stream) {
    TDQ_REQUIRE(ctrl_dev && err_pre && k_last && y1 && partials && out, "null argument");
    TDQ_REQUIRE(n_seg >= 1, "n_seg out of range");
    TDQ_REQUIRE(tdq_dtype_width(dtype) != 0, "unsupported dtype");
    TDQ_REQUIRE((rtol_vec == nullptr) == (atol_vec == nullptr), "rtol_vec and atol_vec go together");
    NormArgs a;
    memset(&a, 0, sizeof(a));
    a.x = err_pre; a.x2 = k_last; a.y0 = y0; a.y1 = y1;
    a.rtol_v = rtol_vec; a.atol_v = atol_vec;
    a.partials = partials; a.out = out; a.q_out = err_over_tol_out; a.n = n;
    bool vec = tdq_aligned16(err_pre) && tdq_aligned16(k_last) && tdq_aligned16(y0) && tdq_aligned16(y1);
    if (err_over_tol_out) vec = false;   // q may be float64 while the state is float32: keep it simple
    TDQ_REQUIRE(norm_common(a, table_dev, n_chunks, n_seg, dtype, table_aligned != 0, &vec) == 0,
                "several segments need a chunk table (tdq_norm_table_fill)");
    if (n == 0) return TDQ_OK;
    dispatch_norm<0>(dtype, (const TdqCtrl *)ctrl_dev, a, vec, (cudaStream_t)stream);
    TDQ_CHECK_CUDA(cudaGetLastError());
    return TDQ_OK;
}

int tdq_scaled_sumsq(void *ctrl_dev, int32_t dtype, const void *x, const void *x2, const void *y0,
                     const double *rtol_vec, const double *atol_vec, const int64_t *table_dev, int64_t n_chunks,
                     int32_t table_aligned, int32_t n_seg, size_t n, double *partials, double *out, void *stream) {
    TDQ_REQUIRE(ctrl_dev && x && partials && out, "null argument");
    TDQ_REQUIRE(n_seg >= 1, "n_seg out of range");
    TDQ_REQUIRE(tdq_dtype_width(dtype) != 0, "unsupported dtype");
    TDQ_REQUIRE((rtol_vec == nullptr) == (atol_vec == nullptr), "rtol_vec and atol_vec go together");
    NormArgs a;
    memset(&a, 0, sizeof(a));
    a.x = x; a.x2 = x2; a.y0 = y0;
    a.rtol_v = rtol_vec; a.atol_v = atol_vec;
    a.partials = partials; a.out = out; a.n = n;
    bool vec = tdq_aligned16(x) && tdq_aligned16(y0) && (x2 == nullptr || tdq_aligned16(x2));
    TDQ_REQUIRE(norm_common(a, table_dev, n_chunks, n_seg, dtype, table_aligned != 0, &vec) == 0,
                "several segments need a chunk table (tdq_norm_table_fill)");
    if (n == 0) return TDQ_OK;
    const TdqCtrl *c = (const TdqCtrl *)ctrl_dev;
    cudaStream_t st = (cudaStream_t)stream;
    if (x2) dispatch_norm<2>(dtype, c, a, vec, st);
    else dispatch_norm<1>(dtype, c, a, vec, st);
    TDQ_CHECK_CUDA(cudaGetLastError());
    return TDQ_OK;
}

int tdq_commit_candidates(void *ctrl_dev, int32_t dtype, const void *y1, const void *k_last, size_t n, void *stream) {
    TDQ_REQUIRE(ctrl_dev && y1 && k_last, "null argument");
    TDQ_REAL_VIEW(dtype, n);
    if (n == 0) return TDQ_OK;
    size_t blocks = (n + kThreads - 1) / kThreads;
    const size_t cap = (size_t)tdq_sm_count() * 8;
    if (blocks > cap) blocks = cap;
    TDQ_DISPATCH_T(dtype, (k_commit<T><<<(unsigned)blocks, kThreads, 0, (cudaStream_t)stream>>>(
                               (const TdqCtrl *)ctrl_dev, (const T *)y1, (const T *)k_last, n)));
    TDQ_CHECK_CUDA(cudaGetLastError());
    return TDQ_OK;
}

}  // extern "C"
