// tdq_stream.cu -- stage combines of the explicit RK hot path.
//
//   k_combine        y_i = y0 + sum_j k_j * c_ij                                  rk_common.py:79, :85
//   k_combine_final  the LAST combine of an attempt (the row that produces y1), fused with the part of the
//                    embedded error estimate that is already computable:          rk_common.py:83-89
//                        y1      = y0 + sum_j k_j * c_sol_j
//                        err_pre = sum_{j available} k_j * fl(dt * e_j)           (ascending j: a prefix of :89's sum)
//
// Both stream each operand exactly once with 128-bit transactions, keep stage slots as separate
// contiguous arrays (structure of arrays; the reference interleaves the stage index innermost,
// rk_common.py:69) and read their scalars from the device control block, so the same launch sequence
// is valid for every attempt and can be replayed from a CUDA graph.  y0 and k_0 (the accepted state and
// its derivative) are read through the control block's pointer table when the caller passes NULL: an
// accepted step flips that table instead of copying y1 -> y0 and k_S -> k_0.
// Arithmetic is contraction free and follows the reference's order of roundings (SURVEY.md 8(a)).
#include "tdq_common.cuh"
#include "tdq_shape.cuh"

namespace {

// ------------------------------------------------------------------------------------------------
// Stage combine.  NK = number of non-zero tableau entries in the row (compile time => the NK+1 loads
// of a thread are all in flight before the first use).
// ------------------------------------------------------------------------------------------------
// Launch shape, from the r1 tuning sweep on B200 (profiles/r1_combine_variants.txt): a persistent
// grid-stride kernel beats one-tile-per-block by 1-15 % at 33.5 MB per operand because the last wave no
// longer drains alone.  Rows with few operands need more bytes in flight per thread:
//   NK <= 2 : 512 threads, 4 vectors per operand per thread, 2 blocks per SM
//   NK >= 3 : 256 threads, 2 vectors per operand per thread, 8 blocks per SM
// The bulk-async (TMA, cp.async.bulk + mbarrier ring through shared memory) variant measured
// SLOWER than plain 128-bit loads for this pure streaming pattern (profiles/r2_tma_sweep.txt), so it is not used.
template <typename T, int NK, int THREADS, int U, bool VECTOR>
__global__ void __launch_bounds__(THREADS)
k_combine(const TdqCtrl *__restrict__ c, int row, T *__restrict__ out, const T *y0, KPtrs kp, size_t n) {
    if (c->halt) return;
    using A = Ar<T>;
    T cf[NK];
    const T *k[NK];
    if (y0 == nullptr) y0 = reinterpret_cast<const T *>(c->y0_cur);
#pragma unroll
    for (int m = 0; m < NK; ++m) {
        cf[m] = (T)c->coef[row][m];
        k[m] = tdq_detach(reinterpret_cast<const T *>(kp.p[m] ? kp.p[m] : c->k0_cur), n);
    }
    y0 = tdq_detach(y0, n);
    if (VECTOR) {
        using V = Vec<T>;
        const size_t nvec = n / V::N;
        const size_t stride = (size_t)gridDim.x * (THREADS * U);
        for (size_t base = (size_t)blockIdx.x * (THREADS * U) + threadIdx.x; base < nvec; base += stride) {
            V a[U], kv[U][NK];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const size_t v = base + (size_t)u * THREADS;
                if (v < nvec) {
                    a[u] = ld_stream<T>(y0 + v * V::N);
#pragma unroll
                    for (int m = 0; m < NK; ++m) kv[u][m] = ld_stream<T>(k[m] + v * V::N);
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const size_t v = base + (size_t)u * THREADS;
                if (v < nvec) {
                    V r;
#pragma unroll
                    for (int e = 0; e < V::N; ++e) {
                        T acc = A::mul(kv[u][0].v[e], cf[0]);
#pragma unroll
                        for (int m = 1; m < NK; ++m) acc = A::add(acc, A::mul(kv[u][m].v[e], cf[m]));
                        r.v[e] = A::add(a[u].v[e], acc);
                    }
                    st_vec<T>(out + v * V::N, r);
                }
            }
        }
        // scalar tail (n not a multiple of the vector width): first threads of block 0
        if (blockIdx.x == 0) {
            const size_t i = nvec * V::N + threadIdx.x;
            if (i < n) {
                T acc = A::mul(k[0][i], cf[0]);
#pragma unroll
                for (int m = 1; m < NK; ++m) acc = A::add(acc, A::mul(k[m][i], cf[m]));
                out[i] = A::add(y0[i], acc);
            }
        }
    } else {
        for (size_t i = (size_t)blockIdx.x * THREADS + threadIdx.x; i < n; i += (size_t)gridDim.x * THREADS) {
            T acc = A::mul(k[0][i], cf[0]);
#pragma unroll
            for (int m = 1; m < NK; ++m) acc = A::add(acc, A::mul(k[m][i], cf[m]));
            out[i] = A::add(y0[i], acc);
        }
    }
}

template <typename T, int NK>
int launch_combine(const TdqCtrl *c, int row, void *out, const void *y0, const KPtrs &kp, size_t n, bool vec,
                   cudaStream_t st) {
    constexpr bool kFew = NK <= 2;
    constexpr int THREADS = kFew ? 512 : 256;
    constexpr int U = kFew ? 4 : 2;
    constexpr int PER_SM = kFew ? 2 : 8;
    if (vec) {
        using V = Vec<T>;
        const size_t nvec = n / V::N;
        size_t blocks = (nvec + (size_t)THREADS * U - 1) / ((size_t)THREADS * U);
        const size_t cap = (size_t)tdq_sm_count() * PER_SM;       // one resident wave; the loop covers the rest
        if (blocks > cap) blocks = cap;
        if (blocks == 0) blocks = 1;
        k_combine<T, NK, THREADS, U, true><<<(unsigned)blocks, THREADS, 0, st>>>(c, row, (T *)out, (const T *)y0, kp, n);
    } else {
        size_t blocks = (n + THREADS - 1) / THREADS;
        const size_t cap = (size_t)tdq_sm_count() * PER_SM * 2;
        if (blocks > cap) blocks = cap;
        if (blocks == 0) blocks = 1;
        k_combine<T, NK, THREADS, U, false><<<(unsigned)blocks, THREADS, 0, st>>>(c, row, (T *)out, (const T *)y0, kp, n);
    }
    return 0;
}

template <typename T>
int dispatch_combine(int nk, const TdqCtrl *c, int row, void *out, const void *y0, const KPtrs &kp, size_t n,
                     bool vec, cudaStream_t st) {
    switch (nk) {
#define TDQ_CASE(N) case N: return launch_combine<T, N>(c, row, out, y0, kp, n, vec, st);
        TDQ_CASE(1) TDQ_CASE(2) TDQ_CASE(3) TDQ_CASE(4) TDQ_CASE(5) TDQ_CASE(6) TDQ_CASE(7) TDQ_CASE(8)
        TDQ_CASE(9) TDQ_CASE(10) TDQ_CASE(11) TDQ_CASE(12) TDQ_CASE(13) TDQ_CASE(14) TDQ_CASE(15)
        TDQ_CASE(16) TDQ_CASE(17)
#undef TDQ_CASE
    }
    return -1;
}

// ------------------------------------------------------------------------------------------------
// Final combine + error prefix.  NU = size of the UNION of the row's and the error weights' stage slots
// that exist when the row is evaluated; rpos[m] / epos[m] give the union term's position in the
// compacted coefficient lists of the control block (coef[row][.], ecoef[.]) or -1.
// Each sum keeps the reference's ascending-j order over its own non-zero terms.
// ------------------------------------------------------------------------------------------------
struct FinalMap {
    signed char rpos[TDQ_MAX_K];
    signed char epos[TDQ_MAX_K];
};

// Coefficients live in registers.  A shared-memory variant (volatile reads at the point of use, ~45 registers and one
// block per SM of occupancy saved) was measured on B200 and is slower: dopri5's last row 0.063 vs 0.038 ms, dopri8/float64
// no better than registers (83 vs 80 us) -- the extra LDS traffic in the inner loop costs more than the occupancy buys.
template <typename T, int NU, bool VECTOR>
__global__ void __launch_bounds__(256)
k_combine_final(const TdqCtrl *__restrict__ c, int row, T *__restrict__ out, T *__restrict__ err_out, const T *y0,
                KPtrs kp, FinalMap fm, size_t n) {
    if (c->halt) return;
    using A = Ar<T>;
    // two vectors per operand per thread for every row width: measured on dopri8/float64 (NU = 9), one vector per
    // operand halves the bandwidth (126 us vs 75 us) even at twice the occupancy -- bytes in flight per thread matter
    constexpr int THREADS = 256, U = 2;
    T cr[NU], ce[NU];
    unsigned mask_r = 0, mask_e = 0;
    const T *k[NU];
    if (y0 == nullptr) y0 = reinterpret_cast<const T *>(c->y0_cur);
#pragma unroll
    for (int m = 0; m < NU; ++m) {
        const bool ur = fm.rpos[m] >= 0, ue = fm.epos[m] >= 0;
        if (ur) mask_r |= 1u << m;
        if (ue) mask_e |= 1u << m;
        const T vr = ur ? (T)c->coef[row][fm.rpos[m]] : (T)0;
        const T ve = ue ? (T)c->ecoef[fm.epos[m]] : (T)0;
        cr[m] = vr;
        ce[m] = ve;
        k[m] = tdq_detach(reinterpret_cast<const T *>(kp.p[m] ? kp.p[m] : c->k0_cur), n);
    }
    y0 = tdq_detach(y0, n);
    auto element = [&](T y, const T *kv, T &yo, T &eo) {
        T ar = (T)0, ae = (T)0;
        bool fr = true, fe = true;
#pragma unroll
        for (int m = 0; m < NU; ++m) {
            if ((mask_r >> m) & 1u) {
                const T p = A::mul(kv[m], cr[m]);
                ar = fr ? p : A::add(ar, p);
                fr = false;
            }
            if ((mask_e >> m) & 1u) {
                const T p = A::mul(kv[m], ce[m]);
                ae = fe ? p : A::add(ae, p);
                fe = false;
            }
        }
        yo = A::add(y, ar);
        eo = ae;
    };
    if (VECTOR) {
        using V = Vec<T>;
        const size_t nvec = n / V::N;
        const size_t stride = (size_t)gridDim.x * (THREADS * U);
        for (size_t base = (size_t)blockIdx.x * (THREADS * U) + threadIdx.x; base < nvec; base += stride) {
            V a[U], kv[U][NU];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const size_t v = base + (size_t)u * THREADS;
                if (v < nvec) {
                    a[u] = ld_stream<T>(y0 + v * V::N);
#pragma unroll
                    for (int m = 0; m < NU; ++m) kv[u][m] = ld_stream<T>(k[m] + v * V::N);
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const size_t v = base + (size_t)u * THREADS;
                if (v < nvec) {
                    V r, q;
#pragma unroll
                    for (int e = 0; e < V::N; ++e) {
                        T ke[NU];
#pragma unroll
                        for (int m = 0; m < NU; ++m) ke[m] = kv[u][m].v[e];
                        element(a[u].v[e], ke, r.v[e], q.v[e]);
                    }
                    st_vec<T>(out + v * V::N, r);
                    st_vec<T>(err_out + v * V::N, q);
                }
            }
        }
        if (blockIdx.x == 0) {
            const size_t i = nvec * V::N + threadIdx.x;
            if (i < n) {
                T ke[NU];
#pragma unroll
                for (int m = 0; m < NU; ++m) ke[m] = k[m][i];
                element(y0[i], ke, out[i], err_out[i]);
            }
        }
    } else {
        for (size_t i = (size_t)blockIdx.x * THREADS + threadIdx.x; i < n; i += (size_t)gridDim.x * THREADS) {
            T ke[NU];
#pragma unroll
            for (int m = 0; m < NU; ++m) ke[m] = k[m][i];
            element(y0[i], ke, out[i], err_out[i]);
        }
    }
}

template <typename T, int NU>
int launch_final(const TdqCtrl *c, int row, void *out, void *err_out, const void *y0, const KPtrs &kp,
                 const FinalMap &fm, size_t n, bool vec, cudaStream_t st) {
    constexpr int THREADS = 256, U = 2;
    if (vec) {
        const size_t nvec = n / Vec<T>::N;
        size_t blocks = (nvec + (size_t)THREADS * U - 1) / ((size_t)THREADS * U);
        const size_t cap = (size_t)tdq_sm_count() * 8;
        if (blocks > cap) blocks = cap;
        if (blocks == 0) blocks = 1;
        k_combine_final<T, NU, true><<<(unsigned)blocks, THREADS, 0, st>>>(c, row, (T *)out, (T *)err_out,
                                                                            (const T *)y0, kp, fm, n);
    } else {
        size_t blocks = (n + THREADS - 1) / THREADS;
        const size_t cap = (size_t)tdq_sm_count() * 16;
        if (blocks > cap) blocks = cap;
        if (blocks == 0) blocks = 1;
        k_combine_final<T, NU, false><<<(unsigned)blocks, THREADS, 0, st>>>(c, row, (T *)out, (T *)err_out,
                                                                             (const T *)y0, kp, fm, n);
    }
    return 0;
}

template <typename T>
int dispatch_final(int nu, const TdqCtrl *c, int row, void *out, void *err_out, const void *y0, const KPtrs &kp,
                   const FinalMap &fm, size_t n, bool vec, cudaStream_t st) {
    switch (nu) {
#define TDQ_CASE(N) case N: return launch_final<T, N>(c, row, out, err_out, y0, kp, fm, n, vec, st);
        TDQ_CASE(1) TDQ_CASE(2) TDQ_CASE(3) TDQ_CASE(4) TDQ_CASE(5) TDQ_CASE(6) TDQ_CASE(7) TDQ_CASE(8)
        TDQ_CASE(9) TDQ_CASE(10) TDQ_CASE(11) TDQ_CASE(12) TDQ_CASE(13) TDQ_CASE(14) TDQ_CASE(15)
        TDQ_CASE(16) TDQ_CASE(17)
#undef TDQ_CASE
    }
    return -1;
}

}  // namespace

int tdq_sm_count() {
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
            sms = 148;
    }
    return sms;
}

void tdq_shape_from_tableau(const tdq_tableau *tab, TdqHostShape *h) {
    memset(h, 0, sizeof(*h));
    const int S = tab->n_stages;
    h->n_stages = S;
    h->fsal = tab->fsal;
    for (int i = 0; i < S; ++i) {
        int m = 0;
        for (int j = 0; j <= i; ++j)
            if (tab->beta[i][j] != 0.0) h->row_idx[i][m++] = j;
        h->row_nnz[i] = m;
    }
    int m = 0;
    for (int j = 0; j <= S; ++j)
        if (tab->c_sol[j] != 0.0) h->row_idx[S][m++] = j;
    h->row_nnz[S] = m;
    m = 0;
    for (int j = 0; j <= S; ++j)
        if (tab->c_err[j] != 0.0) h->err_idx[m++] = j;
    h->err_nnz = m;
    m = 0;
    for (int j = 0; j <= S; ++j)
        if (tab->c_mid[j] != 0.0) h->mid_idx[m++] = j;
    h->mid_nnz = m;
    h->valid = 1;
}

extern "C" {

int tdq_stage_combine(void *ctrl_dev, const tdq_tableau *tab, int32_t dtype, int32_t row, void *y_out,
                      const void *y0, const void *const *k, size_t n, void *stream) {
    TDQ_REQUIRE(ctrl_dev && tab && y_out && k, "null argument");
    TDQ_REAL_VIEW(dtype, n);
    TdqHostShape hs;
    tdq_shape_from_tableau(tab, &hs);
    TDQ_REQUIRE(row >= 0 && row <= hs.n_stages, "row out of range");
    const int nk = hs.row_nnz[row];
    TDQ_REQUIRE(nk >= 1, "empty tableau row");
    KPtrs kp;
    memset(&kp, 0, sizeof(kp));
    bool vec = tdq_aligned16(y_out) && tdq_aligned16(y0);
    for (int m = 0; m < nk; ++m) {
        const int j = hs.row_idx[row][m];
        kp.p[m] = k[j];
        TDQ_REQUIRE(kp.p[m] != nullptr || j == 0, "missing stage slot for a non-zero tableau entry");
        vec = vec && tdq_aligned16(kp.p[m]);
    }
    if (n == 0) return TDQ_OK;
    int rc = -1;
    TDQ_DISPATCH_T(dtype, rc = dispatch_combine<T>(nk, (const TdqCtrl *)ctrl_dev, row, y_out, y0, kp, n, vec,
                                                   (cudaStream_t)stream));
    TDQ_REQUIRE(rc == 0, "unsupported number of stage terms");
    TDQ_CHECK_CUDA(cudaGetLastError());
    return TDQ_OK;
}

int tdq_stage_combine_final(void *ctrl_dev, const tdq_tableau *tab, int32_t dtype, void *y1_out, void *err_out,
                            const void *y0, const void *const *k, size_t n, void *stream) {
    TDQ_REQUIRE(ctrl_dev && tab && y1_out && err_out && k, "null argument");
    TDQ_REAL_VIEW(dtype, n);
    TdqHostShape hs;
    tdq_shape_from_tableau(tab, &hs);
    const int S = hs.n_stages;
    const int row = hs.fsal ? S - 1 : S;          // FSAL: y1 is the last stage value (rk_common.py:83-87)
    const int avail = hs.fsal ? S - 1 : S;        // highest stage slot that exists when the row is evaluated
    // union of the row's and the error weights' slots, ascending
    int used_r[TDQ_MAX_K], used_e[TDQ_MAX_K];
    for (int j = 0; j < TDQ_MAX_K; ++j) used_r[j] = used_e[j] = -1;
    for (int m = 0; m < hs.row_nnz[row]; ++m) used_r[hs.row_idx[row][m]] = m;
    for (int m = 0; m < hs.err_nnz; ++m)
        if (hs.err_idx[m] <= avail) used_e[hs.err_idx[m]] = m;
    KPtrs kp;
    FinalMap fm;
    memset(&kp, 0, sizeof(kp));
    memset(&fm, 0xff, sizeof(fm));
    int nu = 0;
    bool vec = tdq_aligned16(y1_out) && tdq_aligned16(err_out) && tdq_aligned16(y0);
    for (int j = 0; j <= avail; ++j) {
        if (used_r[j] < 0 && used_e[j] < 0) continue;
        kp.p[nu] = k[j];
        TDQ_REQUIRE(kp.p[nu] != nullptr || j == 0, "missing stage slot for a non-zero tableau entry");
        vec = vec && tdq_aligned16(kp.p[nu]);
        fm.rpos[nu] = (signed char)used_r[j];
        fm.epos[nu] = (signed char)used_e[j];
        ++nu;
    }
    TDQ_REQUIRE(nu >= 1, "empty tableau row");
    if (n == 0) return TDQ_OK;
    int rc = -1;
    TDQ_DISPATCH_T(dtype, rc = dispatch_final<T>(nu, (const TdqCtrl *)ctrl_dev, row, y1_out, err_out, y0, kp, fm, n,
                                                 vec, (cudaStream_t)stream));
    TDQ_REQUIRE(rc == 0, "unsupported number of stage terms");
    TDQ_CHECK_CUDA(cudaGetLastError());
    return TDQ_OK;
}

}  // extern "C"
