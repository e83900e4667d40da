/*
 * tdq.h -- C ABI of libtdq (torchdiffeq_b200/csrc), the sm_100a implementation of the
 * explicit Runge-Kutta hot path of rtqichen/torchdiffeq.
 *
 * Boundary rules (SURVEY.md section 8(b)):
 *   - plain pointers and sizes only; no torch types.  Every `void *stream` is a cudaStream_t.
 *   - the CALLER allocates every device buffer (state vectors, stage slots, partials, the control
 *     block).  The library owns nothing but the mapped-host mailbox it hands out on request.
 *   - every launcher is asynchronous and stream ordered, hence capturable into a CUDA graph.
 *   - every entry point returns a tdq_status; tdq_last_error() gives the text for the calling thread.
 *
 * Each entry point names the reference code (file:line under torchdiffeq/_impl/) it replaces.
 * The Python host (torchdiffeq_b200/) binds these with ctypes; INTEGRATION.md shows the binding a
 * reference maintainer would add.
 */
#ifndef TDQ_H_
#define TDQ_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TDQ_ABI_VERSION 2

#define TDQ_MAX_STAGES 16            /* func evaluations per attempt, excluding f0 (dopri8: 13)   */
#define TDQ_MAX_K      (TDQ_MAX_STAGES + 1) /* stage slots k_0 .. k_S                              */
#define TDQ_MAX_SEGS   64            /* segments of a mixed (max-of-rms) norm                      */
#define TDQ_MAX_RANKS  16            /* ranks of one NVLink domain sharing a sharded solve         */

typedef enum {
    TDQ_OK = 0,
    TDQ_ERR_INVALID = 1,   /* bad argument (null pointer, unsupported dtype, too many stages ...)   */
    TDQ_ERR_CUDA = 2,      /* a CUDA runtime call failed; see tdq_last_error()                     */
    TDQ_ERR_UNSUPPORTED = 3
} tdq_status;

/* State dtypes.  A complex state (TDQ_C64 = complex64, TDQ_C128 = complex128) is stored as interleaved (re, im)
 * pairs of its component dtype (float32 / float64).  For a complex code every element count `n`, every segment
 * offset and length and every chunk-table entry counts COMPLEX elements, and every state, stage, coefficient and
 * solution buffer holds n complex values.  Everything that is a real scalar or a real coefficient array stays in the
 * component dtype: tdq_options.dtype, the control block (tdq_ctrl_init takes only TDQ_F32 / TDQ_F64, and tstage /
 * taux are component-dtype scalars), the dtype passed to tdq_prepare_attempt, tdq_controller, tdq_initial_step_h0 /
 * _finish, the dt / slope / cubic-weight arrays of the fixed-grid launchers, and the ratio of tdq_controller.
 * Norms use the complex modulus: |z| = hypot(re, im), one tolerance per complex element, err/tol = err*fl(1/tol)
 * componentwise, and each complex element contributes |err/tol|^2 once.  complex32 has no code. */
typedef enum { TDQ_F32 = 0, TDQ_F64 = 1, TDQ_C64 = 2, TDQ_C128 = 3 } tdq_dtype;

/* Solver status word kept in the control block (device) and mirrored into the mailbox.
 * Mirrors the three assertions of the reference's adaptive loop. */
typedef enum {
    TDQ_RUN_OK = 0,
    TDQ_RUN_DT_UNDERFLOW = 1,   /* rk_common.py:286  assert t0 + dt > t0                          */
    TDQ_RUN_NONFINITE = 2,      /* rk_common.py:287  assert isfinite(y0).all()                     */
    TDQ_RUN_MAX_STEPS = 3,      /* rk_common.py:247  assert n_steps < max_num_steps                */
    TDQ_RUN_EXCHANGE_TIMEOUT = 4 /* a peer rank never delivered its norm partials (sharded solves)  */
} tdq_run_status;

/* Butcher tableau of an explicit embedded RK method, float64 as in the reference
 * (rk_common.py:15 _ButcherTableau; dopri5.py:5-30; dopri8.py:5-70; tsit5.py, bosh3.py,
 * fehlberg2.py, adaptive_heun.py).  beta is lower triangular: row i has i+1 entries. */
typedef struct {
    int32_t n_stages;                 /* S                                                          */
    int32_t order;                    /* controller order (dopri5 5, dopri8 8)                      */
    int32_t fsal;                     /* 1: y1 is the last stage value (rk_common.py:83 shortcut)   */
    int32_t reserved;
    double alpha[TDQ_MAX_STAGES];
    double beta[TDQ_MAX_STAGES][TDQ_MAX_K];
    double c_sol[TDQ_MAX_K];
    double c_err[TDQ_MAX_K];
    double c_mid[TDQ_MAX_K];
} tdq_tableau;

/* Adaptive-solver options; names and defaults follow RKAdaptiveStepsizeODESolver.__init__
 * (rk_common.py:166-177). */
typedef struct {
    int32_t dtype;                    /* tdq_dtype of the state                                     */
    int32_t ratio_f64;                /* 1: error ratio kept in float64 (vector tolerances)         */
    double rtol, atol;                /* scalar tolerances (ignored by the vector-tol norm kernel)  */
    double min_step, max_step;
    double safety, ifactor, dfactor;
    double t_sign;                    /* +1, or -1 when the caller integrates -t (misc.py:273-279): */
                                      /* func sees t_sign*t and stage slots hold RAW func outputs;  */
                                      /* the -1 of _ReverseFunc (misc.py:158-165) is folded into    */
                                      /* every coefficient instead of a pass over f.                */
    int64_t max_num_steps;            /* per output interval (rk_common.py:247)                     */
    int64_t n_global;                 /* element count the RMS mean divides by (all ranks)          */
    /* State pointer table.  The accepted state y0 and its derivative f0 = k_0 live in ybuf[par]/kbuf[par]  */
    /* (par = 0 when a solve starts: the caller puts y(t[0]) into ybuf[0] and f(t[0], y0) into kbuf[0]).     */
    /* tdq_error_norm_commit writes every attempt's candidate (y1, k_S) into the other pair and             */
    /* tdq_controller accepts by flipping par -- rk_common.py:341,:352 without a copy.  Four caller-owned    */
    /* device buffers of n elements, 16-byte aligned; all NULL = no table (every launcher then needs y0 and  */
    /* k[0] explicitly and nothing is committed).                                                           */
    void *ybuf[2];
    void *kbuf[2];
    int32_t always_fit;               /* 1: fit the interpolant on EVERY accepted step (dense output, events) */
    int32_t reserved;
    uint64_t loop_handle;             /* tdq_loop_create's handle when attempts run inside the device-side   */
                                      /* while loop, else 0                                                  */
} tdq_options;

/* Mapped-host mailbox the controller kernel writes after every attempt; the host polls `seq`
 * instead of synchronising the stream. */
typedef struct {
    volatile uint64_t seq;            /* attempts finished so far (written last)                    */
    volatile int32_t status;          /* tdq_run_status                                             */
    volatile int32_t accept;          /* last attempt accepted?                                     */
    volatile int32_t done;            /* all requested output times emitted                         */
    volatile int32_t out_cursor;      /* next output index to emit                                  */
    volatile int64_t n_accept, n_reject;
    volatile double t0, t1, dt;       /* last accepted interval and the next step size              */
    volatile double ratio;            /* error ratio of the last attempt                            */
    volatile double att_t0, att_dt;   /* start time and step size the last attempt used             */
    volatile double next_t0, next_dt; /* the same for the attempt prepared next (callback_step)     */
    volatile int32_t on_jump_t;       /* the accepted attempt ended on a jump_t point: the host must */
                                      /* re-evaluate f at taux[2] = next(T(t1)) (rk_common.py:346-351) */
    volatile int32_t par;             /* which pair of the pointer table holds the accepted state now */
} tdq_mailbox;

/* ---- library ------------------------------------------------------------------------------ */
int tdq_abi_version(void);
/* sizeof the ABI structs as compiled (0: tdq_tableau, 1: tdq_options, 2: tdq_mailbox); lets a foreign
 * binding verify its own struct definitions. */
size_t tdq_sizeof(int32_t which);
const char *tdq_last_error(void);
/* Number of SMs of the current device (grid sizing). */
int tdq_device_sm_count(int *out);

/* Named tableaus: "dopri5", "dopri8", "tsit5", "bosh3", "fehlberg2", "adaptive_heun". */
int tdq_tableau_get(const char *name, tdq_tableau *out);

/* Mapped, pinned host memory for a mailbox (cudaHostAlloc mapped); dev_ptr is what kernels get. */
int tdq_mailbox_create(tdq_mailbox **host_ptr, void **dev_ptr);
int tdq_mailbox_destroy(tdq_mailbox *host_ptr);

/* ---- control block ------------------------------------------------------------------------ */
/* Size in bytes of the device control block, and offsets of the state-dtype scalars torch views
 * alias as func's time argument: tstage[i] = time func sees at stage i (already perturbed and
 * sign-corrected); taux[0] = time of f0, taux[1] = probe time of the initial-step heuristic,
 * taux[2] = Perturb.NEXT time after a jump_t point (taux has 4 slots). */
size_t tdq_ctrl_size(void);
size_t tdq_ctrl_tstage_offset(void);
size_t tdq_ctrl_taux_offset(void);

/* Fill the control block: tableau cast to the state dtype (rk_common.py:201-205), options, start
 * time t_start = t[0], output times (device float64 array of n_out ascending values; misc.py:273-279
 * negates for the caller; must stay alive for the solve).  Replaces
 * RKAdaptiveStepsizeODESolver.__init__ (rk_common.py:166-205) and the scalar part of
 * _before_integrate (:213-221).  Not capturable (host-to-device copy of the block). */
int tdq_ctrl_init(void *ctrl_dev, const tdq_tableau *tab, const tdq_options *opt, const double *t_out_dev,
                  double t_start, int32_t n_out, void *mailbox_dev, void *stream);

/* Optional sorted step_t grid (device float64, values >= t[0]); rk_common.py:223-241, :293-300. */
int tdq_ctrl_set_step_t(void *ctrl_dev, const double *step_t_dev, int32_t n, void *stream);
/* Optional sorted jump_t points (discontinuities of func); rk_common.py:229-241, :302-308, :346-351.
 * Steps are clipped to them on the device; after an accepted step that ended on one, the mailbox says
 * so and taux[2] holds the Perturb.NEXT time at which the host re-evaluates f (lock-step callers). */
int tdq_ctrl_set_jump_t(void *ctrl_dev, const double *jump_t_dev, int32_t n, void *stream);

/* ---- norms: deterministic segmented sum of squares ---------------------------------------- */
/* A norm is max over SEGMENTS of rms(segment) (misc.py:22-23, :30-33, adjoint.py:247-271).  One segment
 * covering [0,n) needs no table.  Anything else -- tuple states, the adjoint's augmented state with one
 * segment per parameter tensor, any number of them -- is described by a CHUNK TABLE in device memory:
 * tdq_norm_table_fill() writes it into a HOST buffer of int64 words that the caller uploads once per solver
 * (the library owns no memory).  Segments must be ascending and disjoint; elements outside every segment
 * (padding, the parameter block under 'seminorm') are still committed and still checked for non-finite
 * values, they just enter no norm.  Returns the number of words needed (call with table_host == NULL to
 * size the buffer), or -1.  table_host[1] = number of chunks, table_host[3] = 1 when every segment starts
 * on a 16-byte boundary (pass both to the launchers below). */
int64_t tdq_norm_table_fill(const int64_t *seg_offsets, const int64_t *seg_lens, int32_t n_seg, int64_t n,
                            int32_t dtype, int64_t *table_host, int64_t capacity_words);
/* Doubles the caller must provide (zero-initialised ONCE) as `partials` for the reductions below;
 * n_chunks = 0 without a table. */
size_t tdq_norm_partials_len(size_t n, int64_t n_chunks);

/* ---- initial step (misc.py:36-77 _select_initial_step) ------------------------------------ */
/* out[s] = sum over segment s of (x/scale)^2 (or ((x - x2)/scale)^2 when x2 != NULL),
 * scale = atol + |y0|*rtol (misc.py:55-58, :69); without x2, out[n_seg] = number of non-finite y0
 * elements (the pass over y0 doubles as the check of rk_common.py:287 for the first attempt).
 * y0 == NULL: the control block's current y0.  table_dev/n_chunks/table_aligned: chunk table or
 * NULL/0/0 with n_seg == 1.  rtol_vec/atol_vec: optional per-element float64. */
int tdq_scaled_sumsq(void *ctrl_dev, int32_t dtype, const void *x, const void *x2, const void *y0,
                     const double *rtol_vec, const double *atol_vec, const int64_t *table_dev, int64_t n_chunks,
                     int32_t table_aligned, int32_t n_seg, size_t n, double *partials, double *out, void *stream);
/* h0 from d0 = norm(y0/scale), d1 = norm(f0/scale) given as (all-reduced) segment sums; also sets
 * taux[1] = probe time t0 + h0 (misc.py:60-67).  seg_counts_dev: GLOBAL element count per segment
 * (device int64) or NULL for a single segment of options.n_global elements. */
int tdq_initial_step_h0(void *ctrl_dev, int32_t dtype, const double *d0_sumsq, const double *d1_sumsq,
                        const int64_t *seg_counts_dev, int32_t n_seg, void *stream);
/* y_probe = y0 + h0*f0 (misc.py:66); f0 is the RAW func output (t_sign applied inside).  NULL y0 / f0: the
 * control block's current pair. */
int tdq_initial_step_probe(void *ctrl_dev, int32_t dtype, void *y_probe, const void *y0, const void *f0,
                           size_t n, void *stream);
/* dt = min(100*h0, h1) from d2 = norm((f1 - f0)/scale)/h0 (misc.py:69-77). */
int tdq_initial_step_finish(void *ctrl_dev, int32_t dtype, const double *d2_sumsq,
                            const int64_t *seg_counts_dev, int32_t n_seg, void *stream);
/* options['first_step'] (rk_common.py:218-219). */
int tdq_set_first_step(void *ctrl_dev, double first_step, void *stream);

/* ---- one adaptive attempt (rk_common.py:266-361 _adaptive_step) --------------------------- */
/* Start-of-attempt scalar work: clamp dt, t1 = t0 + dt, step_t clipping, the dt-underflow and
 * max_num_steps assertions, stage times t_i = T(t0) + alpha_i*T(dt) (or prev(T(t1)) when
 * alpha_i == 1) and coefficients fl_T(beta_ij*T(dt)); rk_common.py:246-247, :269-308, :61-79, :89.
 * tdq_controller already does this for attempt n+1, so the host calls it once per solve. */
/* y0_nonfinite_count_dev: optional device double (tdq_scaled_sumsq's out[n_seg] for x = y0); when it is
 * positive the first attempt fails with TDQ_RUN_NONFINITE exactly where the reference asserts (:287, after
 * the underflow check :286). */
int tdq_prepare_attempt(void *ctrl_dev, int32_t dtype, const double *y0_nonfinite_count_dev, void *stream);

/* y_out = y0 + sum_j k_j * coef[row][j] over the non-zero tableau entries (rk_common.py:79, :85).
 * row in [0, S): stage rows; row == S: the c_sol row of a non-FSAL tableau.  k[j] is stage slot j
 * (RAW func output), NULL allowed where the tableau entry is zero.  `tab` only selects the
 * sparsity pattern; coefficients come from the control block.  No-op once the solve has halted.
 * y0 == NULL and k[0] == NULL select the control block's current pair (pointer table). */
int tdq_stage_combine(void *ctrl_dev, const tdq_tableau *tab, int32_t dtype, int32_t row, void *y_out,
                      const void *y0, const void *const *k, size_t n, void *stream);

/* The LAST combine of an attempt -- the row that yields y1: stage row S-1 for FSAL tableaus
 * (rk_common.py:83-87), the c_sol row otherwise (:85) -- fused with the part of the embedded error
 * estimate (:89) whose stage slots exist at that point:
 *     y1_out  = y0 + sum_j k_j*fl(dt*c_sol_j)
 *     err_out = sum_{j <= avail} k_j*fl(dt*e_j)       ascending j; avail = S-1 (FSAL) or S
 * One pass over k_0..k_avail instead of two.  Same NULL conventions as tdq_stage_combine. */
int tdq_stage_combine_final(void *ctrl_dev, const tdq_tableau *tab, int32_t dtype, void *y1_out, void *err_out,
                            const void *y0, const void *const *k, size_t n, void *stream);

/* Error ratio + candidate commit (rk_common.py:89 tail + misc.py:80-82 + :22-23/:30-33; rk_common.py:338-352):
 *     err = err_pre (+ k_last*fl(dt*e_S) when the tableau is FSAL and e_S != 0; k_last = k_S)
 *     tol = atol + rtol*max(|y0|,|y1|);  out[s] = sum over segment s of (err/tol)^2
 *     out[n_seg] = number of non-finite y1 elements
 * and, in the same pass, y1 -> ybuf[par^1], k_last -> kbuf[par^1] (the candidate the controller accepts by
 * flipping par).  err_over_tol_out, if non-NULL, receives err/tol (state dtype; float64 with vector
 * tolerances) for callers with a custom norm callable.  Chunk table as for tdq_scaled_sumsq. */
int tdq_error_norm_commit(void *ctrl_dev, int32_t dtype, const void *err_pre, const void *k_last, const void *y0,
                          const void *y1, const double *rtol_vec, const double *atol_vec, const int64_t *table_dev,
                          int64_t n_chunks, int32_t table_aligned, int32_t n_seg, size_t n, double *partials,
                          double *out, void *err_over_tol_out, void *stream);
/* The candidate commit alone: y1 -> ybuf[par^1], k_last -> kbuf[par^1]. */
int tdq_commit_candidates(void *ctrl_dev, int32_t dtype, const void *y1, const void *k_last, size_t n, void *stream);

/* Accept/reject, I-controller, bookkeeping, output cursor, the NEXT attempt's constants, mailbox
 * (rk_common.py:323-361, misc.py:85-95, solvers.py:33-34, then :269-308 for the next attempt).
 * norm_in: the (all-reduced) output of tdq_error_norm_commit.  If ratio_dev != NULL (state dtype scalar,
 * float64 when options.ratio_f64) the ratio is read from there instead (custom norm callable). */
int tdq_controller(void *ctrl_dev, int32_t dtype, const double *norm_in, const int64_t *seg_counts_dev,
                   int32_t n_seg, const void *ratio_dev, void *stream);

/* Lazy dense output of the attempt the controller just accepted (rk_common.py:363-369, interp.py:1-48 via
 * rk_common.py:243-250 / solvers.py:28-35).  Does something only when an output time t_j fell into (t0, t1]
 * or options.always_fit is set: forms y_mid and the quartic's coefficients from (y0, y1, k_0, k_S, the
 * mid-point slots) -- y0/k_0 are the pair the accepted step started from -- writes solution[j] for every such
 * t_j (solution is [n_out, n] in the state dtype) and, when coeff != NULL, stores coeff[0..4] = e,d,c,b,a. */
int tdq_interp_fit_eval(void *ctrl_dev, const tdq_tableau *tab, int32_t dtype, const void *y1, const void *const *k,
                        void *const *coeff, void *solution, size_t n, void *stream);
/* Evaluate the current interpolant at one time (device float64 scalar) into out[n] (interp.py:25-48). */
int tdq_interp_eval_at(void *ctrl_dev, int32_t dtype, const void *const *coeff, const double *t_dev, void *out,
                       size_t n, void *stream);
/* out = c0 + x*c1 + x^2*c2 + x^3*c3 + x^4*c4 with x = T(x64) (interp.py:39-46) for coefficient sets the caller keeps
 * itself, e.g. one per accepted step for a dense-output closure (odeint.py:111-157). */
int tdq_poly_eval(int32_t dtype, const void *const *coeff, double x, void *out, size_t n, void *stream);
/* Reset the per-output-interval attempt counter (rk_common.py:245). */
int tdq_ctrl_reset_interval(void *ctrl_dev, void *stream);

/* ---- the adaptive loop itself on the device (solvers.py:28-35, rk_common.py:243-250) ----------- */
/* The reference's `while next_t > t1: _adaptive_step()` is a host loop with a dozen syncs per iteration.
 * Here one attempt is a CUDA graph (captured by the caller: stage combines, func, norm, controller, fit) and
 * the loop is a conditional WHILE node around it: tdq_controller, the last decision of every attempt, calls
 * cudaGraphSetConditional(handle, !halt) from the device, so a whole solve is ONE graph launch with no host
 * in the loop and no attempt executed after the end.
 * tdq_loop_create clones `body_graph` (a cudaGraph_t; it may be destroyed afterwards) into the body of a new
 * executable graph; *handle_out goes into tdq_options.loop_handle (or tdq_ctrl_set_loop) of every solve that
 * is launched with tdq_loop_launch, and must be 0 for attempts launched any other way. */
int tdq_loop_create(void *body_graph, void **loop_out, uint64_t *handle_out);
int tdq_loop_launch(void *loop, void *stream);
int tdq_loop_destroy(void *loop);
int tdq_ctrl_set_loop(void *ctrl_dev, uint64_t loop_handle, void *stream);

/* ---- fixed grid: RK4 3/8 rule (fixed_grid.py:24-29, rk_common.py:110-118) and the other explicit
 *      fixed-step methods euler / midpoint / heun2 / heun3 (fixed_grid.py:6-60, rk_common.py:121-158) -- */
/* which = 1: y0 + (dt*k1)*(1/3);  2: y0 + dt*(k2 - k1*(1/3));  3: y0 + dt*((k1 - k2) + k3);
 * 4: y1 = y0 + ((k1 + 3*(k2 + k3)) + k4)*dt*0.125 (solvers.py:115);
 * 5: y0 + dt*k1 (euler; midpoint and heun2 pass the relevant k as k1);  6: y0 + k1*(0.5*dt) (midpoint stage);
 * 7: y0 + dt*(k1*0.5 + k2*0.5) (heun2);  8: y0 + dt*(k2*(2/3)) (heun3 stage 3);  9: y0 + dt*(k1*0.25 + k3*0.75) (heun3).
 * dt is dt_dev[step_dev[0]] (state dtype array, int64 device step counter; step_dev may be NULL for
 * index 0) so that one captured graph serves every step of the grid. */
int tdq_rk4_stage(int32_t dtype, int32_t which, void *y_out, const void *y0, const void *k1,
                  const void *k2, const void *k3, const void *k4, const void *dt_dev,
                  const int64_t *step_dev, size_t n, void *stream);
/* End of one fixed-grid step (solvers.py:117-126, :175-181, linear interpolation): for every record r
 * in [rec_begin[step], rec_begin[step+1]): solution[out_idx[r]] = y0 | y1 | y0 + slope[r]*(y1 - y0)
 * for mode[r] = 0|1|2; then y0 <- y1, the step counter is incremented and the next step's four func
 * times are copied from tstage_all[step+1][0..4) to tstage_cur[0..4) (state dtype; what func's time
 * argument aliases).  step_dev points at TWO int64 words: [0] the step counter, [1] a ticket the kernel uses
 * (zero-initialised by the caller, self-resetting). */
int tdq_fixed_emit(int32_t dtype, void *y0, const void *y1, void *solution,
                   const int32_t *rec_begin_dev, const int32_t *out_idx_dev, const int32_t *mode_dev,
                   const void *slope_dev, int64_t *step_dev, const void *tstage_all_dev,
                   void *tstage_cur_dev, int64_t n_steps, size_t n, void *stream);

/* The final expression of a step (which = 4 rk4, 5 euler / midpoint, 7 heun2, 9 heun3; operands as for tdq_rk4_stage)
 * fused with tdq_fixed_emit: y1 = y0 + dy is formed in registers, the step's linear-interpolation records are written
 * and y0 <- y1 -- one launch and 2 N*s less than tdq_rk4_stage followed by tdq_fixed_emit. */
int tdq_fixed_final_emit(int32_t dtype, int32_t which, void *y0, const void *k1, const void *k2, const void *k3,
                         const void *k4, const void *dt_dev, void *solution, const int32_t *rec_begin_dev,
                         const int32_t *out_idx_dev, const int32_t *mode_dev, const void *slope_dev, int64_t *step_dev,
                         const void *tstage_all_dev, void *tstage_cur_dev, int64_t n_steps, size_t n, void *stream);

/* Multistep (Adams) predictor / corrector sums (fixed_adams.py:198-215): out = [base +] sum_m x_m * T(coefs[m]), products
 * and sums rounded separately, ascending m, first product initialising the sum (Python's sum()).  x, coefs: HOST
 * arrays of n_terms <= TDQ_MAX_K entries; coefficients are float64 values the kernel casts to the state dtype (what torch
 * does with a 0-dim float64 tensor times a state tensor); base may be NULL. */
int tdq_lincomb(int32_t dtype, void *out, const void *base, const void *const *x, const double *coefs, int32_t n_terms,
                size_t n, void *stream);

/* ---- Stage fused with a LINEAR vector field f(t, y) = y W^T on the tensor cores (tdq_linear.cu) ----------------------------
 * What rk_common.py:79-81 does with two kernels and a round trip of y_i through memory -- y_i = y0 + sum_j coef_ij k_j, then
 * k_i = func(t_i, y_i) -- in one launch when func is `torchdiffeq_b200.LinearField` (float32 states [..., 128], W 128 x 128):
 * y_i is formed in registers (same products, same order as tdq_stage_combine), split into three bfloat16 planes and multiplied
 * on tcgen05 with float32 accumulation in tensor memory (three bf16 planes per operand, six products: float32-grade, rel. rms error 1e-7 against float64).
 * tdq_linear_supported: 1 if (dtype, width) has a fused kernel.  tdq_linear_weights_bytes: size of the split weights.
 * tdq_linear_prepare: W (row-major [width][width], W[n][k] = d k_n / d y_k, i.e. func = y @ W^T) -> split planes (once per solve).
 * tdq_linear_apply: k_out = y W^T for n_rows rows, no control block (f0, tests).
 * tdq_linear_stage: row `row` (0 .. S-1) of the tableau as tdq_stage_combine evaluates it, k_out = k_{row+1}; for the row
 * that yields y1 of an FSAL tableau (row S-1) y1_out and err_out are written as tdq_stage_combine_final writes them
 * (bitwise), otherwise they must be NULL.  y0 NULL / k[0] NULL: the control block's pointer table.  Rows of more than 8
 * terms are rejected (the caller keeps the unfused pair for them).  No-op after halt, like every attempt kernel. */
int tdq_linear_supported(int32_t dtype, int32_t width);
size_t tdq_linear_weights_bytes(int32_t width);
int tdq_linear_prepare(int32_t dtype, const void *weight, int32_t width, void *planes, void *stream);
int tdq_linear_apply(int32_t dtype, const void *y, const void *planes, int32_t width, size_t n_rows, void *k_out,
                     void *stream);
int tdq_linear_stage(void *ctrl_dev, const tdq_tableau *tab, int32_t dtype, int32_t row, void *k_out, void *y1_out,
                     void *err_out, const void *y0, const void *const *k, const void *planes, int32_t width, size_t n,
                     void *stream);

/* ---- A WHOLE attempt of a linear vector field in one launch (tdq_attempt.cu) ---------------------------------------------
 * For f(t, y) = y W^T an attempt is row-local, so one kernel takes every tile of 16 state rows through all S stages on chip:
 * rk_common.py:43-90 (_runge_kutta_step: every y_i, every k_i, y1, the error estimate), the squared error ratio of
 * misc.py:80-82 and the candidate commit of rk_common.py:341/:352 -- what S x tdq_linear_stage + tdq_error_norm_commit do
 * in S + 1 launches.  HBM traffic: 2 reads + 2 writes per element.  Same arithmetic, operation for operation: k_i, y1 and the
 * error prefix are bitwise what tdq_linear_stage writes.
 * tdq_linear_attempt_supported: 1 for float32, width 128 and the FSAL tableaus dopri5 / bosh3.
 * tdq_linear_attempt: y0 / k0 NULL: the control block's pointer table.  k_out[i] (i = 1..S), y1_out, err_out receive k_i, y1
 * and the error-sum prefix ONLY for attempts that can contain an output time (t_out[cursor] <= the attempt's end), when the
 * control block keeps every step (always_fit) or when store_always != 0 -- the lazy interpolant fit is their only reader.
 * partials / norm_out (both or neither): norm_out[0] = sum over the state of ((err_pre + k_S e_S) / (atol + rtol max(|y0|,|y1|)))^2,
 * norm_out[1] = number of non-finite y1 elements (what tdq_error_norm_commit writes for one segment), and y1 -> ybuf[par^1],
 * k_S -> kbuf[par^1]; partials needs tdq_norm_partials_len doubles, zeroed once.  Scalar tolerances only.  No-op after halt.
 * seg_counts_dev != NULL (needs partials / norm_out): the last block to finish also performs the controller step, exactly
 * what tdq_controller(ctrl, dtype, norm_out, seg_counts_dev, 1, NULL) would do next (rk_common.py:323-361, misc.py:85-95,
 * the peer exchange of a sharded solve included) -- the caller then skips that launch. */
int tdq_linear_attempt_supported(const tdq_tableau *tab, int32_t dtype, int32_t width);
int tdq_linear_attempt(void *ctrl_dev, const tdq_tableau *tab, int32_t dtype, void *const *k_out, void *y1_out, void *err_out,
                       const void *y0, const void *k0, const void *planes, int32_t width, size_t n, double *partials,
                       double *norm_out, const int64_t *seg_counts_dev, int32_t store_always, void *stream);

/* interp='cubic' (solvers.py:120-125, :166-173): for records r in [rec_lo, rec_hi) of one step
 * solution[out_idx[r]] = h00*y0 + (h10*dt)*f0 + h01*y1 + (h11*dt)*f1 with the four weights of record r at
 * coef_dev[4*r .. 4*r+4) (state dtype; the caller evaluates them in t's dtype like the reference and folds the
 * reverse-time sign into the two dt*f weights).  f0 = f(t0, y0) and f1 = f(t1, y1) are RAW func outputs.
 * Does not commit y0 <- y1: tdq_fixed_emit (with an empty record range) still ends the step. */
int tdq_fixed_emit_cubic(int32_t dtype, const void *y0, const void *y1, const void *f0, const void *f1, void *solution,
                         const int32_t *out_idx_dev, const void *coef_dev, int32_t rec_lo, int32_t rec_hi, size_t n,
                         void *stream);

/* ---- sharded solves: norm partials exchanged over NVLink peer memory INSIDE tdq_controller ----- */
/* The reference has no multi-GPU path; its RMS norm is a mean over the whole batch (misc.py:22-23), so
 * batch-sharded ranks must sum their n_seg+1 float64 partials before every accept/reject decision.
 * Instead of a separate collective launch, each rank's controller kernel stores its partials straight
 * into every peer's exchange buffer (P2P stores, release flag), spins on its own buffer until all
 * peers' flags for this attempt have arrived, and adds the R vectors in rank order -- every rank gets
 * the bitwise identical sum.  The buffer is the one allocation the library makes itself, because it
 * must be a whole cudaMalloc allocation to be exported with cudaIpcGetMemHandle. */
typedef struct { unsigned char bytes[64]; } tdq_ipc_handle;
int tdq_xchg_create(void **dev_ptr, tdq_ipc_handle *handle_out);
int tdq_xchg_open(const tdq_ipc_handle *handle, void **peer_ptr);
int tdq_xchg_close(void *peer_ptr);
int tdq_xchg_destroy(void *dev_ptr);
/* After tdq_ctrl_init: peer_ptrs[r] = rank r's exchange buffer as mapped in THIS process (own buffer at
 * index `rank`); epoch must be the same on all ranks and differ from solve to solve. */
int tdq_ctrl_set_exchange(void *ctrl_dev, const void *const *peer_ptrs, int32_t rank, int32_t world,
                          uint64_t epoch, void *stream);

/* ---- adjoint augmented state (adjoint.py:72-105, misc.py:137-165) ------------------------- */
/* dst[offset_i .. offset_i + len_i) = scale_i * src_i for i < n_src, one launch
 * (the torch.cat of _TupleFunc, the unary minus on adj_y and the *(-1) of _ReverseFunc).
 * src_i == NULL writes zeros (adjoint.py:100-103).  All arrays are HOST arrays. */
int tdq_pack_segments(int32_t dtype, void *dst, const void *const *src, const int64_t *offsets,
                      const int64_t *lens, const double *scales, int32_t n_src, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* TDQ_H_ */
