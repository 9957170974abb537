/*
 * fpa_b200.h -- C ABI of the B200-native fiber-parametric-amplification (FWM) solver.
 *
 * One shared library (libfpa_b200.so, built by nvcc for sm_100a) exports every
 * entry point declared here.  There are no C++ or torch types in any signature:
 * plain pointers, sizes and int status codes only, so the library can be bound
 * from ctypes / cffi / any FFI.  Exceptions never cross the ABI; every function
 * returns an FPA_* status and `fpa_last_error()` gives the text of the last
 * failure on the calling thread.
 *
 * The reference (pure Python) has no FFI of its own; the interfaces these entry
 * points stand in for are Python call signatures.  Each declaration cites the
 * reference file:line it replaces (paths relative to the reference checkout).
 *
 * Layout conventions
 *   complex128  = two consecutive doubles (re, im), exactly numpy's complex128.
 *   A[B,4]      = C-order, wave order [pump1, pump2, signal, idler].
 *   trace       = A_trace[B, n_saved, 4] complex128, n_saved = n_steps/save_every + 1
 *                 (integrators.py:115); sample 0 is the initial state (:120-122).
 *   "dev" entry points take DEVICE pointers and a cudaStream_t (passed as void*);
 *   they are asynchronous on that stream.  "host" entry points take HOST
 *   pointers, stage through a library-owned device workspace and return after
 *   the results are back in host memory.
 *
 * Alignment
 *   dev entries: the kernels move complex128 values and rows of maxima with 16-byte
 *   vector accesses, so these device pointers must be 16-byte aligned (else
 *   FPA_ERR_INVALID, error text "... must be 16-byte aligned"): yaman4 A0, A_trace,
 *   A_end, Pmax; sweep plan.omega, A_end, Pmax; phase sweep A0_table; Delta-beta
 *   table omega; N-wave A0, A_trace, A_end and `factored`.  (torch and cudaMalloc
 *   allocations are; a complex128 view at an odd element offset is not.)  The transfer
 *   kernels store jac one double at a time: its device pointer must be 8-byte aligned
 *   ("jac must be 8-byte aligned"); their other arrays follow the rules above.
 *   host entries: any naturally aligned array (numpy's rule: 8 bytes for float64 and
 *   complex128).  A page-locked result array the kernel cannot store to directly
 *   is staged like pageable memory.
 */
#ifndef FPA_B200_H
#define FPA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ status */
#define FPA_OK               0
#define FPA_ERR_INVALID      1   /* bad argument (maps to ValueError)              */
#define FPA_ERR_CUDA         2   /* CUDA runtime failure (maps to RuntimeError)    */
#define FPA_ERR_NO_DEVICE    3   /* no usable CUDA device: there is NO CPU fallback */
#define FPA_ERR_UNSUPPORTED  4   /* e.g. N-wave plan too large for the kernel      */

/* ------------------------------------------------------------------- flags */
#define FPA_OUT_TRACE   (1u << 0)  /* write A_trace[B,n_saved,N]                     */
#define FPA_OUT_END     (1u << 1)  /* write A_end[B,N] (state after the last step)   */
#define FPA_OUT_PMAX    (1u << 2)  /* write Pmax[B,N] = max over SAVED samples |A|^2  */
#define FPA_CHECK_NAN   (1u << 3)  /* per-step finite check (integrators.py:132-135) */
#define FPA_PHASE_EXACT (1u << 4)  /* the reference's arithmetic structure step by   *
                                    * step: h_i = z_{i+1}-z_i, sincos at every RK4   *
                                    * abscissa, k_1..k_4 formed (slower; default is  *
                                    * the constant-h / phase-recurrence fast kernel) */
#define FPA_NWAVE_TABLE (1u << 6)   /* N-wave: force the enumerated-triplet kernel even   *
                                    * when grid_slot is given                          */
#define FPA_NWAVE_PLAIN (1u << 8)   /* N-wave table kernel: walk the entry list even when  *
                                    * the factored form (`factored`) is at hand          */
#define FPA_NWAVE_COMB  (1u << 7)   /* N-wave: insist on the convolution-form kernel     *
                                    * (FPA_ERR_UNSUPPORTED beyond its limits); without  *
                                    * either flag the library picks: convolution form   *
                                    * for grid plans within its limits (span <= 512)    *
                                    * unless the plan is so sparse that the table has   *
                                    * less work (span^2 > 5 * n_triplets)               */
#define FPA_UNIFORM_PHYSICS (1u << 5) /* gamma and alpha are the same for every point *
                                    * (stride 0) AND their values are given in       *
                                    * gamma_uniform / alpha_uniform: the kernel then  *
                                    * keeps all stage coefficients in the constant    *
                                    * bank instead of registers                       */

/* status[b] values written by the integrators */
#define FPA_POINT_OK      (-1)     /* otherwise: index of the first step whose result was non-finite */

/* Phase-matching strategies of the sweep front-end (phase_matching.py:50-53) */
#define FPA_PM_GENERAL_TAYLOR 0
#define FPA_PM_SYMMETRIC_EVEN 1
#define FPA_PM_PROVIDED       2

#define FPA_MAX_TAYLOR_ORDER 12

const char* fpa_last_error(void);
const char* fpa_version(void);

/* Number of visible CUDA devices (0 when none; never fails). */
int fpa_device_count(void);
/* SM count, max SM clock [kHz] and name of `device`. */
int fpa_device_info(int device, int* sm_count, int* clock_khz, char* name, int name_cap);
/* Make `device` current for the calling thread in this library's CUDA runtime.  The *_dev entry
 * points run on the current device; call this once per thread when the process also uses another
 * CUDA runtime instance (e.g. PyTorch) to select devices. */
int fpa_set_device(int device);

/* ------------------------------------------------ 4-wave RK4 integrator (hot path)
 * Replaces the call chain
 *   integrators.integrate_interval      integrators.py:150-204
 *   integrators.integrate_fixed_step    integrators.py:68-142
 *   integrators.rk4_step                integrators.py:25-61
 *   yaman_model.rhs_yaman_simplified    yaman_model.py:10-52 (+ :123-186)
 * for a batch of B independent scan points in ONE kernel launch: all four RK4
 * stages and the RHS are fused, the state stays in registers for every z-step.
 *
 * Grid semantics (integrators.py:194-195, numpy.linspace): with z_grid == NULL,
 * z_i = z0 + i*((z_max-z0)/n_steps) for i<n_steps, z_n = z_max exactly, and the
 * per-step h_i = z_{i+1}-z_i by subtraction (:127-128).  With z_grid != NULL
 * (n_steps+1 doubles, shared by all points) those values are used instead and
 * the phase is evaluated with sincos at every abscissa.
 */
typedef struct fpa_yaman4_desc {
    int64_t       n_points;      /* B                                                     */
    const double* dbeta;         /* [B] phase mismatch per point, 1/length                */
    const double* gamma;         /* [B] or [1]                                            */
    int64_t       gamma_stride;  /* 1 = per point, 0 = broadcast                          */
    const double* alpha;         /* [B] or [1]  power attenuation, 1/length               */
    int64_t       alpha_stride;
    const double* A0;            /* [B,4] or [1,4] complex128                             */
    int64_t       A0_stride;     /* in points: 1 = per point, 0 = broadcast               */
    double        z0;            /* first grid value (0 for integrate_interval)           */
    double        z_max;         /* last grid value                                       */
    int64_t       n_steps;       /* >= 1                                                  */
    int64_t       save_every;    /* >= 1                                                  */
    const double* z_grid;        /* NULL, or [n_steps+1] explicit grid                    */
    uint32_t      flags;         /* FPA_OUT_* | FPA_CHECK_NAN | FPA_PHASE_EXACT | FPA_UNIFORM_PHYSICS */
    uint32_t      reserved;
    double*       A_trace;       /* [B,n_saved,4] complex128 or NULL                      */
    double*       A_end;         /* [B,4] complex128 or NULL                              */
    double*       Pmax;          /* [B,4] or NULL                                         */
    int32_t*      status;        /* [B] (always written when non-NULL)                    */
    double        gamma_uniform; /* with FPA_UNIFORM_PHYSICS: the value *gamma points to   */
    double        alpha_uniform; /* with FPA_UNIFORM_PHYSICS: the value *alpha points to   */
    void*         scratch;       /* _dev entry: device memory of fpa_yaman4_scratch_bytes(B)
                                    bytes for the z-segment scheduler, or NULL (whole-run
                                    kernel).  Ignored by the host entry (library workspace). */
    int64_t       scratch_bytes;
} fpa_yaman4_desc;

/* Device scratch that lets a batch of one wave of the resident warps or more run through the
 * z-segment scheduler (persistent kernel, work items = (32 points, 64/128 RK4 steps); results are
 * bit-identical to the whole-run kernel, the tail of the last wave shrinks from one fiber to one
 * segment).  One size serves fpa_yaman4_rk4_batch_dev and fpa_yaman4_sweep_dev. */
int64_t fpa_yaman4_scratch_bytes(int64_t n_points);

/* n_saved for (n_steps, save_every): n_steps/save_every + 1 (integrators.py:115). */
int64_t fpa_n_saved(int64_t n_steps, int64_t save_every);

/* n_steps for integrate_interval: (int)round-half-even(z_max/dz) (integrators.py:194). */
int64_t fpa_interval_steps(double z_max, double dz);

/* Device-pointer variant: asynchronous on `stream` (a cudaStream_t), current device. */
int fpa_yaman4_rk4_batch_dev(const fpa_yaman4_desc* d, void* stream);
/* Host-pointer variant: H2D, one launch, D2H, synchronise.  `device` = CUDA ordinal. */
int fpa_yaman4_rk4_batch_host(const fpa_yaman4_desc* d, int device);
/* The same batch split over several devices of one box from ONE process (the Delta-beta sweep loop
 * scan_mismtach.py:126-170 and any other batch of independent points; SURVEY 8e): contiguous point
 * ranges whose sizes differ by at most one, one kernel per device in flight at once, every device
 * writes its own shard of the caller's host arrays (trace mode included: no collective).  Results are
 * bit-identical to the single-device call for any device list. */
int fpa_yaman4_rk4_batch_multi_host(const fpa_yaman4_desc* d, int n_devices, const int* devices);

/* RHS only: dA[b,:] = rhs_yaman_simplified(z[b], A[b,:]) for B (z, A) pairs.
 * Replaces the direct Python call yaman_model.py:10-52.  Host pointers. */
int fpa_yaman4_rhs_host(int64_t B, const double* z, const double* A, const double* gamma,
                        const double* alpha, const double* dbeta, double* dA, int device);

/* ------------------------------------------------ sweep front-end (Delta-beta table)
 * Replaces, vectorised over the scan points,
 *   frequency_plan.plan_from_wavelengths     frequency_plan.py:291-327
 *   frequency_plan.infer_symmetry_from_omegas frequency_plan.py:215-255
 *   phase_matching.compute_phase_mismatch    phase_matching.py:150-215
 *   dispersion.delta_beta_from_omegas        dispersion.py:282-318
 *   dispersion.delta_beta_symmetric          dispersion.py:321-372
 *   dispersion.beta_taylor                   dispersion.py:233-279
 * Point b = i1*n3 + i3 of the (n1 x n3) grid uses lambda1[i1], lambda2[i1*l2_stride],
 * lambda3[i3].  Arithmetic is done without FMA contraction, in the reference's
 * operation order.  valid[b] = 0 marks points for which the reference raises
 * (non-positive inferred idler, energy-conservation or symmetry check failure);
 * their dbeta is NaN.
 */
typedef struct fpa_plan_desc {
    int64_t       n1;            /* pump-1 wavelengths                                    */
    int64_t       n3;            /* signal wavelengths                                    */
    const double* lambda1;       /* [n1] metres                                           */
    const double* lambda2;       /* [n1] or [1] metres                                    */
    int64_t       lambda2_stride;/* 1 or 0                                                */
    const double* lambda3;       /* [n3] metres                                           */
    int32_t       method;        /* FPA_PM_*                                              */
    int32_t       max_order;     /* GENERAL_TAYLOR: highest Taylor order                  */
    int32_t       n_even;        /* SYMMETRIC_EVEN: number of even orders                 */
    int32_t       even_orders[FPA_MAX_TAYLOR_ORDER];
    double        beta[FPA_MAX_TAYLOR_ORDER + 1]; /* beta_n, n = 0..12 (already per length unit) */
    double        omega_ref;
    double        atol, rtol;    /* energy-conservation tolerances                        */
    double        provided;      /* PROVIDED: the constant                                */
    double*       omega;         /* [n1*n3,4] or NULL                                     */
    double*       dbeta;         /* [n1*n3]                                               */
    int32_t*      valid;         /* [n1*n3]                                               */
} fpa_plan_desc;

int fpa_dbeta_table_dev(const fpa_plan_desc* d, void* stream);
int fpa_dbeta_table_host(const fpa_plan_desc* d, int device);

/* ------------------------------------------------ fused sweep (front-end + integrator + metric)
 * Replaces the per-point loop of
 *   scan_mismtach.plot_max_gain_and_dbeta_vs_lambda_signal  scan_mismtach.py:694-738
 *   scan_mismtach.plot_max_signal_gain_vs_lambda_signal     scan_mismtach.py:357-392
 * including simulation.run_single_simulation's unit handling (simulation.py:279-336):
 * `plan` holds the dispersion as the caller gave it (per length_unit) and yields the
 * reported dbeta; the integration uses dbeta/scale, gamma/scale, alpha/scale,
 * z_max*scale, dz*scale with scale = 1 (m) or 1000 (km).
 * Host pointers: only the wavelength axes go up, only gain/dbeta/status come back.  Result arrays in
 * page-locked memory (fpa_host_alloc, cudaHostAlloc, cudaHostRegister) are written by the kernel itself
 * while it runs; pageable arrays are filled by a copy after the kernel.
 *   gain_lin[b] = Pmax_signal / p_in[2]  (NaN for invalid / non-finite / <= 0 points)
 */
typedef struct fpa_sweep_desc {
    fpa_plan_desc plan;          /* host pointers; plan.omega may be NULL                 */
    double        A0[8];         /* initial amplitudes, 4 x complex128 (simulation.py:103-123,
                                    computed by the host mirror make_initial_amplitudes)  */
    double        p_signal;      /* p_in[2]: the gain reference (scan_mismtach.py:727)    */
    double        gamma, alpha;  /* per length unit                                       */
    double        z_max, dz;     /* per length unit                                       */
    double        length_scale;  /* 1.0 or 1000.0                                         */
    int64_t       save_every;
    uint32_t      flags;         /* FPA_CHECK_NAN (FPA_PHASE_EXACT: FPA_ERR_UNSUPPORTED)  */
    uint32_t      reserved;
    double*       gain_lin;      /* [n1*n3]                                               */
    double*       Pmax;          /* [n1*n3,4] or NULL                                     */
    double*       A_end;         /* [n1*n3,4] complex128 or NULL                          */
    int32_t*      status;        /* [n1*n3] or NULL                                       */
    int64_t       first_point;   /* sub-range of the flattened grid b = i1*n3 + i3 to run: */
    int64_t       n_sub_points;  /*   [first_point, first_point + n_sub_points); 0, 0 = all.
                                    Every output array is then indexed by b - first_point
                                    (pass base + first_point to fill one full-size array).  */
    int32_t       n_peers;       /* _dev entry, 0..FPA_MAX_PEERS: the kernel ALSO stores each point's gain   */
    int32_t       reserved3;     /*   into peer_gain[p][b] (b = index in the WHOLE grid) for every p -- full-  */
    double*       peer_gain[8];  /*   size gain maps in the memory of the GPUs of the box (this one included),
                                    opened with fpa_ipc_open: the final result gather of a multi-GPU sweep
                                    (SURVEY 8e) done by the sweep kernel itself over NVLink peer stores while
                                    the other points still integrate -- no collective after the kernel.      */
} fpa_sweep_desc;
#define FPA_MAX_PEERS 8

int fpa_yaman4_sweep_host(const fpa_sweep_desc* d, int device);
/* The same sweep on several devices of one box from ONE process (SURVEY 8e: scan points are
 * independent, no exchange): the flattened n1*n3 points are split into contiguous ranges whose sizes
 * differ by at most one (a 1-D sweep with n1 = 1 uses every device too), one kernel per device runs
 * concurrently, every device delivers its range into the caller's host arrays (pinned arrays are
 * written by the kernels directly) -- the "final gather" is the result layout itself.  Results are
 * bit-identical to the single-device call for any device count.
 * (bench.py / sharding.py use the other arrangement, one process per GPU with an NCCL all-gather.) */
int fpa_yaman4_sweep_multi_host(const fpa_sweep_desc* d, int n_devices, const int* devices);
/* Same, but all pointers (plan.lambda*, plan.dbeta, plan.valid, gain_lin, ...) are DEVICE
 * pointers and the work is queued on `stream` (asynchronous): ONE kernel launch per sweep
 * (frequency plan + Delta-beta prologue, fused RK4 loop, gain epilogue).  `scratch` is device memory
 * of at least fpa_yaman4_sweep_scratch_bytes(n1*n3) bytes (= fpa_yaman4_scratch_bytes) for the
 * z-segment scheduler; with NULL the sweep runs as the whole-run kernel (same results, longer tail
 * for batches of a few waves).  FPA_PHASE_EXACT is refused with FPA_ERR_UNSUPPORTED (use
 * fpa_dbeta_table_* + fpa_yaman4_rk4_batch_*, which honours it). */
int64_t fpa_yaman4_sweep_scratch_bytes(int64_t n_points);
int fpa_yaman4_sweep_dev(const fpa_sweep_desc* d, void* scratch, int64_t scratch_bytes, void* stream);

/* ------------------------------------------------ phase-sensitive sweep (wavelength grid x input phase)
 * The fused sweep above with an input-phase axis: every grid point g (b = i1*n3 + i3) runs K initial
 * states, A0_table[k] = make_initial_amplitudes(p_in, phase_in + phase_axis[k]*weights)
 * (simulation.py:103-123, built by the host mirror), so run k of grid point g starts from exactly the
 * bits the plain sweep would use with that phase_in.  Run (g, k) is point g*K + k (phases fastest).
 *   gain_lin[g*K + k] = P3 / p_in[2], NaN for failed / non-finite / <= 0 runs, with P3 chosen by `metric`:
 *     FPA_GAIN_MAX_SAVED   max over the saved samples of |A3|^2 -- the plain sweep's metric
 *                          (scan_mismtach.py:723-738)
 *     FPA_GAIN_LAST_SAVED  |A3|^2 of the LAST SAVED sample, the reference's Pz[-1]
 *                          (scan_mismtach.py:27-40): not the fiber end when save_every does not divide
 *                          the step count
 * and, per grid point over its K gains, numpy's nan-reductions (one small kernel on the same stream
 * right after the sweep kernel): gain_max = nanmax, gain_min = nanmin, idx_max / idx_min =
 * nanargmax / nanargmin (first index on ties), n_finite = number of non-NaN gains; a grid point whose K
 * gains are all NaN (e.g. an invalid plan) gives NaN, -1, -1 and 0.
 * Shapes: sweep.plan.dbeta / valid / omega are per GRID point [G] (G = n1*n3, or n_sub_points);
 * sweep.gain_lin, Pmax, A_end and status are per run [G*K]; the reduction outputs are [G] and each may
 * be NULL.  sweep.first_point / n_sub_points select GRID points (the K runs of a grid point are never
 * split).  sweep.A0 is ignored; sweep.n_peers must be 0 (FPA_ERR_INVALID).  Units, check_nan and the
 * FPA_PHASE_EXACT refusal (FPA_ERR_UNSUPPORTED) are those of fpa_yaman4_sweep_*.
 */
#define FPA_GAIN_MAX_SAVED  0
#define FPA_GAIN_LAST_SAVED 1
#define FPA_MAX_PHASES      65536

typedef struct fpa_phase_sweep_desc {
    fpa_sweep_desc sweep;        /* wavelength grid, physics and per-run outputs (see above)        */
    int64_t        n_phases;     /* K, 1..FPA_MAX_PHASES                                            */
    const double*  A0_table;     /* [K,4] complex128                                                */
    int32_t        metric;       /* FPA_GAIN_MAX_SAVED | FPA_GAIN_LAST_SAVED                        */
    int32_t        reserved;
    double*        gain_max;     /* [G] or NULL                                                     */
    double*        gain_min;     /* [G] or NULL                                                     */
    int32_t*       idx_max;      /* [G] or NULL                                                     */
    int32_t*       idx_min;      /* [G] or NULL                                                     */
    int32_t*       n_finite;     /* [G] or NULL                                                     */
} fpa_phase_sweep_desc;

/* Host pointers, as fpa_yaman4_sweep_host.  sweep.gain_lin may be NULL: the [G*K] gain map then stays in
 * the library workspace and only the reductions come back (a 1000 x 1000 x 64 sweep needs no 512 MB
 * host array). */
int fpa_yaman4_phase_sweep_host(const fpa_phase_sweep_desc* d, int device);
/* The grid points split over several devices of one box from ONE process (contiguous ranges whose sizes
 * differ by at most one); bit-identical to the single-device call for any device list. */
int fpa_yaman4_phase_sweep_multi_host(const fpa_phase_sweep_desc* d, int n_devices, const int* devices);
/* Device scratch for the z-segment scheduler of a phase sweep of n_points = G*K runs: one more double of
 * state per run than fpa_yaman4_scratch_bytes (the last saved signal power travels with the segment). */
int64_t fpa_yaman4_phase_sweep_scratch_bytes(int64_t n_points);
/* Device pointers, asynchronous on `stream`: the sweep kernel and the reduction kernel.  sweep.gain_lin
 * must be set.  `scratch` NULL: the whole-run kernel (same results). */
int fpa_yaman4_phase_sweep_dev(const fpa_phase_sweep_desc* d, void* scratch, int64_t scratch_bytes, void* stream);

/* ------------------------------------------------ small-signal transfer matrices (not in the reference)
 * J = dA(L)/dA(z0): the exact derivative of the discrete RK4 map the fast integrator computes (not an
 * approximation of the ODE's derivative; central finite differences of fpa_yaman4_rk4_batch_* converge to it).
 * Each RK4 stage out = base + c*f(in) (yaman_model.py:10-52 weighted by c) is differentiated along a tangent t:
 *   P_j' = 2(x_j x_j' + y_j y_j'),  S' = sum P_j',  G_j' = c*gamma*(2 S' - P_j')
 *   U' = A3'A4 + A3A4',  V' = A1'A2 + A1A2',  W' = qU',  Z' = conj(q)V'
 *   out_j' = base_j' + cn A_j' + i(G_j'A_j + G_jA_j') + i(conj(A_m)'{W|Z} + conj(A_m){W'|Z'})
 * with the base run's phase factors q and the same RK4 combination.  The base state runs with the unchanged
 * arithmetic: A_end, Pmax, status and gain_lin equal those of fpa_yaman4_rk4_batch_* / fpa_yaman4_sweep_* bit for
 * bit.  One GPU thread per (point, column); uniform-grid whole-run kernels only.
 *
 * Batch: the descriptor of fpa_yaman4_rk4_batch_* with all its outputs but the trace; FPA_OUT_TRACE, z_grid and
 * FPA_PHASE_EXACT give FPA_ERR_UNSUPPORTED; `scratch` is ignored.
 * Sweep: the descriptor and units of fpa_yaman4_sweep_*; n_peers must be 0; FPA_PHASE_EXACT gives
 * FPA_ERR_UNSUPPORTED.  gain_lin may be NULL, and only then may p_signal be 0: a zero seed gives the undepleted-pump
 * linearisation.
 * The multi-device entries split the work over several devices of one box from ONE process, the batch's points
 * like fpa_yaman4_rk4_batch_multi_host and the sweep's flattened grid like fpa_yaman4_sweep_multi_host; results
 * are bit-identical to the single-device call for any device list.
 * A point that is not integrated (invalid plan point, non-finite dbeta) and, under FPA_CHECK_NAN, a point whose
 * status is not FPA_POINT_OK get an all-NaN J.  J is dimensionless, the same in m and km units.
 */
typedef struct fpa_transfer_out {
    uint32_t columns;   /* bit c (0..7) set: column d A(L) / d in_c, in_c = Re A_{c/2}(z0) (c even) or Im (c odd); != 0 */
    uint32_t reserved;
    double*  jac;       /* [B, 8, popcount(columns)]: row r = Re/Im of A_{r/2}(L), columns in ascending bit order */
} fpa_transfer_out;

int fpa_yaman4_transfer_batch_dev (const fpa_yaman4_desc* d, const fpa_transfer_out* t, void* stream);
int fpa_yaman4_transfer_batch_host(const fpa_yaman4_desc* d, const fpa_transfer_out* t, int device);
int fpa_yaman4_transfer_batch_multi_host(const fpa_yaman4_desc* d, const fpa_transfer_out* t,
                                         int n_devices, const int* devices);
int fpa_yaman4_transfer_sweep_dev (const fpa_sweep_desc* d, const fpa_transfer_out* t, void* stream);
int fpa_yaman4_transfer_sweep_host(const fpa_sweep_desc* d, const fpa_transfer_out* t, int device);
int fpa_yaman4_transfer_sweep_multi_host(const fpa_sweep_desc* d, const fpa_transfer_out* t,
                                         int n_devices, const int* devices);

/* ------------------------------------------------ linear test RHS  y' = lambda*y
 * Lets the reference's own integrator tests (tests.py:146-226, y' = y on a real
 * state) run on the device: complex lambda per component, complex128 state.
 * y0[B,dim], lam[dim] complex128; outputs as for yaman4 with 4 -> dim. */
int fpa_linear_rk4_batch_host(int64_t B, int64_t dim, const double* y0, const double* lam,
                              double z0, double z_max, int64_t n_steps, int64_t save_every,
                              const double* z_grid, uint32_t flags, double* y_trace,
                              double* y_end, int32_t* status, int device);

/* ------------------------------------------------ N-wave generalisation (not in the reference)
 * dA_n/dz = -(alpha/2) A_n + i*gamma * [ (2*sum_j P_j - P_n) A_n
 *            + sum_{entries e of n} D_e * A_k A_l conj(A_m) * exp(i (b_k+b_l-b_m-b_n) z) ]
 * with the triplet table produced by fpa_enumerate_triplets (entries sorted by n, k, l, m;
 * k <= l, m not in {k,l}; D = 1 for k == l else 2).  Reduces to the 4-wave system with the
 * fixed table {n0:(2,3;1) n1:(2,3;0) n2:(0,1;3) n3:(0,1;2)} and b = [0,0,0,dbeta].
 */
typedef struct fpa_triplet {
    int16_t k, l, m, weight;
} fpa_triplet;

/* Enumerate on an integer frequency grid: wave j sits at grid index g[j]; entry (n;k,l,m)
 * exists iff g[k]+g[l]-g[m] == g[n].  Pass out == NULL to get only the count.
 * row_ptr[N+1] receives CSR offsets per n (may be NULL).  Returns the count, or -1. */
int64_t fpa_enumerate_triplets(int32_t N, const int32_t* g, fpa_triplet* out, int64_t cap,
                               int64_t* row_ptr);

/* The same for a plan that is NOT on an integer grid: entry (n;k,l,m) exists iff the photon energies match
 * within the reference's tolerance rule for its four-wave plan (frequency_plan.enforce_energy_conservation,
 * frequency_plan.py:112-131: numpy.isclose(w_k + w_l, w_m + w_n, atol, rtol), i.e.
 * |lhs - rhs| <= atol + rtol * |rhs| with both sums rounded to double first; defaults atol 0, rtol 1e-12).
 * Same canonical order (n, k <= l, m not in {k, l}) and weights; bit-exact against the CPU restatement. */
int64_t fpa_enumerate_triplets_omega(int32_t N, const double* omega, double atol, double rtol, fpa_triplet* out,
                                     int64_t cap, int64_t* row_ptr);

typedef struct fpa_nwave_desc {
    int64_t            n_points;     /* B                                                  */
    int32_t            n_waves;      /* N (<= 128)                                         */
    int32_t            reserved0;
    const double*      beta;         /* [B,N] or [1,N] per-wave propagation constants      */
    int64_t            beta_stride;  /* in points                                          */
    const double*      gamma;  int64_t gamma_stride;
    const double*      alpha;  int64_t alpha_stride;
    const double*      A0;           /* [B,N] or [1,N] complex128                          */
    int64_t            A0_stride;
    const fpa_triplet* triplets;     /* [n_triplets] shared by all points                  */
    const int64_t*     row_ptr;      /* [N+1]                                              */
    int64_t            n_triplets;
    double             z0, z_max;
    int64_t            n_steps, save_every;
    uint32_t           flags;
    uint32_t           reserved1;
    double*            A_trace;      /* [B,n_saved,N] complex128 or NULL                   */
    double*            A_end;        /* [B,N] or NULL                                      */
    double*            Pmax;         /* [B,N] or NULL                                      */
    int32_t*           status;       /* [B]                                                */
    /* Integer-grid plans (uniform combs): grid_slot[j] = g_j - g_min for every wave, grid_span =
     * g_max - g_min + 1 (<= 512).  When set (and FPA_NWAVE_TABLE is not), the integrator uses the
     * O(span^2) convolution form of the same ODE instead of the enumerated table (csrc/nwave_comb.cu);
     * triplets / row_ptr may then be NULL -- but when they are given too, plans the convolution form
     * does not suit (span > 512, or sparse: span^2 > 5 * n_triplets) run through the table kernel.
     * Slots must be distinct values in [0, grid_span). */
    const int32_t*     grid_slot;    /* [N] or NULL                                        */
    int32_t            grid_span;
    /* Factored form of the table (fpa_nwave_factor_table below; a device pointer for the _dev call): when set,
     * the table kernel forms every pair product At_k At_l once per RHS and every (n, m) cell once, instead of
     * walking the entry list -- same ODE, ~25x less arithmetic for a comb of 64 lines; triplets / row_ptr may
     * then be NULL.  The _host and _multi_host calls build it themselves from triplets / row_ptr. */
    int32_t            n_classes;
    const void*        factored;
} fpa_nwave_desc;

/* Factor a CSR triplet table (host pointers) into the blob `factored` points to.  Returns the blob size in bytes
 * (and the class count in *n_classes); the blob is written when `blob` is not NULL and `cap` is large enough.
 * Any table factors -- nothing is assumed about where it came from; -1 on malformed input (N > 128, indices out
 * of range, row_ptr not a CSR offset array).  The size query and the fill call of one plan cost one
 * factorisation (11 ms at N = 64): the library keeps the calling thread's last result, keyed by a hash of the
 * table, which also serves the host integrator calls that repeat a plan. */
int64_t fpa_nwave_factor_table(int32_t N, const fpa_triplet* triplets, const int64_t* row_ptr, int64_t n_triplets,
                               void* blob, int64_t cap, int32_t* n_classes);

int fpa_nwave_rk4_batch_dev(const fpa_nwave_desc* d, void* stream);
int fpa_nwave_rk4_batch_host(const fpa_nwave_desc* d, int device);
/* The same batch split over several devices of one box from ONE process (BASELINE config 5: B = 1024 pump
 * powers over the 8 GPUs): contiguous balanced point ranges, one kernel per device in flight at once, every
 * device writes its own shard of the caller's host arrays.  Bit-identical to the single-device call as long
 * as every shard stays on the same side of the library's kernel choices (they depend on the batch size). */
int fpa_nwave_rk4_batch_multi_host(const fpa_nwave_desc* d, int n_devices, const int* devices);
/* Algorithmic flops per point.step the N-wave kernel is credited with (see DESIGN.md). */
double fpa_nwave_flops_per_step(int32_t n_waves, int64_t n_triplets, int64_t n_pairs);
/* Same for the table kernel integrating from a factored table (`blob`: the HOST copy fpa_nwave_factor_table
 * wrote): 8 per non-empty cell, 10 per pair product, 30 N per RHS; 0 for a foreign blob. */
double fpa_nwave_factored_flops_per_step(const void* blob);
/* Same for the convolution-form kernel (O(span^2) work: credited with what it executes). */
double fpa_nwave_comb_flops_per_step(int32_t n_waves, int32_t grid_span);

/* ------------------------------------------------ measurement helpers */
/* DFMA micro-benchmark: dependent-chain-free FP64 FMA loop on every SM.  Returns the
 * achieved TFLOP/s (2 flops per FMA) in *tflops and the kernel time in *ms. */
int fpa_fp64_peak_probe(int device, int iters, double* tflops, double* ms);
/* Algorithmic flops per scan-point.RK4-step of the 4-wave model (SURVEY 8d): 568. */
double fpa_yaman4_flops_per_step(void);

/* Pinned host memory for the e2e path. */
int fpa_host_alloc(void** ptr, int64_t bytes);
int fpa_host_free(void* ptr);
/* Device memory that can be shared with the other processes of the box (one rank per GPU): allocate on
 * `device`, export a 64-byte handle, open it in the peer process (device pointer valid on the opener's current
 * device; peer access is enabled by the open), close before the owner frees.  Used for the peer_gain maps above. */
int fpa_dev_alloc(void** ptr, int64_t bytes, int device);
int fpa_dev_free(void* ptr);
int fpa_ipc_export(const void* dev_ptr, void* handle64);
int fpa_ipc_open(const void* handle64, void** dev_ptr);
int fpa_ipc_close(void* dev_ptr);

/* Page-lock memory the caller already owns (e.g. a POSIX shared-memory segment several processes
 * map: every rank registers it and its kernels store their shard of the result straight into the
 * one host array).  Registered memory counts as pinned wherever a host entry point writes results
 * directly: fpa_yaman4_rk4_batch_*host, fpa_yaman4_sweep_*host and fpa_yaman4_phase_sweep_*host; their
 * complex128 outputs and Pmax rows only when 16-byte aligned (else staged, see "Alignment" above).  The
 * N-wave, linear, RHS and Delta-beta table entries always stage their results and copy them back. */
int fpa_host_register(void* ptr, int64_t bytes);
int fpa_host_unregister(void* ptr);

#ifdef __cplusplus
}
#endif
#endif /* FPA_B200_H */
