// yaman4.cu -- fused fixed-step RK4 x 4-wave Yaman/Agrawal FWM right-hand side.
//
// One thread integrates one scan point for ALL z-steps with its state in registers: the four RK4
// stages, the RHS, the per-step finite check, the max-over-saved-samples metric and the trace
// write-out are a single kernel (one launch per batch).
//
// What it stands in for in the reference (paths relative to the reference checkout):
//   integrators.rk4_step              integrators.py:25-61   (stage formulas :54-59)
//   integrators.integrate_fixed_step  integrators.py:68-142  (grid, saving, NaN guard)
//   integrators.integrate_interval    integrators.py:150-204 (linspace grid)
//   yaman_model.rhs_yaman_simplified  yaman_model.py:10-52   (+ _linear_loss_terms :123-132,
//                                     _kerr_terms :135-156, _fwm_terms :159-186)
//
// Why thread-per-point and not warp-per-point for N = 4: the FWM sum has four terms; a warp per
// point would leave 28 lanes idle.  The bound is the FP64 FMA pipe (16 lanes per SM sub-partition:
// one warp-wide FP64 instruction every 2 cycles), so the kernels are written to minimise FP64
// instructions per point.step.  Two kernel families:
//
//  * yaman4_fast_kernel -- uniform grid (integrate_interval).  ~300 FP64 instructions per step:
//      - constant step h = (z_max-z0)/n_steps (the reference's per-step h_i = z_{i+1}-z_i differs
//        from it by <= 1 ulp(z); the sum telescopes to the same z_max);
//      - every stage writes the NEXT STAGE STATE directly: y + c*f(ys) is one 4-FMA chain per
//        component with the stage weight c folded into the Kerr / loss / phase coefficients, so
//        k_1..k_4 are never formed;
//      - the RK4 combination is rebuilt from the stage states,
//            y' = -y/3 + ys2/3 + 2 ys3/3 + ys4/3 + (h/6) f(ys4)       (algebraically identical);
//      - the FWM phase 2*gamma*exp(i*dbeta*z) advances by a constant complex rotation per half
//        step (2 rotations per step) and is re-synchronised with an exact sincos every 32 steps,
//        instead of the reference's 8 complex exp() per step.
//    Measured against the oracle: <= 1e-13 relative on |A|^2 after 10 000 steps at 45 dB gain.
//    Symmetric sweeps (the plain fused sweep only): when the initial state has A1 == A2 and A3 == A4 bit for
//    bit -- the standard dual-pump set-up, p_in = [P, P, Ps, Ps] with no input phase -- every rounded
//    operation of stage() on wave 2 (4) is the one on wave 1 (3) with the same operands, so the state stays
//    on that subspace for the whole fiber.  stage_sym() / fast_integrate<..., SYM> then integrate the
//    4-double state (x1, y1, x3, y3) with the same expressions in the same operand order: 186 instead of
//    298 FP64 instructions per lossy step and the same bits (DESIGN.md §4.1c).  The launcher decides by a
//    memcmp of A0's bit patterns; FPA_SWEEP_SYM=0 forces the 4-wave kernels.
//  * yaman4_exact_kernel -- FPA_PHASE_EXACT or an explicit z-grid: the reference's arithmetic
//    structure step by step (h_i by subtraction, sincos at z, z+h/2, z+h, k_j formed, y + h/6*(..)).
#include "plan_point.cuh"

#include <stdlib.h>

#include <type_traits>

namespace fpa {

constexpr int kResync = 32;  // steps between exact sincos re-synchronisations of the phase

struct Yaman4Coef {  // stage-weighted coefficients; c = {h/2, h, h/6}
    double cg[3];    // c*gamma
    double c2g[3];   // 2*c*gamma
    double cn[3];    // -c*alpha/2
    double q0;       // (h/2)*2*gamma : modulus of the scaled phase factor
};

struct Yaman4Params {
    int64_t       n_points;
    const double* dbeta;
    const double* gamma;
    const double* alpha;
    const double* A0;
    const double* z_grid;
    double*       A_trace;
    double*       A_end;
    double*       Pmax;
    int32_t*      status;
    double        z0, z_max, h;
    int           gamma_stride, alpha_stride, A0_stride;
    int           n_steps, save_every;
    int           check;
    int           lossless;  // uniform physics with alpha == 0
    int64_t       n_saved;
    Yaman4Coef    coef;  // valid when gamma and alpha are the same for every point (UNIFORM)
};

__host__ __device__ inline Yaman4Coef make_coef(double gamma, double alpha, double h) {
    Yaman4Coef c;
    const double w[3] = {0.5 * h, h, h * (1.0 / 6.0)};
    const double nha  = -0.5 * alpha;
    for (int s = 0; s < 3; ++s) {
        c.cg[s]  = w[s] * gamma;
        c.c2g[s] = c.cg[s] + c.cg[s];
        c.cn[s]  = w[s] * nha;
    }
    c.q0 = c.c2g[0];
    return c;
}

// ------------------------------------------------------------------ fast path
// One RK4 stage.  in = stage state (x1,y1,..,x4,y4), base = what the weighted RHS is added to,
// (qr,qi) = c*2*gamma*exp(i*dbeta*z) for this stage's weight c, cg/c2g/cn the matching
// coefficients.  out = base + c*f(in): 32 shared + 32 chain FP64 instructions.  S = sum |in|^2.
template <bool LOSS = true>
__device__ __forceinline__ void stage(const double (&in)[8], const double (&base)[8], double qr, double qi,
                                      double cg, double c2g, double cn, double (&out)[8], double& S) {
    const double x1 = in[0], y1 = in[1], x2 = in[2], y2 = in[3];
    const double x3 = in[4], y3 = in[5], x4 = in[6], y4 = in[7];
    // powers (yaman_model.py:144-147)
    const double P1 = fma(y1, y1, x1 * x1);
    const double P2 = fma(y2, y2, x2 * x2);
    const double P3 = fma(y3, y3, x3 * x3);
    const double P4 = fma(y4, y4, x4 * x4);
    S = (P1 + P2) + (P3 + P4);
    // c*gamma*(P_j + 2*sum_{k!=j} P_k) == c*gamma*(2S - P_j)   (yaman_model.py:148-151)
    const double c2 = c2g * S;
    const double G1 = fma(-cg, P1, c2);
    const double G2 = fma(-cg, P2, c2);
    const double G3 = fma(-cg, P3, c2);
    const double G4 = fma(-cg, P4, c2);
    // pair products shared by two waves each (yaman_model.py:177-181)
    const double Ur = fma(-y3, y4, x3 * x4), Ui = fma(x3, y4, y3 * x4);  // A3*A4
    const double Vr = fma(-y1, y2, x1 * x2), Vi = fma(x1, y2, y1 * x2);  // A1*A2
    // W = q U ,  Z = conj(q) V
    const double Wr = fma(-qi, Ui, qr * Ur), Wi = fma(qr, Ui, qi * Ur);
    const double Zr = fma(qi, Vi, qr * Vr),  Zi = fma(qr, Vi, -(qi * Vr));
    // out_j = base_j + cn*A_j + i*G_j*A_j + i*conj(A_m)*{W|Z}
    //   i*conj(A_m)*W = (ym Wr - xm Wi) + i (xm Wr + ym Wi)
    // The loss term is added FIRST: it needs nothing but the stage input, so the SASS pass
    // (tools/sass_sched.py) can issue it right before an FMA that shares its operand.
    if (LOSS) {
        out[0] = fma(-G1, y1, fma(y2, Wr, fma(-x2, Wi, fma(cn, x1, base[0]))));
        out[1] = fma(G1, x1, fma(x2, Wr, fma(y2, Wi, fma(cn, y1, base[1]))));
        out[2] = fma(-G2, y2, fma(y1, Wr, fma(-x1, Wi, fma(cn, x2, base[2]))));
        out[3] = fma(G2, x2, fma(x1, Wr, fma(y1, Wi, fma(cn, y2, base[3]))));
        out[4] = fma(-G3, y3, fma(y4, Zr, fma(-x4, Zi, fma(cn, x3, base[4]))));
        out[5] = fma(G3, x3, fma(x4, Zr, fma(y4, Zi, fma(cn, y3, base[5]))));
        out[6] = fma(-G4, y4, fma(y3, Zr, fma(-x3, Zi, fma(cn, x4, base[6]))));
        out[7] = fma(G4, x4, fma(x3, Zr, fma(y3, Zi, fma(cn, y4, base[7]))));
    } else {  // alpha == 0: the reference's loss term is exact zeros (yaman_model.py:129-130)
        out[0] = fma(-G1, y1, fma(y2, Wr, fma(-x2, Wi, base[0])));
        out[1] = fma(G1, x1, fma(x2, Wr, fma(y2, Wi, base[1])));
        out[2] = fma(-G2, y2, fma(y1, Wr, fma(-x1, Wi, base[2])));
        out[3] = fma(G2, x2, fma(x1, Wr, fma(y1, Wi, base[3])));
        out[4] = fma(-G3, y3, fma(y4, Zr, fma(-x4, Zi, base[4])));
        out[5] = fma(G3, x3, fma(x4, Zr, fma(y4, Zi, base[5])));
        out[6] = fma(-G4, y4, fma(y3, Zr, fma(-x3, Zi, base[6])));
        out[7] = fma(G4, x4, fma(x3, Zr, fma(y3, Zi, base[7])));
    }
}

// stage() on a symmetric state, in = (x1, y1, x3, y3) standing for (x1, y1, x1, y1, x3, y3, x3, y3), base the
// same way.  Every rounded operation is the one stage() performs with x2 -> x1, y2 -> y1, x4 -> x3, y4 -> y3:
// P2 == P1, P4 == P3, G2 == G1, G4 == G3, and out[2], out[3], out[6], out[7] of stage() are the FMA chains of
// out[0], out[1], out[4], out[5] on the same operands, so they are not computed.  S is stage()'s
// (P1 + P2) + (P3 + P4) with that substitution, the same two adds and the same rounding.  Every product and
// sum is spelled out as in stage(); nothing is left to contraction.
template <bool LOSS = true>
__device__ __forceinline__ void stage_sym(const double (&in)[4], const double (&base)[4], double qr, double qi,
                                          double cg, double c2g, double cn, double (&out)[4], double& S) {
    const double x1 = in[0], y1 = in[1], x3 = in[2], y3 = in[3];
    const double P1 = fma(y1, y1, x1 * x1);
    const double P3 = fma(y3, y3, x3 * x3);
    S = (P1 + P1) + (P3 + P3);
    const double c2 = c2g * S;
    const double G1 = fma(-cg, P1, c2);
    const double G3 = fma(-cg, P3, c2);
    const double Ur = fma(-y3, y3, x3 * x3), Ui = fma(x3, y3, y3 * x3);  // A3*A4
    const double Vr = fma(-y1, y1, x1 * x1), Vi = fma(x1, y1, y1 * x1);  // A1*A2
    const double Wr = fma(-qi, Ui, qr * Ur), Wi = fma(qr, Ui, qi * Ur);
    const double Zr = fma(qi, Vi, qr * Vr),  Zi = fma(qr, Vi, -(qi * Vr));
    if (LOSS) {
        out[0] = fma(-G1, y1, fma(y1, Wr, fma(-x1, Wi, fma(cn, x1, base[0]))));
        out[1] = fma(G1, x1, fma(x1, Wr, fma(y1, Wi, fma(cn, y1, base[1]))));
        out[2] = fma(-G3, y3, fma(y3, Zr, fma(-x3, Zi, fma(cn, x3, base[2]))));
        out[3] = fma(G3, x3, fma(x3, Zr, fma(y3, Zi, fma(cn, y3, base[3]))));
    } else {
        out[0] = fma(-G1, y1, fma(y1, Wr, fma(-x1, Wi, base[0])));
        out[1] = fma(G1, x1, fma(x1, Wr, fma(y1, Wi, base[1])));
        out[2] = fma(-G3, y3, fma(y3, Zr, fma(-x3, Zi, base[2])));
        out[3] = fma(G3, x3, fma(x3, Zr, fma(y3, Zi, base[3])));
    }
}

// One RK4 stage on the full state or (4 doubles) on the symmetric half of one.
template <bool LOSS>
__device__ __forceinline__ void rk_stage(const double (&in)[8], const double (&base)[8], double qr, double qi,
                                         double cg, double c2g, double cn, double (&out)[8], double& S) {
    stage<LOSS>(in, base, qr, qi, cg, c2g, cn, out, S);
}
template <bool LOSS>
__device__ __forceinline__ void rk_stage(const double (&in)[4], const double (&base)[4], double qr, double qi,
                                         double cg, double c2g, double cn, double (&out)[4], double& S) {
    stage_sym<LOSS>(in, base, qr, qi, cg, c2g, cn, out, S);
}

__device__ __forceinline__ void load_state(const Yaman4Params& p, int64_t b, double (&y)[8]) {
    const double2* a0 = reinterpret_cast<const double2*>(p.A0) + b * p.A0_stride * 4;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const double2 v = a0[j];
        y[2 * j] = v.x;
        y[2 * j + 1] = v.y;
    }
}

// A point whose dbeta is not finite: exp(i*dbeta*z) is NaN from the first stage on, every later
// sample is NaN and step 0 is the bad one (integrators.py:132-135).  Invalid scan points of a sweep
// arrive here with dbeta = NaN and cost nothing.
__device__ __noinline__ void write_invalid_point(const Yaman4Params& p, int64_t b, const double (&y)[8]) {
    const double qn = qnan();
    if (p.A_trace) {
        double* t = p.A_trace + b * p.n_saved * 8;
        for (int j = 0; j < 4; ++j) store_c128(t + 2 * j, y[2 * j], y[2 * j + 1]);
        for (int64_t s = 1; s < p.n_saved; ++s)
            for (int j = 0; j < 4; ++j) store_c128(t + s * 8 + 2 * j, qn, qn);
    }
    if (p.A_end)
        for (int j = 0; j < 4; ++j) store_c128(p.A_end + b * 8 + 2 * j, qn, qn);
    if (p.Pmax)
        for (int j = 0; j < 4; ++j) p.Pmax[b * 4 + j] = qn;
    if (p.status) p.status[b] = p.check ? 0 : FPA_POINT_OK;
}

// LAST: *plast = |A3|^2 of this sample, so that after the run it holds the LAST saved sample's signal power (the
// phase sweep's "end" metric, which is not the fiber end when save_every does not divide the step count).
template <bool LAST = false>
__device__ __forceinline__ void save_sample(const double (&y)[8], double*& tr, double (&pm)[4], bool trace,
                                            bool pmax, double* plast = nullptr) {
    if (trace) {
        // one 64-byte row [A1..A4] per saved sample: two 256-bit stores = two full 32 B sectors
        // (A_trace rows are 64-byte aligned whenever the buffer is 32-byte aligned; else 16 B stores)
        if ((reinterpret_cast<uintptr_t>(tr) & 31) == 0) {
            store_2c128(tr, y[0], y[1], y[2], y[3]);
            store_2c128(tr + 4, y[4], y[5], y[6], y[7]);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) store_c128(tr + 2 * j, y[2 * j], y[2 * j + 1]);
        }
        tr += 8;
    }
    if (pmax) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double P = fma(y[2 * j + 1], y[2 * j + 1], y[2 * j] * y[2 * j]);
            // numpy.max semantics: NaN is sticky
            pm[j] = (P != P || pm[j] != pm[j]) ? qnan() : fmax(pm[j], P);
        }
    }
    if (LAST) *plast = fma(y[5], y[5], y[4] * y[4]);
}

// save_sample of a symmetric state (x1, y1, x3, y3): the running maxima of waves 1 and 3 (pm[1] and pm[3] would be
// the same computation on the same bits; the epilogue copies them).  No trace.
template <bool LAST = false>
__device__ __forceinline__ void save_sample(const double (&y)[4], double*&, double (&pm)[4], bool, bool pmax,
                                            double* = nullptr) {
    static_assert(!LAST, "the symmetric path has no last-sample metric");
    if (pmax) {
#pragma unroll
        for (int j = 0; j < 4; j += 2) {
            const double P = fma(y[j + 1], y[j + 1], y[j] * y[j]);
            pm[j] = (P != P || pm[j] != pm[j]) ? qnan() : fmax(pm[j], P);
        }
    }
}

__device__ __forceinline__ void write_results(const Yaman4Params& p, int64_t b, const double (&y)[8],
                                              const double (&pm)[4], bool pmax, int32_t bad) {
    if (p.check && bad == FPA_POINT_OK) {
        bool nf = false;
#pragma unroll
        for (int j = 0; j < 8; ++j) nf |= nonfinite(y[j]);
        if (nf) bad = p.n_steps - 1;
    }
    if (p.status) p.status[b] = p.check ? bad : FPA_POINT_OK;
    if (p.A_end) {
#pragma unroll
        for (int j = 0; j < 4; ++j) store_c128(p.A_end + b * 8 + 2 * j, y[2 * j], y[2 * j + 1]);
    }
    if (pmax) {
        double2* o = reinterpret_cast<double2*>(p.Pmax + b * 4);
        o[0] = make_double2(pm[0], pm[1]);
        o[1] = make_double2(pm[2], pm[3]);
    }
}

// The z-loop of the fast path: advances y over the steps [i0, i1) of the run, keeps the running maxima
// in pm and returns the first step whose result was not finite (or `bad` as given).  The whole run is
// (0, n_steps); the z-segment scheduler (SegParams below) calls it once per segment with the
// state, pm and bad of the previous segment.  i0 must be a multiple of kResync: the phase factor is
// rebuilt by the exact sincos at the first step of the range, exactly where the whole-run loop rebuilds
// it, so a segmented run is bit-identical to a whole one.  LAST: *plast follows the last saved sample (save_sample).
// SYM: y is the symmetric half (x1, y1, x3, y3) of a state with A1 == A2, A3 == A4 (stage_sym); pm[0] and pm[2] are
// kept, pm[1] and pm[3] are left to the caller.
template <bool SYM>
constexpr int kStateLen = SYM ? 4 : 8;
template <bool TRACE, bool PMAX, bool LOSS, bool SEG = false, bool LAST = false, bool SYM = false>
__device__ __forceinline__ int32_t fast_integrate(const Yaman4Params& p, int64_t b, double dbeta,
                                                  const Yaman4Coef& cf, double (&y)[kStateLen<SYM>], double (&pm)[4],
                                                  int i0_in = 0, int i1_in = 0, int32_t bad_in = FPA_POINT_OK,
                                                  double* plast = nullptr) {
    constexpr int NS = kStateLen<SYM>;
    static_assert(!SYM || !TRACE, "the symmetric path writes no trace");
    const int i0 = SEG ? i0_in : 0;
    const int i1 = SEG ? i1_in : p.n_steps;
    double* tr = nullptr;
    if (TRACE) tr = p.A_trace + b * p.n_saved * 8 + (i0 == 0 ? 0 : ((int64_t)(i0 / p.save_every) + 1) * 8);
    if (i0 == 0) {
        if (PMAX) {
#pragma unroll
            for (int j = 0; j < 4; ++j) pm[j] = -1.0;  // |A|^2 >= 0: first sample always replaces it
        }
        save_sample<LAST>(y, tr, pm, TRACE, PMAX, plast);
    }

    const double h = p.h, z0 = p.z0;
    // rotation by half a step
    double rr, ri;
    sincos(dbeta * (0.5 * h), &ri, &rr);

    double  qr = cf.q0, qi = 0.0;  // (h/2)*2*gamma*exp(i*dbeta*z_i)
    int     save_ctr = SEG ? p.save_every - (i0 % p.save_every) : p.save_every;
    int32_t bad = SEG ? bad_in : FPA_POINT_OK;
    // Weights of the stage states in y' = -y/3 + ys2/3 + 2 ys3/3 + ys4/3 + (h/6) f(ys4).  They must sum
    // to EXACTLY one in floating point: fl(1/3) + fl(2/3) = 1 - 2^-54 shrinks |A| by that factor every
    // step (and fl(1/3) + fl(1 - fl(1/3)) = 1 + 2^-54 grows it), and the Kerr phase integrates the
    // amplitude error -- quadratic growth, 3e-10 rad after 2e5 steps (tests/test_gpu_edges.py).  The y and
    // ys2 weights cancel exactly (same constant); 1 - fl(2/3) is exactly representable, so the ys4 weight
    // third_c = 1 - fl(2/3) makes two_thirds + third_c == 1 with no rounding.
    const double third = 1.0 / 3.0, two_thirds = 2.0 / 3.0, third_c = 1.0 - two_thirds;

    for (int i = i0; i < i1; ++i) {
        if ((i & (kResync - 1)) == 0) {
            double s, c;
            sincos(dbeta * fma((double)i, h, z0), &s, &c);
            qr = cf.q0 * c;
            qi = cf.q0 * s;
        }
        // phase at z+h/2 (weight h/2), the same with weight h, and at z+h (weights h/2 and h/6)
        const double qhr = fma(-qi, ri, qr * rr), qhi = fma(qr, ri, qi * rr);
        const double q2r = qhr + qhr, q2i = qhi + qhi;
        const double qfr = fma(-qhi, ri, qhr * rr), qfi = fma(qhr, ri, qhi * rr);
        const double q6r = qfr * third, q6i = qfi * third;

        double ys[NS], yt[NS], acc[NS], S, Sx;
        // stage 1: ys = y + (h/2) f(z, y)
        rk_stage<LOSS>(y, y, qr, qi, cf.cg[0], cf.c2g[0], cf.cn[0], ys, S);
        // S = sum |A|^2 of the state that step i-1 produced: a non-finite component makes S
        // non-finite, so the exact per-component test runs only then (integrators.py:132-135).
        if (nonfinite(S) && bad == FPA_POINT_OK && i > 0) {
            bool nf = false;
#pragma unroll
            for (int j = 0; j < NS; ++j) nf |= nonfinite(y[j]);
            if (nf) bad = i - 1;
        }
#pragma unroll
        for (int j = 0; j < NS; ++j) acc[j] = fma(third, ys[j], y[j] * (-third));
        // stage 2: yt = y + (h/2) f(z+h/2, ys)
        rk_stage<LOSS>(ys, y, qhr, qhi, cf.cg[0], cf.c2g[0], cf.cn[0], yt, Sx);
#pragma unroll
        for (int j = 0; j < NS; ++j) acc[j] = fma(two_thirds, yt[j], acc[j]);
        // stage 3: ys = y + h f(z+h/2, yt)
        rk_stage<LOSS>(yt, y, q2r, q2i, cf.cg[1], cf.c2g[1], cf.cn[1], ys, Sx);
#pragma unroll
        for (int j = 0; j < NS; ++j) acc[j] = fma(third_c, ys[j], acc[j]);
        // stage 4: y' = acc + (h/6) f(z+h, ys)
        rk_stage<LOSS>(ys, acc, q6r, q6i, cf.cg[2], cf.c2g[2], cf.cn[2], y, Sx);

        qr = qfr;
        qi = qfi;

        if (--save_ctr == 0) {  // (i+1) % save_every == 0, integrators.py:137-140
            save_ctr = p.save_every;
            save_sample<LAST>(y, tr, pm, TRACE, PMAX, plast);
        }
    }
    return bad;
}

// UNIFORM: 0 = gamma/alpha per thread; 1 = uniform physics, coefficients from the constant bank;
// 2 = uniform and lossless (alpha == 0): the 32 loss FMAs per step are not issued.
template <bool TRACE, bool PMAX, int UNIFORM, int THREADS, int MIN_BLOCKS>
__global__ void __launch_bounds__(THREADS, MIN_BLOCKS) yaman4_fast_kernel(const Yaman4Params p) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= p.n_points) return;

    double y[8];
    load_state(p, b, y);
    const double dbeta = p.dbeta[b];
    if (nonfinite(dbeta)) {
        write_invalid_point(p, b, y);
        return;
    }
    // stage-weighted coefficients: from the constant bank when the physics is uniform over the
    // batch (sweeps), else per thread
    Yaman4Coef cf;
    if (UNIFORM != 0) {
        cf = p.coef;
    } else {
        cf = make_coef(p.gamma[b * p.gamma_stride], p.alpha[b * p.alpha_stride], p.h);
    }
    double        pm[4] = {0.0, 0.0, 0.0, 0.0};
    const int32_t bad = fast_integrate<TRACE, PMAX, UNIFORM != 2>(p, b, dbeta, cf, y, pm);
    write_results(p, b, y, pm, PMAX, bad);
}

// ------------------------------------------------------------------ z-segment scheduler
// The integrators as PERSISTENT kernels for batches of one wave or more.  Every point costs the same, so a
// batch of 1.65 waves (125 000 points per GPU when the 1e6-point grid is split over 8 GPUs) runs as one
// full wave plus a second wave at 65 % occupancy that takes nearly as long: the sub-partition with the
// most warps sets the time.  Here the fiber is cut into segments of seg_steps RK4 steps and the work
// items (warp of 32 points, segment) are handed out in segment-major order from one atomic counter to
// the resident warps: the chip stays full until the last seg_steps of the last item, so the tail costs
// at most one segment instead of one wave.  Between segments a point's state (y, running maxima, first
// bad step, its Delta-beta: 14 doubles + 1 int, SoA) goes through global memory -- 116 B per point per
// segment, L2-resident -- and done[w] counts the finished segments of warp-item w (release / acquire).
// When item t is handed out at most R-1 older items (R = resident warps) can still be running, and the
// launcher only segments batches of n_warps >= R items per segment, so the item t depends on, t - n_warps,
// is normally finished: the acquire loop is a correctness guard, not a wait.  Segment boundaries are
// multiples of kResync steps, which makes the arithmetic -- phase re-synchronisation, save schedule,
// finite check -- identical to the whole-run loop: results are bit-identical to the whole-run kernels.
struct SegParams {
    unsigned int* counter;    // [1] next work item (zeroed by the launcher)
    int*          done;       // [n_warps] finished segments per warp-item (zeroed by the launcher)
    double*       state;      // [kSegDoubles][n_pad]
    int32_t*      bad;        // [n_pad]
    int64_t       n_pad;      // n_warps * 32
    int           n_warps, n_seg, seg_steps;
};
constexpr int kSegDoubles = 13;  // y[8], pm[4], dbeta
constexpr int kSegDoublesPhase = kSegDoubles + 1;  // the phase sweep adds the last saved signal power

__device__ __forceinline__ int ld_acquire(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(int* p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Next work item of the z-segment scheduler for this warp: (segment, warp-item), or false when the queue
// is empty.  Waits (normally zero iterations) until the item's previous segment has been published.
__device__ __forceinline__ bool seg_next_item(const SegParams& g, int lane, int& seg, int& w) {
    unsigned t = 0;
    if (lane == 0) t = atomicAdd(g.counter, 1u);
    t = __shfl_sync(0xffffffffu, t, 0);
    if (t >= (unsigned)g.n_warps * (unsigned)g.n_seg) return false;
    seg = (int)(t / (unsigned)g.n_warps);
    w   = (int)(t - (unsigned)seg * (unsigned)g.n_warps);
    if (seg > 0) {
        while (ld_acquire(g.done + w) < seg) __nanosleep(100);
    }
    return true;
}

__device__ __forceinline__ void seg_publish(const SegParams& g, int lane, int seg, int w) {
    __threadfence();
    __syncwarp();
    if (lane == 0) st_release(g.done + w, seg + 1);
}

// The batch integrator through the z-segment scheduler:
// same arithmetic as yaman4_fast_kernel, bit-identical results.  Uniform physics only (UNIFORM = 1 | 2).
template <bool TRACE, bool PMAX, int UNIFORM, int THREADS, int MIN_BLOCKS>
__global__ void __launch_bounds__(THREADS, MIN_BLOCKS) yaman4_fast_seg_kernel(const Yaman4Params p, const SegParams g) {
    const int lane = threadIdx.x & 31;
    int       seg, w;
    while (seg_next_item(g, lane, seg, w)) {
        const int64_t b = (int64_t)w * 32 + lane;
        const bool    last = seg == g.n_seg - 1;
        if (b < p.n_points) {
            const double dbeta = p.dbeta[b];
            double       y[8], pm[4] = {0.0, 0.0, 0.0, 0.0};
            int32_t      bad = FPA_POINT_OK;
            double* const st = g.state + b;
            if (nonfinite(dbeta)) {
                if (seg == 0) {
                    load_state(p, b, y);
                    write_invalid_point(p, b, y);
                }
            } else {
                if (seg == 0) {
                    load_state(p, b, y);
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) y[j] = __ldcg(st + j * g.n_pad);
                    if (PMAX) {
#pragma unroll
                        for (int j = 0; j < 4; ++j) pm[j] = __ldcg(st + (8 + j) * g.n_pad);
                    }
                    bad = __ldcg(g.bad + b);
                }
                const int i0 = seg * g.seg_steps;
                const int i1 = last ? p.n_steps : i0 + g.seg_steps;
                bad = fast_integrate<TRACE, PMAX, UNIFORM != 2, true>(p, b, dbeta, p.coef, y, pm, i0, i1, bad);
                if (last) {
                    write_results(p, b, y, pm, PMAX, bad);
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) __stcg(st + j * g.n_pad, y[j]);
                    if (PMAX) {
#pragma unroll
                        for (int j = 0; j < 4; ++j) __stcg(st + (8 + j) * g.n_pad, pm[j]);
                    }
                    __stcg(g.bad + b, bad);
                }
            }
        }
        if (!last) seg_publish(g, lane, seg, w);
    }
}

// ------------------------------------------------------------------ fused sweep
// ONE kernel per sweep: per scan point the prologue builds the frequency plan, the validity flag
// and Delta-beta (plan_point.cuh), the body is the fast RK4 loop above, and the epilogue reduces
// to the sweep's gain metric.  Replaces the loop bodies scan_mismtach.py:694-738 / :357-392 incl.
// simulation.run_single_simulation's unit handling (simulation.py:279-336): the reported dbeta
// uses the dispersion as given, the integration uses every beta_n (or the PROVIDED constant)
// divided by the length scale.
struct SweepExtra {
    PlanParams plan;        // axes, method, coefficient table as given (per length unit)
    double     beta_run[FPA_MAX_TAYLOR_ORDER + 1];  // beta_n / scale
    double     provided_run;
    int        same_run;    // scale == 1: the run's dbeta is the reported one
    double     A0[8];
    double     p_signal;
    double*    gain_lin;    // [B]
    int64_t    first_point; // grid index of point 0 of this launch (sub-range sweeps; outputs are indexed locally)
    double*    peer[FPA_MAX_PEERS];  // full-size gain maps on the GPUs of the box (peer memory), indexed by the grid
    int        n_peers;
};

// The phase sweep (fpa_yaman4_phase_sweep_*): every grid point g runs K initial states, point b = g*K + k of the
// launch is phase k of grid point g (phases fastest: the K runs of a grid point share warps and take the same
// plan / validity branches).  A0_table[k] is make_initial_amplitudes(p_in, phase_in + phase_axis[k]*weights),
// built on the host, so each run starts from the bits the plain sweep would use with that phase_in.
struct PhaseSweepExtra : SweepExtra {
    const double* A0_table;    // [K,4] complex128
    int64_t       n_phases;    // K
    int           last_saved;  // metric: 1 = |A3|^2 of the last saved sample, 0 = max over the saved samples
};
// The sweep kernels take their arguments as X = SweepExtra (plain sweep) or PhaseSweepExtra (phase sweep).
template <typename X>
constexpr bool kPhase = std::is_same<X, PhaseSweepExtra>::value;

// (grid point, phase) of launch point b
template <typename X>
__device__ __forceinline__ void sweep_point(const X& x, int64_t b, int64_t& gp, int64_t& k) {
    if constexpr (kPhase<X>) {
        gp = b / x.n_phases;
        k  = b - gp * x.n_phases;
    } else {
        gp = b;
        k  = 0;
    }
}

template <typename X>
__device__ __forceinline__ void sweep_initial_state(const X& x, int64_t k, double (&y)[8]) {
    if constexpr (kPhase<X>) {
        const double2* a0 = reinterpret_cast<const double2*>(x.A0_table) + k * 4;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double2 v = a0[j];
            y[2 * j] = v.x;
            y[2 * j + 1] = v.y;
        }
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) y[j] = x.A0[j];
    }
}

// Symmetric sweep (A0 waves 2 and 4 are bit copies of waves 1 and 3): the state is (x1, y1, x3, y3).
__device__ __forceinline__ void sweep_initial_state(const SweepExtra& x, int64_t, double (&y)[4]) {
    y[0] = x.A0[0];
    y[1] = x.A0[1];
    y[2] = x.A0[4];
    y[3] = x.A0[5];
}

// The full end state and maxima of a symmetric run: waves 2 and 4 are copies of waves 1 and 3.
__device__ __forceinline__ void sym_expand(const double (&s)[4], double (&y)[8], double (&pm)[4]) {
    y[0] = y[2] = s[0];
    y[1] = y[3] = s[1];
    y[4] = y[6] = s[2];
    y[5] = y[7] = s[3];
    pm[1] = pm[0];
    pm[3] = pm[2];
}

// The signal power the gain is taken from: max over the saved samples, or (phase sweep, "end") the last saved one.
template <typename X>
__device__ __forceinline__ double sweep_metric(const X& x, const double (&pm)[4], double plast) {
    if constexpr (kPhase<X>) return x.last_saved ? plast : pm[2];
    return pm[2];
}

// The final gather of a multi-GPU sweep, fused into the kernel: the thread that finishes a point stores its gain
// into the full-size map of every GPU of the box (NVLink peer stores, posted, 8 B per point and peer) while the
// other points still integrate.
__device__ __forceinline__ void store_gain(const SweepExtra& x, int64_t b, double gain) {
    x.gain_lin[b] = gain;
    if (x.n_peers > 0) {
        const int64_t bg = b + x.first_point;
        for (int q = 0; q < x.n_peers; ++q) x.peer[q][bg] = gain;
        __threadfence_system();
    }
}

// Prologue of grid point b (of this launch): frequency plan, validity, reported and integration Delta-beta; writes
// the plan outputs when `lead` (one lane per grid point of a phase sweep).  Returns false for points the
// reference's per-point try/except turns into NaN.
__device__ __forceinline__ bool sweep_prologue(const SweepExtra& x, int64_t b, double& db_run, bool lead = true) {
    const int64_t bg = b + x.first_point;
    const int64_t i1 = bg / x.plan.n3, i3 = bg - i1 * x.plan.n3;
    double w[4];
    bool   ok = plan_omegas(x.plan.lambda1[i1], x.plan.lambda2[i1 * x.plan.lambda2_stride], x.plan.lambda3[i3], w);
    const double db_report = plan_dbeta(x.plan, x.plan.beta, x.plan.provided, w, ok);
    db_run = db_report;
    if (!x.same_run) {
        bool ok_run = ok;
        db_run = plan_dbeta(x.plan, x.beta_run, x.provided_run, w, ok_run);
        if (!ok_run) db_run = qnan();
    }
    if (lead && x.plan.dbeta) x.plan.dbeta[b] = db_report;
    if (lead && x.plan.valid) x.plan.valid[b] = ok ? 1 : 0;
    if (lead && x.plan.omega) {
        double2* o = reinterpret_cast<double2*>(x.plan.omega + b * 4);
        o[0] = make_double2(w[0], w[1]);
        o[1] = make_double2(w[2], w[3]);
    }
    return ok && !nonfinite(db_run);
}

// the reference's per-point try/except leaves NaN (scan_mismtach.py:736-738)
__device__ __forceinline__ void sweep_invalid(const Yaman4Params& p, const SweepExtra& x, int64_t b) {
    const double qn = qnan();
    if (p.A_end)
        for (int j = 0; j < 4; ++j) store_c128(p.A_end + b * 8 + 2 * j, qn, qn);
    if (p.Pmax)
        for (int j = 0; j < 4; ++j) p.Pmax[b * 4 + j] = qn;
    if (p.status) p.status[b] = p.check ? 0 : FPA_POINT_OK;
    store_gain(x, b, qn);
}

// Epilogue of an integrated point: status, optional end state / maxima, and the sweep's gain metric P3 / p_in[2].
__device__ __forceinline__ void sweep_epilogue(const Yaman4Params& p, const SweepExtra& x, int64_t b,
                                               const double (&y)[8], const double (&pm)[4], int32_t bad, double P3) {
    if (p.check && bad == FPA_POINT_OK) {
        bool nf = false;
#pragma unroll
        for (int j = 0; j < 8; ++j) nf |= nonfinite(y[j]);
        if (nf) bad = p.n_steps - 1;
    }
    if (p.status) p.status[b] = p.check ? bad : FPA_POINT_OK;
    if (p.A_end) {
#pragma unroll
        for (int j = 0; j < 4; ++j) store_c128(p.A_end + b * 8 + 2 * j, y[2 * j], y[2 * j + 1]);
    }
    if (p.Pmax) {
        double2* o = reinterpret_cast<double2*>(p.Pmax + b * 4);
        o[0] = make_double2(pm[0], pm[1]);
        o[1] = make_double2(pm[2], pm[3]);
    }
    // gain = max_saved |A3|^2 / p_in[2]; NaN for failed, non-finite or <= 0 (scan_mismtach.py:723-734).  The
    // phase sweep's "end" metric takes P3 from the last saved sample under the same rule.
    double gain = qnan();
    if (!(p.check && bad != FPA_POINT_OK) && !nonfinite(pm[2])) {
        const double q = P3 / x.p_signal;
        if (!nonfinite(q) && q > 0.0) gain = q;
    }
    store_gain(x, b, gain);
}

// X = PhaseSweepExtra: the phase sweep.  SYM (plain sweep only): A0 is symmetric, the z-loop runs on (A1, A3).
template <bool LOSS, int THREADS, int MIN_BLOCKS, typename X, bool SYM = false>
__global__ void __launch_bounds__(THREADS, MIN_BLOCKS) yaman4_sweep_kernel(const Yaman4Params p, const X x) {
    constexpr bool PHASE = kPhase<X>;
    static_assert(!(SYM && PHASE), "the phase sweep has no symmetric path");
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= p.n_points) return;
    int64_t gp, k;
    sweep_point(x, b, gp, k);
    double db_run;
    if (!sweep_prologue(x, gp, db_run, k == 0)) {
        sweep_invalid(p, x, b);
        return;
    }
    double y[kStateLen<SYM>];
    sweep_initial_state(x, k, y);
    double        pm[4] = {0.0, 0.0, 0.0, 0.0}, plast = 0.0;
    const int32_t bad = fast_integrate<false, true, LOSS, false, PHASE, SYM>(p, b, db_run, p.coef, y, pm, 0, 0,
                                                                             FPA_POINT_OK, &plast);
    if constexpr (SYM) {
        double yf[8];
        sym_expand(y, yf, pm);
        sweep_epilogue(p, x, b, yf, pm, bad, pm[2]);
    } else {
        sweep_epilogue(p, x, b, y, pm, bad, sweep_metric(x, pm, plast));
    }
}

// ------------------------------------------------------------------ fused sweep, z-segment scheduler
// The sweep kernel above as a persistent kernel on the z-segment scheduler: prologue at segment 0, gain
// epilogue at the last segment, the point's integration Delta-beta travels with its state (phase sweep: and the
// last saved signal power, record kSegDoubles of the state).  SYM: the record carries the symmetric state
// (x1, y1, x3, y3) in slots 0-3 and the maxima of waves 1 and 3 in slots 8 and 10.
template <bool LOSS, int THREADS, int MIN_BLOCKS, typename X, bool SYM = false>
__global__ void __launch_bounds__(THREADS, MIN_BLOCKS)
    yaman4_sweep_seg_kernel(const Yaman4Params p, const X x, const SegParams g) {
    constexpr bool PHASE = kPhase<X>;
    static_assert(!(SYM && PHASE), "the phase sweep has no symmetric path");
    constexpr int NS = kStateLen<SYM>, PM_STEP = SYM ? 2 : 1;
    const int lane = threadIdx.x & 31;
    int       seg, w;
    while (seg_next_item(g, lane, seg, w)) {
        const int64_t b = (int64_t)w * 32 + lane;
        const bool    last = seg == g.n_seg - 1;
        if (b < p.n_points) {
            double  y[NS], pm[4] = {0.0, 0.0, 0.0, 0.0}, db_run, plast = 0.0;
            int32_t bad = FPA_POINT_OK;
            bool    run;
            double* const st = g.state + b;
            if (seg == 0) {
                int64_t gp, k;
                sweep_point(x, b, gp, k);
                run = sweep_prologue(x, gp, db_run, k == 0);
                if (!run) {
                    sweep_invalid(p, x, b);
                    db_run = qnan();
                }
                sweep_initial_state(x, k, y);
            } else {
                db_run = __ldcg(st + 12 * g.n_pad);
                run = !nonfinite(db_run);
                if (run) {
#pragma unroll
                    for (int j = 0; j < NS; ++j) y[j] = __ldcg(st + j * g.n_pad);
#pragma unroll
                    for (int j = 0; j < 4; j += PM_STEP) pm[j] = __ldcg(st + (8 + j) * g.n_pad);
                    if (PHASE) plast = __ldcg(st + kSegDoubles * g.n_pad);
                    bad = __ldcg(g.bad + b);
                }
            }
            if (run) {
                const int i0 = seg * g.seg_steps;
                const int i1 = last ? p.n_steps : i0 + g.seg_steps;
                bad = fast_integrate<false, true, LOSS, true, PHASE, SYM>(p, b, db_run, p.coef, y, pm, i0, i1, bad,
                                                                          &plast);
                if (last) {
                    if constexpr (SYM) {
                        double yf[8];
                        sym_expand(y, yf, pm);
                        sweep_epilogue(p, x, b, yf, pm, bad, pm[2]);
                    } else {
                        sweep_epilogue(p, x, b, y, pm, bad, sweep_metric(x, pm, plast));
                    }
                }
            }
            if (!last) {
                __stcg(st + 12 * g.n_pad, db_run);
                if (run) {
#pragma unroll
                    for (int j = 0; j < NS; ++j) __stcg(st + j * g.n_pad, y[j]);
#pragma unroll
                    for (int j = 0; j < 4; j += PM_STEP) __stcg(st + (8 + j) * g.n_pad, pm[j]);
                    if (PHASE) __stcg(st + kSegDoubles * g.n_pad, plast);
                    __stcg(g.bad + b, bad);
                }
            }
        }
        if (!last) seg_publish(g, lane, seg, w);
    }
}

// ------------------------------------------------------------------ exact path
// dA/dz for one point.  (pr,pi) = 2*gamma*exp(i*dbeta*z); nha = -alpha/2.
__device__ __forceinline__ void rhs4(const double (&y)[8], double pr, double pi, double gamma,
                                     double nha, double (&k)[8], double& Ssum) {
    const double zero[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    stage<true>(y, zero, pr, pi, gamma, gamma + gamma, nha, k, Ssum);
}

template <bool GRID>
__global__ void __launch_bounds__(128, 3) yaman4_exact_kernel(const Yaman4Params p) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= p.n_points) return;

    double y[8];
    load_state(p, b, y);
    const double dbeta = p.dbeta[b];
    if (nonfinite(dbeta)) {
        write_invalid_point(p, b, y);
        return;
    }
    const double gamma = p.gamma[b * p.gamma_stride];
    const double nha   = -0.5 * p.alpha[b * p.alpha_stride];
    const double g2    = gamma + gamma;
    const bool   trace = p.A_trace != nullptr, pmax = p.Pmax != nullptr;

    double* tr = trace ? p.A_trace + b * p.n_saved * 8 : nullptr;
    double  pm[4] = {-1.0, -1.0, -1.0, -1.0};
    save_sample(y, tr, pm, trace, pmax);

    const int    n_steps = p.n_steps;
    const double z0 = p.z0, z_max = p.z_max;
    // numpy.linspace: step = (stop-start)/div, z_i = i*step + start, z_n = stop
    const double step = (z_max - z0) / (double)n_steps;
    double  zi = GRID ? p.z_grid[0] : z0;
    double  di = 0.0;
    int     save_ctr = p.save_every;
    int32_t bad = FPA_POINT_OK;

    for (int i = 0; i < n_steps; ++i) {
        double zn;
        if (GRID) {
            zn = p.z_grid[i + 1];
        } else {
            di += 1.0;
            zn = (i + 1 == n_steps) ? z_max : __dadd_rn(__dmul_rn(di, step), z0);
        }
        const double h  = zn - zi;  // integrators.py:128
        const double hh = 0.5 * h;
        const double h6 = h / 6.0;  // integrators.py:59
        const double h3 = h6 + h6;

        double s, c, k[8], ys[8], yn[8], S, Sx;
        sincos(dbeta * zi, &s, &c);
        rhs4(y, g2 * c, g2 * s, gamma, nha, k, S);
        if (nonfinite(S) && bad == FPA_POINT_OK && i > 0) {
            bool nf = false;
#pragma unroll
            for (int j = 0; j < 8; ++j) nf |= nonfinite(y[j]);
            if (nf) bad = i - 1;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            yn[j] = fma(h6, k[j], y[j]);
            ys[j] = fma(hh, k[j], y[j]);
        }
        sincos(dbeta * (zi + hh), &s, &c);  // integrators.py:55-56
        const double phr = g2 * c, phi_ = g2 * s;
        rhs4(ys, phr, phi_, gamma, nha, k, Sx);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            yn[j] = fma(h3, k[j], yn[j]);
            ys[j] = fma(hh, k[j], y[j]);
        }
        rhs4(ys, phr, phi_, gamma, nha, k, Sx);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            yn[j] = fma(h3, k[j], yn[j]);
            ys[j] = fma(h, k[j], y[j]);
        }
        sincos(dbeta * (zi + h), &s, &c);  // integrators.py:57
        rhs4(ys, g2 * c, g2 * s, gamma, nha, k, Sx);
#pragma unroll
        for (int j = 0; j < 8; ++j) y[j] = fma(h6, k[j], yn[j]);
        zi = zn;

        if (--save_ctr == 0) {
            save_ctr = p.save_every;
            save_sample(y, tr, pm, trace, pmax);
        }
    }
    write_results(p, b, y, pm, pmax, bad);
}

// RHS-only kernel (direct calls of yaman_model.rhs_yaman_simplified, yaman_model.py:10-52):
// the phase is evaluated exactly at the caller's z.
__global__ void yaman4_rhs_kernel(int64_t B, const double* z, const double* A, const double* gamma,
                                  const double* alpha, const double* dbeta, double* dA) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double y[8], k[8], S, s, c;
#pragma unroll
    for (int j = 0; j < 8; ++j) y[j] = A[b * 8 + j];
    const double g = gamma[b];
    sincos(dbeta[b] * z[b], &s, &c);
    rhs4(y, (g + g) * c, (g + g) * s, g, -0.5 * alpha[b], k, S);
#pragma unroll
    for (int j = 0; j < 8; ++j) dA[b * 8 + j] = k[j];
}

// Launch shape of the fast kernel: kFastThreads threads per block, kFastMinBlocks resident blocks
// per SM (register cap = 65536 / (threads * blocks)); chosen by measurement (tools/tune_yaman4.cu,
// DESIGN.md).
#ifndef FPA_YAMAN4_THREADS
#define FPA_YAMAN4_THREADS 128
#endif
#ifndef FPA_YAMAN4_MIN_BLOCKS
#define FPA_YAMAN4_MIN_BLOCKS 3
#endif
constexpr int kFastThreads = FPA_YAMAN4_THREADS, kFastMinBlocks = FPA_YAMAN4_MIN_BLOCKS;
// the fused sweep kernel gets its best schedule (fewest 3-register FMAs, tools/sass_cost.py) at 4
constexpr int kSweepMinBlocks = 4;
// the symmetric sweep kernels (stage_sym): resident blocks per SM, chosen by measurement (DESIGN.md §4.1c)
#ifndef FPA_SWEEP_SYM_MIN_BLOCKS
#define FPA_SWEEP_SYM_MIN_BLOCKS 4
#endif
constexpr int kSweepSymMinBlocks = FPA_SWEEP_SYM_MIN_BLOCKS;
// z-segment scheduler: RK4 steps per segment (multiples of kResync), chosen by measurement
// (profiles/r2_seg_tune.txt): 64 below two waves of the resident warps, 128 above -- with those the
// scheduler is at least as fast as the whole-run kernel at every batch of one wave or more
// (1.00 waves 68 -> 83 % of the FP64 peak, 1.65 waves 80.8 -> 86.2 %, 6.6 waves 85.4 -> 87.2 %,
// 13.2 waves 87.2 -> 87.3 %).  Above kSegMaxWaves waves the whole-run kernel is kept: its tail is down
// to ~1 % there, and the state hand-over of a batch that large no longer fits the 126 MB L2 (1e6 points:
// 116 MB per hand-over, 3.9 GB of DRAM traffic per sweep against 0.1 MB for the whole-run kernel).
constexpr int kSegStepsShort = 64, kSegStepsLong = 128, kSegMaxWaves = 8;

// ---- z-segment scheduler: scratch layout and launch geometry
static size_t seg_align(size_t v) { return (v + 255) & ~(size_t)255; }

// seg_doubles: doubles of a point's state record (kSegDoubles, or kSegDoublesPhase for the phase sweep)
static int64_t scratch_bytes(int64_t n_points, int seg_doubles) {
    if (n_points <= 0) return 0;
    const size_t n_warps = (size_t)((n_points + 31) / 32), n_pad = n_warps * 32;
    return (int64_t)(256 + seg_align(n_warps * sizeof(int)) + seg_align(n_pad * seg_doubles * sizeof(double)) +
                     seg_align(n_pad * sizeof(int32_t)));
}
int64_t yaman4_scratch_bytes(int64_t n_points) { return scratch_bytes(n_points, kSegDoubles); }
int64_t yaman4_phase_scratch_bytes(int64_t n_points) { return scratch_bytes(n_points, kSegDoublesPhase); }

static int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

// CTAs of a persistent kernel that are resident at once on the current device.
template <typename Kernel>
static int resident_ctas(Kernel kernel, int threads) {
    int dev = 0, sms = 148, per_sm = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0);
    return sms * (per_sm < 1 ? 1 : per_sm);
}

// Decides whether a batch runs through the scheduler and, if so, fills `g` and clears its counters.
// Legal when the caller gave enough scratch, every segment holds at least one item per resident warp
// (then an item's predecessor is finished when it is handed out) and the run has at least two segments.
// FPA_SWEEP_SEG=0 forces the whole-run kernels, =2 lifts the kSegMaxWaves cap, FPA_SWEEP_SEG_STEPS overrides the
// segment length (tools, tests).
static int seg_plan(int64_t B, int64_t n_steps, int ctas, int threads, void* scratch, int64_t scratch_bytes,
                    cudaStream_t st, SegParams& g, bool& use_seg, int seg_doubles = kSegDoubles) {
    const int64_t n_warps = (B + 31) / 32, resident_warps = (int64_t)ctas * (threads / 32);
    // segment length: 64 steps below two waves of the resident warps, else 128; half that for runs of fewer than
    // 1 000 steps, which would otherwise have too few segments to even out the tail (profiles/r2_seg_tune.txt:
    // 1e5 points x 500 steps 81.6 -> 83.8 % with 32, 2.5e5 points 84.8 -> 85.9 % with 64)
    int seg_default = n_warps < 2 * resident_warps ? kSegStepsShort : kSegStepsLong;
    if (n_steps < 1000) seg_default /= 2;
    int seg_steps = env_int("FPA_SWEEP_SEG_STEPS", seg_default);
    seg_steps = (seg_steps + kResync - 1) / kResync * kResync;
    if (seg_steps < kResync) seg_steps = kResync;
    use_seg = env_int("FPA_SWEEP_SEG", 1) != 0 && scratch != nullptr && scratch_bytes >= ::fpa::scratch_bytes(B, seg_doubles) &&
              n_warps >= resident_warps && (n_warps < kSegMaxWaves * resident_warps || env_int("FPA_SWEEP_SEG", 1) == 2) &&
              n_steps >= 2 * (int64_t)seg_steps &&
              n_warps * ((n_steps + seg_steps - 1) / seg_steps) < 4000000000LL;
    if (!use_seg) return FPA_OK;
    char* base = static_cast<char*>(scratch);
    g.counter   = reinterpret_cast<unsigned int*>(base);
    g.done      = reinterpret_cast<int*>(base + 256);
    g.state     = reinterpret_cast<double*>(base + 256 + seg_align((size_t)n_warps * sizeof(int)));
    g.n_pad     = n_warps * 32;
    g.bad       = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(g.state) +
                                             seg_align((size_t)g.n_pad * seg_doubles * sizeof(double)));
    g.n_warps   = (int)n_warps;
    g.seg_steps = seg_steps;
    g.n_seg     = (int)((n_steps + seg_steps - 1) / seg_steps);
    FPA_CUDA(cudaMemsetAsync(base, 0, 256 + (size_t)n_warps * sizeof(int), st));
    return FPA_OK;
}

template <bool TRACE, bool PMAX>
static int launch_fast(const Yaman4Params& p, bool uniform, void* scratch, int64_t scratch_bytes, cudaStream_t st) {
    const int  threads = kFastThreads;
    const long blocks  = (long)((p.n_points + threads - 1) / threads);
    if (uniform) {  // the z-segment scheduler carries the uniform-physics instantiations
        SegParams g;
        bool      use_seg = false;
        const int ctas = p.lossless ? resident_ctas(yaman4_fast_seg_kernel<TRACE, PMAX, 2, kFastThreads, kFastMinBlocks>, threads)
                                    : resident_ctas(yaman4_fast_seg_kernel<TRACE, PMAX, 1, kFastThreads, kFastMinBlocks>, threads);
        int       rc = seg_plan(p.n_points, p.n_steps, ctas, threads, scratch, scratch_bytes, st, g, use_seg);
        if (rc != FPA_OK) return rc;
        if (use_seg) {
            if (p.lossless)
                yaman4_fast_seg_kernel<TRACE, PMAX, 2, kFastThreads, kFastMinBlocks><<<ctas, threads, 0, st>>>(p, g);
            else
                yaman4_fast_seg_kernel<TRACE, PMAX, 1, kFastThreads, kFastMinBlocks><<<ctas, threads, 0, st>>>(p, g);
            FPA_CUDA(cudaGetLastError());
            return FPA_OK;
        }
    }
    if (uniform && p.lossless)
        yaman4_fast_kernel<TRACE, PMAX, 2, kFastThreads, kFastMinBlocks><<<blocks, threads, 0, st>>>(p);
    else if (uniform)
        yaman4_fast_kernel<TRACE, PMAX, 1, kFastThreads, kFastMinBlocks><<<blocks, threads, 0, st>>>(p);
    else
        yaman4_fast_kernel<TRACE, PMAX, 0, kFastThreads, kFastMinBlocks><<<blocks, threads, 0, st>>>(p);
    FPA_CUDA(cudaGetLastError());
    return FPA_OK;
}

// The checks of a batch descriptor, for the device and the host entries alike.  FPA_UNIFORM_PHYSICS is checked by
// yaman4_launch alone: the host entry sets or clears that flag itself.
int yaman4_check(const fpa_yaman4_desc* d) {
    FPA_REQUIRE(d != nullptr, "descriptor is NULL");
    FPA_REQUIRE(d->n_points >= 0, "n_points must be >= 0");
    FPA_REQUIRE(d->n_steps >= 1 && d->n_steps < 2147483647LL, "n_steps must be in [1, 2^31)");
    FPA_REQUIRE(d->save_every >= 1, "save_every must be a positive integer");
    FPA_REQUIRE(d->dbeta && d->gamma && d->alpha && d->A0, "dbeta/gamma/alpha/A0 must be set");
    FPA_REQUIRE((d->gamma_stride | 1) == 1 && (d->alpha_stride | 1) == 1 && (d->A0_stride | 1) == 1,
                "strides must be 0 (broadcast) or 1 (per point)");
    FPA_REQUIRE(!(d->flags & FPA_OUT_TRACE) || d->A_trace, "FPA_OUT_TRACE needs A_trace");
    FPA_REQUIRE(!(d->flags & FPA_OUT_PMAX) || d->Pmax, "FPA_OUT_PMAX needs Pmax");
    FPA_REQUIRE(!(d->flags & FPA_OUT_END) || d->A_end, "FPA_OUT_END needs A_end");
    return FPA_OK;
}

int yaman4_launch(const fpa_yaman4_desc* d, cudaStream_t st) {
    int rc = yaman4_check(d);
    if (rc != FPA_OK) return rc;
    const bool trace = (d->flags & FPA_OUT_TRACE) != 0;
    const bool pmax  = (d->flags & FPA_OUT_PMAX) != 0;
    const bool endo  = (d->flags & FPA_OUT_END) != 0;
    const bool uniform = (d->flags & FPA_UNIFORM_PHYSICS) != 0;
    FPA_REQUIRE(!uniform || (d->gamma_stride == 0 && d->alpha_stride == 0),
                "FPA_UNIFORM_PHYSICS needs broadcast gamma and alpha (stride 0)");
    if (d->n_points == 0) return FPA_OK;

    Yaman4Params p;
    p.n_points     = d->n_points;
    p.dbeta        = d->dbeta;
    p.gamma        = d->gamma;
    p.alpha        = d->alpha;
    p.A0           = d->A0;
    p.z_grid       = d->z_grid;
    p.A_trace      = trace ? d->A_trace : nullptr;
    p.A_end        = endo ? d->A_end : nullptr;
    p.Pmax         = pmax ? d->Pmax : nullptr;
    p.status       = d->status;
    p.z0           = d->z0;
    p.z_max        = d->z_max;
    p.h            = (d->z_max - d->z0) / (double)d->n_steps;
    p.gamma_stride = (int)d->gamma_stride;
    p.alpha_stride = (int)d->alpha_stride;
    p.A0_stride    = (int)d->A0_stride;
    p.n_steps      = (int)d->n_steps;
    // save_every > n_steps never fires; clamp so the countdown fits an int
    p.save_every   = (int)(d->save_every > d->n_steps ? d->n_steps + 1 : d->save_every);
    p.check        = (d->flags & FPA_CHECK_NAN) ? 1 : 0;
    p.n_saved      = fpa_n_saved(d->n_steps, d->save_every);
    p.coef         = make_coef(uniform ? d->gamma_uniform : 0.0, uniform ? d->alpha_uniform : 0.0, p.h);
    p.lossless     = (uniform && d->alpha_uniform == 0.0) ? 1 : 0;

    const int    threads = 128;
    const long   blocks  = (long)((p.n_points + threads - 1) / threads);
    if (d->z_grid || (d->flags & FPA_PHASE_EXACT)) {
        if (d->z_grid)
            yaman4_exact_kernel<true><<<blocks, threads, 0, st>>>(p);
        else
            yaman4_exact_kernel<false><<<blocks, threads, 0, st>>>(p);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return cuda_fail(e, "yaman4_exact_kernel launch");
        return FPA_OK;
    }
    if (trace && pmax) return launch_fast<true, true>(p, uniform, d->scratch, d->scratch_bytes, st);
    if (trace) return launch_fast<true, false>(p, uniform, d->scratch, d->scratch_bytes, st);
    if (pmax) return launch_fast<false, true>(p, uniform, d->scratch, d->scratch_bytes, st);
    return launch_fast<false, false>(p, uniform, d->scratch, d->scratch_bytes, st);
}

// plan: the sweep's plan descriptor (device axis pointers); run_scale = 1 or 1000 (length unit);
// gamma/alpha/z_max/dz per length unit, exactly as fpa_sweep_desc carries them.
int plan_fill(const fpa_plan_desc* d, PlanParams& p);

// The grid points a sweep runs: the whole n1*n3 grid, or the sub-range [first_point, first_point + n_sub_points).
int sweep_grid_points(const fpa_sweep_desc* d, int64_t* n_grid) {
    const int64_t grid = d->plan.n1 * d->plan.n3;
    FPA_REQUIRE(d->first_point >= 0 && d->n_sub_points >= 0 && d->first_point + d->n_sub_points <= grid,
                "first_point / n_sub_points must select a range of the n1*n3 grid");
    *n_grid = (d->first_point == 0 && d->n_sub_points == 0) ? grid : d->n_sub_points;
    return FPA_OK;
}

// Checks a sweep descriptor and fills the kernel arguments for its n_grid grid points (the whole grid or the
// sub-range) x n_phases runs each; the plain sweep is n_phases = 1.
static int sweep_setup(const fpa_sweep_desc* d, int64_t n_phases, Yaman4Params& p, SweepExtra& x, int64_t& n_grid) {
    FPA_REQUIRE(d != nullptr, "sweep descriptor is NULL");
    if (d->flags & FPA_PHASE_EXACT) {
        set_error("FPA_PHASE_EXACT is not available for the fused sweep: build the table with fpa_dbeta_table_* "
                  "and integrate with fpa_yaman4_rk4_batch_* (which honours the flag)");
        return FPA_ERR_UNSUPPORTED;
    }
    int rc = plan_fill(&d->plan, x.plan);
    if (rc != FPA_OK) return rc;
    rc = sweep_grid_points(d, &n_grid);
    if (rc != FPA_OK) return rc;
    const int64_t B = n_grid * n_phases;
    FPA_REQUIRE(d->gain_lin != nullptr || B == 0, "gain_lin must be set");
    FPA_REQUIRE(d->length_scale == 1.0 || d->length_scale == 1000.0, "length_scale must be 1 or 1000");
    FPA_REQUIRE(d->z_max > 0.0, "z_max must be positive");
    FPA_REQUIRE(d->dz > 0.0, "dz must be positive");
    FPA_REQUIRE(d->save_every >= 1, "save_every must be a positive integer");
    FPA_REQUIRE(d->p_signal > 0.0, "p_in[2] (signal seed power) must be > 0 to define gain");
    if (B == 0) return FPA_OK;
    const double sc = d->length_scale;
    const int64_t n_steps = fpa_interval_steps(d->z_max * sc, d->dz * sc);
    FPA_REQUIRE(n_steps >= 1 && n_steps < 2147483647LL, "z_max/dz must round to a step count in [1, 2^31)");

    x.same_run = sc == 1.0 ? 1 : 0;
    for (int n = 0; n <= FPA_MAX_TAYLOR_ORDER; ++n) x.beta_run[n] = d->plan.beta[n] / sc;  // simulation.py:126-150
    x.provided_run = d->plan.provided / sc;                                               // simulation.py:153-175
    for (int j = 0; j < 8; ++j) x.A0[j] = d->A0[j];
    x.p_signal = d->p_signal;
    x.gain_lin = d->gain_lin;
    x.first_point = d->first_point;
    FPA_REQUIRE(d->n_peers >= 0 && d->n_peers <= FPA_MAX_PEERS, "n_peers must be in [0, %d]", FPA_MAX_PEERS);
    x.n_peers = d->n_peers;
    for (int q = 0; q < FPA_MAX_PEERS; ++q) {
        x.peer[q] = q < d->n_peers ? d->peer_gain[q] : nullptr;
        FPA_REQUIRE(q >= d->n_peers || x.peer[q] != nullptr, "peer_gain[%d] is NULL", q);
    }

    memset(&p, 0, sizeof(p));
    p.n_points   = B;
    p.A_end      = d->A_end;
    p.Pmax       = d->Pmax;
    p.status     = d->status;
    p.z0         = 0.0;
    p.z_max      = d->z_max * sc;
    p.h          = p.z_max / (double)n_steps;
    p.n_steps    = (int)n_steps;
    p.save_every = (int)(d->save_every > n_steps ? n_steps + 1 : d->save_every);
    p.check      = (d->flags & FPA_CHECK_NAN) ? 1 : 0;
    p.n_saved    = fpa_n_saved(n_steps, d->save_every);
    p.coef       = make_coef(d->gamma / sc, d->alpha / sc, p.h);
    p.lossless   = d->alpha == 0.0 ? 1 : 0;
    return FPA_OK;
}

// z-segment scheduler when the batch is a wave or more, else the whole-run kernel.  SYM: the symmetric kernels (their
// own launch shape); resident_ctas and seg_plan see the kernel that will run.
template <typename X, bool SYM = false>
static int sweep_run(const Yaman4Params& p, const X& x, void* scratch, int64_t scratch_bytes, cudaStream_t st) {
    constexpr bool PHASE = kPhase<X>;
    constexpr int  MB = SYM ? kSweepSymMinBlocks : kSweepMinBlocks;
    const int64_t B = p.n_points;
    const bool    lossless = p.lossless != 0;
    const int ctas = lossless ? resident_ctas(yaman4_sweep_seg_kernel<false, kFastThreads, MB, X, SYM>, kFastThreads)
                              : resident_ctas(yaman4_sweep_seg_kernel<true, kFastThreads, MB, X, SYM>, kFastThreads);
    SegParams g;
    bool      use_seg = false;
    int rc = seg_plan(B, p.n_steps, ctas, kFastThreads, scratch, scratch_bytes, st, g, use_seg,
                      PHASE ? kSegDoublesPhase : kSegDoubles);
    if (rc != FPA_OK) return rc;
    if (use_seg) {
        if (lossless)
            yaman4_sweep_seg_kernel<false, kFastThreads, MB, X, SYM><<<ctas, kFastThreads, 0, st>>>(p, x, g);
        else
            yaman4_sweep_seg_kernel<true, kFastThreads, MB, X, SYM><<<ctas, kFastThreads, 0, st>>>(p, x, g);
    } else {
        const long blocks = (long)((B + kFastThreads - 1) / kFastThreads);
        if (lossless)
            yaman4_sweep_kernel<false, kFastThreads, MB, X, SYM><<<blocks, kFastThreads, 0, st>>>(p, x);
        else
            yaman4_sweep_kernel<true, kFastThreads, MB, X, SYM><<<blocks, kFastThreads, 0, st>>>(p, x);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "yaman4_sweep_kernel launch");
    return FPA_OK;
}

// A0 has A1 == A2 and A3 == A4 BIT FOR BIT (a value test would take -0.0 for 0.0, and the runs would then differ in
// the sign of a zero); FPA_SWEEP_SYM=0 turns the symmetric kernels off (tests, A/B timing).
static bool sweep_symmetric(const SweepExtra& x) {
    return env_int("FPA_SWEEP_SYM", 1) != 0 && memcmp(&x.A0[0], &x.A0[2], 2 * sizeof(double)) == 0 &&
           memcmp(&x.A0[4], &x.A0[6], 2 * sizeof(double)) == 0;
}

int yaman4_sweep_launch(const fpa_sweep_desc* d, void* scratch, int64_t scratch_bytes, cudaStream_t st) {
    Yaman4Params p;
    SweepExtra   x;
    int64_t      n_grid;
    int rc = sweep_setup(d, 1, p, x, n_grid);
    if (rc != FPA_OK || n_grid == 0) return rc;
    if (sweep_symmetric(x)) return sweep_run<SweepExtra, true>(p, x, scratch, scratch_bytes, st);
    return sweep_run(p, x, scratch, scratch_bytes, st);
}

// The arguments of the phase axis, for the device and the host entries alike.
int phase_sweep_check(const fpa_phase_sweep_desc* d) {
    FPA_REQUIRE(d != nullptr, "phase sweep descriptor is NULL");
    FPA_REQUIRE(d->sweep.n_peers == 0, "the phase sweep has no peer-store gather: n_peers must be 0");
    FPA_REQUIRE(d->n_phases >= 1 && d->n_phases <= FPA_MAX_PHASES, "n_phases must be in [1, %d]", FPA_MAX_PHASES);
    FPA_REQUIRE(d->A0_table != nullptr, "A0_table must be set");
    FPA_REQUIRE(d->metric == FPA_GAIN_MAX_SAVED || d->metric == FPA_GAIN_LAST_SAVED, "unknown gain metric %d", d->metric);
    return FPA_OK;
}

// The sweep kernels with the phase axis: n_grid * K points, plan outputs per grid point, everything else per point.
int yaman4_phase_sweep_launch(const fpa_phase_sweep_desc* d, void* scratch, int64_t scratch_bytes, cudaStream_t st) {
    Yaman4Params    p;
    PhaseSweepExtra x;
    int64_t         n_grid;
    if (d && (d->sweep.flags & FPA_PHASE_EXACT)) return sweep_setup(&d->sweep, 1, p, x, n_grid);  // FPA_ERR_UNSUPPORTED
    int rc = phase_sweep_check(d);
    if (rc != FPA_OK) return rc;
    const int64_t K = d->n_phases;
    rc = sweep_setup(&d->sweep, K, p, x, n_grid);
    if (rc != FPA_OK || n_grid == 0) return rc;
    x.A0_table   = d->A0_table;
    x.n_phases   = K;
    x.last_saved = d->metric == FPA_GAIN_LAST_SAVED ? 1 : 0;
    return sweep_run(p, x, scratch, scratch_bytes, st);
}

int yaman4_rhs_launch(int64_t B, const double* z, const double* A, const double* gamma,
                      const double* alpha, const double* dbeta, double* dA, cudaStream_t st) {
    if (B == 0) return FPA_OK;
    const int threads = 128;
    yaman4_rhs_kernel<<<(unsigned)((B + threads - 1) / threads), threads, 0, st>>>(B, z, A, gamma, alpha,
                                                                                 dbeta, dA);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "yaman4_rhs_kernel launch");
    return FPA_OK;
}

}  // namespace fpa
