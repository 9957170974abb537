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
//    298 FP64 instructions per lossy step and the same bits (DESIGN.md §4.1c).  The symmetric kernels run
//    stage_sym_fast() (178 per step: exact identities that hold while |A1|^2 + |A3|^2 < 2^1023) and replay a
//    run or segment that left that range with stage_sym().  The launcher decides by a memcmp of A0's bit
//    patterns; FPA_SWEEP_SYM=0 forces the 4-wave kernels.
//    Each family -- the batch (yaman4_fast_kernel) and the fused sweep (yaman4_sweep_kernel) -- has one per-point
//    body, fast_point / sweep_run_point.  Its whole-run kernel runs it once, for the single segment [0, n_steps); its
//    z-segment scheduler kernel (yaman4_fast_seg_kernel / yaman4_sweep_seg_kernel) runs it once per work item through
//    seg_items, with the point carried between segments in a SegRecord.  Both families write a point's outputs with
//    write_results / write_nan_outputs, and launch_fast_family makes the lossy / lossless and segmented / whole-run
//    choice for both.
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

// stage_sym() with fewer FP64 instructions, the same bits whenever T = P1 + P3 < 2^1023 (DESIGN.md §4.1c):
//  * S = (P1 + P1) + (P3 + P3) is exactly 2T (doublings are exact, scaling by 2 commutes with rounding), so
//    c2g * S and c4g * T = (2 c2g) * T are products of the same real numbers: 2 adds fewer.
//  * DBL (stage 2, whose doubled phase (q2r, q2i) = 2 (qr, qi) the z-loop forms anyway for stage 3): with m = y x,
//    fma(x, y, m) is exactly 2m (m's rounding error is below half the spacing at 2m; a subnormal tie rounds to the
//    even 2m), so fma(-qi, Ui, .) == fma(-q2i, m3, .) and the same for Wi, Zr, Zi: Ui and Vi are not formed.
// Both fail only when a doubling overflows, which needs T >= 2^1023.  The high word of T (>= +0 or NaN) is folded
// into `guard` by an unsigned max: guard >= 0x7FE00000 flags T >= 2^1023, inf or NaN, and the caller then replays
// the run with stage_sym().
template <bool LOSS, bool DBL>
__device__ __forceinline__ void stage_sym_fast(const double (&in)[4], const double (&base)[4], double qr, double qi,
                                               double q2r, double q2i, double cg, double c4g, double cn,
                                               double (&out)[4], unsigned& guard) {
    const double x1 = in[0], y1 = in[1], x3 = in[2], y3 = in[3];
    const double P1 = fma(y1, y1, x1 * x1);
    const double P3 = fma(y3, y3, x3 * x3);
    const double T  = P1 + P3;
    const unsigned hiT = (unsigned)__double2hiint(T);
    guard = hiT > guard ? hiT : guard;
    const double c2 = c4g * T;
    const double G1 = fma(-cg, P1, c2);
    const double G3 = fma(-cg, P3, c2);
    const double Ur = fma(-y3, y3, x3 * x3), m3 = y3 * x3;
    const double Vr = fma(-y1, y1, x1 * x1), m1 = y1 * x1;
    double Wr, Wi, Zr, Zi;
    if (DBL) {
        Wr = fma(-q2i, m3, qr * Ur), Wi = fma(q2r, m3, qi * Ur);
        Zr = fma(q2i, m1, qr * Vr),  Zi = fma(q2r, m1, -(qi * Vr));
    } else {
        const double Ui = fma(x3, y3, m3), Vi = fma(x1, y1, m1);
        Wr = fma(-qi, Ui, qr * Ur), Wi = fma(qr, Ui, qi * Ur);
        Zr = fma(qi, Vi, qr * Vr),  Zi = fma(qr, Vi, -(qi * Vr));
    }
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

// Tangent of stage() along t (DESIGN.md §4.1d): tout = tbase + c*Df(in)*t, where in, (qr, qi) and the coefficients
// are those of the base run's stage.  Term by term, with A_j = x_j + i y_j and A_j' = t_{2j} + i t_{2j+1}:
//   P_j' = 2(x_j x_j' + y_j y_j'),  S' = sum_j P_j',  G_j' = c2g S' - cg P_j'
//   U' = A3' A4 + A3 A4',  V' = A1' A2 + A1 A2',  W' = q U',  Z' = conj(q) V'
//   out_j' = base_j' + cn A_j' + i (G_j' A_j + G_j A_j') + i (conj(A_m)' {W|Z} + conj(A_m) {W'|Z'})
// The half powers h_j = x_j x_j' + y_j y_j' are formed and G_j' = fma(-2cg, h_j, 4cg hS), which is exactly
// fma(-cg, P_j', c2g S') (the factors of 2 are exact).  G_j, W and Z are stage()'s expressions on the same operands
// (the compiler shares them with the base stage).  Every product and sum is spelled out with fma, __dmul_rn and
// __dadd_rn: nothing is left to contraction, so oracle/transfer_model.py reproduces it operation for operation.
template <bool LOSS>
__device__ __forceinline__ void tan_wave(double xj, double yj, double dxj, double dyj, double xm, double ym, double dxm,
                                         double dym, double G, double dG, double Cr, double Ci, double dCr, double dCi,
                                         double cn, double tbr, double tbi, double& outr, double& outi) {
    double r = LOSS ? fma(cn, dxj, tbr) : tbr;
    double i = LOSS ? fma(cn, dyj, tbi) : tbi;
    r = fma(-G, dyj, fma(-dG, yj, fma(ym, dCr, fma(dym, Cr, fma(-xm, dCi, fma(-dxm, Ci, r))))));
    i = fma(G, dxj, fma(dG, xj, fma(xm, dCr, fma(dxm, Cr, fma(ym, dCi, fma(dym, Ci, i))))));
    outr = r;
    outi = i;
}

template <bool LOSS>
__device__ __forceinline__ void stage_tan(const double (&in)[8], const double (&t)[8], const double (&tbase)[8],
                                          double qr, double qi, double cg, double c2g, double cn, double (&out)[8]) {
    const double x1 = in[0], y1 = in[1], x2 = in[2], y2 = in[3];
    const double x3 = in[4], y3 = in[5], x4 = in[6], y4 = in[7];
    const double dx1 = t[0], dy1 = t[1], dx2 = t[2], dy2 = t[3];
    const double dx3 = t[4], dy3 = t[5], dx4 = t[6], dy4 = t[7];
    // the base stage's G_j, W, Z (stage())
    const double P1 = fma(y1, y1, x1 * x1);
    const double P2 = fma(y2, y2, x2 * x2);
    const double P3 = fma(y3, y3, x3 * x3);
    const double P4 = fma(y4, y4, x4 * x4);
    const double S  = (P1 + P2) + (P3 + P4);
    const double c2 = c2g * S;
    const double G1 = fma(-cg, P1, c2), G2 = fma(-cg, P2, c2), G3 = fma(-cg, P3, c2), G4 = fma(-cg, P4, c2);
    const double Ur = fma(-y3, y4, x3 * x4), Ui = fma(x3, y4, y3 * x4);
    const double Vr = fma(-y1, y2, x1 * x2), Vi = fma(x1, y2, y1 * x2);
    const double Wr = fma(-qi, Ui, qr * Ur), Wi = fma(qr, Ui, qi * Ur);
    const double Zr = fma(qi, Vi, qr * Vr),  Zi = fma(qr, Vi, -(qi * Vr));
    // the tangent
    const double h1 = fma(y1, dy1, __dmul_rn(x1, dx1));
    const double h2 = fma(y2, dy2, __dmul_rn(x2, dx2));
    const double h3 = fma(y3, dy3, __dmul_rn(x3, dx3));
    const double h4 = fma(y4, dy4, __dmul_rn(x4, dx4));
    const double hS = __dadd_rn(__dadd_rn(h1, h2), __dadd_rn(h3, h4));
    const double c4g = __dadd_rn(c2g, c2g);
    const double d2  = __dmul_rn(c4g, hS);
    const double dG1 = fma(-c2g, h1, d2), dG2 = fma(-c2g, h2, d2), dG3 = fma(-c2g, h3, d2), dG4 = fma(-c2g, h4, d2);
    const double dUr = fma(x3, dx4, fma(-y3, dy4, fma(-dy3, y4, __dmul_rn(dx3, x4))));
    const double dUi = fma(x3, dy4, fma(y3, dx4, fma(dy3, x4, __dmul_rn(dx3, y4))));
    const double dVr = fma(x1, dx2, fma(-y1, dy2, fma(-dy1, y2, __dmul_rn(dx1, x2))));
    const double dVi = fma(x1, dy2, fma(y1, dx2, fma(dy1, x2, __dmul_rn(dx1, y2))));
    const double dWr = fma(-qi, dUi, __dmul_rn(qr, dUr)), dWi = fma(qr, dUi, __dmul_rn(qi, dUr));
    const double dZr = fma(qi, dVi, __dmul_rn(qr, dVr)),  dZi = fma(qr, dVi, -__dmul_rn(qi, dVr));
    tan_wave<LOSS>(x1, y1, dx1, dy1, x2, y2, dx2, dy2, G1, dG1, Wr, Wi, dWr, dWi, cn, tbase[0], tbase[1], out[0], out[1]);
    tan_wave<LOSS>(x2, y2, dx2, dy2, x1, y1, dx1, dy1, G2, dG2, Wr, Wi, dWr, dWi, cn, tbase[2], tbase[3], out[2], out[3]);
    tan_wave<LOSS>(x3, y3, dx3, dy3, x4, y4, dx4, dy4, G3, dG3, Zr, Zi, dZr, dZi, cn, tbase[4], tbase[5], out[4], out[5]);
    tan_wave<LOSS>(x4, y4, dx4, dy4, x3, y3, dx3, dy3, G4, dG4, Zr, Zi, dZr, dZi, cn, tbase[6], tbase[7], out[6], out[7]);
}

// The z-loop hook of fast_integrate: NoTangent (every existing kernel) adds nothing; Tangent carries one tangent
// column t through the run.  stage<s>(in, ...) is called after stage s of a step with that stage's input state and
// coefficients and mirrors it on the tangent, including the RK4 combination with the same exact-sum weights.
struct NoTangent {};

template <bool LOSS>
struct Tangent {
    double t[8], ts[8], tt[8], ta[8];

    template <int S>
    __device__ __forceinline__ void stage(const double (&in)[8], double qr, double qi, double cg, double c2g, double cn) {
        const double third = 1.0 / 3.0, two_thirds = 2.0 / 3.0, third_c = 1.0 - two_thirds;  // as fast_integrate
        if constexpr (S == 0) {
            stage_tan<LOSS>(in, t, t, qr, qi, cg, c2g, cn, ts);
#pragma unroll
            for (int j = 0; j < 8; ++j) ta[j] = fma(third, ts[j], __dmul_rn(t[j], -third));
        } else if constexpr (S == 1) {
            stage_tan<LOSS>(in, ts, t, qr, qi, cg, c2g, cn, tt);
#pragma unroll
            for (int j = 0; j < 8; ++j) ta[j] = fma(two_thirds, tt[j], ta[j]);
        } else if constexpr (S == 2) {
            stage_tan<LOSS>(in, tt, t, qr, qi, cg, c2g, cn, ts);
#pragma unroll
            for (int j = 0; j < 8; ++j) ta[j] = fma(third_c, ts[j], ta[j]);
        } else {
            stage_tan<LOSS>(in, ts, ta, qr, qi, cg, c2g, cn, t);
        }
    }
};

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

// One state (4 x complex128, 16-byte aligned): A0 of a batch point, a row of the phase sweep's A0_table.
__device__ __forceinline__ void load_c128x4(const double* a, double (&y)[8]) {
    const double2* a2 = reinterpret_cast<const double2*>(a);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const double2 v = a2[j];
        y[2 * j] = v.x;
        y[2 * j + 1] = v.y;
    }
}

__device__ __forceinline__ void load_state(const Yaman4Params& p, int64_t b, double (&y)[8]) {
    load_c128x4(p.A0 + b * p.A0_stride * 8, y);
}

// A_end and Pmax all NaN and status 0 (failed at step 0) under the check: the outputs of a point that is not
// integrated.
__device__ __forceinline__ void write_nan_outputs(const Yaman4Params& p, int64_t b) {
    const double qn = qnan();
    if (p.A_end)
        for (int j = 0; j < 4; ++j) store_c128(p.A_end + b * 8 + 2 * j, qn, qn);
    if (p.Pmax)
        for (int j = 0; j < 4; ++j) p.Pmax[b * 4 + j] = qn;
    if (p.status) p.status[b] = p.check ? 0 : FPA_POINT_OK;
}

// A point whose dbeta is not finite: exp(i*dbeta*z) is NaN from the first stage on, every later
// sample is NaN and step 0 is the bad one (integrators.py:132-135).  Invalid scan points of a sweep
// arrive here with dbeta = NaN and cost nothing.
__device__ __noinline__ void write_invalid_point(const Yaman4Params& p, int64_t b, const double (&y)[8]) {
    if (p.A_trace) {
        const double qn = qnan();
        double*      t  = p.A_trace + b * p.n_saved * 8;
        for (int j = 0; j < 4; ++j) store_c128(t + 2 * j, y[2 * j], y[2 * j + 1]);
        for (int64_t s = 1; s < p.n_saved; ++s)
            for (int j = 0; j < 4; ++j) store_c128(t + s * 8 + 2 * j, qn, qn);
    }
    write_nan_outputs(p, b);
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

// Outputs of an integrated point: status (the end state's finite check decides a run that was finite until its
// last step), A_end and, when pmax, Pmax.  Returns the point's first bad step (FPA_POINT_OK: none).
__device__ __forceinline__ int32_t write_results(const Yaman4Params& p, int64_t b, const double (&y)[8],
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
    return bad;
}

// The z-loop of the fast path: advances y over the steps [i0, i1) of the run, keeps the running maxima
// in pm and returns the first step whose result was not finite (or `bad` as given).  The whole run is
// (0, n_steps); the z-segment scheduler (SegParams below) calls it once per segment with the
// state, pm and bad of the previous segment.  i0 must be a multiple of kResync: the phase factor is
// rebuilt by the exact sincos at the first step of the range, exactly where the whole-run loop rebuilds
// it, so a segmented run is bit-identical to a whole one.  LAST: *plast follows the last saved sample (save_sample).
// SYM: y is the symmetric half (x1, y1, x3, y3) of a state with A1 == A2, A3 == A4 (stage_sym); pm[0] and pm[2] are
// kept, pm[1] and pm[3] are left to the caller.
// GUARD (SYM only): the stages are stage_sym_fast(), and no step runs the finite check.  Returns kSymReplay when a
// stage's guard tripped (some T >= 2^1023, inf or NaN: the only states where stage_sym_fast() may differ from
// stage_sym(), and the only ones where the finite check could have fired); the caller then replays the range with
// GUARD = false.  Otherwise the results are those of GUARD = false, and `bad` is returned as given.
template <bool SYM>
constexpr int kStateLen = SYM ? 4 : 8;
constexpr int32_t kSymReplay = -2;
// (double)i, the same bits, through an asm statement: the compiler then cannot keep a floating-point copy of the loop
// counter (one DADD per step) for the re-sync block, which needs it every kResync steps only.
__device__ __forceinline__ double int_to_double_opaque(int i) {
    double d;
    asm("cvt.rn.f64.s32 %0, %1;" : "=d"(d) : "r"(i));
    return d;
}
// Tan: the tangent hook (NoTangent, or Tangent<LOSS> for the transfer kernels: full state, *tan advanced with y).
template <bool TRACE, bool PMAX, bool LOSS, bool SEG = false, bool LAST = false, bool SYM = false, bool GUARD = false,
          typename Tan = NoTangent>
__device__ __forceinline__ int32_t fast_integrate(const Yaman4Params& p, int64_t b, double dbeta,
                                                  const Yaman4Coef& cf, double (&y)[kStateLen<SYM>], double (&pm)[4],
                                                  int i0_in = 0, int i1_in = 0, int32_t bad_in = FPA_POINT_OK,
                                                  double* plast = nullptr, Tan* tan = nullptr) {
    constexpr int NS = kStateLen<SYM>;
    constexpr bool TAN = !std::is_same<Tan, NoTangent>::value;
    static_assert(!SYM || !TRACE, "the symmetric path writes no trace");
    static_assert(!TAN || !SYM, "tangent directions leave the symmetric subspace");
    static_assert(!GUARD || SYM, "the guarded stages are those of the symmetric path");
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
    unsigned     guard = 0;
    // 4*c*gamma of stage_sym_fast(), in registers: a field of Yaman4Coef would grow the parameter block, and with it
    // the machine code of every kernel.  It is finite: sweep_symmetric() sends any other sweep to the 4-wave kernels.
    const double c4g[3] = {cf.c2g[0] + cf.c2g[0], cf.c2g[1] + cf.c2g[1], cf.c2g[2] + cf.c2g[2]};

    for (int i = i0; i < i1; ++i) {
        if ((i & (kResync - 1)) == 0) {
            double s, c;
            sincos(dbeta * fma(GUARD ? int_to_double_opaque(i) : (double)i, h, z0), &s, &c);
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
        if constexpr (GUARD) {
            stage_sym_fast<LOSS, false>(y, y, qr, qi, q2r, q2i, cf.cg[0], c4g[0], cf.cn[0], ys, guard);
        } else {
            rk_stage<LOSS>(y, y, qr, qi, cf.cg[0], cf.c2g[0], cf.cn[0], ys, S);
            // S = sum |A|^2 of the state that step i-1 produced: a non-finite component makes S
            // non-finite, so the exact per-component test runs only then (integrators.py:132-135).
            if (nonfinite(S) && bad == FPA_POINT_OK && i > 0) {
                bool nf = false;
#pragma unroll
                for (int j = 0; j < NS; ++j) nf |= nonfinite(y[j]);
                if (nf) bad = i - 1;
            }
        }
#pragma unroll
        for (int j = 0; j < NS; ++j) acc[j] = fma(third, ys[j], y[j] * (-third));
        if constexpr (TAN) tan->template stage<0>(y, qr, qi, cf.cg[0], cf.c2g[0], cf.cn[0]);
        // stage 2: yt = y + (h/2) f(z+h/2, ys)
        if constexpr (GUARD)
            stage_sym_fast<LOSS, true>(ys, y, qhr, qhi, q2r, q2i, cf.cg[0], c4g[0], cf.cn[0], yt, guard);
        else
            rk_stage<LOSS>(ys, y, qhr, qhi, cf.cg[0], cf.c2g[0], cf.cn[0], yt, Sx);
#pragma unroll
        for (int j = 0; j < NS; ++j) acc[j] = fma(two_thirds, yt[j], acc[j]);
        if constexpr (TAN) tan->template stage<1>(ys, qhr, qhi, cf.cg[0], cf.c2g[0], cf.cn[0]);
        // stage 3: ys = y + h f(z+h/2, yt)
        if constexpr (GUARD)
            stage_sym_fast<LOSS, false>(yt, y, q2r, q2i, q2r, q2i, cf.cg[1], c4g[1], cf.cn[1], ys, guard);
        else
            rk_stage<LOSS>(yt, y, q2r, q2i, cf.cg[1], cf.c2g[1], cf.cn[1], ys, Sx);
#pragma unroll
        for (int j = 0; j < NS; ++j) acc[j] = fma(third_c, ys[j], acc[j]);
        if constexpr (TAN) tan->template stage<2>(yt, q2r, q2i, cf.cg[1], cf.c2g[1], cf.cn[1]);
        // stage 4: y' = acc + (h/6) f(z+h, ys)
        if constexpr (GUARD)
            stage_sym_fast<LOSS, false>(ys, acc, q6r, q6i, q2r, q2i, cf.cg[2], c4g[2], cf.cn[2], y, guard);
        else
            rk_stage<LOSS>(ys, acc, q6r, q6i, cf.cg[2], cf.c2g[2], cf.cn[2], y, Sx);
        if constexpr (TAN) tan->template stage<3>(ys, q6r, q6i, cf.cg[2], cf.c2g[2], cf.cn[2]);

        qr = qfr;
        qi = qfi;

        if (--save_ctr == 0) {  // (i+1) % save_every == 0, integrators.py:137-140
            save_ctr = p.save_every;
            save_sample<LAST>(y, tr, pm, TRACE, PMAX, plast);
        }
    }
    if (GUARD && guard >= 0x7FE00000u) return kSymReplay;
    return bad;
}

// ------------------------------------------------------------------ z-segment scheduler
// The integrators as PERSISTENT kernels for batches of one wave or more.  Every point costs the same, so a
// batch of 1.65 waves (125 000 points per GPU when the 1e6-point grid is split over 8 GPUs) runs as one
// full wave plus a second wave at 65 % occupancy that takes nearly as long: the sub-partition with the
// most warps sets the time.  Here the fiber is cut into segments of seg_steps RK4 steps and the work
// items (warp of 32 points, segment) are handed out in segment-major order from one atomic counter to
// the resident warps: the chip stays full until the last seg_steps of the last item, so the tail costs
// at most one segment instead of one wave.  Between segments a point's record (y, running maxima, first
// bad step and, for the sweeps, its Delta-beta: at most 14 doubles + 1 int, SoA) goes through global memory --
// up to 116 B per point per segment, L2-resident -- and done[w] counts the finished segments of warp-item w
// (release / acquire).
// When item t is handed out at most R-1 older items (R = resident warps) can still be running, and the
// launcher only segments batches of n_warps >= R items per segment, so the item t depends on, t - n_warps,
// is normally finished: the acquire loop is a correctness guard, not a wait.  Segment boundaries are
// multiples of kResync steps, which makes the arithmetic -- phase re-synchronisation, save schedule,
// finite check -- identical to the whole-run loop: results are bit-identical to the whole-run kernels.
struct SegParams {
    unsigned int* counter;    // [1] next work item (zeroed by the launcher)
    int*          done;       // [n_warps] finished segments per warp-item (zeroed by the launcher)
    double*       state;      // [kSegDoubles or kSegDoublesPhase][n_pad]: the records below
    int32_t*      bad;        // [n_pad]
    int64_t       n_pad;      // n_warps * 32
    int           n_warps, n_seg, seg_steps;
};
// The record of point b: slot s at state[s * n_pad + b], the first bad step at bad[b].  Slots: the state y from
// kSegY (8 doubles; symmetric path: the 4 of (x1, y1, x3, y3)), the running maxima from kSegPmax (symmetric path:
// those of waves 1 and 3 only), the sweep's integration Delta-beta at kSegDbeta (the batch path re-reads dbeta[b]
// and leaves it unused) and the phase sweep's last saved signal power at kSegPlast.
constexpr int kSegY = 0, kSegPmax = 8, kSegDbeta = 12, kSegPlast = 13;
constexpr int kSegDoubles      = kSegDbeta + 1;  // batch, plain sweep
constexpr int kSegDoublesPhase = kSegPlast + 1;  // phase sweep

// Point b's view of its record.
struct SegRecord {
    const SegParams& g;
    int64_t          b;
    double*          st;  // slot 0 of point b
    __device__ __forceinline__ SegRecord(const SegParams& g, int64_t b) : g(g), b(b), st(g.state + b) {}
    __device__ __forceinline__ double* slot(int s) const { return st + s * g.n_pad; }

    // Saves (store) or restores (load) the state y of NS doubles, the maxima when PMAX (NS = 4: those of waves 1
    // and 3), the last saved signal power when LAST, and the first bad step.
    template <bool PMAX, bool LAST, int NS>
    __device__ __forceinline__ void store(const double (&y)[NS], const double (&pm)[4], double plast, int32_t bad) const {
        constexpr int PM_STEP = NS == 8 ? 1 : 2;
#pragma unroll
        for (int j = 0; j < NS; ++j) __stcg(slot(kSegY + j), y[j]);
        if (PMAX) {
#pragma unroll
            for (int j = 0; j < 4; j += PM_STEP) __stcg(slot(kSegPmax + j), pm[j]);
        }
        if (LAST) __stcg(slot(kSegPlast), plast);
        __stcg(g.bad + b, bad);
    }
    template <bool PMAX, bool LAST, int NS>
    __device__ __forceinline__ void load(double (&y)[NS], double (&pm)[4], double& plast, int32_t& bad) const {
        constexpr int PM_STEP = NS == 8 ? 1 : 2;
#pragma unroll
        for (int j = 0; j < NS; ++j) y[j] = __ldcg(slot(kSegY + j));
        if (PMAX) {
#pragma unroll
            for (int j = 0; j < 4; j += PM_STEP) pm[j] = __ldcg(slot(kSegPmax + j));
        }
        if (LAST) plast = __ldcg(slot(kSegPlast));
        bad = __ldcg(g.bad + b);
    }
};

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

// The persistent kernels' loop: point(b, seg, last) for point b = 32 w + lane of every work item (w, seg) this warp
// takes, b past the batch included; last: seg is the fiber's last segment.
template <typename Point>
__device__ __forceinline__ void seg_items(const SegParams& g, Point point) {
    const int lane = threadIdx.x & 31;
    int       seg, w;
    while (seg_next_item(g, lane, seg, w)) {
        const bool last = seg == g.n_seg - 1;
        point((int64_t)w * 32 + lane, seg, last);
        if (!last) seg_publish(g, lane, seg, w);
    }
}

// ------------------------------------------------------------------ batch integrator
// Point b of a batch (nothing when b >= n_points): the whole run (SEG = false, seg = 0, last), or segment `seg` of
// it on the z-segment scheduler.  y is the kernel's array, and A0 is read ahead of dbeta[b] on the whole run only:
// write_invalid_point takes y's address, and with y a local of this function, or one read order for both kernels,
// the compiler emits different machine code for the two kernels (same results).
// UNIFORM: 0 = gamma/alpha per thread (whole run only); 1 = uniform physics, coefficients from the constant bank;
// 2 = uniform and lossless (alpha == 0): the 32 loss FMAs per step are not issued.
template <bool TRACE, bool PMAX, int UNIFORM, bool SEG>
__device__ __forceinline__ void fast_point(const Yaman4Params& p, const SegParams& g, int64_t b, int seg, bool last,
                                           double (&y)[8]) {
    if (b >= p.n_points) return;
    if (!SEG) load_state(p, b, y);
    const double    dbeta = p.dbeta[b];
    double          pm[4] = {0.0, 0.0, 0.0, 0.0}, plast;
    int32_t         bad = FPA_POINT_OK;
    const SegRecord rec(g, b);
    if (nonfinite(dbeta)) {
        if (seg == 0) {
            if (SEG) load_state(p, b, y);
            write_invalid_point(p, b, y);
        }
        return;
    }
    if (seg == 0) {
        if (SEG) load_state(p, b, y);
    } else {
        rec.load<PMAX, false>(y, pm, plast, bad);
    }
    const int i0 = seg * g.seg_steps;
    const int i1 = last ? p.n_steps : i0 + g.seg_steps;
    if constexpr (UNIFORM != 0) {
        bad = fast_integrate<TRACE, PMAX, UNIFORM != 2, SEG>(p, b, dbeta, p.coef, y, pm, i0, i1, bad);
    } else {
        const Yaman4Coef cf = make_coef(p.gamma[b * p.gamma_stride], p.alpha[b * p.alpha_stride], p.h);
        bad = fast_integrate<TRACE, PMAX, UNIFORM != 2, SEG>(p, b, dbeta, cf, y, pm, i0, i1, bad);
    }
    if (last) {
        write_results(p, b, y, pm, PMAX, bad);
    } else {
        rec.store<PMAX, false>(y, pm, plast, bad);
    }
}

template <bool TRACE, bool PMAX, int UNIFORM, int THREADS, int MIN_BLOCKS>
__global__ void __launch_bounds__(THREADS, MIN_BLOCKS) yaman4_fast_kernel(const Yaman4Params p) {
    double y[8];
    fast_point<TRACE, PMAX, UNIFORM, false>(p, SegParams{}, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, 0, true, y);
}

// The batch integrator on the z-segment scheduler: uniform physics only (UNIFORM = 1 | 2).
template <bool TRACE, bool PMAX, int UNIFORM, int THREADS, int MIN_BLOCKS>
__global__ void __launch_bounds__(THREADS, MIN_BLOCKS) yaman4_fast_seg_kernel(const Yaman4Params p, const SegParams g) {
    double y[8];
    seg_items(g, [&](int64_t b, int seg, bool last) { fast_point<TRACE, PMAX, UNIFORM, true>(p, g, b, seg, last, y); });
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
        load_c128x4(x.A0_table + k * 8, y);
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
    write_nan_outputs(p, b);
    store_gain(x, b, qnan());
}

// Epilogue of an integrated point: status, optional end state / maxima, and the sweep's gain metric P3 / p_in[2].
__device__ __forceinline__ void sweep_epilogue(const Yaman4Params& p, const SweepExtra& x, int64_t b,
                                               const double (&y)[8], const double (&pm)[4], int32_t bad, double P3) {
    bad = write_results(p, b, y, pm, p.Pmax != nullptr, bad);
    // gain = max_saved |A3|^2 / p_in[2]; NaN for failed, non-finite or <= 0 (scan_mismtach.py:723-734).  The
    // phase sweep's "end" metric takes P3 from the last saved sample under the same rule.
    double gain = qnan();
    if (!(p.check && bad != FPA_POINT_OK) && !nonfinite(pm[2])) {
        const double q = P3 / x.p_signal;
        if (!nonfinite(q) && q > 0.0) gain = q;
    }
    store_gain(x, b, gain);
}

// Point b of a sweep launch (nothing when b >= n_points): the whole run (SEG = false, seg = 0, last), or segment
// `seg` of it on the z-segment scheduler.  The prologue runs at segment 0, the gain epilogue at the last; between
// segments the record carries the integration Delta-beta, NaN for an invalid point, which then runs no segment.
// X = PhaseSweepExtra: the phase sweep.  SYM (plain sweep only): A0 is symmetric, the z-loop runs on (A1, A3).
template <bool LOSS, typename X, bool SYM, bool SEG>
__device__ __forceinline__ void sweep_run_point(const Yaman4Params& p, const X& x, const SegParams& g, int64_t b,
                                                int seg, bool last) {
    constexpr bool PHASE = kPhase<X>;
    static_assert(!(SYM && PHASE), "the phase sweep has no symmetric path");
    if (b >= p.n_points) return;
    double          y[kStateLen<SYM>], pm[4] = {0.0, 0.0, 0.0, 0.0}, db_run, plast = 0.0;
    int32_t         bad = FPA_POINT_OK;
    bool            run;
    const SegRecord rec(g, b);
    if (seg == 0) {
        int64_t gp, k;
        sweep_point(x, b, gp, k);
        run = sweep_prologue(x, gp, db_run, k == 0);
        if (!run) {
            sweep_invalid(p, x, b);
            if (!SEG) return;
            db_run = qnan();
        }
        sweep_initial_state(x, k, y);
    } else {
        db_run = __ldcg(rec.slot(kSegDbeta));
        run = !nonfinite(db_run);
        if (run) rec.load<true, PHASE>(y, pm, plast, bad);
    }
    if (run) {
        const int i0 = seg * g.seg_steps;
        const int i1 = last ? p.n_steps : i0 + g.seg_steps;
        if constexpr (SYM) {
            // The guarded loop; a range where it tripped runs again from its start (A0, or the record, which is only
            // overwritten after the range) with stage_sym(), and the outputs are the replay's.
            bad = fast_integrate<false, true, LOSS, SEG, false, true, true>(p, b, db_run, p.coef, y, pm, i0, i1, bad);
            if (bad == kSymReplay) {
                bad = FPA_POINT_OK;
                if (seg == 0)
                    sweep_initial_state(x, 0, y);
                else
                    rec.load<true, false>(y, pm, plast, bad);
                bad = fast_integrate<false, true, LOSS, SEG, false, true>(p, b, db_run, p.coef, y, pm, i0, i1, bad);
            }
        } else {
            bad = fast_integrate<false, true, LOSS, SEG, PHASE>(p, b, db_run, p.coef, y, pm, i0, i1, bad, &plast);
        }
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
        __stcg(rec.slot(kSegDbeta), db_run);
        if (run) rec.store<true, PHASE>(y, pm, plast, bad);
    }
}

template <bool LOSS, int THREADS, int MIN_BLOCKS, typename X, bool SYM = false>
__global__ void __launch_bounds__(THREADS, MIN_BLOCKS) yaman4_sweep_kernel(const Yaman4Params p, const X x) {
    sweep_run_point<LOSS, X, SYM, false>(p, x, SegParams{}, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, 0, true);
}

// The sweep kernel on the z-segment scheduler.
template <bool LOSS, int THREADS, int MIN_BLOCKS, typename X, bool SYM = false>
__global__ void __launch_bounds__(THREADS, MIN_BLOCKS)
    yaman4_sweep_seg_kernel(const Yaman4Params p, const X x, const SegParams g) {
    seg_items(g, [&](int64_t b, int seg, bool last) { sweep_run_point<LOSS, X, SYM, true>(p, x, g, b, seg, last); });
}

// ------------------------------------------------------------------ small-signal transfer matrices
// J = dA(L)/dA(0) of the discrete map fast_integrate computes (DESIGN.md §4.1d).  One thread per (point, column):
// every lane of a point runs the point's base trajectory with the unchanged stage() calls, so A_end, Pmax, status and
// the gain are those of the batch / sweep kernels bit for bit, and carries one tangent column beside it.  Lane
// k = t mod nc of point b = t / nc starts from the unit vector of component col[k] (2j: Re A_j(z0), 2j+1: Im) and
// stores jac[b, r, k] for the 8 rows r.  Lane 0 writes the point's other outputs.  Whole-run kernels only.
struct TransferParams {
    double*  jac;   // [B, 8, nc]
    int      nc;    // columns per point
    uint32_t cols;  // 4 bits per slot: bits 4k..4k+3 = the state component of slot k
};

struct BatchPoints {};  // X of the batch transfer kernel: the points are fpa_yaman4_desc's

// Lane t of a transfer launch.  X = BatchPoints (batch) or SweepExtra (fused sweep; gain_lin may be NULL).
// UNIFORM as for fast_point: 0 = gamma / alpha per point (batch only), 1 = uniform, 2 = uniform and lossless.
template <int UNIFORM, typename X>
__device__ __forceinline__ void transfer_point(const Yaman4Params& p, const X& x, const TransferParams& tp, int64_t t) {
    constexpr bool SWEEP = std::is_same<X, SweepExtra>::value;
    constexpr bool LOSS  = UNIFORM != 2;
    const int64_t  b = t / tp.nc;
    if (b >= p.n_points) return;
    const int  k    = (int)(t - b * tp.nc);
    const bool lead = k == 0;
    double     y[8], pm[4] = {0.0, 0.0, 0.0, 0.0}, dbeta;
    bool       run;
    if constexpr (SWEEP) {
        run = sweep_prologue(x, b, dbeta, lead);
        sweep_initial_state(x, 0, y);
    } else {
        load_state(p, b, y);
        dbeta = p.dbeta[b];
        run   = !nonfinite(dbeta);
    }
    Tangent<LOSS> tan;
#pragma unroll
    for (int j = 0; j < 8; ++j) tan.t[j] = j == (int)((tp.cols >> (4 * k)) & 15u) ? 1.0 : 0.0;
    bool ok = false;
    if (run) {
        int32_t bad;
        if constexpr (UNIFORM != 0) {
            bad = fast_integrate<false, true, LOSS>(p, b, dbeta, p.coef, y, pm, 0, 0, FPA_POINT_OK, nullptr, &tan);
        } else {
            const Yaman4Coef cf = make_coef(p.gamma[b * p.gamma_stride], p.alpha[b * p.alpha_stride], p.h);
            bad = fast_integrate<false, true, LOSS>(p, b, dbeta, cf, y, pm, 0, 0, FPA_POINT_OK, nullptr, &tan);
        }
        // write_results' status rule, in every lane
        bool nf = false;
#pragma unroll
        for (int j = 0; j < 8; ++j) nf |= nonfinite(y[j]);
        ok = !(p.check && (bad != FPA_POINT_OK || nf));
        if (lead) {
            if constexpr (SWEEP) {
                if (x.gain_lin) sweep_epilogue(p, x, b, y, pm, bad, pm[2]);
                else write_results(p, b, y, pm, p.Pmax != nullptr, bad);
            } else {
                write_results(p, b, y, pm, p.Pmax != nullptr, bad);
            }
        }
    } else if (lead) {
        if constexpr (SWEEP) {
            if (x.gain_lin) sweep_invalid(p, x, b);
            else write_nan_outputs(p, b);
        } else {
            write_nan_outputs(p, b);
        }
    }
    double* J = tp.jac + b * 8 * tp.nc + k;
#pragma unroll
    for (int r = 0; r < 8; ++r) J[r * tp.nc] = ok ? tan.t[r] : qnan();
}

// 128 threads, 2 resident blocks per SM: the lane holds two RK4 states (base and tangent, 4 x 8 doubles each) and
// needs ~200 registers (DESIGN.md §4.1d).
constexpr int kTransferThreads = 128, kTransferMinBlocks = 2;

template <int UNIFORM, typename X>
__global__ void __launch_bounds__(kTransferThreads, kTransferMinBlocks)
    yaman4_transfer_kernel(const Yaman4Params p, const X x, const TransferParams tp) {
    transfer_point<UNIFORM>(p, x, tp, (int64_t)blockIdx.x * blockDim.x + threadIdx.x);
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
                    cudaStream_t st, SegParams& g, bool& use_seg, int seg_doubles) {
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

// Runs p.n_points points of a fast-path kernel family: its z-segment scheduler kernel (seg*, arguments (p, x..., g))
// when seg_plan takes the batch, else its whole-run kernel (run*, arguments (p, x...)); the *_lossless kernels when
// p.lossless.  resident_ctas and seg_plan see the scheduler kernel that would run; seg_doubles is its record size.
template <typename SegK, typename RunK, typename... X>
static int launch_fast_family(SegK seg, SegK seg_lossless, RunK run, RunK run_lossless, int seg_doubles,
                              const char* what, const Yaman4Params& p, void* scratch, int64_t scratch_bytes,
                              cudaStream_t st, const X&... x) {
    const bool lossless = p.lossless != 0;
    const SegK seg_kernel = lossless ? seg_lossless : seg;
    const int  ctas = resident_ctas(seg_kernel, kFastThreads);
    SegParams  g;
    bool       use_seg = false;
    int rc = seg_plan(p.n_points, p.n_steps, ctas, kFastThreads, scratch, scratch_bytes, st, g, use_seg, seg_doubles);
    if (rc != FPA_OK) return rc;
    if (use_seg) {
        seg_kernel<<<ctas, kFastThreads, 0, st>>>(p, x..., g);
    } else {
        const long blocks = (long)((p.n_points + kFastThreads - 1) / kFastThreads);
        (lossless ? run_lossless : run)<<<blocks, kFastThreads, 0, st>>>(p, x...);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, what);
    return FPA_OK;
}

// Uniform physics: the family of UNIFORM = 1 (lossless: 2); per-point physics: the whole-run kernel of UNIFORM = 0.
template <bool TRACE, bool PMAX>
static int launch_fast(const Yaman4Params& p, bool uniform, void* scratch, int64_t scratch_bytes, cudaStream_t st) {
    if (uniform)
        return launch_fast_family(yaman4_fast_seg_kernel<TRACE, PMAX, 1, kFastThreads, kFastMinBlocks>,
                                  yaman4_fast_seg_kernel<TRACE, PMAX, 2, kFastThreads, kFastMinBlocks>,
                                  yaman4_fast_kernel<TRACE, PMAX, 1, kFastThreads, kFastMinBlocks>,
                                  yaman4_fast_kernel<TRACE, PMAX, 2, kFastThreads, kFastMinBlocks>, kSegDoubles,
                                  "cudaGetLastError()", p, scratch, scratch_bytes, st);
    const long blocks = (long)((p.n_points + kFastThreads - 1) / kFastThreads);
    yaman4_fast_kernel<TRACE, PMAX, 0, kFastThreads, kFastMinBlocks><<<blocks, kFastThreads, 0, st>>>(p);
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

// The kernel arguments of a checked batch descriptor (yaman4_launch, yaman4_transfer_launch).
static void batch_params(const fpa_yaman4_desc* d, bool uniform, Yaman4Params& p) {
    p.n_points     = d->n_points;
    p.dbeta        = d->dbeta;
    p.gamma        = d->gamma;
    p.alpha        = d->alpha;
    p.A0           = d->A0;
    p.z_grid       = d->z_grid;
    p.A_trace      = (d->flags & FPA_OUT_TRACE) ? d->A_trace : nullptr;
    p.A_end        = (d->flags & FPA_OUT_END) ? d->A_end : nullptr;
    p.Pmax         = (d->flags & FPA_OUT_PMAX) ? d->Pmax : nullptr;
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
    // load_state, save_sample and write_results access these with 16-byte (trace: also 32-byte) vector accesses
    FPA_REQUIRE_ALIGNED16(d->A0, "A0");
    if (trace) FPA_REQUIRE_ALIGNED16(d->A_trace, "A_trace");
    if (endo) FPA_REQUIRE_ALIGNED16(d->A_end, "A_end");
    if (pmax) FPA_REQUIRE_ALIGNED16(d->Pmax, "Pmax");
    if (d->n_points == 0) return FPA_OK;

    Yaman4Params p;
    batch_params(d, uniform, p);

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
// transfer: the transfer sweep, whose gain_lin may be NULL (and only then p_signal 0).
static int sweep_setup(const fpa_sweep_desc* d, int64_t n_phases, Yaman4Params& p, SweepExtra& x, int64_t& n_grid,
                       bool transfer = false) {
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
    FPA_REQUIRE(d->gain_lin != nullptr || B == 0 || transfer, "gain_lin must be set");
    FPA_REQUIRE(d->length_scale == 1.0 || d->length_scale == 1000.0, "length_scale must be 1 or 1000");
    FPA_REQUIRE(d->z_max > 0.0, "z_max must be positive");
    FPA_REQUIRE(d->dz > 0.0, "dz must be positive");
    FPA_REQUIRE(d->save_every >= 1, "save_every must be a positive integer");
    FPA_REQUIRE(d->p_signal > 0.0 || (transfer && d->gain_lin == nullptr),
                "p_in[2] (signal seed power) must be > 0 to define gain");
    // sweep_prologue and sweep_epilogue store these with 16-byte vector stores
    FPA_REQUIRE_ALIGNED16(d->plan.omega, "plan.omega");
    FPA_REQUIRE_ALIGNED16(d->A_end, "A_end");
    FPA_REQUIRE_ALIGNED16(d->Pmax, "Pmax");
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

// SYM: the symmetric kernels, with their own launch shape.
template <typename X, bool SYM = false>
static int sweep_run(const Yaman4Params& p, const X& x, void* scratch, int64_t scratch_bytes, cudaStream_t st) {
    constexpr int MB = SYM ? kSweepSymMinBlocks : kSweepMinBlocks;
    return launch_fast_family(yaman4_sweep_seg_kernel<true, kFastThreads, MB, X, SYM>,
                              yaman4_sweep_seg_kernel<false, kFastThreads, MB, X, SYM>,
                              yaman4_sweep_kernel<true, kFastThreads, MB, X, SYM>,
                              yaman4_sweep_kernel<false, kFastThreads, MB, X, SYM>,
                              kPhase<X> ? kSegDoublesPhase : kSegDoubles, "yaman4_sweep_kernel launch", p, scratch,
                              scratch_bytes, st, x);
}

// A0 has A1 == A2 and A3 == A4 BIT FOR BIT (a value test would take -0.0 for 0.0, and the runs would then differ in
// the sign of a zero); FPA_SWEEP_SYM=0 turns the symmetric kernels off (tests, A/B timing).  The symmetric kernels'
// 4*c*gamma must be finite (stage_sym_fast): an absurd gamma*h takes the 4-wave kernels, which compute the same bits.
static bool sweep_symmetric(const Yaman4Params& p, const SweepExtra& x) {
    bool c4g_finite = true;
    for (int s = 0; s < 3; ++s) c4g_finite &= std::isfinite(p.coef.c2g[s] + p.coef.c2g[s]);
    return env_int("FPA_SWEEP_SYM", 1) != 0 && memcmp(&x.A0[0], &x.A0[2], 2 * sizeof(double)) == 0 &&
           memcmp(&x.A0[4], &x.A0[6], 2 * sizeof(double)) == 0 && c4g_finite;
}

int yaman4_sweep_launch(const fpa_sweep_desc* d, void* scratch, int64_t scratch_bytes, cudaStream_t st) {
    Yaman4Params p;
    SweepExtra   x;
    int64_t      n_grid;
    int rc = sweep_setup(d, 1, p, x, n_grid);
    if (rc != FPA_OK || n_grid == 0) return rc;
    if (sweep_symmetric(p, x)) return sweep_run<SweepExtra, true>(p, x, scratch, scratch_bytes, st);
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
    FPA_REQUIRE_ALIGNED16(d->A0_table, "A0_table");  // read with 16-byte loads (sweep_initial_state)
    const int64_t K = d->n_phases;
    rc = sweep_setup(&d->sweep, K, p, x, n_grid);
    if (rc != FPA_OK || n_grid == 0) return rc;
    x.A0_table   = d->A0_table;
    x.n_phases   = K;
    x.last_saved = d->metric == FPA_GAIN_LAST_SAVED ? 1 : 0;
    return sweep_run(p, x, scratch, scratch_bytes, st);
}

// ---- small-signal transfer matrices
// The column mask and jac of a transfer output (the kernels store jac with 8-byte stores).
static int transfer_params(const fpa_transfer_out* t, TransferParams& tp) {
    FPA_REQUIRE(t != nullptr, "transfer output is NULL");
    FPA_REQUIRE(t->columns != 0 && (t->columns >> 8) == 0, "columns must be a non-zero mask of bits 0..7 (got %#x)",
                t->columns);
    FPA_REQUIRE(t->jac != nullptr, "jac must be set");
    FPA_REQUIRE_ALIGNED8(t->jac, "jac");
    tp.jac  = t->jac;
    tp.nc   = 0;
    tp.cols = 0;
    for (uint32_t c = 0; c < 8; ++c) {
        if ((t->columns >> c) & 1u) {
            tp.cols |= c << (4 * tp.nc);
            ++tp.nc;
        }
    }
    return FPA_OK;
}

// The checks of a batch transfer, for the device and the host entries alike: the batch descriptor's, the transfer
// output's, and the paths the tangent kernels do not cover (FPA_ERR_UNSUPPORTED).
int yaman4_transfer_check(const fpa_yaman4_desc* d, const fpa_transfer_out* t) {
    if (d && ((d->flags & (FPA_OUT_TRACE | FPA_PHASE_EXACT)) || d->z_grid)) {
        set_error("transfer matrices follow the uniform-grid fast integrator: FPA_OUT_TRACE, z_grid and "
                  "FPA_PHASE_EXACT are not available");
        return FPA_ERR_UNSUPPORTED;
    }
    int rc = yaman4_check(d);
    if (rc != FPA_OK) return rc;
    TransferParams tp;
    return transfer_params(t, tp);
}

int yaman4_transfer_launch(const fpa_yaman4_desc* d, const fpa_transfer_out* t, cudaStream_t st) {
    int rc = yaman4_transfer_check(d, t);
    if (rc != FPA_OK) return rc;
    const bool uniform = (d->flags & FPA_UNIFORM_PHYSICS) != 0;
    FPA_REQUIRE(!uniform || (d->gamma_stride == 0 && d->alpha_stride == 0),
                "FPA_UNIFORM_PHYSICS needs broadcast gamma and alpha (stride 0)");
    FPA_REQUIRE_ALIGNED16(d->A0, "A0");
    if (d->flags & FPA_OUT_END) FPA_REQUIRE_ALIGNED16(d->A_end, "A_end");
    if (d->flags & FPA_OUT_PMAX) FPA_REQUIRE_ALIGNED16(d->Pmax, "Pmax");
    if (d->n_points == 0) return FPA_OK;
    Yaman4Params   p;
    TransferParams tp;
    batch_params(d, uniform, p);
    transfer_params(t, tp);
    const BatchPoints x{};
    const long        blocks = (long)((p.n_points * tp.nc + kTransferThreads - 1) / kTransferThreads);
    if (!uniform)
        yaman4_transfer_kernel<0><<<blocks, kTransferThreads, 0, st>>>(p, x, tp);
    else if (p.lossless)
        yaman4_transfer_kernel<2><<<blocks, kTransferThreads, 0, st>>>(p, x, tp);
    else
        yaman4_transfer_kernel<1><<<blocks, kTransferThreads, 0, st>>>(p, x, tp);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "yaman4_transfer_kernel launch");
    return FPA_OK;
}

int yaman4_transfer_sweep_launch(const fpa_sweep_desc* d, const fpa_transfer_out* t, cudaStream_t st) {
    Yaman4Params   p;
    SweepExtra     x;
    TransferParams tp;
    int64_t        n_grid;
    if (d && (d->flags & FPA_PHASE_EXACT)) return sweep_setup(d, 1, p, x, n_grid);  // FPA_ERR_UNSUPPORTED
    FPA_REQUIRE(d != nullptr, "sweep descriptor is NULL");
    FPA_REQUIRE(d->n_peers == 0, "the transfer sweep has no peer-store gather: n_peers must be 0");
    int rc = transfer_params(t, tp);
    if (rc != FPA_OK) return rc;
    rc = sweep_setup(d, 1, p, x, n_grid, true);
    if (rc != FPA_OK || n_grid == 0) return rc;
    const long blocks = (long)((p.n_points * tp.nc + kTransferThreads - 1) / kTransferThreads);
    if (p.lossless)
        yaman4_transfer_kernel<2><<<blocks, kTransferThreads, 0, st>>>(p, x, tp);
    else
        yaman4_transfer_kernel<1><<<blocks, kTransferThreads, 0, st>>>(p, x, tp);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "yaman4_transfer_kernel launch");
    return FPA_OK;
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
