// nwave.cu -- N-wave generalisation of the fused RK4 x FWM integrator (NOT in the reference).
//
//   dA_n/dz = -(alpha/2) A_n + i*gamma * [ (2*sum_j P_j - P_n) A_n
//               + conj(E_n) * sum_{e in row n} D_e * At_k At_l conj(At_m) ],   At_j = A_j E_j,
//   E_j = exp(i*beta_j*z)
// which is the reference's 4-wave system (yaman_model.py:22-25, :135-186) for the fixed table
// {0:(2,3;1) 1:(2,3;0) 2:(0,1;3) 3:(0,1;2)}, weight 2 and beta = [0,0,0,dbeta].
//
// Mapping: one CTA per scan point (a single warp when the plan is small).  The point's complex
// amplitudes, its per-wave phase table and -- when it fits -- the frequency plan's triplet
// index/weight list live in shared memory for all z-steps; each warp owns rows n = w, w+W, ...
// of the triplet sum, lanes stride over the row's entries and the partial sums are combined
// with warp shuffles.  The four RK4 stages are fused: nothing goes to HBM between stages.
//
// The triplet enumerator (integer-grid matching, canonical order n,k,l,m) is host code in this
// file as well; tests compare it bit-for-bit with the Python restatement in oracle/.
#include "fpa_common.cuh"

#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <map>
#include <vector>

// compute-sanitizer is not available on the B200 pool: -DFPA_BOUNDS_CHECK checks every index the factored-table
// kernel takes from its blob (device assert); tools/bounds_check.py builds that variant and runs the shapes.
#ifdef FPA_BOUNDS_CHECK
#include <assert.h>
#define FPA_IN_RANGE(idx, n) assert((long long)(idx) >= 0 && (long long)(idx) < (long long)(n))
#else
#define FPA_IN_RANGE(idx, n) ((void)0)
#endif

namespace fpa {

struct NwaveParams {
    int64_t            n_points;
    int                n_waves;
    int                beta_stride, gamma_stride, alpha_stride, A0_stride;
    const double*      beta;
    const double*      gamma;
    const double*      alpha;
    const double*      A0;
    const fpa_triplet* triplets;
    const int64_t*     row_ptr;
    int64_t            n_triplets;
    int                table_in_smem;
    int                table_in_smem_only_one_cta;
    double             z0, z_max;
    int                n_steps, save_every;
    int64_t            n_saved;
    const double*      z_grid;
    double*            A_trace;
    double*            A_end;
    double*            Pmax;
    int32_t*           status;
    int                check;
    const unsigned char* fact;        // factored table (FactHeader + arrays, see below) or NULL
    int                n_classes;
};

// Factored form of a triplet table (host: fpa_nwave_factor_table below).  The entries of row n are grouped by
// their conjugated wave m; the (k, l, weight) list of a group is a CLASS, and groups with the same list share it:
//   R_n = sum_m conj(At_m) * T_{c(n,m)} - At_n * sum_m w_own(n,m) P_m,     T_c = sum_{(k,l,w) in c} w At_k At_l.
// For a table that came from a frequency plan every group of the same sum frequency w_n + w_m holds the same
// pairs except its own {n, m} (the enumerator's "m not in {k, l}"), so the factoriser may add that pair to the
// group (weight 1 for n == m, else 2) and take it out again through w_own -- then N = 64 has 127 classes with
// 2 080 pairs in all and 4 096 (n, m) cells instead of 84 320 entries.  Any table factors (worst case one class
// per cell); nothing about the plan is assumed.  Modes: 0 no own pairs (w_own = 0); 1 own pairs where a group
// has entries, w_own matrix; 2 own pairs in EVERY cell, so sum_m w_own P_m = 2 S - P_n needs no matrix.
//
// Layout for the kernel: pair records {k*16, l*16, weight}, classes in order of falling size (lanes that work side
// by side get lists of similar length) with every class padded to a multiple of 4 (weight 0); cls[c] = {first
// pair, byte offset of the class sum's slot in T} -- the slots are numbered in order of first appearance in the
// cell map, which for a comb is the order of the sum frequency, so the lanes of a row read neighbouring slots;
// the cell map holds for every row n the byte offsets into T of its N_pad = 2^np_log cells (empty and padding
// cells point at a zero slot T[C]) in BIT-REVERSED order of m: the cells m = r (mod L) are then contiguous for
// every power of two L, so whatever number of lanes shares a row, each lane reads its cells with 16-byte loads.
struct FactHeader {
    uint32_t magic;
    int32_t  n_waves, n_classes, n_pairs, mode, np_log, reserved;
    int32_t  off_cls, off_pairs, off_cmap, off_wown;   // bytes from the start of the blob
    int32_t  bytes;
};
struct FactPair {
    uint16_t k16, l16;   // byte offsets of At_k, At_l (index * 16)
    float    w;
};
constexpr uint32_t kFactMagic   = 0x33504146u;   // "FAP3"
constexpr int      kFactMaxCls  = 1 << 20;

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Shared-memory layout (doubles): y[2N] ys[2N] yn[2N] At[2N] E[2N] beta[N] P[N] red[34] | rows[N+1] | table
struct Smem {
    double *y, *ys, *yn, *At, *E, *beta, *P, *red;
    int*                rows;
    const fpa_triplet*  table;
    double2*            T;      // factored form: class sums, in place of rows | table
};

__device__ __forceinline__ Smem carve(double* base, int N, const NwaveParams& p) {
    Smem s;
    s.y    = base;
    s.ys   = s.y + 2 * N;
    s.yn   = s.ys + 2 * N;
    s.At   = s.yn + 2 * N;
    s.E    = s.At + 2 * N;
    s.beta = s.E + 2 * N;
    s.P    = s.beta + N;
    s.red  = s.P + N;
    s.rows = reinterpret_cast<int*>(s.red + 34);
    s.T    = reinterpret_cast<double2*>(s.red + 34);
    // table is 8-byte aligned: (N+1) ints rounded up to an even count
    s.table = reinterpret_cast<const fpa_triplet*>(s.rows + ((N + 2) & ~1));
    return s;
}

// One RHS evaluation at abscissa z on stage state s.ys; afterwards, for every wave n, the row owner
// applies   yn_n += wa*k_n   and   ys_n = y_n + wb*k_n   (or y_n = yn_n + wa*k_n when `last`).
// Returns S = sum |ys|^2 (used by the finite check).
__device__ double rhs_stage(const Smem& s, const NwaveParams& p, const fpa_triplet* __restrict__ table,
                            double z, double gamma, double nha, double wa, double wb, bool last) {
    const int N = p.n_waves;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;

    // phases, rotated amplitudes, powers
    double part = 0.0;
    for (int j = tid; j < N; j += blockDim.x) {
        double sn, cs;
        sincos(s.beta[j] * z, &sn, &cs);
        const double xr = s.ys[2 * j], xi = s.ys[2 * j + 1];
        s.E[2 * j]      = cs;
        s.E[2 * j + 1]  = sn;
        s.At[2 * j]     = fma(-xi, sn, xr * cs);
        s.At[2 * j + 1] = fma(xr, sn, xi * cs);
        const double P  = fma(xi, xi, xr * xr);
        s.P[j] = P;
        part += P;
    }
    part = warp_sum(part);
    if (lane == 0) s.red[warp] = part;
    __syncthreads();
    double S = 0.0;
    for (int w = 0; w < nwarps; ++w) S += s.red[w];

    // triplet sums, one warp per row
    for (int n = warp; n < N; n += nwarps) {
        const int e0 = s.rows[n], e1 = s.rows[n + 1];
        double rr = 0.0, ri = 0.0;
        // one entry: D * At_k At_l conj(At_m)
        auto term = [&](const fpa_triplet t, double& ar, double& ai) {
            const double kr = s.At[2 * t.k], ki = s.At[2 * t.k + 1];
            const double lr = s.At[2 * t.l], li = s.At[2 * t.l + 1];
            const double mr = s.At[2 * t.m], mi = s.At[2 * t.m + 1];
            const double w  = (double)t.weight;
            const double qr = w * fma(-ki, li, kr * lr);
            const double qi = w * fma(kr, li, ki * lr);
            ar = fma(qr, mr, fma(qi, mi, ar));   // q * conj(m)
            ai = fma(qi, mr, fma(-qr, mi, ai));
        };
        // A table that does not fit into shared memory streams from L2 (N = 64: 674 KB per RHS and scan point):
        // four entries per lane are requested before the first one is used, and two accumulator pairs keep the
        // FMA chains apart -- the rolled loop ran at the latency of one load per entry (~800 cycles).
        double r2 = 0.0, i2 = 0.0;
        int    e = e0 + lane;
        for (; e + 96 < e1; e += 128) {
            const fpa_triplet t0 = table[e], t1 = table[e + 32], t2 = table[e + 64], t3 = table[e + 96];
            term(t0, rr, ri);
            term(t1, r2, i2);
            term(t2, rr, ri);
            term(t3, r2, i2);
        }
        for (; e < e1; e += 32) term(table[e], rr, ri);
        rr += r2;
        ri += i2;
        rr = warp_sum(rr);
        ri = warp_sum(ri);
        if (lane == 0) {
            const double xr = s.ys[2 * n], xi = s.ys[2 * n + 1];
            const double er = s.E[2 * n], ei = s.E[2 * n + 1];
            // F = conj(E_n) * R
            const double fr = fma(ri, ei, rr * er);
            const double fi = fma(ri, er, -(rr * ei));
            const double G  = gamma * ((S + S) - s.P[n]);
            // k = nha*x + i*(G*x + gamma*F)
            const double kr = fma(nha, xr, -fma(G, xi, gamma * fi));
            const double ki = fma(nha, xi, fma(G, xr, gamma * fr));
            if (last) {
                s.y[2 * n]     = fma(wa, kr, s.yn[2 * n]);
                s.y[2 * n + 1] = fma(wa, ki, s.yn[2 * n + 1]);
            } else {
                const double a = s.y[2 * n], bq = s.y[2 * n + 1];
                // first stage starts the accumulator from y (wb == 0 marks "yn not yet initialised")
                s.yn[2 * n]     = fma(wa, kr, s.yn[2 * n]);
                s.yn[2 * n + 1] = fma(wa, ki, s.yn[2 * n + 1]);
                s.ys[2 * n]     = fma(wb, kr, a);
                s.ys[2 * n + 1] = fma(wb, ki, bq);
            }
        }
    }
    __syncthreads();
    return S;
}

#ifdef FPA_FACT_TIMING   // tools/fact_phase_timing.py: thread 0 of point 0 accumulates clock64() between the phases
__shared__ long long g_fact_ticks[12];
#define FPA_FTICK(k)                                        \
    do {                                                    \
        if (threadIdx.x == 0) {                             \
            const long long t_now = clock64();              \
            g_fact_ticks[k] += t_now - t_last;              \
            t_last = t_now;                                 \
        }                                                   \
    } while (0)
#else
#define FPA_FTICK(k)
#endif

struct FactView {
    const int2*     cls;
    const FactPair* pairs;
    const uint32_t* cmap;
    const int16_t*  wown;
    int             C, mode, np_log, lpr_log, lpc_log, ok;
};

__device__ __forceinline__ FactView fact_view(const NwaveParams& p) {
    const FactHeader* h = reinterpret_cast<const FactHeader*>(p.fact);
    FactView          f;
    f.ok     = h->magic == kFactMagic && h->n_waves == p.n_waves && h->n_classes == p.n_classes;
    f.cls    = reinterpret_cast<const int2*>(p.fact + h->off_cls);
    f.pairs  = reinterpret_cast<const FactPair*>(p.fact + h->off_pairs);
    f.cmap   = reinterpret_cast<const uint32_t*>(p.fact + h->off_cmap);
    f.wown   = reinterpret_cast<const int16_t*>(p.fact + h->off_wown);
    f.C      = h->n_classes;
    f.mode   = h->mode;
    f.np_log = h->np_log;
    // lanes per row: as many as the CTA has for N_pad rows, at least four cells per lane (one 16-byte load)
    const int t_log = 31 - __clz((int)blockDim.x);
    f.lpr_log = max(0, min(min(5, f.np_log - 2), t_log - f.np_log));
    // lanes per class: 4, more when the CTA has lanes to spare for all classes at once (8 lanes per class make the
    // operand loads of a quarter-warp conflict-free -- one class, neighbouring words -- but cost a shuffle level and
    // a second pass over the classes: measured 6 % slower at N = 64)
    f.lpc_log = 2;
    while (f.lpc_log < 5 && (f.C << (f.lpc_log + 1)) <= (int)blockDim.x) ++f.lpc_log;
    return f;
}

// The same stage as rhs_stage through the factored table: class sums with 4 lanes per class, then the rows with
// lpr lanes per row.  Phases are the exact sincos of rhs_stage.
__device__ double fact_stage(const Smem& s, const NwaveParams& p, const FactView& f, double z, double gamma,
                             double nha, double wa, double wb, bool last) {
    const int N = p.n_waves;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const double2*       At2 = reinterpret_cast<const double2*>(s.At);
    const unsigned char* Atb = reinterpret_cast<const unsigned char*>(s.At);
    const unsigned char* Tb  = reinterpret_cast<const unsigned char*>(s.T);
#ifdef FPA_FACT_TIMING
    long long t_last = clock64(), t_sub = 0;
#define FPA_FSUB0() do { if (threadIdx.x == 0) t_sub = clock64(); } while (0)
#define FPA_FSUB(k, dep) do { if (threadIdx.x == 0 && (dep) == (dep)) { const long long t_n = clock64(); g_fact_ticks[k] += t_n - t_sub; t_sub = t_n; } } while (0)
#else
#define FPA_FSUB0()
#define FPA_FSUB(k, dep)
#endif

    double part = 0.0;
    for (int j = tid; j < N; j += blockDim.x) {
        double sn, cs;
        sincos(s.beta[j] * z, &sn, &cs);
        const double xr = s.ys[2 * j], xi = s.ys[2 * j + 1];
        s.E[2 * j]      = cs;
        s.E[2 * j + 1]  = sn;
        s.At[2 * j]     = fma(-xi, sn, xr * cs);
        s.At[2 * j + 1] = fma(xr, sn, xi * cs);
        const double P  = fma(xi, xi, xr * xr);
        s.P[j] = P;
        part += P;
    }
    FPA_FTICK(0);
    part = warp_sum(part);
    if (lane == 0) s.red[warp] = part;
    __syncthreads();
    FPA_FTICK(1);
    const int nw_sum = min(nwarps, (N + 31) >> 5);      // the warps that had waves to rotate
    double    S = 0.0, S1 = 0.0;
    for (int w = 0; w + 1 < nw_sum; w += 2) {
        S += s.red[w];
        S1 += s.red[w + 1];
    }
    if (nw_sum & 1) S += s.red[nw_sum - 1];
    S += S1;

    // class sums T_c: lpc lanes per class, two pairs of a lane in flight
    const int lpc_log = f.lpc_log, lpc = 1 << lpc_log, csub = tid & (lpc - 1);
    auto      pair_term = [&](const uint2 u, double& qr, double& qi) {
        FPA_IN_RANGE(u.x & 0xFFFFu, 16 * N);
        FPA_IN_RANGE(u.x >> 16, 16 * N);
        const double2 a = *reinterpret_cast<const double2*>(Atb + (u.x & 0xFFFFu));
        const double2 b = *reinterpret_cast<const double2*>(Atb + (u.x >> 16));
        const double  w = (double)__uint_as_float(u.y);
        const double  pr = fma(-a.y, b.y, a.x * b.x);
        const double  pi = fma(a.x, b.y, a.y * b.x);
        qr = fma(w, pr, qr);
        qi = fma(w, pi, qi);
    };
    for (int base = 0; base < f.C; base += (int)(blockDim.x >> lpc_log)) {
        const int c = base + (tid >> lpc_log);
        double    qr = 0.0, qi = 0.0, q2 = 0.0, j2 = 0.0;
        int       slot = 0;
        FPA_FSUB0();
        if (c < f.C) {
            const uint2* pp = reinterpret_cast<const uint2*>(f.pairs);
            const int2   c0 = __ldg(f.cls + c);
            const int    e1 = __ldg(f.cls + c + 1).x;
            int          e = c0.x + csub;
            slot           = c0.y;
            FPA_IN_RANGE(slot, 16 * f.C);
            FPA_IN_RANGE(c0.x, e1 + 1);
            for (; e + lpc < e1; e += 2 * lpc) {
                const uint2 u0 = __ldg(pp + e), u1 = __ldg(pp + e + lpc);
                pair_term(u0, qr, qi);
                pair_term(u1, q2, j2);
            }
            if (e < e1) pair_term(__ldg(pp + e), qr, qi);
            qr += q2;
            qi += j2;
        }
        FPA_FSUB(6, qr + qi);
        for (int o = lpc >> 1; o > 0; o >>= 1) {
            qr += __shfl_xor_sync(0xffffffffu, qr, o);
            qi += __shfl_xor_sync(0xffffffffu, qi, o);
        }
        FPA_FSUB(7, qr + qi);
        if (c < f.C && csub == 0) *reinterpret_cast<double2*>(const_cast<unsigned char*>(Tb) + slot) = make_double2(qr, qi);
        FPA_FSUB(8, 0.0);
    }
    FPA_FTICK(2);
    __syncthreads();
    FPA_FTICK(3);

    // rows: lpr lanes per row; a lane's cells are one contiguous run of the bit-reversed map, four per 16-byte
    // load; cells beyond N point at the zero slot (their At index is clamped), so the body has no branches and its
    // eight shared-memory loads go out together
    const int lpr_log = f.lpr_log, lpr = 1 << lpr_log, rsub = tid & (lpr - 1);
    const int cpl = 1 << (f.np_log - lpr_log), rev_shift = 32 - f.np_log;
    for (int base = 0; base < N; base += (int)(blockDim.x >> lpr_log)) {
        const int n = base + (tid >> lpr_log);
        double    rr = 0.0, ri = 0.0, r2 = 0.0, i2 = 0.0, r3 = 0.0, i3 = 0.0, r4 = 0.0, i4 = 0.0, cw = 0.0;
        FPA_FSUB0();
        if (n < N) {
            const int    q0 = rsub * cpl;
            const uint4* cm = reinterpret_cast<const uint4*>(f.cmap + ((size_t)n << f.np_log) + q0);
            auto         wave_of = [&](int q) { return min((int)(__brev((unsigned)q) >> rev_shift), N - 1); };
            if (cpl >= 4) {
                uint4 o = __ldg(cm);
                for (int i = 0; i < cpl; i += 4) {
                    const uint4   on = __ldg(cm + (i + 4 < cpl ? (i >> 2) + 1 : 0));
                    FPA_IN_RANGE(o.x, 16 * (f.C + 1));
                    FPA_IN_RANGE(o.y, 16 * (f.C + 1));
                    FPA_IN_RANGE(o.z, 16 * (f.C + 1));
                    FPA_IN_RANGE(o.w, 16 * (f.C + 1));
                    FPA_IN_RANGE(q0 + i + 3, 1 << f.np_log);
                    const double2 t0 = *reinterpret_cast<const double2*>(Tb + o.x);
                    const double2 t1 = *reinterpret_cast<const double2*>(Tb + o.y);
                    const double2 t2 = *reinterpret_cast<const double2*>(Tb + o.z);
                    const double2 t3 = *reinterpret_cast<const double2*>(Tb + o.w);
                    const double2 b0 = At2[wave_of(q0 + i)], b1 = At2[wave_of(q0 + i + 1)];
                    const double2 b2 = At2[wave_of(q0 + i + 2)], b3 = At2[wave_of(q0 + i + 3)];
                    rr = fma(t0.x, b0.x, fma(t0.y, b0.y, rr));   // T * conj(At_m)
                    ri = fma(t0.y, b0.x, fma(-t0.x, b0.y, ri));
                    r2 = fma(t1.x, b1.x, fma(t1.y, b1.y, r2));
                    i2 = fma(t1.y, b1.x, fma(-t1.x, b1.y, i2));
                    r3 = fma(t2.x, b2.x, fma(t2.y, b2.y, r3));
                    i3 = fma(t2.y, b2.x, fma(-t2.x, b2.y, i3));
                    r4 = fma(t3.x, b3.x, fma(t3.y, b3.y, r4));
                    i4 = fma(t3.y, b3.x, fma(-t3.x, b3.y, i4));
                    o = on;
                }
            } else {      // N_pad < 4: one lane, one to two cells
                for (int i = 0; i < cpl; ++i) {
                    const double2 t0 = *reinterpret_cast<const double2*>(Tb + __ldg(f.cmap + ((size_t)n << f.np_log) + q0 + i));
                    const double2 b0 = At2[wave_of(q0 + i)];
                    rr = fma(t0.x, b0.x, fma(t0.y, b0.y, rr));
                    ri = fma(t0.y, b0.x, fma(-t0.x, b0.y, ri));
                }
            }
            rr = (rr + r2) + (r3 + r4);
            ri = (ri + i2) + (i3 + i4);
            if (f.mode == 1) {
                const int16_t* wo = f.wown + n * N;
                for (int m = rsub; m < N; m += lpr) cw = fma((double)__ldg(wo + m), s.P[m], cw);
            }
        }
        FPA_FSUB(9, rr + ri);
        for (int o = lpr >> 1; o > 0; o >>= 1) {
            rr += __shfl_xor_sync(0xffffffffu, rr, o);
            ri += __shfl_xor_sync(0xffffffffu, ri, o);
            if (f.mode == 1) cw += __shfl_xor_sync(0xffffffffu, cw, o);
        }
        FPA_FSUB(10, rr + ri);
        if (n < N && rsub == 0) {
            const double xr = s.ys[2 * n], xi = s.ys[2 * n + 1];
            const double er = s.E[2 * n], ei = s.E[2 * n + 1];
            // the own pairs the factoriser added come out again: R -= At_n * sum_m w_own P_m
            if (f.mode == 2) cw = (S + S) - s.P[n];
            rr = fma(-cw, s.At[2 * n], rr);
            ri = fma(-cw, s.At[2 * n + 1], ri);
            const double fr = fma(ri, ei, rr * er);
            const double fi = fma(ri, er, -(rr * ei));
            const double G  = gamma * ((S + S) - s.P[n]);
            const double kr = fma(nha, xr, -fma(G, xi, gamma * fi));
            const double ki = fma(nha, xi, fma(G, xr, gamma * fr));
            if (last) {
                s.y[2 * n]     = fma(wa, kr, s.yn[2 * n]);
                s.y[2 * n + 1] = fma(wa, ki, s.yn[2 * n + 1]);
            } else {
                const double a = s.y[2 * n], bq = s.y[2 * n + 1];
                s.yn[2 * n]     = fma(wa, kr, s.yn[2 * n]);
                s.yn[2 * n + 1] = fma(wa, ki, s.yn[2 * n + 1]);
                s.ys[2 * n]     = fma(wb, kr, a);
                s.ys[2 * n + 1] = fma(wb, ki, bq);
            }
        }
        FPA_FSUB(11, 0.0);
    }
    FPA_FTICK(4);
    __syncthreads();
    FPA_FTICK(5);
    return S;
}

template <bool FACT>
__global__ void __launch_bounds__(1024) nwave_rk4_kernel(const NwaveParams p) {
    extern __shared__ double smem_raw[];
    const int     N = p.n_waves;
    const int64_t b = blockIdx.x;
    const int     tid = threadIdx.x;
    Smem          s = carve(smem_raw, N, p);

    const double gamma = p.gamma[b * p.gamma_stride];
    const double nha   = -0.5 * p.alpha[b * p.alpha_stride];

    for (int j = tid; j < N; j += blockDim.x) {
        s.beta[j] = p.beta[b * p.beta_stride * N + j];
        const double re = p.A0[(b * p.A0_stride * N + j) * 2];
        const double im = p.A0[(b * p.A0_stride * N + j) * 2 + 1];
        s.y[2 * j] = re;
        s.y[2 * j + 1] = im;
    }
    const fpa_triplet* table = p.triplets;
    FactView           fv = {};
    if (FACT) {
        fv = fact_view(p);
        if (fv.ok && tid == 0) s.T[fv.C] = make_double2(0.0, 0.0);   // the slot empty cells point at
#ifdef FPA_FACT_TIMING
        if (tid < 12) g_fact_ticks[tid] = 0;
#endif
    } else {
        for (int j = tid; j <= N; j += blockDim.x) s.rows[j] = (int)p.row_ptr[j];
        if (p.table_in_smem) {
            fpa_triplet* dst = const_cast<fpa_triplet*>(s.table);
            for (int64_t e = tid; e < p.n_triplets; e += blockDim.x) dst[e] = p.triplets[e];
            table = s.table;
        }
    }
    __syncthreads();
    if (FACT && !fv.ok) {   // not the blob of this plan: no result rather than a wrong one
        if (p.status && tid == 0) p.status[b] = 0;
        if (p.A_end)
            for (int j = tid; j < 2 * N; j += blockDim.x) p.A_end[b * 2 * N + j] = qnan();
        if (p.Pmax)
            for (int j = tid; j < N; j += blockDim.x) p.Pmax[b * N + j] = qnan();
        return;
    }
    auto stage = [&](double z, double wa, double wb, bool last) {
        return FACT ? fact_stage(s, p, fv, z, gamma, nha, wa, wb, last)
                    : rhs_stage(s, p, table, z, gamma, nha, wa, wb, last);
    };

    double* tr = p.A_trace ? p.A_trace + b * p.n_saved * 2 * N : nullptr;
    if (tr) {
        for (int j = tid; j < 2 * N; j += blockDim.x) tr[j] = s.y[j];
        tr += 2 * N;
    }
    // per-thread running max for the waves this thread owns (j = tid, tid+blockDim, ...): at most
    // ceil(128/32) = 4 waves per thread
    double pm[4] = {0.0, 0.0, 0.0, 0.0};
    if (p.Pmax) {
        int q = 0;
        for (int j = tid; j < N; j += blockDim.x, ++q) pm[q] = fma(s.y[2 * j + 1], s.y[2 * j + 1], s.y[2 * j] * s.y[2 * j]);
    }

    const int    n_steps = p.n_steps;
    const double z0 = p.z0, z_max = p.z_max;
    const double step = (z_max - z0) / (double)n_steps;
    double       zi = p.z_grid ? p.z_grid[0] : z0;
    double       di = 0.0;
    int          save_ctr = p.save_every;
    int32_t      bad = FPA_POINT_OK;

    for (int i = 0; i < n_steps; ++i) {
        double zn;
        if (p.z_grid) {
            zn = p.z_grid[i + 1];
        } else {
            di += 1.0;
            zn = (i + 1 == n_steps) ? z_max : __dadd_rn(__dmul_rn(di, step), z0);
        }
        const double h = zn - zi, hh = 0.5 * h, h6 = h / 6.0, h3 = h6 + h6;

        // stage state and accumulator start from y
        for (int j = tid; j < 2 * N; j += blockDim.x) {
            const double v = s.y[j];
            s.ys[j] = v;
            s.yn[j] = v;
        }
        __syncthreads();

        const double S = stage(zi, h6, hh, false);
        if (p.check && i > 0 && bad == FPA_POINT_OK && nonfinite(S)) {
            int nf = 0;
            for (int j = tid; j < 2 * N; j += blockDim.x) nf |= nonfinite(s.y[j]) ? 1 : 0;
            if (__syncthreads_or(nf)) bad = i - 1;
        }
        stage(zi + hh, h3, hh, false);
        stage(zi + hh, h3, h, false);
        stage(zi + h, h6, 0.0, true);
        zi = zn;

        if (--save_ctr == 0) {
            save_ctr = p.save_every;
            if (tr) {
                for (int j = tid; j < 2 * N; j += blockDim.x) tr[j] = s.y[j];
                tr += 2 * N;
            }
            if (p.Pmax) {
                int q = 0;
                for (int j = tid; j < N; j += blockDim.x, ++q) {
                    const double P = fma(s.y[2 * j + 1], s.y[2 * j + 1], s.y[2 * j] * s.y[2 * j]);
                    pm[q] = (P != P || pm[q] != pm[q]) ? qnan() : fmax(pm[q], P);
                }
            }
        }
    }

    if (p.check && bad == FPA_POINT_OK) {
        int nf = 0;
        for (int j = tid; j < 2 * N; j += blockDim.x) nf |= nonfinite(s.y[j]) ? 1 : 0;
        if (__syncthreads_or(nf)) bad = n_steps - 1;
    }
    if (p.status && tid == 0) p.status[b] = bad;
#ifdef FPA_FACT_TIMING
    if (FACT && b == 0 && tid == 0) {
        const double per = 1.0 / (4.0 * n_steps);
        printf("fact stage cycles (thread 0 of point 0, per stage): phases %.0f | sum+sync %.0f | classes %.0f | sync %.0f | rows %.0f | sync %.0f"
               " || classes: loads+products %.0f, shuffles %.0f, store %.0f || rows: cells %.0f, shuffles %.0f, owner %.0f\n",
               g_fact_ticks[0] * per, g_fact_ticks[1] * per, g_fact_ticks[2] * per, g_fact_ticks[3] * per,
               g_fact_ticks[4] * per, g_fact_ticks[5] * per, g_fact_ticks[6] * per, g_fact_ticks[7] * per,
               g_fact_ticks[8] * per, g_fact_ticks[9] * per, g_fact_ticks[10] * per, g_fact_ticks[11] * per);
    }
#endif
    if (p.A_end)
        for (int j = tid; j < 2 * N; j += blockDim.x) p.A_end[b * 2 * N + j] = s.y[j];
    if (p.Pmax) {
        int q = 0;
        for (int j = tid; j < N; j += blockDim.x, ++q) p.Pmax[b * N + j] = pm[q];
    }
}

static size_t nwave_smem_bytes(int N, int64_t n_table_entries) {
    size_t doubles = (size_t)(5 * 2 * N + 2 * N + 34);
    size_t bytes   = doubles * sizeof(double) + (size_t)((N + 2) & ~1) * sizeof(int);
    return bytes + (size_t)n_table_entries * sizeof(fpa_triplet);
}

// The checks of an N-wave descriptor that the table kernel and the comb kernel share, for the device and the host
// entries alike.  Each launcher adds its kernel's own limits.
int nwave_check(const fpa_nwave_desc* d) {
    FPA_REQUIRE(d != nullptr, "descriptor is NULL");
    FPA_REQUIRE(d->n_points >= 0, "n_points must be >= 0");
    FPA_REQUIRE(d->n_waves >= 1, "n_waves must be >= 1");
    FPA_REQUIRE(d->n_steps >= 1 && d->n_steps < 2147483647LL, "n_steps must be in [1, 2^31)");
    FPA_REQUIRE(d->save_every >= 1, "save_every must be a positive integer");
    FPA_REQUIRE(d->beta && d->gamma && d->alpha && d->A0, "beta/gamma/alpha/A0 must be set");
    FPA_REQUIRE((d->gamma_stride | 1) == 1 && (d->alpha_stride | 1) == 1 && (d->A0_stride | 1) == 1 &&
                    (d->beta_stride | 1) == 1,
                "strides must be 0 (broadcast) or 1 (per point)");
    FPA_REQUIRE(!(d->flags & FPA_OUT_TRACE) || d->A_trace, "FPA_OUT_TRACE needs A_trace");
    FPA_REQUIRE(!(d->flags & FPA_OUT_PMAX) || d->Pmax, "FPA_OUT_PMAX needs Pmax");
    FPA_REQUIRE(!(d->flags & FPA_OUT_END) || d->A_end, "FPA_OUT_END needs A_end");
    return FPA_OK;
}

int nwave_launch(const fpa_nwave_desc* d, cudaStream_t st) {
    int rc = nwave_check(d);
    if (rc != FPA_OK) return rc;
    if (d->n_waves > 128) {
        set_error("n_waves = %d exceeds the kernel limit of 128", d->n_waves);
        return FPA_ERR_UNSUPPORTED;
    }
    // the factored form of the table (fpa_nwave_factor_table) replaces the entry list when the caller supplies it
    const bool fact = d->factored != nullptr && !(d->flags & FPA_NWAVE_PLAIN) && getenv("FPA_NWAVE_PLAIN") == nullptr;
    if (fact) {
        FPA_REQUIRE(d->n_classes >= 0 && d->n_classes < kFactMaxCls, "n_classes must be the class count of `factored`");
    } else {
        FPA_REQUIRE(d->n_triplets >= 0 && d->n_triplets < 2147483647LL, "bad n_triplets");
        FPA_REQUIRE(d->row_ptr != nullptr, "row_ptr must be set");
        FPA_REQUIRE(d->n_triplets == 0 || d->triplets, "triplets must be set");
    }
    const bool trace = (d->flags & FPA_OUT_TRACE) != 0;
    const bool pmax  = (d->flags & FPA_OUT_PMAX) != 0;
    const bool endo  = (d->flags & FPA_OUT_END) != 0;
    if (d->n_points == 0) return FPA_OK;

    NwaveParams p;
    p.n_points     = d->n_points;
    p.n_waves      = d->n_waves;
    p.beta_stride  = (int)d->beta_stride;
    p.gamma_stride = (int)d->gamma_stride;
    p.alpha_stride = (int)d->alpha_stride;
    p.A0_stride    = (int)d->A0_stride;
    p.beta         = d->beta;
    p.gamma        = d->gamma;
    p.alpha        = d->alpha;
    p.A0           = d->A0;
    p.triplets     = d->triplets;
    p.row_ptr      = d->row_ptr;
    p.n_triplets   = d->n_triplets;
    p.z0           = d->z0;
    p.z_max        = d->z_max;
    p.n_steps      = (int)d->n_steps;
    p.save_every   = (int)(d->save_every > d->n_steps ? d->n_steps + 1 : d->save_every);
    p.n_saved      = fpa_n_saved(d->n_steps, d->save_every);
    p.z_grid       = nullptr;  // the C ABI exposes linspace grids only for the N-wave model
    p.A_trace      = trace ? d->A_trace : nullptr;
    p.A_end        = endo ? d->A_end : nullptr;
    p.Pmax         = pmax ? d->Pmax : nullptr;
    p.status       = d->status;
    p.check        = (d->flags & FPA_CHECK_NAN) ? 1 : 0;
    p.fact         = fact ? static_cast<const unsigned char*>(d->factored) : nullptr;
    p.n_classes    = fact ? d->n_classes : 0;
    p.table_in_smem = p.table_in_smem_only_one_cta = 0;
    FPA_REQUIRE(d->n_points < 2147483647LL, "n_points too large for one launch");

    if (fact) {
        // state + class sums: 8.4 KB for N = 64 -- one CTA of 256 threads per point, several per SM
        const size_t smem = nwave_smem_bytes(d->n_waves, 0) + (size_t)(p.n_classes + 1) * sizeof(double2);
        if (smem <= 200 * 1024) {
            // threads per point (profiles/r2_fact_thread_sweep.txt): about 1 024 per SM in all -- 64 (128 above 64
            // waves) for large batches: many small CTAs per SM hide each other's barriers and load latencies best --
            // up to 512 when the batch leaves SMs to spare: a single run is one CTA whatever its size, the latencies
            // of its own passes are all there is to hide (1 024 threads cost more in instructions issued by lanes
            // without work than they hide).  FPA_FACT_THREADS overrides (tools)
            int dev = 0, sms = 148;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            const int env_threads = getenv("FPA_FACT_THREADS") ? atoi(getenv("FPA_FACT_THREADS")) : 0;
            const int     lo = d->n_waves <= 64 ? 64 : 128, hi = d->n_waves <= 12 ? 64 : (d->n_waves <= 32 ? 256 : 512);
            const int64_t per_sm = (d->n_points + sms - 1) / sms;      // points an SM gets at once
            int           threads = hi;
            while (threads > lo && threads * per_sm > 1024) threads >>= 1;
            if (env_threads >= 32 && env_threads <= 1024) threads = env_threads & ~31;
            cudaError_t      e = cudaFuncSetAttribute(nwave_rk4_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(nwave_rk4_kernel<factored>)");
            nwave_rk4_kernel<true><<<(unsigned)d->n_points, threads, smem, st>>>(p);
            e = cudaGetLastError();
            if (e != cudaSuccess) return cuda_fail(e, "nwave_rk4_kernel<factored> launch");
            return FPA_OK;
        }
        // more classes than shared memory holds: the entry list it is
        p.fact = nullptr;
        FPA_REQUIRE(d->row_ptr != nullptr && (d->n_triplets == 0 || d->triplets), "triplet table must be set");
    }

    // the triplet list stays in shared memory when it fits beside the state (<= 200 KB in total)
    const size_t with_table = nwave_smem_bytes(d->n_waves, d->n_triplets);
    p.table_in_smem = with_table <= 200 * 1024 ? 1 : 0;
    const size_t smem = p.table_in_smem ? with_table : nwave_smem_bytes(d->n_waves, 0);
    p.table_in_smem_only_one_cta = smem > 100 * 1024 ? 1 : 0;
    // Warps per point: one warp per row of the triplet sum (up to 32 warps) when the batch is too
    // small to fill the GPU with points -- a single run (B = 1) is one CTA and its only parallelism
    // is across rows and entries; for large batches 8 warps per point leave room for several CTAs
    // per SM.
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int warps = d->n_waves < 32 ? d->n_waves : 32;
    if (d->n_points >= 4 * (int64_t)sms && !p.table_in_smem_only_one_cta) warps = warps < 8 ? warps : 8;
    const int threads = 32 * warps;

    cudaError_t e = cudaFuncSetAttribute(nwave_rk4_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(nwave_rk4_kernel)");
    nwave_rk4_kernel<false><<<(unsigned)d->n_points, threads, smem, st>>>(p);
    e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "nwave_rk4_kernel launch");
    return FPA_OK;
}

}  // namespace fpa

// ------------------------------------------------------------------ host: triplet enumeration
extern "C" int64_t fpa_enumerate_triplets(int32_t N, const int32_t* g, fpa_triplet* out, int64_t cap,
                                          int64_t* row_ptr) {
    if (N < 1 || N > 32767 || g == nullptr) {
        fpa::set_error("fpa_enumerate_triplets: need 1 <= N <= 32767 and a grid index array");
        return -1;
    }
    int64_t count = 0;
    for (int32_t n = 0; n < N; ++n) {
        if (row_ptr) row_ptr[n] = count;
        for (int32_t k = 0; k < N; ++k) {
            for (int32_t l = k; l < N; ++l) {
                const int64_t target = (int64_t)g[k] + (int64_t)g[l] - (int64_t)g[n];
                for (int32_t m = 0; m < N; ++m) {
                    if (m == k || m == l) continue;
                    if ((int64_t)g[m] != target) continue;
                    if (out) {
                        if (count >= cap) {
                            fpa::set_error("fpa_enumerate_triplets: output capacity %lld too small",
                                           (long long)cap);
                            return -1;
                        }
                        out[count].k = (int16_t)k;
                        out[count].l = (int16_t)l;
                        out[count].m = (int16_t)m;
                        out[count].weight = (int16_t)(k == l ? 1 : 2);
                    }
                    ++count;
                }
            }
        }
    }
    if (row_ptr) row_ptr[N] = count;
    return count;
}

extern "C" int64_t fpa_enumerate_triplets_omega(int32_t N, const double* omega, double atol, double rtol, fpa_triplet* out,
                                                int64_t cap, int64_t* row_ptr) {
    if (N < 1 || N > 32767 || omega == nullptr || !(atol >= 0.0) || !(rtol >= 0.0)) {
        fpa::set_error("fpa_enumerate_triplets_omega: need 1 <= N <= 32767, an omega array and non-negative tolerances");
        return -1;
    }
    int64_t count = 0;
    for (int32_t n = 0; n < N; ++n) {
        if (row_ptr) row_ptr[n] = count;
        for (int32_t k = 0; k < N; ++k) {
            for (int32_t l = k; l < N; ++l) {
                const volatile double lhs = omega[k] + omega[l];   // rounded to double, as numpy does
                for (int32_t m = 0; m < N; ++m) {
                    if (m == k || m == l) continue;
                    const volatile double rhs = omega[m] + omega[n];
                    // numpy.isclose for finite values: |a - b| <= atol + rtol * |b|
                    const volatile double diff = lhs - rhs;
                    const volatile double tol = rtol * fabs(rhs);
                    if (!(fabs(diff) <= atol + tol)) continue;
                    if (out) {
                        if (count >= cap) {
                            fpa::set_error("fpa_enumerate_triplets_omega: output capacity %lld too small", (long long)cap);
                            return -1;
                        }
                        out[count].k = (int16_t)k;
                        out[count].l = (int16_t)l;
                        out[count].m = (int16_t)m;
                        out[count].weight = (int16_t)(k == l ? 1 : 2);
                    }
                    ++count;
                }
            }
        }
    }
    if (row_ptr) row_ptr[N] = count;
    return count;
}

// ------------------------------------------------------------------ host: table factorisation
namespace {
struct PairW {
    int16_t k, l;
    int32_t w;
    bool operator<(const PairW& o) const { return k != o.k ? k < o.k : (l != o.l ? l < o.l : w < o.w); }
};
struct Factored {
    std::vector<std::vector<PairW>> classes;
    std::vector<int>                cmap;   // [N*N] class or -1
    std::vector<int>                wown;   // [N*N]
    int64_t                         n_pairs = 0;
    int                             mode = 0;
};

// groups[n*N+m] = merged, sorted (k <= l, weight) list of the entries (n; k, l, m).
// mode 0: the groups as they are; 1: plus the own pair {n, m} of every group that has entries and lacks it;
// 2: plus the own pair of EVERY cell -- only if no cell holds it already (then w_own is the same for all plans).
bool factor_groups(int N, const std::vector<std::vector<PairW>>& groups, int mode, Factored* out) {
    Factored&                         f = *out;
    std::map<std::vector<PairW>, int> ids;
    f = Factored();
    f.mode = mode;
    f.cmap.assign((size_t)N * N, -1);
    f.wown.assign((size_t)N * N, 0);
    for (int n = 0; n < N; ++n)
        for (int m = 0; m < N; ++m) {
            std::vector<PairW> key = groups[(size_t)n * N + m];
            if (key.empty() && mode != 2) continue;
            if (mode != 0) {
                const PairW own = {(int16_t)(n < m ? n : m), (int16_t)(n < m ? m : n), n == m ? 1 : 2};
                bool        present = false;
                for (const PairW& q : key) present |= q.k == own.k && q.l == own.l;
                if (present && mode == 2) return false;
                if (!present) {
                    key.insert(std::lower_bound(key.begin(), key.end(), own), own);
                    f.wown[(size_t)n * N + m] = own.w;
                }
            }
            auto it = ids.find(key);
            if (it == ids.end()) {
                it = ids.emplace(key, (int)f.classes.size()).first;
                f.n_pairs += (int64_t)key.size();
                f.classes.push_back(key);
            }
            f.cmap[(size_t)n * N + m] = it->second;
        }
    return true;
}
}  // namespace

// Factor the table into *out (resized).  Returns the blob size or -1.
static int64_t factor_build(int32_t N, const fpa_triplet* triplets, const int64_t* row_ptr, int64_t n_triplets,
                            std::vector<unsigned char>* out, int32_t* n_classes) {
    using fpa::FactHeader;
    using fpa::FactPair;
    if (N < 1 || N > 128 || row_ptr == nullptr || n_triplets < 0 || (n_triplets > 0 && triplets == nullptr)) {
        fpa::set_error("fpa_nwave_factor_table: need 1 <= N <= 128 and a CSR triplet table");
        return -1;
    }
    if (row_ptr[0] != 0 || row_ptr[N] != n_triplets) {
        fpa::set_error("fpa_nwave_factor_table: row_ptr must run from 0 to n_triplets");
        return -1;
    }
    std::vector<std::vector<PairW>> groups((size_t)N * N);
    for (int n = 0; n < N; ++n) {
        if (row_ptr[n + 1] < row_ptr[n]) {
            fpa::set_error("fpa_nwave_factor_table: row_ptr must not decrease");
            return -1;
        }
        for (int64_t e = row_ptr[n]; e < row_ptr[n + 1]; ++e) {
            const fpa_triplet t = triplets[e];
            if (t.k < 0 || t.k >= N || t.l < 0 || t.l >= N || t.m < 0 || t.m >= N) {
                fpa::set_error("fpa_nwave_factor_table: entry %lld has a wave index outside [0, %d)", (long long)e, N);
                return -1;
            }
            std::vector<PairW>& g = groups[(size_t)n * N + t.m];
            const PairW         q = {t.k < t.l ? t.k : t.l, t.k < t.l ? t.l : t.k, t.weight};
            bool                merged = false;
            for (PairW& o : g)
                if (o.k == q.k && o.l == q.l) {
                    o.w += q.w;
                    merged = true;
                }
            if (!merged) g.push_back(q);
        }
    }
    for (auto& g : groups) {
        std::sort(g.begin(), g.end());
        for (const PairW& q : g)
            if (q.w < -(1 << 24) || q.w > (1 << 24)) {      // exact in the record's float
                fpa::set_error("fpa_nwave_factor_table: merged weight %d is out of range", q.w);
                return -1;
            }
    }
    // whichever of the three forms leaves the least to do per RHS: pair products, plus a pass over the w_own
    // matrix for mode 1
    Factored best, cand;
    int64_t  best_cost = -1;
    for (int mode = 0; mode < 3; ++mode) {
        if (!factor_groups(N, groups, mode, &cand)) continue;
        const int64_t cost = 6 * cand.n_pairs + (mode == 1 ? 2 * (int64_t)N * N : 0);
        if (best_cost < 0 || cost < best_cost) {
            best_cost = cost;
            best      = cand;
        }
    }
    Factored& f = best;
    const int C = (int)f.classes.size();
    if (C >= fpa::kFactMaxCls) {
        fpa::set_error("fpa_nwave_factor_table: %d classes exceed the format's limit", C);
        return -1;
    }
    // processing order: classes of similar size next to each other (lanes that work side by side); slot order:
    // first appearance in the row-major cell map
    std::vector<int> order((size_t)C), slot((size_t)C, -1);
    for (int c = 0; c < C; ++c) order[(size_t)c] = c;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return f.classes[(size_t)a].size() > f.classes[(size_t)b].size(); });
    int n_slots = 0;
    for (size_t i = 0; i < (size_t)N * N; ++i)
        if (f.cmap[i] >= 0 && slot[(size_t)f.cmap[i]] < 0) slot[(size_t)f.cmap[i]] = n_slots++;
    int64_t n_padded = 0;
    for (const auto& c : f.classes) n_padded += ((int64_t)c.size() + 3) & ~(int64_t)3;

    int np_log = 0;
    while ((1 << np_log) < N) ++np_log;
    const int n_pad = 1 << np_log;

    auto       up16 = [](int64_t v) { return (v + 15) & ~(int64_t)15; };
    FactHeader h = {};
    h.magic      = fpa::kFactMagic;
    h.n_waves    = N;
    h.n_classes  = C;
    h.n_pairs    = (int32_t)n_padded;
    h.mode       = f.mode;
    h.np_log     = np_log;
    h.off_cls    = (int32_t)up16(sizeof(FactHeader));
    h.off_pairs  = (int32_t)up16(h.off_cls + (int64_t)(C + 1) * 8);
    h.off_cmap   = (int32_t)up16(h.off_pairs + n_padded * (int64_t)sizeof(FactPair));
    h.off_wown   = (int32_t)up16(h.off_cmap + (int64_t)N * n_pad * 4);
    h.bytes      = (int32_t)up16(h.off_wown + (f.mode == 1 ? (int64_t)N * N * 2 : 0));
    if (n_classes) *n_classes = C;
    out->assign((size_t)h.bytes, 0);
    unsigned char* base = out->data();
    memcpy(base, &h, sizeof h);
    int32_t*  cls   = reinterpret_cast<int32_t*>(base + h.off_cls);      // {first pair, slot byte offset} per class
    FactPair* pairs = reinterpret_cast<FactPair*>(base + h.off_pairs);
    uint32_t* cmap  = reinterpret_cast<uint32_t*>(base + h.off_cmap);
    int16_t*  wown  = reinterpret_cast<int16_t*>(base + h.off_wown);
    int32_t   at = 0;
    for (int r = 0; r < C; ++r) {
        const int c    = order[(size_t)r];
        cls[2 * r]     = at;
        cls[2 * r + 1] = slot[(size_t)c] * 16;
        for (const PairW& q : f.classes[(size_t)c]) {
            pairs[at].k16 = (uint16_t)(q.k * 16);
            pairs[at].l16 = (uint16_t)(q.l * 16);
            pairs[at].w   = (float)q.w;
            ++at;
        }
        while (at & 3) pairs[at++] = FactPair{0, 0, 0.0f};     // padding: weight 0
    }
    cls[2 * C]     = at;
    cls[2 * C + 1] = C * 16;
    for (int n = 0; n < N; ++n)
        for (int q = 0; q < n_pad; ++q) {
            int m = 0;      // bit reversal of q over np_log bits
            for (int bit = 0; bit < np_log; ++bit) m |= ((q >> bit) & 1) << (np_log - 1 - bit);
            const int c = m < N ? f.cmap[(size_t)n * N + m] : -1;
            cmap[(size_t)n * n_pad + q] = (uint32_t)(c < 0 ? C : slot[(size_t)c]) * 16u;
        }
    if (f.mode == 1)
        for (size_t i = 0; i < (size_t)N * N; ++i) wown[i] = (int16_t)f.wown[i];
    return h.bytes;
}

// The C entry point is called twice per plan (size, then fill) and the host integrator entry points call it on
// every launch: the last factorisation of each thread is kept, keyed by a hash of the table.
extern "C" int64_t fpa_nwave_factor_table(int32_t N, const fpa_triplet* triplets, const int64_t* row_ptr, int64_t n_triplets,
                                          void* blob, int64_t cap, int32_t* n_classes) {
    if (N < 1 || N > 128 || row_ptr == nullptr || n_triplets < 0 || (n_triplets > 0 && triplets == nullptr)) {
        fpa::set_error("fpa_nwave_factor_table: need 1 <= N <= 128 and a CSR triplet table");
        return -1;
    }
    struct Cached {
        uint64_t                   key = 0;
        int32_t                    N = 0, C = 0;
        int64_t                    nt = -1;
        std::vector<unsigned char> blob;
    };
    static thread_local Cached last;
    auto fnv = [](uint64_t h, const void* data, size_t bytes) {
        const unsigned char* p = static_cast<const unsigned char*>(data);
        size_t               i = 0;
        for (; i + 8 <= bytes; i += 8) {     // word at a time: the table is ~0.7 MB at N = 64
            uint64_t w;
            memcpy(&w, p + i, 8);
            h = (h ^ w) * 1099511628211ull;
        }
        for (; i < bytes; ++i) h = (h ^ p[i]) * 1099511628211ull;
        return h;
    };
    uint64_t key = fnv(14695981039346656037ull, row_ptr, (size_t)(N + 1) * sizeof(int64_t));
    key          = fnv(key, triplets, (size_t)n_triplets * sizeof(fpa_triplet));
    if (!(last.nt == n_triplets && last.N == N && last.key == key && !last.blob.empty())) {
        Cached        fresh;
        const int64_t nb = factor_build(N, triplets, row_ptr, n_triplets, &fresh.blob, &fresh.C);
        if (nb < 0) return -1;
        fresh.key = key;
        fresh.N   = N;
        fresh.nt  = n_triplets;
        last      = std::move(fresh);
    }
    if (n_classes) *n_classes = last.C;
    const int64_t bytes = (int64_t)last.blob.size();
    if (blob != nullptr && cap >= bytes) memcpy(blob, last.blob.data(), (size_t)bytes);
    return bytes;
}

extern "C" double fpa_nwave_factored_flops_per_step(const void* blob) {
    // per RHS: 8 per non-empty cell (T * conj(At_m), accumulated), 10 per pair product (complex product 6, weighted
    // accumulate 4), c*N as for the entry list (c = 30); per step 4 RHS + 26*N
    if (blob == nullptr) return 0.0;
    const unsigned char*   base = static_cast<const unsigned char*>(blob);
    const fpa::FactHeader* h = reinterpret_cast<const fpa::FactHeader*>(base);
    if (h->magic != fpa::kFactMagic) return 0.0;
    const fpa::FactPair* pairs = reinterpret_cast<const fpa::FactPair*>(base + h->off_pairs);
    const uint32_t*      cmap = reinterpret_cast<const uint32_t*>(base + h->off_cmap);
    int64_t              live = 0, cells = 0;
    for (int32_t e = 0; e < h->n_pairs; ++e) live += pairs[e].w != 0.0f;
    for (int64_t i = 0; i < ((int64_t)h->n_waves << h->np_log); ++i) cells += cmap[i] != (uint32_t)h->n_classes * 16u;
    const double rhs = 8.0 * (double)cells + 10.0 * (double)live + 30.0 * (double)h->n_waves;
    return 4.0 * rhs + 26.0 * (double)h->n_waves;
}

extern "C" double fpa_nwave_flops_per_step(int32_t n_waves, int64_t n_triplets, int64_t n_pairs) {
    // SURVEY 8(d): per RHS 8*T_terms + 6*T_pairs + c*N with c = 30 (phase rotate 6, power 3,
    // Kerr factor 3, conj(E_n)*R 6, assemble 12); per step 4 RHS + 26*N for the RK4 combine.
    const double rhs = 8.0 * (double)n_triplets + 6.0 * (double)n_pairs + 30.0 * (double)n_waves;
    return 4.0 * rhs + 26.0 * (double)n_waves;
}
