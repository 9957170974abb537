// nwave_comb.cu -- N-wave RK4 for plans on an integer frequency grid, in correlation form
// (NOT in the reference; SURVEY App. C "uniform-comb shortcut").
//
// On a grid w_j = w_0 + g_j*dw the matching condition w_k + w_l - w_m = w_n is g_k + g_l - g_m = g_n,
// so with At_j = A_j exp(i*beta_j*z) placed at grid slot g_j - g_min (empty slots hold 0) the whole
// FWM + SPM + XPM sum of wave n is
//
//     R_n = sum_{k,l,m : k+l-m=n} At_k At_l conj(At_m) = sum_k At_k * X_{n-k},
//     X_d = sum_m At_{m+d} conj(At_m)            (auto-correlation, X_{-d} = conj(X_d))
//
// i.e. one correlation and one convolution of length-M sequences (M = grid span): 2*M^2 complex
// MACs per RHS instead of O(N^3) table entries, with exactly the weights of the analytic Kerr
// factor (2*sum P - P_n) for the m = k / m = l terms, and
//
//     dA_n/dz = -(alpha/2) A_n + i*gamma * conj(E_n) * R_n ,   E_n = exp(i*beta_n*z).
//
// Same ODE as nwave.cu integrates from the enumerated triplet table (tests compare both with the
// oracle).  Both sums have the shape  out[o] = sum_i a[i] * w[i + o]:  a thread owns a tile of
// adjacent outputs and a contiguous part of the i-range, keeps the tile's accumulators and a sliding
// window of w in registers, and the parts are combined with warp shuffles.
//
// Two kernels, chosen by batch size (nwave_comb_launch):
//   nwave_comb_kernel   one CTA of 4 warps per point, tiles of 2, sums split 4 ways: latency, for single
//                       runs and batches below 4 x SM count;
//   nwave_comb8_kernel  one warp per point, tiles of 8 with a rolling window: throughput, for larger batches.
// Other mappings of the batch path were measured and removed, each slower at every batch size tried (N = 64,
// B200, profiles/r2_comb_bench.txt, point.steps/s): the round-1 warp per point with tiles of 4
// (B = 592 / 1024 / 9472: 5.2e7 / 6.5e7 / 8.9e7 against 6.8e7 / 7.4e7 / 9.3e7), half a warp per point
// (B = 1024 / 4736: 6.5e7 / 9.0e7 against 7.4e7 / 9.3e7) and two warps per point (B = 1024: 5.8e7 against 6.6e7).
// exp(i*beta_n*z) advances by a constant rotation per half step (exact sincos every kResync steps),
// the step is the constant h = (z_max - z0)/n_steps like the 4-wave fast kernel.
#include "fpa_common.cuh"

#include <assert.h>

// compute-sanitizer is not available on the B200 pool: -DFPA_BOUNDS_CHECK turns every shared-memory
// sequence access of this file into a checked one (device assert), tools/bounds_check.py builds that
// variant and runs the N-wave tests on it.
// -DFPA_COMB_TIMING: thread 0 of point 0 accumulates clock64() between the phases of a stage and prints
// the averages when the kernel ends (tools only; never in the shipped library).
#ifdef FPA_COMB_TIMING
#include <cstdio>
#define FPA_TICK(k)                                   \
    do {                                              \
        if (b == 0 && tid == 0) {                     \
            const long long now_ = clock64();         \
            tk[k] += now_ - t_prev;                   \
            t_prev = now_;                            \
        }                                             \
    } while (0)
#else
#define FPA_TICK(k) ((void)0)
#endif

#ifdef FPA_BOUNDS_CHECK
#define FPA_IN_RANGE(idx, n) assert((idx) >= 0 && (idx) < (n))
#else
#define FPA_IN_RANGE(idx, n) ((void)0)
#endif

namespace fpa {

struct CombParams {
    int64_t        n_points;
    int            n_waves, span;  // N lines on M = span grid slots
    int            beta_stride, gamma_stride, alpha_stride, A0_stride;
    const double*  beta;
    const double*  gamma;
    const double*  alpha;
    const double*  A0;
    const int32_t* slot;  // [N] grid slot of each wave (g_j - g_min), device memory
    double         z0, z_max;
    int            n_steps, save_every;
    int64_t        n_saved;
    double*        A_trace;
    double*        A_end;
    double*        Pmax;
    int32_t*       status;
    int            check;
};

constexpr int kCombThreads = 256;
constexpr int kCombResync  = 32;
constexpr int kPad         = 8;  // spare words of R

struct CombSmem {
    double2 *y, *ys, *yn, *E, *Eh, *rot;  // [N] state, stage state, accumulator, phases
    double2 *At;                          // [seq_words]  At on the grid at padx(slot), zeros above M
    double2 *Y;                           // [seq_words]  Y[padx(q)] = X_{M-1-q}, zeros above 2M-2
    double2 *R;                           // [comb_r_words(M)]
    double*  beta;
    int*     slot;
};

// words of a zero-padded, bank-skewed sequence buffer (At and Y): the sums run over whole blocks of 8
// terms per part (at most 8 parts), so indices reach 2*roundup(M, 64) + 16
__host__ __device__ inline int comb_seq_words(int M, int sk) {
    const int e = 2 * ((M + 63) & ~63) + 16;
    return e + (e >> sk) + 1;
}

__host__ __device__ inline int comb_r_words(int M) { return M + (M >> 3) + kPad; }  // room for the padx<3> layout

__host__ __device__ inline size_t comb_point_doubles(int N, int M, int sk) {
    const size_t d = 2 * (size_t)(6 * N + 2 * comb_seq_words(M, sk) + comb_r_words(M)) + (size_t)N + (size_t)(N + 1) / 2 + 2;
    return (d + 1) & ~(size_t)1;  // keeps every point's block 16-byte aligned
}

__device__ __forceinline__ CombSmem comb_carve(double* base, int N, int M, int sk) {
    CombSmem s;
    s.y    = reinterpret_cast<double2*>(base);
    s.ys   = s.y + N;
    s.yn   = s.ys + N;
    s.E    = s.yn + N;
    s.Eh   = s.E + N;
    s.rot  = s.Eh + N;
    s.At   = s.rot + N;
    s.Y    = s.At + comb_seq_words(M, sk);
    s.R    = s.Y + comb_seq_words(M, sk);
    s.beta = reinterpret_cast<double*>(s.R + comb_r_words(M));
    s.slot = reinterpret_cast<int*>(s.beta + N);
    return s;
}

// Shared-memory position of sequence element e: one spare word after every 2^SK words (the tile width: 2 in
// nwave_comb_kernel, 8 in nwave_comb8_kernel), so that the windows of eight neighbouring tiles (16-byte words
// 3 resp. 9 apart) fall into distinct bank groups (3*tau mod 8 resp. 9*tau mod 8 are permutations) and every
// operand of a block of terms sits at a compile-time offset from the block's first word.
template <int SK>
__host__ __device__ __forceinline__ int padx(int e) { return e + (e >> SK); }

// =====================================================================================================
// CTA-per-point kernel for single runs and small batches (nwave_comb_kernel): 4 warps per point, tiles of
// kTile = 2 outputs, the term range of a sum split kSplit = 4 ways (the fastest of seven shapes tried).
// =====================================================================================================
constexpr int kCtaWarps = 4;
constexpr int kTile = 2, kSplit = 4, kSk = 1;

// acc[t] += a[i] (x) w[wbase + i + t]  for i in [i0, i1), t in [0, kTile);  (x) = conj(a)*w when CONJ
// else a*w.  i0 and i1 are multiples of 8 and wbase of kTile, so inside a block of K = 8 terms every
// operand sits at a compile-time offset from two base addresses; all operands of a block are loaded first
// (independent loads in flight together), then K*kTile complex MACs run from registers.  No bounds
// tests: the sequences are zero beyond their last element.
template <bool CONJ>
__device__ __forceinline__ void sliding_mac(const double2* __restrict__ a, const double2* __restrict__ w, int wbase,
                                            int i0, int i1, int words, double (&re)[kTile], double (&im)[kTile]) {
    constexpr int K = 8;  // K = 4 or 2 and unrolling the block loop: 0 ... -12 % (measured)
    for (int i = i0; i < i1; i += K) {
        const double2* ap = a + padx<kSk>(i);
        const double2* wp = w + padx<kSk>(wbase + i);
        FPA_IN_RANGE(padx<kSk>(i) + (K - 1) + ((K - 1) >> kSk), words);
        FPA_IN_RANGE(padx<kSk>(wbase + i) + (K + kTile - 2) + ((K + kTile - 2) >> kSk), words);
        double2 av[K], wv[K + kTile - 1];
#pragma unroll
        for (int k = 0; k < K; ++k) av[k] = ap[k + (k >> kSk)];
#pragma unroll
        for (int k = 0; k < K + kTile - 1; ++k) wv[k] = wp[k + (k >> kSk)];
#pragma unroll
        for (int k = 0; k < K; ++k) {
#pragma unroll
            for (int t = 0; t < kTile; ++t) {
                if (CONJ) {  // conj(a) * w
                    re[t] = fma(av[k].x, wv[k + t].x, fma(av[k].y, wv[k + t].y, re[t]));
                    im[t] = fma(av[k].x, wv[k + t].y, fma(-av[k].y, wv[k + t].x, im[t]));
                } else {     // a * w
                    re[t] = fma(av[k].x, wv[k + t].x, fma(-av[k].y, wv[k + t].y, re[t]));
                    im[t] = fma(av[k].x, wv[k + t].y, fma(av[k].y, wv[k + t].x, im[t]));
                }
            }
        }
    }
}

// out[o] = sum_{i<n_terms} a[i] (x) w[i + o] for o in [0, n_out): tiles of kTile outputs, shared by the
// kCtaWarps warps of the CTA; the i-range is split into kSplit contiguous parts held by lanes LP = 32/kSplit
// apart in the same warp (so the eight lanes of a shared-memory wavefront work on eight neighbouring tiles of
// one part), combined by shuffles; the part-0 lane calls store(o, re, im).
template <bool CONJ, typename Store>
__device__ __forceinline__ void tiled_correlation(const double2* a, const double2* w, int n_terms, int n_out, int tid,
                                                  int words, Store store) {
    // the parts are whole blocks of 8 terms; the last part reads the zeros behind the sequence
    constexpr int LP = 32 / kSplit;
    const int lane = tid & 31, warp = tid >> 5;
    const int part = lane / LP, tl = lane % LP;
    const int n_tiles = (n_out + kTile - 1) / kTile;
    const int chunk   = ((n_terms + kSplit - 1) / kSplit + 7) & ~7;
    const int i0      = part * chunk;
    const int i1      = i0 + chunk;
    // every lane of a warp runs the same number of rounds (the shuffles below need all of them)
    const int rounds = (n_tiles + kCtaWarps * LP - 1) / (kCtaWarps * LP);
    for (int r = 0; r < rounds; ++r) {
        const int  tile = (r * kCtaWarps + warp) * LP + tl;
        const bool live = tile < n_tiles;
        double     re[kTile], im[kTile];
#pragma unroll
        for (int t = 0; t < kTile; ++t) re[t] = im[t] = 0.0;
        if (live) sliding_mac<CONJ>(a, w, tile * kTile, i0, i1, words, re, im);
#pragma unroll
        for (int d = LP; d < 32; d <<= 1) {
#pragma unroll
            for (int t = 0; t < kTile; ++t) {
                re[t] += __shfl_xor_sync(0xffffffffu, re[t], d);
                im[t] += __shfl_xor_sync(0xffffffffu, im[t], d);
            }
        }
        if (live && part == 0) {
#pragma unroll
            for (int t = 0; t < kTile; ++t)
                if (tile * kTile + t < n_out) store(tile * kTile + t, re[t], im[t]);
        }
    }
}

__global__ void __launch_bounds__(kCombThreads, 2) nwave_comb_kernel(const CombParams p) {
    constexpr int T = 32 * kCtaWarps;  // threads per scan point
    extern __shared__ __align__(16) double comb_smem_raw[];
    const int     N = p.n_waves, M = p.span;
    const int     tid = threadIdx.x;
    const int64_t b = blockIdx.x;
    CombSmem s = comb_carve(comb_smem_raw, N, M, kSk);
    // Per-wave state (y, stage state, accumulator, phases) in registers: T >= N, so a thread owns at most one
    // wave and every `j` loop below runs at most once -- four dependent shared-memory round trips per RK4 stage
    // less than with the state in shared memory, on a path whose cost is latency.
    double2 r_y = {0, 0}, r_ys = {0, 0}, r_yn = {0, 0}, r_E = {0, 0}, r_Eh = {0, 0}, r_rot = {0, 0};
    double  r_beta = 0.0;
    int     r_slot = 0;

    const double gamma = p.gamma[b * p.gamma_stride];
    const double nha   = -0.5 * p.alpha[b * p.alpha_stride];
    const int    n_steps = p.n_steps;
    const double z0 = p.z0;
    const double h = (p.z_max - z0) / (double)n_steps, hh = 0.5 * h, h6 = h / 6.0, h3 = h6 + h6;

    for (int j = tid; j < N; j += T) {
        const double bj = p.beta[b * p.beta_stride * N + j];
        r_beta = bj;
        r_slot = p.slot[j];
        const double2* a0 = reinterpret_cast<const double2*>(p.A0) + b * p.A0_stride * N;
        r_y = a0[j];
        double sn, cs;
        sincos(bj * hh, &sn, &cs);
        r_rot = make_double2(cs, sn);
    }
    for (int m = tid; m < comb_seq_words(M, kSk); m += T) {
        s.At[m] = make_double2(0.0, 0.0);  // empty grid slots and the padding stay 0
        s.Y[m]  = make_double2(0.0, 0.0);
    }
    for (int m = tid; m < M + kPad; m += T) s.R[m] = make_double2(0.0, 0.0);
    __syncthreads();

    double2* tr = p.A_trace ? reinterpret_cast<double2*>(p.A_trace) + b * p.n_saved * N : nullptr;
    if (tr) {
        for (int j = tid; j < N; j += T) tr[j] = r_y;
        tr += N;
    }
    double pm[4] = {0.0, 0.0, 0.0, 0.0};
    if (p.Pmax) {
        int q = 0;
        for (int j = tid; j < N; j += T, ++q) pm[q] = fma(r_y.y, r_y.y, r_y.x * r_y.x);
    }
    int     save_ctr = p.save_every;
    int32_t bad = FPA_POINT_OK;
    double2* const Yc = s.Y;  // Yc[q] = X_{M-1-q}, q in [0, 2M-2]
    const int      words = comb_seq_words(M, kSk);

#ifdef FPA_COMB_TIMING
    long long tk[8] = {0, 0, 0, 0, 0, 0, 0, 0}, t_prev = clock64();
#endif
    for (int i = 0; i < n_steps; ++i) {
        const bool resync = (i % kCombResync) == 0;
        const double zi = fma((double)i, h, z0);
        int nf = 0;
        // the four stages unrolled: no stage-dependent branches on the latency path (-7 ... -14 % per step)
#pragma unroll
        for (int stage = 0; stage < 4; ++stage) {
            FPA_TICK(0);  // loop overhead, save block, finite vote
            // ---- phases and the rotated stage state on the grid (thread j owns wave j)
            for (int j = tid; j < N; j += T) {
                double2 e;
                if (stage == 0) {
                    if (resync) {
                        double sn, cs;
                        sincos(r_beta * zi, &sn, &cs);
                        e = make_double2(cs, sn);
                    } else {
                        e = r_E;
                    }
                    const double2 v = r_y;
                    r_ys = v;
                    r_yn = v;
                    if (p.check && (nonfinite(v.x) || nonfinite(v.y))) nf = 1;
                } else if (stage == 2) {
                    e = r_Eh;
                } else {  // stage 1: z + h/2, stage 3: z + h
                    const double2 r = r_rot, e0 = stage == 1 ? r_E : r_Eh;
                    e = make_double2(fma(-e0.y, r.y, e0.x * r.x), fma(e0.x, r.y, e0.y * r.x));
                }
                if (stage == 1) r_Eh = e;
                if (stage == 0 || stage == 3) r_E = e;  // after stage 3: the next step's phase
                const double2 a = r_ys;
                FPA_IN_RANGE(r_slot, M);
                s.At[padx<kSk>(r_slot)] = make_double2(fma(-a.y, e.y, a.x * e.x), fma(a.x, e.y, a.y * e.x));
                if (stage == 3) r_Eh = e;               // phase this stage's conj(E) uses
            }
            FPA_TICK(1);  // phases + At
            __syncthreads();
            FPA_TICK(2);  // barrier 1
            // ---- X_d = sum_m At[m+d] conj(At[m]), d in [0, M): stored mirrored for the convolution
            tiled_correlation<true>(s.At, s.At, M, M, tid, words, [&](int d, double re, double im) {
                FPA_IN_RANGE(padx<kSk>(M - 1 - d), words);
                FPA_IN_RANGE(padx<kSk>(M - 1 + d), words);
                Yc[padx<kSk>(M - 1 - d)] = make_double2(re, im);
                Yc[padx<kSk>(M - 1 + d)] = make_double2(re, -im);
            });
            FPA_TICK(3);  // auto-correlation
            __syncthreads();
            FPA_TICK(4);  // barrier 2
            // ---- R_n = sum_k At[k] X_{n-k} = sum_k At[k] Yc[(M-1-n) + k]; output o = M-1-n
            tiled_correlation<false>(s.At, Yc, M, M, tid, words, [&](int o, double re, double im) {
                FPA_IN_RANGE(M - 1 - o, M + kPad);
                s.R[M - 1 - o] = make_double2(re, im);
            });
            FPA_TICK(5);  // convolution
            __syncthreads();
            FPA_TICK(6);  // barrier 3
            // ---- k_n = -(alpha/2) x + i*gamma*conj(E_n) R_n and the RK4 bookkeeping
            const double wa = (stage == 0 || stage == 3) ? h6 : h3;
            const double wb = stage == 2 ? h : hh;
            for (int j = tid; j < N; j += T) {
                const double2 r = s.R[r_slot];
                const double2 e = stage == 0 ? r_E : r_Eh;
                const double2 x = r_ys;
                const double  fr = fma(r.y, e.y, r.x * e.x);
                const double  fi = fma(r.y, e.x, -(r.x * e.y));
                const double  kr = fma(nha, x.x, -(gamma * fi));
                const double  ki = fma(nha, x.y, gamma * fr);
                const double2 acc = r_yn;
                if (stage == 3) {
                    r_y = make_double2(fma(wa, kr, acc.x), fma(wa, ki, acc.y));
                } else {
                    const double2 y0 = r_y;
                    r_yn = make_double2(fma(wa, kr, acc.x), fma(wa, ki, acc.y));
                    r_ys = make_double2(fma(wb, kr, y0.x), fma(wb, ki, y0.y));
                }
            }
            FPA_TICK(7);  // k and the RK4 bookkeeping
            // no barrier: the next stage's first loop touches only what this thread wrote
        }
        if (p.check && i > 0 && bad == FPA_POINT_OK) {
            if (__syncthreads_or(nf)) bad = i - 1;  // the state produced by step i-1 was not finite
        }
        if (--save_ctr == 0) {
            save_ctr = p.save_every;
            if (tr) {
                for (int j = tid; j < N; j += T) tr[j] = r_y;
                tr += N;
            }
            if (p.Pmax) {
                int q = 0;
                for (int j = tid; j < N; j += T, ++q) {
                    const double P = fma(r_y.y, r_y.y, r_y.x * r_y.x);
                    pm[q] = (P != P || pm[q] != pm[q]) ? qnan() : fmax(pm[q], P);
                }
            }
        }
    }
    if (p.check && bad == FPA_POINT_OK) {
        int nf = 0;
        for (int j = tid; j < N; j += T) nf |= (nonfinite(r_y.x) || nonfinite(r_y.y)) ? 1 : 0;
        if (__syncthreads_or(nf)) bad = n_steps - 1;
    }
#ifdef FPA_COMB_TIMING
    if (b == 0 && tid == 0) {
        const double st = 4.0 * n_steps;
        printf("comb (CTA per point) cycles per stage: other %.0f | phases+At %.0f | bar %.0f | autocorr %.0f | bar %.0f | "
               "conv %.0f | bar %.0f | k+RK4 %.0f\n", tk[0] / st, tk[1] / st, tk[2] / st, tk[3] / st, tk[4] / st, tk[5] / st,
               tk[6] / st, tk[7] / st);
    }
#endif
    if (p.status && tid == 0) p.status[b] = bad;
    if (p.A_end) {
        double2* o = reinterpret_cast<double2*>(p.A_end) + b * N;
        for (int j = tid; j < N; j += T) o[j] = r_y;
    }
    if (p.Pmax) {
        int q = 0;
        for (int j = tid; j < N; j += T, ++q) p.Pmax[b * N + j] = pm[q];
    }
}

// =====================================================================================================
// Warp-per-point kernel for batches (nwave_comb8_kernel): tiles of EIGHT outputs with a rolling window.
//
// The round-1 batch mapping (sliding_mac above, one warp per point, tiles of 4) was bound by shared-memory
// wavefronts, not by the FP64 pipe (ncu: LSU 79 % busy at 63 % FP64 activity): a block of 8 terms loads 19 words
// for 128 FMAs.  Here a lane owns 8 adjacent outputs and walks its part of the term range one term at a time:
// the 8-word window of w slides
// by one word per term, so a term costs ONE new word of w and one (broadcast) word of a for 32 FMAs --
// 40 loads per 512 FMAs.  The loads of term k+1 are issued before the FMAs of term k (software pipeline);
// the window lives in registers and rotates by renaming (the 8-term body is fully unrolled).
// Sequences are stored with one spare word after every 8 (padx<3>): the eight lanes of a quarter-warp hold
// neighbouring tiles, 9 words apart, i.e. in eight different 16-byte bank groups -- conflict-free.
// Lane layout: LP = 2^lp lanes hold the tiles of one part of the term range (LP >= number of tiles), the
// 32 / LP parts are summed by xor-shuffles.  For M = 64: 8 tiles x 4 parts.
// =====================================================================================================
constexpr int kSk8 = 3;

// acc[t] += a * win[(k + t) & 7] for the 8 outputs of a tile, as two runs of 16 FMAs that share one operand
// each (first a.y, then a.x): consecutive FP64 instructions with a common operand get it from the operand-reuse
// cache and fetch two registers instead of three -- an FMA fetching three registers holds the pipe for 3 cycles
// instead of 2 (tools/dfma_operand_probe.cu).  The two FMAs of one accumulator are 16 instructions apart.
template <int K>
__device__ __forceinline__ void term8(double (&re)[8], double (&im)[8], const double2 a, const double2 (&win)[8]) {
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        re[t] = fma(-a.y, win[(K + t) & 7].y, re[t]);
        im[t] = fma(a.y, win[(K + t) & 7].x, im[t]);
    }
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        re[t] = fma(a.x, win[(K + t) & 7].x, re[t]);
        im[t] = fma(a.x, win[(K + t) & 7].y, im[t]);
    }
}

// (a.x, +-a.y): conj(a) * w is computed as a' * w with the sign bit of a.y flipped after the load (an integer
// operation on the high word: the FP64 pipe does not see it), so ONE instance of the loop below serves the
// auto-correlation (conj) and the convolution -- the unrolled body is 4.4 KB of code, and three inlined copies
// of it plus the four warps of a sub-partition at different places thrashed the instruction cache
// (stall_no_instruction 0.72 per issue in the first version of this kernel).
__device__ __forceinline__ double2 load_a(const double2* p, int sign_flip) {
    double2 v = *p;
    v.y = __hiloint2double(__double2hiint(v.y) ^ sign_flip, __double2loint(v.y));
    return v;
}

// acc[t] += a'[i] * w[obase + i + t] for i in [i0, i1), t in [0, 8).  obase and i0 are multiples of 8 and
// i1 - i0 is a multiple of 8.  Reads up to w[obase + i1 + 7] and a[i1].
__device__ __forceinline__ void roll8_mac(const double2* __restrict__ a, const double2* __restrict__ w, int obase,
                                          int i0, int i1, int sign_flip, double (&re)[8], double (&im)[8]) {
    double2        win[8];
    const double2* wp = w + padx<kSk8>(obase + i0);
    const double2* ap = a + padx<kSk8>(i0);
#pragma unroll
    for (int t = 0; t < 8; ++t) win[t] = wp[t];
    double2 av = load_a(ap, sign_flip);
    for (int i = i0; i < i1; i += 8) {
        wp += 9;  // the next 8 words of w (one spare word in between)
        // operands of the next term are requested before this term's 32 FMAs
#define FPA_TERM(K)                                                                     \
        {                                                                               \
            const double2 nw = wp[K];                                                   \
            const double2 an = load_a(ap + (K < 7 ? K + 1 : 9), sign_flip);             \
            term8<K>(re, im, av, win);                                                  \
            win[K] = nw;                                                                \
            av = an;                                                                    \
        }
        FPA_TERM(0) FPA_TERM(1) FPA_TERM(2) FPA_TERM(3) FPA_TERM(4) FPA_TERM(5) FPA_TERM(6) FPA_TERM(7)
#undef FPA_TERM
        ap += 9;
    }
}

// The same for exactly FOUR terms starting at i0 (a multiple of 4): the short parts of small plans.
__device__ __forceinline__ void roll4_mac(const double2* __restrict__ a, const double2* __restrict__ w, int obase,
                                          int i0, int sign_flip, double (&re)[8], double (&im)[8]) {
    double2 win[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) win[t] = w[padx<kSk8>(obase + i0 + t)];
    const double2* ap = a + padx<kSk8>(i0);                  // 4 words, no pad inside (i0 % 4 == 0)
    const double2* wp = w + padx<kSk8>(obase + i0 + 8);
#define FPA_TERM4(K)                                                                    \
    {                                                                                   \
        const double2 av = load_a(ap + K, sign_flip);                                   \
        double2       nw = make_double2(0.0, 0.0);                                      \
        if (K < 3) nw = wp[K];                                                          \
        term8<K>(re, im, av, win);                                                      \
        win[K] = nw;                                                                    \
    }
    FPA_TERM4(0) FPA_TERM4(1) FPA_TERM4(2) FPA_TERM4(3)
#undef FPA_TERM4
}

// One level of the reduce-scatter over the parts: lanes d apart exchange HALF of the CNT values they hold
// and keep the sum of the other half (the lane whose bit d is set keeps the upper half).  Against a
// butterfly all-reduce this moves 8+4+2 instead of 16+16+16 doubles for three levels, and leaves the outputs
// of a tile spread over the parts, so that all of them store.
template <int CNT>
__device__ __forceinline__ void scatter_level(double (&re)[8], double (&im)[8], int d, bool up) {
    if (CNT > 1) {
        constexpr int H = CNT / 2 > 0 ? CNT / 2 : 1;
#pragma unroll
        for (int t = 0; t < H; ++t) {
            const double sr = up ? re[t] : re[t + H], si = up ? im[t] : im[t + H];
            const double kr = up ? re[t + H] : re[t], ki = up ? im[t + H] : im[t];
            re[t] = kr + __shfl_xor_sync(0xffffffffu, sr, d);
            im[t] = ki + __shfl_xor_sync(0xffffffffu, si, d);
        }
    } else {  // one value left: plain all-reduce (only the lane with all upper part bits clear stores)
        re[0] += __shfl_xor_sync(0xffffffffu, re[0], d);
        im[0] += __shfl_xor_sync(0xffffffffu, im[0], d);
    }
}

// What a lane does in every correlation of the run -- both sums of a stage have the same shape (M outputs,
// M terms), so this is computed ONCE per kernel: LP = 2^lp lanes hold the tiles of one part of the term range
// (LP >= number of tiles, or all 32 lanes and several rounds of tiles), the 32 / LP parts are combined by the
// reduce-scatter, after which the lane owns outputs [off, off + cnt) of its tile.
struct Corr8Lane {
    int lp, parts_log;   // log2 of lanes per part and of the number of parts
    int tl, part;        // tile within a round, part
    int i0, i1, half;    // term range of the part (half: exactly four terms)
    int off, cnt;        // outputs of the tile this lane ends up with
    int rounds, n_tiles, n_out, idle;
};

// `lane` = lane of the point's warp
__device__ __forceinline__ Corr8Lane corr8_lane(int n_terms, int n_out, int lane) {
    Corr8Lane c;
    c.n_out = n_out;
    c.n_tiles = (n_out + 7) >> 3;
    c.lp = 0;
    while ((1 << c.lp) < c.n_tiles && (1 << c.lp) < 32) ++c.lp;
    int parts = 32 >> c.lp;
    c.parts_log = 0;
    while ((1 << c.parts_log) < parts) ++c.parts_log;
    int chunk = (n_terms + parts - 1) / parts;
    c.half = chunk <= 4;
    chunk = c.half ? 4 : (chunk + 7) & ~7;
    c.tl = lane & ((1 << c.lp) - 1);
    c.part = lane >> c.lp;
    c.i0 = c.part * chunk;
    c.i1 = c.i0 + chunk;
    const int end8 = (n_terms + 7) & ~7;
    if (c.i1 > end8) c.i1 = end8;
    c.idle = c.i0 >= n_terms;
    c.rounds = (c.n_tiles + (1 << c.lp) - 1) >> c.lp;
    c.off = ((c.part & 1) && c.parts_log >= 1 ? 4 : 0) + ((c.part & 2) && c.parts_log >= 2 ? 2 : 0) +
            ((c.part & 4) && c.parts_log >= 3 ? 1 : 0);
    c.cnt = 8 >> (c.parts_log < 3 ? c.parts_log : 3);
    if (c.part >> 3) c.cnt = 0;            // more than 8 parts: the upper ones hold copies
    return c;
}

#ifdef FPA_COMB_TIMING
__device__ long long g_corr_ticks[8];
#define FPA_CTICK(k)                                                           \
    do {                                                                       \
        if (blockIdx.x == 0 && threadIdx.x == 0) {                             \
            const long long now_ = clock64();                                  \
            g_corr_ticks[k] += now_ - ct_prev;                                 \
            ct_prev = now_;                                                    \
        }                                                                      \
    } while (0)
#define FPA_TICK8(k)                                  \
    do {                                              \
        if (b == 0 && gl == 0) {                      \
            const long long now_ = clock64();         \
            tk8[k] += now_ - t_prev8;                 \
            t_prev8 = now_;                           \
        }                                             \
    } while (0)
#else
#define FPA_CTICK(k) ((void)0)
#define FPA_TICK8(k) ((void)0)
#endif

// out[o] = sum_{i < n_terms} a'[i] * w[i + o] for o in [0, n_out), on the warp of one point.  The lane
// that ends up with output o writes it: TO_R -> dst[padx(M-1-o)] (the convolution result R, o = M-1-n);
// else -> dst[padx(M-1-o)] = X_o and dst[padx(M-1+o)] = conj(X_o) (the mirrored auto-correlation).
// PLOG = log2 of the number of parts when it is known at compile time (the usual plan sizes), -1 = taken
// from c.parts_log: with PLOG >= 0 the reduce-scatter and the stores are straight-line code.  Stores are
// branch-free: a lane without a valid output writes to `trash` (a spare word nobody reads).
template <int PLOG, bool TO_R>
__device__ __forceinline__ void corr8(const double2* a, const double2* w, const Corr8Lane& c, int sign_flip, int M,
                                      double2* dst, double2* trash) {
    const int LP = 1 << c.lp;
    const int plog = PLOG >= 0 ? PLOG : c.parts_log;
#ifdef FPA_COMB_TIMING
    long long ct_prev = clock64();
#endif
    for (int r = 0; r < c.rounds; ++r) {
        const int  tile = r * LP + c.tl;
        const bool live = tile < c.n_tiles && !c.idle;
        double     re[8], im[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) re[t] = im[t] = 0.0;
        FPA_CTICK(0);
        if (live) {
            if (c.half)
                roll4_mac(a, w, tile * 8, c.i0, sign_flip, re, im);
            else
                roll8_mac(a, w, tile * 8, c.i0, c.i1, sign_flip, re, im);
        }
        FPA_CTICK(1);
        // reduce-scatter over the parts (the level count is uniform over the warp: shuffles stay convergent)
        if (plog >= 1) scatter_level<8>(re, im, LP, (c.part & 1) != 0);
        if (plog >= 2) scatter_level<4>(re, im, 2 * LP, (c.part & 2) != 0);
        if (plog >= 3) scatter_level<2>(re, im, 4 * LP, (c.part & 4) != 0);
        if (plog >= 4) scatter_level<1>(re, im, 8 * LP, false);
        if (plog >= 5) scatter_level<1>(re, im, 16 * LP, false);
        FPA_CTICK(2);
        const int o0 = tile * 8 + c.off;
        constexpr int kMaxOut = PLOG < 0 ? 8 : (8 >> (PLOG < 3 ? PLOG : 3));
#pragma unroll
        for (int t = 0; t < kMaxOut; ++t) {
            const bool ok = t < c.cnt && o0 + t < c.n_out && tile < c.n_tiles;
            double2* q1 = ok ? dst + padx<kSk8>(M - 1 - (o0 + t)) : trash;
            *q1 = make_double2(re[t], im[t]);
            if (!TO_R) {
                double2* q2 = ok ? dst + padx<kSk8>(M - 1 + (o0 + t)) : trash;
                *q2 = make_double2(re[t], -im[t]);
            }
        }
        FPA_CTICK(3);
    }
}

// After the convolution of stage S: k_n = -(alpha/2) x + i*gamma*conj(E_n) R_n, the RK4 bookkeeping of that
// stage AND the phase / rotated state of the NEXT stage (or of stage 0 of the next step) for one wave, in
// one pass: the wave's state makes one shared-memory round trip per stage.  E holds exp(i*beta*z) at the
// start of the step (from S = 2 on: at its end), Eh the phase the current stage's conj(E) uses.
struct CombStep {
    double gamma, nha, hh, h, h6, h3;
};

template <int S, int K>
__device__ __forceinline__ void wave_pass(const CombSmem& s, const int (&j)[K], const int (&slot_pad)[K], const CombStep& k,
                                          bool resync_next, double z_next, bool check, int& nf) {
    // all loads of the K waves first, then K independent chains: a lane's waves overlap their latencies
    double2 r[K], e[K], x[K], acc[K], y0[K], rot[K];
#pragma unroll
    for (int q = 0; q < K; ++q) {
        r[q]   = s.R[slot_pad[q]];
        e[q]   = S == 0 ? s.E[j[q]] : s.Eh[j[q]];
        x[q]   = s.ys[j[q]];
        acc[q] = s.yn[j[q]];
        if (S != 3) y0[q] = s.y[j[q]];
        if (S == 0 || S == 2) rot[q] = s.rot[j[q]];
    }
#pragma unroll
    for (int q = 0; q < K; ++q) {
        const double fr = fma(r[q].y, e[q].y, r[q].x * e[q].x);
        const double fi = fma(r[q].y, e[q].x, -(r[q].x * e[q].y));
        const double kr = fma(k.nha, x[q].x, -(k.gamma * fi));
        const double ki = fma(k.nha, x[q].y, k.gamma * fr);
        const double wa = (S == 0 || S == 3) ? k.h6 : k.h3;
        double2      ysn, en;
        if (S == 3) {
            ysn = make_double2(fma(wa, kr, acc[q].x), fma(wa, ki, acc[q].y));    // the step's result
            s.y[j[q]] = ysn;
            s.yn[j[q]] = ysn;
            if (check && (nonfinite(ysn.x) || nonfinite(ysn.y))) nf = 1;
            if (resync_next) {   // exact phase every kCombResync steps
                double sn, cs;
                sincos(s.beta[j[q]] * z_next, &sn, &cs);
                en = make_double2(cs, sn);
            } else {
                en = e[q];       // stage 3 ran at z + h: that is the next step's starting phase
            }
            s.E[j[q]] = en;
        } else {
            const double wb = S == 2 ? k.h : k.hh;
            s.yn[j[q]] = make_double2(fma(wa, kr, acc[q].x), fma(wa, ki, acc[q].y));
            ysn = make_double2(fma(wb, kr, y0[q].x), fma(wb, ki, y0[q].y));
            if (S == 1) {
                en = e[q];       // stages 1 and 2 share the abscissa z + h/2
            } else {             // S = 0 -> z + h/2 ; S = 2 -> z + h
                en = make_double2(fma(-e[q].y, rot[q].y, e[q].x * rot[q].x), fma(e[q].x, rot[q].y, e[q].y * rot[q].x));
                s.Eh[j[q]] = en;
                if (S == 2) s.E[j[q]] = en;
            }
        }
        s.ys[j[q]] = ysn;
        s.At[slot_pad[q]] = make_double2(fma(-ysn.y, en.y, ysn.x * en.x), fma(ysn.x, en.y, ysn.y * en.x));
    }
}

// The waves a lane owns (gl, gl + LW, ...; at most OWN of them) in pairs, so that two chains share one
// straight-line region; a lane of the last, partly filled round handles its single wave alone.
template <int S, int OWN, int LW>
__device__ __forceinline__ void wave_passes(const CombSmem& s, int gl, int N, const int (&slot_pad)[OWN], const CombStep& k,
                                            bool resync_next, double z_next, bool check, int& nf) {
#pragma unroll
    for (int q = 0; q < OWN; q += 2) {
        const int j0 = gl + q * LW, j1 = j0 + LW;
        if (OWN - q >= 2 && j1 < N) {
            const int jj[2] = {j0, j1}, sp[2] = {slot_pad[q], slot_pad[q + 1 < OWN ? q + 1 : q]};
            wave_pass<S, 2>(s, jj, sp, k, resync_next, z_next, check, nf);
        } else if (j0 < N) {
            const int jj[1] = {j0}, sp[1] = {slot_pad[q]};
            wave_pass<S, 1>(s, jj, sp, k, resync_next, z_next, check, nf);
        }
    }
}

// One warp per scan point, up to 8 points per CTA; the warps of a CTA never wait for each other.
template <int PLOG>
__global__ void __launch_bounds__(kCombThreads, 2) nwave_comb8_kernel(const CombParams p) {
    extern __shared__ __align__(16) double comb_smem_raw[];
    constexpr int LW = 32;                   // lanes of a point
    constexpr int kOwn = 128 / LW;           // waves a lane owns at most (N <= 128)
    const int     N = p.n_waves, M = p.span;
    const int     gl = threadIdx.x & 31;     // lane within the point
    const int     sub = threadIdx.x >> 5;    // point slot inside the CTA
    const int     ppc = blockDim.x >> 5;     // points per CTA
    const int64_t b = (int64_t)blockIdx.x * ppc + sub;
    if (b >= p.n_points) return;             // whole warps beyond the batch leave
    CombSmem s = comb_carve(comb_smem_raw + (size_t)sub * comb_point_doubles(N, M, kSk8), N, M, kSk8);

    const int    n_steps = p.n_steps;
    const double z0 = p.z0;
    const double h = (p.z_max - z0) / (double)n_steps;
    CombStep     ks;
    ks.gamma = p.gamma[b * p.gamma_stride];
    ks.nha   = -0.5 * p.alpha[b * p.alpha_stride];
    ks.h     = h;
    ks.hh    = 0.5 * h;
    ks.h6    = h / 6.0;
    ks.h3    = ks.h6 + ks.h6;

    const int words = comb_seq_words(M, kSk8);
    for (int m = gl; m < words; m += LW) {
        s.At[m] = make_double2(0.0, 0.0);  // empty grid slots and the padding stay 0
        s.Y[m]  = make_double2(0.0, 0.0);
    }
    for (int m = gl; m < comb_r_words(M); m += LW) s.R[m] = make_double2(0.0, 0.0);
    __syncwarp();
    // per-wave state; stage 0 of the first step: exact phase at z0, ys = yn = y, At = y * E
    for (int j = gl; j < N; j += LW) {
        const double bj = p.beta[b * p.beta_stride * N + j];
        s.beta[j] = bj;
        const double2 v = (reinterpret_cast<const double2*>(p.A0) + b * p.A0_stride * N)[j];
        s.y[j] = s.ys[j] = s.yn[j] = v;
        double sn, cs;
        sincos(bj * ks.hh, &sn, &cs);
        s.rot[j] = make_double2(cs, sn);
        sincos(bj * z0, &sn, &cs);
        s.E[j] = s.Eh[j] = make_double2(cs, sn);
        s.At[padx<kSk8>(p.slot[j])] = make_double2(fma(-v.y, sn, v.x * cs), fma(v.x, sn, v.y * cs));
    }

    double2* tr = p.A_trace ? reinterpret_cast<double2*>(p.A_trace) + b * p.n_saved * N : nullptr;
    if (tr) {
        for (int j = gl; j < N; j += LW) tr[j] = s.y[j];
        tr += N;
    }
    double pm[kOwn];
#pragma unroll
    for (int q = 0; q < kOwn; ++q) {
        const int j = gl + q * LW;
        pm[q] = (p.Pmax && j < N) ? fma(s.y[j].y, s.y[j].y, s.y[j].x * s.y[j].x) : 0.0;
    }
    int      save_ctr = p.save_every;
    int32_t  bad = FPA_POINT_OK;
    int      nf = 0;                                    // a component of the state entering the step is not finite
    if (p.check)
        for (int j = gl; j < N; j += LW) nf |= (nonfinite(s.y[j].x) || nonfinite(s.y[j].y)) ? 1 : 0;
    double2* const Yc = s.Y;                            // Yc[padx(q)] = X_{M-1-q}, q in [0, 2M-2]
    double2* const trash = s.R + comb_r_words(M) - 1;   // spare word: target of the stores of lanes without an output
    // padded positions of this lane's waves on the grid (At, R) -- fixed for the whole run
    int slot_pad[kOwn];
#pragma unroll
    for (int q = 0; q < kOwn; ++q) slot_pad[q] = gl + q * LW < N ? padx<kSk8>(p.slot[gl + q * LW]) : 0;
    const Corr8Lane cl = corr8_lane(M, M, gl);          // both correlations of a stage: M outputs, M terms
#ifdef FPA_COMB_TIMING
    long long tk8[8] = {0, 0, 0, 0, 0, 0, 0, 0}, t_prev8 = clock64();
#endif

    for (int i = 0; i < n_steps; ++i) {
        if (p.check && i > 0 && bad == FPA_POINT_OK) {
            if (__ballot_sync(0xffffffffu, nf) != 0u) bad = i - 1;  // the state produced by step i-1 was not finite
        }
        nf = 0;
        const bool   resync_next = ((i + 1) % kCombResync) == 0;
        const double z_next = fma((double)(i + 1), h, z0);
        for (int stage = 0; stage < 4; ++stage) {
            FPA_TICK8(0);
            __syncwarp();
            // ---- X_d = sum_m conj(At[m]) At[m+d], d in [0, M), stored mirrored: Yc[M-1-d] = X_d, Yc[M-1+d] = conj(X_d)
            corr8<PLOG, false>(s.At, s.At, cl, (int)0x80000000, M, Yc, trash);
            FPA_TICK8(1);
            __syncwarp();
            // ---- R_n = sum_k At[k] X_{n-k} = sum_k At[k] Yc[(M-1-n) + k]; output o = M-1-n
            corr8<PLOG, true>(s.At, Yc, cl, 0, M, s.R, trash);
            FPA_TICK8(2);
            __syncwarp();
            // ---- k, RK4 bookkeeping and the next stage's phases / rotated state: one pass per wave, straight-line
            // code per stage (one uniform jump instead of a chain of stage tests)
            switch (stage) {
            case 0: wave_passes<0, kOwn, LW>(s, gl, N, slot_pad, ks, false, 0.0, false, nf); break;
            case 1: wave_passes<1, kOwn, LW>(s, gl, N, slot_pad, ks, false, 0.0, false, nf); break;
            case 2: wave_passes<2, kOwn, LW>(s, gl, N, slot_pad, ks, false, 0.0, false, nf); break;
            default: wave_passes<3, kOwn, LW>(s, gl, N, slot_pad, ks, resync_next, z_next, p.check != 0, nf); break;
            }
            FPA_TICK8(3);
        }
        if (--save_ctr == 0) {
            save_ctr = p.save_every;
            if (tr) {
                for (int j = gl; j < N; j += LW) tr[j] = s.y[j];
                tr += N;
            }
            if (p.Pmax) {
#pragma unroll
                for (int q = 0; q < kOwn; ++q) {
                    const int j = gl + q * LW;
                    if (j < N) {
                        const double P = fma(s.y[j].y, s.y[j].y, s.y[j].x * s.y[j].x);
                        pm[q] = (P != P || pm[q] != pm[q]) ? qnan() : fmax(pm[q], P);
                    }
                }
            }
        }
    }
    if (p.check && bad == FPA_POINT_OK) {
        if (__ballot_sync(0xffffffffu, nf) != 0u) bad = n_steps - 1;
    }
#ifdef FPA_COMB_TIMING
    if (b == 0 && gl == 0) {
        const double st = 4.0 * n_steps;
        printf("comb8<PLOG=%d> cycles per stage: other %.0f | auto-correlation %.0f | convolution %.0f | wave pass %.0f\n",
               PLOG, tk8[0] / st, tk8[1] / st, tk8[2] / st, tk8[3] / st);
        printf("   per correlation: setup %.0f | window + terms %.0f | reduce-scatter %.0f | stores %.0f\n", g_corr_ticks[0] / (2 * st),
               g_corr_ticks[1] / (2 * st), g_corr_ticks[2] / (2 * st), g_corr_ticks[3] / (2 * st));
        for (int k = 0; k < 8; ++k) g_corr_ticks[k] = 0;
    }
#endif
    if (p.status && gl == 0) p.status[b] = bad;
    if (p.A_end) {
        double2* o = reinterpret_cast<double2*>(p.A_end) + b * N;
        for (int j = gl; j < N; j += LW) o[j] = s.y[j];
    }
    if (p.Pmax) {
#pragma unroll
        for (int q = 0; q < kOwn; ++q) {
            const int j = gl + q * LW;
            if (j < N) p.Pmax[b * N + j] = pm[q];
        }
    }
}

template <int PLOG>
static cudaError_t comb8_launch_p(const CombParams& p, int sms, cudaStream_t st) {
    const size_t smem_point = comb_point_doubles(p.n_waves, p.span, kSk8) * sizeof(double);
    // points (= warps) per CTA: as many (up to 8) as fit the shared memory and still leave two CTAs for every SM,
    // so that a mid-sized batch spreads over the whole chip
    int ppc = kCombThreads / 32;
    while (ppc > 1 && (smem_point * ppc > 200 * 1024 || (p.n_points + ppc - 1) / ppc < 2 * (int64_t)sms)) ppc >>= 1;
    const size_t smem = smem_point * ppc;
    cudaError_t  e = cudaFuncSetAttribute(nwave_comb8_kernel<PLOG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const unsigned blocks = (unsigned)((p.n_points + ppc - 1) / ppc);
    nwave_comb8_kernel<PLOG><<<blocks, 32 * ppc, smem, st>>>(p);
    return cudaGetLastError();
}

// The number of parts of the term range follows from the plan's span (tiles of 8 outputs, 32 lanes): the usual
// sizes get the kernel with a compile-time reduce-scatter, everything else the generic one.
static cudaError_t comb8_launch(const CombParams& p, int sms, cudaStream_t st) {
    const int tiles = (p.span + 7) >> 3;
    int       lp = 0;
    while ((1 << lp) < tiles && (1 << lp) < 32) ++lp;
    const int plog = 5 - lp;
    if (plog == 1) return comb8_launch_p<1>(p, sms, st);   // span 65..128
    if (plog == 2) return comb8_launch_p<2>(p, sms, st);   // span 33..64
    return comb8_launch_p<-1>(p, sms, st);
}

static cudaError_t comb_launch(const CombParams& p, cudaStream_t st) {
    const size_t smem = comb_point_doubles(p.n_waves, p.span, kSk) * sizeof(double);
    cudaError_t  e = cudaFuncSetAttribute(nwave_comb_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    nwave_comb_kernel<<<(unsigned)p.n_points, 32 * kCtaWarps, smem, st>>>(p);
    return cudaGetLastError();
}

int nwave_check(const fpa_nwave_desc* d);          // nwave.cu
int nwave_check_aligned(const fpa_nwave_desc* d);  // nwave.cu

// The limits of the convolution form: n_waves <= 128, grid_span <= 512.
bool nwave_comb_fits(const fpa_nwave_desc* d) { return d->n_waves <= 128 && d->grid_span <= 512; }

// d->grid_slot: device pointer to the N grid slots; span = number of grid slots covered.
int nwave_comb_launch(const fpa_nwave_desc* d, cudaStream_t st) {
    int rc = nwave_check(d);
    if (rc == FPA_OK) rc = nwave_check_aligned(d);
    if (rc != FPA_OK) return rc;
    FPA_REQUIRE(d->n_points < 2147483647LL, "bad n_points");
    if (!nwave_comb_fits(d)) {
        set_error("comb kernel limits: n_waves <= 128, grid_span <= 512 (got %d, %d)", d->n_waves, d->grid_span);
        return FPA_ERR_UNSUPPORTED;
    }
    FPA_REQUIRE(d->grid_span >= d->n_waves, "grid_span must cover all waves");
    if (d->n_points == 0) return FPA_OK;
    const int N = d->n_waves, M = d->grid_span;
    CombParams p;
    p.n_points     = d->n_points;
    p.n_waves      = N;
    p.span         = M;
    p.beta_stride  = (int)d->beta_stride;
    p.gamma_stride = (int)d->gamma_stride;
    p.alpha_stride = (int)d->alpha_stride;
    p.A0_stride    = (int)d->A0_stride;
    p.beta         = d->beta;
    p.gamma        = d->gamma;
    p.alpha        = d->alpha;
    p.A0           = d->A0;
    p.slot         = d->grid_slot;
    p.z0           = d->z0;
    p.z_max        = d->z_max;
    p.n_steps      = (int)d->n_steps;
    p.save_every   = (int)(d->save_every > d->n_steps ? d->n_steps + 1 : d->save_every);
    p.n_saved      = fpa_n_saved(d->n_steps, d->save_every);
    p.A_trace      = (d->flags & FPA_OUT_TRACE) ? d->A_trace : nullptr;
    p.A_end        = (d->flags & FPA_OUT_END) ? d->A_end : nullptr;
    p.Pmax         = (d->flags & FPA_OUT_PMAX) ? d->Pmax : nullptr;
    p.status       = d->status;
    p.check        = (d->flags & FPA_CHECK_NAN) ? 1 : 0;

    int          dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // one warp per point once the batch can give every SM sub-partition a point of its own (and 8 points
    // fit into a CTA's shared memory); below that one CTA per point, for latency
    const size_t smem_w1 = comb_point_doubles(N, M, kSk8) * sizeof(double);
    const bool   wide = d->n_points >= 4 * (int64_t)sms && smem_w1 <= 200 * 1024;
    const cudaError_t e = wide ? comb8_launch(p, sms, st) : comb_launch(p, st);
    if (e != cudaSuccess) return cuda_fail(e, "nwave_comb_kernel launch");
    return FPA_OK;
}

}  // namespace fpa

extern "C" double fpa_nwave_comb_flops_per_step(int32_t n_waves, int32_t grid_span) {
    // per RHS: X_d for d >= 0 over the non-zero products, M^2/2 complex MACs (8 flops) = 4*M^2; the
    // convolution with X on the N occupied slots, 8*N*M; 30*N for phases, rotation, conj(E)*R and the
    // assembly.  Per step 4 RHS + 26*N for the RK4 combination.  (The kernel executes the regular,
    // zero-padded M^2 + M^2 form: the padding is not credited.)
    const double M = grid_span, N = n_waves;
    return 4.0 * (4.0 * M * M + 8.0 * N * M + 30.0 * N) + 26.0 * N;
}
