// api.cu -- the extern "C" surface of libfpa_b200.so (declared in include/fpa_b200.h).
//
// Everything in this file is plumbing around the kernels of yaman4.cu / frontend.cu / nwave.cu /
// linear.cu / probe.cu: argument checks, device selection, a grow-only device workspace for the
// host-pointer entry points, H2D / D2H staging and error text.  No arithmetic of the hot path
// lives here and nothing here can run the path on the CPU: without a CUDA device every compute
// entry point returns FPA_ERR_NO_DEVICE.
#include "fpa_common.cuh"

#include <math.h>
#include <stdarg.h>

#include <map>
#include <tuple>
#include <vector>

namespace fpa {

// launchers and descriptor checks implemented next to their kernels
int yaman4_check(const fpa_yaman4_desc* d);
int yaman4_launch(const fpa_yaman4_desc* d, cudaStream_t st);
int yaman4_transfer_check(const fpa_yaman4_desc* d, const fpa_transfer_out* t);
int yaman4_transfer_launch(const fpa_yaman4_desc* d, const fpa_transfer_out* t, cudaStream_t st);
int yaman4_transfer_sweep_launch(const fpa_sweep_desc* d, const fpa_transfer_out* t, cudaStream_t st);
int yaman4_rhs_launch(int64_t B, const double* z, const double* A, const double* gamma,
                      const double* alpha, const double* dbeta, double* dA, cudaStream_t st);
int plan_launch(const fpa_plan_desc* d, double* dbeta_masked, cudaStream_t st);
int sweep_grid_points(const fpa_sweep_desc* d, int64_t* n_grid);
int yaman4_sweep_launch(const fpa_sweep_desc* d, void* scratch, int64_t scratch_bytes, cudaStream_t st);
int phase_sweep_check(const fpa_phase_sweep_desc* d);
int yaman4_phase_sweep_launch(const fpa_phase_sweep_desc* d, void* scratch, int64_t scratch_bytes, cudaStream_t st);
int phase_reduce_launch(int64_t G, int K, const double* gain, double* gmax, double* gmin, int32_t* imax, int32_t* imin,
                        int32_t* nfin, cudaStream_t st);
int64_t yaman4_scratch_bytes(int64_t n_points);
int64_t yaman4_phase_scratch_bytes(int64_t n_points);
int linear_launch(int64_t B, int dim, const double* y0, const double* lam, double z0, double z_max,
                  int64_t n_steps, int64_t save_every, const double* z_grid, uint32_t flags,
                  double* y_trace, double* y_end, int32_t* bad_scratch, int32_t* status,
                  cudaStream_t st);
int nwave_check(const fpa_nwave_desc* d);
int nwave_launch(const fpa_nwave_desc* d, cudaStream_t st);
bool nwave_comb_fits(const fpa_nwave_desc* d);
int nwave_comb_launch(const fpa_nwave_desc* d, cudaStream_t st);
int probe_run(int device, int iters, double* tflops, double* ms_out);

#define FPA_TRY(expr)                  \
    do {                               \
        int rc__ = (expr);             \
        if (rc__ != FPA_OK) return rc__; \
    } while (0)

// ----------------------------------------------------------------- error text (per host thread)
static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
    set_error("CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
    // leave the runtime's sticky "last error" clean for the next call
    cudaGetLastError();
    if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) return FPA_ERR_NO_DEVICE;
    return FPA_ERR_CUDA;
}

// FPA_ERR_NO_DEVICE unless a CUDA device is visible; `why` completes the error text.
static int need_device(const char* why = "libfpa_b200 has no CPU path") {
    if (fpa_device_count() > 0) return FPA_OK;
    set_error("no CUDA device is visible: %s", why);
    return FPA_ERR_NO_DEVICE;
}

int use_device(int device) {
    FPA_TRY(need_device());
    const int n = fpa_device_count();
    if (device < 0 || device >= n) {
        set_error("device %d out of range [0, %d)", device, n);
        return FPA_ERR_INVALID;
    }
    FPA_CUDA(cudaSetDevice(device));
    return FPA_OK;
}

// ----------------------------------------------------------------- grow-only workspace
struct Slab {
    void*  ptr = nullptr;
    size_t cap = 0;
};
static thread_local std::map<std::pair<int, int>, Slab> g_slabs;

int workspace(int device, int slot, size_t bytes, void** out) {
    Slab& s = g_slabs[std::make_pair(device, slot)];
    if (bytes > s.cap) {
        if (s.ptr) {
            FPA_CUDA(cudaDeviceSynchronize());
            FPA_CUDA(cudaFree(s.ptr));
            s.ptr = nullptr;
            s.cap = 0;
        }
        // round up so that slowly growing batches do not reallocate every call
        size_t want = (bytes + ((size_t)1 << 20) - 1) & ~(((size_t)1 << 20) - 1);
        FPA_CUDA(cudaMalloc(&s.ptr, want));
        s.cap = want;
    }
    *out = s.ptr;
    return FPA_OK;
}

static int up(void* dst, const void* src, size_t bytes, cudaStream_t st) {
    if (bytes == 0) return FPA_OK;
    FPA_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
    return FPA_OK;
}
static int down(void* dst, const void* src, size_t bytes, cudaStream_t st) {
    if (bytes == 0 || dst == nullptr) return FPA_OK;
    FPA_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st));
    return FPA_OK;
}

// Address at which a kernel can write `host_ptr` directly (pinned / registered host memory under
// unified addressing), or nullptr for pageable memory.  The reduce-mode sweep writes its 24 bytes
// per scan point straight into such buffers while it runs: no staging copy after the kernel.
template <typename T>
static T* mapped(T* host_ptr) {
    if (host_ptr == nullptr) return nullptr;
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, host_ptr) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    if (at.type != cudaMemoryTypeHost || at.devicePointer == nullptr) return nullptr;
    return static_cast<T*>(at.devicePointer);
}

// One non-blocking stream per (host thread, device) for the host-pointer entry points.
static thread_local std::map<int, cudaStream_t> g_streams;
static int host_stream(int device, cudaStream_t* st) {
    auto it = g_streams.find(device);
    if (it == g_streams.end()) {
        cudaStream_t s;
        FPA_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        it = g_streams.emplace(device, s).first;
    }
    *st = it->second;
    return FPA_OK;
}

// ----------------------------------------------------------------- host-pointer calls
// A host-pointer call in flight: its stream (NULL: nothing was queued) and the copies of results into the
// caller's arrays that are still to be queued after the kernel.
struct Pending {
    struct Copy {
        void*       host;
        const void* dev;
        size_t      bytes;
    };
    cudaStream_t      st = nullptr;
    std::vector<Copy> copies;
};

static int collect(const Pending& p, int device) {
    if (!p.st) return FPA_OK;
    FPA_TRY(use_device(device));
    for (const Pending::Copy& c : p.copies) FPA_TRY(down(c.host, c.dev, c.bytes, p.st));
    return FPA_OK;
}

// The end of a single-device call: queue the result copies, wait for the stream.
static int finish(const Pending& p, int device) {
    FPA_TRY(collect(p, device));
    if (p.st) FPA_CUDA(cudaStreamSynchronize(p.st));
    return FPA_OK;
}

template <typename Desc>
static int run_on_device(int (*launch)(const Desc*, int, Pending*), const Desc* d, int device) {
    Pending p;
    FPA_TRY(launch(d, device, &p));
    return finish(p, device);
}

// Alignment the kernels need of the arrays they access with 16-byte vector loads and stores (complex128 data, rows of
// four maxima).
constexpr size_t kVecAlign = 16;

// The device buffers of one host-pointer call, carved in 256-byte aligned pieces from one workspace slot.
// stage() runs the entry's declaring code twice: a sizing pass that only adds up the pieces, then, with the
// workspace at that size, the placing pass that hands out addresses, queues the uploads and records the copies
// back.  The workspace size and the carve thus come from one list of declarations.
struct Staging {
    char*              base = nullptr;  // NULL during the sizing pass
    size_t             off  = 0;
    Pending*           pend = nullptr;
    std::vector<void*> maps;            // out(): the mapped address of each call, found in the sizing pass
    size_t             n_out = 0;
    int                rc = FPA_OK;     // first failed upload

    // a device-only buffer of n elements
    template <class T>
    T* tmp(size_t n) {
        T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
        off += (n * sizeof(T) + 255) & ~(size_t)255;
        return p;
    }
    // a buffer holding the n elements at `host`, uploaded before the kernel
    template <class T>
    T* in(const T* host, size_t n) {
        T* p = tmp<T>(n);
        if (base && rc == FPA_OK) rc = up(p, host, n * sizeof(T), pend->st);
        return p;
    }
    // where the kernel writes the n elements meant for `host`: the device address of `host` when may_map is set,
    // `host` is page-locked and `host` is aligned to `align` bytes, the width of the kernel's stores into it (16
    // for complex128 data and rows of maxima, which numpy only aligns to 8); else a buffer that is copied to `host`
    // after the kernel (a NULL `host` gets none)
    template <class T>
    T* out(T* host, size_t n, bool may_map, size_t align = alignof(T)) {
        if (!base) maps.push_back(may_map && reinterpret_cast<uintptr_t>(host) % align == 0 ? mapped(host) : nullptr);
        if (T* m = static_cast<T*>(maps[n_out++])) return m;
        T* p = tmp<T>(n);
        if (base && host) pend->copies.push_back({host, p, n * sizeof(T)});
        return p;
    }
};

template <typename Declare>
static int stage(int device, int slot, Pending* pend, Declare declare) {
    Staging s;
    s.pend = pend;
    declare(s);
    void* ws = nullptr;
    FPA_TRY(workspace(device, slot, s.off, &ws));
    FPA_TRY(host_stream(device, &pend->st));
    s.base  = static_cast<char*>(ws);
    s.off   = 0;
    s.n_out = 0;
    declare(s);
    return s.rc;
}

// Contiguous share of n items for part k of `parts`: sizes differ by at most one.
static void balanced_range(int64_t n, int parts, int k, int64_t* lo, int64_t* hi) {
    const int64_t base = n / parts, extra = n % parts;
    *lo = (int64_t)k * base + (k < extra ? k : extra);
    *hi = *lo + base + (k < extra ? 1 : 0);
}

// Drive several devices from one host thread: every part's kernel is put in flight first (a copy into
// pageable memory blocks the host until the kernel is done), then the result copies are queued, then
// every stream is synchronised -- also after an error on a later device.  A device that is listed twice
// shares one workspace and stream, so the earlier part's copies are queued before its next kernel may
// overwrite the staging buffers.
template <typename Launch>
static int run_on_devices(int n_devices, const int* devices, Launch launch) {
    std::vector<Pending> pend((size_t)n_devices);
    bool collected[64] = {};
    int  used = 0, rc = FPA_OK;
    for (int k = 0; k < n_devices && rc == FPA_OK; ++k) {
        used = k + 1;
        for (int j = 0; j < k && rc == FPA_OK; ++j) {
            if (devices[j] == devices[k] && pend[j].st && !collected[j]) {
                rc = collect(pend[j], devices[j]);
                collected[j] = true;
            }
        }
        if (rc == FPA_OK) rc = launch(k, &pend[k]);
    }
    for (int k = 0; k < used && rc == FPA_OK; ++k)
        if (!collected[k]) rc = collect(pend[k], devices[k]);
    for (int k = 0; k < used; ++k) {
        if (!pend[k].st) continue;
        if (cudaSetDevice(devices[k]) != cudaSuccess || cudaStreamSynchronize(pend[k].st) != cudaSuccess) {
            if (rc == FPA_OK) rc = cuda_fail(cudaGetLastError(), "multi-device call: stream synchronize");
        }
    }
    return rc;
}

static int check_devices(int n_devices, const int* devices) {
    FPA_REQUIRE(n_devices >= 1 && n_devices <= 64 && devices != nullptr, "need 1..64 device ordinals");
    return FPA_OK;
}

// ----------------------------------------------------------------- 4-wave batch
// t != NULL: the transfer batch (jac staged like the other outputs, no scheduler scratch).
static int batch_host_launch(const fpa_yaman4_desc* d, int device, Pending* p, const fpa_transfer_out* t) {
    FPA_TRY(t ? yaman4_transfer_check(d, t) : yaman4_check(d));
    FPA_TRY(use_device(device));
    const size_t B = (size_t)d->n_points;
    if (B == 0) return FPA_OK;
    const size_t     ns      = (size_t)fpa_n_saved(d->n_steps, d->save_every);
    const size_t     n_sched = t ? 0 : (size_t)yaman4_scratch_bytes((int64_t)B);
    const size_t     nc      = t ? (size_t)__builtin_popcount(t->columns) : 0;
    fpa_yaman4_desc  dd;
    fpa_transfer_out tt = {};
    // outputs in pinned host memory are written by the kernel itself (no staging, no copy)
    FPA_TRY(stage(device, 0, p, [&](Staging& s) {
        dd         = *d;
        dd.dbeta   = s.in(d->dbeta, B);
        dd.gamma   = s.in(d->gamma, d->gamma_stride ? B : 1);
        dd.alpha   = s.in(d->alpha, d->alpha_stride ? B : 1);
        dd.A0      = s.in(d->A0, (d->A0_stride ? B : 1) * 8);
        dd.z_grid  = d->z_grid ? s.in(d->z_grid, (size_t)d->n_steps + 1) : nullptr;
        dd.A_trace = (d->flags & FPA_OUT_TRACE) ? s.out(d->A_trace, B * ns * 8, true, kVecAlign) : nullptr;
        dd.A_end   = (d->flags & FPA_OUT_END) ? s.out(d->A_end, B * 8, true, kVecAlign) : nullptr;
        dd.Pmax    = (d->flags & FPA_OUT_PMAX) ? s.out(d->Pmax, B * 4, true, kVecAlign) : nullptr;
        dd.status  = s.out(d->status, B, true);  // the kernel always gets one
        dd.scratch = s.tmp<char>(n_sched);
        if (t) {
            tt     = *t;
            tt.jac = s.out(t->jac, B * 8 * nc, true);
        }
    }));
    dd.scratch_bytes = (int64_t)n_sched;
    if (d->gamma_stride == 0 && d->alpha_stride == 0) {  // host pointers: the broadcast values are known here
        dd.flags |= FPA_UNIFORM_PHYSICS;
        dd.gamma_uniform = d->gamma[0];
        dd.alpha_uniform = d->alpha[0];
    } else {
        dd.flags &= ~FPA_UNIFORM_PHYSICS;
    }
    return t ? yaman4_transfer_launch(&dd, &tt, p->st) : yaman4_launch(&dd, p->st);
}

static int batch_host_launch(const fpa_yaman4_desc* d, int device, Pending* p) {
    return batch_host_launch(d, device, p, nullptr);
}

// Part k of a batch: a contiguous range of the points, sizes differing by at most one.
static fpa_yaman4_desc batch_part(const fpa_yaman4_desc* d, int n_devices, int k, int64_t* lo) {
    int64_t hi;
    balanced_range(d->n_points, n_devices, k, lo, &hi);
    const int64_t   ns   = fpa_n_saved(d->n_steps, d->save_every);
    fpa_yaman4_desc part = *d;
    part.n_points = hi - *lo;
    part.dbeta    = d->dbeta + *lo;
    part.gamma    = d->gamma + *lo * d->gamma_stride;
    part.alpha    = d->alpha + *lo * d->alpha_stride;
    part.A0       = d->A0 + *lo * d->A0_stride * 8;
    if (d->A_trace) part.A_trace = d->A_trace + *lo * ns * 8;
    if (d->A_end) part.A_end = d->A_end + *lo * 8;
    if (d->Pmax) part.Pmax = d->Pmax + *lo * 4;
    if (d->status) part.status = d->status + *lo;
    return part;
}

// ----------------------------------------------------------------- sweeps
// Phase sweep: the sweep kernel, then the per-grid-point reductions over its gain map on the same stream.
static int phase_sweep_dev(const fpa_phase_sweep_desc* d, void* scratch, int64_t scratch_bytes, cudaStream_t st) {
    FPA_TRY(yaman4_phase_sweep_launch(d, scratch, scratch_bytes, st));
    const fpa_sweep_desc& w = d->sweep;
    const int64_t G = (w.first_point == 0 && w.n_sub_points == 0) ? w.plan.n1 * w.plan.n3 : w.n_sub_points;
    return phase_reduce_launch(G, (int)d->n_phases, w.gain_lin, d->gain_max, d->gain_min, d->idx_max, d->idx_min,
                               d->n_finite, st);
}

// The host checks of a sweep and the grid points it runs (*G); selects the device.
static int sweep_host_points(const fpa_sweep_desc* d, int device, int64_t* G) {
    const fpa_plan_desc& pl = d->plan;
    FPA_REQUIRE(pl.n1 >= 0 && pl.n3 >= 0, "grid sizes must be >= 0");
    FPA_REQUIRE(pl.lambda1 && pl.lambda2 && pl.lambda3, "wavelength axes must be set");
    FPA_TRY(sweep_grid_points(d, G));
    return use_device(device);
}

// The buffers of a sweep of B grid points and P runs (P = B*K for a phase sweep).  Outputs in pinned host
// memory are written by the kernel itself (each thread stores its results when it finishes, so the PCIe
// traffic hides behind the integration of the other points; measured with 8 GPUs storing into one host at
// once: 44.1 ms per 8e6-point sweep against 46.0 ms with staging and copies).  Pageable outputs go through
// the device workspace and a copy.  `map_gain` false: the gain map stays in device memory, where the phase
// sweep's reduction kernel reads it.
static void stage_sweep(Staging& s, const fpa_sweep_desc* d, fpa_sweep_desc& dd, size_t B, size_t P, bool map_gain) {
    const fpa_plan_desc& pl = d->plan;
    const size_t         n1 = (size_t)pl.n1, n3 = (size_t)pl.n3;
    dd              = *d;
    dd.n_peers      = 0;  // peer maps are device pointers: a feature of the _dev entry
    dd.plan.lambda1 = s.in(pl.lambda1, n1);
    dd.plan.lambda2 = s.in(pl.lambda2, pl.lambda2_stride ? n1 : 1);
    dd.plan.lambda3 = s.in(pl.lambda3, n3);
    dd.plan.omega   = pl.omega ? s.out(pl.omega, B * 4, false) : nullptr;
    dd.plan.dbeta   = s.out(pl.dbeta, B, true);
    dd.plan.valid   = s.out(pl.valid, B, true);
    dd.gain_lin     = s.out(d->gain_lin, P, map_gain);
    dd.Pmax         = d->Pmax ? s.out(d->Pmax, P * 4, true, kVecAlign) : nullptr;
    dd.A_end        = d->A_end ? s.out(d->A_end, P * 8, true, kVecAlign) : nullptr;
    dd.status       = s.out(d->status, P, true);
}

// t != NULL: the transfer sweep (gain_lin may be NULL, jac staged like the other outputs, no scheduler scratch).
static int sweep_host_launch(const fpa_sweep_desc* d, int device, Pending* p, const fpa_transfer_out* t) {
    FPA_REQUIRE(d != nullptr, "sweep descriptor is NULL");
    FPA_REQUIRE(t == nullptr || t->columns != 0, "columns must be a non-zero mask of bits 0..7 (got 0)");
    int64_t G;
    FPA_TRY(sweep_host_points(d, device, &G));
    if (G == 0) return FPA_OK;
    FPA_REQUIRE(d->gain_lin != nullptr || t, "gain_lin must be set");
    const size_t     n_sched = t ? 0 : (size_t)yaman4_scratch_bytes(G);
    const size_t     nc      = t ? (size_t)__builtin_popcount(t->columns) : 0;
    fpa_sweep_desc   dd;
    fpa_transfer_out tt = {};
    char*            sched;
    FPA_TRY(stage(device, 3, p, [&](Staging& s) {
        stage_sweep(s, d, dd, (size_t)G, (size_t)G, true);
        sched = s.tmp<char>(n_sched);
        if (t) {
            tt     = *t;
            tt.jac = s.out(t->jac, (size_t)G * 8 * nc, true);
        }
    }));
    if (!t) return yaman4_sweep_launch(&dd, sched, (int64_t)n_sched, p->st);
    if (d->gain_lin == nullptr) dd.gain_lin = nullptr;  // no gain map: the seed power may be 0
    dd.n_peers = d->n_peers;                            // refused by the launcher when set
    return yaman4_transfer_sweep_launch(&dd, &tt, p->st);
}

static int sweep_host_launch(const fpa_sweep_desc* d, int device, Pending* p) {
    return sweep_host_launch(d, device, p, nullptr);
}

// K = n_phases runs per grid point: the per-run arrays hold G*K entries, the plan outputs and the reductions G.
static int phase_sweep_host_launch(const fpa_phase_sweep_desc* d, int device, Pending* p) {
    FPA_TRY(phase_sweep_check(d));
    int64_t G;
    FPA_TRY(sweep_host_points(&d->sweep, device, &G));
    if (G == 0) return FPA_OK;
    const size_t         K = (size_t)d->n_phases, P = (size_t)G * K;
    const size_t         n_sched = (size_t)yaman4_phase_scratch_bytes((int64_t)P);
    fpa_phase_sweep_desc pd;
    char*                sched;
    FPA_TRY(stage(device, 3, p, [&](Staging& s) {
        pd = *d;
        stage_sweep(s, &d->sweep, pd.sweep, (size_t)G, P, false);  // a NULL gain_lin stays in the workspace
        pd.A0_table = s.in(d->A0_table, K * 8);
        pd.gain_max = d->gain_max ? s.out(d->gain_max, (size_t)G, false) : nullptr;
        pd.gain_min = d->gain_min ? s.out(d->gain_min, (size_t)G, false) : nullptr;
        pd.idx_max  = d->idx_max ? s.out(d->idx_max, (size_t)G, false) : nullptr;
        pd.idx_min  = d->idx_min ? s.out(d->idx_min, (size_t)G, false) : nullptr;
        pd.n_finite = d->n_finite ? s.out(d->n_finite, (size_t)G, false) : nullptr;
        sched       = s.tmp<char>(n_sched);
    }));
    return phase_sweep_dev(&pd, sched, (int64_t)n_sched, p->st);
}

// The checks of a multi-device sweep; the grid is split over the devices (see the header).
static int sweep_multi_check(const fpa_sweep_desc* d, int n_devices, const int* devices) {
    FPA_TRY(check_devices(n_devices, devices));
    FPA_REQUIRE(d->plan.n1 >= 0 && d->plan.n3 >= 0, "grid sizes must be >= 0");
    FPA_REQUIRE(d->first_point == 0 && d->n_sub_points == 0, "the multi-device sweep splits the whole grid itself");
    return FPA_OK;
}

// Part k of the grid: a contiguous range of the FLATTENED grid, sizes differing by at most one (a 1-D sweep,
// n1 = 1, or a grid with fewer pump rows than devices still uses every device); K runs per grid point.
static fpa_sweep_desc sweep_part(const fpa_sweep_desc* d, int n_devices, int k, int64_t K, int64_t* lo) {
    int64_t hi;
    balanced_range(d->plan.n1 * d->plan.n3, n_devices, k, lo, &hi);
    fpa_sweep_desc part = *d;
    part.first_point  = *lo;
    part.n_sub_points = hi - *lo;
    if (d->plan.omega) part.plan.omega = d->plan.omega + *lo * 4;
    if (d->plan.dbeta) part.plan.dbeta = d->plan.dbeta + *lo;
    if (d->plan.valid) part.plan.valid = d->plan.valid + *lo;
    if (d->gain_lin) part.gain_lin = d->gain_lin + *lo * K;
    if (d->Pmax) part.Pmax = d->Pmax + *lo * K * 4;
    if (d->A_end) part.A_end = d->A_end + *lo * K * 8;
    if (d->status) part.status = d->status + *lo * K;
    return part;
}

// ----------------------------------------------------------------- N-wave batch
// Which kernel integrates an N-wave batch: the convolution form needs an integer-grid plan within its limits
// (n_waves <= 128, span <= 512) and pays off unless the plan is sparse (2*span^2 complex MACs per RHS against
// ~one per table entry; the table kernel gathers, so it is given a factor: span^2 > 5 * n_triplets -> table).
// FPA_NWAVE_TABLE / FPA_NWAVE_COMB force the choice; a forced comb beyond its limits is FPA_ERR_UNSUPPORTED.
static bool nwave_use_comb(const fpa_nwave_desc* d) {
    if (d == nullptr || d->grid_slot == nullptr || (d->flags & FPA_NWAVE_TABLE)) return false;
    if (d->flags & FPA_NWAVE_COMB) return true;
    const bool table_given = d->row_ptr != nullptr && (d->n_triplets == 0 || d->triplets != nullptr);
    if (!table_given) return true;
    if (!nwave_comb_fits(d)) return false;
    return (int64_t)d->grid_span * d->grid_span <= 5 * d->n_triplets || d->n_triplets == 0;
}

static int nwave_dispatch(const fpa_nwave_desc* d, cudaStream_t st) {
    return nwave_use_comb(d) ? nwave_comb_launch(d, st) : nwave_launch(d, st);
}

// What only the host entry can check: the flags that pick the kernel, and the grid slots (host pointers here).
static int nwave_host_check(const fpa_nwave_desc* d) {
    FPA_TRY(nwave_check(d));
    FPA_REQUIRE(!((d->flags & FPA_NWAVE_TABLE) && (d->flags & FPA_NWAVE_COMB)), "FPA_NWAVE_TABLE and FPA_NWAVE_COMB exclude each other");
    FPA_REQUIRE(!(d->flags & FPA_NWAVE_COMB) || d->grid_slot, "FPA_NWAVE_COMB needs grid_slot");
    FPA_REQUIRE(nwave_use_comb(d) || (d->n_triplets >= 0 && d->row_ptr), "triplet table must be set");
    if (d->grid_slot) {
        FPA_REQUIRE(d->grid_span >= 1, "grid_span must be >= 1");
        std::vector<char> seen((size_t)d->grid_span, 0);
        for (int j = 0; j < d->n_waves; ++j) {
            const int32_t g = d->grid_slot[j];
            FPA_REQUIRE(g >= 0 && g < d->grid_span, "grid_slot[%d] = %d is outside [0, grid_span = %d)", j, g, d->grid_span);
            FPA_REQUIRE(!seen[(size_t)g], "grid_slot values must be distinct (slot %d appears twice)", g);
            seen[(size_t)g] = 1;
        }
    }
    return FPA_OK;
}

static int nwave_host_launch(const fpa_nwave_desc* d, int device, Pending* p) {
    FPA_TRY(nwave_host_check(d));
    const bool comb = nwave_use_comb(d);
    FPA_TRY(use_device(device));
    const size_t B = (size_t)d->n_points, N = (size_t)d->n_waves;
    if (B == 0) return FPA_OK;
    const size_t ns = (size_t)fpa_n_saved(d->n_steps, d->save_every);
    // the table kernel gets the factored form of the table (unless the caller insists on the entry list)
    std::vector<unsigned char> blob;
    int32_t                    n_classes = 0;
    if (!comb && !(d->flags & FPA_NWAVE_PLAIN) && N <= 128) {
        const int64_t nb = fpa_nwave_factor_table((int32_t)N, d->triplets, d->row_ptr, d->n_triplets, nullptr, 0, &n_classes);
        if (nb < 0) return FPA_ERR_INVALID;
        blob.resize((size_t)nb);
        if (fpa_nwave_factor_table((int32_t)N, d->triplets, d->row_ptr, d->n_triplets, blob.data(), nb, &n_classes) != nb) return FPA_ERR_INVALID;
    }
    fpa_nwave_desc dd;
    FPA_TRY(stage(device, 5, p, [&](Staging& s) {
        dd           = *d;
        dd.beta      = s.in(d->beta, (d->beta_stride ? B : 1) * N);
        dd.gamma     = s.in(d->gamma, d->gamma_stride ? B : 1);
        dd.alpha     = s.in(d->alpha, d->alpha_stride ? B : 1);
        dd.A0        = s.in(d->A0, (d->A0_stride ? B : 1) * N * 2);
        dd.grid_slot = comb ? s.in(d->grid_slot, N) : nullptr;
        dd.triplets  = comb ? nullptr : s.in(d->triplets, (size_t)d->n_triplets);
        dd.row_ptr   = comb ? nullptr : s.in(d->row_ptr, N + 1);
        dd.factored  = blob.empty() ? nullptr : s.in(blob.data(), blob.size());
        dd.A_trace   = (d->flags & FPA_OUT_TRACE) ? s.out(d->A_trace, B * ns * N * 2, false) : nullptr;
        dd.A_end     = (d->flags & FPA_OUT_END) ? s.out(d->A_end, B * N * 2, false) : nullptr;
        dd.Pmax      = (d->flags & FPA_OUT_PMAX) ? s.out(d->Pmax, B * N, false) : nullptr;
        dd.status    = s.out(d->status, B, false);  // the kernel always gets one
    }));
    dd.n_classes = n_classes;
    dd.flags = (d->flags & ~(FPA_NWAVE_TABLE | FPA_NWAVE_COMB)) | (comb ? FPA_NWAVE_COMB : FPA_NWAVE_TABLE);  // decided above
    return nwave_dispatch(&dd, p->st);
}

}  // namespace fpa

using namespace fpa;

// =================================================================== extern "C"
extern "C" {

const char* fpa_last_error(void) { return g_err; }
const char* fpa_version(void) {
#if defined(FPA_SASS_PASS) && FPA_SASS_PASS
    return "fpa_b200 0.2 (sm_100a; FP64 hot loops re-scheduled after ptxas: tools/sass_sched.py)";
#else
    return "fpa_b200 0.2 (sm_100a; ptxas schedule)";
#endif
}

int fpa_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int fpa_device_info(int device, int* sm_count, int* clock_khz, char* name, int name_cap) {
    FPA_TRY(use_device(device));
    cudaDeviceProp prop;
    FPA_CUDA(cudaGetDeviceProperties(&prop, device));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (clock_khz) {
        int khz = 0;
        FPA_CUDA(cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, device));
        *clock_khz = khz;
    }
    if (name && name_cap > 0) {
        strncpy(name, prop.name, (size_t)name_cap - 1);
        name[name_cap - 1] = '\0';
    }
    return FPA_OK;
}

int fpa_set_device(int device) { return use_device(device); }

int64_t fpa_n_saved(int64_t n_steps, int64_t save_every) {
    if (n_steps < 0 || save_every < 1) return -1;
    return n_steps / save_every + 1;
}

int64_t fpa_interval_steps(double z_max, double dz) {
    // Python's round() on a float is round-half-to-even == nearbyint in the default FP mode
    const double q = z_max / dz;
    if (!(q == q) || fabs(q) > 9.0e15) return -1;
    return (int64_t)nearbyint(q);
}

double fpa_yaman4_flops_per_step(void) { return 568.0; }

// ------------------------------------------------------------------ 4-wave integrator
int fpa_yaman4_rk4_batch_dev(const fpa_yaman4_desc* d, void* stream) {
    FPA_TRY(need_device());
    return yaman4_launch(d, static_cast<cudaStream_t>(stream));
}

int fpa_yaman4_rk4_batch_host(const fpa_yaman4_desc* d, int device) {
    return run_on_device(batch_host_launch, d, device);
}

int fpa_yaman4_rk4_batch_multi_host(const fpa_yaman4_desc* d, int n_devices, const int* devices) {
    FPA_TRY(yaman4_check(d));
    FPA_TRY(check_devices(n_devices, devices));
    if (n_devices == 1) return fpa_yaman4_rk4_batch_host(d, devices[0]);
    return run_on_devices(n_devices, devices, [&](int k, Pending* p) {
        int64_t               lo;
        const fpa_yaman4_desc part = batch_part(d, n_devices, k, &lo);
        return part.n_points > 0 ? batch_host_launch(&part, devices[k], p) : (int)FPA_OK;
    });
}

int fpa_yaman4_rhs_host(int64_t B, const double* z, const double* A, const double* gamma,
                        const double* alpha, const double* dbeta, double* dA, int device) {
    FPA_REQUIRE(B >= 0, "B must be >= 0");
    FPA_REQUIRE(B == 0 || (z && A && gamma && alpha && dbeta && dA), "NULL argument");
    FPA_TRY(use_device(device));
    if (B == 0) return FPA_OK;
    const size_t b = (size_t)B;
    Pending      p;
    const double *dz, *dA_in, *dg, *da, *db;
    double*       dA_out;
    FPA_TRY(stage(device, 1, &p, [&](Staging& s) {
        dz     = s.in(z, b);
        dg     = s.in(gamma, b);
        da     = s.in(alpha, b);
        db     = s.in(dbeta, b);
        dA_in  = s.in(A, b * 8);
        dA_out = s.out(dA, b * 8, false);
    }));
    FPA_TRY(yaman4_rhs_launch(B, dz, dA_in, dg, da, db, dA_out, p.st));
    return finish(p, device);
}

// ------------------------------------------------------------------ Delta-beta table
int fpa_dbeta_table_dev(const fpa_plan_desc* d, void* stream) {
    FPA_TRY(need_device());
    return plan_launch(d, nullptr, static_cast<cudaStream_t>(stream));
}

int fpa_dbeta_table_host(const fpa_plan_desc* d, int device) {
    FPA_REQUIRE(d != nullptr, "plan descriptor is NULL");
    FPA_REQUIRE(d->n1 >= 0 && d->n3 >= 0, "grid sizes must be >= 0");
    FPA_REQUIRE(d->lambda1 && d->lambda2 && d->lambda3, "wavelength axes must be set");
    FPA_REQUIRE(d->dbeta != nullptr, "dbeta output must be set");
    FPA_TRY(use_device(device));
    const size_t n1 = (size_t)d->n1, n3 = (size_t)d->n3, B = n1 * n3;
    if (B == 0) return FPA_OK;
    Pending       p;
    fpa_plan_desc dd;
    FPA_TRY(stage(device, 2, &p, [&](Staging& s) {
        dd         = *d;
        dd.lambda1 = s.in(d->lambda1, n1);
        dd.lambda2 = s.in(d->lambda2, d->lambda2_stride ? n1 : 1);
        dd.lambda3 = s.in(d->lambda3, n3);
        dd.omega   = d->omega ? s.out(d->omega, B * 4, false) : nullptr;
        dd.dbeta   = s.out(d->dbeta, B, false);
        dd.valid   = s.out(d->valid, B, false);
    }));
    FPA_TRY(plan_launch(&dd, nullptr, p.st));
    return finish(p, device);
}

// ------------------------------------------------------------------ fused sweep
int64_t fpa_yaman4_scratch_bytes(int64_t n_points) { return yaman4_scratch_bytes(n_points); }

int64_t fpa_yaman4_sweep_scratch_bytes(int64_t n_points) {
    // scheduler counters + one state record per point for the z-segment scheduler (csrc/yaman4.cu); a
    // sweep launched without it (scratch == NULL) runs as the whole-run kernel
    return yaman4_scratch_bytes(n_points);
}

// One fused kernel per sweep.  FPA_PHASE_EXACT is refused (FPA_ERR_UNSUPPORTED): the reference's
// arithmetic structure is available through fpa_dbeta_table_* + fpa_yaman4_rk4_batch_*.
int fpa_yaman4_sweep_dev(const fpa_sweep_desc* d, void* scratch, int64_t scratch_bytes, void* stream) {
    FPA_TRY(need_device());
    return yaman4_sweep_launch(d, scratch, scratch_bytes, static_cast<cudaStream_t>(stream));
}

int fpa_yaman4_sweep_host(const fpa_sweep_desc* d, int device) {
    return run_on_device(sweep_host_launch, d, device);
}

int fpa_yaman4_sweep_multi_host(const fpa_sweep_desc* d, int n_devices, const int* devices) {
    FPA_REQUIRE(d != nullptr, "sweep descriptor is NULL");
    FPA_TRY(sweep_multi_check(d, n_devices, devices));
    if (n_devices == 1) return fpa_yaman4_sweep_host(d, devices[0]);
    return run_on_devices(n_devices, devices, [&](int k, Pending* p) {
        int64_t              lo;
        const fpa_sweep_desc part = sweep_part(d, n_devices, k, 1, &lo);
        return part.n_sub_points > 0 ? sweep_host_launch(&part, devices[k], p) : (int)FPA_OK;
    });
}

// ------------------------------------------------------------------ small-signal transfer matrices
int fpa_yaman4_transfer_batch_dev(const fpa_yaman4_desc* d, const fpa_transfer_out* t, void* stream) {
    FPA_TRY(need_device());
    return yaman4_transfer_launch(d, t, static_cast<cudaStream_t>(stream));
}

int fpa_yaman4_transfer_batch_host(const fpa_yaman4_desc* d, const fpa_transfer_out* t, int device) {
    FPA_REQUIRE(t != nullptr, "transfer output is NULL");
    Pending p;
    FPA_TRY(batch_host_launch(d, device, &p, t));
    return finish(p, device);
}

int fpa_yaman4_transfer_batch_multi_host(const fpa_yaman4_desc* d, const fpa_transfer_out* t, int n_devices,
                                         const int* devices) {
    FPA_TRY(yaman4_transfer_check(d, t));
    FPA_TRY(check_devices(n_devices, devices));
    if (n_devices == 1) return fpa_yaman4_transfer_batch_host(d, t, devices[0]);
    const int64_t nc = __builtin_popcount(t->columns);
    return run_on_devices(n_devices, devices, [&](int k, Pending* p) {
        int64_t               lo;
        const fpa_yaman4_desc part = batch_part(d, n_devices, k, &lo);
        fpa_transfer_out      tp   = *t;
        tp.jac += lo * 8 * nc;
        return part.n_points > 0 ? batch_host_launch(&part, devices[k], p, &tp) : (int)FPA_OK;
    });
}

int fpa_yaman4_transfer_sweep_dev(const fpa_sweep_desc* d, const fpa_transfer_out* t, void* stream) {
    FPA_TRY(need_device());
    return yaman4_transfer_sweep_launch(d, t, static_cast<cudaStream_t>(stream));
}

int fpa_yaman4_transfer_sweep_host(const fpa_sweep_desc* d, const fpa_transfer_out* t, int device) {
    FPA_REQUIRE(t != nullptr, "transfer output is NULL");
    Pending p;
    FPA_TRY(sweep_host_launch(d, device, &p, t));
    return finish(p, device);
}

int fpa_yaman4_transfer_sweep_multi_host(const fpa_sweep_desc* d, const fpa_transfer_out* t, int n_devices,
                                         const int* devices) {
    FPA_REQUIRE(d != nullptr, "sweep descriptor is NULL");
    FPA_REQUIRE(t != nullptr, "transfer output is NULL");
    FPA_TRY(sweep_multi_check(d, n_devices, devices));
    if (n_devices == 1) return fpa_yaman4_transfer_sweep_host(d, t, devices[0]);
    const int64_t nc = __builtin_popcount(t->columns);
    return run_on_devices(n_devices, devices, [&](int k, Pending* p) {
        int64_t              lo;
        const fpa_sweep_desc part = sweep_part(d, n_devices, k, 1, &lo);
        fpa_transfer_out     tp   = *t;
        if (tp.jac) tp.jac += lo * 8 * nc;
        return part.n_sub_points > 0 ? sweep_host_launch(&part, devices[k], p, &tp) : (int)FPA_OK;
    });
}

// ------------------------------------------------------------------ phase sweep
int64_t fpa_yaman4_phase_sweep_scratch_bytes(int64_t n_points) { return yaman4_phase_scratch_bytes(n_points); }

int fpa_yaman4_phase_sweep_dev(const fpa_phase_sweep_desc* d, void* scratch, int64_t scratch_bytes, void* stream) {
    FPA_TRY(need_device());
    return phase_sweep_dev(d, scratch, scratch_bytes, static_cast<cudaStream_t>(stream));
}

int fpa_yaman4_phase_sweep_host(const fpa_phase_sweep_desc* d, int device) {
    return run_on_device(phase_sweep_host_launch, d, device);
}

// The K runs of a grid point stay together on one device.
int fpa_yaman4_phase_sweep_multi_host(const fpa_phase_sweep_desc* d, int n_devices, const int* devices) {
    FPA_REQUIRE(d != nullptr, "phase sweep descriptor is NULL");
    FPA_TRY(sweep_multi_check(&d->sweep, n_devices, devices));
    if (n_devices == 1) return fpa_yaman4_phase_sweep_host(d, devices[0]);
    return run_on_devices(n_devices, devices, [&](int k, Pending* p) {
        int64_t              lo;
        fpa_phase_sweep_desc part = *d;
        part.sweep = sweep_part(&d->sweep, n_devices, k, d->n_phases, &lo);
        if (part.sweep.n_sub_points == 0) return (int)FPA_OK;
        if (d->gain_max) part.gain_max = d->gain_max + lo;
        if (d->gain_min) part.gain_min = d->gain_min + lo;
        if (d->idx_max) part.idx_max = d->idx_max + lo;
        if (d->idx_min) part.idx_min = d->idx_min + lo;
        if (d->n_finite) part.n_finite = d->n_finite + lo;
        return phase_sweep_host_launch(&part, devices[k], p);
    });
}

// ------------------------------------------------------------------ linear test RHS
int fpa_linear_rk4_batch_host(int64_t B, int64_t dim, const double* y0, const double* lam, double z0,
                              double z_max, int64_t n_steps, int64_t save_every, const double* z_grid,
                              uint32_t flags, double* y_trace, double* y_end, int32_t* status,
                              int device) {
    FPA_REQUIRE(B >= 0 && dim >= 1 && dim < (1 << 20), "need B >= 0 and 1 <= dim < 2^20");
    FPA_REQUIRE(n_steps >= 1, "n_steps must be >= 1");
    FPA_REQUIRE(save_every >= 1, "save_every must be a positive integer");
    FPA_REQUIRE(y0 && lam, "y0 and lam must be set");
    const bool trace = (flags & FPA_OUT_TRACE) != 0, endo = (flags & FPA_OUT_END) != 0;
    FPA_REQUIRE(!trace || y_trace, "FPA_OUT_TRACE needs y_trace");
    FPA_REQUIRE(!endo || y_end, "FPA_OUT_END needs y_end");
    FPA_TRY(use_device(device));
    if (B == 0) return FPA_OK;
    const size_t n = (size_t)B * (size_t)dim, ns = (size_t)fpa_n_saved(n_steps, save_every);
    Pending      p;
    const double *dy0, *dlam, *grid;
    double *      dtr, *dye;
    int32_t *     bad, *stt;
    FPA_TRY(stage(device, 4, &p, [&](Staging& s) {
        dy0  = s.in(y0, n * 2);
        dlam = s.in(lam, (size_t)dim * 2);
        grid = z_grid ? s.in(z_grid, (size_t)n_steps + 1) : nullptr;
        dtr  = s.out(trace ? y_trace : nullptr, trace ? n * ns * 2 : 0, false);
        dye  = s.out(endo ? y_end : nullptr, n * 2, false);
        bad  = s.tmp<int32_t>(n);
        stt  = s.out(status, (size_t)B, false);
    }));
    FPA_TRY(linear_launch(B, (int)dim, dy0, dlam, z0, z_max, n_steps, save_every, grid, flags, dtr, dye, bad, stt,
                          p.st));
    return finish(p, device);
}

// ------------------------------------------------------------------ N-wave integrator
int fpa_nwave_rk4_batch_dev(const fpa_nwave_desc* d, void* stream) {
    FPA_TRY(need_device());
    return nwave_dispatch(d, static_cast<cudaStream_t>(stream));
}

int fpa_nwave_rk4_batch_host(const fpa_nwave_desc* d, int device) {
    return run_on_device(nwave_host_launch, d, device);
}

int fpa_nwave_rk4_batch_multi_host(const fpa_nwave_desc* d, int n_devices, const int* devices) {
    FPA_TRY(nwave_host_check(d));
    FPA_TRY(check_devices(n_devices, devices));
    if (n_devices == 1) return fpa_nwave_rk4_batch_host(d, devices[0]);
    const int64_t ns = fpa_n_saved(d->n_steps, d->save_every), N = d->n_waves;
    return run_on_devices(n_devices, devices, [&](int k, Pending* p) {
        int64_t lo, hi;
        balanced_range(d->n_points, n_devices, k, &lo, &hi);
        if (hi <= lo) return (int)FPA_OK;
        fpa_nwave_desc part = *d;
        part.n_points = hi - lo;
        part.beta     = d->beta + lo * d->beta_stride * N;
        part.gamma    = d->gamma + lo * d->gamma_stride;
        part.alpha    = d->alpha + lo * d->alpha_stride;
        part.A0       = d->A0 + lo * d->A0_stride * N * 2;
        if (d->A_trace) part.A_trace = d->A_trace + lo * ns * N * 2;
        if (d->A_end) part.A_end = d->A_end + lo * N * 2;
        if (d->Pmax) part.Pmax = d->Pmax + lo * N;
        if (d->status) part.status = d->status + lo;
        return nwave_host_launch(&part, devices[k], p);
    });
}

// ------------------------------------------------------------------ measurement helpers
int fpa_fp64_peak_probe(int device, int iters, double* tflops, double* ms) {
    return probe_run(device, iters, tflops, ms);
}

int fpa_host_alloc(void** ptr, int64_t bytes) {
    FPA_REQUIRE(ptr != nullptr && bytes >= 0, "bad arguments");
    FPA_TRY(need_device("pinned host memory needs the CUDA runtime"));
    FPA_CUDA(cudaMallocHost(ptr, (size_t)(bytes > 0 ? bytes : 1)));
    return FPA_OK;
}

int fpa_host_free(void* ptr) {
    if (ptr == nullptr) return FPA_OK;
    FPA_CUDA(cudaFreeHost(ptr));
    return FPA_OK;
}

int fpa_dev_alloc(void** ptr, int64_t bytes, int device) {
    FPA_REQUIRE(ptr != nullptr && bytes > 0, "bad arguments");
    FPA_TRY(use_device(device));
    FPA_CUDA(cudaMalloc(ptr, (size_t)bytes));
    return FPA_OK;
}

int fpa_dev_free(void* ptr) {
    if (ptr == nullptr) return FPA_OK;
    FPA_CUDA(cudaFree(ptr));
    return FPA_OK;
}

int fpa_ipc_export(const void* dev_ptr, void* handle64) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "the ABI documents a 64-byte handle");
    FPA_REQUIRE(dev_ptr != nullptr && handle64 != nullptr, "bad arguments");
    cudaIpcMemHandle_t h;
    FPA_CUDA(cudaIpcGetMemHandle(&h, const_cast<void*>(dev_ptr)));
    memcpy(handle64, &h, sizeof(h));
    return FPA_OK;
}

int fpa_ipc_open(const void* handle64, void** dev_ptr) {
    FPA_REQUIRE(dev_ptr != nullptr && handle64 != nullptr, "bad arguments");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, sizeof(h));
    FPA_CUDA(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return FPA_OK;
}

int fpa_ipc_close(void* dev_ptr) {
    if (dev_ptr == nullptr) return FPA_OK;
    FPA_CUDA(cudaIpcCloseMemHandle(dev_ptr));
    return FPA_OK;
}

int fpa_host_register(void* ptr, int64_t bytes) {
    FPA_REQUIRE(ptr != nullptr && bytes > 0, "bad arguments");
    FPA_TRY(need_device("page-locking host memory needs the CUDA runtime"));
    FPA_CUDA(cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterPortable | cudaHostRegisterMapped));
    return FPA_OK;
}

int fpa_host_unregister(void* ptr) {
    if (ptr == nullptr) return FPA_OK;
    FPA_CUDA(cudaHostUnregister(ptr));
    return FPA_OK;
}

}  // extern "C"
