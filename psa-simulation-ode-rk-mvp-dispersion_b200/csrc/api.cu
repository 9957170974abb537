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

// launchers implemented next to their kernels
int yaman4_launch(const fpa_yaman4_desc* d, cudaStream_t st);
int yaman4_rhs_launch(int64_t B, const double* z, const double* A, const double* gamma,
                      const double* alpha, const double* dbeta, double* dA, cudaStream_t st);
int plan_launch(const fpa_plan_desc* d, double* dbeta_masked, cudaStream_t st);
int yaman4_sweep_launch(const fpa_sweep_desc* d, void* scratch, int64_t scratch_bytes, cudaStream_t st);
int yaman4_phase_sweep_launch(const fpa_phase_sweep_desc* d, void* scratch, int64_t scratch_bytes, cudaStream_t st);
int phase_reduce_launch(int64_t G, int K, const double* gain, double* gmax, double* gmin, int32_t* imax, int32_t* imin,
                        int32_t* nfin, cudaStream_t st);
int64_t yaman4_scratch_bytes(int64_t n_points);
int64_t yaman4_phase_scratch_bytes(int64_t n_points);
int linear_launch(int64_t B, int dim, const double* y0, const double* lam, double z0, double z_max,
                  int64_t n_steps, int64_t save_every, const double* z_grid, uint32_t flags,
                  double* y_trace, double* y_end, int32_t* bad_scratch, int32_t* status,
                  cudaStream_t st);
int nwave_launch(const fpa_nwave_desc* d, cudaStream_t st);
int nwave_comb_launch(const fpa_nwave_desc* d, cudaStream_t st);
int probe_run(int device, int iters, double* tflops, double* ms_out);

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

int use_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        cudaGetLastError();
        set_error("no CUDA device is visible: libfpa_b200 has no CPU path");
        return FPA_ERR_NO_DEVICE;
    }
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

// bump allocator over one workspace slab (256-byte aligned pieces)
struct Carver {
    char*  base = nullptr;
    size_t off  = 0;
    template <class T>
    T* take(size_t count) {
        T* p = reinterpret_cast<T*>(base + off);
        off += (count * sizeof(T) + 255) & ~(size_t)255;
        return p;
    }
    static size_t need(size_t bytes) { return (bytes + 255) & ~(size_t)255; }
};

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

#define FPA_TRY(expr)                  \
    do {                               \
        int rc__ = (expr);             \
        if (rc__ != FPA_OK) return rc__; \
    } while (0)

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

// ----------------------------------------------------------------- N-wave dispatch
// Which kernel integrates an N-wave batch: the convolution form needs an integer-grid plan within its limits
// (n_waves <= 128, span <= 512) and pays off unless the plan is sparse (2*span^2 complex MACs per RHS against
// ~one per table entry; the table kernel gathers, so it is given a factor: span^2 > 5 * n_triplets -> table).
// FPA_NWAVE_TABLE / FPA_NWAVE_COMB force the choice; a forced comb beyond its limits is FPA_ERR_UNSUPPORTED.
static bool nwave_use_comb(const fpa_nwave_desc* d) {
    if (d->grid_slot == nullptr || (d->flags & FPA_NWAVE_TABLE)) return false;
    if (d->flags & FPA_NWAVE_COMB) return true;
    const bool table_given = d->row_ptr != nullptr && (d->n_triplets == 0 || d->triplets != nullptr);
    if (!table_given) return true;
    if (d->n_waves > 128 || d->grid_span > 512) return false;
    return (int64_t)d->grid_span * d->grid_span <= 5 * d->n_triplets || d->n_triplets == 0;
}

static int nwave_dispatch(const fpa_nwave_desc* d, cudaStream_t st) {
    if (!nwave_use_comb(d)) return nwave_launch(d, st);
    FPA_REQUIRE(d->n_points >= 0 && d->n_points < 2147483647LL, "bad n_points");
    FPA_REQUIRE(d->n_waves >= 1, "n_waves must be >= 1");
    if (d->n_waves > 128 || d->grid_span > 512) {
        set_error("comb kernel limits: n_waves <= 128, grid_span <= 512 (got %d, %d)", d->n_waves, d->grid_span);
        return FPA_ERR_UNSUPPORTED;
    }
    FPA_REQUIRE(d->grid_span >= d->n_waves, "grid_span must cover all waves");
    FPA_REQUIRE(d->n_steps >= 1 && d->n_steps < 2147483647LL, "n_steps must be in [1, 2^31)");
    FPA_REQUIRE(d->save_every >= 1, "save_every must be a positive integer");
    FPA_REQUIRE(d->beta && d->gamma && d->alpha && d->A0, "beta/gamma/alpha/A0 must be set");
    FPA_REQUIRE((d->gamma_stride | 1) == 1 && (d->alpha_stride | 1) == 1 && (d->A0_stride | 1) == 1 &&
                    (d->beta_stride | 1) == 1,
                "strides must be 0 (broadcast) or 1 (per point)");
    FPA_REQUIRE(!(d->flags & FPA_OUT_TRACE) || d->A_trace, "FPA_OUT_TRACE needs A_trace");
    FPA_REQUIRE(!(d->flags & FPA_OUT_PMAX) || d->Pmax, "FPA_OUT_PMAX needs Pmax");
    FPA_REQUIRE(!(d->flags & FPA_OUT_END) || d->A_end, "FPA_OUT_END needs A_end");
    if (d->n_points == 0) return FPA_OK;
    return nwave_comb_launch(d, st);
}

// ----------------------------------------------------------------- sweep (device pointers)
// One fused kernel per sweep.  FPA_PHASE_EXACT is refused (FPA_ERR_UNSUPPORTED): the reference's
// arithmetic structure is available through fpa_dbeta_table_* + fpa_yaman4_rk4_batch_*.
static int sweep_dev(const fpa_sweep_desc* d, void* scratch, int64_t scratch_bytes, cudaStream_t st) {
    return yaman4_sweep_launch(d, scratch, scratch_bytes, st);
}

// Phase sweep: the sweep kernel, then the per-grid-point reductions over its gain map on the same stream.
static int phase_sweep_dev(const fpa_phase_sweep_desc* d, void* scratch, int64_t scratch_bytes, cudaStream_t st) {
    FPA_TRY(yaman4_phase_sweep_launch(d, scratch, scratch_bytes, st));
    const fpa_sweep_desc& w = d->sweep;
    const int64_t G = (w.first_point == 0 && w.n_sub_points == 0) ? w.plan.n1 * w.plan.n3 : w.n_sub_points;
    return phase_reduce_launch(G, (int)d->n_phases, w.gain_lin, d->gain_max, d->gain_min, d->idx_max, d->idx_min,
                               d->n_finite, st);
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
template <typename Pending, typename Launch, typename Collect>
static int run_on_devices(int n_devices, const int* devices, Pending* pend, Launch launch, Collect collect) {
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
    int n = fpa_device_count();
    if (n <= 0) {
        set_error("no CUDA device is visible: libfpa_b200 has no CPU path");
        return FPA_ERR_NO_DEVICE;
    }
    return yaman4_launch(d, static_cast<cudaStream_t>(stream));
}

// One batch with host pointers in two steps (see the sweep below for why): batch_host_launch queues the
// uploads and the kernel, batch_host_collect queues the result copies; the caller synchronises.
struct PendingBatch {
    cudaStream_t st = nullptr;
    size_t       B = 0, n_tr = 0;
    // device staging buffers, NULL where the kernel wrote straight into the caller's pinned array
    double * tr = nullptr, *Ae = nullptr, *Pm = nullptr;
    int32_t* stt = nullptr;
    fpa_yaman4_desc user;
};

static int batch_host_check(const fpa_yaman4_desc* d) {
    FPA_REQUIRE(d != nullptr, "descriptor is NULL");
    FPA_REQUIRE(d->n_points >= 0, "n_points must be >= 0");
    FPA_REQUIRE(d->n_steps >= 1, "n_steps must be >= 1");
    FPA_REQUIRE(d->save_every >= 1, "save_every must be a positive integer");
    FPA_REQUIRE(d->dbeta && d->gamma && d->alpha && d->A0, "dbeta/gamma/alpha/A0 must be set");
    FPA_REQUIRE((d->gamma_stride | 1) == 1 && (d->alpha_stride | 1) == 1 && (d->A0_stride | 1) == 1,
                "strides must be 0 (broadcast) or 1 (per point)");
    FPA_REQUIRE(!(d->flags & FPA_OUT_TRACE) || d->A_trace, "FPA_OUT_TRACE needs A_trace");
    FPA_REQUIRE(!(d->flags & FPA_OUT_PMAX) || d->Pmax, "FPA_OUT_PMAX needs Pmax");
    FPA_REQUIRE(!(d->flags & FPA_OUT_END) || d->A_end, "FPA_OUT_END needs A_end");
    return FPA_OK;
}

static int batch_host_launch(const fpa_yaman4_desc* d, int device, PendingBatch* pb) {
    FPA_TRY(batch_host_check(d));
    FPA_TRY(use_device(device));
    *pb = PendingBatch();
    const size_t B = (size_t)d->n_points;
    if (B == 0) return FPA_OK;
    const size_t ns     = (size_t)fpa_n_saved(d->n_steps, d->save_every);
    const size_t n_g    = d->gamma_stride ? B : 1, n_a = d->alpha_stride ? B : 1;
    const size_t n_A0   = (d->A0_stride ? B : 1) * 8;
    const size_t n_grid = d->z_grid ? (size_t)d->n_steps + 1 : 0;
    const bool   trace = (d->flags & FPA_OUT_TRACE) != 0, endo = (d->flags & FPA_OUT_END) != 0;
    const bool   pmax = (d->flags & FPA_OUT_PMAX) != 0;
    // outputs in pinned host memory are written by the kernel itself (no staging, no copy)
    double*  m_tr = trace ? mapped(d->A_trace) : nullptr;
    double*  m_Ae = endo ? mapped(d->A_end) : nullptr;
    double*  m_Pm = pmax ? mapped(d->Pmax) : nullptr;
    int32_t* m_st = mapped(d->status);
    const size_t n_tr = (trace && !m_tr) ? B * ns * 8 : 0;
    const size_t n_sched = (size_t)yaman4_scratch_bytes((int64_t)B);

    size_t need = Carver::need(B * 8) + Carver::need(n_g * 8) + Carver::need(n_a * 8) +
                  Carver::need(n_A0 * 8) + Carver::need(n_grid * 8) + Carver::need(n_tr * 8) +
                  Carver::need(B * 64) + Carver::need(B * 32) + Carver::need(B * 4) + Carver::need(n_sched);
    void* ws = nullptr;
    FPA_TRY(workspace(device, 0, need, &ws));
    cudaStream_t st;
    FPA_TRY(host_stream(device, &st));
    Carver cv;
    cv.base = static_cast<char*>(ws);
    double*  dbeta = cv.take<double>(B);
    double*  gam   = cv.take<double>(n_g);
    double*  alp   = cv.take<double>(n_a);
    double*  A0    = cv.take<double>(n_A0);
    double*  grid  = cv.take<double>(n_grid);
    double*  tr    = cv.take<double>(n_tr);
    double*  Aend  = cv.take<double>(B * 8);
    double*  Pm    = cv.take<double>(B * 4);
    int32_t* stat  = cv.take<int32_t>(B);
    char*    sched = cv.take<char>(n_sched);

    FPA_TRY(up(dbeta, d->dbeta, B * 8, st));
    FPA_TRY(up(gam, d->gamma, n_g * 8, st));
    FPA_TRY(up(alp, d->alpha, n_a * 8, st));
    FPA_TRY(up(A0, d->A0, n_A0 * 8, st));
    FPA_TRY(up(grid, d->z_grid, n_grid * 8, st));

    fpa_yaman4_desc dd = *d;
    dd.dbeta   = dbeta;
    dd.gamma   = gam;
    dd.alpha   = alp;
    dd.A0      = A0;
    dd.z_grid  = d->z_grid ? grid : nullptr;
    dd.A_trace = trace ? (m_tr ? m_tr : tr) : nullptr;
    dd.A_end   = endo ? (m_Ae ? m_Ae : Aend) : nullptr;
    dd.Pmax    = pmax ? (m_Pm ? m_Pm : Pm) : nullptr;
    dd.status  = d->status ? (m_st ? m_st : stat) : stat;
    dd.scratch = sched;
    dd.scratch_bytes = (int64_t)n_sched;
    if (d->gamma_stride == 0 && d->alpha_stride == 0) {  // host pointers: the broadcast values are known here
        dd.flags |= FPA_UNIFORM_PHYSICS;
        dd.gamma_uniform = d->gamma[0];
        dd.alpha_uniform = d->alpha[0];
    } else {
        dd.flags &= ~FPA_UNIFORM_PHYSICS;
    }
    FPA_TRY(yaman4_launch(&dd, st));
    pb->st   = st;
    pb->B    = B;
    pb->n_tr = n_tr;
    pb->user = *d;
    pb->tr   = (trace && !m_tr) ? tr : nullptr;
    pb->Ae   = (endo && !m_Ae) ? Aend : nullptr;
    pb->Pm   = (pmax && !m_Pm) ? Pm : nullptr;
    pb->stt  = (d->status && !m_st) ? stat : nullptr;
    return FPA_OK;
}

static int batch_host_collect(const PendingBatch& pb, int device) {
    if (!pb.st) return FPA_OK;
    FPA_TRY(use_device(device));
    if (pb.tr) FPA_TRY(down(pb.user.A_trace, pb.tr, pb.n_tr * 8, pb.st));
    if (pb.Ae) FPA_TRY(down(pb.user.A_end, pb.Ae, pb.B * 64, pb.st));
    if (pb.Pm) FPA_TRY(down(pb.user.Pmax, pb.Pm, pb.B * 32, pb.st));
    if (pb.stt) FPA_TRY(down(pb.user.status, pb.stt, pb.B * 4, pb.st));
    return FPA_OK;
}

int fpa_yaman4_rk4_batch_host(const fpa_yaman4_desc* d, int device) {
    PendingBatch pb;
    FPA_TRY(batch_host_launch(d, device, &pb));
    FPA_TRY(batch_host_collect(pb, device));
    if (pb.st) FPA_CUDA(cudaStreamSynchronize(pb.st));
    return FPA_OK;
}

int fpa_yaman4_rk4_batch_multi_host(const fpa_yaman4_desc* d, int n_devices, const int* devices) {
    FPA_TRY(batch_host_check(d));
    FPA_REQUIRE(n_devices >= 1 && n_devices <= 64 && devices != nullptr, "need 1..64 device ordinals");
    if (n_devices == 1) return fpa_yaman4_rk4_batch_host(d, devices[0]);
    const int64_t ns = fpa_n_saved(d->n_steps, d->save_every);
    PendingBatch  pend[64];
    return run_on_devices(
        n_devices, devices, pend,
        [&](int k, PendingBatch* pb) {
            int64_t lo, hi;
            balanced_range(d->n_points, n_devices, k, &lo, &hi);
            *pb = PendingBatch();
            if (hi <= lo) return (int)FPA_OK;
            fpa_yaman4_desc part = *d;
            part.n_points = hi - lo;
            part.dbeta    = d->dbeta + lo;
            part.gamma    = d->gamma + lo * d->gamma_stride;
            part.alpha    = d->alpha + lo * d->alpha_stride;
            part.A0       = d->A0 + lo * d->A0_stride * 8;
            if (d->A_trace) part.A_trace = d->A_trace + lo * ns * 8;
            if (d->A_end) part.A_end = d->A_end + lo * 8;
            if (d->Pmax) part.Pmax = d->Pmax + lo * 4;
            if (d->status) part.status = d->status + lo;
            return batch_host_launch(&part, devices[k], pb);
        },
        batch_host_collect);
}

int fpa_yaman4_rhs_host(int64_t B, const double* z, const double* A, const double* gamma,
                        const double* alpha, const double* dbeta, double* dA, int device) {
    FPA_REQUIRE(B >= 0, "B must be >= 0");
    FPA_REQUIRE(B == 0 || (z && A && gamma && alpha && dbeta && dA), "NULL argument");
    FPA_TRY(use_device(device));
    if (B == 0) return FPA_OK;
    const size_t b = (size_t)B;
    void* ws = nullptr;
    FPA_TRY(workspace(device, 1, 4 * Carver::need(b * 8) + 2 * Carver::need(b * 64), &ws));
    cudaStream_t st;
    FPA_TRY(host_stream(device, &st));
    Carver cv;
    cv.base = static_cast<char*>(ws);
    double* dz = cv.take<double>(b);
    double* dg = cv.take<double>(b);
    double* da = cv.take<double>(b);
    double* db = cv.take<double>(b);
    double* dA_in = cv.take<double>(b * 8);
    double* dA_out = cv.take<double>(b * 8);
    FPA_TRY(up(dz, z, b * 8, st));
    FPA_TRY(up(dg, gamma, b * 8, st));
    FPA_TRY(up(da, alpha, b * 8, st));
    FPA_TRY(up(db, dbeta, b * 8, st));
    FPA_TRY(up(dA_in, A, b * 64, st));
    FPA_TRY(yaman4_rhs_launch(B, dz, dA_in, dg, da, db, dA_out, st));
    FPA_TRY(down(dA, dA_out, b * 64, st));
    FPA_CUDA(cudaStreamSynchronize(st));
    return FPA_OK;
}

// ------------------------------------------------------------------ Delta-beta table
int fpa_dbeta_table_dev(const fpa_plan_desc* d, void* stream) {
    if (fpa_device_count() <= 0) {
        set_error("no CUDA device is visible: libfpa_b200 has no CPU path");
        return FPA_ERR_NO_DEVICE;
    }
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
    const size_t n2 = d->lambda2_stride ? n1 : 1;
    void*        ws = nullptr;
    FPA_TRY(workspace(device, 2,
                      Carver::need(n1 * 8) + Carver::need(n2 * 8) + Carver::need(n3 * 8) +
                          Carver::need(B * 32) + Carver::need(B * 8) + Carver::need(B * 4),
                      &ws));
    cudaStream_t st;
    FPA_TRY(host_stream(device, &st));
    Carver cv;
    cv.base = static_cast<char*>(ws);
    double*  l1 = cv.take<double>(n1);
    double*  l2 = cv.take<double>(n2);
    double*  l3 = cv.take<double>(n3);
    double*  om = cv.take<double>(B * 4);
    double*  db = cv.take<double>(B);
    int32_t* va = cv.take<int32_t>(B);
    FPA_TRY(up(l1, d->lambda1, n1 * 8, st));
    FPA_TRY(up(l2, d->lambda2, n2 * 8, st));
    FPA_TRY(up(l3, d->lambda3, n3 * 8, st));
    fpa_plan_desc dd = *d;
    dd.lambda1 = l1;
    dd.lambda2 = l2;
    dd.lambda3 = l3;
    dd.omega   = d->omega ? om : nullptr;
    dd.dbeta   = db;
    dd.valid   = va;
    FPA_TRY(plan_launch(&dd, nullptr, st));
    FPA_TRY(down(d->omega, om, B * 32, st));
    FPA_TRY(down(d->dbeta, db, B * 8, st));
    FPA_TRY(down(d->valid, va, B * 4, st));
    FPA_CUDA(cudaStreamSynchronize(st));
    return FPA_OK;
}

// ------------------------------------------------------------------ fused sweep
int64_t fpa_yaman4_scratch_bytes(int64_t n_points) { return yaman4_scratch_bytes(n_points); }

int64_t fpa_yaman4_sweep_scratch_bytes(int64_t n_points) {
    // scheduler counters + one state record per point for the z-segment scheduler (csrc/yaman4.cu); a
    // sweep launched without it (scratch == NULL) runs as the whole-run kernel
    return yaman4_scratch_bytes(n_points);
}

int fpa_yaman4_sweep_dev(const fpa_sweep_desc* d, void* scratch, int64_t scratch_bytes, void* stream) {
    if (fpa_device_count() <= 0) {
        set_error("no CUDA device is visible: libfpa_b200 has no CPU path");
        return FPA_ERR_NO_DEVICE;
    }
    return sweep_dev(d, scratch, scratch_bytes, static_cast<cudaStream_t>(stream));
}

// One sweep with host pointers in two steps, so that several devices can be driven from one thread:
// sweep_host_launch queues the axes upload and the kernel; sweep_host_collect queues the result
// copies (a copy into pageable memory blocks the host until the kernel is done, so every device's
// kernel has to be in flight before the first collect) and the caller synchronises the stream.
// A phase sweep (`ph` set) runs K = ph->n_phases initial states per grid point: the per-run arrays hold B*K entries,
// the plan outputs and the reductions B.
struct PendingSweep {
    cudaStream_t st = nullptr;
    size_t       B = 0, P = 0;  // grid points, runs (P = B*K)
    // device staging buffers, NULL where the kernel wrote straight into the caller's pinned array
    double * gain = nullptr, *db = nullptr, *Pm = nullptr, *Ae = nullptr, *om = nullptr;
    int32_t *va = nullptr, *stt = nullptr;
    double * gmax = nullptr, *gmin = nullptr;  // phase sweep reductions
    int32_t *imax = nullptr, *imin = nullptr, *nfin = nullptr;
    fpa_sweep_desc       user;  // the caller's (host) pointers
    fpa_phase_sweep_desc puser;
};

static int sweep_host_launch(const fpa_sweep_desc* d, const fpa_phase_sweep_desc* ph, int device, PendingSweep* ps) {
    FPA_REQUIRE(d != nullptr, "sweep descriptor is NULL");
    FPA_REQUIRE(!ph || (ph->n_phases >= 1 && ph->n_phases <= FPA_MAX_PHASES), "n_phases must be in [1, %d]",
                FPA_MAX_PHASES);
    FPA_REQUIRE(!ph || ph->A0_table != nullptr, "A0_table must be set");
    FPA_REQUIRE(!ph || d->n_peers == 0, "the phase sweep has no peer-store gather: n_peers must be 0");
    const fpa_plan_desc& pl = d->plan;
    FPA_REQUIRE(pl.n1 >= 0 && pl.n3 >= 0, "grid sizes must be >= 0");
    FPA_REQUIRE(pl.lambda1 && pl.lambda2 && pl.lambda3, "wavelength axes must be set");
    FPA_TRY(use_device(device));
    *ps = PendingSweep();
    const size_t n1 = (size_t)pl.n1, n3 = (size_t)pl.n3;
    FPA_REQUIRE(d->first_point >= 0 && d->n_sub_points >= 0 &&
                    (size_t)(d->first_point + d->n_sub_points) <= n1 * n3,
                "first_point / n_sub_points must select a range of the n1*n3 grid");
    // points of this call: the whole grid, or the sub-range (outputs are indexed from its first point)
    const size_t B = (d->first_point == 0 && d->n_sub_points == 0) ? n1 * n3 : (size_t)d->n_sub_points;
    if (B == 0) return FPA_OK;
    // the phase sweep may leave its gain map in the workspace (only the reductions come back)
    FPA_REQUIRE(ph || d->gain_lin != nullptr, "gain_lin must be set");
    const size_t K = ph ? (size_t)ph->n_phases : 1, P = B * K;
    const size_t n2 = pl.lambda2_stride ? n1 : 1;
    const size_t n_sched = (size_t)(ph ? yaman4_phase_scratch_bytes((int64_t)P) : yaman4_scratch_bytes((int64_t)B));
    const size_t n_red = ph ? B : 0;
    size_t need = Carver::need(n1 * 8) + Carver::need(n2 * 8) + Carver::need(n3 * 8) +
                  Carver::need(P * 8) /*gain*/ + Carver::need(B * 8) /*dbeta*/ +
                  Carver::need(B * 4) /*valid*/ + Carver::need(P * 4) /*status*/ +
                  Carver::need(P * 32) /*Pmax*/ + Carver::need(P * 64) /*A_end*/ +
                  Carver::need(B * 32) /*omega*/ + Carver::need(n_sched) +
                  Carver::need(K * 64) /*A0 table*/ + 2 * Carver::need(n_red * 8) + 3 * Carver::need(n_red * 4);
    void* ws = nullptr;
    FPA_TRY(workspace(device, 3, need, &ws));
    cudaStream_t st;
    FPA_TRY(host_stream(device, &st));
    Carver cv;
    cv.base = static_cast<char*>(ws);
    double*  l1   = cv.take<double>(n1);
    double*  l2   = cv.take<double>(n2);
    double*  l3   = cv.take<double>(n3);
    double*  gain = cv.take<double>(P);
    double*  db   = cv.take<double>(B);
    int32_t* va   = cv.take<int32_t>(B);
    int32_t* stt  = cv.take<int32_t>(P);
    double*  Pm   = cv.take<double>(P * 4);
    double*  Ae   = cv.take<double>(P * 8);
    double*  om   = cv.take<double>(B * 4);
    char*    sched = cv.take<char>(n_sched);
    double*  tab  = cv.take<double>(K * 8);
    double*  gmax = cv.take<double>(n_red);
    double*  gmin = cv.take<double>(n_red);
    int32_t* imax = cv.take<int32_t>(n_red);
    int32_t* imin = cv.take<int32_t>(n_red);
    int32_t* nfin = cv.take<int32_t>(n_red);

    FPA_TRY(up(l1, pl.lambda1, n1 * 8, st));
    FPA_TRY(up(l2, pl.lambda2, n2 * 8, st));
    FPA_TRY(up(l3, pl.lambda3, n3 * 8, st));
    if (ph) FPA_TRY(up(tab, ph->A0_table, K * 64, st));
    // Outputs in pinned host memory are written by the kernel itself (each thread stores its results
    // when it finishes, so the PCIe traffic hides behind the integration of the other points; measured
    // with 8 GPUs storing into one host at once: 44.1 ms per 8e6-point sweep against 46.0 ms with staging
    // and copies).  Pageable outputs go through the device workspace and a copy.  The phase sweep keeps its gain map
    // in device memory: the reduction kernel reads it there.
    double*  m_gain = ph ? nullptr : mapped(d->gain_lin);
    double*  m_db   = mapped(pl.dbeta);
    int32_t* m_va   = mapped(pl.valid);
    int32_t* m_st   = mapped(d->status);
    double*  m_Pm   = mapped(d->Pmax);
    double*  m_Ae   = mapped(d->A_end);
    fpa_sweep_desc dd = *d;
    dd.n_peers      = 0;   // peer maps are device pointers: a feature of the _dev entry
    dd.plan.lambda1 = l1;
    dd.plan.lambda2 = l2;
    dd.plan.lambda3 = l3;
    dd.plan.omega   = pl.omega ? om : nullptr;
    dd.plan.dbeta   = m_db ? m_db : db;
    dd.plan.valid   = m_va ? m_va : va;
    dd.gain_lin     = m_gain ? m_gain : gain;
    dd.Pmax         = d->Pmax ? (m_Pm ? m_Pm : Pm) : nullptr;
    dd.A_end        = d->A_end ? (m_Ae ? m_Ae : Ae) : nullptr;
    dd.status       = m_st ? m_st : stt;
    if (ph) {
        fpa_phase_sweep_desc pd = *ph;
        pd.sweep    = dd;
        pd.A0_table = tab;
        pd.gain_max = ph->gain_max ? gmax : nullptr;
        pd.gain_min = ph->gain_min ? gmin : nullptr;
        pd.idx_max  = ph->idx_max ? imax : nullptr;
        pd.idx_min  = ph->idx_min ? imin : nullptr;
        pd.n_finite = ph->n_finite ? nfin : nullptr;
        FPA_TRY(phase_sweep_dev(&pd, sched, (int64_t)n_sched, st));
        ps->puser = *ph;
        ps->gmax  = pd.gain_max;
        ps->gmin  = pd.gain_min;
        ps->imax  = pd.idx_max;
        ps->imin  = pd.idx_min;
        ps->nfin  = pd.n_finite;
    } else {
        FPA_TRY(sweep_dev(&dd, sched, (int64_t)n_sched, st));
    }
    ps->st   = st;
    ps->B    = B;
    ps->P    = P;
    ps->user = *d;
    ps->gain = (m_gain || !d->gain_lin) ? nullptr : gain;
    ps->db   = m_db ? nullptr : db;
    ps->va   = m_va ? nullptr : va;
    ps->om   = om;
    ps->stt  = m_st ? nullptr : stt;
    ps->Pm   = m_Pm ? nullptr : Pm;
    ps->Ae   = m_Ae ? nullptr : Ae;
    return FPA_OK;
}

static int sweep_host_collect(const PendingSweep& ps, int device) {
    if (!ps.st) return FPA_OK;
    FPA_TRY(use_device(device));
    const size_t B = ps.B, P = ps.P;
    if (ps.gain) FPA_TRY(down(ps.user.gain_lin, ps.gain, P * 8, ps.st));
    if (ps.db) FPA_TRY(down(ps.user.plan.dbeta, ps.db, B * 8, ps.st));
    if (ps.va) FPA_TRY(down(ps.user.plan.valid, ps.va, B * 4, ps.st));
    FPA_TRY(down(ps.user.plan.omega, ps.om, B * 32, ps.st));
    if (ps.stt) FPA_TRY(down(ps.user.status, ps.stt, P * 4, ps.st));
    if (ps.Pm) FPA_TRY(down(ps.user.Pmax, ps.Pm, P * 32, ps.st));
    if (ps.Ae) FPA_TRY(down(ps.user.A_end, ps.Ae, P * 64, ps.st));
    if (ps.gmax) FPA_TRY(down(ps.puser.gain_max, ps.gmax, B * 8, ps.st));
    if (ps.gmin) FPA_TRY(down(ps.puser.gain_min, ps.gmin, B * 8, ps.st));
    if (ps.imax) FPA_TRY(down(ps.puser.idx_max, ps.imax, B * 4, ps.st));
    if (ps.imin) FPA_TRY(down(ps.puser.idx_min, ps.imin, B * 4, ps.st));
    if (ps.nfin) FPA_TRY(down(ps.puser.n_finite, ps.nfin, B * 4, ps.st));
    return FPA_OK;
}

int fpa_yaman4_sweep_host(const fpa_sweep_desc* d, int device) {
    PendingSweep ps;
    FPA_TRY(sweep_host_launch(d, nullptr, device, &ps));
    FPA_TRY(sweep_host_collect(ps, device));
    if (ps.st) FPA_CUDA(cudaStreamSynchronize(ps.st));
    return FPA_OK;
}

// The grid split over several devices (see the header); `ph` set: a phase sweep, its K runs per grid point stay
// together.
static int sweep_multi_host(const fpa_sweep_desc* d, const fpa_phase_sweep_desc* ph, int n_devices, const int* devices) {
    FPA_REQUIRE(d != nullptr, "sweep descriptor is NULL");
    FPA_REQUIRE(n_devices >= 1 && n_devices <= 64 && devices != nullptr, "need 1..64 device ordinals");
    const int64_t n1 = d->plan.n1, n3 = d->plan.n3;
    FPA_REQUIRE(n1 >= 0 && n3 >= 0, "grid sizes must be >= 0");
    FPA_REQUIRE(d->first_point == 0 && d->n_sub_points == 0, "the multi-device sweep splits the whole grid itself");
    if (n_devices == 1) return ph ? fpa_yaman4_phase_sweep_host(ph, devices[0]) : fpa_yaman4_sweep_host(d, devices[0]);
    const int64_t K = ph ? ph->n_phases : 1;
    // contiguous ranges of the FLATTENED grid, sizes differing by at most one: a 1-D sweep (n1 = 1) or a
    // grid with fewer pump rows than devices still uses every device
    PendingSweep pend[64];
    return run_on_devices(
        n_devices, devices, pend,
        [&](int k, PendingSweep* ps) {
            int64_t lo, hi;
            balanced_range(n1 * n3, n_devices, k, &lo, &hi);
            *ps = PendingSweep();
            if (hi <= lo) return (int)FPA_OK;
            fpa_sweep_desc part = *d;
            part.first_point  = lo;
            part.n_sub_points = hi - lo;
            if (d->plan.omega) part.plan.omega = d->plan.omega + lo * 4;
            if (d->plan.dbeta) part.plan.dbeta = d->plan.dbeta + lo;
            if (d->plan.valid) part.plan.valid = d->plan.valid + lo;
            if (d->gain_lin) part.gain_lin = d->gain_lin + lo * K;
            if (d->Pmax) part.Pmax = d->Pmax + lo * K * 4;
            if (d->A_end) part.A_end = d->A_end + lo * K * 8;
            if (d->status) part.status = d->status + lo * K;
            if (!ph) return sweep_host_launch(&part, nullptr, devices[k], ps);
            fpa_phase_sweep_desc pp = *ph;
            if (ph->gain_max) pp.gain_max = ph->gain_max + lo;
            if (ph->gain_min) pp.gain_min = ph->gain_min + lo;
            if (ph->idx_max) pp.idx_max = ph->idx_max + lo;
            if (ph->idx_min) pp.idx_min = ph->idx_min + lo;
            if (ph->n_finite) pp.n_finite = ph->n_finite + lo;
            return sweep_host_launch(&part, &pp, devices[k], ps);
        },
        sweep_host_collect);
}

int fpa_yaman4_sweep_multi_host(const fpa_sweep_desc* d, int n_devices, const int* devices) {
    return sweep_multi_host(d, nullptr, n_devices, devices);
}

// ------------------------------------------------------------------ phase sweep
int64_t fpa_yaman4_phase_sweep_scratch_bytes(int64_t n_points) { return yaman4_phase_scratch_bytes(n_points); }

int fpa_yaman4_phase_sweep_dev(const fpa_phase_sweep_desc* d, void* scratch, int64_t scratch_bytes, void* stream) {
    if (fpa_device_count() <= 0) {
        set_error("no CUDA device is visible: libfpa_b200 has no CPU path");
        return FPA_ERR_NO_DEVICE;
    }
    return phase_sweep_dev(d, scratch, scratch_bytes, static_cast<cudaStream_t>(stream));
}

int fpa_yaman4_phase_sweep_host(const fpa_phase_sweep_desc* d, int device) {
    FPA_REQUIRE(d != nullptr, "phase sweep descriptor is NULL");
    PendingSweep ps;
    FPA_TRY(sweep_host_launch(&d->sweep, d, device, &ps));
    FPA_TRY(sweep_host_collect(ps, device));
    if (ps.st) FPA_CUDA(cudaStreamSynchronize(ps.st));
    return FPA_OK;
}

int fpa_yaman4_phase_sweep_multi_host(const fpa_phase_sweep_desc* d, int n_devices, const int* devices) {
    FPA_REQUIRE(d != nullptr, "phase sweep descriptor is NULL");
    return sweep_multi_host(&d->sweep, d, n_devices, devices);
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
    const size_t n_grid = z_grid ? (size_t)n_steps + 1 : 0;
    const size_t n_tr = trace ? n * ns * 2 : 0;
    void* ws = nullptr;
    FPA_TRY(workspace(device, 4,
                      2 * Carver::need(n * 16) + Carver::need((size_t)dim * 16) + Carver::need(n_grid * 8) +
                          Carver::need(n_tr * 8) + Carver::need(n * 4) + Carver::need((size_t)B * 4),
                      &ws));
    cudaStream_t st;
    FPA_TRY(host_stream(device, &st));
    Carver cv;
    cv.base = static_cast<char*>(ws);
    double*  dy0  = cv.take<double>(n * 2);
    double*  dye  = cv.take<double>(n * 2);
    double*  dlam = cv.take<double>((size_t)dim * 2);
    double*  grid = cv.take<double>(n_grid);
    double*  dtr  = cv.take<double>(n_tr);
    int32_t* bad  = cv.take<int32_t>(n);
    int32_t* stt  = cv.take<int32_t>((size_t)B);
    FPA_TRY(up(dy0, y0, n * 16, st));
    FPA_TRY(up(dlam, lam, (size_t)dim * 16, st));
    FPA_TRY(up(grid, z_grid, n_grid * 8, st));
    FPA_TRY(linear_launch(B, (int)dim, dy0, dlam, z0, z_max, n_steps, save_every, z_grid ? grid : nullptr,
                          flags, dtr, dye, bad, stt, st));
    if (trace) FPA_TRY(down(y_trace, dtr, n_tr * 8, st));
    if (endo) FPA_TRY(down(y_end, dye, n * 16, st));
    FPA_TRY(down(status, stt, (size_t)B * 4, st));
    FPA_CUDA(cudaStreamSynchronize(st));
    return FPA_OK;
}

// ------------------------------------------------------------------ N-wave integrator
int fpa_nwave_rk4_batch_dev(const fpa_nwave_desc* d, void* stream) {
    if (fpa_device_count() <= 0) {
        set_error("no CUDA device is visible: libfpa_b200 has no CPU path");
        return FPA_ERR_NO_DEVICE;
    }
    return nwave_dispatch(d, static_cast<cudaStream_t>(stream));
}

struct PendingNwave {
    cudaStream_t st = nullptr;
    size_t       B = 0, N = 0, n_tr = 0;
    double * tr = nullptr, *Ae = nullptr, *Pm = nullptr;
    int32_t* stt = nullptr;
    fpa_nwave_desc user;
};

static int nwave_host_check(const fpa_nwave_desc* d) {
    FPA_REQUIRE(d != nullptr, "descriptor is NULL");
    FPA_REQUIRE(d->n_points >= 0, "n_points must be >= 0");
    FPA_REQUIRE(d->n_waves >= 1, "n_waves must be >= 1");
    FPA_REQUIRE(d->n_steps >= 1, "n_steps must be >= 1");
    FPA_REQUIRE(d->save_every >= 1, "save_every must be a positive integer");
    FPA_REQUIRE(d->beta && d->gamma && d->alpha && d->A0, "beta/gamma/alpha/A0 must be set");
    FPA_REQUIRE(!((d->flags & FPA_NWAVE_TABLE) && (d->flags & FPA_NWAVE_COMB)), "FPA_NWAVE_TABLE and FPA_NWAVE_COMB exclude each other");
    FPA_REQUIRE(!(d->flags & FPA_NWAVE_COMB) || d->grid_slot, "FPA_NWAVE_COMB needs grid_slot");
    const bool comb = nwave_use_comb(d);
    FPA_REQUIRE(comb || (d->n_triplets >= 0 && d->row_ptr), "triplet table must be set");
    FPA_REQUIRE((d->gamma_stride | 1) == 1 && (d->alpha_stride | 1) == 1 && (d->A0_stride | 1) == 1 &&
                    (d->beta_stride | 1) == 1,
                "strides must be 0 (broadcast) or 1 (per point)");
    FPA_REQUIRE(!(d->flags & FPA_OUT_TRACE) || d->A_trace, "FPA_OUT_TRACE needs A_trace");
    FPA_REQUIRE(!(d->flags & FPA_OUT_PMAX) || d->Pmax, "FPA_OUT_PMAX needs Pmax");
    FPA_REQUIRE(!(d->flags & FPA_OUT_END) || d->A_end, "FPA_OUT_END needs A_end");
    if (d->grid_slot) {   // host pointers here: the slots can be checked
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

static int nwave_host_launch(const fpa_nwave_desc* d, int device, PendingNwave* pn) {
    FPA_TRY(nwave_host_check(d));
    const bool comb = nwave_use_comb(d);
    const bool trace = (d->flags & FPA_OUT_TRACE) != 0, endo = (d->flags & FPA_OUT_END) != 0;
    const bool pmax = (d->flags & FPA_OUT_PMAX) != 0;
    FPA_TRY(use_device(device));
    *pn = PendingNwave();
    const size_t B = (size_t)d->n_points, N = (size_t)d->n_waves;
    if (B == 0) return FPA_OK;
    const size_t ns = (size_t)fpa_n_saved(d->n_steps, d->save_every);
    const size_t n_b = (d->beta_stride ? B : 1) * N, n_g = d->gamma_stride ? B : 1;
    const size_t n_a = d->alpha_stride ? B : 1, n_A0 = (d->A0_stride ? B : 1) * N * 2;
    const size_t n_t = comb ? 0 : (size_t)d->n_triplets;
    const size_t n_tr = trace ? B * ns * N * 2 : 0;
    // the table kernel gets the factored form of the table (unless the caller insists on the entry list)
    std::vector<unsigned char> blob;
    int32_t                    n_classes = 0;
    if (!comb && !(d->flags & FPA_NWAVE_PLAIN) && N <= 128) {
        const int64_t nb = fpa_nwave_factor_table((int32_t)N, d->triplets, d->row_ptr, d->n_triplets, nullptr, 0, &n_classes);
        if (nb < 0) return FPA_ERR_INVALID;
        blob.resize((size_t)nb);
        if (fpa_nwave_factor_table((int32_t)N, d->triplets, d->row_ptr, d->n_triplets, blob.data(), nb, &n_classes) != nb) return FPA_ERR_INVALID;
    }
    void* ws = nullptr;
    FPA_TRY(workspace(device, 5,
                      Carver::need(blob.size()) + Carver::need(n_b * 8) + Carver::need(n_g * 8) + Carver::need(n_a * 8) +
                          Carver::need(n_A0 * 8) + Carver::need(n_t * sizeof(fpa_triplet)) +
                          Carver::need((N + 1) * 8) + Carver::need(n_tr * 8) +
                          Carver::need(B * N * 16) + Carver::need(B * N * 8) + Carver::need(B * 4) +
                          Carver::need(N * 4),
                      &ws));
    cudaStream_t st;
    FPA_TRY(host_stream(device, &st));
    Carver cv;
    cv.base = static_cast<char*>(ws);
    double*      beta = cv.take<double>(n_b);
    double*      gam  = cv.take<double>(n_g);
    double*      alp  = cv.take<double>(n_a);
    double*      A0   = cv.take<double>(n_A0);
    fpa_triplet* tab  = cv.take<fpa_triplet>(n_t);
    int64_t*     rows = cv.take<int64_t>(N + 1);
    double*      tr   = cv.take<double>(n_tr);
    double*      Ae   = cv.take<double>(B * N * 2);
    double*      Pm   = cv.take<double>(B * N);
    int32_t*     stt  = cv.take<int32_t>(B);
    int32_t*     slot = cv.take<int32_t>(N);
    unsigned char* fact = cv.take<unsigned char>(blob.size());
    if (comb) FPA_TRY(up(slot, d->grid_slot, N * 4, st));
    if (!blob.empty()) FPA_TRY(up(fact, blob.data(), blob.size(), st));
    FPA_TRY(up(beta, d->beta, n_b * 8, st));
    FPA_TRY(up(gam, d->gamma, n_g * 8, st));
    FPA_TRY(up(alp, d->alpha, n_a * 8, st));
    FPA_TRY(up(A0, d->A0, n_A0 * 8, st));
    if (!comb) {
        FPA_TRY(up(tab, d->triplets, n_t * sizeof(fpa_triplet), st));
        FPA_TRY(up(rows, d->row_ptr, (N + 1) * 8, st));
    }
    fpa_nwave_desc dd = *d;
    dd.beta     = beta;
    dd.gamma    = gam;
    dd.alpha    = alp;
    dd.A0       = A0;
    dd.triplets = tab;
    dd.row_ptr  = rows;
    dd.A_trace  = trace ? tr : nullptr;
    dd.A_end    = endo ? Ae : nullptr;
    dd.Pmax     = pmax ? Pm : nullptr;
    dd.status   = stt;
    dd.grid_slot = comb ? slot : nullptr;
    dd.factored  = blob.empty() ? nullptr : fact;
    dd.n_classes = n_classes;
    dd.flags = (d->flags & ~(FPA_NWAVE_TABLE | FPA_NWAVE_COMB)) | (comb ? FPA_NWAVE_COMB : FPA_NWAVE_TABLE);  // decided above
    FPA_TRY(nwave_dispatch(&dd, st));
    pn->st   = st;
    pn->B    = B;
    pn->N    = N;
    pn->n_tr = n_tr;
    pn->user = *d;
    pn->tr   = trace ? tr : nullptr;
    pn->Ae   = endo ? Ae : nullptr;
    pn->Pm   = pmax ? Pm : nullptr;
    pn->stt  = stt;
    return FPA_OK;
}

static int nwave_host_collect(const PendingNwave& pn, int device) {
    if (!pn.st) return FPA_OK;
    FPA_TRY(use_device(device));
    if (pn.tr) FPA_TRY(down(pn.user.A_trace, pn.tr, pn.n_tr * 8, pn.st));
    if (pn.Ae) FPA_TRY(down(pn.user.A_end, pn.Ae, pn.B * pn.N * 16, pn.st));
    if (pn.Pm) FPA_TRY(down(pn.user.Pmax, pn.Pm, pn.B * pn.N * 8, pn.st));
    FPA_TRY(down(pn.user.status, pn.stt, pn.B * 4, pn.st));
    return FPA_OK;
}

int fpa_nwave_rk4_batch_host(const fpa_nwave_desc* d, int device) {
    PendingNwave pn;
    FPA_TRY(nwave_host_launch(d, device, &pn));
    FPA_TRY(nwave_host_collect(pn, device));
    if (pn.st) FPA_CUDA(cudaStreamSynchronize(pn.st));
    return FPA_OK;
}

int fpa_nwave_rk4_batch_multi_host(const fpa_nwave_desc* d, int n_devices, const int* devices) {
    FPA_TRY(nwave_host_check(d));
    FPA_REQUIRE(n_devices >= 1 && n_devices <= 64 && devices != nullptr, "need 1..64 device ordinals");
    if (n_devices == 1) return fpa_nwave_rk4_batch_host(d, devices[0]);
    const int64_t ns = fpa_n_saved(d->n_steps, d->save_every), N = d->n_waves;
    PendingNwave  pend[64];
    return run_on_devices(
        n_devices, devices, pend,
        [&](int k, PendingNwave* pn) {
            int64_t lo, hi;
            balanced_range(d->n_points, n_devices, k, &lo, &hi);
            *pn = PendingNwave();
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
            return nwave_host_launch(&part, devices[k], pn);
        },
        nwave_host_collect);
}

// ------------------------------------------------------------------ measurement helpers
int fpa_fp64_peak_probe(int device, int iters, double* tflops, double* ms) {
    return probe_run(device, iters, tflops, ms);
}

int fpa_host_alloc(void** ptr, int64_t bytes) {
    FPA_REQUIRE(ptr != nullptr && bytes >= 0, "bad arguments");
    if (fpa_device_count() <= 0) {
        set_error("no CUDA device is visible: pinned host memory needs the CUDA runtime");
        return FPA_ERR_NO_DEVICE;
    }
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
    if (fpa_device_count() <= 0) {
        set_error("no CUDA device is visible: page-locking host memory needs the CUDA runtime");
        return FPA_ERR_NO_DEVICE;
    }
    FPA_CUDA(cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterPortable | cudaHostRegisterMapped));
    return FPA_OK;
}

int fpa_host_unregister(void* ptr) {
    if (ptr == nullptr) return FPA_OK;
    FPA_CUDA(cudaHostUnregister(ptr));
    return FPA_OK;
}

}  // extern "C"
