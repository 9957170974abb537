// frontend.cu -- stand-alone Delta-beta table kernel (fpa_dbeta_table_*): frequency plan ->
// validity -> Delta-beta for every point of a (pump x signal) wavelength grid.  The per-point
// arithmetic lives in plan_point.cuh (shared with the fused sweep kernel in yaman4.cu), which
// cites the reference lines it restates.  Also the per-grid-point reductions of the phase sweep
// (fpa_yaman4_phase_sweep_*), which run right after its sweep kernel.
#include "plan_point.cuh"

namespace fpa {

__global__ void plan_dbeta_kernel(const PlanParams p) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t B = p.n1 * p.n3;
    if (b >= B) return;
    const int64_t i1 = b / p.n3, i3 = b - i1 * p.n3;
    double w[4];
    bool   ok = plan_omegas(p.lambda1[i1], p.lambda2[i1 * p.lambda2_stride], p.lambda3[i3], w);
    const double db = plan_dbeta(p, p.beta, p.provided, w, ok);

    if (p.dbeta) p.dbeta[b] = db;
    if (p.dbeta_masked) p.dbeta_masked[b] = ok ? db : 0.0;
    if (p.valid) p.valid[b] = ok ? 1 : 0;
    if (p.omega) {
        double2* o = reinterpret_cast<double2*>(p.omega + b * 4);
        o[0] = make_double2(w[0], w[1]);
        o[1] = make_double2(w[2], w[3]);
    }
}

// Validate a plan descriptor and copy it into the kernel-side struct.
int plan_fill(const fpa_plan_desc* d, PlanParams& p) {
    FPA_REQUIRE(d != nullptr, "plan descriptor is NULL");
    FPA_REQUIRE(d->n1 >= 0 && d->n3 >= 0, "grid sizes must be >= 0");
    FPA_REQUIRE(d->lambda1 && d->lambda2 && d->lambda3, "wavelength axes must be set");
    FPA_REQUIRE(d->method >= 0 && d->method <= 2, "unknown phase-matching method %d", d->method);
    FPA_REQUIRE(d->max_order >= 0, "max_order must be >= 0");
    FPA_REQUIRE(d->n_even >= 0 && d->n_even <= FPA_MAX_TAYLOR_ORDER, "too many even orders");
    FPA_REQUIRE((d->lambda2_stride | 1) == 1, "lambda2_stride must be 0 or 1");
    if (d->method == FPA_PM_GENERAL_TAYLOR && d->max_order > FPA_MAX_TAYLOR_ORDER) {
        set_error("max_order %d exceeds the supported Taylor order %d", d->max_order, FPA_MAX_TAYLOR_ORDER);
        return FPA_ERR_UNSUPPORTED;
    }
    for (int e = 0; e < d->n_even; ++e) {
        if (d->method == FPA_PM_SYMMETRIC_EVEN && d->even_orders[e] > FPA_MAX_TAYLOR_ORDER) {
            set_error("even order %d exceeds the supported Taylor order %d", d->even_orders[e],
                      FPA_MAX_TAYLOR_ORDER);
            return FPA_ERR_UNSUPPORTED;
        }
    }
    p.n1 = d->n1;
    p.n3 = d->n3;
    p.lambda1 = d->lambda1;
    p.lambda2 = d->lambda2;
    p.lambda3 = d->lambda3;
    p.lambda2_stride = (int)d->lambda2_stride;
    p.method = d->method;
    p.max_order = d->max_order;
    p.n_even = d->n_even;
    for (int i = 0; i < FPA_MAX_TAYLOR_ORDER; ++i) p.even_orders[i] = d->even_orders[i];
    for (int i = 0; i <= FPA_MAX_TAYLOR_ORDER; ++i) p.beta[i] = d->beta[i];
    p.omega_ref = d->omega_ref;
    p.atol = d->atol;
    p.rtol = d->rtol;
    p.provided = d->provided;
    p.omega = d->omega;
    p.dbeta = d->dbeta;
    p.dbeta_masked = nullptr;
    p.valid = d->valid;
    return FPA_OK;
}

int plan_launch(const fpa_plan_desc* d, double* dbeta_masked, cudaStream_t st) {
    PlanParams p;
    int rc = plan_fill(d, p);
    if (rc != FPA_OK) return rc;
    FPA_REQUIRE(d->dbeta || dbeta_masked, "a dbeta output must be set");
    FPA_REQUIRE_ALIGNED16(d->omega, "omega");  // stored with 16-byte vector stores
    p.dbeta_masked = dbeta_masked;
    const int64_t B = d->n1 * d->n3;
    if (B == 0) return FPA_OK;

    const int threads = 256;
    plan_dbeta_kernel<<<(unsigned)((B + threads - 1) / threads), threads, 0, st>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "plan_dbeta_kernel launch");
    return FPA_OK;
}

// Per-grid-point reductions of a phase sweep (fpa_yaman4_phase_sweep_*): one thread per grid point over the K gains
// gain[g*K .. g*K+K-1], with numpy's semantics -- nanmax / nanmin, nanargmax / nanargmin (first index on ties),
// the count of non-NaN gains; an all-NaN row gives NaN, -1, -1, 0.
__global__ void phase_reduce_kernel(int64_t G, int K, const double* gain, double* gmax, double* gmin, int32_t* imax,
                                    int32_t* imin, int32_t* nfin) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    const double* r  = gain + g * K;
    double        hi = qnan(), lo = qnan();
    int           ih = -1, il = -1, n = 0;
    for (int k = 0; k < K; ++k) {
        const double v = r[k];
        if (v != v) continue;
        ++n;
        if (ih < 0 || v > hi) {
            hi = v;
            ih = k;
        }
        if (il < 0 || v < lo) {
            lo = v;
            il = k;
        }
    }
    if (gmax) gmax[g] = hi;
    if (gmin) gmin[g] = lo;
    if (imax) imax[g] = ih;
    if (imin) imin[g] = il;
    if (nfin) nfin[g] = n;
}

int phase_reduce_launch(int64_t G, int K, const double* gain, double* gmax, double* gmin, int32_t* imax, int32_t* imin,
                        int32_t* nfin, cudaStream_t st) {
    if (G == 0 || !(gmax || gmin || imax || imin || nfin)) return FPA_OK;
    const int threads = 256;
    phase_reduce_kernel<<<(unsigned)((G + threads - 1) / threads), threads, 0, st>>>(G, K, gain, gmax, gmin, imax, imin,
                                                                                  nfin);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "phase_reduce_kernel launch");
    return FPA_OK;
}

}  // namespace fpa
