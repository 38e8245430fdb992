// Handle lifetime, error reporting and kernel hyper-parameter set-up of the gpexp_b200 C ABI.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include "gpx_common.cuh"

#include <atomic>

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};  // kernel launches issued by this library (every launch site checks once)

void gpx_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int gpx_check_launch(const char* what) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        gpx_set_error("%s: %s", what, cudaGetErrorString(e));
        return (int)e;
    }
    return GPX_OK;
}

int gpx_ensure_smem(gpx_handle h, const void* func, size_t bytes, const char* name) {
    for (int i = 0; i < h->n_smem_ready; ++i)
        if (h->smem_ready[i] == func) return GPX_OK;
    int cur = -1;
    cudaGetDevice(&cur);
    if (cur != h->device) cudaSetDevice(h->device);
    cudaError_t e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (cur != h->device && cur >= 0) cudaSetDevice(cur);
    if (e != cudaSuccess) {
        gpx_set_error("%s: cannot opt in to %zu bytes of shared memory: %s", name, bytes, cudaGetErrorString(e));
        return (int)e;
    }
    if (h->n_smem_ready < GPX_SMEM_FUNCS) h->smem_ready[h->n_smem_ready++] = func;
    return GPX_OK;
}

extern "C" int gpx_version(void) { return GPX_VERSION; }

extern "C" int64_t gpx_launch_count(void) { return (int64_t)g_launches.load(std::memory_order_relaxed); }

extern "C" const char* gpx_last_error(void) { return g_err; }

extern "C" int gpx_create(int device, gpx_handle* out) {
    GPX_REQUIRE(out != nullptr, GPX_EINVAL, "out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        gpx_set_error("gpx_create: no CUDA device (%s); this library has no CPU fallback",
                      e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
        return e == cudaSuccess ? (int)cudaErrorNoDevice : (int)e;
    }
    GPX_REQUIRE(device >= 0 && device < count, GPX_EINVAL, "device out of range");
    e = cudaSetDevice(device);
    if (e != cudaSuccess) {
        gpx_set_error("gpx_create: cudaSetDevice: %s", cudaGetErrorString(e));
        return (int)e;
    }
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    if (prop.major < 10) {
        gpx_set_error("gpx_create: device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major,
                      prop.minor);
        return (int)cudaErrorInvalidDevice;
    }
    gpx_context* c = new gpx_context();
    memset(c, 0, sizeof(*c));
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    {
        const char* e = getenv("GPX_IVAR_RING");
        c->ivar_ring = (e && e[0] >= '0' && e[0] <= '2' && e[1] == 0) ? (e[0] - '0') : GPX_DEFAULT_IVAR_RING;
        const char* k = getenv("GPX_IVAR_CORE");
        c->ivar_core = (k && strcmp(k, "dmma") == 0) ? GPX_CORE_DMMA : GPX_CORE_I8;
    }
    bool ok = cudaMalloc(&c->red_val, GPX_RED_SLOTS * sizeof(double)) == cudaSuccess &&
              cudaMalloc(&c->red_idx, GPX_RED_SLOTS * sizeof(int64_t)) == cudaSuccess &&
              cudaMalloc(&c->red_counter, 16 * sizeof(unsigned int)) == cudaSuccess &&
              cudaMalloc(&c->scal, 16 * sizeof(double)) == cudaSuccess &&
              cudaMalloc(&c->iscal, 16 * sizeof(int64_t)) == cudaSuccess;
    if (!ok) {
        gpx_set_error("gpx_create: cudaMalloc of the reduction scratch failed");
        gpx_destroy(c);
        return (int)cudaErrorMemoryAllocation;
    }
    cudaMemset(c->red_counter, 0, 16 * sizeof(unsigned int));
    cudaMemset(c->scal, 0, 16 * sizeof(double));
    cudaMemset(c->iscal, 0, 16 * sizeof(int64_t));
    *out = c;
    return GPX_OK;
}

extern "C" int gpx_destroy(gpx_handle h) {
    if (!h) return GPX_OK;
    cudaFree(h->red_val);
    cudaFree(h->red_idx);
    cudaFree(h->red_counter);
    cudaFree(h->scal);
    cudaFree(h->iscal);
    delete h;
    return GPX_OK;
}

extern "C" int gpx_set_kernel(gpx_handle h, int family, int d, const double* p, int nparams) {
    GPX_REQUIRE(h != nullptr, GPX_EINVAL, "handle is NULL");
    GPX_REQUIRE(p != nullptr, GPX_EINVAL, "params_host is NULL");
    GPX_REQUIRE(d >= 1 && d <= GPX_MAX_DIM, GPX_ESIZE, "dimension must be in 1..GPX_MAX_DIM");
    KParams kp;
    memset(&kp, 0, sizeof(kp));
    kp.family = family;
    kp.d = d;
    if (family == GPX_SE) {
        GPX_REQUIRE(nparams == d + 1, GPX_EINVAL, "SE expects cl[d], signalSize");
        for (int i = 0; i < d; ++i) {
            GPX_REQUIRE(p[i] != 0.0, GPX_EINVAL, "correlation length must be non-zero");
            kp.a[i] = pow(p[i], -2.0);  // np: cl**-2.0 (kernels.py:122)
        }
        kp.signal = p[d];
    } else if (family == GPX_MATERN32) {
        GPX_REQUIRE(nparams == 2, GPX_EINVAL, "MATERN32 expects rho, signalSize");
        GPX_REQUIRE(p[0] != 0.0, GPX_EINVAL, "rho must be non-zero");
        kp.c0 = sqrt(3.0) / p[0];
        kp.signal = p[1];
    } else if (family == GPX_MATERN12 || family == GPX_MATERN52) {
        // c0 = sqrt(2 nu) / rho, the scaling kernels.py:87-89 uses for nu = 3/2
        GPX_REQUIRE(nparams == 2, GPX_EINVAL, "MATERN12 / MATERN52 expect rho, signalSize");
        GPX_REQUIRE(p[0] != 0.0, GPX_EINVAL, "rho must be non-zero");
        kp.c0 = (family == GPX_MATERN12 ? 1.0 : sqrt(5.0)) / p[0];
        kp.signal = p[1];
    } else if (family == GPX_MEHLER) {
        GPX_REQUIRE(nparams == d, GPX_EINVAL, "MEHLER expects t[d]");
        double pref = 1.0;
        for (int i = 0; i < d; ++i) {
            const double t = p[i];
            GPX_REQUIRE(fabs(t) < 1.0, GPX_EINVAL, "Mehler parameter must satisfy |t| < 1");
            kp.a[i] = t * t;
            kp.b[i] = 2.0 * t;
            kp.c[i] = 1.0 / (2.0 * (1.0 - t * t));
            pref *= pow(1.0 - t * t, -0.5);
        }
        kp.signal = pref;
    } else {
        GPX_REQUIRE(false, GPX_EINVAL, "unknown kernel family");
    }
    h->kp = kp;
    h->has_kernel = true;
    h->has_measure = false;  // a measure's constants belong to one kernel
    memset(h->center, 0, sizeof(h->center));  // a centre belongs to one kernel / data set
    return GPX_OK;
}
