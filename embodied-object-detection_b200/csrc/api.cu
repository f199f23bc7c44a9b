// libeod_memory.so: error reporting and device queries shared by all entry points.
#include <stdarg.h>
#include <string.h>

#include "eod_common.cuh"
#include "tmap_cache.cuh"

static thread_local char g_err[512] = "";

void eod_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int eod_check_launch(const char *what)
{
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        eod_set_error("%s: %s", what, cudaGetErrorString(e));
        return EOD_ERR_LAUNCH;
    }
    return EOD_OK;
}

int eod_num_sms()
{
    static int cache[64] = {0};                 // per device ordinal (a process may drive several GPUs)
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
    int &n = cache[dev & 63];
    if (!n) {
        int v = 0;
        n = (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0) ? v : EOD_NUM_SMS_FALLBACK;
    }
    return n;
}

PFN_eodEncodeTiled eod_encode_tiled_fn()
{
    static const PFN_eodEncodeTiled fn = [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        const bool ok = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess;
        return ok ? reinterpret_cast<PFN_eodEncodeTiled>(p) : nullptr;
    }();
    return fn;
}

// Work tickets for persistent kernels that claim their tiles dynamically: a pool of zeroed {next, done} int pairs per device.
// A launch takes the next pair of the pool; the kernel's last CTA re-arms it (both words back to 0), so a pair is reusable as
// soon as its launch has finished.  1024 pairs per device, handed out round-robin: two launches on DIFFERENT streams could only meet on
// one pair if one stream ran more than a thousand ticketed launches behind the other (launches of one stream are ordered anyway).  The pool is allocated at the first call on a device (never
// call it inside a CUDA graph capture: captured launches take the static partition); nullptr = allocation failed (callers fall back to static partitioning).
int *eod_work_tickets()
{
    constexpr int kPairs = 1024;
    static int *pool[64] = {nullptr};
    static unsigned next[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
    int *p = __atomic_load_n(&pool[dev & 63], __ATOMIC_ACQUIRE);
    if (!p) {
        int *fresh = nullptr;
        if (cudaMalloc(&fresh, kPairs * 2 * sizeof(int)) != cudaSuccess || cudaMemset(fresh, 0, kPairs * 2 * sizeof(int)) != cudaSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        int *expected = nullptr;
        if (__atomic_compare_exchange_n(&pool[dev & 63], &expected, fresh, false, __ATOMIC_ACQ_REL, __ATOMIC_ACQUIRE)) p = fresh;
        else { cudaFree(fresh); p = expected; }
    }
    const unsigned k = __atomic_fetch_add(&next[dev & 63], 1u, __ATOMIC_RELAXED) % kPairs;
    return p + 2 * k;
}

extern "C" int eod_version(void) { return 100; /* 0.1.0 */ }
extern "C" const char *eod_last_error(void) { return g_err; }
