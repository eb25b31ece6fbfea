// mc3_b200 -- error state, device queries, FMA-peak microbenchmark.
#include <stdarg.h>
#include <string.h>
#include "common.cuh"

static thread_local char g_err[512] = "";

void mc3b_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int mc3b_sm_count() {
    static int cached[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); return -1; }
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
            cudaGetLastError();
            return -1;
        }
        cached[dev] = n;
    }
    return cached[dev];
}

extern "C" int mc3b_version(void) { return MC3B_VERSION; }
extern "C" const char* mc3b_last_error(void) { return g_err; }
extern "C" int mc3b_device_sms(void) { return mc3b_sm_count(); }

// ---- peer memory (CUDA IPC) for the multi-GPU exchange ------------------------
extern "C" int mc3b_peer_alloc(int64_t nbytes, void** ptr, unsigned char* handle64) {
    MC3B_CHECK_ARG(nbytes > 0 && ptr && handle64, "bad arguments");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    void* p = nullptr;
    MC3B_CUDA(cudaMalloc(&p, (size_t)nbytes));
    MC3B_CUDA(cudaMemset(p, 0, (size_t)nbytes));
    MC3B_CUDA(cudaDeviceSynchronize());
    cudaIpcMemHandle_t h;
    MC3B_CUDA(cudaIpcGetMemHandle(&h, p));
    memcpy(handle64, &h, 64);
    *ptr = p;
    return MC3B_OK;
}
extern "C" int mc3b_peer_open(const unsigned char* handle64, void** ptr) {
    MC3B_CHECK_ARG(handle64 && ptr, "bad arguments");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    void* p = nullptr;
    MC3B_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    *ptr = p;
    return MC3B_OK;
}
extern "C" int mc3b_peer_close(void* ptr) {
    MC3B_CHECK_ARG(ptr, "null pointer");
    MC3B_CUDA(cudaIpcCloseMemHandle(ptr));
    return MC3B_OK;
}
extern "C" int mc3b_peer_free(void* ptr) {
    MC3B_CHECK_ARG(ptr, "null pointer");
    MC3B_CUDA(cudaFree(ptr));
    return MC3B_OK;
}

extern "C" int mc3b_host_device_pointer(void* host, void** dev) {
    MC3B_CHECK_ARG(host && dev, "bad arguments");
    MC3B_CUDA(cudaHostGetDevicePointer(dev, host, 0));
    return MC3B_OK;
}

// Roofline denominator: 8 independent accumulators per thread, each a chain of
// dependent FMAs; 256 threads x 8 CTAs per SM keeps the pipe full.
namespace {
template <typename T>
__global__ void __launch_bounds__(256) k_fma_peak(int64_t iters, double* sink) {
    T a[8];
#pragma unroll
    for (int k = 0; k < 8; k++) a[k] = (T)(threadIdx.x + k) * (T)1e-3;
    const T m = (T)0.999999, c = (T)1e-7;
    for (int64_t i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 8; k++) a[k] = fma(a[k], m, c);
    }
    T s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) s += a[k];
    if (s == (T)123456.789) sink[0] = (double)s;     // never true; keeps the loop alive
}
}  // namespace

// Variants that mimic the model kernel's operand kinds (fp64 only):
//   1: 8 chains per thread, c operand from the constant bank / uniform registers
//   2: 4 chains per thread (the kernel's ILP), constant operands, 6 CTAs of 128
__device__ __constant__ double kPeakC[8] = {1e-7, 2e-7, 3e-7, 4e-7, 5e-7, 6e-7, 7e-7, 8e-7};
template <int NCH>
__global__ void k_fma_const(int64_t iters, double* sink) {
    double a[NCH];
#pragma unroll
    for (int k = 0; k < NCH; k++) a[k] = (double)(threadIdx.x + k) * 1e-3;
    const double m = 0.999999 + 1e-9 * threadIdx.x;
    for (int64_t i = 0; i < iters; i++) {
#pragma unroll
        for (int j = 0; j < 8; j++) {
#pragma unroll
            for (int k = 0; k < NCH; k++) a[k] = fma(a[k], m, kPeakC[j]);
        }
    }
    double s = 0;
#pragma unroll
    for (int k = 0; k < NCH; k++) s += a[k];
    if (s == 123456.789) sink[0] = s;
}

//   5: every FMA reads three different vector registers that no neighbour shares
//      (register-file operand bandwidth instead of pipe issue rate)
//   6: two different vector registers + one shared multiplier
template <int MODE>
__global__ void __launch_bounds__(128, 6) k_fma_regs(int64_t iters, double* sink) {
    double a[8], b[8], c[8];
#pragma unroll
    for (int k = 0; k < 8; k++) {
        a[k] = (double)(threadIdx.x + k) * 1e-3;
        b[k] = 0.999999 + 1e-9 * (threadIdx.x + k);
        c[k] = 1e-7 * (threadIdx.x + 3 * k + 1);
    }
    for (int64_t i = 0; i < iters; i++) {
#pragma unroll
        for (int j = 0; j < 8; j++) {
#pragma unroll
            for (int k = 0; k < 8; k++) {
                if (MODE == 5) a[k] = fma(a[k], b[(k + j) & 7], c[(k + 3 * j + 1) & 7]);
                else a[k] = fma(a[k], b[0], c[(k + 3 * j + 1) & 7]);
            }
        }
    }
    double s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) s += a[k];
    if (s == 123456.789) sink[0] = s;
}

extern "C" int mc3b_fma_peak_variant(int variant, int64_t iters, double* sink, double* flops, void* stream) {
    MC3B_CHECK_ARG(sink && flops && iters > 0, "bad arguments");
    int sms = mc3b_sm_count();
    MC3B_CHECK_ARG(sms > 0, "no CUDA device");
    if (variant == 1) {
        k_fma_const<8><<<sms * 8, 256, 0, (cudaStream_t)stream>>>(iters, sink);
        *flops = 2.0 * 8.0 * 8.0 * 256.0 * sms * 8.0 * (double)iters;
    } else if (variant == 2) {
        k_fma_const<4><<<sms * 6, 128, 0, (cudaStream_t)stream>>>(iters, sink);
        *flops = 2.0 * 8.0 * 4.0 * 128.0 * sms * 6.0 * (double)iters;
    } else if (variant == 3) {
        k_fma_const<2><<<sms * 8, 128, 0, (cudaStream_t)stream>>>(iters, sink);
        *flops = 2.0 * 8.0 * 2.0 * 128.0 * sms * 8.0 * (double)iters;
    } else if (variant == 4) {
        k_fma_const<1><<<sms * 8, 128, 0, (cudaStream_t)stream>>>(iters, sink);
        *flops = 2.0 * 8.0 * 1.0 * 128.0 * sms * 8.0 * (double)iters;
    } else if (variant == 5 || variant == 6) {
        if (variant == 5) k_fma_regs<5><<<sms * 6, 128, 0, (cudaStream_t)stream>>>(iters, sink);
        else k_fma_regs<6><<<sms * 6, 128, 0, (cudaStream_t)stream>>>(iters, sink);
        *flops = 2.0 * 8.0 * 8.0 * 128.0 * sms * 6.0 * (double)iters;
    } else { mc3b_set_error("bad variant %d", variant); return MC3B_ERR_ARG; }
    MC3B_CHECK_LAUNCH("k_fma_const");
    return MC3B_OK;
}

extern "C" int mc3b_fma_peak(int dtype, int64_t iters, double* sink, double* flops, void* stream) {
    MC3B_CHECK_ARG(sink && flops && iters > 0, "bad arguments");
    int sms = mc3b_sm_count();
    MC3B_CHECK_ARG(sms > 0, "no CUDA device");
    const int ctas = sms * 8;
    if (dtype == MC3B_F64) k_fma_peak<double><<<ctas, 256, 0, (cudaStream_t)stream>>>(iters, sink);
    else if (dtype == MC3B_F32) k_fma_peak<float><<<ctas, 256, 0, (cudaStream_t)stream>>>(iters, sink);
    else { mc3b_set_error("bad dtype %d", dtype); return MC3B_ERR_ARG; }
    MC3B_CHECK_LAUNCH("k_fma_peak");
    *flops = 2.0 * 8.0 * 256.0 * (double)ctas * (double)iters;
    return MC3B_OK;
}
