// fnn_common.h — error plumbing shared by the translation units of libfastnn.so.
#pragma once
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdio>
#include "fastnn.h"

namespace fnn {
void set_error(const char* fmt, ...);
const char* last_error();
}  // namespace fnn

// frees a handful of cudaMalloc'ed scratch buffers on every exit path of a C-ABI entry point
struct DevScratch {
    void* ptr[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    int count = 0;
    cudaError_t alloc(void** out, size_t bytes) {
        cudaError_t e = cudaMalloc(out, bytes);
        if (e == cudaSuccess && count < 8) ptr[count++] = *out;
        return e;
    }
    ~DevScratch() { for (int i = 0; i < count; ++i) cudaFree(ptr[i]); }
};

// a cudaEvent_t that is destroyed on every exit path
struct DevEvent {
    cudaEvent_t e = nullptr;
    cudaError_t create() { return cudaEventCreate(&e); }
    operator cudaEvent_t() const { return e; }
    ~DevEvent() { if (e) cudaEventDestroy(e); }
};

// internal accessors across translation units (not part of the ABI)
int64_t fnn_ctx_n_(fnn_ctx* c);
void fnn_ctx_mark_loaded_(fnn_ctx* c);
void fnn_ctx_mark_unloaded_(fnn_ctx* c);
fnn_stats* fnn_ctx_stats_(fnn_ctx* c);
int fnn_ctx_device_(fnn_ctx* c);
int fnn_ctx_sms_(fnn_ctx* c);
cudaStream_t fnn_ctx_stream_(fnn_ctx* c);

// CUDA errors are fatal for the call (no CPU fallback): record and return FNN_E_CUDA.
#define FNN_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t err_ = (call);                                                              \
        if (err_ != cudaSuccess) {                                                              \
            fnn::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(err_)); \
            cudaGetLastError();                                                                 \
            return FNN_E_CUDA;                                                                  \
        }                                                                                       \
    } while (0)
