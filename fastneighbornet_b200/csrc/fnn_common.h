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

// ---- alignment distances (csrc/fnn_dist.cu) ----
struct DistTimes {
    float upload_ms = 0, pack_ms = 0, pairs_ms = 0;
};
// the argument checks of fnn_distances; FNN_E_ARG with the message prefixed by `who`
int fnn_dist_check_args_(const char* who, const uint8_t* codes, int64_t n, int64_t sites, int32_t model, double undef);
// An alignment resident on the device: upload() copies the codes once and allocates the bit-planes (and, with resample, the
// site list); run() packs and computes the distances into dD, as often as needed.  sites (host, L entries, or NULL for the
// alignment as given) lists the columns of a resampled alignment.  An undefined pair fails the call, naming the pair with
// its counts in the packed alignment; `where` is inserted before "the <model> distance" ("" or e.g. "replicate 3: ").
struct DistJob {
    cudaStream_t stream = nullptr;
    int sms = 0;
    const uint8_t* codes = nullptr;   // host, kept for the error message's counts
    int64_t n = 0, L = 0;
    uint8_t* d_codes = nullptr;
    unsigned long long* d_planes = nullptr;
    unsigned long long* d_flags = nullptr;   // [0] = first undefined pair key, [1] = bad-code flag
    int32_t* d_sites = nullptr;
    DevScratch scratch;
    int upload(cudaStream_t stream, int sms, const uint8_t* codes, int64_t n, int64_t L, bool resample, DistTimes* tm);
    int run(const char* who, const char* where, int32_t model, double undef, const int32_t* sites, double* dD, int64_t ld,
            DistTimes* tm);
};

// ---- the network chain of fnn_network (csrc/fnn_csw.cu) ----
// One split-weight workspace for networks of n taxa, reused from one run to the next.  fnn_chain_run_ takes a loaded
// context: packed upper triangle of its matrix -> fnn_ctx_order -> split weights -> the splits with x > cutoff compacted
// on the device.  Only the count of kept splits is read back (*kept); fnn_chain_kept_idx_ points at their packed (i, j)
// indices on the device, increasing, valid until the next run; fnn_chain_copy_kept_ converts them for the host.
struct NetChain;
struct ChainTimes {
    double order_ms = 0, csw_ms = 0;   // CUDA-event ms: fnn_ctx_order; triangle packing + solve + compaction
    long long cg_iters = 0;            // CG iterations of the solve
};
int fnn_chain_create_(const fnn_opts* o, int64_t n, NetChain** out);
void fnn_chain_destroy_(NetChain* w);
int fnn_chain_run_(NetChain* w, fnn_ctx* ctx, double cutoff, int32_t* ordering_out, int64_t* kept, ChainTimes* tm);
const int* fnn_chain_kept_idx_(NetChain* w);
cudaStream_t fnn_chain_stream_(NetChain* w);
int fnn_chain_copy_kept_(NetChain* w, int64_t kept, int32_t* split_i, int32_t* split_j, double* weight);

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
