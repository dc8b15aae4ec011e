// Shared host-side helpers of libeaglegpu: error state, launch checks, device properties.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cuda_runtime.h>

#include "../../include/eagle_gpu.h"

namespace eg {

int set_error(int code, const char* fmt, ...);   // stores the message for eg_last_error(); returns code
int check_cuda(cudaError_t e, const char* what); // EG_OK or EG_ERR_CUDA (+message)
int check_launch(const char* kernel);            // cudaGetLastError() after a launch
int num_sms();                                   // SM count of the current device (148 on B200)
void pool_give_back();                           // release the library's cached device memory to the driver (retry after an OOM)
cudaError_t scratch_alloc(void** p, size_t bytes, cudaStream_t st);  // pool block usable on st (capi.cu)
void scratch_free(void* p, cudaStream_t st);                         // back to the pool after the work queued on st
// cudaMalloc with one retry after pool_give_back()
static inline cudaError_t malloc_retry(void** p, size_t bytes) {
    cudaError_t e = cudaMalloc(p, bytes);
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        pool_give_back();
        e = cudaMalloc(p, bytes);
    }
    return e;
}

#define EG_TRY(expr)                 \
    do {                             \
        int _rc = (expr);            \
        if (_rc != EG_OK) return _rc; \
    } while (0)
#define EG_CUDA(expr) EG_TRY(::eg::check_cuda((expr), #expr))

static inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }
// row pitch of a genotype store: room for one extra (zero) column, 128-byte multiple
static inline int64_t store_pitch(int64_t cols) { return round_up(cols + 1, 128); }

}  // namespace eg
