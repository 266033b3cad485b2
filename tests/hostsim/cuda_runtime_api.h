/*
 * tests/hostsim/cuda_runtime_api.h — TEST SCAFFOLDING ONLY: a malloc-backed stand-in for the
 * handful of CUDA runtime calls smx_host.c makes, so the host shim compiles with gcc for the
 * CPU-side host-logic tests (see hostsim.h).  "Device" allocations are filled with 0xCD so that
 * a missing cudaMemset shows up as a test failure.
 */
#pragma once
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif
typedef int cudaError_t;
typedef void* cudaStream_t;
typedef void* cudaEvent_t;
enum { cudaSuccess = 0, cudaErrorMemoryAllocation = 2, cudaErrorPeerAccessAlreadyEnabled = 704 };
enum { cudaMemcpyHostToDevice = 1, cudaMemcpyDeviceToHost = 2, cudaMemcpyDeviceToDevice = 3, cudaMemcpyDefault = 4 };
enum { cudaMemoryTypeUnregistered = 0, cudaMemoryTypeHost = 1, cudaMemoryTypeDevice = 2, cudaMemoryTypeManaged = 3 };
enum { cudaStreamNonBlocking = 1, cudaEventDefault = 0, cudaEventDisableTiming = 2, cudaHostAllocDefault = 0 };
enum { cudaDevAttrMultiProcessorCount = 16 };
struct cudaPointerAttributes { int type; int device; void* devicePointer; void* hostPointer; };
cudaError_t cudaGetDeviceCount(int* n);
cudaError_t cudaSetDevice(int d);
cudaError_t cudaGetDevice(int* d);
cudaError_t cudaDeviceGetAttribute(int* v, int attr, int dev);
cudaError_t cudaMalloc(void** p, size_t n);
cudaError_t cudaFree(void* p);
cudaError_t cudaHostAlloc(void** p, size_t n, unsigned flags);
cudaError_t cudaFreeHost(void* p);
cudaError_t cudaMemset(void* p, int v, size_t n);
cudaError_t cudaMemsetAsync(void* p, int v, size_t n, cudaStream_t s);
cudaError_t cudaMemcpy(void* d, const void* s, size_t n, int kind);
cudaError_t cudaMemcpyAsync(void* d, const void* s, size_t n, int kind, cudaStream_t st);
cudaError_t cudaStreamCreateWithFlags(cudaStream_t* s, unsigned flags);
cudaError_t cudaStreamDestroy(cudaStream_t s);
cudaError_t cudaStreamSynchronize(cudaStream_t s);
cudaError_t cudaStreamWaitEvent(cudaStream_t s, cudaEvent_t e, unsigned flags);
cudaError_t cudaEventCreateWithFlags(cudaEvent_t* e, unsigned flags);
cudaError_t cudaEventCreate(cudaEvent_t* e);
cudaError_t cudaEventDestroy(cudaEvent_t e);
cudaError_t cudaEventRecord(cudaEvent_t e, cudaStream_t s);
cudaError_t cudaEventSynchronize(cudaEvent_t e);
cudaError_t cudaEventElapsedTime(float* ms, cudaEvent_t a, cudaEvent_t b);
typedef struct { char reserved[64]; } cudaIpcMemHandle_t;
enum { cudaIpcMemLazyEnablePeerAccess = 1 };
cudaError_t cudaIpcGetMemHandle(cudaIpcMemHandle_t* h, void* p);
cudaError_t cudaIpcOpenMemHandle(void** p, cudaIpcMemHandle_t h, unsigned flags);
cudaError_t cudaIpcCloseMemHandle(void* p);
cudaError_t cudaDeviceEnablePeerAccess(int peer, unsigned flags);
cudaError_t cudaPointerGetAttributes(struct cudaPointerAttributes* a, const void* p);
cudaError_t cudaMemGetInfo(size_t* free_b, size_t* total_b);
cudaError_t cudaGetLastError(void);
cudaError_t cudaDeviceSynchronize(void);
const char* cudaGetErrorString(cudaError_t e);
#ifdef __cplusplus
}
#endif
