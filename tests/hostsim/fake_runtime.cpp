// tests/hostsim/fake_runtime.cpp — TEST SCAFFOLDING ONLY (see hostsim.h).
#include "cuda_runtime_api.h"
#include "hostsim.h"
#include <map>
#include <mutex>

thread_local uint3_sim blockIdx, threadIdx;
thread_local dim3 gridDim, blockDim;

static std::map<uintptr_t, size_t> g_dev;   // "device" allocations
static std::mutex g_mu;
static size_t g_dev_bytes = 0;

extern "C" {
cudaError_t cudaGetDeviceCount(int* n) { *n = 1; return 0; }
cudaError_t cudaSetDevice(int d) { return d == 0 ? 0 : 1; }
cudaError_t cudaGetDevice(int* d) { *d = 0; return 0; }
cudaError_t cudaDeviceGetAttribute(int* v, int, int) { *v = 2; return 0; }
cudaError_t cudaMalloc(void** p, size_t n) {
  void* q = nullptr;
  if (posix_memalign(&q, 256, n ? n : 256)) return cudaErrorMemoryAllocation;
  memset(q, 0xCD, n);
  std::lock_guard<std::mutex> lk(g_mu);
  g_dev[(uintptr_t)q] = n;
  g_dev_bytes += n;
  *p = q;
  return 0;
}
cudaError_t cudaFree(void* p) {
  if (!p) return 0;
  std::lock_guard<std::mutex> lk(g_mu);
  auto it = g_dev.find((uintptr_t)p);
  if (it == g_dev.end()) return 1;
  g_dev_bytes -= it->second;
  g_dev.erase(it);
  free(p);
  return 0;
}
cudaError_t cudaHostAlloc(void** p, size_t n, unsigned) { *p = malloc(n ? n : 1); return *p ? 0 : 2; }
cudaError_t cudaFreeHost(void* p) { free(p); return 0; }
cudaError_t cudaMemset(void* p, int v, size_t n) { memset(p, v, n); return 0; }
cudaError_t cudaMemsetAsync(void* p, int v, size_t n, cudaStream_t) { memset(p, v, n); return 0; }
cudaError_t cudaMemcpy(void* d, const void* s, size_t n, int) { memmove(d, s, n); return 0; }
cudaError_t cudaMemcpyAsync(void* d, const void* s, size_t n, int, cudaStream_t) { memmove(d, s, n); return 0; }
cudaError_t cudaStreamCreateWithFlags(cudaStream_t* s, unsigned) { *s = (void*)1; return 0; }
cudaError_t cudaStreamDestroy(cudaStream_t) { return 0; }
cudaError_t cudaStreamSynchronize(cudaStream_t) { return 0; }
cudaError_t cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned) { return 0; }
cudaError_t cudaEventCreateWithFlags(cudaEvent_t* e, unsigned) { *e = (void*)1; return 0; }
cudaError_t cudaEventCreate(cudaEvent_t* e) { *e = (void*)1; return 0; }
cudaError_t cudaEventDestroy(cudaEvent_t) { return 0; }
cudaError_t cudaEventRecord(cudaEvent_t, cudaStream_t) { return 0; }
cudaError_t cudaEventSynchronize(cudaEvent_t) { return 0; }
cudaError_t cudaEventElapsedTime(float* ms, cudaEvent_t, cudaEvent_t) { *ms = 1.0f; return 0; }
cudaError_t cudaPointerGetAttributes(struct cudaPointerAttributes* a, const void* p) {
  std::lock_guard<std::mutex> lk(g_mu);
  a->type = cudaMemoryTypeUnregistered;
  a->device = 0;
  auto it = g_dev.upper_bound((uintptr_t)p);
  if (it != g_dev.begin()) {
    --it;
    if ((uintptr_t)p < it->first + it->second) a->type = cudaMemoryTypeDevice;
  }
  return 0;
}
// "IPC" inside one process: the handle carries the raw pointer (ranks are threads in the CPU tests)
cudaError_t cudaIpcGetMemHandle(cudaIpcMemHandle_t* h, void* p) { memset(h, 0, sizeof *h); memcpy(h->reserved, &p, sizeof p); return 0; }
cudaError_t cudaIpcOpenMemHandle(void** p, cudaIpcMemHandle_t h, unsigned) { memcpy(p, h.reserved, sizeof *p); return *p ? 0 : 1; }
cudaError_t cudaIpcCloseMemHandle(void*) { return 0; }
cudaError_t cudaDeviceEnablePeerAccess(int, unsigned) { return 0; }
cudaError_t cudaMemGetInfo(size_t* f, size_t* t) { *t = (size_t)8 << 30; *f = *t - g_dev_bytes; return 0; }
cudaError_t cudaGetLastError(void) { return 0; }
cudaError_t cudaDeviceSynchronize(void) { return 0; }
const char* cudaGetErrorString(cudaError_t) { return "hostsim error"; }
}
