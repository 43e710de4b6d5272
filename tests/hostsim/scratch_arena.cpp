// TEST-ONLY host build of the scratch arena (schnorr-sig_b200/csrc/scratch.cuh) with g++ against the stand-in
// cuda_runtime.h in stub/, for tests/test_scratch_arena_hostsim.py.  cudaMalloc hands out addresses of a fake device
// address space (nothing is dereferenced) and fails once on request; every cudaMalloc, cudaFree and
// cudaStreamSynchronize is logged.  Scopes are
// kept on a stack so that the test can open and close them one call at a time.
#include <cstdint>
#include <memory>
#include <vector>

#include "cuda_runtime.h"
#include "../../schnorr-sig_b200/csrc/scratch.cuh"

#define API extern "C" __attribute__((visibility("default")))

enum { EV_MALLOC = 1, EV_FREE = 2, EV_SYNC = 3 };
struct event {
    uint64_t kind, ptr, bytes, device;
};
static std::vector<event> g_log;
static uint64_t g_next = 0x100000000ull;
static int g_fail_next = 0;
static int g_device = 0;   // the current device

cudaError_t cudaMalloc(void** p, size_t bytes) {
    if (g_fail_next) {
        g_fail_next = 0;
        return cudaErrorMemoryAllocation;
    }
    *p = (void*)(uintptr_t)g_next;
    g_log.push_back({EV_MALLOC, g_next, bytes, (uint64_t)g_device});
    g_next += (bytes + 4095) / 4096 * 4096 + 4096;   // a gap after every block
    return cudaSuccess;
}
cudaError_t cudaFree(void* p) {
    g_log.push_back({EV_FREE, (uint64_t)(uintptr_t)p, 0, (uint64_t)g_device});
    return cudaSuccess;
}
cudaError_t cudaStreamSynchronize(cudaStream_t) {
    g_log.push_back({EV_SYNC, 0, 0, (uint64_t)g_device});
    return cudaSuccess;
}
cudaError_t cudaGetLastError(void) { return cudaSuccess; }
cudaError_t cudaGetDevice(int* device) {
    *device = g_device;
    return cudaSuccess;
}
cudaError_t cudaSetDevice(int device) {
    g_device = device;
    return cudaSuccess;
}

static std::unique_ptr<scratch_arena> g_arena;
static std::vector<std::unique_ptr<scratch_scope>> g_scopes;

API void hs_reset() {
    g_scopes.clear();
    g_arena.reset();
    g_log.clear();
    g_device = 0;
    g_arena.reset(new scratch_arena());
}
API void hs_destroy() {
    g_scopes.clear();
    g_arena.reset();
}
API void hs_open() { g_scopes.emplace_back(new scratch_scope(*g_arena, nullptr)); }
API void hs_close() { g_scopes.pop_back(); }
// 0 and the region's address in *out, or the error of cudaMalloc
API int hs_take(uint64_t bytes, uint64_t* out) {
    void* p = nullptr;
    cudaError_t e = g_arena->take(bytes, &p);
    *out = (uint64_t)(uintptr_t)p;
    return e;
}
API void hs_fail_next_malloc() { g_fail_next = 1; }
API void hs_set_device(int device) { g_device = device; }
API uint64_t hs_log_size() { return g_log.size(); }
API void hs_log(uint64_t* out) {
    for (size_t i = 0; i < g_log.size(); i++) {
        out[4 * i] = g_log[i].kind;
        out[4 * i + 1] = g_log[i].ptr;
        out[4 * i + 2] = g_log[i].bytes;
        out[4 * i + 3] = g_log[i].device;
    }
}
