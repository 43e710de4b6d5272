// TEST-ONLY stand-in for the CUDA runtime header, with just what schnorr-sig_b200/csrc/scratch.cuh uses, so that
// tests/hostsim/scratch_arena.cpp can build the arena with g++ and record every allocator and synchronisation call.
#pragma once
#include <cstddef>

typedef int cudaError_t;
static constexpr cudaError_t cudaSuccess = 0;
static constexpr cudaError_t cudaErrorMemoryAllocation = 2;
typedef struct CUstream_st* cudaStream_t;

cudaError_t cudaMalloc(void** p, size_t bytes);
cudaError_t cudaFree(void* p);
cudaError_t cudaStreamSynchronize(cudaStream_t stream);
cudaError_t cudaGetLastError(void);
cudaError_t cudaGetDevice(int* device);
cudaError_t cudaSetDevice(int device);
