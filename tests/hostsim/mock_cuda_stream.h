// mock_cuda_stream.h -- TEST INFRASTRUCTURE ONLY.  The part of the CUDA runtime that the stream entry points of
// fourq_b200/csrc/capi.cu use beyond mock_cuda_runtime.h: stream-ordered pool allocation, capture status, the device of a stream
// and the current device.  capi.cu includes this header in every mock build (-DFQ_MOCK_CUDA).  The functions are declared weak:
// the mock builds that do not link mock_cuda_stream.cpp (build.sh, build_fixed_base.sh) still link, and capi.cu refuses stream
// calls there.  build_stream.sh links mock_cuda_stream.cpp and compiles capi.cu and the mock kernels with -DFQ_MOCK_COUNT, which
// routes their runtime calls through counting wrappers, so the tests can see every synchronisation, allocation and enqueue.
#pragma once
#include <cstdint>
#include "mock_cuda_runtime.h"

struct MockPool;
typedef MockPool* cudaMemPool_t;
enum cudaStreamCaptureStatus { cudaStreamCaptureStatusNone = 0, cudaStreamCaptureStatusActive = 1, cudaStreamCaptureStatusInvalidated = 2 };
enum cudaMemAllocationType { cudaMemAllocationTypeInvalid = 0, cudaMemAllocationTypePinned = 1 };
enum cudaMemLocationType { cudaMemLocationTypeInvalid = 0, cudaMemLocationTypeDevice = 1 };
enum cudaMemPoolAttr { cudaMemPoolAttrReleaseThreshold = 4 };
struct cudaMemLocation { cudaMemLocationType type; int id; };
struct cudaMemPoolProps { cudaMemAllocationType allocType; int handleTypes; cudaMemLocation location; };

#define FQ_MOCK_WEAK __attribute__((weak))
cudaError_t cudaGetDevice(int* dev) FQ_MOCK_WEAK;
cudaError_t cudaStreamGetDevice(cudaStream_t s, int* dev) FQ_MOCK_WEAK;
cudaError_t cudaStreamIsCapturing(cudaStream_t s, cudaStreamCaptureStatus* st) FQ_MOCK_WEAK;
cudaError_t cudaMemPoolCreate(cudaMemPool_t* pool, const cudaMemPoolProps* props) FQ_MOCK_WEAK;
cudaError_t cudaMemPoolDestroy(cudaMemPool_t pool) FQ_MOCK_WEAK;
cudaError_t cudaMemPoolSetAttribute(cudaMemPool_t pool, cudaMemPoolAttr attr, void* value) FQ_MOCK_WEAK;
cudaError_t cudaMemPoolTrimTo(cudaMemPool_t pool, size_t keep) FQ_MOCK_WEAK;
cudaError_t cudaMallocFromPoolAsync(void** p, size_t bytes, cudaMemPool_t pool, cudaStream_t s) FQ_MOCK_WEAK;
cudaError_t cudaFreeAsync(void* p, cudaStream_t s) FQ_MOCK_WEAK;

// counting wrappers of mock_cuda_stream.cpp around the runtime of mock_cuda_runtime.cpp
cudaError_t mock_count_cudaMalloc(void** p, size_t bytes);
cudaError_t mock_count_cudaFree(void* p);
cudaError_t mock_count_cudaHostAlloc(void** p, size_t bytes, unsigned flags);
cudaError_t mock_count_cudaFreeHost(void* p);
cudaError_t mock_count_cudaStreamSynchronize(cudaStream_t s);
cudaError_t mock_count_cudaDeviceSynchronize();
cudaError_t mock_count_cudaEventSynchronize(cudaEvent_t e);
cudaError_t mock_count_cudaMemcpy(void* dst, const void* src, size_t bytes, cudaMemcpyKind kind);
cudaError_t mock_count_cudaMemcpyAsync(void* dst, const void* src, size_t bytes, cudaMemcpyKind kind, cudaStream_t s);
cudaError_t mock_count_cudaMemsetAsync(void* p, int v, size_t bytes, cudaStream_t s);
cudaError_t mock_count_cudaEventRecord(cudaEvent_t e, cudaStream_t s);
cudaError_t mock_count_cudaSetDevice(int dev);
void mock_count_stream_enqueue(cudaStream_t s, std::function<void()> fn);

#ifdef FQ_MOCK_COUNT
#define cudaMalloc mock_count_cudaMalloc
#define cudaFree mock_count_cudaFree
#define cudaHostAlloc mock_count_cudaHostAlloc
#define cudaFreeHost mock_count_cudaFreeHost
#define cudaStreamSynchronize mock_count_cudaStreamSynchronize
#define cudaDeviceSynchronize mock_count_cudaDeviceSynchronize
#define cudaEventSynchronize mock_count_cudaEventSynchronize
#define cudaMemcpy mock_count_cudaMemcpy
#define cudaMemcpyAsync mock_count_cudaMemcpyAsync
#define cudaMemsetAsync mock_count_cudaMemsetAsync
#define cudaEventRecord mock_count_cudaEventRecord
#define cudaSetDevice mock_count_cudaSetDevice
#define mock_stream_enqueue mock_count_stream_enqueue
#endif
