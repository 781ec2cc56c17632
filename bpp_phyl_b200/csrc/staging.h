// Pageable host memory <-> device at PCIe speed, shared by the entry points that take large host buffers (site patterns,
// pairwise distances).
//
// A plain cudaMemcpy of pageable memory is bounded by ONE host thread copying through the driver's staging buffer (about 10 GB/s);
// an alignment (1 GB for 1M sites x 1024 taxa) going in and the tip codes coming back dominate such a call.  staged_copy moves the
// 4 MB chunks of a large pageable buffer through two pinned buffers per copy thread, each thread on its own stream, so that the
// host-side memcpy of one chunk overlaps the DMA of the others.  The pinned pool is allocated once per process.  Buffers the
// runtime already knows (pinned / registered / device / managed) and small ones take the direct copy.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <mutex>

namespace bppgpu {

constexpr size_t kStageChunk = (size_t)4 << 20;
constexpr int kCopyThreadsMax = 8;
struct StagePool {
  std::mutex mu;
  int device = -1, threads = 0;
  void* pinned[kCopyThreadsMax][2] = {};
  cudaStream_t stream[kCopyThreadsMax] = {};
  cudaEvent_t done[kCopyThreadsMax][2] = {};
  cudaError_t ensure(int dev);
};

// Blocking copy of `bytes` between host (any kind) or device memory and device memory of `device`; h2d says which side is the
// host candidate.  The caller has synchronised the work that produced `src` (device to host) / launches consumers afterwards.
cudaError_t staged_copy(void* dst, const void* src, size_t bytes, bool h2d, int device);

}  // namespace bppgpu
