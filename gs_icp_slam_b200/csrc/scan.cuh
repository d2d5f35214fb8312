// scan.cuh — stream compaction offsets: out[i] = number of j < i with flag(j) != 0.
#pragma once
#include <cub/cub.cuh>
#include "host_common.h"

namespace gsicp {

// Exclusive sum of flag(0..n-1) into out (Out[n]); tmp holds cub's workspace.  Both buffers grow on demand.
template <typename Out, typename Flag>
int flag_exclusive_scan(int n, Flag flag, Scratch& out, Scratch& tmp, cudaStream_t stream) {
  if (int e = out.ensure((size_t)n * sizeof(Out))) return e;
  cub::CountingInputIterator<int> counting(0);
  cub::TransformInputIterator<Out, Flag, cub::CountingInputIterator<int>> flags(counting, flag);
  size_t bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, bytes, flags, out.as<Out>(), n, stream);
  if (int e = tmp.ensure(bytes)) return e;
  bytes = tmp.cap;
  GSICP_CUDA(cub::DeviceScan::ExclusiveSum(tmp.ptr, bytes, flags, out.as<Out>(), n, stream));
  return GSICP_OK;
}

}  // namespace gsicp
