// vad_resample.cu -- the launchers of vad_resample.cuh's kernels, in a translation unit of their own so that the
// fused kernels of vadb200.cu compile exactly as they do without them.  vadb200.cu validates every argument and
// counts the launches; these functions only enqueue.
#define VADB_RESAMPLE_KERNELS
#include "vad_resample.cuh"

#include <algorithm>
#include <cstring>

namespace vadb {

cudaError_t resample_allow_smem(int bytes) {
  cudaError_t e = cudaFuncSetAttribute(resample_kernel<int16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(resample_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  return e;
}

void enqueue_decode_pcm(int fmt, dim3 grid, cudaStream_t st, const uint8_t* raw, int channels, int be,
                        const long long* src, const long long* dst_off, const long long* len, float* dst) {
  switch (fmt) {
    case kPcmS16: decode_pcm_kernel<kPcmS16><<<grid, 256, 0, st>>>(raw, channels, be, src, dst_off, len, dst); break;
    case kPcmU8: decode_pcm_kernel<kPcmU8><<<grid, 256, 0, st>>>(raw, channels, be, src, dst_off, len, dst); break;
    case kPcmS24: decode_pcm_kernel<kPcmS24><<<grid, 256, 0, st>>>(raw, channels, be, src, dst_off, len, dst); break;
    case kPcmS32: decode_pcm_kernel<kPcmS32><<<grid, 256, 0, st>>>(raw, channels, be, src, dst_off, len, dst); break;
    case kPcmF32: decode_pcm_kernel<kPcmF32><<<grid, 256, 0, st>>>(raw, channels, be, src, dst_off, len, dst); break;
    default: decode_pcm_kernel<kPcmF64><<<grid, 256, 0, st>>>(raw, channels, be, src, dst_off, len, dst); break;
  }
}

void enqueue_resample(bool s16, const ResampleParams& a, const ResampleUtt* list, long long n, long long tiles,
                      size_t smem, cudaStream_t st) {
  ResampleFill f;
  for (long long u0 = 0; u0 < n; u0 += kResampleFill) {
    const int cnt = static_cast<int>(std::min<long long>(kResampleFill, n - u0));
    std::memcpy(f.u, list + u0, cnt * sizeof(ResampleUtt));
    resample_fill_kernel<<<1, 256, 0, st>>>(const_cast<ResampleUtt*>(a.utts) + u0, cnt, f);
  }
  if (s16) resample_kernel<int16_t><<<static_cast<unsigned>(tiles), kResampleThreads, smem, st>>>(a);
  else resample_kernel<float><<<static_cast<unsigned>(tiles), kResampleThreads, smem, st>>>(a);
}

}  // namespace vadb
