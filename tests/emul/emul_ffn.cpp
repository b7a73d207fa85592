// Host shim over the tensor-core FFN's weight packing (TEST INFRASTRUCTURE).
// Compiles the host part of vad_b200/csrc/ffn_tc.cuh with g++ (cuda_fp16.h / cuda_runtime.h from the CUDA
// toolkit's include directory) so that the CPU suite can read the fp16 scales, the folded epilogue constants and
// both operand blobs exactly as a handle builds them.  The product never links this file.
#include <cstring>

#include "../../vad_b200/csrc/ffn_tc.cuh"

using namespace vadb;

extern "C" {

int emul_ffn_blob_bytes(int fp16) { return fp16 ? kTc16BlobBytes : kTcBlobBytes; }

// weights: W1,b1,W2,b2,W3,b3,W4,b4 concatenated (5219 floats).
// scales: pre[4], post[4], postp[4];  cbias: c1[64], c2[32], c3[16];  blob16: kTc16BlobBytes;  blob32: kTcBlobBytes.
// Returns tc16_pack_weights' result (1: the fp16 scales are in range).
int emul_ffn_pack(const float* weights, float* scales, float* cbias, unsigned char* blob16, unsigned char* blob32) {
  static FfnParams p;
  static FfnBias fb;
  std::memset(&p, 0, sizeof(p));
  std::memset(&fb, 0, sizeof(fb));
  const size_t n = kNFeat * kH1 + kH1 + kH1 * kH2 + kH2 + kH2 * kH3 + kH3 + kH3 * kNCls + kNCls;
  std::memcpy(p.W1, weights, n * sizeof(float));
  std::memset(blob16, 0, kTc16BlobBytes);
  const bool ok = tc16_pack_weights(p, blob16, fb);
  tc_pack_weights(p, blob32);
  std::memcpy(scales, fb.pre, sizeof(fb.pre));
  std::memcpy(scales + 4, fb.post, sizeof(fb.post));
  std::memcpy(scales + 8, fb.postp, sizeof(fb.postp));
  std::memcpy(cbias, fb.c1, sizeof(fb.c1));
  std::memcpy(cbias + kH1, fb.c2, sizeof(fb.c2));
  std::memcpy(cbias + kH1 + kH2, fb.c3, sizeof(fb.c3));
  return ok ? 1 : 0;
}

}  // extern "C"
