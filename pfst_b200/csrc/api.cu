// Library-level entry points: version, error strings, device check.
#include <stdio.h>
#include <string.h>

#include "common.cuh"

namespace pfst {

static thread_local char g_last_error[512] = "";

void set_last_cuda_error(cudaError_t e, const char* where) {
  snprintf(g_last_error, sizeof(g_last_error), "%s: %s (%s)", where,
           cudaGetErrorName(e), cudaGetErrorString(e));
}

}  // namespace pfst

extern "C" {

const char* pfst_version(void) { return "pfst_sm100 0.4.0 (sm_100a)"; }

const char* pfst_error_string(int code) {
  switch (code) {
    case PFST_OK: return "ok";
    case PFST_ERR_INVALID_ARG: return "invalid argument";
    case PFST_ERR_UNSUPPORTED: return "unsupported configuration";
    case PFST_ERR_CUDA: return "CUDA error (see pfst_last_cuda_error)";
    case PFST_ERR_NO_DEVICE: return "no sm_100 (B200) device is current";
    default: return "unknown error code";
  }
}

const char* pfst_last_cuda_error(void) { return pfst::g_last_error; }

int pfst_copy_async(void* dst, const void* src, int64_t bytes, void* stream) {
  if (!dst || !src || bytes < 0) return PFST_ERR_INVALID_ARG;
  if (bytes == 0) return PFST_OK;
  PFST_CUDA_TRY(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDefault, static_cast<cudaStream_t>(stream)),
                "pfst_copy_async");
  return PFST_OK;
}

int pfst_classmix_draw(const uint64_t* words, int64_t n_words, const int64_t* classes, int32_t n_classes,
                        int32_t batch, uint32_t* masks, int32_t* state, int64_t* words_missing) {
  if (!classes || !masks || !state || !words_missing || n_classes < 0 || n_classes > 256 || batch < 0 ||
      n_words < 0 || (n_words > 0 && !words))
    return PFST_ERR_INVALID_ARG;
  const int n = n_classes, k = (n + n % 2) / 2;
  int b = state[0], i = state[1];
  int* perm = state + 2;
  if (b < 0 || b > batch || i < 0 || i >= (n > 0 ? n : 1)) return PFST_ERR_INVALID_ARG;
  for (int c = 0; c < n; ++c)
    if (classes[c] < 0 || classes[c] > 255) return PFST_ERR_INVALID_ARG;
  int64_t pos = 0;
  *words_missing = 0;
  for (; b < batch; ++b) {
    if (i == 0) {                               // a new image: identity permutation, first swap index n-1
      for (int c = 0; c < n; ++c) perm[c] = c;
      i = n - 1;
    }
    // numpy legacy RandomState.shuffle: for i = n-1 .. 1: j = random_interval(i) (masked rejection on
    // successive 32-bit outputs), swap(perm[i], perm[j])
    for (; i >= 1; --i) {
      uint32_t mask = (uint32_t)i;
      mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16;
      uint32_t v;
      do {
        if (pos >= n_words) {
          // out of words: at least one more for this swap and one for each swap still to come
          state[0] = b; state[1] = i;
          *words_missing = (int64_t)i + (int64_t)(batch - 1 - b) * (n - 1);
          return PFST_OK;
        }
        v = (uint32_t)words[pos++] & mask;
      } while (v > (uint32_t)i);
      const int t = perm[i]; perm[i] = perm[v]; perm[v] = t;
    }
    uint32_t* m = masks + (size_t)b * 8;
    for (int w = 0; w < 8; ++w) m[w] = 0;
    for (int c = 0; c < k; ++c) {
      const int cl = (int)classes[perm[c]];
      m[cl >> 5] |= 1u << (cl & 31);
    }
    i = 0;
  }
  state[0] = batch; state[1] = 0;
  return pos == n_words ? PFST_OK : PFST_ERR_INVALID_ARG;     // more words than the shuffles consume
}

int pfst_device_check(void) {
  int dev = -1;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    pfst::set_last_cuda_error(e, "pfst_device_check/cudaGetDevice");
    cudaGetLastError();
    return PFST_ERR_NO_DEVICE;
  }
  int major = 0;
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess) {
    pfst::set_last_cuda_error(e, "pfst_device_check/cudaDeviceGetAttribute");
    cudaGetLastError();
    return PFST_ERR_NO_DEVICE;
  }
  return major == 10 ? PFST_OK : PFST_ERR_NO_DEVICE;
}

}  // extern "C"
