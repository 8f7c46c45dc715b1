// Library-level entry points of the C ABI: error channel, version, device check, launch counter.
#include "../../include/mocha_b200.h"
#include "common.cuh"
#include "gemm_tc.cuh"

#include <atomic>

namespace mocha {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
const char* last_error() { return g_err; }
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

}  // namespace mocha

extern "C" const char* mocha_last_error(void) { return mocha::last_error(); }
extern "C" int mocha_version(void) { return 100; }
extern "C" long long mocha_launch_count(void) { return mocha::g_launches.load(); }
extern "C" void mocha_reset_launch_count(void) { mocha::g_launches.store(0); }

extern "C" int mocha_check_device(void) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess)
    return mocha::set_error(MOCHA_ERR_CUDA, "no CUDA device: %s", cudaGetErrorString(e));
  int major = 0, minor = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
  if (major != 10)
    return mocha::set_error(MOCHA_ERR_ARCH, "device is sm_%d%d; this library is built for sm_100a only", major, minor);
  return MOCHA_OK;
}

// Register the bf16 mirror of an fp32 weight blob so MOCHA_BF16 layers can find W16 for a W pointer.
extern "C" int mocha_register_bf16_blob(const float* blob32, const void* blob16, size_t elems) {
  // blob16 == NULL unregisters the range (call before freeing the blob)
  if (!blob32 || elems == 0)
    return mocha::set_error(MOCHA_ERR_ARG, "mocha_register_bf16_blob: bad argument");
  mocha::tc_register_blob(blob32, blob16, elems);
  return MOCHA_OK;
}

// Workspace size queries (mocha_*_workspace_bytes) answer for this precision mode from now on (process-wide; the
// default covers MOCHA_FP32 and MOCHA_BF16; MOCHA_TF32X3 adds room for its split operands).
extern "C" int mocha_workspace_precision(int precision) {
  if (precision != MOCHA_FP32 && precision != MOCHA_BF16 && precision != MOCHA_TF32X3)
    return mocha::set_error(MOCHA_ERR_ARG, "mocha_workspace_precision: unknown precision %d", precision);
  mocha::tc_set_workspace_precision(precision);
  return MOCHA_OK;
}

// sizeof() of every ABI struct, so a binding can verify its mirror definitions at load time.
// order: dims, enc_layer, dec_layer, generator_weights, cvae_enc_layer, cvae_dec_layer, cvae_weights,
//        clip_state, post_params, frame_out
extern "C" int mocha_struct_sizes(size_t* out, int n) {
  const size_t s[10] = {sizeof(mocha_dims), sizeof(mocha_enc_layer), sizeof(mocha_dec_layer),
                        sizeof(mocha_generator_weights), sizeof(mocha_cvae_enc_layer), sizeof(mocha_cvae_dec_layer),
                        sizeof(mocha_cvae_weights), sizeof(mocha_clip_state), sizeof(mocha_post_params),
                        sizeof(mocha_frame_out)};
  if (!out || n < 10) return mocha::set_error(MOCHA_ERR_ARG, "mocha_struct_sizes: need room for 10 entries");
  for (int i = 0; i < 10; ++i) out[i] = s[i];
  return MOCHA_OK;
}
