// ABI bookkeeping: version, error strings, launch counter; the shared-memory opt-in table.
#include <map>
#include <mutex>
#include <utility>
#include "common.cuh"

namespace irs {

long long g_launches = 0;

cudaError_t opt_in_smem(const void* kernel, size_t bytes) {
  static std::mutex mu;
  static std::map<std::pair<const void*, int>, size_t> granted;
  int dev;
  const cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lock(mu);
  size_t& have = granted[{kernel, dev}];
  if (bytes <= have) return cudaSuccess;
  const cudaError_t r = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (r == cudaSuccess) have = bytes;
  return r;
}

}  // namespace irs

extern "C" int irs_abi_version(void) { return IRS_B200_ABI_VERSION; }

extern "C" const char* irs_error_string(int code) {
  if (code == 0) return "ok";
  if (code > 0) return cudaGetErrorString((cudaError_t)code);
  switch (code) {
    case IRS_E_BADARG: return "irs_b200: bad argument (null pointer or non-positive size)";
    case IRS_E_SHAPE: return "irs_b200: shape/alignment outside what the kernel supports";
    case IRS_E_WORKSPACE: return "irs_b200: workspace too small (use the *_workspace_bytes query)";
    case IRS_E_OVERFLOW: return "irs_b200: candidate buffer overflow";
    default: return "irs_b200: unknown error";
  }
}

extern "C" long long irs_launch_count(void) { return irs::g_launches; }
extern "C" void irs_launch_count_reset(void) { irs::g_launches = 0; }
