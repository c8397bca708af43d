// Error reporting of the C-ABI entry points (host).  No CUDA headers: gemm_plan.cuh uses it and the host compiler builds that too.
#pragma once

namespace dsb {

void set_error(const char* fmt, ...);  // the message dsb_last_error() returns (api.cu)

}  // namespace dsb

#define DSB_REQUIRE(cond, ...)                                                                  \
  do {                                                                                          \
    if (!(cond)) {                                                                              \
      dsb::set_error(__VA_ARGS__);                                                              \
      return 2;                                                                                 \
    }                                                                                           \
  } while (0)
