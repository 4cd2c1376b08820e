// Error reporting and device selection shared by the host code of every C ABI unit (taco_env.cu, taco_actor.cu,
// taco_critic.cu, taco_gae.cu, taco_ppo.cu).
#pragma once
#include <string>

#include <cuda_runtime.h>

#include "../../include/taco_b200.h"

namespace taco {

// records msg as this thread's error (taco_last_error) and returns code; defined in taco_env.cu, one error slot for the library
int fail(int code, const std::string& msg);

// makes `dev` the current device for the guard's lifetime
struct DevGuard {
    int prev = -1;
    explicit DevGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

}  // namespace taco

// returns TACO_E_CUDA from the enclosing function when a CUDA runtime call fails; the message names the call and the error
#define TACO_CUDA(expr)                                                                               \
    do {                                                                                              \
        cudaError_t _e = (expr);                                                                      \
        if (_e != cudaSuccess)                                                                        \
            return ::taco::fail(TACO_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));    \
    } while (0)
