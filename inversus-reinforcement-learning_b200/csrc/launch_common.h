// launch_common.h -- host code every kernel file shares (defined in inversus_b200.cu, and the last
// four functions in host_expand.cpp).
#pragma once

#include <cuda_runtime.h>

#include "../../include/inversus_b200.h"

namespace inv_host {

// sets the calling thread's inv_last_error() text to "<who>: <msg>"; returns code
int set_error(int code, const char *who, const char *msg);
// INV_OK if the current device is an sm_100 part, else INV_ERR_NO_DEVICE (INV_ERR_CUDA if the query fails)
int require_sm100(const char *who);
// the current device's SM count, cached per device; 148 (a B200's) when it cannot be read
int sm_count();
// raises kernel's dynamic shared-memory limit on the current device to bytes; calls
// cudaFuncSetAttribute only when bytes exceeds the largest value already set there
cudaError_t allow_dynamic_smem(const void *kernel, size_t bytes);
// INV_OK, or INV_ERR_CUDA with "<who>: <cudaGetErrorString>" for what cudaGetLastError() returns
int launch_status(const char *who);

void expand_f32(const uint32_t *bits, float *dst, int64_t lo, int64_t hi, int nthreads);
int hardware_threads();
bool stage_action_ids(int8_t *dst, const int8_t *src, int64_t n);
bool check_action_ids(const int8_t *src, int64_t n);

} // namespace inv_host
