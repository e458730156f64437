// internal.h -- what the library's .cu files share beyond include/msda_b200.h. Not installed, not part of the ABI: the
// symbols below are defined once (msda_b200.cu, msda_bwd_det.cu) and only the library's own files call them.
// Included at file scope, after msda_b200.h and cuda_runtime.h.
#pragma once

#include <cstdio>

struct DetLayout;  // msda_bwd_det.cuh

extern "C" {
// msda_b200.cu: sets msda_b200_last_error() to `msg` and returns `code`
int msda_b200_internal_fail(int code, const char* msg);
// msda_b200.cu: the descriptor checks of forward / backward
int msda_b200_internal_validate(const msda_b200_desc* desc);
// msda_b200.cu: the geometry limit of msda_b200_backward (shared memory per block) for a validated descriptor
int msda_b200_internal_check_backward(const msda_b200_desc* desc);
// msda_b200.cu: one more launch for msda_b200_launch_count()
void msda_b200_internal_count_launch(void);

// msda_bwd_det.cu (CUB stays in that file). The caller has checked records <= INT_MAX and keys <= 2^32 - 1.
// Bytes of the sort's scratch, as CUB reports them for the current device (0 without records):
int msda_b200_internal_det_sort_bytes(const DetLayout* lay, size_t* bytes);
// The sort of the records in the first buffers of `workspace` (at least lay->sort_off + the bytes above); *keys and
// *vals receive the buffers that hold the sorted records. Counts as one launch.
int msda_b200_internal_det_sort(const DetLayout* lay, void* workspace, const unsigned** keys,
                                const unsigned long long** vals, cudaStream_t stream);
// The deterministic MSDA backward's workspace for a validated descriptor, and its grad_value from the records that
// msda_bwd_kernel<ACC = 2> wrote.
int msda_b200_internal_det_workspace_bytes(const msda_b200_desc* desc, size_t* bytes);
int msda_b200_internal_det_grad_value(const msda_b200_desc* desc, const void* grad_out, void* grad_value,
                                      void* workspace, cudaStream_t stream);
}

// A failed CUDA call: last_error = "<what>: <CUDA's message>", returns MSDA_B200_ERR_CUDA. The failure is also the
// thread's last CUDA error; it is cleared so that the next launch check does not report it again.
inline int cuda_error(const char* what, cudaError_t e) {
  (void)cudaGetLastError();
  char msg[256];
  snprintf(msg, sizeof(msg), "%s: %s", what, cudaGetErrorString(e));
  return msda_b200_internal_fail(MSDA_B200_ERR_CUDA, msg);
}

// The end of every kernel launch site: counts the launch and checks it.
inline int launched(const char* what) {
  msda_b200_internal_count_launch();
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? MSDA_B200_OK : cuda_error(what, e);
}
