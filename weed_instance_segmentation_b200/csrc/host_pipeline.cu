// Host-buffer pipeline over the C ABI (include/msda_b200.h, "Host-buffer pipeline").
//
// The op's tensors live in host memory; a step cuts the batch into chunks of whole images and moves every chunk
// through H2D copy -> msda_b200_forward (+ msda_b200_backward) -> D2H copy on three streams.  A ring of staging
// slots decouples the stages: while chunk i computes, chunk i+1 is on its way in and chunk i-1 on its way out, so
// the step costs about max(H2D, D2H) of its bytes instead of H2D + kernels + D2H.  Ordering is carried only by CUDA
// events (no host waits inside step), which also lets consecutive steps overlap.
//
// kCopyLanes: streams per copy direction (chunks alternate between them).  Measured on B200 / PCIe Gen5 at BASELINE
// config 2 (tools/host_pipeline_sweep.py): raw duplex 6.8-7.0 ms for the step's 2 x 341 MB, the pipeline 7.4-7.9 ms
// with one lane and 8.0-8.2 ms with two -- the gap to the raw figure is not per-copy latency, so one lane it is.
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdlib>
#include <new>
#include <vector>

#include "msda_b200.h"
#include "internal.h"

namespace {

constexpr int kCopyLanes = 1;

struct Slot {
  char* in = nullptr;    // value | loc | attn | grad_out for one chunk
  char* out = nullptr;   // out | grad_value | grad_loc | grad_attn
  char* ws = nullptr;    // backward workspace
  cudaEvent_t in_done = nullptr, comp_done = nullptr, out_done = nullptr;
};

inline size_t align256(size_t n) { return (n + 255) & ~size_t(255); }

inline size_t dtype_size(int code) { return code == MSDA_B200_BF16 ? 2 : 4; }

}  // namespace

struct msda_b200_host_pipeline {
  msda_b200_desc desc{};  // whole batch; pointers into the two vectors below
  std::vector<int32_t> shapes;
  std::vector<int64_t> starts;
  int32_t chunk = 1, nslots = 0, with_backward = 1, device = 0;
  const int32_t* query_order = nullptr;
  // per-image byte counts
  size_t value_b = 0, loc_b = 0, attn_b = 0, out_b = 0;
  // offsets inside a slot's `in` / `out` block (sized for a full chunk)
  size_t in_off[4] = {0, 0, 0, 0}, out_off[4] = {0, 0, 0, 0};
  size_t ws_bytes = 0;
  std::vector<Slot> slots;
  cudaStream_t s_h2d[kCopyLanes] = {}, s_comp = nullptr, s_d2h[kCopyLanes] = {};
  cudaEvent_t fork = nullptr, tail[kCopyLanes] = {};
  uint64_t next = 0;  // chunks enqueued so far (slot = next % nslots)
  bool poisoned = false;  // a step failed half way: its batch is incomplete, further steps are refused
};

namespace {

#define HP_CUDA(expr)                                              \
  do {                                                             \
    cudaError_t e_ = (expr);                                       \
    if (e_ != cudaSuccess) return cuda_error("host_pipeline", e_); \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  bool changed = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) changed = cudaSetDevice(dev) == cudaSuccess;
  }
  ~DeviceGuard() {
    if (changed) cudaSetDevice(prev);
  }
};

void release(msda_b200_host_pipeline* p) {
  for (Slot& s : p->slots) {
    if (s.in) cudaFree(s.in);
    if (s.out) cudaFree(s.out);
    if (s.ws) cudaFree(s.ws);
    if (s.in_done) cudaEventDestroy(s.in_done);
    if (s.comp_done) cudaEventDestroy(s.comp_done);
    if (s.out_done) cudaEventDestroy(s.out_done);
  }
  if (p->fork) cudaEventDestroy(p->fork);
  for (int i = 0; i < kCopyLanes; ++i) {
    if (p->tail[i]) cudaEventDestroy(p->tail[i]);
    if (p->s_h2d[i]) cudaStreamDestroy(p->s_h2d[i]);
    if (p->s_d2h[i]) cudaStreamDestroy(p->s_d2h[i]);
  }
  if (p->s_comp) cudaStreamDestroy(p->s_comp);
  delete p;
}

}  // namespace

extern "C" int msda_b200_host_pipeline_create(const msda_b200_desc* desc, int32_t chunk_images, int32_t slots,
                                              int32_t with_backward, const int32_t* query_order,
                                              msda_b200_host_pipeline** pipeline) {
  if (!desc || !pipeline) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "host_pipeline_create: NULL argument");
  *pipeline = nullptr;
  if (chunk_images < 1 || slots < 2 || slots > 16)
    return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "host_pipeline_create: chunk_images >= 1 and 2 <= slots <= 16");
  if (desc->B < 1 || desc->L < 1 || !desc->spatial_shapes_hw || !desc->level_start_index)
    return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "host_pipeline_create: incomplete descriptor");
  // The library's own descriptor checks FIRST (L <= MSDA_B200_MAX_LEVELS, positive sizes, level table inside S):
  // only a validated descriptor says how many entries of the caller's arrays may be read.
  if (int rc = msda_b200_internal_validate(desc)) return rc;  // last_error set by validate
  if (with_backward)
    if (int rc = msda_b200_internal_check_backward(desc)) return rc;
  msda_b200_host_pipeline* p = new (std::nothrow) msda_b200_host_pipeline();
  if (!p) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "host_pipeline_create: out of host memory");
  p->desc = *desc;
  p->desc.flags &= ~MSDA_B200_FLAG_PROFILE;  // per-launch events would serialise the streams
  p->shapes.assign(desc->spatial_shapes_hw, desc->spatial_shapes_hw + 2 * desc->L);
  p->starts.assign(desc->level_start_index, desc->level_start_index + desc->L);
  p->desc.spatial_shapes_hw = p->shapes.data();
  p->desc.level_start_index = p->starts.data();
  p->chunk = chunk_images < desc->B ? chunk_images : desc->B;
  p->nslots = slots;
  p->with_backward = with_backward ? 1 : 0;
  p->query_order = query_order;

  const size_t vs = dtype_size(desc->value_dtype), as = dtype_size(desc->attn_dtype);
  const size_t hd = size_t(desc->H) * desc->D, lp = size_t(desc->L) * desc->P;
  p->value_b = size_t(desc->S) * hd * vs;
  p->loc_b = size_t(desc->Q) * desc->H * lp * 2 * sizeof(float);
  p->attn_b = size_t(desc->Q) * desc->H * lp * as;
  p->out_b = size_t(desc->Q) * hd * vs;

  // The library's own descriptor checks, then the workspace one chunk needs.
  msda_b200_desc cd = p->desc;
  cd.B = p->chunk;
  if (int rc = msda_b200_internal_validate(&cd)) {
    delete p;
    return rc;  // last_error set by validate
  }
  if (p->with_backward) p->ws_bytes = msda_b200_backward_workspace_bytes(&cd);
  const size_t c = size_t(p->chunk);
  const size_t in_sz[4] = {p->value_b * c, p->loc_b * c, p->attn_b * c, p->with_backward ? p->out_b * c : 0};
  const size_t out_sz[4] = {p->out_b * c, p->with_backward ? p->value_b * c : 0, p->with_backward ? p->loc_b * c : 0,
                            p->with_backward ? p->attn_b * c : 0};
  size_t in_total = 0, out_total = 0;
  for (int i = 0; i < 4; ++i) {
    p->in_off[i] = in_total;
    in_total += align256(in_sz[i]);
    p->out_off[i] = out_total;
    out_total += align256(out_sz[i]);
  }

  cudaError_t e = cudaGetDevice(&p->device);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&p->s_comp, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->fork, cudaEventDisableTiming);
  for (int i = 0; i < kCopyLanes; ++i) {
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&p->s_h2d[i], cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&p->s_d2h[i], cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->tail[i], cudaEventDisableTiming);
  }
  p->slots.resize(size_t(slots));
  for (Slot& s : p->slots) {
    if (e == cudaSuccess) e = cudaMalloc(&s.in, in_total);
    if (e == cudaSuccess) e = cudaMalloc(&s.out, out_total);
    if (e == cudaSuccess && p->ws_bytes) e = cudaMalloc(&s.ws, p->ws_bytes);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.in_done, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.comp_done, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.out_done, cudaEventDisableTiming);
  }
  if (e != cudaSuccess) {
    release(p);
    return cuda_error("host_pipeline_create", e);
  }
  *pipeline = p;
  return MSDA_B200_OK;
}

extern "C" int msda_b200_host_pipeline_step(msda_b200_host_pipeline* p, const void* value, const float* sampling_loc,
                                            const void* attn_weight, const void* grad_output, void* output,
                                            void* grad_value, float* grad_sampling_loc, void* grad_attn_weight,
                                            void* stream) {
  if (!p) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "host_pipeline_step: NULL pipeline");
  if (p->poisoned)
    return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "host_pipeline_step: an earlier step failed; destroy the pipeline");
  const bool bw = p->with_backward != 0;
  if (!value || !sampling_loc || !attn_weight || !output ||
      (bw && (!grad_output || !grad_value || !grad_sampling_loc || !grad_attn_weight)))
    return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "host_pipeline_step: NULL host tensor pointer");
  DeviceGuard guard(p->device);
  HP_CUDA(cudaEventRecord(p->fork, static_cast<cudaStream_t>(stream)));
  for (int i = 0; i < kCopyLanes; ++i) HP_CUDA(cudaStreamWaitEvent(p->s_h2d[i], p->fork, 0));

  const char* h_in[4] = {static_cast<const char*>(value), reinterpret_cast<const char*>(sampling_loc),
                         static_cast<const char*>(attn_weight), static_cast<const char*>(grad_output)};
  char* h_out[4] = {static_cast<char*>(output), static_cast<char*>(grad_value),
                    reinterpret_cast<char*>(grad_sampling_loc), static_cast<char*>(grad_attn_weight)};
  const size_t in_img[4] = {p->value_b, p->loc_b, p->attn_b, p->out_b};
  const size_t out_img[4] = {p->out_b, p->value_b, p->loc_b, p->attn_b};
  const int n_io = bw ? 4 : 3;  // inputs copied in
  const int n_res = bw ? 4 : 1; // results copied out

  for (int32_t b0 = 0; b0 < p->desc.B; b0 += p->chunk) {
    const int32_t nb = (p->desc.B - b0 < p->chunk) ? p->desc.B - b0 : p->chunk;
    Slot& s = p->slots[size_t(p->next % uint64_t(p->nslots))];
    cudaStream_t s_in = p->s_h2d[p->next % kCopyLanes], s_out = p->s_d2h[p->next % kCopyLanes];
    ++p->next;
    // H2D: the slot's inputs are free once its previous kernels have run.
    HP_CUDA(cudaStreamWaitEvent(s_in, s.comp_done, 0));
    for (int i = 0; i < n_io; ++i)
      HP_CUDA(cudaMemcpyAsync(s.in + p->in_off[i], h_in[i] + size_t(b0) * in_img[i], size_t(nb) * in_img[i],
                              cudaMemcpyHostToDevice, s_in));
    HP_CUDA(cudaEventRecord(s.in_done, s_in));
    // Compute: inputs have landed, and the slot's previous results have left.
    HP_CUDA(cudaStreamWaitEvent(p->s_comp, s.in_done, 0));
    HP_CUDA(cudaStreamWaitEvent(p->s_comp, s.out_done, 0));
    msda_b200_desc cd = p->desc;
    cd.B = nb;
    int rc = msda_b200_forward(&cd, s.in + p->in_off[0], reinterpret_cast<const float*>(s.in + p->in_off[1]),
                               s.in + p->in_off[2], s.out + p->out_off[0], p->query_order, p->s_comp);
    if (rc == MSDA_B200_OK && bw)
      rc = msda_b200_backward(&cd, s.in + p->in_off[0], reinterpret_cast<const float*>(s.in + p->in_off[1]),
                              s.in + p->in_off[2], s.in + p->in_off[3], s.out + p->out_off[1],
                              reinterpret_cast<float*>(s.out + p->out_off[2]), s.out + p->out_off[3], s.ws,
                              p->ws_bytes, p->query_order, p->s_comp);
    if (rc != MSDA_B200_OK) {
      // keep the slot's event chain intact (later waits must not see a stale comp_done / out_done) and refuse
      // further steps: part of this batch never ran
      cudaEventRecord(s.comp_done, p->s_comp);
      cudaEventRecord(s.out_done, s_out);
      p->poisoned = true;
      return rc;
    }
    HP_CUDA(cudaEventRecord(s.comp_done, p->s_comp));
    // D2H
    HP_CUDA(cudaStreamWaitEvent(s_out, s.comp_done, 0));
    for (int i = 0; i < n_res; ++i)
      HP_CUDA(cudaMemcpyAsync(h_out[i] + size_t(b0) * out_img[i], s.out + p->out_off[i], size_t(nb) * out_img[i],
                              cudaMemcpyDeviceToHost, s_out));
    HP_CUDA(cudaEventRecord(s.out_done, s_out));
  }
  return MSDA_B200_OK;
}

extern "C" int msda_b200_host_pipeline_join(msda_b200_host_pipeline* p, void* stream) {
  if (!p) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "host_pipeline_join: NULL pipeline");
  DeviceGuard guard(p->device);
  // Every chunk ends with a D2H copy and each D2H stream runs its copies in order: their tails cover everything.
  for (int i = 0; i < kCopyLanes; ++i) {
    HP_CUDA(cudaEventRecord(p->tail[i], p->s_d2h[i]));
    HP_CUDA(cudaStreamWaitEvent(static_cast<cudaStream_t>(stream), p->tail[i], 0));
  }
  return MSDA_B200_OK;
}

extern "C" int msda_b200_host_pipeline_sync(msda_b200_host_pipeline* p) {
  if (!p) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "host_pipeline_sync: NULL pipeline");
  DeviceGuard guard(p->device);
  for (int i = 0; i < kCopyLanes; ++i) HP_CUDA(cudaStreamSynchronize(p->s_h2d[i]));
  HP_CUDA(cudaStreamSynchronize(p->s_comp));
  for (int i = 0; i < kCopyLanes; ++i) HP_CUDA(cudaStreamSynchronize(p->s_d2h[i]));
  return MSDA_B200_OK;
}

extern "C" int msda_b200_host_pipeline_destroy(msda_b200_host_pipeline* p) {
  if (!p) return MSDA_B200_OK;
  DeviceGuard guard(p->device);
  for (int i = 0; i < kCopyLanes; ++i) cudaStreamSynchronize(p->s_h2d[i]);
  cudaStreamSynchronize(p->s_comp);
  for (int i = 0; i < kCopyLanes; ++i) cudaStreamSynchronize(p->s_d2h[i]);
  release(p);
  return MSDA_B200_OK;
}
