// gemm_f32.cu -- float32 projections of the encoder layer on the Blackwell tensor cores (round 2).
//
// The reference trains in float32 (REF/models/mask2former/train.py never casts), and for float32 tensors PyTorch runs
// the attention module's and the FFN's projections (M2F:947-956, 981, 1052-1056) as CUDA-core SGEMMs: 52-58 TFLOP/s on a
// B200, 15 of the 20 ms of an encoder layer at BASELINE config 2. cuBLASLt 12.9 can run the same float32 GEMM on the
// bf16 tensor cores by splitting every operand into three bfloat16 terms and accumulating the nine products in float32
// (CUBLAS_COMPUTE_32F_EMULATED_16BFX9). Measured on B200 for the layer's shapes (profiles/micro/gemm_emul.cu,
// profiles/r02_gemm_emul.log): 78-129 TFLOP/s, 1.7-2.3x the SGEMM, with a SMALLER error against float64 (0.4-1.3e-7 of
// max |y|, SGEMM 1.6-5.8e-7; TF32 would be 7-10x faster but 1-3.5e-4 off) -- so this is not a precision trade.
//
// The GEMMs stay library calls (north star: "the value/output projections use tensor cores only because they are dense
// GEMMs"). The PyTorch wheel bundles its own cuBLASLt without the emulated compute type, and a library with the same
// SONAME cannot be linked a second time, so the CUDA toolkit's libcublasLt is opened by ABSOLUTE path at first use
// (dlopen, RTLD_LOCAL: a private second copy) and called through function pointers. Where it is missing or refuses the
// compute type, msda_b200_linear_f32_available() returns 0 and the Python side keeps torch's SGEMM -- loudly visible in
// bench_layer.py's numbers, never silently wrong.
//
// Row-major contract (what F.linear uses):  y[M,N] = x[M,K] . w[N,K]^T (+ bias[N]) (+ ReLU)
//                                           grad_x[M,K] = grad_y[M,N] . w[N,K]
//                                           grad_w[N,K] = grad_y[M,N]^T . x[M,K]
// mapped onto cuBLASLt's column-major GEMM by computing the transposed product (no copies).
#include <cublasLt.h>
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <mutex>

#include "msda_b200.h"
#include "internal.h"

namespace {

struct Lt {
  void* dl = nullptr;
  bool ok = false;
  decltype(&cublasLtCreate) Create;
  decltype(&cublasLtMatmulDescCreate) DescCreate;
  decltype(&cublasLtMatmulDescDestroy) DescDestroy;
  decltype(&cublasLtMatmulDescSetAttribute) DescSet;
  decltype(&cublasLtMatrixLayoutCreate) LayoutCreate;
  decltype(&cublasLtMatrixLayoutDestroy) LayoutDestroy;
  decltype(&cublasLtMatmulPreferenceCreate) PrefCreate;
  decltype(&cublasLtMatmulPreferenceDestroy) PrefDestroy;
  decltype(&cublasLtMatmulPreferenceSetAttribute) PrefSet;
  decltype(&cublasLtMatmulAlgoGetHeuristic) Heuristic;
  decltype(&cublasLtMatmul) Matmul;
};
Lt g_lt;
std::once_flag g_lt_once;

template <typename F>
bool sym(void* dl, const char* name, F& f) {
  f = reinterpret_cast<F>(dlsym(dl, name));
  return f != nullptr;
}

void load_lt() {
  const char* env = getenv("MSDA_B200_CUBLASLT");
  const char* paths[] = {env, "/usr/local/cuda/lib64/libcublasLt.so.12", "/usr/local/cuda-12.9/lib64/libcublasLt.so.12"};
  for (const char* p : paths) {
    if (!p || !*p) continue;
    void* dl = dlopen(p, RTLD_NOW | RTLD_LOCAL);
    if (!dl) continue;
    Lt t;
    t.dl = dl;
    if (sym(dl, "cublasLtCreate", t.Create) && sym(dl, "cublasLtMatmulDescCreate", t.DescCreate) &&
        sym(dl, "cublasLtMatmulDescDestroy", t.DescDestroy) && sym(dl, "cublasLtMatmulDescSetAttribute", t.DescSet) &&
        sym(dl, "cublasLtMatrixLayoutCreate", t.LayoutCreate) && sym(dl, "cublasLtMatrixLayoutDestroy", t.LayoutDestroy) &&
        sym(dl, "cublasLtMatmulPreferenceCreate", t.PrefCreate) && sym(dl, "cublasLtMatmulPreferenceDestroy", t.PrefDestroy) &&
        sym(dl, "cublasLtMatmulPreferenceSetAttribute", t.PrefSet) && sym(dl, "cublasLtMatmulAlgoGetHeuristic", t.Heuristic) &&
        sym(dl, "cublasLtMatmul", t.Matmul)) {
      t.ok = true;
      g_lt = t;
      return;
    }
    dlclose(dl);
  }
}

// one handle and a small plan cache per host thread (the autograd thread and the main thread each get their own)
struct Plan {
  int kind = -1, device = -1, epilogue = 0;
  long long M = 0;
  int N = 0, K = 0;
  size_t ws = 0;
  cublasLtMatmulDesc_t op = nullptr;
  cublasLtMatrixLayout_t a = nullptr, b = nullptr, c = nullptr;
  cublasLtMatmulAlgo_t algo;
};
constexpr int kPlans = 32;
struct ThreadState {
  int device = -1;
  cublasLtHandle_t handle = nullptr;
  Plan plans[kPlans];
  int next = 0;
};
thread_local ThreadState g_ts;

enum { KIND_FWD = 0, KIND_GRAD_X = 1, KIND_GRAD_W = 2 };

void destroy(Plan& p) {
  if (p.op) g_lt.DescDestroy(p.op);
  if (p.a) g_lt.LayoutDestroy(p.a);
  if (p.b) g_lt.LayoutDestroy(p.b);
  if (p.c) g_lt.LayoutDestroy(p.c);
  p = Plan();
}

// Column-major view of the three row-major products (see the file header): C[m x n] = op(A) . op(B)
int make_plan(Plan& p, int kind, long long M, int N, int K, int epilogue, size_t ws) {
  cublasOperation_t ta, tb;
  long long m, n, k, lda, ldb, ldc, ar, ac, br, bc;  // stored (untransposed) column-major shapes of A and B
  if (kind == KIND_FWD) {            // y^T[N,M] = w[N,K] . x^T[K,M]:  A = w as (K x N) col-major, transposed
    ta = CUBLAS_OP_T; tb = CUBLAS_OP_N; m = N; n = M; k = K; ar = K; ac = N; lda = K; br = K; bc = M; ldb = K; ldc = N;
  } else if (kind == KIND_GRAD_X) {  // gx^T[K,M] = w^T[K,N] . gy^T[N,M]: A = w as (K x N), B = gy as (N x M)
    ta = CUBLAS_OP_N; tb = CUBLAS_OP_N; m = K; n = M; k = N; ar = K; ac = N; lda = K; br = N; bc = M; ldb = N; ldc = K;
  } else {                           // gw^T[K,N] = x^T[K,M] . gy[M,N]:   A = x as (K x M), B = gy as (N x M), transposed
    ta = CUBLAS_OP_N; tb = CUBLAS_OP_T; m = K; n = N; k = M; ar = K; ac = M; lda = K; br = N; bc = M; ldb = N; ldc = K;
  }
  (void)k;
  if (g_lt.DescCreate(&p.op, CUBLAS_COMPUTE_32F_EMULATED_16BFX9, CUDA_R_32F) != CUBLAS_STATUS_SUCCESS) return 1;
  if (g_lt.DescSet(p.op, CUBLASLT_MATMUL_DESC_TRANSA, &ta, sizeof(ta)) != CUBLAS_STATUS_SUCCESS) return 1;
  if (g_lt.DescSet(p.op, CUBLASLT_MATMUL_DESC_TRANSB, &tb, sizeof(tb)) != CUBLAS_STATUS_SUCCESS) return 1;
  if (epilogue) {
    const cublasLtEpilogue_t ep = epilogue == 2 ? CUBLASLT_EPILOGUE_RELU_BIAS : CUBLASLT_EPILOGUE_BIAS;
    if (g_lt.DescSet(p.op, CUBLASLT_MATMUL_DESC_EPILOGUE, &ep, sizeof(ep)) != CUBLAS_STATUS_SUCCESS) return 1;
  }
  if (g_lt.LayoutCreate(&p.a, CUDA_R_32F, (uint64_t)ar, (uint64_t)ac, lda) != CUBLAS_STATUS_SUCCESS) return 1;
  if (g_lt.LayoutCreate(&p.b, CUDA_R_32F, (uint64_t)br, (uint64_t)bc, ldb) != CUBLAS_STATUS_SUCCESS) return 1;
  if (g_lt.LayoutCreate(&p.c, CUDA_R_32F, (uint64_t)m, (uint64_t)n, ldc) != CUBLAS_STATUS_SUCCESS) return 1;
  cublasLtMatmulPreference_t pref = nullptr;
  if (g_lt.PrefCreate(&pref) != CUBLAS_STATUS_SUCCESS) return 1;
  g_lt.PrefSet(pref, CUBLASLT_MATMUL_PREF_MAX_WORKSPACE_BYTES, &ws, sizeof(ws));
  cublasLtMatmulHeuristicResult_t h;
  int found = 0;
  const cublasStatus_t st = g_lt.Heuristic(g_ts.handle, p.op, p.a, p.b, p.c, p.c, pref, 1, &h, &found);
  g_lt.PrefDestroy(pref);
  if (st != CUBLAS_STATUS_SUCCESS || found == 0) return 2;
  p.algo = h.algo;
  p.kind = kind; p.M = M; p.N = N; p.K = K; p.epilogue = epilogue; p.ws = ws; p.device = g_ts.device;
  return 0;
}

int ensure_thread_state() {
  std::call_once(g_lt_once, load_lt);
  if (!g_lt.ok) return 1;
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess) return 1;
  if (g_ts.handle && g_ts.device != dev) {  // another device on this thread: plans and handle belong to the old context
    for (Plan& p : g_ts.plans) destroy(p);
    g_ts.handle = nullptr;                  // (the old handle is left to its context; one process per GPU never gets here)
  }
  if (!g_ts.handle) {
    if (g_lt.Create(&g_ts.handle) != CUBLAS_STATUS_SUCCESS) return 1;
    g_ts.device = dev;
  }
  return 0;
}

int run(int kind, long long M, int N, int K, int epilogue, const float* A, const float* B, float* C, const float* bias,
        void* workspace, size_t ws, cudaStream_t st, const char* what) {
  if (M < 0 || N <= 0 || K <= 0) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "linear_f32: bad shape");
  if (M == 0) return MSDA_B200_OK;
  if (!A || !B || !C || (epilogue && !bias)) return msda_b200_internal_fail(MSDA_B200_ERR_INVALID, "linear_f32: NULL tensor pointer");
  if (ensure_thread_state())
    return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "linear_f32: cuBLASLt with float32 emulation is not available");
  Plan* p = nullptr;
  for (Plan& q : g_ts.plans)
    if (q.kind == kind && q.M == M && q.N == N && q.K == K && q.epilogue == epilogue && q.ws == ws && q.device == g_ts.device) {
      p = &q;
      break;
    }
  if (!p) {
    Plan& slot = g_ts.plans[g_ts.next];
    g_ts.next = (g_ts.next + 1) % kPlans;
    destroy(slot);
    const int rc = make_plan(slot, kind, M, N, K, epilogue, ws);
    if (rc) {
      destroy(slot);
      return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED,
                                     rc == 2 ? "linear_f32: cuBLASLt offers no algorithm for the emulated float32 product"
                                             : "linear_f32: cuBLASLt descriptor setup failed");
    }
    p = &slot;
  }
  if (epilogue && g_lt.DescSet(p->op, CUBLASLT_MATMUL_DESC_BIAS_POINTER, &bias, sizeof(bias)) != CUBLAS_STATUS_SUCCESS)
    return msda_b200_internal_fail(MSDA_B200_ERR_CUDA, "linear_f32: cannot set the bias pointer");
  const float one = 1.f, zero = 0.f;
  const cublasStatus_t s = g_lt.Matmul(g_ts.handle, p->op, &one, A, p->a, B, p->b, &zero, C, p->c, C, p->c, &p->algo,
                                       workspace, ws, st);
  if (s != CUBLAS_STATUS_SUCCESS) {
    char msg[96];
    snprintf(msg, sizeof(msg), "%s: cublasLtMatmul failed (%d)", what, (int)s);
    return msda_b200_internal_fail(MSDA_B200_ERR_CUDA, msg);
  }
  return MSDA_B200_OK;
}

}  // namespace

extern "C" {

int msda_b200_linear_f32_available(void) {
  if (ensure_thread_state()) return 0;
  // probe once per thread: does this cuBLASLt accept the emulated compute type for a small product?
  static thread_local int probed = -1;
  if (probed < 0) {
    Plan p;
    probed = make_plan(p, KIND_FWD, 128, 128, 128, 0, 0) == 0 ? 1 : 0;
    destroy(p);
  }
  return probed;
}

int msda_b200_linear_f32_forward(const float* x, const float* weight, const float* bias, int relu, float* y, int64_t rows,
                                 int32_t out_features, int32_t in_features, void* workspace, size_t workspace_bytes,
                                 void* stream) {
  const int ep = bias ? (relu ? 2 : 1) : 0;
  if (relu && !bias) return msda_b200_internal_fail(MSDA_B200_ERR_UNSUPPORTED, "linear_f32_forward: ReLU needs a bias");
  return run(KIND_FWD, rows, out_features, in_features, ep, weight, x, y, bias, workspace, workspace_bytes,
             reinterpret_cast<cudaStream_t>(stream), "linear_f32_forward");
}

int msda_b200_linear_f32_grad_input(const float* grad_y, const float* weight, float* grad_x, int64_t rows,
                                    int32_t out_features, int32_t in_features, void* workspace, size_t workspace_bytes,
                                    void* stream) {
  return run(KIND_GRAD_X, rows, out_features, in_features, 0, weight, grad_y, grad_x, nullptr, workspace, workspace_bytes,
             reinterpret_cast<cudaStream_t>(stream), "linear_f32_grad_input");
}

int msda_b200_linear_f32_grad_weight(const float* grad_y, const float* x, float* grad_weight, int64_t rows,
                                     int32_t out_features, int32_t in_features, void* workspace, size_t workspace_bytes,
                                     void* stream) {
  return run(KIND_GRAD_W, rows, out_features, in_features, 0, x, grad_y, grad_weight, nullptr, workspace, workspace_bytes,
             reinterpret_cast<cudaStream_t>(stream), "linear_f32_grad_weight");
}

}  // extern "C"
