// extern "C" entry points of libgrafp_b200.so: argument validation + dispatch.
#include <atomic>
#include <cctype>
#include <cstring>
#include <mutex>
#include <string>

#include "knn.cuh"

namespace grafp {

namespace {
thread_local std::string g_error;
thread_local const char* g_knn_algo = "none";
thread_local const char* g_knn_variant = "none";
}  // namespace

void set_error(const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_error = buf;
}
void clear_error() { g_error.clear(); }

int check_launch(const char* what) {
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: launch failed: %s", what, cudaGetErrorString(e));
    return static_cast<int>(e);
  }
  return GRAFP_OK;
}

int current_device() {
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return -1; }
  return dev;
}

// ---- run-time options: defaults, overridden once at load by GRAFP_<NAME>, then by grafp_set_option ----
namespace {
struct OptionSpec { const char* name; int def; };
const OptionSpec kOptionSpecs[OPT_COUNT] = {
    {"mr_fwd_form", 2}, {"mr_bwd_form", 2}, {"knn_epilogue", 0}, {"edge_bwd_row", 1}, {"gather_row", 1},
    {"edge_row", 1},    {"maxk_row", 1},    {"bn_reverse", 1},   {"bn_persistent", 1}, {"bn_l2_keep_mb", 80}, {"check_index", 0},
    {"conv_gemm", 1},
};
std::atomic<int> g_options[OPT_COUNT];
std::once_flag g_options_once;
void init_options() {
  for (int i = 0; i < OPT_COUNT; ++i) {
    int v = kOptionSpecs[i].def;
    char env[64] = "GRAFP_";
    size_t n = strlen(env);
    for (const char* c = kOptionSpecs[i].name; *c && n + 1 < sizeof(env); ++c) env[n++] = (char)toupper((unsigned char)*c);
    env[n] = 0;
    if (const char* e = getenv(env)) v = atoi(e);
    g_options[i].store(v, std::memory_order_relaxed);
  }
}
int option_index(const char* name) {
  if (name == nullptr) return -1;
  for (int i = 0; i < OPT_COUNT; ++i)
    if (strcmp(name, kOptionSpecs[i].name) == 0) return i;
  return -1;
}
}  // namespace

int option(Option o) {
  std::call_once(g_options_once, init_options);
  return g_options[o].load(std::memory_order_relaxed);
}

int num_sms() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

// Every entry point refuses to run anywhere but on an sm_100 device with device pointers.
static int require_device(const char* fn) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    set_error("%s: no CUDA device available (%s); this library has no CPU path", fn, cudaGetErrorString(e));
    cudaGetLastError();
    return GRAFP_ENODEVICE;
  }
  static int major[64] = {0};
  if (dev >= 0 && dev < 64 && major[dev] == 0) {
    int m = 0;
    cudaDeviceGetAttribute(&m, cudaDevAttrComputeCapabilityMajor, dev);
    major[dev] = m;
  }
  if (dev >= 0 && dev < 64 && major[dev] != 10) {
    set_error("%s: device %d has compute capability %d.x; libgrafp_b200 is built for sm_100a only", fn, dev, major[dev]);
    return GRAFP_ENODEVICE;
  }
  return GRAFP_OK;
}

static int require_device_ptr(const char* fn, const char* name, const void* p) {
  cudaPointerAttributes a;
  const cudaError_t e = cudaPointerGetAttributes(&a, p);
  if (e != cudaSuccess || (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged)) {
    cudaGetLastError();
    set_error("%s: %s is not a device pointer (there is no CPU path)", fn, name);
    return GRAFP_EINVAL;
  }
  return GRAFP_OK;
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace grafp

using namespace grafp;

#define COMMON_SHAPE_CHECKS(fn)                                                                                 \
  clear_error();                                                                                                \
  GRAFP_REQUIRE(B > 0 && N > 0 && M > 0 && C > 0 && k > 0, GRAFP_EINVAL, fn ": B, N, M, C, k must be positive"); \
  GRAFP_REQUIRE(dtype == GRAFP_F32 || dtype == GRAFP_BF16, GRAFP_EUNSUPPORTED, fn ": dtype %d not supported", dtype); \
  GRAFP_REQUIRE(k <= 255, GRAFP_EUNSUPPORTED, fn ": k = %d exceeds the uint8 argmax range", k);                 \
  { int rc_ = require_device(fn); if (rc_ != GRAFP_OK) return rc_; }

extern "C" {

int grafp_abi_version(void) { return GRAFP_ABI_VERSION; }

int grafp_set_option(const char* name, int value) {
  clear_error();
  const int i = option_index(name);
  GRAFP_REQUIRE(i >= 0, GRAFP_EINVAL, "grafp_set_option: unknown option '%s'", name ? name : "(null)");
  std::call_once(g_options_once, init_options);
  g_options[i].store(value, std::memory_order_relaxed);
  return GRAFP_OK;
}

int grafp_check_index(const void* idx, int idx_is_i64, long long count, int limit, int* bad_count, void* stream) {
  clear_error();
  GRAFP_REQUIRE(idx && bad_count && count > 0 && limit > 0, GRAFP_EINVAL, "grafp_check_index: idx, bad_count must be non-null, count and limit positive");
  { int rc = require_device("grafp_check_index"); if (rc != GRAFP_OK) return rc; }
  { int rc = require_device_ptr("grafp_check_index", "idx", idx); if (rc) return rc; }
  return launch_check_index(idx, idx_is_i64, count, limit, bad_count, static_cast<cudaStream_t>(stream));
}

int grafp_get_option(const char* name) {
  const int i = option_index(name);
  if (i < 0) return GRAFP_EINVAL;
  return option(static_cast<Option>(i));
}
const char* grafp_last_error(void) { return g_error.c_str(); }
const char* grafp_knn_last_algo(void) { return g_knn_algo; }
const char* grafp_knn_last_variant(void) { return g_knn_variant; }

size_t grafp_knn_workspace_bytes(int B, int N, int M, int C, int K, int dtype) {
  (void)K; (void)dtype;
  if (B <= 0 || N <= 0 || M <= 0 || C <= 0) return 0;
  const size_t qx = align_up((size_t)B * N * C * sizeof(float), 1024);
  const size_t qy = align_up((size_t)B * M * C * sizeof(float), 1024);
  const size_t sx = align_up((size_t)B * N * sizeof(float), 1024);
  const size_t sy = align_up((size_t)B * M * sizeof(float), 1024);
  // hi+lo (or x_hat) for queries and keys, squared norms, round hand-over bounds (K > 16), base alignment
  return 2 * (qx + qy) + sx + sy + 2 * sx + 1024;
}

int grafp_knn_fwd(const void* x, const void* y, const float* relpos, int64_t* nn_idx, int32_t* nn_idx32, int B, int N,
                  int M, int C, int k, int dilation, int emit_all, int normalize, int dtype, int algo, int metric,
                  void* workspace, size_t workspace_bytes, void* stream) {
  COMMON_SHAPE_CHECKS("grafp_knn_fwd");
  GRAFP_REQUIRE(metric == GRAFP_METRIC_L2 || metric == GRAFP_METRIC_COSINE, GRAFP_EINVAL, "grafp_knn_fwd: unknown metric %d", metric);
  GRAFP_REQUIRE(x && nn_idx && workspace, GRAFP_EINVAL, "grafp_knn_fwd: x, nn_idx and workspace must be non-null");
  GRAFP_REQUIRE(dilation > 0, GRAFP_EINVAL, "grafp_knn_fwd: dilation must be positive");
  GRAFP_REQUIRE(y != nullptr || M == N, GRAFP_EINVAL, "grafp_knn_fwd: M (%d) must equal N (%d) when y is null", M, N);
  GRAFP_REQUIRE(B <= 65535, GRAFP_EUNSUPPORTED, "grafp_knn_fwd: B = %d exceeds 65535", B);
  const long long K = (long long)k * dilation;
  GRAFP_REQUIRE(K <= M, GRAFP_EINVAL, "grafp_knn_fwd: k*dilation = %lld exceeds the number of key nodes %d", K, M);
  GRAFP_REQUIRE(K <= GRAFP_KNN_MAX_K, GRAFP_EUNSUPPORTED, "grafp_knn_fwd: k*dilation = %lld exceeds %d", K, GRAFP_KNN_MAX_K);
  GRAFP_REQUIRE(algo >= GRAFP_KNN_AUTO && algo <= GRAFP_KNN_TC_TF32, GRAFP_EINVAL, "grafp_knn_fwd: unknown algo %d", algo);
  GRAFP_REQUIRE(workspace_bytes >= grafp_knn_workspace_bytes(B, N, M, C, (int)K, dtype), GRAFP_EWORKSPACE,
                "grafp_knn_fwd: workspace of %zu bytes is smaller than grafp_knn_workspace_bytes()", workspace_bytes);
  { int rc = require_device_ptr("grafp_knn_fwd", "x", x); if (rc) return rc; }
  { int rc = require_device_ptr("grafp_knn_fwd", "nn_idx", nn_idx); if (rc) return rc; }
  cudaStream_t s = static_cast<cudaStream_t>(stream);

  // tensor-core kernels: f16x3 (knn_tc2.cu, K <= 64) preferred, tf32x3 (knn_tc.cu) for the rest of the envelope
  // (f16x3 needs |x| <= 1, i.e. the normalised features DenseDilatedKnnGraph always passes)
  const bool tc2_ok = relpos == nullptr && normalize != 0 && knn_tc2_supported(N, M, C, (int)K, dtype, y == nullptr);
  const bool tc1_ok = relpos == nullptr && knn_tc_supported(N, M, C, (int)K, dtype);
  if ((algo == GRAFP_KNN_TC && !tc2_ok && !tc1_ok) || (algo == GRAFP_KNN_TC_TF32 && !tc1_ok)) {
    set_error("grafp_knn_fwd: the tcgen05 path does not support N=%d M=%d C=%d K=%lld dtype=%d", N, M, C, K, dtype);
    return GRAFP_EUNSUPPORTED;
  }
  const bool use_tc2 = tc2_ok && (algo == GRAFP_KNN_TC || algo == GRAFP_KNN_AUTO);
  const bool use_tc = use_tc2 || algo == GRAFP_KNN_TC_TF32 || (tc1_ok && (algo == GRAFP_KNN_TC || algo == GRAFP_KNN_AUTO));

  // carve the workspace
  char* base = reinterpret_cast<char*>(align_up(reinterpret_cast<size_t>(workspace), 1024));
  const size_t qx = align_up((size_t)B * N * C * sizeof(float), 1024);
  const size_t qy = align_up((size_t)B * M * C * sizeof(float), 1024);
  const size_t sx = align_up((size_t)B * N * sizeof(float), 1024);
  float* x_hi = reinterpret_cast<float*>(base);
  float* x_lo = reinterpret_cast<float*>(base + qx);
  float* y_hi = reinterpret_cast<float*>(base + 2 * qx);
  float* y_lo = reinterpret_cast<float*>(base + 2 * qx + qy);
  float* x_sq = reinterpret_cast<float*>(base + 2 * qx + 2 * qy);
  float* y_sq = reinterpret_cast<float*>(base + 2 * qx + 2 * qy + sx);
  void* bounds = base + 2 * qx + 2 * qy + sx + align_up((size_t)B * M * sizeof(float), 1024);

  const int mode = use_tc2 ? 3 : (use_tc ? 1 : 0);  // fp16 hi/lo planes, tf32 hi/lo planes, or plain fp32 x_hat
  int rc;
  if (dtype == GRAFP_F32) {
    rc = launch_knn_normalize<float>(x, x_hi, x_lo, x_sq, (long long)B * N, C, mode, normalize != 0, s);
    if (rc == GRAFP_OK && y) rc = launch_knn_normalize<float>(y, y_hi, y_lo, y_sq, (long long)B * M, C, mode, normalize != 0, s);
  } else {
    rc = launch_knn_normalize<__nv_bfloat16>(x, x_hi, x_lo, x_sq, (long long)B * N, C, mode, normalize != 0, s);
    if (rc == GRAFP_OK && y) rc = launch_knn_normalize<__nv_bfloat16>(y, y_hi, y_lo, y_sq, (long long)B * M, C, mode, normalize != 0, s);
  }
  if (rc != GRAFP_OK) return rc;
  if (metric == GRAFP_METRIC_COSINE) {  // 2 (1 - x.y) = (1 - 2 x.y) + 1: the L2 epilogue with unit squared norms
    rc = launch_fill_f32(x_sq, (long long)B * N, 1.f, s);
    if (rc == GRAFP_OK && y) rc = launch_fill_f32(y_sq, (long long)B * M, 1.f, s);
    if (rc != GRAFP_OK) return rc;
  }
  if (!y) { y_hi = x_hi; y_lo = x_lo; y_sq = x_sq; }

  const int k_out = emit_all ? (int)K : k;
  const int stride = emit_all ? 1 : dilation;
  if (use_tc2) {
    g_knn_algo = "tcgen05";
    g_knn_variant = "f16x3";
    return launch_knn_tc2(x_hi, x_lo, x_sq, y_hi, y_lo, y_sq, reinterpret_cast<long long*>(nn_idx), nn_idx32, B, N, M, C,
                          (int)K, k_out, stride, dtype, y == nullptr, bounds, s);
  }
  if (use_tc) {
    g_knn_algo = "tcgen05";
    g_knn_variant = "tf32x3";
    return launch_knn_tc(x_hi, x_lo, x_sq, y_hi, y_lo, y_sq, relpos, reinterpret_cast<long long*>(nn_idx), nn_idx32, B, N,
                         M, C, (int)K, k_out, stride, dtype, s);
  }
  g_knn_algo = "simt";
  g_knn_variant = "fp32";
  return launch_knn_simt(x_hi, x_sq, y_hi, y_sq, relpos, reinterpret_cast<long long*>(nn_idx), nn_idx32, B, N, M, C,
                         (int)K, k_out, stride, s);
}

#define DISPATCH_DTYPE(call_f32, call_bf16) (dtype == GRAFP_F32 ? (call_f32) : (call_bf16))

int grafp_mr_aggregate_fwd(const void* x, const void* y, const void* nbr_idx, const void* ctr_idx, int idx_is_i64,
                           void* out, uint8_t* argmax, int B, int N, int M, int C, int k, int dtype, void* stream) {
  COMMON_SHAPE_CHECKS("grafp_mr_aggregate_fwd");
  GRAFP_REQUIRE(x && nbr_idx && out, GRAFP_EINVAL, "grafp_mr_aggregate_fwd: x, nbr_idx and out must be non-null");
  GRAFP_REQUIRE(y != nullptr || M == N, GRAFP_EINVAL, "grafp_mr_aggregate_fwd: M must equal N when y is null");
  { int rc = require_device_ptr("grafp_mr_aggregate_fwd", "x", x); if (rc) return rc; }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  return DISPATCH_DTYPE(launch_mr_aggregate_fwd<float>(x, y, nbr_idx, ctr_idx, idx_is_i64, out, argmax, B, N, M, C, k, s),
                        launch_mr_aggregate_fwd<__nv_bfloat16>(x, y, nbr_idx, ctr_idx, idx_is_i64, out, argmax, B, N, M, C, k, s));
}

size_t grafp_mr_aggregate_bwd_workspace_bytes(int B, int N, int k) {
  if (B <= 0 || N <= 0 || k <= 0) return 0;
  return mr_bwd_workspace_bytes(B, N, k);
}

int grafp_mr_aggregate_bwd(const void* grad_out, const uint8_t* argmax, const void* nbr_idx, const void* ctr_idx,
                           int idx_is_i64, void* grad_x, void* grad_y, int B, int N, int M, int C, int k, int dtype,
                           void* workspace, size_t workspace_bytes, void* stream) {
  COMMON_SHAPE_CHECKS("grafp_mr_aggregate_bwd");
  GRAFP_REQUIRE(grad_out && argmax && nbr_idx && grad_x, GRAFP_EINVAL,
                "grafp_mr_aggregate_bwd: grad_out, argmax, nbr_idx and grad_x must be non-null");
  GRAFP_REQUIRE(grad_y != nullptr || M == N, GRAFP_EINVAL, "grafp_mr_aggregate_bwd: M must equal N when grad_y is null");
  { int rc = require_device_ptr("grafp_mr_aggregate_bwd", "grad_out", grad_out); if (rc) return rc; }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  return DISPATCH_DTYPE(launch_mr_aggregate_bwd<float>(grad_out, argmax, nbr_idx, ctr_idx, idx_is_i64, grad_x, grad_y, B, N, M, C, k, workspace, workspace_bytes, s),
                        launch_mr_aggregate_bwd<__nv_bfloat16>(grad_out, argmax, nbr_idx, ctr_idx, idx_is_i64, grad_x, grad_y, B, N, M, C, k, workspace, workspace_bytes, s));
}

int grafp_gather_fwd(const void* src, const void* idx, int idx_is_i64, void* out, int B, int N, int M, int C, int k,
                     int dtype, void* stream) {
  COMMON_SHAPE_CHECKS("grafp_gather_fwd");
  GRAFP_REQUIRE(src && idx && out, GRAFP_EINVAL, "grafp_gather_fwd: src, idx and out must be non-null");
  { int rc = require_device_ptr("grafp_gather_fwd", "src", src); if (rc) return rc; }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  return DISPATCH_DTYPE(launch_gather_fwd<float>(src, idx, idx_is_i64, out, B, N, M, C, k, s),
                        launch_gather_fwd<__nv_bfloat16>(src, idx, idx_is_i64, out, B, N, M, C, k, s));
}

int grafp_gather_bwd(const void* grad_out, const void* idx, int idx_is_i64, void* grad_src, int B, int N, int M, int C,
                     int k, int dtype, void* stream) {
  COMMON_SHAPE_CHECKS("grafp_gather_bwd");
  GRAFP_REQUIRE(grad_out && idx && grad_src, GRAFP_EINVAL, "grafp_gather_bwd: grad_out, idx and grad_src must be non-null");
  { int rc = require_device_ptr("grafp_gather_bwd", "grad_out", grad_out); if (rc) return rc; }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  return DISPATCH_DTYPE(launch_gather_bwd<float>(grad_out, idx, idx_is_i64, grad_src, B, N, M, C, k, s),
                        launch_gather_bwd<__nv_bfloat16>(grad_out, idx, idx_is_i64, grad_src, B, N, M, C, k, s));
}

int grafp_neighbor_sum_fwd(const void* src, const void* idx, int idx_is_i64, void* out, int B, int N, int M, int C, int k,
                           int dtype, void* stream) {
  COMMON_SHAPE_CHECKS("grafp_neighbor_sum_fwd");
  GRAFP_REQUIRE(src && idx && out, GRAFP_EINVAL, "grafp_neighbor_sum_fwd: src, idx and out must be non-null");
  { int rc = require_device_ptr("grafp_neighbor_sum_fwd", "src", src); if (rc) return rc; }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  return DISPATCH_DTYPE(launch_neighbor_sum_fwd<float>(src, idx, idx_is_i64, out, B, N, M, C, k, s),
                        launch_neighbor_sum_fwd<__nv_bfloat16>(src, idx, idx_is_i64, out, B, N, M, C, k, s));
}

int grafp_neighbor_sum_bwd(const void* grad_out, const void* idx, int idx_is_i64, void* grad_src, int B, int N, int M,
                           int C, int k, int dtype, void* stream) {
  COMMON_SHAPE_CHECKS("grafp_neighbor_sum_bwd");
  GRAFP_REQUIRE(grad_out && idx && grad_src, GRAFP_EINVAL, "grafp_neighbor_sum_bwd: grad_out, idx and grad_src must be non-null");
  { int rc = require_device_ptr("grafp_neighbor_sum_bwd", "grad_out", grad_out); if (rc) return rc; }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  return DISPATCH_DTYPE(launch_neighbor_sum_bwd<float>(grad_out, idx, idx_is_i64, grad_src, B, N, M, C, k, s),
                        launch_neighbor_sum_bwd<__nv_bfloat16>(grad_out, idx, idx_is_i64, grad_src, B, N, M, C, k, s));
}

int grafp_edge_gather_fwd(const void* x, const void* y, const void* nbr_idx, const void* ctr_idx, int idx_is_i64,
                          void* out, int B, int N, int M, int C, int k, int dtype, void* stream) {
  COMMON_SHAPE_CHECKS("grafp_edge_gather_fwd");
  GRAFP_REQUIRE(x && nbr_idx && out, GRAFP_EINVAL, "grafp_edge_gather_fwd: x, nbr_idx and out must be non-null");
  GRAFP_REQUIRE(y != nullptr || M == N, GRAFP_EINVAL, "grafp_edge_gather_fwd: M must equal N when y is null");
  { int rc = require_device_ptr("grafp_edge_gather_fwd", "x", x); if (rc) return rc; }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  return DISPATCH_DTYPE(launch_edge_gather_fwd<float>(x, y, nbr_idx, ctr_idx, idx_is_i64, out, B, N, M, C, k, s),
                        launch_edge_gather_fwd<__nv_bfloat16>(x, y, nbr_idx, ctr_idx, idx_is_i64, out, B, N, M, C, k, s));
}

int grafp_edge_gather_bwd(const void* grad_out, const void* nbr_idx, const void* ctr_idx, int idx_is_i64, void* grad_x,
                          void* grad_y, int B, int N, int M, int C, int k, int dtype, void* stream) {
  COMMON_SHAPE_CHECKS("grafp_edge_gather_bwd");
  GRAFP_REQUIRE(grad_out && nbr_idx && grad_x, GRAFP_EINVAL, "grafp_edge_gather_bwd: grad_out, nbr_idx and grad_x must be non-null");
  GRAFP_REQUIRE(grad_y != nullptr || M == N, GRAFP_EINVAL, "grafp_edge_gather_bwd: M must equal N when grad_y is null");
  { int rc = require_device_ptr("grafp_edge_gather_bwd", "grad_out", grad_out); if (rc) return rc; }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  return DISPATCH_DTYPE(launch_edge_gather_bwd<float>(grad_out, nbr_idx, ctr_idx, idx_is_i64, grad_x, grad_y, B, N, M, C, k, s),
                        launch_edge_gather_bwd<__nv_bfloat16>(grad_out, nbr_idx, ctr_idx, idx_is_i64, grad_x, grad_y, B, N, M, C, k, s));
}

int grafp_max_over_k_fwd(const void* h, void* out, uint8_t* argmax, int B, int N, int C, int k, int dtype, void* stream) {
  const int M = 1;
  COMMON_SHAPE_CHECKS("grafp_max_over_k_fwd");
  GRAFP_REQUIRE(h && out, GRAFP_EINVAL, "grafp_max_over_k_fwd: h and out must be non-null");
  { int rc = require_device_ptr("grafp_max_over_k_fwd", "h", h); if (rc) return rc; }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  return DISPATCH_DTYPE(launch_max_over_k_fwd<float>(h, out, argmax, B, N, C, k, s),
                        launch_max_over_k_fwd<__nv_bfloat16>(h, out, argmax, B, N, C, k, s));
}

int grafp_max_over_k_bwd(const void* grad_out, const uint8_t* argmax, void* grad_h, int B, int N, int C, int k, int dtype,
                         void* stream) {
  const int M = 1;
  COMMON_SHAPE_CHECKS("grafp_max_over_k_bwd");
  GRAFP_REQUIRE(grad_out && argmax && grad_h, GRAFP_EINVAL, "grafp_max_over_k_bwd: grad_out, argmax and grad_h must be non-null");
  { int rc = require_device_ptr("grafp_max_over_k_bwd", "grad_out", grad_out); if (rc) return rc; }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  return DISPATCH_DTYPE(launch_max_over_k_bwd<float>(grad_out, argmax, grad_h, B, N, C, k, s),
                        launch_max_over_k_bwd<__nv_bfloat16>(grad_out, argmax, grad_h, B, N, C, k, s));
}

}  // extern "C"

namespace grafp {
static int search_envelope(const char* fn, int n_q, int n_db, int d, int k) {
  GRAFP_REQUIRE(n_q > 0 && n_db > 0 && d > 0 && k > 0, GRAFP_EINVAL, "%s: n_q, n_db, d and k must be positive", fn);
  GRAFP_REQUIRE(d % 8 == 0 && d >= 64 && d <= 256, GRAFP_EUNSUPPORTED, "%s: d = %d is not a multiple of 8 in [64, 256]", fn, d);
  GRAFP_REQUIRE(k <= GRAFP_KNN_MAX_K, GRAFP_EUNSUPPORTED, "%s: k = %d exceeds %d", fn, k, GRAFP_KNN_MAX_K);
  GRAFP_REQUIRE(k <= n_db, GRAFP_EINVAL, "%s: k = %d exceeds the %d database rows", fn, k, n_db);
  return GRAFP_OK;
}
}  // namespace grafp

extern "C" {

int grafp_search_prepare(const float* rows, long long n, int d, void* hi, void* lo, float* sq, void* stream) {
  clear_error();
  GRAFP_REQUIRE(n > 0 && d > 0, GRAFP_EINVAL, "grafp_search_prepare: n and d must be positive");
  GRAFP_REQUIRE(d % 8 == 0 && d >= 64 && d <= 256, GRAFP_EUNSUPPORTED, "grafp_search_prepare: d = %d is not a multiple of 8 in [64, 256]", d);
  GRAFP_REQUIRE(rows && hi && lo && sq, GRAFP_EINVAL, "grafp_search_prepare: rows, hi, lo and sq must be non-null");
  { int rc = require_device("grafp_search_prepare"); if (rc != GRAFP_OK) return rc; }
  { int rc = require_device_ptr("grafp_search_prepare", "rows", rows); if (rc) return rc; }
  { int rc = require_device_ptr("grafp_search_prepare", "hi", hi); if (rc) return rc; }
  { int rc = require_device_ptr("grafp_search_prepare", "lo", lo); if (rc) return rc; }
  { int rc = require_device_ptr("grafp_search_prepare", "sq", sq); if (rc) return rc; }
  return launch_knn_normalize<float>(rows, static_cast<float*>(hi), static_cast<float*>(lo), sq, n, d, 3, false,
                                     static_cast<cudaStream_t>(stream));
}

size_t grafp_search_workspace_bytes(int n_q, int n_db, int d, int k) {
  if (search_envelope("grafp_search_workspace_bytes", n_q, n_db, d, k) != GRAFP_OK) return 0;
  return search_workspace_bytes(n_q, n_db, d, k);
}

int grafp_search_fwd(const float* q, int n_q, const void* hi, const void* lo, const float* sq, int n_db, int d, int k,
                     int64_t* ids, float* dist, void* workspace, size_t workspace_bytes, void* stream) {
  clear_error();
  { int rc = search_envelope("grafp_search_fwd", n_q, n_db, d, k); if (rc != GRAFP_OK) return rc; }
  GRAFP_REQUIRE(q && hi && lo && sq && ids && dist && workspace, GRAFP_EINVAL,
                "grafp_search_fwd: q, hi, lo, sq, ids, dist and workspace must be non-null");
  GRAFP_REQUIRE(aligned16(q) && aligned16(hi) && aligned16(lo) && aligned16(sq), GRAFP_EINVAL,
                "grafp_search_fwd: q, hi, lo and sq must be 16-byte aligned");
  { int rc = require_device("grafp_search_fwd"); if (rc != GRAFP_OK) return rc; }
  { int rc = require_device_ptr("grafp_search_fwd", "q", q); if (rc) return rc; }
  { int rc = require_device_ptr("grafp_search_fwd", "hi", hi); if (rc) return rc; }
  { int rc = require_device_ptr("grafp_search_fwd", "lo", lo); if (rc) return rc; }
  { int rc = require_device_ptr("grafp_search_fwd", "sq", sq); if (rc) return rc; }
  { int rc = require_device_ptr("grafp_search_fwd", "ids", ids); if (rc) return rc; }
  { int rc = require_device_ptr("grafp_search_fwd", "dist", dist); if (rc) return rc; }
  { int rc = require_device_ptr("grafp_search_fwd", "workspace", workspace); if (rc) return rc; }
  return launch_search(q, n_q, hi, lo, sq, n_db, d, k, reinterpret_cast<long long*>(ids), dist, workspace, workspace_bytes,
                       static_cast<cudaStream_t>(stream));
}

size_t grafp_bn_workspace_bytes(int C) { return C > 0 ? bn_workspace_bytes(C) : 0; }

int grafp_bn_train_fwd(const void* x, const void* residual, const float* weight, const float* bias, float* running_mean,
                       float* running_var, const float* conv_bias, long long* num_batches_tracked, void* out, float* save_mean,
                       float* save_invstd, long long R, int C, float eps, float momentum, int relu, int dtype, void* workspace,
                       size_t workspace_bytes, void* stream) {
  clear_error();
  GRAFP_REQUIRE(R > 1 && C > 0, GRAFP_EINVAL, "grafp_bn_train_fwd: needs at least two rows and C > 0");
  GRAFP_REQUIRE(dtype == GRAFP_F32 || dtype == GRAFP_BF16, GRAFP_EUNSUPPORTED, "grafp_bn_train_fwd: dtype %d not supported", dtype);
  GRAFP_REQUIRE(x && weight && bias && out && save_mean && save_invstd && workspace, GRAFP_EINVAL,
                "grafp_bn_train_fwd: x, weight, bias, out, save_mean, save_invstd and workspace must be non-null");
  GRAFP_REQUIRE(aligned16(x) && aligned16(out) && (residual == nullptr || aligned16(residual)),
                GRAFP_EINVAL, "grafp_bn_train_fwd: x, out and residual must be 16-byte aligned");
  GRAFP_REQUIRE(workspace_bytes >= bn_workspace_bytes(C), GRAFP_EWORKSPACE, "grafp_bn_train_fwd: workspace too small");
  { int rc = require_device("grafp_bn_train_fwd"); if (rc != GRAFP_OK) return rc; }
  { int rc = require_device_ptr("grafp_bn_train_fwd", "x", x); if (rc) return rc; }
  return launch_bn_train_fwd(x, residual, weight, bias, running_mean, running_var, conv_bias, num_batches_tracked, out, save_mean,
                             save_invstd, R, C, eps, momentum, relu, dtype, workspace, false, static_cast<cudaStream_t>(stream));
}

int grafp_bn_train_fwd_from_moments(const void* x, const void* residual, const float* weight, const float* bias,
                                    float* running_mean, float* running_var, const float* conv_bias,
                                    long long* num_batches_tracked, void* out, float* save_mean, float* save_invstd, long long R,
                                    int C, float eps, float momentum, int relu, int dtype, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  clear_error();
  GRAFP_REQUIRE(R > 1 && C > 0, GRAFP_EINVAL, "grafp_bn_train_fwd_from_moments: needs at least two rows and C > 0");
  GRAFP_REQUIRE(dtype == GRAFP_F32 || dtype == GRAFP_BF16, GRAFP_EUNSUPPORTED,
                "grafp_bn_train_fwd_from_moments: dtype %d not supported", dtype);
  GRAFP_REQUIRE(x && weight && bias && out && save_mean && save_invstd && workspace, GRAFP_EINVAL,
                "grafp_bn_train_fwd_from_moments: x, weight, bias, out, save_mean, save_invstd and workspace must be non-null");
  GRAFP_REQUIRE(aligned16(x) && aligned16(out) && (residual == nullptr || aligned16(residual)), GRAFP_EINVAL,
                "grafp_bn_train_fwd_from_moments: x, out and residual must be 16-byte aligned");
  GRAFP_REQUIRE(workspace_bytes >= bn_workspace_bytes(C), GRAFP_EWORKSPACE, "grafp_bn_train_fwd_from_moments: workspace too small");
  { int rc = require_device("grafp_bn_train_fwd_from_moments"); if (rc != GRAFP_OK) return rc; }
  { int rc = require_device_ptr("grafp_bn_train_fwd_from_moments", "x", x); if (rc) return rc; }
  return launch_bn_train_fwd(x, residual, weight, bias, running_mean, running_var, conv_bias, num_batches_tracked, out, save_mean,
                             save_invstd, R, C, eps, momentum, relu, dtype, workspace, true, static_cast<cudaStream_t>(stream));
}

int grafp_conv1x1_bn_stats_supported(long long R, int Cin, int Cout, int groups, int dtype) {
  return conv1x1_stats_supported(R, Cin, Cout, groups, dtype) ? 1 : 0;
}

int grafp_conv1x1_bn_stats_fwd(const void* x, const void* w, void* y, long long R, int Cin, int Cout, int groups, int dtype,
                               void* workspace, size_t workspace_bytes, void* stream) {
  clear_error();
  GRAFP_REQUIRE(R > 0 && Cin > 0 && Cout > 0 && groups > 0, GRAFP_EINVAL,
                "grafp_conv1x1_bn_stats_fwd: R, Cin, Cout and groups must be positive");
  GRAFP_REQUIRE(x && w && y && workspace, GRAFP_EINVAL, "grafp_conv1x1_bn_stats_fwd: x, w, y and workspace must be non-null");
  GRAFP_REQUIRE(workspace_bytes >= bn_workspace_bytes(Cout), GRAFP_EWORKSPACE,
                "grafp_conv1x1_bn_stats_fwd: workspace smaller than grafp_bn_workspace_bytes(Cout)");
  { int rc = require_device("grafp_conv1x1_bn_stats_fwd"); if (rc != GRAFP_OK) return rc; }
  { int rc = require_device_ptr("grafp_conv1x1_bn_stats_fwd", "x", x); if (rc) return rc; }
  return launch_conv1x1_stats(x, w, y, bn_workspace_sums(workspace), R, Cin, Cout, groups, dtype,
                              static_cast<cudaStream_t>(stream));
}

int grafp_bn_train_bwd(const void* dy, const void* x, const float* weight, const float* bias, const float* save_mean,
                       const float* save_invstd, void* dx, float* dweight, float* dbias, float* dx_colsum, long long R, int C,
                       int relu, int dtype, void* workspace, size_t workspace_bytes, void* stream) {
  clear_error();
  GRAFP_REQUIRE(R > 1 && C > 0, GRAFP_EINVAL, "grafp_bn_train_bwd: needs at least two rows and C > 0");
  GRAFP_REQUIRE(dtype == GRAFP_F32 || dtype == GRAFP_BF16, GRAFP_EUNSUPPORTED, "grafp_bn_train_bwd: dtype %d not supported", dtype);
  GRAFP_REQUIRE(dy && x && weight && bias && save_mean && save_invstd && dx && dweight && dbias && workspace, GRAFP_EINVAL,
                "grafp_bn_train_bwd: all pointers must be non-null");
  GRAFP_REQUIRE(aligned16(dy) && aligned16(x) && aligned16(dx), GRAFP_EINVAL,
                "grafp_bn_train_bwd: dy, x and dx must be 16-byte aligned");
  GRAFP_REQUIRE(workspace_bytes >= bn_workspace_bytes(C), GRAFP_EWORKSPACE, "grafp_bn_train_bwd: workspace too small");
  { int rc = require_device("grafp_bn_train_bwd"); if (rc != GRAFP_OK) return rc; }
  { int rc = require_device_ptr("grafp_bn_train_bwd", "dy", dy); if (rc) return rc; }
  return launch_bn_train_bwd(dy, x, weight, bias, save_mean, save_invstd, dx, dweight, dbias, dx_colsum, R, C, relu, dtype,
                             workspace, static_cast<cudaStream_t>(stream));
}

int grafp_ntxent_fwd(const float* z, float* lse, float* row_loss, float* loss, int n2, int d, float inv_tau, void* stream) {
  clear_error();
  GRAFP_REQUIRE(z && lse && row_loss && loss, GRAFP_EINVAL, "grafp_ntxent_fwd: z, lse, row_loss and loss must be non-null");
  GRAFP_REQUIRE(ntxent_supported(n2, d), GRAFP_EUNSUPPORTED, "grafp_ntxent_fwd: needs an even n2 >= 2 and d %% 4 == 0, d <= 256 (got %d, %d)", n2, d);
  GRAFP_REQUIRE(aligned16(z), GRAFP_EINVAL, "grafp_ntxent_fwd: z must be 16-byte aligned");
  { int rc = require_device("grafp_ntxent_fwd"); if (rc != GRAFP_OK) return rc; }
  { int rc = require_device_ptr("grafp_ntxent_fwd", "z", z); if (rc) return rc; }
  return launch_ntxent_fwd(z, lse, row_loss, loss, n2, d, inv_tau, 0, n2, static_cast<cudaStream_t>(stream));
}

int grafp_ntxent_bwd(const float* z, const float* lse, const float* grad_loss, float* dz, int n2, int d, float inv_tau,
                     void* stream) {
  clear_error();
  GRAFP_REQUIRE(z && lse && grad_loss && dz, GRAFP_EINVAL, "grafp_ntxent_bwd: z, lse, grad_loss and dz must be non-null");
  GRAFP_REQUIRE(ntxent_supported(n2, d), GRAFP_EUNSUPPORTED, "grafp_ntxent_bwd: needs an even n2 >= 2 and d %% 4 == 0, d <= 256 (got %d, %d)", n2, d);
  GRAFP_REQUIRE(aligned16(z) && aligned16(dz), GRAFP_EINVAL, "grafp_ntxent_bwd: z and dz must be 16-byte aligned");
  { int rc = require_device("grafp_ntxent_bwd"); if (rc != GRAFP_OK) return rc; }
  { int rc = require_device_ptr("grafp_ntxent_bwd", "z", z); if (rc) return rc; }
  return launch_ntxent_bwd(z, lse, grad_loss, dz, n2, d, inv_tau, 0, n2, 1.f, static_cast<cudaStream_t>(stream));
}

int grafp_ntxent_rows_fwd(const float* z, float* lse, float* row_loss, float* loss_part, int n2, int d, int row_lo, int row_hi,
                          float inv_tau, void* stream) {
  clear_error();
  GRAFP_REQUIRE(z && lse && row_loss && loss_part, GRAFP_EINVAL, "grafp_ntxent_rows_fwd: z, lse, row_loss and loss_part must be non-null");
  GRAFP_REQUIRE(ntxent_supported(n2, d), GRAFP_EUNSUPPORTED, "grafp_ntxent_rows_fwd: needs an even n2 >= 2 and d %% 4 == 0, d <= 256 (got %d, %d)", n2, d);
  GRAFP_REQUIRE(row_lo >= 0 && row_lo < row_hi && row_hi <= n2 && row_lo % 2 == 0 && row_hi % 2 == 0, GRAFP_EINVAL,
                "grafp_ntxent_rows_fwd: needs 0 <= row_lo < row_hi <= n2, both even (got %d, %d)", row_lo, row_hi);
  GRAFP_REQUIRE(aligned16(z), GRAFP_EINVAL, "grafp_ntxent_rows_fwd: z must be 16-byte aligned");
  { int rc = require_device("grafp_ntxent_rows_fwd"); if (rc != GRAFP_OK) return rc; }
  { int rc = require_device_ptr("grafp_ntxent_rows_fwd", "z", z); if (rc) return rc; }
  return launch_ntxent_fwd(z, lse, row_loss, loss_part, n2, d, inv_tau, row_lo, row_hi, static_cast<cudaStream_t>(stream));
}

int grafp_ntxent_rows_bwd(const float* z, const float* lse, const float* grad_loss, float* dz_rows, int n2, int d, int row_lo,
                          int row_hi, float inv_tau, float grad_scale, void* stream) {
  clear_error();
  GRAFP_REQUIRE(z && lse && grad_loss && dz_rows, GRAFP_EINVAL, "grafp_ntxent_rows_bwd: z, lse, grad_loss and dz_rows must be non-null");
  GRAFP_REQUIRE(ntxent_supported(n2, d), GRAFP_EUNSUPPORTED, "grafp_ntxent_rows_bwd: needs an even n2 >= 2 and d %% 4 == 0, d <= 256 (got %d, %d)", n2, d);
  GRAFP_REQUIRE(row_lo >= 0 && row_lo < row_hi && row_hi <= n2 && row_lo % 2 == 0 && row_hi % 2 == 0, GRAFP_EINVAL,
                "grafp_ntxent_rows_bwd: needs 0 <= row_lo < row_hi <= n2, both even (got %d, %d)", row_lo, row_hi);
  GRAFP_REQUIRE(aligned16(z) && aligned16(dz_rows), GRAFP_EINVAL, "grafp_ntxent_rows_bwd: z and dz_rows must be 16-byte aligned");
  { int rc = require_device("grafp_ntxent_rows_bwd"); if (rc != GRAFP_OK) return rc; }
  { int rc = require_device_ptr("grafp_ntxent_rows_bwd", "z", z); if (rc) return rc; }
  return launch_ntxent_bwd(z, lse, grad_loss, dz_rows, n2, d, inv_tau, row_lo, row_hi, grad_scale, static_cast<cudaStream_t>(stream));
}

int grafp_downsample_taps_fwd(const void* x, void* taps, int B, int N, int C, int dtype, void* stream) {
  clear_error();
  GRAFP_REQUIRE(x && taps && B > 0, GRAFP_EINVAL, "grafp_downsample_taps_fwd: x and taps must be non-null, B positive");
  GRAFP_REQUIRE(downsample_taps_supported(N, C, dtype), GRAFP_EUNSUPPORTED,
                "grafp_downsample_taps_fwd: needs an even N >= 2 and fp32 / bf16 rows of a multiple of 16 bytes (N=%d C=%d)", N, C);
  GRAFP_REQUIRE(aligned16(x) && aligned16(taps), GRAFP_EINVAL, "grafp_downsample_taps_fwd: x and taps must be 16-byte aligned");
  { int rc = require_device("grafp_downsample_taps_fwd"); if (rc != GRAFP_OK) return rc; }
  { int rc = require_device_ptr("grafp_downsample_taps_fwd", "x", x); if (rc) return rc; }
  return launch_downsample_taps_fwd(x, taps, B, N, C, dtype, static_cast<cudaStream_t>(stream));
}

int grafp_downsample_taps_bwd(const void* dtaps, void* dx, int B, int N, int C, int dtype, void* stream) {
  clear_error();
  GRAFP_REQUIRE(dtaps && dx && B > 0, GRAFP_EINVAL, "grafp_downsample_taps_bwd: dtaps and dx must be non-null, B positive");
  GRAFP_REQUIRE(downsample_taps_supported(N, C, dtype), GRAFP_EUNSUPPORTED,
                "grafp_downsample_taps_bwd: needs an even N >= 2 and fp32 / bf16 rows of a multiple of 16 bytes (N=%d C=%d)", N, C);
  GRAFP_REQUIRE(aligned16(dtaps) && aligned16(dx), GRAFP_EINVAL, "grafp_downsample_taps_bwd: dtaps and dx must be 16-byte aligned");
  { int rc = require_device("grafp_downsample_taps_bwd"); if (rc != GRAFP_OK) return rc; }
  { int rc = require_device_ptr("grafp_downsample_taps_bwd", "dtaps", dtaps); if (rc) return rc; }
  return launch_downsample_taps_bwd(dtaps, dx, B, N, C, dtype, static_cast<cudaStream_t>(stream));
}

size_t grafp_peak_extract_workspace_bytes(int B, int kh, int kw) {
  return (B > 0 && kh > 0 && kw > 0) ? peak_extract_workspace_bytes(B, kh, kw) : 0;
}

int grafp_peak_extract_fwd(const float* spec, const float* weight, const float* bias, float* out, int B, int H, int W, int F,
                           int kh, int kw, int stride_h, void* stream) {
  clear_error();
  GRAFP_REQUIRE(spec && weight && bias && out && B > 0, GRAFP_EINVAL, "grafp_peak_extract_fwd: spec, weight, bias, out must be non-null, B positive");
  GRAFP_REQUIRE(peak_extract_supported(H, W, F, kh, kw, stride_h), GRAFP_EUNSUPPORTED,
                "grafp_peak_extract_fwd: needs F == 8, odd kh / kw and planes that fit shared memory (H=%d W=%d F=%d kh=%d kw=%d)", H, W, F, kh, kw);
  GRAFP_REQUIRE(aligned16(out), GRAFP_EINVAL, "grafp_peak_extract_fwd: out must be 16-byte aligned");
  { int rc = require_device("grafp_peak_extract_fwd"); if (rc != GRAFP_OK) return rc; }
  { int rc = require_device_ptr("grafp_peak_extract_fwd", "spec", spec); if (rc) return rc; }
  return launch_peak_extract_fwd(spec, weight, bias, out, B, H, W, kh, kw, stride_h, static_cast<cudaStream_t>(stream));
}

int grafp_peak_extract_bwd(const float* spec, const float* out, const float* grad_out, void* partial, size_t partial_bytes,
                           float* dweight, float* dbias, int B, int H, int W, int F, int kh, int kw, int stride_h, void* stream) {
  clear_error();
  GRAFP_REQUIRE(spec && out && grad_out && partial && dweight && dbias && B > 0, GRAFP_EINVAL, "grafp_peak_extract_bwd: all pointers must be non-null, B positive");
  GRAFP_REQUIRE(peak_extract_supported(H, W, F, kh, kw, stride_h), GRAFP_EUNSUPPORTED, "grafp_peak_extract_bwd: unsupported shape");
  GRAFP_REQUIRE(partial_bytes >= peak_extract_workspace_bytes(B, kh, kw), GRAFP_EWORKSPACE, "grafp_peak_extract_bwd: workspace too small");
  GRAFP_REQUIRE(aligned16(out) && aligned16(grad_out) && aligned16(partial), GRAFP_EINVAL, "grafp_peak_extract_bwd: out, grad_out and partial must be 16-byte aligned");
  { int rc = require_device("grafp_peak_extract_bwd"); if (rc != GRAFP_OK) return rc; }
  { int rc = require_device_ptr("grafp_peak_extract_bwd", "spec", spec); if (rc) return rc; }
  return launch_peak_extract_bwd(spec, out, grad_out, static_cast<float*>(partial), dweight, dbias, B, H, W, kh, kw, stride_h,
                                 static_cast<cudaStream_t>(stream));
}

}  // extern "C"
