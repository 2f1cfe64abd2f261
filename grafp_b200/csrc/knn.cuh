// Internal declarations shared by the k-NN translation units.
#pragma once
#include "common.cuh"

namespace grafp {

__device__ __forceinline__ float to_float(float v) { return v; }
__device__ __forceinline__ float to_float(__nv_bfloat16 v) { return __bfloat162float(v); }

// mode 0: x_hat fp32 -> xhat;  1: tf32 hi -> xhat, lo -> lo;  2: bf16 x_hat -> xhat (as bf16);
// 3: fp16 planes of x_hat * 2^12: hi -> xhat, lo -> lo (both as __half)
template <typename T>
int launch_knn_normalize(const void* x, float* xhat, float* lo, float* sq, long long rows, int C, int mode,
                         bool normalize, cudaStream_t s);

int launch_fill_f32(float* p, long long n, float v, cudaStream_t s);

int launch_knn_simt(const float* xh, const float* xsq, const float* yh, const float* ysq, const float* relpos,
                    long long* nn_idx, int* nn_idx32, int B, int N, int M, int C, int K, int k_out, int stride,
                    cudaStream_t s);

// tensor-core path (knn_tc.cu).  Returns GRAFP_EUNSUPPORTED when the shape is outside its envelope.
bool knn_tc_supported(int N, int M, int C, int K, int dtype);
int launch_knn_tc(const void* xhi, const void* xlo, const float* xsq, const void* yhi, const void* ylo,
                  const float* ysq, const float* relpos, long long* nn_idx, int* nn_idx32, int B, int N, int M, int C,
                  int K, int k_out, int stride, int dtype, cudaStream_t s);

// second-generation tensor-core path (knn_tc2.cu): fp16 hi/lo planes, kind::f16, K <= 64 (K > 16 in rounds of 16
// ranks; `bounds` = B * N * 8 bytes of scratch for the hand-over between rounds).
// `self`: the keys are the queries (y == NULL).
bool knn_tc2_supported(int N, int M, int C, int K, int dtype, bool self);
int launch_knn_tc2(const void* xhi, const void* xlo, const float* xsq, const void* yhi, const void* ylo,
                   const float* ysq, long long* nn_idx, int* nn_idx32, int B, int N, int M, int C, int K, int k_out,
                   int stride, int dtype, bool self, void* bounds, cudaStream_t s);

// exact flat search (knn_tc2.cu): fp16 planes + |x|^2 of n_db database rows (launch_knn_normalize, mode 3, no
// normalisation), queries fp32 (n_q, d); ids / dist (n_q, k) ascending.  0 bytes: no plan for the shape.
size_t search_workspace_bytes(int n_q, int n_db, int d, int k);
int launch_search(const float* q, int n_q, const void* hi, const void* lo, const float* sq, int n_db, int d, int k,
                  long long* ids, float* dist, void* workspace, size_t workspace_bytes, cudaStream_t s);

}  // namespace grafp
