// Operand twins (fp16 value + fp16 residual, the f16x3 form of gemm_tc.cu) for callers outside the decoder's Ctx: the two
// networks of the eval pre-step (sort.cu, ssp.cu) allocate their own pairs and let their pointwise kernels write them.
// Everything here is per translation unit (anonymous namespace).
#pragma once
#include "common.cuh"

namespace vsr {
namespace {

// fp16 value + fp16 residual of one activation element (the f16x3 operand form of gemm_tc.cu)
__device__ __forceinline__ void put_twin(const TwinOut& o, size_t off, float v) {
  if (o.hi == nullptr) return;
  v = fminf(fmaxf(v, -65504.f), 65504.f);
  const __half h = __float2half_rn(v);
  reinterpret_cast<__half*>(o.hi)[off] = h;
  reinterpret_cast<__half*>(o.lo)[off] = __float2half_rn(v - __half2float(h));
}

// operand twins of max(0, x): the feed-forward activation between its two tensor-core projections
__global__ void k_relu_twin(const float* __restrict__ x, size_t n4, const TwinOut tw) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  const float4 v = reinterpret_cast<const float4*>(x)[i];
  store_twin4(tw, i * 4, make_float4(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f)));
}

void free_pair(F16Pair* b, bool view = false) {
  if (!view) { if (b->hi) cudaFree(b->hi); if (b->lo) cudaFree(b->lo); if (b->scale) cudaFree(b->scale); }
  b->hi = b->lo = nullptr; b->scale = nullptr;
}

// fp16 value / residual arrays + tensor maps of a [rows][ld] operand (rows a multiple of 128); weights also get their scale pair
int make_pair(F16Pair* b, int rows, int ld, bool weight) {
  free_pair(b);
  VSR_CHECK_CUDA(cudaMalloc(&b->hi, (size_t)rows * ld * 2));
  VSR_CHECK_CUDA(cudaMalloc(&b->lo, (size_t)rows * ld * 2));
  VSR_CHECK_CUDA(cudaMemset(b->hi, 0, (size_t)rows * ld * 2));
  VSR_CHECK_CUDA(cudaMemset(b->lo, 0, (size_t)rows * ld * 2));
  if (weight) VSR_CHECK_CUDA(cudaMalloc((void**)&b->scale, 2 * sizeof(float)));
  b->rows = rows; b->ld = ld; b->box_rows = 128; b->n_valid = rows; b->act_scale = 1.f; b->alt_bn = 0; b->pair_rows = 0;
  VSR_TRY(make_tmap_f16(b->map_hi, b->hi, rows, ld, ld, 128));
  VSR_TRY(make_tmap_f16(b->map_lo, b->lo, rows, ld, ld, 128));
  return VSR_OK;
}

// rows [r0, r0 + rows) of a weight pair as a pair of its own (same arrays, same scale)
int make_view(F16Pair* v, const F16Pair& of, int r0, int rows) {
  *v = of;
  v->hi = reinterpret_cast<__half*>(of.hi) + (size_t)r0 * of.ld;
  v->lo = reinterpret_cast<__half*>(of.lo) + (size_t)r0 * of.ld;
  v->rows = rows; v->n_valid = rows;
  VSR_TRY(make_tmap_f16(v->map_hi, v->hi, rows, of.ld, of.ld, 128));
  VSR_TRY(make_tmap_f16(v->map_lo, v->lo, rows, of.ld, of.ld, 128));
  return VSR_OK;
}

}  // namespace
}  // namespace vsr
