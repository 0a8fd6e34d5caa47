// R-level SSP of the eval pre-step (SURVEY.md 8 f2): SinkhornNet forward + optimal assignment, batched on the device.
//
// Reference: models/sinkhorn_network.py:30-51 (MLP over the 2352-d rows of a repeated role's slots -> tanh logits ->
// exp(x / tau) -> n_iters x column / row normalisation) and coco_scripts/eval_coco.py:184-189, where the reference
// moves every 10 x 10 matrix to the host (.cpu()) and runs munkres on it, once per (caption, verb, repeated role).
// Batches of problems run the four MLP layers as GEMMs over ALL rows of the batch (B x N rows) on the decoder path's
// tcgen05 f16x3 kernels — the weights are read once per batch instead of once per problem — with small kernels writing the
// operand twins in between (input split, ReLU, concatenation); then one CTA per problem does the N-output head, the Sinkhorn
// iterations on its N x N shared-memory tile and the Hungarian algorithm (O(N^3), one thread, double-precision potentials) on
// the transposed matrix, so nothing returns to the host but B x N column indices.  A few problems (or VSRDEC_GEMM=simt) take
// the one-CTA-per-problem kernel that runs the MLP itself with warp-per-output fp32 FFMA layers.
#include <math.h>

#include "common.cuh"
#include "twin_util.cuh"

namespace vsr {

namespace {

constexpr int SSP_THREADS = 256;
constexpr int SSP_MAXN = 16;
constexpr int D_TXT = 300, D_VIS = 2048, D_POS = 4, D_IN = D_TXT + D_VIS + D_POS;      // 2352 (eval_coco.py:146)
constexpr int H_TXT = 128, H_VIS1 = 512, H_VIS2 = 128, H_Z = H_TXT + H_VIS2 + D_POS, H_FC = 256;

struct SspWeights {
  const float *w1_txt, *b1_txt, *w1_vis, *b1_vis, *w2_vis, *b2_vis, *w_pos, *b_pos, *w_fc, *b_fc;
};

// out[r][o] = act(bias[o] + sum_k W[o][k] * in[r][k]) for r < N: one warp per output o, lanes stride k (coalesced rows of
// W), N accumulators per lane, one shuffle reduction per row.  ACT: 0 = relu, 1 = tanh.
template <int ACT>
__device__ __forceinline__ void layer(const float* __restrict__ W, const float* __restrict__ bias, int n_out, int K,
                                      const float* in, int ld_in, float* out, int ld_out, int N, int warp, int lane) {
  constexpr int NW = SSP_THREADS / 32;
  for (int o = warp; o < n_out; o += NW) {
    float acc[SSP_MAXN];
#pragma unroll
    for (int r = 0; r < SSP_MAXN; ++r) acc[r] = 0.f;
    const float* w = W + (size_t)o * K;
    for (int k = lane * 4; k < K; k += 128) {           // K % 4 == 0 for every layer; rows of `in` are 16-byte aligned
      const float4 wv = __ldg(reinterpret_cast<const float4*>(w + k));
#pragma unroll
      for (int r = 0; r < SSP_MAXN; ++r) {
        if (r < N) {
          const float4 xv = *reinterpret_cast<const float4*>(in + r * ld_in + k);
          acc[r] = fmaf(wv.x, xv.x, fmaf(wv.y, xv.y, fmaf(wv.z, xv.z, fmaf(wv.w, xv.w, acc[r]))));
        }
      }
    }
#pragma unroll
    for (int r = 0; r < SSP_MAXN; ++r) {
      if (r >= N) break;
      float v = acc[r];
#pragma unroll
      for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
      if (lane == 0) {
        v += bias[o];
        out[r * ld_out + o] = ACT == 0 ? fmaxf(v, 0.f) : tanhf(v);
      }
    }
  }
}

// Hungarian algorithm (potentials, O(n^3)) for the MAXIMUM-profit assignment of the n x n matrix prof[i][j]:
// col[i] = column assigned to row i.  Minimises cost = -profit; 1-based working arrays.
__device__ void hungarian_max(const float* prof, int ld, int n, int* col) {
  double u[SSP_MAXN + 1], v[SSP_MAXN + 1], minv[SSP_MAXN + 1];
  int p[SSP_MAXN + 1], way[SSP_MAXN + 1];
  bool used[SSP_MAXN + 1];
  for (int i = 0; i <= n; ++i) { u[i] = 0.0; v[i] = 0.0; p[i] = 0; way[i] = 0; }
  for (int i = 1; i <= n; ++i) {
    p[0] = i;
    int j0 = 0;
    for (int j = 0; j <= n; ++j) { minv[j] = 1e300; used[j] = false; }
    do {
      used[j0] = true;
      const int i0 = p[j0];
      double delta = 1e300;
      int j1 = 0;
      for (int j = 1; j <= n; ++j) {
        if (used[j]) continue;
        const double cur = -(double)prof[(i0 - 1) * ld + (j - 1)] - u[i0] - v[j];
        if (cur < minv[j]) { minv[j] = cur; way[j] = j0; }
        if (minv[j] < delta) { delta = minv[j]; j1 = j; }
      }
      for (int j = 0; j <= n; ++j) {
        if (used[j]) { u[p[j]] += delta; v[j] -= delta; } else { minv[j] -= delta; }
      }
      j0 = j1;
    } while (p[j0] != 0);
    do {
      const int j1 = way[j0];
      p[j0] = p[j1];
      j0 = j1;
    } while (j0 != 0);
  }
  for (int j = 1; j <= n; ++j) col[p[j] - 1] = j - 1;
}

// f_in == nullptr: the whole network for problem blockIdx.x from its input rows.  f_in != nullptr: the batched GEMM path has
// already produced the pre-activation of W_fc_pos for every row ([B*N][256]); only the head and the matrix work remain.
__global__ void __launch_bounds__(SSP_THREADS) k_sinkhorn(const SspWeights W, const float* __restrict__ seq, const float* __restrict__ f_in,
                                                          int N, int n_iters, float tau, float* __restrict__ matrix,
                                                          int32_t* __restrict__ assign) {
  extern __shared__ __align__(16) float sm[];
  const bool tail = f_in != nullptr;
  float* x = sm;                                   // [N][2352] input rows
  float* h1 = x + (tail ? 0 : N * D_IN);           // [N][512]
  float* z = h1 + (tail ? 0 : N * H_VIS1);         // [N][260] = [txt 128 | vis 128 | pos 4]
  float* f = z + (tail ? 0 : N * H_Z);             // [N][256]
  float* m = f + N * H_FC;                // [N][N] logits -> doubly stochastic matrix
  float* mt = m + N * N;                  // [N][N] its transpose (the profit matrix of eval_coco.py:187)
  __shared__ float s_sum[SSP_MAXN];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tail) {
    const float* src = f_in + (size_t)b * N * H_FC;
    for (int i = tid * 4; i < N * H_FC; i += SSP_THREADS * 4) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(src + i));
      *reinterpret_cast<float4*>(f + i) = make_float4(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f));   // relu  :47
    }
    __syncthreads();
  } else {
  const float* src = seq + (size_t)b * N * D_IN;
  for (int i = tid * 4; i < N * D_IN; i += SSP_THREADS * 4) *reinterpret_cast<float4*>(x + i) = __ldg(reinterpret_cast<const float4*>(src + i));
  __syncthreads();
  // x_txt = seq[..., :300], x_vis = seq[..., 300:2348], x_pos = seq[..., 2348:]     (sinkhorn_network.py:40-42)
  layer<0>(W.w1_txt, W.b1_txt, H_TXT, D_TXT, x, D_IN, z, H_Z, N, warp, lane);                      // relu(W1_txt x_txt)   :43
  layer<0>(W.w1_vis, W.b1_vis, H_VIS1, D_VIS, x + D_TXT, D_IN, h1, H_VIS1, N, warp, lane);         // relu(W1_vis x_vis)   :44
  for (int i = tid; i < N * D_POS; i += SSP_THREADS) z[(i / D_POS) * H_Z + H_TXT + H_VIS2 + (i % D_POS)] = x[(i / D_POS) * D_IN + D_TXT + D_VIS + (i % D_POS)];
  __syncthreads();
  layer<0>(W.w2_vis, W.b2_vis, H_VIS2, H_VIS1, h1, H_VIS1, z + H_TXT, H_Z, N, warp, lane);         // relu(W2_vis .)       :45
  __syncthreads();
  layer<0>(W.w_pos, W.b_pos, H_FC, H_Z, z, H_Z, f, H_FC, N, warp, lane);                           // relu(W_fc_pos cat)   :46-47
  __syncthreads();
  }
  layer<1>(W.w_fc, W.b_fc, N, H_FC, f, H_FC, m, N, N, warp, lane);                                 // tanh(W_fc .)         :49
  __syncthreads();
  // sinkhorn (:30-37): x = exp(x / tau); n_iters x { x /= (1e-7 + sum over rows) ; x /= (1e-7 + sum over columns) }
  const int i = tid / N, j = tid - i * N;
  const bool cell = tid < N * N;
  if (cell) m[tid] = expf(m[tid] / tau);
  __syncthreads();
  for (int it = 0; it < n_iters; ++it) {
    if (tid < N) { float s = 0.f; for (int r = 0; r < N; ++r) s += m[r * N + tid]; s_sum[tid] = s; }     // torch.sum(x, -2)
    __syncthreads();
    if (cell) m[tid] = m[tid] / (10e-8f + s_sum[j]);
    __syncthreads();
    if (tid < N) { float s = 0.f; for (int c = 0; c < N; ++c) s += m[tid * N + c]; s_sum[tid] = s; }     // torch.sum(x, -1)
    __syncthreads();
    if (cell) m[tid] = m[tid] / (10e-8f + s_sum[i]);
    __syncthreads();
  }
  if (cell) {
    matrix[(size_t)b * N * N + tid] = m[tid];
    mt[j * N + i] = m[tid];
  }
  __syncthreads();
  if (assign != nullptr && tid == 0) {
    int col[SSP_MAXN];
    hungarian_max(mt, N, N, col);
    for (int r = 0; r < N; ++r) assign[(size_t)b * N + r] = col[r];
  }
}

// dynamic shared memory of the one-CTA kernel that runs the whole network: input rows, hidden layers and the two N x N tiles
size_t ssp_smem_full(int N) { return sizeof(float) * ((size_t)N * (D_IN + H_VIS1 + H_Z + H_FC) + 2 * (size_t)N * N); }

constexpr int K_TXT = 320, K_Z = 320;      // K of the text layer (300) and of W_fc_pos (260) padded to whole 64-element k-blocks

// input rows -> operand twins of the two first-layer GEMMs: txt = columns [0, 300) (the pad columns stay zero), vis = [300, 2348)
__global__ void k_ssp_split(const float* __restrict__ seq, int rows, const TwinOut txt, const TwinOut vis) {
  const int r = blockIdx.x;
  const float4* src = reinterpret_cast<const float4*>(seq + (size_t)r * D_IN);
  for (int c4 = threadIdx.x; c4 < (D_TXT + D_VIS) / 4; c4 += blockDim.x) {
    const float4 v = __ldg(src + c4);
    if (c4 < D_TXT / 4) store_twin4(txt, (size_t)r * K_TXT + 4 * c4, v);
    else store_twin4(vis, (size_t)r * D_VIS + 4 * c4 - D_TXT, v);
  }
}
// z = [relu(txt branch) 128 | relu(vis branch) 128 | pos 4] -> operand twins of the W_fc_pos GEMM (pad columns stay zero)
__global__ void k_ssp_cat(const float* __restrict__ t1, const float* __restrict__ v2, const float* __restrict__ seq, int rows,
                          const TwinOut z) {
  const int r = blockIdx.x, c = threadIdx.x;      // 260 live columns, blockDim = 288
  if (c >= H_Z) return;
  float v;
  if (c < H_TXT) v = fmaxf(t1[(size_t)r * H_TXT + c], 0.f);
  else if (c < H_TXT + H_VIS2) v = fmaxf(v2[(size_t)r * H_VIS2 + c - H_TXT], 0.f);
  else v = seq[(size_t)r * D_IN + D_TXT + D_VIS + (c - H_TXT - H_VIS2)];
  put_twin(z, (size_t)r * K_Z + c, v);
}

struct SspCtx {
  int device, N, n_iters;
  float tau;
  float* w[10];
  size_t n[10];
  bool attr_set = false;
  size_t smem_cap = 0;      // dynamic shared memory k_sinkhorn may use on this device (opt-in maximum less its static part)
  // batched GEMM path: padded fp32 copies of the two weights whose K is not a whole number of k-blocks, operand twins of the
  // four MLP weights, and a workspace for cap_rows input rows
  bool use_tc = true;
  float *wpad_txt = nullptr, *wpad_pos = nullptr;
  F16Pair w_txt_p, w_vis1_p, w_vis2_p, w_pos_p;
  int cap_rows = 0;
  F16Pair txt_b, vis_b, h1_b, z_b;
  float *t1 = nullptr, *h1 = nullptr, *v2 = nullptr, *f = nullptr;
};

int ssp_split_weights(SspCtx* c, cudaStream_t st) {
  if (!c->use_tc) return VSR_OK;
  if (c->w_vis1_p.hi == nullptr) {
    VSR_CHECK_CUDA(cudaMalloc((void**)&c->wpad_txt, sizeof(float) * H_TXT * K_TXT));
    VSR_CHECK_CUDA(cudaMalloc((void**)&c->wpad_pos, sizeof(float) * H_FC * K_Z));
    VSR_CHECK_CUDA(cudaMemset(c->wpad_txt, 0, sizeof(float) * H_TXT * K_TXT));
    VSR_CHECK_CUDA(cudaMemset(c->wpad_pos, 0, sizeof(float) * H_FC * K_Z));
    VSR_TRY(make_pair(&c->w_txt_p, H_TXT, K_TXT, true)); VSR_TRY(make_pair(&c->w_vis1_p, H_VIS1, D_VIS, true));
    VSR_TRY(make_pair(&c->w_vis2_p, H_VIS2, H_VIS1, true)); VSR_TRY(make_pair(&c->w_pos_p, H_FC, K_Z, true));
  }
  VSR_CHECK_CUDA(cudaMemcpy2DAsync(c->wpad_txt, sizeof(float) * K_TXT, c->w[0], sizeof(float) * D_TXT, sizeof(float) * D_TXT, H_TXT,
                                   cudaMemcpyDeviceToDevice, st));
  VSR_CHECK_CUDA(cudaMemcpy2DAsync(c->wpad_pos, sizeof(float) * K_Z, c->w[6], sizeof(float) * H_Z, sizeof(float) * H_Z, H_FC,
                                   cudaMemcpyDeviceToDevice, st));
  VSR_TRY(launch_split_pair(c->wpad_txt, c->w_txt_p, (size_t)H_TXT * K_TXT, st, true));
  VSR_TRY(launch_split_pair(c->w[2], c->w_vis1_p, (size_t)H_VIS1 * D_VIS, st, true));
  VSR_TRY(launch_split_pair(c->w[4], c->w_vis2_p, (size_t)H_VIS2 * H_VIS1, st, true));
  VSR_TRY(launch_split_pair(c->wpad_pos, c->w_pos_p, (size_t)H_FC * K_Z, st, true));
  return VSR_OK;
}

int ssp_ensure_rows(SspCtx* c, int rows) {
  if (rows <= c->cap_rows) return VSR_OK;
  if (c->cap_rows > 0) { VSR_CHECK_CUDA(cudaDeviceSynchronize()); cudaFree(c->t1); c->t1 = nullptr; c->cap_rows = 0; }
  const int rp = (rows + 127) / 128 * 128;
  VSR_TRY(make_pair(&c->txt_b, rp, K_TXT, false)); VSR_TRY(make_pair(&c->vis_b, rp, D_VIS, false));
  VSR_TRY(make_pair(&c->h1_b, rp, H_VIS1, false)); VSR_TRY(make_pair(&c->z_b, rp, K_Z, false));
  VSR_CHECK_CUDA(cudaMalloc((void**)&c->t1, sizeof(float) * (size_t)rp * (H_TXT + H_VIS1 + H_VIS2 + H_FC)));
  c->h1 = c->t1 + (size_t)rp * H_TXT; c->v2 = c->h1 + (size_t)rp * H_VIS1; c->f = c->v2 + (size_t)rp * H_VIS2;
  c->cap_rows = rp;
  return VSR_OK;
}

// out = a . w^T + bias on the tcgen05 f16x3 kernels
int ssp_lin(const F16Pair* a_b, int K, const F16Pair* w_b, const float* bias, float* out, int M, int N, cudaStream_t st) {
  GemmArgs g{};
  g.nseg = 1; g.seg[0] = {nullptr, K, K, K, a_b};
  g.ldw = K; g.bias = bias; g.wb = w_b;
  g.c = out; g.ldc = N; g.M = M; g.N = N;
  return launch_gemm_tc(g, nullptr, st);
}

}  // namespace
}  // namespace vsr

using vsr::SspCtx;

extern "C" {

static const size_t kSspShape[10] = {(size_t)vsr::H_TXT * vsr::D_TXT, vsr::H_TXT, (size_t)vsr::H_VIS1 * vsr::D_VIS, vsr::H_VIS1,
                                     (size_t)vsr::H_VIS2 * vsr::H_VIS1, vsr::H_VIS2, (size_t)vsr::H_FC * vsr::H_Z, vsr::H_FC, 0, 0};

int vsr_ssp_load_weights(vsr_ssp_handle h, const float* const* weights, void* stream) {
  if (!h || !weights) { vsr::set_error("vsr_ssp_load_weights: null argument"); return VSR_EINVAL; }
  SspCtx* c = (SspCtx*)h;
  for (int i = 0; i < 10; ++i)
    VSR_CHECK_CUDA(cudaMemcpyAsync(c->w[i], weights[i], c->n[i] * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return vsr::ssp_split_weights(c, (cudaStream_t)stream);
}

int vsr_ssp_create(const float* const* weights, int32_t N, int32_t n_iters, float tau, vsr_ssp_handle* out) {
  if (!out || !weights) { vsr::set_error("vsr_ssp_create: null argument"); return VSR_EINVAL; }
  *out = nullptr;
  VSR_REQUIRE(N >= 1 && N <= vsr::SSP_MAXN && N * N <= vsr::SSP_THREADS, VSR_EINVAL, "vsr_ssp_create: N=%d not in [1,%d]", N, vsr::SSP_MAXN);
  VSR_REQUIRE(n_iters >= 0 && tau > 0.f, VSR_EINVAL, "vsr_ssp_create: bad n_iters / tau");
  int ndev = 0;
  VSR_REQUIRE(cudaGetDeviceCount(&ndev) == cudaSuccess && ndev > 0, VSR_ECUDA, "vsr_ssp_create: no CUDA device (no CPU fallback)");
  // the one-CTA kernel serves a few problems and VSRDEC_GEMM=simt: every N accepted here must fit its shared memory
  int dev = 0, optin = 0;
  cudaFuncAttributes fa{};
  VSR_CHECK_CUDA(cudaGetDevice(&dev));
  VSR_CHECK_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  VSR_CHECK_CUDA(cudaFuncGetAttributes(&fa, vsr::k_sinkhorn));
  const size_t smem_cap = (size_t)optin - fa.sharedSizeBytes;
  VSR_REQUIRE(vsr::ssp_smem_full(N) <= smem_cap, VSR_EINVAL, "vsr_ssp_create: N=%d needs %zu B of shared memory, the device allows %zu",
              N, vsr::ssp_smem_full(N), smem_cap);
  SspCtx* c = new SspCtx();
  c->N = N; c->n_iters = n_iters; c->tau = tau;
  c->device = dev; c->smem_cap = smem_cap;
  if (const char* e = getenv("VSRDEC_GEMM")) c->use_tc = strcmp(e, "simt") != 0;
  for (int i = 0; i < 10; ++i) {
    c->n[i] = i == 8 ? (size_t)N * vsr::H_FC : i == 9 ? (size_t)N : kSspShape[i];
    c->w[i] = nullptr;
  }
  for (int i = 0; i < 10; ++i) {
    if (cudaMalloc((void**)&c->w[i], c->n[i] * sizeof(float)) != cudaSuccess) {
      vsr::set_error("vsr_ssp_create: cudaMalloc failed");
      for (int j = 0; j < i; ++j) cudaFree(c->w[j]);
      delete c;
      return VSR_ENOMEM;
    }
  }
  const int r = vsr_ssp_load_weights((vsr_ssp_handle)c, weights, nullptr);
  if (r != VSR_OK) { for (int i = 0; i < 10; ++i) cudaFree(c->w[i]); delete c; return r; }
  VSR_CHECK_CUDA(cudaStreamSynchronize(nullptr));
  *out = (vsr_ssp_handle)c;
  return VSR_OK;
}

void vsr_ssp_destroy(vsr_ssp_handle h) {
  if (!h) return;
  SspCtx* c = (SspCtx*)h;
  cudaDeviceSynchronize();
  for (int i = 0; i < 10; ++i) cudaFree(c->w[i]);
  if (c->wpad_txt) cudaFree(c->wpad_txt);
  if (c->wpad_pos) cudaFree(c->wpad_pos);
  if (c->t1) cudaFree(c->t1);
  for (vsr::F16Pair* b : {&c->w_txt_p, &c->w_vis1_p, &c->w_vis2_p, &c->w_pos_p, &c->txt_b, &c->vis_b, &c->h1_b, &c->z_b}) vsr::free_pair(b);
  delete c;
}

int vsr_ssp_forward(vsr_ssp_handle h, const float* seq, int32_t B, float* matrix, int32_t* assign, void* stream) {
  if (!h) { vsr::set_error("vsr_ssp_forward: null handle"); return VSR_EINVAL; }
  SspCtx* c = (SspCtx*)h;
  VSR_REQUIRE(seq != nullptr && matrix != nullptr && B >= 0, VSR_EINVAL, "vsr_ssp_forward: null argument");
  VSR_REQUIRE(((uintptr_t)seq % 16) == 0, VSR_EINVAL, "vsr_ssp_forward: seq must be 16-byte aligned");
  if (B == 0) return VSR_OK;
  int prev = -1;
  cudaGetDevice(&prev);
  if (prev != c->device) cudaSetDevice(c->device);
  const int N = c->N;
  if (!c->attr_set) {
    VSR_CHECK_CUDA(cudaFuncSetAttribute(vsr::k_sinkhorn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_cap));
    c->attr_set = true;
  }
  vsr::SspWeights W{c->w[0], c->w[1], c->w[2], c->w[3], c->w[4], c->w[5], c->w[6], c->w[7], c->w[8], c->w[9]};
  cudaStream_t st = (cudaStream_t)stream;
  if (c->use_tc && B >= 8) {
    // the four MLP layers over all B * N rows at once (weights read once per batch), then one CTA per problem for the head
    using namespace vsr;
    const int R = B * N;
    int rc = ssp_ensure_rows(c, R);
    if (rc == VSR_OK) {
      k_ssp_split<<<R, 256, 0, st>>>(seq, R, twin_out(&c->txt_b), twin_out(&c->vis_b));
      rc = ssp_lin(&c->txt_b, K_TXT, &c->w_txt_p, c->w[1], c->t1, R, H_TXT, st);                        // W1_txt           :43
    }
    if (rc == VSR_OK) rc = ssp_lin(&c->vis_b, D_VIS, &c->w_vis1_p, c->w[3], c->h1, R, H_VIS1, st);    // W1_vis           :44
    if (rc == VSR_OK) {
      const size_t n4 = (size_t)R * H_VIS1 / 4;
      k_relu_twin<<<(unsigned)((n4 + 255) / 256), 256, 0, st>>>(c->h1, n4, twin_out(&c->h1_b));
      rc = ssp_lin(&c->h1_b, H_VIS1, &c->w_vis2_p, c->w[5], c->v2, R, H_VIS2, st);                     // W2_vis           :45
    }
    if (rc == VSR_OK) {
      k_ssp_cat<<<R, 288, 0, st>>>(c->t1, c->v2, seq, R, twin_out(&c->z_b));                           // relu, cat        :43-46
      rc = ssp_lin(&c->z_b, K_Z, &c->w_pos_p, c->w[7], c->f, R, H_FC, st);                             // W_fc_pos         :47
    }
    if (rc != VSR_OK) { if (prev != c->device && prev >= 0) cudaSetDevice(prev); return rc; }
    const size_t smem_tail = sizeof(float) * ((size_t)N * H_FC + 2 * (size_t)N * N);
    k_sinkhorn<<<B, SSP_THREADS, smem_tail, st>>>(W, seq, c->f, N, c->n_iters, c->tau, matrix, assign);
  } else {
    const size_t smem = vsr::ssp_smem_full(N);
    VSR_REQUIRE(smem <= c->smem_cap, VSR_EINVAL, "vsr_ssp_forward: N=%d rows do not fit shared memory", N);
    vsr::k_sinkhorn<<<B, vsr::SSP_THREADS, smem, st>>>(W, seq, nullptr, N, c->n_iters, c->tau, matrix, assign);
  }
  const cudaError_t e = cudaGetLastError();
  if (prev != c->device && prev >= 0) cudaSetDevice(prev);
  VSR_CHECK_CUDA(e);
  return VSR_OK;
}

}  // extern "C"
