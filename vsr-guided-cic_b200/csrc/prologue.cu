// Weight packing and the once-per-batch prologue (time-invariant terms of step()/step_v()).
//
// Hoisted out of the per-step path (SURVEY.md Appendix A):
//   img[b]   = sum_d det[b,d,:] / #{d : sum_f det[b,d,f] != 0}   controllable_captioning.py:126-128, 203-205
//   valid    = (sum_f x != 0) for every slot row                  :159, :240
//   P[b,l,r] = att_va.weight . det_seqs[b,l,r,:]                   :161, :242
//   U[b]     = S1[:, img cols] . img[b] + stacked biases           :151-152, :181 (img part of input_1)
//   U2[b]    = lstm_cell_2.weight_ih[:, img cols] . img[b]         :174 (img_second_lstm only)
#include <cuda_fp16.h>

#include "common.cuh"

namespace vsr {

namespace {

// the prologue's activation twins (slot rows, image descriptors): fp16 hi + fp16 residual, row stride ld
struct PairOut { TwinOut tw; int ld; __device__ __host__ bool on() const { return tw.hi != nullptr; } };
__device__ __forceinline__ void store_pair4(const PairOut& o, size_t i, const float4& v) { store_twin4(o.tw, i, v); }

// dst[r0+r][c0+c] = src[r][sc0+c]
__global__ void k_pack_block(float* __restrict__ dst, int ld_dst, int r0, int c0,
                             const float* __restrict__ src, int ld_src, int sc0, int rows, int cols) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int r = blockIdx.y;
  if (c < cols && r < rows) dst[(size_t)(r0 + r) * ld_dst + c0 + c] = src[(size_t)r * ld_src + sc0 + c];
}

// gate-interleaved variants: source row/element r (a hidden unit) goes to row/element cell_col(gate, r, ng)
__global__ void k_pack_block_perm(float* __restrict__ dst, int ld_dst, int r0, int c0,
                                  const float* __restrict__ src, int ld_src, int sc0, int rows, int cols,
                                  int gate, int ng) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int r = blockIdx.y;
  if (c < cols && r < rows)
    dst[(size_t)(r0 + cell_col(gate, r, ng)) * ld_dst + c0 + c] = src[(size_t)r * ld_src + sc0 + c];
}
__global__ void k_pack_bias_perm(float* __restrict__ dst, const float* __restrict__ a,
                                 const float* __restrict__ b, int n, int gate, int ng) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[cell_col(gate, i, ng)] = a[i] + (b != nullptr ? b[i] : 0.f);
}

// dst[o0+i] = a[i] (+ b[i])
__global__ void k_pack_bias(float* __restrict__ dst, int o0, const float* __restrict__ a,
                            const float* __restrict__ b, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[o0 + i] = a[i] + (b != nullptr ? b[i] : 0.f);
}

// The kernels that read caller features are templates on their element type T (float, __half, __nv_bfloat16):
// each value is widened to fp32 as it is loaded (ldg_feat4), after which the arithmetic is T-independent.

// one warp per row: flag[row] = (sum_f x[row][f] != 0).  Row r of image/caption g lives at
// base + g*group_stride + (r % rows_per_group)*F.
// Optionally also writes the row's fp16 hi/lo split (operand of the tcgen05 att_va projection).
template <typename T>
__global__ void k_row_valid(const T* __restrict__ x, int64_t group_stride, int rows_per_group,
                            int total_rows, int F, uint8_t* __restrict__ flag, PairOut split) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= total_rows) return;
  const T* p = x + (size_t)(row / rows_per_group) * group_stride + (size_t)(row % rows_per_group) * F;
  float s = 0.f;
  for (int f = lane * 4; f < F; f += 128) {
    const float4 v = ldg_feat4(p + f);
    s += (v.x + v.y) + (v.z + v.w);
    if (split.on()) store_pair4(split, (size_t)row * split.ld + f, v);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) flag[row] = (s != 0.f) ? 1 : 0;
}

// one 64-bit validity mask per slot tile (R <= 64 regions)
__global__ void k_slot_masks(const uint8_t* __restrict__ valid, int R, int n_slots, unsigned long long* __restrict__ mask) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_slots) return;
  unsigned long long m = 0;
  for (int r = 0; r < R; ++r) if (valid[(size_t)s * R + r]) m |= 1ull << r;
  mask[s] = m;
}

// Compaction of the valid slot rows (tensor-core path): exclusive scan of the slots' valid-row counts -> first P row
// of every slot, and the in-use flags of the compact rows.  One block; n_slots is ~1000.
__global__ void __launch_bounds__(1024) k_slot_scan(const unsigned long long* __restrict__ mask, int n_slots,
                                                    int32_t* __restrict__ slot_base, uint8_t* __restrict__ comp_valid,
                                                    int comp_rows) {
  __shared__ int s_part[1024];
  __shared__ int s_total;
  const int tid = threadIdx.x;
  const int per = (n_slots + 1023) / 1024;
  const int lo = tid * per, hi = min(lo + per, n_slots);
  int cnt = 0;
  for (int s = lo; s < hi; ++s) cnt += __popcll(mask[s]);
  s_part[tid] = cnt;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {       // Hillis-Steele inclusive scan
    const int v = tid >= off ? s_part[tid - off] : 0;
    __syncthreads();
    s_part[tid] += v;
    __syncthreads();
  }
  int base = s_part[tid] - cnt;
  for (int s = lo; s < hi; ++s) { slot_base[s] = base; base += __popcll(mask[s]); }
  if (tid == 1023) s_total = s_part[1023];
  __syncthreads();
  const int total = s_total;
  for (int i = tid; i < comp_rows; i += 1024) comp_valid[i] = i < total ? 1 : 0;
}

// one warp per source row: valid rows are split to fp16 hi/lo at their compact position
template <typename T>
__global__ void k_split_compact(const T* __restrict__ x, int R, int total_rows, int F,
                                const unsigned long long* __restrict__ mask, const int32_t* __restrict__ slot_base,
                                PairOut split) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= total_rows) return;
  const int s = row / R, r = row - s * R;
  const unsigned long long m = mask[s];
  if (!((m >> r) & 1ull)) return;
  const int dst = slot_base[s] + __popcll(m & ((1ull << r) - 1ull));
  const T* p = x + (size_t)row * F;
  for (int f = lane * 4; f < F; f += 128)
    store_pair4(split, (size_t)dst * split.ld + f, ldg_feat4(p + f));
}

// index form: validity mask of a slot from its detection indices (-2 = image mean row, valid iff the image
// has any valid detection; -1 = padding)
__global__ void k_slot_masks_indexed(const int32_t* __restrict__ slot_index, const uint8_t* __restrict__ det_valid,
                                     int R, int L, int D, int n_slots, int img_mul, unsigned long long* __restrict__ mask) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_slots) return;
  const int img = (s / L) * img_mul;
  int any = 0;
  for (int d = 0; d < D; ++d) any |= det_valid[img * D + d];
  unsigned long long m = 0;
  for (int r = 0; r < R; ++r) {
    const int idx = slot_index[(size_t)s * R + r];
    const bool v = idx >= 0 ? (idx < D && det_valid[img * D + idx]) : (idx == -2 && any);
    if (v) m |= 1ull << r;
  }
  mask[s] = m;
}

// img[g][f] = sum_d det[g][d][f] / count(valid rows of g).  Block (128, POOL_Y): thread (x, y) sums the rows
// d = y, y + POOL_Y, ... of float4 column x; the POOL_Y partial sums are combined in a fixed order (deterministic).
constexpr int POOL_Y = 4;
template <typename T>
__global__ void __launch_bounds__(128 * POOL_Y) k_pool(const T* __restrict__ det, int64_t img_stride, int D, int F,
                       const uint8_t* __restrict__ valid, float* __restrict__ img, int ld_img, PairOut split) {
  __shared__ float4 s_part[POOL_Y][128];
  __shared__ int s_cnt;
  const int g = blockIdx.y;
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int f = (blockIdx.x * 128 + tx) * 4;
  if (tx == 0 && ty == 0) s_cnt = 0;
  __syncthreads();
  {   // valid-row count of the image
    int c = 0;
    for (int d = ty * 128 + tx; d < D; d += 128 * POOL_Y) c += valid[g * D + d];
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((tx & 31) == 0 && c != 0) atomicAdd(&s_cnt, c);
  }
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  if (f < F) {
    const T* p = det + (size_t)g * img_stride + f;
    for (int d0 = ty; d0 < D; d0 += 8 * POOL_Y) {     // 8 independent row loads in flight
      float4 v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int d = d0 + u * POOL_Y;
        v[u] = d < D ? ldg_feat4(p + (size_t)d * F) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) { s.x += v[u].x; s.y += v[u].y; s.z += v[u].z; s.w += v[u].w; }
    }
  }
  s_part[ty][tx] = s;
  __syncthreads();
  if (ty != 0 || f >= F) return;
#pragma unroll
  for (int y = 1; y < POOL_Y; ++y) { const float4 q = s_part[y][tx]; s.x += q.x; s.y += q.y; s.z += q.z; s.w += q.w; }
  const float n = (float)s_cnt;
  const float4 o = make_float4(s.x / n, s.y / n, s.z / n, s.w / n);
  *reinterpret_cast<float4*>(img + (size_t)g * ld_img + f) = o;
  if (split.on()) store_pair4(split, (size_t)g * split.ld + f, o);
}

}  // namespace

static int pack_block(Ctx* c, float* dst, int ld_dst, int r0, int c0, const float* src, int ld_src,
                      int sc0, int rows, int cols, cudaStream_t st) {
  if (rows == 0 || cols == 0) return VSR_OK;
  dim3 grid((cols + 255) / 256, rows);
  k_pack_block<<<grid, 256, 0, st>>>(dst, ld_dst, r0, c0, src, ld_src, sc0, rows, cols);
  VSR_CHECK_CUDA(cudaGetLastError());
  c->launches++;
  return VSR_OK;
}
static int pack_bias(Ctx* c, float* dst, int o0, const float* a, const float* b, int n, cudaStream_t st) {
  k_pack_bias<<<(n + 255) / 256, 256, 0, st>>>(dst, o0, a, b, n);
  VSR_CHECK_CUDA(cudaGetLastError());
  c->launches++;
  return VSR_OK;
}

static int pack_perm(Ctx* c, float* dst, int ld_dst, int r0, int c0, const float* src, int ld_src, int sc0,
                     int units, int cols, int gate, int ng, cudaStream_t st) {
  if (units == 0 || cols == 0) return VSR_OK;
  dim3 grid((cols + 255) / 256, units);
  k_pack_block_perm<<<grid, 256, 0, st>>>(dst, ld_dst, r0, c0, src, ld_src, sc0, units, cols, gate, ng);
  VSR_CHECK_CUDA(cudaGetLastError());
  c->launches++;
  return VSR_OK;
}
static int pack_bias_perm(Ctx* c, float* dst, const float* a, const float* b, int n, int gate, int ng, cudaStream_t st) {
  k_pack_bias_perm<<<(n + 255) / 256, 256, 0, st>>>(dst, a, b, n, gate, ng);
  VSR_CHECK_CUDA(cudaGetLastError());
  c->launches++;
  return VSR_OK;
}

// Build the stacked, K-padded weight blocks S1..S7 of SURVEY.md Appendix A from the 28
// state_dict tensors (order documented in include/vsrdec.h).
int pack_weights(Ctx* c, const float* const* w, cudaStream_t st) {
  const int H = c->H, E = c->E, F = c->F, A = c->A, V = c->V;
  const int Hp = c->Hp, Ep = c->Ep;
  const bool h2f = c->d.h2_first_lstm != 0, img2 = c->d.img_second_lstm != 0;
  const int in1 = (h2f ? H : 0) + F + E;
  const int in2 = H + F + (img2 ? F : 0);
  const int c_img = h2f ? H : 0;        // column of the img block inside input_1
  const int c_xt = c_img + F;           // column of the xt block
  // column offsets inside WA's K axis
  const int ka_h2 = 0, ka_h1 = h2f ? Hp : 0;

  // all packed buffers were zero-filled at allocation; re-zero for repacks
  VSR_CHECK_CUDA(cudaMemsetAsync(c->WA, 0, sizeof(float) * (size_t)c->NA * c->KA, st));
  VSR_CHECK_CUDA(cudaMemsetAsync(c->WAx, 0, sizeof(float) * (size_t)c->NA * Ep, st));
  VSR_CHECK_CUDA(cudaMemsetAsync(c->WU, 0, sizeof(float) * (size_t)c->NA * c->Fp, st));
  VSR_CHECK_CUDA(cudaMemsetAsync(c->bU, 0, sizeof(float) * (size_t)c->NA, st));

  // ---- S1 / S2 -> WA, WU, bU.  Six "gates" per hidden unit, rows gate-interleaved (cell_col(g, u, 6)):
  //      0..3 = lstm_cell_1 i,f,g,o | 4 = sentinel gate (W1_is + W1_hs) | 5 = shift gate, input_1 part (W1_ig)
  struct Gate { const float* wi; const float* wh; const float* bi; const float* bh; };
  Gate gates[6];
  for (int g = 0; g < 4; ++g)       // lstm_cell_1: W_ih / W_hh act on (input_1, h1_old)
    gates[g] = {w[10] + (size_t)g * H * in1, w[11] + (size_t)g * H * H, w[12] + g * H, w[13] + g * H};
  gates[4] = {w[1], w[3], w[2], w[4]};           // W1_is(input_1) + W1_hs(h1_old)            (:151)
  gates[5] = {w[22], nullptr, w[23], w[25]};     // W1_ig(input_1); W1_hg acts on h1' (:181) -> WB2
  for (int g = 0; g < 6; ++g) {
    const Gate& k = gates[g];
    if (h2f) VSR_TRY(pack_perm(c, c->WA, c->KA, 0, ka_h2, k.wi, in1, 0, H, H, g, 6, st));
    VSR_TRY(pack_perm(c, c->WAx, Ep, 0, 0, k.wi, in1, c_xt, H, E, g, 6, st));
    if (k.wh != nullptr) VSR_TRY(pack_perm(c, c->WA, c->KA, 0, ka_h1, k.wh, H, 0, H, H, g, 6, st));
    VSR_TRY(pack_perm(c, c->WU, c->Fp, 0, 0, k.wi, in1, c_img, H, F, g, 6, st));
    VSR_TRY(pack_bias_perm(c, c->bU, k.bi, k.bh, H, g, 6, st));
  }
  // ---- S3 -> WB1: s_fc (F rows) | att_sa (A rows)
  VSR_CHECK_CUDA(cudaMemsetAsync(c->WB1, 0, sizeof(float) * (size_t)c->NB1 * Hp, st));
  VSR_CHECK_CUDA(cudaMemsetAsync(c->bB1, 0, sizeof(float) * (size_t)c->NB1, st));
  VSR_TRY(pack_block(c, c->WB1, Hp, 0, 0, w[20], H, 0, F, H, st));
  VSR_TRY(pack_block(c, c->WB1, Hp, c->oB1_sa, 0, w[8], H, 0, A, H, st));
  VSR_TRY(pack_bias(c, c->bB1, 0, w[21], nullptr, F, st));
  // ---- S4 -> WB2: W1_hg (H) | att_ha (A)
  VSR_CHECK_CUDA(cudaMemsetAsync(c->WB2, 0, sizeof(float) * (size_t)c->NB2 * Hp, st));
  VSR_TRY(pack_block(c, c->WB2, Hp, 0, 0, w[24], H, 0, H, H, st));
  VSR_TRY(pack_block(c, c->WB2, Hp, c->oB2_ha, 0, w[6], H, 0, A, H, st));
  // ---- S5 -> WC: att_ga
  VSR_CHECK_CUDA(cudaMemsetAsync(c->WC, 0, sizeof(float) * (size_t)c->NC * Hp, st));
  VSR_TRY(pack_block(c, c->WC, Hp, 0, 0, w[26], H, 0, A, H, st));
  // ---- S6 -> WD: lstm2.W_ih[:, H:H+F] (att) | lstm2.W_ih[:, 0:H] (h1') | lstm2.W_hh (h2) ; bias b_ih2 + b_hh2
  // (h1' rides in GEMM-D rather than in the h1' projection GEMM-B: B then fits one wave of 148 CTAs)
  VSR_CHECK_CUDA(cudaMemsetAsync(c->WD, 0, sizeof(float) * (size_t)c->ND * c->KD, st));
  VSR_CHECK_CUDA(cudaMemsetAsync(c->bD, 0, sizeof(float) * (size_t)c->ND, st));
  if (img2) VSR_CHECK_CUDA(cudaMemsetAsync(c->WU2, 0, sizeof(float) * (size_t)c->ND * c->Fp, st));
  for (int g = 0; g < 4; ++g) {
    const float* wi = w[14] + (size_t)g * H * in2;
    VSR_TRY(pack_perm(c, c->WD, c->KD, 0, 0, wi, in2, H, H, F, g, 4, st));
    VSR_TRY(pack_perm(c, c->WD, c->KD, 0, c->Fp, wi, in2, 0, H, H, g, 4, st));
    VSR_TRY(pack_perm(c, c->WD, c->KD, 0, c->Fp + Hp, w[15] + (size_t)g * H * H, H, 0, H, H, g, 4, st));
    VSR_TRY(pack_bias_perm(c, c->bD, w[16] + g * H, w[17] + g * H, H, g, 4, st));
    if (img2) VSR_TRY(pack_perm(c, c->WU2, c->Fp, 0, 0, wi, in2, H + F, H, F, g, 4, st));
  }
  // ---- S7 -> WE: out_fc
  VSR_CHECK_CUDA(cudaMemsetAsync(c->WE, 0, sizeof(float) * (size_t)c->NE * Hp, st));
  VSR_CHECK_CUDA(cudaMemsetAsync(c->bE, 0, sizeof(float) * (size_t)c->NE, st));
  VSR_TRY(pack_block(c, c->WE, Hp, 0, 0, w[18], H, 0, V, H, st));
  VSR_TRY(pack_bias(c, c->bE, 0, w[19], nullptr, V, st));
  // ---- att_va, attention vectors, embedding
  VSR_CHECK_CUDA(cudaMemsetAsync(c->Wva, 0, sizeof(float) * (size_t)c->NVA * c->Fp, st));
  VSR_TRY(pack_block(c, c->Wva, c->Fp, 0, 0, w[5], F, 0, A, F, st));
  VSR_CHECK_CUDA(cudaMemsetAsync(c->v_a, 0, sizeof(float) * c->Ap, st));
  VSR_CHECK_CUDA(cudaMemsetAsync(c->v_s, 0, sizeof(float) * c->Ap, st));
  VSR_CHECK_CUDA(cudaMemsetAsync(c->v_g, 0, sizeof(float) * c->Ap, st));
  VSR_TRY(pack_bias(c, c->v_a, 0, w[7], nullptr, A, st));
  VSR_TRY(pack_bias(c, c->v_s, 0, w[9], nullptr, A, st));
  VSR_TRY(pack_bias(c, c->v_g, 0, w[27], nullptr, A, st));
  VSR_CHECK_CUDA(cudaMemsetAsync(c->embed, 0, sizeof(float) * (size_t)V * Ep, st));
  VSR_TRY(pack_block(c, c->embed, Ep, 0, 0, w[0], E, 0, V, E, st));
  {  // X[v] = WAx . embed[v]  (exact fp32 FFMA, once per weight load): the xt third of input_1 never enters
     // the per-step GEMM; step t adds row X[word] in the GEMM-A epilogue instead (SURVEY.md Appendix A)
    GemmArgs g{};
    g.nseg = 1; g.seg[0] = {c->embed, Ep, Ep, Ep};
    g.w = c->WAx; g.ldw = Ep;
    g.c = c->X; g.ldc = c->NA; g.M = V; g.N = c->NA;
    VSR_TRY(launch_gemm_simt(g, st));
    c->launches++;
  }
  // fp16 hi/lo twins of the per-step weights and of the embedding table (tcgen05 operands)
  struct Tw { const float* f; F16Pair* b; size_t n; };
  const Tw tw[] = {{c->WU, &c->WU_b, (size_t)c->NA * c->Fp}, {c->WU2, &c->WU2_b, (size_t)c->ND * c->Fp},
                   {c->Wva, &c->Wva_b, (size_t)c->NVA * c->Fp},
                   {c->WA, &c->WA_b, (size_t)c->NA * c->KA}, {c->WB1, &c->WB1_b, (size_t)c->NB1 * Hp},
                   {c->WB2, &c->WB2_b, (size_t)c->NB2 * Hp}, {c->WC, &c->WC_b, (size_t)c->NC * Hp},
                   {c->WD, &c->WD_b, (size_t)c->ND * c->KD}, {c->WE, &c->WE_b, (size_t)c->NE * Hp}};
  for (const Tw& t : tw) {
    if (t.b->hi == nullptr || t.f == nullptr) continue;
    VSR_TRY(launch_split_pair(t.f, *t.b, t.n, st, true));
    c->launches += t.b->scale != nullptr ? 3 : 1;
  }
  return VSR_OK;
}

// calls fn(T()) with T the element type of feature dtype tag dt (validated by prologue_impl)
template <typename Fn>
static int with_feat_type(int dt, Fn&& fn) {
  if (dt == VSR_DT_F16) return fn(__half());
  if (dt == VSR_DT_BF16) return fn(__nv_bfloat16());
  return fn(float());
}

template <typename T>
static int run_prologue_t(Ctx* c, const T* det, int64_t det_stride, cudaStream_t st) {
  PhaseScope ps(c, PH_PROLOGUE, st);
  const int F = c->F, D = c->D, b = c->b, L = c->L, R = c->R;
  const T* det_seqs = static_cast<const T*>(c->det_seqs);
  const int n_img = c->n_img;
  // validity of detection rows and slot rows
  {
    const int rows = n_img * D;
    const PairOut none{twin_out(nullptr), 0};
    k_row_valid<<<(rows * 32 + 255) / 256, 256, 0, st>>>(det, det_stride, D, rows, F, c->det_valid, none);
    VSR_CHECK_CUDA(cudaGetLastError());
    const int srows = b * L * R;
    k_row_valid<<<(int)(((size_t)srows * 32 + 255) / 256), 256, 0, st>>>(det_seqs, (int64_t)L * R * F, L * R,
                                                                          srows, F, c->seq_valid, none);
    VSR_CHECK_CUDA(cudaGetLastError());
    k_slot_masks<<<(b * L + 127) / 128, 128, 0, st>>>(c->seq_valid, R, b * L, c->slot_mask);
    VSR_CHECK_CUDA(cudaGetLastError());
    c->launches += 3;
    if (c->p_compact) {
      // about half of the slot rows are padding: only the valid ones are split to fp16 and projected
      const PairOut dsp{twin_out(&c->ds_b), c->Fp};
      k_slot_scan<<<1, 1024, 0, st>>>(c->slot_mask, b * L, c->slot_base, c->comp_valid, round_up(srows, MPAD));
      VSR_CHECK_CUDA(cudaGetLastError());
      k_split_compact<<<(int)(((size_t)srows * 32 + 255) / 256), 256, 0, st>>>(det_seqs, R, srows, F, c->slot_mask,
                                                                               c->slot_base, dsp);
      VSR_CHECK_CUDA(cudaGetLastError());
      c->launches += 2;
    }
  }
  // image descriptor
  {
    dim3 grid((F / 4 + 127) / 128, n_img);
    const PairOut ip{twin_out(&c->img_b, c->use_tc), c->Fp};
    k_pool<<<grid, dim3(128, POOL_Y), 0, st>>>(det, det_stride, D, F, c->det_valid, c->img, c->Fp, ip);
    VSR_CHECK_CUDA(cudaGetLastError());
    c->launches++;
  }
  // U = WU . img + biases ; U2 likewise
  {
    GemmArgs g{};
    g.nseg = 1; g.seg[0] = {c->img, c->Fp, c->Fp, c->Fp, &c->img_b};
    g.w = c->WU; g.ldw = c->Fp; g.bias = c->bU; g.wb = &c->WU_b;
    g.c = c->U; g.ldc = c->NA; g.M = n_img; g.N = c->NA;
    VSR_TRY(launch_gemm(c, g, st));
    c->launches++;
    if (c->d.img_second_lstm) {
      GemmArgs g2{};
      g2.nseg = 1; g2.seg[0] = {c->img, c->Fp, c->Fp, c->Fp, &c->img_b};
      g2.w = c->WU2; g2.ldw = c->Fp; g2.wb = &c->WU2_b;
      g2.c = c->U2; g2.ldc = c->ND; g2.M = n_img; g2.N = c->ND;
      VSR_TRY(launch_gemm(c, g2, st));
      c->launches++;
    }
  }
  // P = att_va . det_seqs rows (tiles of padding rows are skipped).  The tensor-core path reads the fp16 twins
  // written above; the fp32 FFMA twin reads det_seqs in place, which prologue_impl allows only for fp32 features.
  {
    GemmArgs g{};
    g.nseg = 1; g.seg[0] = {reinterpret_cast<const float*>(det_seqs), F, c->Fp, F, &c->ds_b};
    g.w = c->Wva; g.ldw = c->Fp; g.wb = &c->Wva_b;
    g.c = c->P; g.ldc = c->NVA; g.M = b * L * R; g.N = c->NVA;
    g.row_skip = c->p_compact ? c->comp_valid : c->seq_valid;     // compact: the tiles past the last valid row are skipped
    VSR_TRY(launch_gemm(c, g, st));
    c->launches++;
  }
  return VSR_OK;
}

int run_prologue(Ctx* c, const void* det, int64_t det_stride, cudaStream_t st) {
  return with_feat_type(c->feat_dtype, [&](auto t) {
    return run_prologue_t(c, static_cast<const decltype(t)*>(det), det_stride, st);
  });
}

// Index form (vsr_prologue_indexed): projections per DETECTION row + one per image mean row; slot tiles are
// never materialised.
template <typename T>
static int run_prologue_indexed_t(Ctx* c, const T* det, int64_t det_stride, cudaStream_t st) {
  PhaseScope ps(c, PH_PROLOGUE, st);
  const int F = c->F, D = c->D, b = c->b, L = c->L, R = c->R;
  const int n_img = c->n_img;
  const int rows = n_img * D;
  {
    const PairOut dsp{twin_out(&c->ds_b, c->use_tc), c->Fp};
    k_row_valid<<<(rows * 32 + 255) / 256, 256, 0, st>>>(det, det_stride, D, rows, F, c->det_valid, dsp);
    VSR_CHECK_CUDA(cudaGetLastError());
    k_slot_masks_indexed<<<(b * L + 127) / 128, 128, 0, st>>>(c->slot_index, c->det_valid, R, L, D, b * L,
                                                              n_img == 1 ? 0 : 1, c->slot_mask);
    VSR_CHECK_CUDA(cudaGetLastError());
    dim3 grid((F / 4 + 127) / 128, n_img);
    const PairOut ip{twin_out(&c->img_b, c->use_tc), c->Fp};
    k_pool<<<grid, dim3(128, POOL_Y), 0, st>>>(det, det_stride, D, F, c->det_valid, c->img, c->Fp, ip);
    VSR_CHECK_CUDA(cudaGetLastError());
    c->launches += 3;
  }
  {
    GemmArgs g{};
    g.nseg = 1; g.seg[0] = {c->img, c->Fp, c->Fp, c->Fp, &c->img_b};
    g.w = c->WU; g.ldw = c->Fp; g.bias = c->bU; g.wb = &c->WU_b;
    g.c = c->U; g.ldc = c->NA; g.M = n_img; g.N = c->NA;
    VSR_TRY(launch_gemm(c, g, st));
    c->launches++;
    if (c->d.img_second_lstm) {
      GemmArgs g2{};
      g2.nseg = 1; g2.seg[0] = {c->img, c->Fp, c->Fp, c->Fp, &c->img_b};
      g2.w = c->WU2; g2.ldw = c->Fp; g2.wb = &c->WU2_b;
      g2.c = c->U2; g2.ldc = c->ND; g2.M = n_img; g2.N = c->ND;
      VSR_TRY(launch_gemm(c, g2, st));
      c->launches++;
    }
  }
  {  // P per detection row, and per image mean row
    GemmArgs g{};
    // the fp32 FFMA twin reads the detections in place (fp32 features only); their rows are contiguous only when
    // images are dense
    g.nseg = 1; g.seg[0] = {reinterpret_cast<const float*>(det), F, c->Fp, F, &c->ds_b};
    g.w = c->Wva; g.ldw = c->Fp; g.wb = &c->Wva_b;
    g.c = c->P; g.ldc = c->NVA; g.M = rows; g.N = c->NVA;
    g.row_skip = c->det_valid;
    VSR_TRY(launch_gemm(c, g, st));
    GemmArgs gm{};
    gm.nseg = 1; gm.seg[0] = {c->img, c->Fp, c->Fp, c->Fp, &c->img_b};
    gm.w = c->Wva; gm.ldw = c->Fp; gm.wb = &c->Wva_b;
    gm.c = c->Pmean; gm.ldc = c->NVA; gm.M = n_img; gm.N = c->NVA;
    VSR_TRY(launch_gemm(c, gm, st));
    c->launches += 2;
  }
  return VSR_OK;
}

int run_prologue_indexed(Ctx* c, const void* det, int64_t det_stride, cudaStream_t st) {
  return with_feat_type(c->feat_dtype, [&](auto t) {
    return run_prologue_indexed_t(c, static_cast<const decltype(t)*>(det), det_stride, st);
  });
}

}  // namespace vsr
