// vit.cu — ViT inference forward (CBIR extract path with a Transformer backbone) on the same tcgen05 GEMM, plus the one
// kernel the ConvNeXt path does not have: softmax(Q K^T / sqrt(d)) V.
//
// Replaces, for `timm-vit_*` backbones, the eval forward of TimmWrapper (models/faceX/backbone/timm_wrapper.py:51-54: timm's
// VisionTransformer.forward_features + the Transformer neck LayerNorm -> Flatten -> Linear -> BatchNorm1d of :39-47) that
// FeatureExtractor.extract_cbir (models/faceX/face_model.py:120-144) runs per batch.
//
//   patchify (NCHW fp32 -> [B*N, 3*P*P] bf16)  -> GEMM(+bias)          patch embedding (Conv2d(3,C,P,P) as a GEMM)
//   assemble: x[b,0] = cls + pos[0]; x[b,1+i] = tok[b,i] + pos[1+i]
//   per block:  y = LN1(x); qkv = GEMM(y)+b; a = attention(qkv); x = x + GEMM(a)+b        (residual in the GEMM epilogue)
//               y = LN2(x); h = GELU(GEMM(y)+b); x = x + GEMM(h)+b
//   y = LN_neck(LN_final(x)); embeddings = split-K GEMM over (token, channel) with BatchNorm1d folded [+ L2 normalise]
//
// Attention: one CTA = 64 query rows of one (image, head), 4 warps x 16 rows, K/V streamed in 64-row tiles through
// swizzled shared memory, mma.sync m16n8k16 (bf16 in, fp32 accumulate) with the online-softmax recurrence in registers
// (scores never leave the SM).  Attention is 4 % of a ViT-B's FLOPs; the tcgen05 version is the next step for it.
#include "vdk_host.h"
#include "vdk_ptx.cuh"
#include "convnext_internal.h"
#include "train_gemm.h"

#include <algorithm>
#include <cstdlib>

namespace vdk {

// ------------------------------------------------------------------------------------------------
// patchify: NCHW fp32 image -> rows of Kp >= 3*P*P bf16 in (c, kh, kw) order (Conv2d weight order), zero padded to Kp
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
vit_patchify_kernel(const float* __restrict__ x, int B, int S, int P, int Kp, __nv_bfloat16* __restrict__ out) {
  const int G = S / P;  // patches per side
  const int64_t total = static_cast<int64_t>(B) * G * G * Kp;
  for (int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int kidx = static_cast<int>(t % Kp);
    const int64_t patch = t / Kp;
    float v = 0.f;
    if (kidx < 3 * P * P) {
      const int c = kidx / (P * P), r = kidx - c * P * P, kh = r / P, kw = r - kh * P;
      const int pw = static_cast<int>(patch % G), ph = static_cast<int>((patch / G) % G);
      const int b = static_cast<int>(patch / (static_cast<int64_t>(G) * G));
      v = x[((static_cast<int64_t>(b) * 3 + c) * S + (ph * P + kh)) * S + pw * P + kw];
    }
    out[t] = __float2bfloat16_rn(v);
  }
}

// x[b, 0, :] = cls + pos[0];  x[b, 1 + i, :] = tok[b, i, :] + pos[1 + i]
__global__ void __launch_bounds__(256)
vit_assemble_kernel(const __nv_bfloat16* __restrict__ tok, const float* __restrict__ cls, const float* __restrict__ pos, int B,
                    int N, int C, __nv_bfloat16* __restrict__ x) {
  const int64_t total = static_cast<int64_t>(B) * (N + 1) * (C / 2);
  for (int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c2 = static_cast<int>(t % (C / 2));
    const int64_t row = t / (C / 2);
    const int tk = static_cast<int>(row % (N + 1));
    const int b = static_cast<int>(row / (N + 1));
    float2 v;
    if (tk == 0) {
      v = make_float2(cls[2 * c2], cls[2 * c2 + 1]);
    } else {
      v = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(tok + (static_cast<int64_t>(b) * N + tk - 1) * C + 2 * c2));
    }
    const float2 p = *reinterpret_cast<const float2*>(pos + static_cast<int64_t>(tk) * C + 2 * c2);
    *reinterpret_cast<__nv_bfloat162*>(x + row * C + 2 * c2) = __floats2bfloat162_rn(v.x + p.x, v.y + p.y);
  }
}

// ------------------------------------------------------------------------------------------------
// attention forward, head_dim 64
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

constexpr int kAttD = 64;        // head dim
constexpr int kAttBN = 64;       // key/value rows per shared-memory tile
constexpr int kAttMaxWarps = 16; // query rows per CTA = 16 per warp

// [rows] x 64 bf16 tile in shared memory: 128-byte rows, 16-byte chunk index XOR (row & 7) (conflict-free ldmatrix)
__device__ __forceinline__ uint32_t att_tile_addr(uint32_t base, int row, int col /*multiple of 8*/) {
  return base + row * 128 + (((col >> 3) ^ (row & 7)) << 4);
}

// qkv: [B, N, 3, H, 64] bf16 (the qkv Linear's output as stored);  out: [B, N, H*64] bf16.
// CTA = up to 16 warps, each owning 16 query rows of one (image, head); K / V stream through 64-row tiles loaded once per
// CTA (ViT-B/16: 197 tokens -> ONE CTA of 13 warps per (image, head), K and V read once); 8-column score tiles and 16-row
// P.V steps that lie entirely beyond N are skipped.
__global__ void __launch_bounds__(kAttMaxWarps * 32)
attention_fwd_kernel(const __nv_bfloat16* __restrict__ qkv, int B, int N, int H, float scale_log2e, __nv_bfloat16* __restrict__ out,
                     float* __restrict__ lse2 /*[B,H,N] log2-domain log-sum-exp per row, or null*/) {
  extern __shared__ __align__(128) uint8_t att_smem[];
  const int nwarps = blockDim.x >> 5;
  uint8_t* sq = att_smem;                       // [nwarps * 16][64]
  uint8_t* skv = att_smem + nwarps * 16 * 128;  // 2 stages x { K [64][64], V [64][64] }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int q0 = (blockIdx.x * nwarps + warp) * 16, h = blockIdx.y, b = blockIdx.z;
  const int64_t ld = static_cast<int64_t>(3) * H * kAttD;
  const __nv_bfloat16* base = qkv + static_cast<int64_t>(b) * N * ld + h * kAttD;
  const __nv_bfloat16* kp = base + static_cast<int64_t>(H) * kAttD;
  const __nv_bfloat16* vp = base + static_cast<int64_t>(2) * H * kAttD;

  // this warp's 16 query rows -> its private slice of sq -> A fragments for the 4 k-steps over d
  uint32_t qa[4][4];
  {
    uint8_t* mine = sq + warp * 16 * 128;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int idx = lane + c * 32;
      const int r = idx >> 3, ch = idx & 7;
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (q0 + r < N) v = __ldg(reinterpret_cast<const uint4*>(base + static_cast<int64_t>(q0 + r) * ld + ch * 8));
      *reinterpret_cast<uint4*>(mine + r * 128 + ((ch ^ (r & 7)) << 4)) = v;
    }
    __syncwarp();
    const uint32_t sqb = smem_u32(mine);
    const int i = lane >> 3, r = lane & 7;
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) ldmatrix_x4(qa[kk], att_tile_addr(sqb, (i & 1) * 8 + r, kk * 16 + (i >> 1) * 8));
  }
  float o[8][4];
#pragma unroll
  for (int j = 0; j < 8; ++j)
#pragma unroll
    for (int c = 0; c < 4; ++c) o[j][c] = 0.f;
  float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};  // rows g and g + 8

  // K / V tiles are double buffered with cp.async: tile t+1 is in flight while tile t is multiplied
  auto issue_tile = [&](int kv0, int stage) {
    uint8_t* dstb = skv + stage * (2 * kAttBN * 128);
    for (int idx = threadIdx.x; idx < 2 * kAttBN * 8; idx += blockDim.x) {
      const int m = idx >> 9, rem = idx & 511;  // m: 0 = K, 1 = V
      const int r = rem >> 3, ch = rem & 7;
      const bool ok = kv0 + r < N;
      const __nv_bfloat16* src = (m ? vp : kp) + static_cast<int64_t>(ok ? kv0 + r : 0) * ld + ch * 8;
      const uint32_t dst = smem_u32(dstb + m * (kAttBN * 128) + r * 128 + ((ch ^ (r & 7)) << 4));
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(ok ? 16 : 0) : "memory");  // 0: zero fill
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  const int n_tiles = (N + kAttBN - 1) / kAttBN;
  issue_tile(0, 0);
  for (int tile = 0; tile < n_tiles; ++tile) {
    const int kv0 = tile * kAttBN;
    if (tile + 1 < n_tiles) {
      issue_tile(kv0 + kAttBN, (tile + 1) & 1);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();  // every thread's part of tile `tile` has landed
    const uint32_t skb = smem_u32(skv + (tile & 1) * (2 * kAttBN * 128)), svb = skb + kAttBN * 128;
    const int n_valid = min(kAttBN, N - kv0);  // key columns of this tile that exist
    // S = Q K^T for 16 rows x 64 key columns
    float sacc[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
      for (int c = 0; c < 4; ++c) sacc[j][c] = 0.f;
    {
      const int i = lane >> 3, r = lane & 7;
#pragma unroll
      for (int jp = 0; jp < 4; ++jp) {  // pairs of 8-column tiles
        if (jp * 16 < n_valid) {
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            uint32_t kb[4];
            ldmatrix_x4(kb, att_tile_addr(skb, jp * 16 + (i >> 1) * 8 + r, kk * 16 + (i & 1) * 8));
            mma_bf16_16816(sacc[2 * jp], qa[kk], kb[0], kb[1]);
            mma_bf16_16816(sacc[2 * jp + 1], qa[kk], kb[2], kb[3]);
          }
        }
      }
    }
    // scale, mask the columns beyond N, online softmax
    float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int col = j * 8 + 2 * t + (c & 1);
        const float v = col < n_valid ? sacc[j][c] * scale_log2e : -INFINITY;
        sacc[j][c] = v;
        mx[c >> 1] = fmaxf(mx[c >> 1], v);
      }
    }
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
      mx[rr] = fmaxf(mx[rr], __shfl_xor_sync(0xffffffffu, mx[rr], 1));
      mx[rr] = fmaxf(mx[rr], __shfl_xor_sync(0xffffffffu, mx[rr], 2));
    }
    float corr[2], m_new[2];
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
      m_new[rr] = fmaxf(m_run[rr], mx[rr]);  // finite: every tile has at least one valid column
      corr[rr] = fast_exp2(m_run[rr] - m_new[rr]);
      m_run[rr] = m_new[rr];
    }
    float rs[2] = {0.f, 0.f};
    uint32_t pa[4][4];  // P as A fragments: k-step kk covers key columns 16 kk .. 16 kk + 15 = score tiles 2kk, 2kk+1
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float p0 = fast_exp2(sacc[j][0] - m_new[0]), p1 = fast_exp2(sacc[j][1] - m_new[0]);
      const float p2 = fast_exp2(sacc[j][2] - m_new[1]), p3 = fast_exp2(sacc[j][3] - m_new[1]);
      rs[0] += p0 + p1;
      rs[1] += p2 + p3;
      __nv_bfloat162 lo = __floats2bfloat162_rn(p0, p1), hi = __floats2bfloat162_rn(p2, p3);
      pa[j >> 1][(j & 1) * 2] = *reinterpret_cast<uint32_t*>(&lo);
      pa[j >> 1][(j & 1) * 2 + 1] = *reinterpret_cast<uint32_t*>(&hi);
    }
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
      rs[rr] += __shfl_xor_sync(0xffffffffu, rs[rr], 1);
      rs[rr] += __shfl_xor_sync(0xffffffffu, rs[rr], 2);
      l_run[rr] = l_run[rr] * corr[rr] + rs[rr];
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      o[j][0] *= corr[0]; o[j][1] *= corr[0];
      o[j][2] *= corr[1]; o[j][3] *= corr[1];
    }
    // O += P V
    {
      const int i = lane >> 3, r = lane & 7;
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        if (kk * 16 < n_valid) {
#pragma unroll
          for (int jp = 0; jp < 4; ++jp) {  // pairs of 8-wide d tiles
            uint32_t vb[4];
            ldmatrix_x4_trans(vb, att_tile_addr(svb, kk * 16 + (i & 1) * 8 + r, jp * 16 + (i >> 1) * 8));
            mma_bf16_16816(o[2 * jp], pa[kk], vb[0], vb[1]);
            mma_bf16_16816(o[2 * jp + 1], pa[kk], vb[2], vb[3]);
          }
        }
      }
    }
    __syncthreads();  // this stage is free again for the tile after next
  }
  // normalise and store: rows q0 + g (+8), columns h*64 + 8j + 2t
  const float inv0 = 1.0f / l_run[0], inv1 = 1.0f / l_run[1];
  const int r0 = q0 + g, r1 = r0 + 8;
  if (lse2 != nullptr && t == 0) {  // saved for the backward: P = exp2(s * scale_log2e - lse2)
    float* lp = lse2 + (static_cast<int64_t>(b) * H + h) * N;
    if (r0 < N) lp[r0] = m_run[0] + log2f(l_run[0]);
    if (r1 < N) lp[r1] = m_run[1] + log2f(l_run[1]);
  }
  __nv_bfloat16* ob = out + static_cast<int64_t>(b) * N * H * kAttD + h * kAttD;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (r0 < N)
      *reinterpret_cast<__nv_bfloat162*>(ob + static_cast<int64_t>(r0) * H * kAttD + j * 8 + 2 * t) =
          __floats2bfloat162_rn(o[j][0] * inv0, o[j][1] * inv0);
    if (r1 < N)
      *reinterpret_cast<__nv_bfloat162*>(ob + static_cast<int64_t>(r1) * H * kAttD + j * 8 + 2 * t) =
          __floats2bfloat162_rn(o[j][2] * inv1, o[j][3] * inv1);
  }
}

int launch_attention_tc(const __nv_bfloat16* qkv, int B, int N, int H, __nv_bfloat16* out, float* lse2, cudaStream_t s);  // attention_tc.cu

static int launch_attention_mma_sync(const __nv_bfloat16* qkv, int B, int N, int H, int head_dim, __nv_bfloat16* out, float* lse2,
                                     cudaStream_t s);

// Forward attention: the tcgen05 kernel (attention_tc.cu) by default; VDK_ATT_TC=0 selects the earlier mma.sync kernel (kept as
// the comparison baseline of profiles/ and for A/B parity tests).
static int launch_attention(const __nv_bfloat16* qkv, int B, int N, int H, int head_dim, __nv_bfloat16* out, float* lse2,
                            cudaStream_t s) {
  static const bool use_tc = [] {
    const char* e = getenv("VDK_ATT_TC");
    return e ? atoi(e) != 0 : true;
  }();
  if (!use_tc) return launch_attention_mma_sync(qkv, B, N, H, head_dim, out, lse2, s);
  VDK_REQUIRE(head_dim == kAttD, "attention: head_dim must be 64 (got %d)", head_dim);
  ProfScope prof(kProfAttention, 4.0 * static_cast<double>(B) * H * N * N * 64.0, 2.0 * static_cast<double>(B) * N * H * 64.0 * 4.0, s);
  return launch_attention_tc(qkv, B, N, H, out, lse2, s);
}

static int launch_attention_mma_sync(const __nv_bfloat16* qkv, int B, int N, int H, int head_dim, __nv_bfloat16* out, float* lse2,
                                     cudaStream_t s) {
  // algorithmic work: QK^T and PV = 4 * N^2 * head_dim flops per (image, head); qkv (+ o, do, dqkv) read / written once
  ProfScope prof(kProfAttention, 4.0 * static_cast<double>(B) * H * N * N * 64.0,
                 2.0 * static_cast<double>(B) * N * H * 64.0 * 4.0, s);

  VDK_REQUIRE(head_dim == kAttD, "attention: head_dim must be 64 (got %d)", head_dim);
  VDK_REQUIRE(B > 0 && N > 0 && H > 0 && H <= 65535 && B <= 65535, "attention: bad shape");
  const float scale_log2e = 1.4426950408889634f / sqrtf(static_cast<float>(head_dim));
  const int row_groups = (N + 15) / 16;
  static const int warp_cap = [] {  // tuning switch: query-row groups (warps) per CTA
    const char* e = getenv("VDK_ATT_WARPS");
    const int v = e ? atoi(e) : 8;  // measured on ViT-B/16 batch 256: 16 -> 13.06 ms, 8 -> 12.68 ms, 4 -> 12.87 ms per forward
    return v < 1 ? 1 : (v > kAttMaxWarps ? kAttMaxWarps : v);
  }();
  const int ctas = (row_groups + warp_cap - 1) / warp_cap;
  const int nwarps = (row_groups + ctas - 1) / ctas;  // balanced: 197 tokens -> 1 CTA x 13 warps; 577 -> 3 CTAs x 13 warps
  const int smem = nwarps * 16 * 128 + 2 * (2 * kAttBN * 128);
  static bool attr = false;
  if (!attr) {
    VDK_CUDA_OK(cudaFuncSetAttribute(attention_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    attr = true;
  }
  attention_fwd_kernel<<<dim3(ctas, H, B), nwarps * 32, smem, s>>>(qkv, B, N, H, scale_log2e, out, lse2);
  VDK_CUDA_OK(cudaGetLastError());
  return VDK_OK;
}

// ------------------------------------------------------------------------------------------------
// attention backward for N <= 208 tokens (ViT-*/16 at 224^2: 197): one CTA per (image, head) keeps Q, K, V, dO and the
// whole probability matrix in shared memory and runs the five products of the backward as in-CTA GEMMs on mma.sync:
//   P = exp2(scale' Q K^T - lse2)                    (recomputed from the saved log-sum-exp)
//   dV = P^T dO;  dP = dO V^T;  dS = scale P (dP - D),  D_i = sum_d dO_id O_id;  dQ = dS K;  dK = dS^T Q
// Warp w owns rows 16w .. 16w+15 of whichever matrix is being produced.
// ------------------------------------------------------------------------------------------------
constexpr int kAttBwdMaxRows = 208;
constexpr int kAttPStride = 432;  // bytes per row of P (208 bf16 = 416, padded so that 8 rows hit 8 distinct 16-byte bank groups)

__device__ __forceinline__ uint32_t att_p_addr(uint32_t base, int row, int col /*multiple of 8*/) {
  return base + row * kAttPStride + col * 2;
}

__global__ void __launch_bounds__(13 * 32)
attention_bwd_kernel(const __nv_bfloat16* __restrict__ qkv, const __nv_bfloat16* __restrict__ o, const __nv_bfloat16* __restrict__ d_o,
                     const float* __restrict__ lse2, int B, int N, int H, float scale, float scale_log2e,
                     __nv_bfloat16* __restrict__ dqkv) {
  extern __shared__ __align__(128) uint8_t att_smem[];
  const int nwarps = blockDim.x >> 5;  // = ceil(N / 16)
  const int Np = nwarps * 16;
  uint8_t* sq = att_smem;
  uint8_t* sk = sq + Np * 128;
  uint8_t* sv = sk + Np * 128;
  uint8_t* sdo = sv + Np * 128;
  uint8_t* sp = sdo + Np * 128;                                   // [Np][kAttPStride]
  float* sD = reinterpret_cast<float*>(sp + Np * kAttPStride);    // [Np]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int h = blockIdx.x, b = blockIdx.y;
  const int64_t ld = static_cast<int64_t>(3) * H * kAttD, ldo = static_cast<int64_t>(H) * kAttD;
  const __nv_bfloat16* qb = qkv + static_cast<int64_t>(b) * N * ld + h * kAttD;
  const __nv_bfloat16* ob = o + static_cast<int64_t>(b) * N * ldo + h * kAttD;
  const __nv_bfloat16* dob = d_o + static_cast<int64_t>(b) * N * ldo + h * kAttD;
  __nv_bfloat16* dqb = dqkv + static_cast<int64_t>(b) * N * ld + h * kAttD;

  // ---- stage Q, K, V, dO (rows >= N zero) ----
  for (int idx = threadIdx.x; idx < 4 * Np * 8; idx += blockDim.x) {
    const int m = idx / (Np * 8), rem = idx - m * (Np * 8);
    const int r = rem >> 3, ch = rem & 7;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (r < N) {
      const __nv_bfloat16* src = m < 3 ? qb + static_cast<int64_t>(m) * H * kAttD + static_cast<int64_t>(r) * ld
                                       : dob + static_cast<int64_t>(r) * ldo;
      v = __ldg(reinterpret_cast<const uint4*>(src + ch * 8));
    }
    *reinterpret_cast<uint4*>(sq + m * (Np * 128) + r * 128 + ((ch ^ (r & 7)) << 4)) = v;
  }
  // D_i = sum_d dO_id O_id: 2 lanes per row (32 columns each)
  {
    const int r = warp * 16 + (lane >> 1), half = lane & 1;
    float acc = 0.f;
    if (r < N) {
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const uint4 a = __ldg(reinterpret_cast<const uint4*>(ob + static_cast<int64_t>(r) * ldo + half * 32 + c * 8));
        const uint4 d = __ldg(reinterpret_cast<const uint4*>(dob + static_cast<int64_t>(r) * ldo + half * 32 + c * 8));
        const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, dw[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float2 fa = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&aw[k]));
          const float2 fd = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&dw[k]));
          acc = fmaf(fa.x, fd.x, fmaf(fa.y, fd.y, acc));
        }
      }
    }
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    if (half == 0) sD[r] = acc;
  }
  __syncthreads();
  const uint32_t sqb = smem_u32(sq), skb = smem_u32(sk), svb = smem_u32(sv), sdob = smem_u32(sdo), spb = smem_u32(sp);
  const int li = lane >> 3, lr = lane & 7;
  const int row0 = warp * 16;  // this warp's rows
  const float* lp = lse2 + (static_cast<int64_t>(b) * H + h) * N;
  const float l0 = row0 + g < N ? lp[row0 + g] : 0.f, l1 = row0 + g + 8 < N ? lp[row0 + g + 8] : 0.f;

  // ---- phase 1: P rows of this warp = exp2(scale' Q K^T - lse2), stored bf16 ----
  {
    uint32_t qa[4][4];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) ldmatrix_x4(qa[kk], att_tile_addr(sqb, row0 + (li & 1) * 8 + lr, kk * 16 + (li >> 1) * 8));
    for (int c0 = 0; c0 < Np; c0 += 16) {  // two 8-column tiles at a time
      float s0[4] = {0.f, 0.f, 0.f, 0.f}, s1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        uint32_t kb[4];
        ldmatrix_x4(kb, att_tile_addr(skb, c0 + (li >> 1) * 8 + lr, kk * 16 + (li & 1) * 8));
        mma_bf16_16816(s0, qa[kk], kb[0], kb[1]);
        mma_bf16_16816(s1, qa[kk], kb[2], kb[3]);
      }
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const float* sv4 = half ? s1 : s0;
        const int col = c0 + half * 8 + 2 * t;
        const bool ok0 = col < N, ok1 = col + 1 < N;
        const float p00 = ok0 && row0 + g < N ? fast_exp2(sv4[0] * scale_log2e - l0) : 0.f;
        const float p01 = ok1 && row0 + g < N ? fast_exp2(sv4[1] * scale_log2e - l0) : 0.f;
        const float p10 = ok0 && row0 + g + 8 < N ? fast_exp2(sv4[2] * scale_log2e - l1) : 0.f;
        const float p11 = ok1 && row0 + g + 8 < N ? fast_exp2(sv4[3] * scale_log2e - l1) : 0.f;
        *reinterpret_cast<__nv_bfloat162*>(sp + (row0 + g) * kAttPStride + col * 2) = __floats2bfloat162_rn(p00, p01);
        *reinterpret_cast<__nv_bfloat162*>(sp + (row0 + g + 8) * kAttPStride + col * 2) = __floats2bfloat162_rn(p10, p11);
      }
    }
  }
  __syncthreads();  // the whole P is in shared memory

  // ---- phase 2: dV rows (key index) of this warp = sum_i P[i][kv] dO[i][:] ----
  {
    float acc[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[j][c] = 0.f;
    for (int i0 = 0; i0 < Np; i0 += 16) {
      uint32_t a[4];  // A = P^T: rows m = kv (this warp), cols k = i
      ldmatrix_x4_trans(a, att_p_addr(spb, i0 + (li >> 1) * 8 + lr, row0 + (li & 1) * 8));
#pragma unroll
      for (int jp = 0; jp < 4; ++jp) {
        uint32_t bb[4];
        ldmatrix_x4_trans(bb, att_tile_addr(sdob, i0 + (li & 1) * 8 + lr, jp * 16 + (li >> 1) * 8));
        mma_bf16_16816(acc[2 * jp], a, bb[0], bb[1]);
        mma_bf16_16816(acc[2 * jp + 1], a, bb[2], bb[3]);
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (row0 + g < N)
        *reinterpret_cast<__nv_bfloat162*>(dqb + static_cast<int64_t>(2) * H * kAttD + static_cast<int64_t>(row0 + g) * ld + j * 8 + 2 * t) =
            __floats2bfloat162_rn(acc[j][0], acc[j][1]);
      if (row0 + g + 8 < N)
        *reinterpret_cast<__nv_bfloat162*>(dqb + static_cast<int64_t>(2) * H * kAttD + static_cast<int64_t>(row0 + g + 8) * ld + j * 8 + 2 * t) =
            __floats2bfloat162_rn(acc[j][2], acc[j][3]);
    }
  }
  __syncthreads();  // every warp has read P: it may now be overwritten by dS

  // ---- phase 3: dS rows (query index) of this warp = scale * P * (dO V^T - D), in place over P ----
  {
    uint32_t da[4][4];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) ldmatrix_x4(da[kk], att_tile_addr(sdob, row0 + (li & 1) * 8 + lr, kk * 16 + (li >> 1) * 8));
    const float d0 = sD[row0 + g], d1 = sD[row0 + g + 8];
    for (int c0 = 0; c0 < Np; c0 += 16) {
      float s0[4] = {0.f, 0.f, 0.f, 0.f}, s1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        uint32_t vb[4];
        ldmatrix_x4(vb, att_tile_addr(svb, c0 + (li >> 1) * 8 + lr, kk * 16 + (li & 1) * 8));
        mma_bf16_16816(s0, da[kk], vb[0], vb[1]);
        mma_bf16_16816(s1, da[kk], vb[2], vb[3]);
      }
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const float* dp = half ? s1 : s0;
        const int col = c0 + half * 8 + 2 * t;
        __nv_bfloat162* p0 = reinterpret_cast<__nv_bfloat162*>(sp + (row0 + g) * kAttPStride + col * 2);
        __nv_bfloat162* p1 = reinterpret_cast<__nv_bfloat162*>(sp + (row0 + g + 8) * kAttPStride + col * 2);
        const float2 pa = __bfloat1622float2(*p0), pb = __bfloat1622float2(*p1);
        *p0 = __floats2bfloat162_rn(scale * pa.x * (dp[0] - d0), scale * pa.y * (dp[1] - d0));
        *p1 = __floats2bfloat162_rn(scale * pb.x * (dp[2] - d1), scale * pb.y * (dp[3] - d1));
      }
    }
  }
  __syncthreads();  // the whole dS is in shared memory

  // ---- phase 4: dQ rows of this warp = dS K;  phase 5: dK rows of this warp = dS^T Q ----
#pragma unroll 1
  for (int which = 0; which < 2; ++which) {
    float acc[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[j][c] = 0.f;
    const uint32_t bmat = which == 0 ? skb : sqb;
    for (int k0 = 0; k0 < Np; k0 += 16) {
      uint32_t a[4];
      if (which == 0) ldmatrix_x4(a, att_p_addr(spb, row0 + (li & 1) * 8 + lr, k0 + (li >> 1) * 8));          // A = dS
      else ldmatrix_x4_trans(a, att_p_addr(spb, k0 + (li >> 1) * 8 + lr, row0 + (li & 1) * 8));               // A = dS^T
#pragma unroll
      for (int jp = 0; jp < 4; ++jp) {
        uint32_t bb[4];
        ldmatrix_x4_trans(bb, att_tile_addr(bmat, k0 + (li & 1) * 8 + lr, jp * 16 + (li >> 1) * 8));
        mma_bf16_16816(acc[2 * jp], a, bb[0], bb[1]);
        mma_bf16_16816(acc[2 * jp + 1], a, bb[2], bb[3]);
      }
    }
    __nv_bfloat16* dst = dqb + static_cast<int64_t>(which) * H * kAttD;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (row0 + g < N)
        *reinterpret_cast<__nv_bfloat162*>(dst + static_cast<int64_t>(row0 + g) * ld + j * 8 + 2 * t) =
            __floats2bfloat162_rn(acc[j][0], acc[j][1]);
      if (row0 + g + 8 < N)
        *reinterpret_cast<__nv_bfloat162*>(dst + static_cast<int64_t>(row0 + g + 8) * ld + j * 8 + 2 * t) =
            __floats2bfloat162_rn(acc[j][2], acc[j][3]);
    }
  }
}

static int launch_attention_bwd(const __nv_bfloat16* qkv, const __nv_bfloat16* o, const __nv_bfloat16* d_o, const float* lse2, int B,
                                int N, int H, int head_dim, __nv_bfloat16* dqkv, cudaStream_t s) {
  // algorithmic work: S, dP, dV, dQ, dK = 10 * N^2 * head_dim flops per (image, head); qkv (+ o, do, dqkv) read / written once
  ProfScope prof(kProfAttention, 10.0 * static_cast<double>(B) * H * N * N * 64.0,
                 2.0 * static_cast<double>(B) * N * H * 64.0 * 8.0, s);

  VDK_REQUIRE(head_dim == kAttD, "attention backward: head_dim must be 64 (got %d)", head_dim);
  VDK_REQUIRE(N > 0 && N <= kAttBwdMaxRows, "attention backward: at most %d tokens (got %d): the probability matrix of one head is kept "
              "in shared memory", kAttBwdMaxRows, N);
  VDK_REQUIRE(B > 0 && H > 0 && H <= 65535 && B <= 65535, "attention backward: bad shape");
  const int nwarps = (N + 15) / 16, Np = nwarps * 16;
  const int smem = 4 * Np * 128 + Np * kAttPStride + Np * 4;
  static bool attr = false;
  if (!attr) {
    VDK_CUDA_OK(cudaFuncSetAttribute(attention_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    attr = true;
  }
  const float scale = 1.0f / sqrtf(static_cast<float>(head_dim));
  attention_bwd_kernel<<<dim3(H, B), nwarps * 32, smem, s>>>(qkv, o, d_o, lse2, B, N, H, scale, scale * 1.4426950408889634f, dqkv);
  VDK_CUDA_OK(cudaGetLastError());
  return VDK_OK;
}

size_t attention_bwd_tc_workspace_bytes(int B, int N, int H);  // attention_bwd_tc.cu
int launch_attention_bwd_tc(const __nv_bfloat16* qkv, const __nv_bfloat16* out, const __nv_bfloat16* d_out, const float* lse2, int B,
                            int N, int H, __nv_bfloat16* dqkv, void* workspace, size_t workspace_bytes, cudaStream_t s);

// The tcgen05 pair (attention_bwd_tc.cu) for any token count: kernel Q writes D_i = sum_d dO_id O_id into the workspace and dQ,
// kernel KV reads D and writes dK, dV.  It executes 14 N^2 64 flops per (image, head) (no atomics: dS is recomputed on the key side);
// the profile keeps the algorithmic 10 N^2 64 of the mma.sync kernel, so both report the same rate for the same time.
static int launch_attention_bwd_pair(const __nv_bfloat16* qkv, const __nv_bfloat16* o, const __nv_bfloat16* d_o, const float* lse2,
                                     int B, int N, int H, int head_dim, __nv_bfloat16* dqkv, void* workspace, size_t workspace_bytes,
                                     cudaStream_t s) {
  ProfScope prof(kProfAttention, 10.0 * static_cast<double>(B) * H * N * N * 64.0,
                 2.0 * static_cast<double>(B) * N * H * 64.0 * 8.0, s);
  VDK_REQUIRE(head_dim == kAttD, "attention backward: head_dim must be 64 (got %d)", head_dim);
  return launch_attention_bwd_tc(qkv, o, d_o, lse2, B, N, H, dqkv, workspace, workspace_bytes, s);
}

static size_t up256v(size_t v) { return (v + 255) & ~static_cast<size_t>(255); }

struct VitLayout {
  int N, T, C, Kp;  // patches, tokens, width, padded patch-row length
  size_t M;         // batch * tokens
  size_t x, y, big, total;
};

static int vit_layout(const vdk_vit_net* n, int batch, VitLayout* L) {
  VDK_REQUIRE(n, "vdk_vit: null network");
  VDK_REQUIRE(n->patch > 0 && n->image_size > 0 && n->image_size % n->patch == 0, "vdk_vit: image_size must be a multiple of patch");
  VDK_REQUIRE(n->dim > 0 && n->heads > 0 && n->dim == n->heads * kAttD, "vdk_vit: dim must be heads * 64");
  VDK_REQUIRE(n->dim % 256 == 0 || n->dim % 8 == 0, "vdk_vit: dim must be a multiple of 8");
  VDK_REQUIRE(n->depth > 0 && n->depth <= VDK_VIT_MAX_BLOCKS, "vdk_vit: bad depth");
  VDK_REQUIRE(n->feat_dim > 0 && n->feat_dim % 8 == 0, "vdk_vit: feat_dim must be a multiple of 8");
  const int G = n->image_size / n->patch;
  L->N = G * G;
  L->T = L->N + 1;
  L->C = n->dim;
  L->Kp = (3 * n->patch * n->patch + 7) & ~7;
  L->M = static_cast<size_t>(batch) * L->T;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += up256v(bytes); return o; };
  L->x = take(L->M * L->C * 2);
  L->y = take(L->M * L->C * 2);
  // qkv / MLP hidden / patch rows + patch tokens / neck split-K slabs share one buffer
  size_t big = L->M * 4 * static_cast<size_t>(L->C) * 2;
  big = std::max(big, static_cast<size_t>(batch) * L->N * (static_cast<size_t>(L->Kp) + L->C) * 2 + 256);
  big = std::max(big, static_cast<size_t>(batch) * n->feat_dim * 4 * 64);
  L->big = take(big);
  L->total = off + 256;
  return VDK_OK;
}

}  // namespace vdk

using namespace vdk;

extern "C" size_t vdk_vit_workspace_bytes(const vdk_vit_net* net, int batch) {
  VitLayout L;
  if (!net || batch <= 0 || vit_layout(net, batch, &L) != VDK_OK) return 0;
  return L.total;
}

extern "C" int vdk_attention_fwd(const void* qkv, int batch, int tokens, int heads, int head_dim, void* out, void* stream) {
  VDK_REQUIRE(qkv && out, "vdk_attention_fwd: null operand");
  return launch_attention(reinterpret_cast<const __nv_bfloat16*>(qkv), batch, tokens, heads, head_dim,
                          reinterpret_cast<__nv_bfloat16*>(out), nullptr, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int vdk_attention_fwd_lse(const void* qkv, int batch, int tokens, int heads, int head_dim, void* out, float* lse2,
                                     void* stream) {
  VDK_REQUIRE(qkv && out && lse2, "vdk_attention_fwd_lse: null operand");
  return launch_attention(reinterpret_cast<const __nv_bfloat16*>(qkv), batch, tokens, heads, head_dim,
                          reinterpret_cast<__nv_bfloat16*>(out), lse2, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int vdk_attention_bwd(const void* qkv, const void* out, const void* d_out, const float* lse2, int batch, int tokens,
                                 int heads, int head_dim, void* dqkv, void* stream) {
  VDK_REQUIRE(qkv && out && d_out && lse2 && dqkv, "vdk_attention_bwd: null operand");
  return launch_attention_bwd(reinterpret_cast<const __nv_bfloat16*>(qkv), reinterpret_cast<const __nv_bfloat16*>(out),
                              reinterpret_cast<const __nv_bfloat16*>(d_out), lse2, batch, tokens, heads, head_dim,
                              reinterpret_cast<__nv_bfloat16*>(dqkv), reinterpret_cast<cudaStream_t>(stream));
}

extern "C" size_t vdk_attention_bwd_tc_workspace_bytes(int batch, int tokens, int heads, int head_dim) {
  if (head_dim != kAttD) return 0;
  return attention_bwd_tc_workspace_bytes(batch, tokens, heads);
}

extern "C" int vdk_attention_bwd_tc(const void* qkv, const void* out, const void* d_out, const float* lse2, int batch, int tokens,
                                    int heads, int head_dim, void* dqkv, void* workspace, size_t workspace_bytes, void* stream) {
  VDK_REQUIRE(qkv && out && d_out && lse2 && dqkv, "vdk_attention_bwd_tc: null operand");
  return launch_attention_bwd_pair(reinterpret_cast<const __nv_bfloat16*>(qkv), reinterpret_cast<const __nv_bfloat16*>(out),
                                   reinterpret_cast<const __nv_bfloat16*>(d_out), lse2, batch, tokens, heads, head_dim,
                                   reinterpret_cast<__nv_bfloat16*>(dqkv), workspace, workspace_bytes, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int vdk_vit_forward(const vdk_vit_net* net, const float* images, int batch, int l2_normalize, float* embeddings,
                               void* workspace, size_t workspace_bytes, void* stream) {
  VitLayout L;
  int rc = vit_layout(net, batch, &L);
  if (rc != VDK_OK) return rc;
  VDK_REQUIRE(images && embeddings && batch > 0, "vdk_vit_forward: null image/embedding buffer");
  VDK_REQUIRE(workspace && workspace_bytes >= L.total && (reinterpret_cast<uintptr_t>(workspace) & 255) == 0,
              "vdk_vit_forward: workspace too small or misaligned");
  VDK_REQUIRE(net->patch_w && net->cls_token && net->pos_embed && net->ones && net->norm_w && net->norm_b &&
                  net->neck_ln_w && net->neck_ln_b && net->neck_w && net->neck_b,
              "vdk_vit_forward: null parameter");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  __nv_bfloat16* x = reinterpret_cast<__nv_bfloat16*>(ws + L.x);
  __nv_bfloat16* y = reinterpret_cast<__nv_bfloat16*>(ws + L.y);
  __nv_bfloat16* big = reinterpret_cast<__nv_bfloat16*>(ws + L.big);
  const int C = L.C, T = L.T, N = L.N, M = static_cast<int>(L.M);
  const float eps = net->ln_eps > 0.f ? net->ln_eps : 1e-6f;
  VDK_REQUIRE((net->norm_pre_w == nullptr) == (net->norm_pre_b == nullptr), "vdk_vit_forward: norm_pre needs weight and bias");

  auto gemm = [&](const void* A, const void* Bw, void* D, int m, int n, int k, int lda, int epi, const float* bias, const float* gamma,
                  const void* res) {
    vdk_gemm_desc g{};
    g.A = A; g.B = Bw; g.D = D;
    g.M = m; g.N = n; g.K = k; g.lda = lda; g.ldb = k; g.ldd = n;
    g.in_dtype = VDK_DTYPE_BF16; g.out_dtype = VDK_DTYPE_BF16; g.epilogue = epi;
    g.bias = bias; g.gamma = gamma; g.residual = res; g.ldr = n; g.ln_eps = 1e-6f; g.split_k = 1;
    return gemm_run(g, s);
  };

  // ---- patch embedding + cls / position ----
  {
    __nv_bfloat16* rows = big;                                                        // [B*N, Kp]
    __nv_bfloat16* tok = big + (static_cast<size_t>(batch) * N * L.Kp + 127) / 128 * 128;  // [B*N, C]
    const int64_t total = static_cast<int64_t>(batch) * N * L.Kp;
    vit_patchify_kernel<<<static_cast<int>(std::min<int64_t>((total + 255) / 256, 148 * 32)), 256, 0, s>>>(images, batch, net->image_size,
                                                                                                         net->patch, L.Kp, rows);
    VDK_CUDA_OK(cudaGetLastError());
    rc = gemm(rows, net->patch_w, tok, batch * N, C, L.Kp, L.Kp, VDK_EPI_NONE, net->patch_b, nullptr, nullptr);
    if (rc != VDK_OK) return rc;
    const int64_t tot2 = static_cast<int64_t>(M) * (C / 2);
    vit_assemble_kernel<<<static_cast<int>(std::min<int64_t>((tot2 + 255) / 256, 148 * 32)), 256, 0, s>>>(tok, net->cls_token, net->pos_embed,
                                                                                                        batch, N, C, x);
    VDK_CUDA_OK(cudaGetLastError());
    if (net->norm_pre_w) {  // timm pre_norm=True (CLIP towers): LayerNorm over every token before the first block
      rc = launch_ln_patchify(x, batch, T, 1, C, net->norm_pre_w, net->norm_pre_b, eps, 1, y, nullptr, s);
      if (rc != VDK_OK) return rc;
      std::swap(x, y);
    }
  }
  // ---- blocks ----
  for (int i = 0; i < net->depth; ++i) {
    const vdk_vit_block* b = &net->blocks[i];
    VDK_REQUIRE(b->ln1_w && b->ln1_b && b->qkv_w && b->qkv_b && b->proj_w && b->proj_b && b->ln2_w && b->ln2_b && b->fc1_w &&
                    b->fc1_b && b->fc2_w && b->fc2_b,
                "vdk_vit_forward: null parameter in block %d", i);
    rc = launch_ln_patchify(x, batch, T, 1, C, b->ln1_w, b->ln1_b, eps, 1, y, nullptr, s);
    if (rc != VDK_OK) return rc;
    rc = gemm(y, b->qkv_w, big, M, 3 * C, C, C, VDK_EPI_NONE, b->qkv_b, nullptr, nullptr);
    if (rc != VDK_OK) return rc;
    rc = launch_attention(big, batch, T, net->heads, kAttD, y, nullptr, s);
    if (rc != VDK_OK) return rc;
    rc = gemm(y, b->proj_w, x, M, C, C, C, VDK_EPI_SCALE_RESIDUAL, b->proj_b, net->ones, x);  // x += proj(a), in place per tile
    if (rc != VDK_OK) return rc;
    rc = launch_ln_patchify(x, batch, T, 1, C, b->ln2_w, b->ln2_b, eps, 1, y, nullptr, s);
    if (rc != VDK_OK) return rc;
    rc = gemm(y, b->fc1_w, big, M, 4 * C, C, C, VDK_EPI_GELU, b->fc1_b, nullptr, nullptr);
    if (rc != VDK_OK) return rc;
    rc = gemm(big, b->fc2_w, x, M, C, 4 * C, 4 * C, VDK_EPI_SCALE_RESIDUAL, b->fc2_b, net->ones, x);
    if (rc != VDK_OK) return rc;
  }
  // ---- final LayerNorm, neck LayerNorm, Linear over (token, channel) with BatchNorm1d folded ----
  rc = launch_ln_patchify(x, batch, T, 1, C, net->norm_w, net->norm_b, eps, 1, y, nullptr, s);
  if (rc != VDK_OK) return rc;
  rc = launch_ln_patchify(y, batch, T, 1, C, net->neck_ln_w, net->neck_ln_b, 1e-5f, 1, x, nullptr, s);
  if (rc != VDK_OK) return rc;
  {
    const int Kn = T * C, F = net->feat_dim;
    const int tiles = ((batch + 127) / 128) * ((F + 255) / 256);
    const size_t slab = static_cast<size_t>(batch) * F;
    int split = std::max(1, std::min(64, (2 * sm_count()) / std::max(1, tiles)));
    split = vdk_gemm_effective_splits(Kn, split);
    float* slabs = reinterpret_cast<float*>(big);
    vdk_gemm_desc g{};
    g.A = x; g.B = net->neck_w; g.D = slabs;
    g.M = batch; g.N = F; g.K = Kn; g.lda = Kn; g.ldb = Kn; g.ldd = F;
    g.in_dtype = VDK_DTYPE_BF16; g.out_dtype = VDK_DTYPE_FP32; g.epilogue = VDK_EPI_NONE;
    g.split_k = split;
    g.split_stride = split > 1 ? static_cast<long long>(slab) : 0;
    rc = gemm_run(g, s);
    if (rc != VDK_OK) return rc;
    rc = launch_neck_finalize(slabs, split, slab, batch, F, net->neck_b, l2_normalize, embeddings, s);
    if (rc != VDK_OK) return rc;
  }
  return VDK_OK;
}

// ================================================================================================================
// ViT TRAINING: forward with saved activations, full backward (fp32 gradients accumulated in timm layouts)
// ================================================================================================================
// Replaces, for `timm-vit_*` backbones in train mode, TimmWrapper.forward (models/faceX/backbone/timm_wrapper.py:51-54; the
// Transformer neck :42-47 with BatchNorm1d on batch statistics) and its autograd backward inside
// `scaler.scale(loss).backward()` (engine/procedure/train.py:206).  BASELINE config 3 (ViT-B/16 + CircleLoss).
namespace vdk {

struct VitTrainLayout {
  int N, T, C, Kp, depth;
  size_t M;
  size_t rows, x0;                                   // patch rows [B*N, Kp], x after patch embed + cls + pos
  size_t y1[VDK_VIT_MAX_BLOCKS], r1[VDK_VIT_MAX_BLOCKS], qkv[VDK_VIT_MAX_BLOCKS], att[VDK_VIT_MAX_BLOCKS], lse[VDK_VIT_MAX_BLOCKS];
  size_t xm[VDK_VIT_MAX_BLOCKS], y2[VDK_VIT_MAX_BLOCKS], r2[VDK_VIT_MAX_BLOCKS], hpre[VDK_VIT_MAX_BLOCKS], hpost[VDK_VIT_MAX_BLOCKS];
  size_t xo[VDK_VIT_MAX_BLOCKS];                     // block outputs (residual stream)
  size_t f1, rf1, f2, rf2, z, zslab, bn_mean, bn_rstd;
  size_t dxa, dxb, dy, dbig, dz, dzb, gw, wslab, tok, dtok;
  size_t att_d;                                      // D = rowsum(dO * O) [batch, heads, T] of the tcgen05 attention backward
  size_t total;
};

static int vit_train_layout(const vdk_vit_net* n, int batch, VitTrainLayout* L) {
  VitLayout base;
  int rc = vit_layout(n, batch, &base);
  if (rc != VDK_OK) return rc;
  VDK_REQUIRE(base.Kp == 3 * n->patch * n->patch, "vdk_vit_train: 3*patch*patch must be a multiple of 8 (patch %d)", n->patch);
  VDK_REQUIRE(batch > 1, "vdk_vit_train: batch must be > 1 (BatchNorm1d batch statistics)");
  L->N = base.N; L->T = base.T; L->C = base.C; L->Kp = base.Kp; L->M = base.M; L->depth = n->depth;
  const size_t M = L->M, C = L->C, F = n->feat_dim;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += up256v(bytes); return o; };
  L->rows = take(static_cast<size_t>(batch) * L->N * L->Kp * 2);
  L->tok = take(static_cast<size_t>(batch) * L->N * C * 2);
  L->x0 = take(M * C * 2);
  for (int i = 0; i < n->depth; ++i) {
    L->y1[i] = take(M * C * 2);  L->r1[i] = take(M * 4);
    L->qkv[i] = take(M * 3 * C * 2);
    L->att[i] = take(M * C * 2); L->lse[i] = take(static_cast<size_t>(batch) * n->heads * L->T * 4);
    L->xm[i] = take(M * C * 2);
    L->y2[i] = take(M * C * 2);  L->r2[i] = take(M * 4);
    L->hpre[i] = take(M * 4 * C * 2);
    L->hpost[i] = take(M * 4 * C * 2);
    L->xo[i] = take(M * C * 2);
  }
  L->f1 = take(M * C * 2); L->rf1 = take(M * 4);
  L->f2 = take(M * C * 2); L->rf2 = take(M * 4);
  L->z = take(static_cast<size_t>(batch) * F * 4);
  L->zslab = take(static_cast<size_t>(batch) * F * 4 * 64);
  L->bn_mean = take(F * 4); L->bn_rstd = take(F * 4);
  // backward scratch
  L->dxa = take(M * C * 2); L->dxb = take(M * C * 2); L->dy = take(M * C * 2);
  L->dbig = take(M * 4 * C * 2);
  L->dz = take(static_cast<size_t>(batch) * F * 4); L->dzb = take(static_cast<size_t>(batch) * F * 2);
  L->gw = take(F * static_cast<size_t>(L->T) * C * 4);
  L->dtok = take(static_cast<size_t>(batch) * L->N * C * 2);
  L->att_d = take(static_cast<size_t>(batch) * n->heads * L->T * 4);
  size_t slab = wgrad_slab_bytes(static_cast<int>(C), L->Kp, static_cast<size_t>(batch) * L->N);
  slab = std::max(slab, wgrad_slab_bytes(static_cast<int>(3 * C), static_cast<int>(C), M));
  slab = std::max(slab, wgrad_slab_bytes(static_cast<int>(C), static_cast<int>(C), M));
  slab = std::max(slab, wgrad_slab_bytes(static_cast<int>(4 * C), static_cast<int>(C), M));
  slab = std::max(slab, wgrad_slab_bytes(static_cast<int>(C), static_cast<int>(4 * C), M));
  L->wslab = take(slab);
  L->total = off + 256;
  return VDK_OK;
}

__global__ void vit_slab_bias_kernel(const float* __restrict__ slabs, int n_slabs, size_t stride, const float* __restrict__ bias, int rows,
                                     int cols, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  float v = bias[i % cols];
  for (int s = 0; s < n_slabs; ++s) v += slabs[s * stride + i];
  out[i] = v;
}
__global__ void vit_colsum_f32_kernel(const float* __restrict__ x, int rows, int cols, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  float s = 0.f;
  for (int r = 0; r < rows; ++r) s += x[static_cast<size_t>(r) * cols + c];
  out[c] += s;
}
// backward of vit_assemble: dtok[b, i] = dx[b, 1 + i];  dpos[t] += sum_b dx[b, t];  dcls += sum_b dx[b, 0]
__global__ void __launch_bounds__(256)
vit_assemble_bwd_kernel(const __nv_bfloat16* __restrict__ dx, int B, int N, int C, __nv_bfloat16* __restrict__ dtok,
                        float* __restrict__ dpos, float* __restrict__ dcls) {
  const int64_t total = static_cast<int64_t>(N + 1) * C;  // one thread per (token, channel), loop over the batch
  for (int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(t % C), tk = static_cast<int>(t / C);
    float s = 0.f;
    for (int b = 0; b < B; ++b) {
      const __nv_bfloat16 v = dx[(static_cast<int64_t>(b) * (N + 1) + tk) * C + c];
      s += __bfloat162float(v);
      if (tk > 0) dtok[(static_cast<int64_t>(b) * N + tk - 1) * C + c] = v;
    }
    dpos[t] += s;
    if (tk == 0) dcls[c] += s;
  }
}

}  // namespace vdk

extern "C" int vdk_vit_pack(const vdk_vit_tensors* p, vdk_vit_net* net, void* stream) {
  VDK_REQUIRE(p && net, "vdk_vit_pack: null argument");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  VitLayout L;
  RC(vit_layout(net, 2, &L));
  VDK_REQUIRE(L.Kp == 3 * net->patch * net->patch, "vdk_vit_pack: 3*patch*patch must be a multiple of 8");
  auto bf = [](const void* q) { return reinterpret_cast<__nv_bfloat16*>(const_cast<void*>(q)); };
  const int64_t C = net->dim;
  RC(launch_cast_bf16(p->patch_w, C * L.Kp, bf(net->patch_w), s));
  for (int i = 0; i < net->depth; ++i) {
    const vdk_vit_block_tensors* b = &p->blocks[i];
    const vdk_vit_block* o = &net->blocks[i];
    RC(launch_cast_bf16(b->qkv_w, 3 * C * C, bf(o->qkv_w), s));
    RC(launch_cast_bf16(b->proj_w, C * C, bf(o->proj_w), s));
    RC(launch_cast_bf16(b->fc1_w, 4 * C * C, bf(o->fc1_w), s));
    RC(launch_cast_bf16(b->fc2_w, 4 * C * C, bf(o->fc2_w), s));
  }
  RC(launch_cast_bf16(p->lin_w, static_cast<int64_t>(net->feat_dim) * L.T * C, bf(net->neck_w), s));
  return VDK_OK;
}

extern "C" size_t vdk_vit_train_workspace_bytes(const vdk_vit_net* net, int batch) {
  VitTrainLayout L;
  if (!net || batch <= 1 || vit_train_layout(net, batch, &L) != VDK_OK) return 0;
  return L.total;
}

static int refuse_pre_norm(const vdk_vit_net* net) {
  VDK_REQUIRE(net && net->norm_pre_w == nullptr && !(net->ln_eps > 0.f && net->ln_eps != 1e-6f),
              "vdk_vit_train: pre_norm / non-default LayerNorm eps variants (CLIP towers) are built for inference only");
  return VDK_OK;
}

extern "C" int vdk_vit_train_forward(const vdk_vit_net* net, const vdk_vit_tensors* p, const float* images, int batch,
                                     float bn_momentum, float* out_feats, void* workspace, size_t workspace_bytes, void* stream) {
  VDK_REQUIRE(net && p && images && out_feats, "vdk_vit_train_forward: null argument");
  RC(refuse_pre_norm(net));
  VitTrainLayout L;
  RC(vit_train_layout(net, batch, &L));
  VDK_REQUIRE(workspace && workspace_bytes >= L.total && (reinterpret_cast<uintptr_t>(workspace) & 255) == 0,
              "vdk_vit_train_forward: workspace too small or misaligned");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  auto B16 = [&](size_t off) { return reinterpret_cast<__nv_bfloat16*>(ws + off); };
  auto F32 = [&](size_t off) { return reinterpret_cast<float*>(ws + off); };
  const Gemm G{s};
  const int C = L.C, T = L.T, N = L.N, M = static_cast<int>(L.M), F = net->feat_dim;

  {
    const int64_t total = static_cast<int64_t>(batch) * N * L.Kp;
    vit_patchify_kernel<<<static_cast<int>(std::min<int64_t>((total + 255) / 256, 148 * 32)), 256, 0, s>>>(images, batch, net->image_size,
                                                                                                         net->patch, L.Kp, B16(L.rows));
    VDK_CUDA_OK(cudaGetLastError());
    RC(G.run(B16(L.rows), net->patch_w, B16(L.tok), batch * N, C, L.Kp, L.Kp, L.Kp, C, VDK_EPI_NONE, net->patch_b, nullptr, nullptr, 0,
             VDK_DTYPE_BF16, 1, 0, 0, 0));
    const int64_t tot2 = static_cast<int64_t>(M) * (C / 2);
    vit_assemble_kernel<<<static_cast<int>(std::min<int64_t>((tot2 + 255) / 256, 148 * 32)), 256, 0, s>>>(B16(L.tok), net->cls_token,
                                                                                                        net->pos_embed, batch, N, C, B16(L.x0));
    VDK_CUDA_OK(cudaGetLastError());
  }
  const __nv_bfloat16* x = B16(L.x0);
  for (int i = 0; i < net->depth; ++i) {
    const vdk_vit_block* b = &net->blocks[i];
    RC(launch_ln_patchify(x, batch, T, 1, C, b->ln1_w, b->ln1_b, 1e-6f, 1, B16(L.y1[i]), F32(L.r1[i]), s));
    RC(G.run(B16(L.y1[i]), b->qkv_w, B16(L.qkv[i]), M, 3 * C, C, C, C, 3 * C, VDK_EPI_NONE, b->qkv_b, nullptr, nullptr, 0, VDK_DTYPE_BF16,
             1, 0, 0, 0));
    RC(launch_attention(B16(L.qkv[i]), batch, T, net->heads, kAttD, B16(L.att[i]), F32(L.lse[i]), s));
    RC(G.run(B16(L.att[i]), b->proj_w, B16(L.xm[i]), M, C, C, C, C, C, VDK_EPI_SCALE_RESIDUAL, b->proj_b, net->ones, x, C, VDK_DTYPE_BF16,
             1, 0, 0, 0));
    RC(launch_ln_patchify(B16(L.xm[i]), batch, T, 1, C, b->ln2_w, b->ln2_b, 1e-6f, 1, B16(L.y2[i]), F32(L.r2[i]), s));
    RC(G.run(B16(L.y2[i]), b->fc1_w, B16(L.hpost[i]), M, 4 * C, C, C, C, 4 * C, VDK_EPI_GELU, b->fc1_b, nullptr, nullptr, 0, VDK_DTYPE_BF16,
             1, 0, 0, 0, B16(L.hpre[i])));
    RC(G.run(B16(L.hpost[i]), b->fc2_w, B16(L.xo[i]), M, C, 4 * C, 4 * C, 4 * C, C, VDK_EPI_SCALE_RESIDUAL, b->fc2_b, net->ones,
             B16(L.xm[i]), C, VDK_DTYPE_BF16, 1, 0, 0, 0));
    x = B16(L.xo[i]);
  }
  RC(launch_ln_patchify(x, batch, T, 1, C, net->norm_w, net->norm_b, 1e-6f, 1, B16(L.f1), F32(L.rf1), s));
  RC(launch_ln_patchify(B16(L.f1), batch, T, 1, C, net->neck_ln_w, net->neck_ln_b, 1e-5f, 1, B16(L.f2), F32(L.rf2), s));
  {
    const int Kn = T * C;
    const int tiles = ((batch + 127) / 128) * ((F + 255) / 256);
    int split = std::max(1, std::min(64, (2 * sm_count()) / std::max(1, tiles)));
    split = vdk_gemm_effective_splits(Kn, split);
    const size_t slab = static_cast<size_t>(batch) * F;
    RC(G.run(B16(L.f2), net->neck_w, F32(L.zslab), batch, F, Kn, Kn, Kn, F, VDK_EPI_NONE, nullptr, nullptr, nullptr, 0, VDK_DTYPE_FP32, split,
             split > 1 ? static_cast<long long>(slab) : 0, 0, 0));
    vit_slab_bias_kernel<<<(batch * F + 255) / 256, 256, 0, s>>>(F32(L.zslab), split, slab, p->lin_b, batch, F, F32(L.z));
    VDK_CUDA_OK(cudaGetLastError());
    RC(launch_bn_fwd_f32(F32(L.z), batch, F, p->bn1_w, p->bn1_b, 1e-5f, bn_momentum, out_feats, F32(L.bn_mean), F32(L.bn_rstd),
                         p->bn1_running_mean, p->bn1_running_var, s));
  }
  return VDK_OK;
}

// Units of the backward in execution order: 0 = neck + final LayerNorm; 1 .. depth = blocks depth-1 .. 0; depth + 1 = cls / position /
// patch embedding.  Consecutive ranges let the caller overlap the DDP all-reduce of finished gradients with the rest.
extern "C" int vdk_vit_train_backward_units(const vdk_vit_net* net) { return net ? net->depth + 2 : 0; }

static int vit_backward_range(const vdk_vit_net* net, const vdk_vit_tensors* p, const vdk_vit_tensors* g, const float* d_feats, int batch,
                              void* workspace, size_t workspace_bytes, void* stream, int u_begin, int u_end) {
  VDK_REQUIRE(net && p && g && d_feats, "vdk_vit_train_backward: null argument");
  VDK_REQUIRE(u_begin >= 0 && u_begin < u_end && u_end <= net->depth + 2, "vdk_vit_train_backward: bad unit range [%d, %d)", u_begin, u_end);
  auto active = [&](int unit) { return unit >= u_begin && unit < u_end; };
  VitTrainLayout L;
  RC(vit_train_layout(net, batch, &L));
  VDK_REQUIRE(workspace && workspace_bytes >= L.total, "vdk_vit_train_backward: workspace too small");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  auto B16 = [&](size_t off) { return reinterpret_cast<__nv_bfloat16*>(ws + off); };
  auto F32 = [&](size_t off) { return reinterpret_cast<float*>(ws + off); };
  const Gemm G{s};
  const int C = L.C, T = L.T, N = L.N, M = static_cast<int>(L.M), F = net->feat_dim, Kn = T * C;
  float* slabs = F32(L.wslab);

  // ---- neck: BatchNorm1d (batch statistics) <- Linear <- LayerNorm(neck) <- LayerNorm(final) ----
  if (active(0)) {
  RC(launch_bn_bwd_f32(d_feats, F32(L.z), batch, F, p->bn1_w, F32(L.bn_mean), F32(L.bn_rstd), F32(L.dz), g->bn1_w, g->bn1_b, s));
  vit_colsum_f32_kernel<<<(F + 255) / 256, 256, 0, s>>>(F32(L.dz), batch, F, g->lin_b);
  VDK_CUDA_OK(cudaGetLastError());
  RC(launch_cast_bf16(F32(L.dz), static_cast<int64_t>(batch) * F, B16(L.dzb), s));
  // dW[F, Kn] = dZ^T . f2 (contraction over the batch): plain stores into scratch, then += into the gradient
  RC(G.run(B16(L.dzb), B16(L.f2), F32(L.gw), F, Kn, batch, F, Kn, Kn, VDK_EPI_NONE, nullptr, nullptr, nullptr, 0, VDK_DTYPE_FP32, 1, 0, 1, 1));
  RC(launch_add_f32(g->lin_w, F32(L.gw), static_cast<int64_t>(F) * Kn, s));
  // df2[B, Kn] = dZ . W
  RC(G.run(B16(L.dzb), net->neck_w, B16(L.dy), batch, Kn, F, F, Kn, Kn, VDK_EPI_NONE, nullptr, nullptr, nullptr, 0, VDK_DTYPE_BF16, 1, 0, 0, 1));
  RC(launch_ln_bwd(B16(L.dy), B16(L.f2), F32(L.rf2), batch, T, 1, C, net->neck_ln_w, net->neck_ln_b, 1, B16(L.dxb), nullptr, g->neck_ln_w,
                   g->neck_ln_b, s));
  RC(launch_ln_bwd(B16(L.dxb), B16(L.f1), F32(L.rf1), batch, T, 1, C, net->norm_w, net->norm_b, 1, B16(L.dxa), nullptr, g->norm_w, g->norm_b, s));
  }
  // the residual-stream gradient ping-pongs between two buffers; every block swaps them twice, so it enters and leaves each
  // block in dxa and skipped units need no bookkeeping
  size_t dx = L.dxa, dx_other = L.dxb;
  // ---- blocks ----
  for (int i = net->depth - 1; i >= 0; --i) {
    if (!active(1 + (net->depth - 1 - i))) continue;
    const vdk_vit_block* b = &net->blocks[i];
    const vdk_vit_block_tensors* gb = &g->blocks[i];
    // MLP: x_out = x_mid + fc2(gelu(fc1(LN2(x_mid))))
    RC(launch_col_sum(B16(dx), M, C, C, gb->fc2_b, s));
    RC(G.wgrad(B16(dx), B16(L.hpost[i]), gb->fc2_w, C, 4 * C, M, C, 4 * C, slabs, true));
    RC(G.run(B16(dx), b->fc2_w, B16(L.dbig), M, 4 * C, C, C, 4 * C, 4 * C, VDK_EPI_MUL_GELU_GRAD, nullptr, nullptr, B16(L.hpre[i]), 4 * C,
             VDK_DTYPE_BF16, 1, 0, 0, 1));
    RC(launch_col_sum(B16(L.dbig), M, 4 * C, 4 * C, gb->fc1_b, s));
    RC(G.wgrad(B16(L.dbig), B16(L.y2[i]), gb->fc1_w, 4 * C, C, M, 4 * C, C, slabs, true));
    RC(G.run(B16(L.dbig), b->fc1_w, B16(L.dy), M, C, 4 * C, 4 * C, C, C, VDK_EPI_NONE, nullptr, nullptr, nullptr, 0, VDK_DTYPE_BF16, 1, 0, 0, 1));
    RC(launch_ln_bwd(B16(L.dy), B16(L.y2[i]), F32(L.r2[i]), batch, T, 1, C, b->ln2_w, b->ln2_b, 1, B16(dx_other), B16(dx), gb->ln2_w,
                     gb->ln2_b, s));  // d x_mid = LN2 backward + the residual branch
    std::swap(dx, dx_other);
    // attention: x_mid = x_in + proj(attn(qkv(LN1(x_in))))
    RC(launch_col_sum(B16(dx), M, C, C, gb->proj_b, s));
    RC(G.wgrad(B16(dx), B16(L.att[i]), gb->proj_w, C, C, M, C, C, slabs, true));
    RC(G.run(B16(dx), b->proj_w, B16(L.dy), M, C, C, C, C, C, VDK_EPI_NONE, nullptr, nullptr, nullptr, 0, VDK_DTYPE_BF16, 1, 0, 0, 1));
    // up to 208 tokens (ViT-*/16 at 224^2) the mma.sync kernel that holds a head's whole P in shared memory; beyond, the tcgen05 pair
    if (T <= kAttBwdMaxRows)
      RC(launch_attention_bwd(B16(L.qkv[i]), B16(L.att[i]), B16(L.dy), F32(L.lse[i]), batch, T, net->heads, kAttD, B16(L.dbig), s));
    else
      RC(launch_attention_bwd_pair(B16(L.qkv[i]), B16(L.att[i]), B16(L.dy), F32(L.lse[i]), batch, T, net->heads, kAttD, B16(L.dbig),
                                   ws + L.att_d, up256v(static_cast<size_t>(batch) * net->heads * T * 4), s));
    RC(launch_col_sum(B16(L.dbig), M, 3 * C, 3 * C, gb->qkv_b, s));
    RC(G.wgrad(B16(L.dbig), B16(L.y1[i]), gb->qkv_w, 3 * C, C, M, 3 * C, C, slabs, true));
    RC(G.run(B16(L.dbig), b->qkv_w, B16(L.dy), M, C, 3 * C, 3 * C, C, C, VDK_EPI_NONE, nullptr, nullptr, nullptr, 0, VDK_DTYPE_BF16, 1, 0, 0, 1));
    RC(launch_ln_bwd(B16(L.dy), B16(L.y1[i]), F32(L.r1[i]), batch, T, 1, C, b->ln1_w, b->ln1_b, 1, B16(dx_other), B16(dx), gb->ln1_w,
                     gb->ln1_b, s));
    std::swap(dx, dx_other);
  }
  // ---- cls / position embeddings, patch embedding ----
  if (active(net->depth + 1)) {
    const int64_t tot = static_cast<int64_t>(T) * C;
    vit_assemble_bwd_kernel<<<static_cast<int>(std::min<int64_t>((tot + 255) / 256, 148 * 8)), 256, 0, s>>>(B16(dx), batch, N, C, B16(L.dtok),
                                                                                                           g->pos_embed, g->cls_token);
    VDK_CUDA_OK(cudaGetLastError());
    RC(launch_col_sum(B16(L.dtok), static_cast<int64_t>(batch) * N, C, C, g->patch_b, s));
    RC(G.wgrad(B16(L.dtok), B16(L.rows), g->patch_w, C, L.Kp, batch * N, C, L.Kp, slabs, true));
  }
  return VDK_OK;
}

extern "C" int vdk_vit_train_backward(const vdk_vit_net* net, const vdk_vit_tensors* p, const vdk_vit_tensors* g, const float* d_feats,
                                      int batch, void* workspace, size_t workspace_bytes, void* stream) {
  VDK_REQUIRE(net, "vdk_vit_train_backward: null net");
  return vit_backward_range(net, p, g, d_feats, batch, workspace, workspace_bytes, stream, 0, net->depth + 2);
}

extern "C" int vdk_vit_train_backward_range(const vdk_vit_net* net, const vdk_vit_tensors* p, const vdk_vit_tensors* g,
                                            const float* d_feats, int batch, void* workspace, size_t workspace_bytes, void* stream,
                                            int unit_begin, int unit_end) {
  VDK_REQUIRE(net, "vdk_vit_train_backward_range: null net");
  return vit_backward_range(net, p, g, d_feats, batch, workspace, workspace_bytes, stream, unit_begin, unit_end);
}

