// attention_bwd_tc.cu — the backward of softmax(Q K^T / 8) V on the 5th-generation tensor cores (tcgen05), head_dim 64, bf16, any
// token count.
//
// Replaces timm's Attention backward inside `scaler.scale(loss).backward()` (engine/procedure/train.py:206) for sequences longer
// than the 208 tokens the mma.sync kernel of vit.cu holds in shared memory (ViT-*/8 at 224^2: 785 tokens; ViT-*/16 at 384^2: 577).
// Inputs as the forward left them: qkv bf16 [B, N, 3, H, 64], out / d_out bf16 [B, N, H*64], lse2 fp32 [B, H, N] (log2 domain);
// output dqkv bf16 [B, N, 3, H, 64].  With scale = 1/8 and c = scale * log2(e):
//   P = exp2(c S - lse2),  S = Q K^T;   D_i = sum_d dO_id O_id;   dS = scale * P (dO V^T - D)
//   dV = P^T dO;   dQ = dS K;   dK = dS^T Q
// Scores, probabilities and dS live in TMEM and shared memory only.  P and dS are rounded to bf16 before they feed a product, as in
// the mma.sync kernel.  No atomics: every dqkv element is written once, by one CTA, after a fixed-order sum, so the result is the
// same bits on every run.  That costs two products more than an atomic-dQ design: 7 MMAs per (query tile, key tile) here, i.e.
// 14 N^2 64 flops executed per (image, head) against the algorithmic 10 N^2 64.
//
// Two persistent kernels on the same stream, 192 threads each: warps 0-3 epilogue (TMEM lane = the tile row this thread owns),
// warp 4 TMA producer, warp 5 tcgen05.mma issuer.  An item is one (image, head, 128-row tile); items are strided over the grid.
//
// Kernel Q (dQ).  Q and dO of one 128-query tile stay resident; 128-key K / V tiles stream through a two-deep ring.  The epilogue
// first computes D for its row (written to the [B, H, N] workspace for kernel KV).  Per key tile j:
//   MMA  S = Q K_j^T (128x128x64, both K-major)          -> TMEM cols [0, 128)
//   MMA  dP = dO V_j^T (128x128x64, both K-major)        -> TMEM cols [128, 256)
//   epilogue: dS = scale * bf16(P) (dP - D) -> bf16 -> shared memory (K-major, 128-byte swizzle, two 64-key halves)
//   MMA  dQ += dS K_j (128x64x128, K as stored = MN-major) -> TMEM cols [256, 320)
// Kernel KV (dK, dV).  K and V of one 128-key tile stay resident; 128-query Q / dO tiles stream.  Per query tile i:
//   MMA  S^T = K Q_i^T                                   -> TMEM cols [0, 128)
//   MMA  dP^T = V dO_i^T                                 -> TMEM cols [128, 256)
//   epilogue: P^T and dS^T (lse2 and D of the 128 queries staged in shared memory) -> bf16 -> shared memory
//   MMA  dV += P^T dO_i (128x64x128, dO MN-major)        -> TMEM cols [256, 320)
//   MMA  dK += dS^T Q_i (128x64x128, Q MN-major)         -> TMEM cols [320, 384)
// TMEM: 320 (Q) / 384 (KV) columns, allocated as 512.  Ordering: the tensor core runs one thread's MMAs in issue order, so the
// commit that publishes S / dP of tile j also covers the dQ (dV, dK) product of tile j-1 that read the bf16 tile in shared memory:
// the epilogue overwrites that tile only after it has seen the S of tile j.  Rows and key / query columns beyond N are read as
// zero by TMA and their P is set to exactly 0 (lse2 and D beyond N are never read); only rows < N of dqkv are written.
#include "vdk_host.h"
#include "vdk_ptx.cuh"

#include <algorithm>
#include <cmath>

namespace vdk {

constexpr int kBtD = 64;                      // head dim
constexpr int kBtM = 128;                     // tile rows (TMEM lanes) and streamed tile rows
constexpr int kBtThreads = 192;
constexpr int kBtTile = kBtM * kBtD * 2;      // 16 KB: a 128 x 64 bf16 tile
constexpr int kBtStages = 2;                  // streamed ring: [stage][two 16 KB tiles]
constexpr uint32_t kBtTmemCols = 512;
constexpr int kBtSmemQ = 2 * kBtTile + kBtStages * 2 * kBtTile + 2 * kBtTile + 256 + 1024;
constexpr int kBtSmemKV = 2 * kBtTile + kBtStages * 2 * kBtTile + 4 * kBtTile + 2 * 2 * kBtM * 4 + 256 + 1024;
static_assert(kBtSmemKV <= 227 * 1024, "attention backward shared memory budget");

struct AttBwdParams {
  int B, N, H, n_tiles;
  float scale, scale_log2e;
  const __nv_bfloat16* out;
  const __nv_bfloat16* d_out;
  const float* lse2;
  float* D;  // [B, H, N]: written by kernel Q, read by kernel KV
  __nv_bfloat16* dqkv;
};

__device__ __forceinline__ float bt_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t bt_pack(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ float bt_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bt_hi(uint32_t w) { return __uint_as_float(w & 0xFFFF0000u); }

// One 32-column chunk c (0..3) of a 128-column bf16 row into a K-major, 128-byte-swizzled [128 rows][128] tile stored as two
// [128][64] halves of 16 KB each.
__device__ __forceinline__ void bt_store_chunk(uint8_t* tile, int r, int c, const uint32_t (&pk)[16]) {
  uint8_t* row = tile + (c >> 1) * kBtTile + r * 128;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int chunk = (c & 1) * 4 + q;
    *reinterpret_cast<uint4*>(row + ((chunk ^ (r & 7)) << 4)) = make_uint4(pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
  }
}

// 64 fp32 accumulator columns of this thread's TMEM lane -> 64 bf16 at dst (skipped, but still loaded, for rows beyond N)
__device__ __forceinline__ void bt_store_acc(uint32_t taddr, __nv_bfloat16* dst, bool ok) {
#pragma unroll
  for (int hc = 0; hc < 2; ++hc) {
    uint32_t v[32];
    tmem_ld_32x32b_x32(taddr + hc * 32, v);
    tmem_ld_wait();
    if (ok) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint4 w;
        w.x = bt_pack(__uint_as_float(v[8 * q]), __uint_as_float(v[8 * q + 1]));
        w.y = bt_pack(__uint_as_float(v[8 * q + 2]), __uint_as_float(v[8 * q + 3]));
        w.z = bt_pack(__uint_as_float(v[8 * q + 4]), __uint_as_float(v[8 * q + 5]));
        w.w = bt_pack(__uint_as_float(v[8 * q + 6]), __uint_as_float(v[8 * q + 7]));
        *reinterpret_cast<uint4*>(dst + hc * 32 + q * 8) = w;
      }
    }
  }
}

// 128x128x64: D[tmem] = A[128 rows] B[128 rows]^T, both K-major 16 KB tiles
__device__ __forceinline__ void bt_mma_nt(uint32_t d, const uint8_t* a, const uint8_t* b) {
  constexpr uint32_t idesc = umma_idesc_f16<true>(kBtM, kBtM);
  const uint64_t da = umma_desc_k_sw128(smem_u32(a)), db = umma_desc_k_sw128(smem_u32(b));
#pragma unroll
  for (int k = 0; k < kBtD / 16; ++k) umma_f16_ss(d, da + 2 * k, db + 2 * k, idesc, k > 0 ? 1u : 0u);
}
// 128x64x128: D[tmem] (+)= A[128 x 128, K-major, two 64-column halves] B, B = a [128 contraction rows][64] tile as stored (MN-major)
__device__ __forceinline__ void bt_mma_nn(uint32_t d, const uint8_t* a, const uint8_t* b, bool accumulate) {
  constexpr uint32_t idesc = umma_idesc_f16<true>(kBtM, kBtD, 0u, 1u);
  const uint64_t db = umma_desc_mn_sw128(smem_u32(b), 8192);
#pragma unroll
  for (int k = 0; k < kBtM / 16; ++k) {
    const uint64_t da = umma_desc_k_sw128(smem_u32(a + (k >> 2) * kBtTile)) + 2 * (k & 3);
    umma_f16_ss(d, da, db + 128u * k, idesc, (accumulate || k > 0) ? 1u : 0u);
  }
}

__device__ __forceinline__ void bt_decode(const AttBwdParams& p, int item, int& t, int& h, int& b) {
  t = item % p.n_tiles;
  const int r = item / p.n_tiles;
  h = r % p.H;
  b = r / p.H;
}

// ===================================================================================================================
// kernel Q: dQ (and D)
// ===================================================================================================================
__global__ void __launch_bounds__(kBtThreads, 1)
attention_bwd_dq_tc_kernel(const __grid_constant__ CUtensorMap map_qkv, const __grid_constant__ CUtensorMap map_do, const AttBwdParams p) {
  extern __shared__ uint8_t bt_smem_raw[];
  uint8_t* smem = bt_smem_raw + ((1024u - (smem_u32(bt_smem_raw) & 1023u)) & 1023u);
  uint8_t* s_q = smem;                                  // Q tile, then dO tile
  uint8_t* s_do = s_q + kBtTile;
  uint8_t* s_kv = s_do + kBtTile;                       // [stage][K | V]
  uint8_t* s_ds = s_kv + kBtStages * 2 * kBtTile;       // dS: [2 halves][128][64]
  uint64_t* q_full = reinterpret_cast<uint64_t*>(s_ds + 2 * kBtTile);
  uint64_t* q_empty = q_full + 1;
  uint64_t* kv_full = q_empty + 1;             // [stages]
  uint64_t* kv_empty = kv_full + kBtStages;    // [stages]
  uint64_t* s_full = kv_empty + kBtStages;     // S and dP of the current key tile are in TMEM
  uint64_t* ds_full = s_full + 1;              // dS is in shared memory and S / dP have been read (4 warp arrivals)
  uint64_t* dq_full = ds_full + 1;             // the item's dQ is final in TMEM
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(dq_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int J = p.n_tiles, N = p.N;
  const int n_items = p.n_tiles * p.H * p.B;

  if (threadIdx.x == 0) {
    prefetch_tensormap(&map_qkv);
    prefetch_tensormap(&map_do);
    mbar_init(q_full, 1);
    mbar_init(q_empty, 1);
    for (int i = 0; i < kBtStages; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(ds_full, 4);
    mbar_init(dq_full, 1);
    fence_mbar_init();
  }
  if (warp == 5) tmem_alloc<kBtTmemCols>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 4) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int ic = 0, kvc = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++ic) {
        int qt, h, b;
        bt_decode(p, item, qt, h, b);
        if (ic >= 1) mbar_wait_relaxed(q_empty, (ic - 1) & 1);  // every MMA that read the previous item's Q / dO has retired
        mbar_arrive_expect_tx(q_full, 2 * kBtTile);
        tma_load_3d(s_q, &map_qkv, q_full, h * kBtD, qt * kBtM, b);
        tma_load_3d(s_do, &map_do, q_full, h * kBtD, qt * kBtM, b);
        for (int j = 0; j < J; ++j, ++kvc) {
          const int st = kvc % kBtStages;
          if (kvc >= kBtStages) mbar_wait_relaxed(&kv_empty[st], ((kvc / kBtStages) - 1) & 1);
          mbar_arrive_expect_tx(&kv_full[st], 2 * kBtTile);
          tma_load_3d(s_kv + st * 2 * kBtTile, &map_qkv, &kv_full[st], (p.H + h) * kBtD, j * kBtM, b);
          tma_load_3d(s_kv + st * 2 * kBtTile + kBtTile, &map_qkv, &kv_full[st], (2 * p.H + h) * kBtD, j * kBtM, b);
        }
      }
    }
  } else if (warp == 5) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t t_s = tmem_base, t_dp = tmem_base + kBtM, t_dq = tmem_base + 2 * kBtM;
      int ic = 0, kvc = 0, g = 0;  // items, K/V tiles, (item, key tile) pairs so far
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++ic) {
        mbar_wait(q_full, ic & 1);
        tc_fence_after();
        for (int j = 0; j < J; ++j, ++g) {
          const int st = (kvc + j) % kBtStages;
          mbar_wait(&kv_full[st], ((kvc + j) / kBtStages) & 1);
          tc_fence_after();
          if (j > 0) {  // dS of the previous key tile is in shared memory, and S / dP of TMEM have been read
            const int pst = (kvc + j - 1) % kBtStages;
            mbar_wait(ds_full, (g - 1) & 1);
            tc_fence_after();
            bt_mma_nn(t_dq, s_ds, s_kv + pst * 2 * kBtTile, j > 1);
            umma_commit(&kv_empty[pst]);
          }
          bt_mma_nt(t_s, s_q, s_kv + st * 2 * kBtTile);
          bt_mma_nt(t_dp, s_do, s_kv + st * 2 * kBtTile + kBtTile);
          umma_commit(s_full);
          if (j + 1 == J) umma_commit(q_empty);
        }
        mbar_wait(ds_full, (g - 1) & 1);
        tc_fence_after();
        const int lst = (kvc + J - 1) % kBtStages;
        bt_mma_nn(t_dq, s_ds, s_kv + lst * 2 * kBtTile, J > 1);
        umma_commit(&kv_empty[lst]);
        umma_commit(dq_full);
        kvc += J;
      }
    }
  } else {
    // ===================== epilogue: one query row per thread =====================
    const int lane_base = warp * 32, r = lane_base + lane;
    const uint32_t lane_off = static_cast<uint32_t>(lane_base) << 16;
    const uint32_t t_s = tmem_base + lane_off, t_dp = t_s + kBtM, t_dq = t_s + 2 * kBtM;
    const size_t ld = static_cast<size_t>(p.H) * kBtD;
    int ic = 0, g = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++ic) {
      int qt, h, b;
      bt_decode(p, item, qt, h, b);
      const int row = qt * kBtM + r;
      const bool rv = row < N;
      const size_t bh = static_cast<size_t>(b) * p.H + h;
      // D = rowsum(dO * O) in fp32 from the bf16 tensors; lse2 of this row (rows beyond N: never read, D = lse = 0)
      float Dr = 0.f, lse = 0.f;
      if (rv) {
        const uint4* o4 = reinterpret_cast<const uint4*>(p.out + (static_cast<size_t>(b) * N + row) * ld + h * kBtD);
        const uint4* d4 = reinterpret_cast<const uint4*>(p.d_out + (static_cast<size_t>(b) * N + row) * ld + h * kBtD);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const uint4 a = __ldg(o4 + c), d = __ldg(d4 + c);
          const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, dw[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) Dr = fmaf(bt_lo(aw[k]), bt_lo(dw[k]), fmaf(bt_hi(aw[k]), bt_hi(dw[k]), Dr));
        }
        p.D[bh * N + row] = Dr;
        lse = p.lse2[bh * N + row];
      }
      for (int j = 0; j < J; ++j, ++g) {
        mbar_wait(s_full, g & 1);
        tc_fence_after();
        const int valid = rv ? min(kBtM, N - j * kBtM) : 0;  // key columns of this tile whose P is computed
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          uint32_t sv[32], dp[32], pk[16];
          tmem_ld_32x32b_x32(t_s + c * 32, sv);
          tmem_ld_32x32b_x32(t_dp + c * 32, dp);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            const int col = c * 32 + i;
            const float p0 = col < valid ? bt_ex2(__uint_as_float(sv[i]) * p.scale_log2e - lse) : 0.f;
            const float p1 = col + 1 < valid ? bt_ex2(__uint_as_float(sv[i + 1]) * p.scale_log2e - lse) : 0.f;
            const uint32_t pb = bt_pack(p0, p1);  // P rounded to bf16 as the mma.sync kernel stores it
            pk[i >> 1] = bt_pack(p.scale * bt_lo(pb) * (__uint_as_float(dp[i]) - Dr),
                                 p.scale * bt_hi(pb) * (__uint_as_float(dp[i + 1]) - Dr));
          }
          bt_store_chunk(s_ds, r, c, pk);
        }
        tc_fence_before();
        fence_proxy_async_smem();  // generic-proxy stores of dS -> visible to the tensor core's async proxy
        __syncwarp();
        if (lane == 0) mbar_arrive(ds_full);
      }
      mbar_wait(dq_full, ic & 1);
      tc_fence_after();
      bt_store_acc(t_dq, p.dqkv + ((static_cast<size_t>(b) * N + (rv ? row : 0)) * 3) * ld + h * kBtD, rv);
      tc_fence_before();  // dQ is read before the next item's first ds_full lets its first dQ product overwrite it
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    tmem_dealloc<kBtTmemCols>(tmem_base);
  }
}

// ===================================================================================================================
// kernel KV: dK, dV
// ===================================================================================================================
__global__ void __launch_bounds__(kBtThreads, 1)
attention_bwd_dkv_tc_kernel(const __grid_constant__ CUtensorMap map_qkv, const __grid_constant__ CUtensorMap map_do, const AttBwdParams p) {
  extern __shared__ uint8_t bt_smem_raw[];
  uint8_t* smem = bt_smem_raw + ((1024u - (smem_u32(bt_smem_raw) & 1023u)) & 1023u);
  uint8_t* s_k = smem;                                  // K tile, then V tile
  uint8_t* s_v = s_k + kBtTile;
  uint8_t* s_qd = s_v + kBtTile;                        // [stage][Q | dO]
  uint8_t* s_pt = s_qd + kBtStages * 2 * kBtTile;       // P^T: [2 halves][128][64]
  uint8_t* s_dst = s_pt + 2 * kBtTile;                  // dS^T: [2 halves][128][64]
  float* s_lse = reinterpret_cast<float*>(s_dst + 2 * kBtTile);  // [2 buffers][128]
  float* s_D = s_lse + 2 * kBtM;                                  // [2 buffers][128]
  uint64_t* kv_full = reinterpret_cast<uint64_t*>(s_D + 2 * kBtM);
  uint64_t* kv_empty = kv_full + 1;
  uint64_t* qd_full = kv_empty + 1;            // [stages]
  uint64_t* qd_empty = qd_full + kBtStages;    // [stages]
  uint64_t* s_full = qd_empty + kBtStages;     // S^T and dP^T of the current query tile are in TMEM
  uint64_t* p_full = s_full + 1;               // P^T / dS^T are in shared memory and S^T / dP^T have been read (4 warp arrivals)
  uint64_t* acc_full = p_full + 1;             // the item's dV, dK are final in TMEM
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(acc_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int J = p.n_tiles, N = p.N;
  const int n_items = p.n_tiles * p.H * p.B;

  if (threadIdx.x == 0) {
    prefetch_tensormap(&map_qkv);
    prefetch_tensormap(&map_do);
    mbar_init(kv_full, 1);
    mbar_init(kv_empty, 1);
    for (int i = 0; i < kBtStages; ++i) {
      mbar_init(&qd_full[i], 1);
      mbar_init(&qd_empty[i], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(p_full, 4);
    mbar_init(acc_full, 1);
    fence_mbar_init();
  }
  if (warp == 5) tmem_alloc<kBtTmemCols>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 4) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int ic = 0, qdc = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++ic) {
        int kt, h, b;
        bt_decode(p, item, kt, h, b);
        if (ic >= 1) mbar_wait_relaxed(kv_empty, (ic - 1) & 1);
        mbar_arrive_expect_tx(kv_full, 2 * kBtTile);
        tma_load_3d(s_k, &map_qkv, kv_full, (p.H + h) * kBtD, kt * kBtM, b);
        tma_load_3d(s_v, &map_qkv, kv_full, (2 * p.H + h) * kBtD, kt * kBtM, b);
        for (int j = 0; j < J; ++j, ++qdc) {
          const int st = qdc % kBtStages;
          if (qdc >= kBtStages) mbar_wait_relaxed(&qd_empty[st], ((qdc / kBtStages) - 1) & 1);
          mbar_arrive_expect_tx(&qd_full[st], 2 * kBtTile);
          tma_load_3d(s_qd + st * 2 * kBtTile, &map_qkv, &qd_full[st], h * kBtD, j * kBtM, b);
          tma_load_3d(s_qd + st * 2 * kBtTile + kBtTile, &map_do, &qd_full[st], h * kBtD, j * kBtM, b);
        }
      }
    }
  } else if (warp == 5) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t t_s = tmem_base, t_dp = tmem_base + kBtM, t_dv = tmem_base + 2 * kBtM, t_dk = t_dv + kBtD;
      int ic = 0, qdc = 0, g = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++ic) {
        mbar_wait(kv_full, ic & 1);
        tc_fence_after();
        for (int j = 0; j < J; ++j, ++g) {
          const int st = (qdc + j) % kBtStages;
          mbar_wait(&qd_full[st], ((qdc + j) / kBtStages) & 1);
          tc_fence_after();
          if (j > 0) {
            const int pst = (qdc + j - 1) % kBtStages;
            mbar_wait(p_full, (g - 1) & 1);
            tc_fence_after();
            bt_mma_nn(t_dv, s_pt, s_qd + pst * 2 * kBtTile + kBtTile, j > 1);
            bt_mma_nn(t_dk, s_dst, s_qd + pst * 2 * kBtTile, j > 1);
            umma_commit(&qd_empty[pst]);
          }
          bt_mma_nt(t_s, s_k, s_qd + st * 2 * kBtTile);
          bt_mma_nt(t_dp, s_v, s_qd + st * 2 * kBtTile + kBtTile);
          umma_commit(s_full);
          if (j + 1 == J) umma_commit(kv_empty);
        }
        mbar_wait(p_full, (g - 1) & 1);
        tc_fence_after();
        const int lst = (qdc + J - 1) % kBtStages;
        bt_mma_nn(t_dv, s_pt, s_qd + lst * 2 * kBtTile + kBtTile, J > 1);
        bt_mma_nn(t_dk, s_dst, s_qd + lst * 2 * kBtTile, J > 1);
        umma_commit(&qd_empty[lst]);
        umma_commit(acc_full);
        qdc += J;
      }
    }
  } else {
    // ===================== epilogue: one key row per thread =====================
    const int lane_base = warp * 32, r = lane_base + lane;
    const uint32_t lane_off = static_cast<uint32_t>(lane_base) << 16;
    const uint32_t t_s = tmem_base + lane_off, t_dp = t_s + kBtM, t_dv = t_s + 2 * kBtM, t_dk = t_dv + kBtD;
    const size_t ld = static_cast<size_t>(p.H) * kBtD;
    int ic = 0, g = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++ic) {
      int kt, h, b;
      bt_decode(p, item, kt, h, b);
      const int row = kt * kBtM + r;
      const bool rv = row < N;
      const size_t bh = static_cast<size_t>(b) * p.H + h;
      for (int j = 0; j < J; ++j, ++g) {
        // lse2 and D of this tile's 128 queries -> shared memory (double-buffered: the other buffer may still be read)
        const int buf = g & 1;
        const int qi = j * kBtM + r;
        s_lse[buf * kBtM + r] = qi < N ? p.lse2[bh * N + qi] : 0.f;
        s_D[buf * kBtM + r] = qi < N ? p.D[bh * N + qi] : 0.f;
        named_bar_sync(1, 4 * 32);
        const float* lse = s_lse + buf * kBtM;
        const float* Dq = s_D + buf * kBtM;
        mbar_wait(s_full, g & 1);
        tc_fence_after();
        const int valid = rv ? min(kBtM, N - j * kBtM) : 0;  // query columns of this tile whose P is computed
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          uint32_t sv[32], dp[32], pp[16], pd[16];
          tmem_ld_32x32b_x32(t_s + c * 32, sv);
          tmem_ld_32x32b_x32(t_dp + c * 32, dp);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            const int col = c * 32 + i;
            const float p0 = col < valid ? bt_ex2(__uint_as_float(sv[i]) * p.scale_log2e - lse[col]) : 0.f;
            const float p1 = col + 1 < valid ? bt_ex2(__uint_as_float(sv[i + 1]) * p.scale_log2e - lse[col + 1]) : 0.f;
            const uint32_t pb = bt_pack(p0, p1);
            pp[i >> 1] = pb;
            pd[i >> 1] = bt_pack(p.scale * bt_lo(pb) * (__uint_as_float(dp[i]) - Dq[col]),
                                 p.scale * bt_hi(pb) * (__uint_as_float(dp[i + 1]) - Dq[col + 1]));
          }
          bt_store_chunk(s_pt, r, c, pp);
          bt_store_chunk(s_dst, r, c, pd);
        }
        tc_fence_before();
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_full);
      }
      mbar_wait(acc_full, ic & 1);
      tc_fence_after();
      __nv_bfloat16* dst = p.dqkv + ((static_cast<size_t>(b) * N + (rv ? row : 0)) * 3) * ld + h * kBtD;
      bt_store_acc(t_dk, dst + ld, rv);
      bt_store_acc(t_dv, dst + 2 * ld, rv);
      tc_fence_before();
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    tmem_dealloc<kBtTmemCols>(tmem_base);
  }
}

size_t attention_bwd_tc_workspace_bytes(int B, int N, int H) {
  if (B <= 0 || N <= 0 || H <= 0) return 0;
  return (static_cast<size_t>(B) * H * N * sizeof(float) + 255) & ~static_cast<size_t>(255);
}

// qkv bf16 [B, N, 3, H, 64], out / d_out bf16 [B, N, H*64], lse2 fp32 [B, H, N] -> dqkv bf16 [B, N, 3, H, 64];
// workspace >= attention_bwd_tc_workspace_bytes(B, N, H) holds D
int launch_attention_bwd_tc(const __nv_bfloat16* qkv, const __nv_bfloat16* out, const __nv_bfloat16* d_out, const float* lse2, int B,
                            int N, int H, __nv_bfloat16* dqkv, void* workspace, size_t workspace_bytes, cudaStream_t s) {
  VDK_REQUIRE(B > 0 && N > 0 && H > 0 && H <= 65535 && B <= 65535, "attention backward (tcgen05): bad shape");
  VDK_REQUIRE(workspace && workspace_bytes >= attention_bwd_tc_workspace_bytes(B, N, H) &&
                  (reinterpret_cast<uintptr_t>(workspace) & 15) == 0,
              "attention backward (tcgen05): workspace too small or misaligned (need %zu bytes)", attention_bwd_tc_workspace_bytes(B, N, H));
  static bool attr = false;
  if (!attr) {
    VDK_CUDA_OK(cudaFuncSetAttribute(attention_bwd_dq_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kBtSmemQ));
    VDK_CUDA_OK(cudaFuncSetAttribute(attention_bwd_dkv_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kBtSmemKV));
    attr = true;
  }
  CUtensorMap map_qkv, map_do;  // [B][N][3*H*64] and [B][N][H*64], 128-row boxes of one head's 64 columns
  const uint64_t pitch = 3ull * H * kBtD, pitch_o = static_cast<uint64_t>(H) * kBtD;
  int rc = make_tma_3d_16bit(&map_qkv, qkv, pitch, static_cast<uint64_t>(N), static_cast<uint64_t>(B), pitch, pitch * N, kBtM);
  if (rc != VDK_OK) return rc;
  rc = make_tma_3d_16bit(&map_do, d_out, pitch_o, static_cast<uint64_t>(N), static_cast<uint64_t>(B), pitch_o, pitch_o * N, kBtM);
  if (rc != VDK_OK) return rc;
  AttBwdParams p{};
  p.B = B; p.N = N; p.H = H;
  p.n_tiles = (N + kBtM - 1) / kBtM;
  p.scale = 1.0f / sqrtf(static_cast<float>(kBtD));
  p.scale_log2e = p.scale * 1.4426950408889634f;
  p.out = out; p.d_out = d_out; p.lse2 = lse2;
  p.D = reinterpret_cast<float*>(workspace);
  p.dqkv = dqkv;
  const long long n_items = static_cast<long long>(p.n_tiles) * H * B;
  VDK_REQUIRE(n_items < (1ll << 31), "attention backward (tcgen05): too many (image, head, tile) items");
  const int grid = static_cast<int>(std::min<long long>(n_items, sm_count()));
  attention_bwd_dq_tc_kernel<<<grid, kBtThreads, kBtSmemQ, s>>>(map_qkv, map_do, p);
  VDK_CUDA_OK(cudaGetLastError());
  attention_bwd_dkv_tc_kernel<<<grid, kBtThreads, kBtSmemKV, s>>>(map_qkv, map_do, p);
  VDK_CUDA_OK(cudaGetLastError());
  return VDK_OK;
}

}  // namespace vdk
