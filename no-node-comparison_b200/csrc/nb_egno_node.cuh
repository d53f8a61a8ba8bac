// nb_egno_node.cuh — EGNO's node-level work after an edge sweep as ONE kernel per layer (forward).
//
// Reference: EGNN_Layer.forward after the aggregation (EGNO/model/basic.py:172-185):
//   U5 = [h, M] W5^T + b5 ; h' = SiLU(U5) W6^T + b6                      node_net     (basic.py:183-185)
//   UV = h Wv1^T + bv1    ; s  = w_v2 . SiLU(UV) + b_v2                   node_v_net   (basic.py:172-176)
//   x' = x + s v + clamp(Fsum / (N - 1), +-100)                                         (basic.py:177-178)
// These were three launches per layer (a two-job k_gemm64_tc batch, a second k_gemm64_tc, k_egno_xupd_fwd), each of
// which streams a 13 MB node tensor through HBM again.  Here a CTA owns a 128-row tile: h and M rows are split in
// registers and written to tensor memory as the A operands (no shared-memory copy of activations), the four weight
// blocks come from the call's pre-split images (64 KB, staged once per CTA), SiLU(U5) goes back into tensor memory as
// the A operand of the second product, and the 64 -> 1 head of node_v_net is a per-row dot finished through shared
// memory.  HBM: reads h, M, x, v, Fsum once; writes U5, UV (kept for the backward), h', x' once.
// Two CTAs per SM (66 KB of shared memory, 256 of 512 TMEM columns each): [0,64) D1 (U5, then h') | [64,128) D2 (UV) |
// [128,192) A0 hi|lo (h, then SiLU(U5)) | [192,256) A1 hi|lo (M).
#pragma once
#ifndef NB_EMU
#include "nb_edge_sel.cuh"

struct NbEgnoNodeFwdArgs {
  int rows, N;
  const unsigned char* img;   // 4 images, 16 KB each: W5 h half | W5 M half | W6 | Wv1   (egno_weight_images, slots 2..5)
  const float *h, *M;         // [rows][64]
  const float *b5, *b6, *bv1, *wv2, *bv2;
  const float *x, *v, *Fsum;  // [rows][3]
  float *U5, *UV;             // [rows][64] pre-activations (the backward's saved state; null: not stored)
  float *h_out, *x_out;
};
#define NB_ENF_W_BYTES (4 * 2 * NB_TC_TILE_BYTES(64))
#define NB_ENF_SMEM (NB_ENF_W_BYTES + (4 * NB_H + 2 * NB_TILE) * 4 + 64 + 1024)

__device__ __forceinline__ void nb_enf_load32(const float* p, bool live, float (&v)[32]) {
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float4 t = live ? nb_ld4(p + 4 * k) : make_float4(0.f, 0.f, 0.f, 0.f);
    v[4 * k] = t.x; v[4 * k + 1] = t.y; v[4 * k + 2] = t.z; v[4 * k + 3] = t.w;
  }
}
__device__ __forceinline__ void nb_enf_store32(float* p, bool live, const float (&v)[32]) {
  if (!live) return;
#pragma unroll
  for (int k = 0; k < 8; ++k) nb_st4(p + 4 * k, make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]));
}

__global__ void __launch_bounds__(NB_THREADS, 2) k_egno_node_fwd(NbEgnoNodeFwdArgs a) {
  NB_PDL_ENTER();
  extern __shared__ __align__(1024) unsigned char nb_smraw[];
  unsigned char* base = nb_smraw + ((1024u - (nb_smem_u32(nb_smraw) & 1023u)) & 1023u);
  float* sb5 = reinterpret_cast<float*>(base + NB_ENF_W_BYTES);
  float* sb6 = sb5 + NB_H;
  float* sbv1 = sb6 + NB_H;
  float* swv2 = sbv1 + NB_H;
  float* cpart = swv2 + NB_H;   // [2][128]
  uint64_t* bar = reinterpret_cast<uint64_t*>(cpart + 2 * NB_TILE);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, hf = warp >> 2;
  const int row = 32 * q + lane, cb = 32 * hf;
  const int ntiles = (a.rows + NB_TILE - 1) / NB_TILE;
  const uint32_t lane_base = (uint32_t)(32 * q) << 16;
  const uint32_t mine = lane_base + 16u * (uint32_t)hf;
  float v[32];
  // the first tile's h rows are requested before the weight copy (the kernel is a latency chain)
  {
    const int64_t gr0 = (int64_t)blockIdx.x * NB_TILE + row;
    nb_enf_load32(a.h + gr0 * NB_H + cb, (int)blockIdx.x < ntiles && gr0 < a.rows, v);
  }
  uint64_t* wbar = bar + 2;   // weight images have landed
  if (tid == 0) {
    nb_mbar_init(bar, 1);
    nb_mbar_init(wbar, 1);
    nb_mbar_fence_init();
    nb_bulk_g2s(base, a.img, (uint32_t)NB_ENF_W_BYTES, wbar);
  }
  if (tid < NB_H) {
    sb5[tid] = __ldg(a.b5 + tid);
    sb6[tid] = __ldg(a.b6 + tid);
    sbv1[tid] = __ldg(a.bv1 + tid);
    swv2[tid] = __ldg(a.wv2 + tid);
  }
  if (warp == 0) nb_tmem_alloc(tmem_slot, 256);
  nb_fence_async_smem();
  nb_tc_fence_before();
  __syncthreads();
  nb_tc_fence_after();
  const uint32_t tm = *tmem_slot;
  const uint32_t d1 = tm + lane_base + (uint32_t)cb;
  const uint32_t a0h = tm + 128, a0l = tm + 160, a1h = tm + 192, a1l = tm + 224;
  const uint32_t idesc_fwd = nb_idesc_bf16(128, 64, 0, 0);
  const uint32_t sW = nb_smem_u32(base);
#define NB_ENF_WH(i) (sW + (uint32_t)(i) * 2u * (uint32_t)NB_TC_TILE_BYTES(64))
#define NB_ENF_WL(i) (NB_ENF_WH(i) + (uint32_t)NB_TC_TILE_BYTES(64))
  const float bv2 = __ldg(a.bv2);
  const float cnt = (float)(a.N - 1 > 1 ? a.N - 1 : 1);
  uint32_t phase = 0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t gr = (int64_t)tile * NB_TILE + row;
    const bool live = gr < a.rows;
    const int64_t off = gr * NB_H + cb;
    if (tile != (int)blockIdx.x) nb_enf_load32(a.h + off, live, v);
    nb_store32_ta(nullptr, nullptr, row, hf, v, a0h + mine, a0l + mine);
    nb_enf_load32(a.M + off, live, v);
    nb_store32_ta(nullptr, nullptr, row, hf, v, a1h + mine, a1l + mine);
    nb_tmem_st_wait();
    nb_tc_fence_before();
    __syncthreads();   // (also: every thread has finished the previous tile's reads of D1 / cpart)
    if (NB_ISSUER(0)) {
      if (tile == (int)blockIdx.x) nb_mbar_wait(wbar, 0);
      nb_tc_fence_after();
      nb_issue_w3_ta(tm, a0h, a0l, NB_ENF_WH(0), NB_ENF_WL(0), false, idesc_fwd, 0u);        // U5  = h W5a^T
      nb_issue_w3_ta(tm, a1h, a1l, NB_ENF_WH(1), NB_ENF_WL(1), false, idesc_fwd, 1u);        //     + M W5b^T
      nb_issue_w3_ta(tm + 64, a0h, a0l, NB_ENF_WH(3), NB_ENF_WL(3), false, idesc_fwd, 0u);   // UV  = h Wv1^T
      nb_mma_commit(bar);
    }
    // coordinate operands of this row, requested under the MMAs (one thread per row)
    float xr[3] = {0.f, 0.f, 0.f}, vr[3] = {0.f, 0.f, 0.f}, fr[3] = {0.f, 0.f, 0.f};
    if (hf == 0 && live) {
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        xr[d] = a.x[gr * 3 + d];
        vr[d] = a.v[gr * 3 + d];
        fr[d] = a.Fsum[gr * 3 + d];
      }
    }
    nb_mbar_wait(bar, phase);
    phase ^= 1;
    nb_tc_fence_after();
    // ---- U5 (kept for the backward) ; SiLU(U5) -> A operand of the second product
    nb_tmem_ld32(d1, v);
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] += sb5[cb + i];
    if (a.U5) nb_enf_store32(a.U5 + off, live, v);   // inference keeps nothing for a backward
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = live ? nb_silu(v[i]) : 0.f;
    nb_store32_ta(nullptr, nullptr, row, hf, v, a0h + mine, a0l + mine);
    // ---- UV (kept for the backward) ; this half's share of s = w_v2 . SiLU(UV)
    nb_tmem_ld32(d1 + 64, v);
    float cp = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      v[i] += sbv1[cb + i];
      cp = fmaf(swv2[cb + i], nb_silu(v[i]), cp);
    }
    if (a.UV) nb_enf_store32(a.UV + off, live, v);
    cpart[hf * NB_TILE + row] = cp;
    nb_tmem_st_wait();
    nb_tc_fence_before();
    __syncthreads();
    if (NB_ISSUER(0)) {
      nb_tc_fence_after();
      nb_issue_w3_ta(tm, a0h, a0l, NB_ENF_WH(2), NB_ENF_WL(2), false, idesc_fwd, 0u);        // h' = SiLU(U5) W6^T
      nb_mma_commit(bar);
    }
    if (hf == 0 && live) {   // x' = x + s v + clamp(mean force)      (basic.py:176-178)
      const float s = (cpart[row] + cpart[NB_TILE + row]) + bv2;
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        float f = fr[d] / cnt;
        f = fminf(fmaxf(f, -100.f), 100.f);
        a.x_out[gr * 3 + d] = xr[d] + s * vr[d] + f;
      }
    }
    nb_mbar_wait(bar, phase);
    phase ^= 1;
    nb_tc_fence_after();
    nb_tmem_ld32(d1, v);
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] += sb6[cb + i];
    nb_enf_store32(a.h_out + off, live, v);
    nb_tc_fence_before();
  }
  if ((int)blockIdx.x >= ntiles && tid == 0) nb_mbar_wait(wbar, 0);   // never exit under a copy in flight
  nb_tc_fence_before();
  __syncthreads();
  if (warp == 0) nb_tmem_dealloc(tm, 256);
}

// ----------------------------------------------------------------------------- backward
// The same three pieces backwards, before the edge sweep of the layer (autograd of basic.py:172-185):
//   x' = x + s v + clamp(Fsum/(N-1)):  gv1 = gv + s gx ; gFsum = gx / (N-1) inside the clamp ; gs = gx . v
//   s  = w_v2 . SiLU(UV) + b_v2     :  GUV = gs w_v2 * SiLU'(UV) ; dL/dw_v2 = sum_rows gs SiLU(UV) ; dL/db_v2 = sum_rows gs
//   h' = SiLU(U5) W6^T + b6         :  GU5 = (gh W6) * SiLU'(U5)
//   U5 = [h, M] W5^T ; UV = h Wv1^T :  gh1 = GU5 W5[:, :64] + GUV Wv1 ;  gM = GU5 W5[:, 64:]
// (was: k_egno_xupd_bwd + two k_gemm64_tc launches).  GU5 and GUV are stored for the weight-gradient reductions; the
// head's weight gradient is reduced over the rows of a warp with a transposing shuffle tree (31 shuffles leave column j's
// sum on lane j), accumulated in ONE register per thread over the CTA's tiles, and written as a [65]-float partial slice
// per CTA for k_finalize — fixed order, no atomics.
// TMEM (256 columns): [0,64) D1 (gh W6, then gM) | [64,128) D3 (gh1) | [128,192) A0 (gh, then GU5) | [192,256) A1 (GUV).
struct NbEgnoNodeBwdArgs {
  int rows, N;
  const unsigned char* img;     // W5 h half | W5 M half | W6 | Wv1
  const float *gh, *U5, *UV;    // [rows][64]: dL/dh', saved pre-activations
  const float *wv2, *bv2;
  const float *gx, *gv, *v, *Fsum;   // [rows][3]
  float *gv_out, *gFsum;        // [rows][3]
  float *GU5, *GUV, *gh1, *gM;  // [rows][64]
  float* partial;               // [grid][65]: dL/dw_v2[64], dL/db_v2
};
#define NB_ENB_SMEM (NB_ENF_W_BYTES + (NB_H + 2 * NB_TILE + 8 * 32 + 8) * 4 + 64 + 1024)

// h[j] summed over the 32 lanes ends up on lane j (h is destroyed)
__device__ __forceinline__ float nb_warp_colsum32(float (&h)[32], int lane) {
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) {
    const bool up = (lane & m) != 0;
#pragma unroll
    for (int i = 0; i < m; ++i) {
      const float send = up ? h[i] : h[i + m];
      const float recv = __shfl_xor_sync(0xffffffffu, send, m);
      h[i] = (up ? h[i + m] : h[i]) + recv;
    }
  }
  return h[0];
}

__global__ void __launch_bounds__(NB_THREADS, 2) k_egno_node_bwd(NbEgnoNodeBwdArgs a) {
  NB_PDL_ENTER();
  extern __shared__ __align__(1024) unsigned char nb_smraw[];
  unsigned char* base = nb_smraw + ((1024u - (nb_smem_u32(nb_smraw) & 1023u)) & 1023u);
  float* swv2 = reinterpret_cast<float*>(base + NB_ENF_W_BYTES);
  float* cpart = swv2 + NB_H;      // [2][128]
  float* red = cpart + 2 * NB_TILE;  // [8][32] + [8]
  uint64_t* bar = reinterpret_cast<uint64_t*>(red + 8 * 32 + 8);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, hf = warp >> 2;
  const int row = 32 * q + lane, cb = 32 * hf;
  const int ntiles = (a.rows + NB_TILE - 1) / NB_TILE;
  const uint32_t lane_base = (uint32_t)(32 * q) << 16;
  const uint32_t mine = lane_base + 16u * (uint32_t)hf;
  float v[32];
  {
    const int64_t gr0 = (int64_t)blockIdx.x * NB_TILE + row;
    nb_enf_load32(a.UV + gr0 * NB_H + cb, (int)blockIdx.x < ntiles && gr0 < a.rows, v);
  }
  uint64_t* wbar = bar + 2;   // weight images have landed
  if (tid == 0) {
    nb_mbar_init(bar, 1);
    nb_mbar_init(wbar, 1);
    nb_mbar_fence_init();
    nb_bulk_g2s(base, a.img, (uint32_t)NB_ENF_W_BYTES, wbar);
  }
  if (tid < NB_H) swv2[tid] = __ldg(a.wv2 + tid);
  if (warp == 0) nb_tmem_alloc(tmem_slot, 256);
  nb_fence_async_smem();
  nb_tc_fence_before();
  __syncthreads();
  nb_tc_fence_after();
  const uint32_t tm = *tmem_slot;
  const uint32_t d1 = tm + lane_base + (uint32_t)cb;
  const uint32_t a0h = tm + 128, a0l = tm + 160, a1h = tm + 192, a1l = tm + 224;
  const uint32_t idesc_mn = nb_idesc_bf16(128, 64, 0, 1);
  const uint32_t sW = nb_smem_u32(base);
  const float bv2 = __ldg(a.bv2);
  const float cnt = (float)(a.N - 1 > 1 ? a.N - 1 : 1);
  float gw2acc = 0.f, gb2acc = 0.f;   // lane j: column cb + j of dL/dw_v2 over this warp's rows; dL/db_v2 (warps with hf = 0)
  uint32_t phase = 0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t gr = (int64_t)tile * NB_TILE + row;
    const bool live = gr < a.rows;
    const int64_t off = gr * NB_H + cb;
    if (tile != (int)blockIdx.x) nb_enf_load32(a.UV + off, live, v);
    float gxr[3] = {0.f, 0.f, 0.f}, vr[3] = {0.f, 0.f, 0.f};
    if (live) {
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        gxr[d] = a.gx[gr * 3 + d];
        vr[d] = a.v[gr * 3 + d];
      }
    }
    const float gs = gxr[0] * vr[0] + gxr[1] * vr[1] + gxr[2] * vr[2];   // dL/ds of this row (0 for padding rows)
    {
      float hz[32];
      float cp = 0.f;
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        float z, d;
        nb_silu_grad(v[i], z, d);
        const float w = swv2[cb + i];
        cp = fmaf(w, z, cp);
        hz[i] = gs * z;
        v[i] = gs * w * d;   // GUV
      }
      cpart[hf * NB_TILE + row] = cp;
      nb_enf_store32(a.GUV + off, live, v);
      nb_store32_ta(nullptr, nullptr, row, hf, v, a1h + mine, a1l + mine);
      gw2acc += nb_warp_colsum32(hz, lane);
      if (hf == 0) {
        float t = gs;
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) t += __shfl_xor_sync(0xffffffffu, t, m);
        gb2acc += t;
      }
    }
    nb_enf_load32(a.gh + off, live, v);
    nb_store32_ta(nullptr, nullptr, row, hf, v, a0h + mine, a0l + mine);
    nb_tmem_st_wait();
    nb_tc_fence_before();
    __syncthreads();
    if (NB_ISSUER(0)) {
      if (tile == (int)blockIdx.x) nb_mbar_wait(wbar, 0);
      nb_tc_fence_after();
      nb_issue_w3_ta(tm, a0h, a0l, NB_ENF_WH(2), NB_ENF_WL(2), true, idesc_mn, 0u);        // gh W6
      nb_issue_w3_ta(tm + 64, a1h, a1l, NB_ENF_WH(3), NB_ENF_WL(3), true, idesc_mn, 0u);   // gh1 = GUV Wv1
      nb_mma_commit(bar);
    }
    nb_enf_load32(a.U5 + off, live, v);   // requested under the MMAs
    if (hf == 0 && live) {   // gv1 = gv + s gx ; gFsum = gx / (N - 1) where the mean force was not clamped
      const float s = (cpart[row] + cpart[NB_TILE + row]) + bv2;
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        a.gv_out[gr * 3 + d] = (a.gv ? a.gv[gr * 3 + d] : 0.f) + s * gxr[d];
        const float f = a.Fsum[gr * 3 + d] / cnt;
        a.gFsum[gr * 3 + d] = (f >= -100.f && f <= 100.f) ? gxr[d] / cnt : 0.f;
      }
    }
    nb_mbar_wait(bar, phase);
    phase ^= 1;
    nb_tc_fence_after();
    {
      float t[32];
      nb_tmem_ld32(d1, t);
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = live ? t[i] * nb_dsilu(v[i]) : 0.f;   // GU5 = (gh W6) * SiLU'(U5)
    }
    nb_enf_store32(a.GU5 + off, live, v);
    nb_store32_ta(nullptr, nullptr, row, hf, v, a0h + mine, a0l + mine);
    nb_tmem_st_wait();
    nb_tc_fence_before();
    __syncthreads();
    if (NB_ISSUER(0)) {
      nb_tc_fence_after();
      nb_issue_w3_ta(tm + 64, a0h, a0l, NB_ENF_WH(0), NB_ENF_WL(0), true, idesc_mn, 1u);   // gh1 += GU5 W5[:, :64]
      nb_issue_w3_ta(tm, a0h, a0l, NB_ENF_WH(1), NB_ENF_WL(1), true, idesc_mn, 0u);        // gM   = GU5 W5[:, 64:]
      nb_mma_commit(bar);
    }
    nb_mbar_wait(bar, phase);
    phase ^= 1;
    nb_tc_fence_after();
    nb_tmem_ld32(d1 + 64, v);
    nb_enf_store32(a.gh1 + off, live, v);
    nb_tmem_ld32(d1, v);
    nb_enf_store32(a.gM + off, live, v);
    nb_tc_fence_before();
  }
  // ---- this CTA's slice of the head's weight gradient: sum the four row quarters of each column half in a fixed order
  red[warp * 32 + lane] = gw2acc;
  if (lane == 0) red[8 * 32 + warp] = gb2acc;
  nb_tc_fence_before();
  __syncthreads();
  if (tid < NB_H) {
    const int h2 = tid >> 5, j = tid & 31;
    a.partial[(int64_t)blockIdx.x * 65 + tid] =
        (red[(4 * h2 + 0) * 32 + j] + red[(4 * h2 + 1) * 32 + j]) + (red[(4 * h2 + 2) * 32 + j] + red[(4 * h2 + 3) * 32 + j]);
  }
  if (tid == 0) a.partial[(int64_t)blockIdx.x * 65 + 64] = (red[8 * 32 + 0] + red[8 * 32 + 1]) + (red[8 * 32 + 2] + red[8 * 32 + 3]);
  if ((int)blockIdx.x >= ntiles && tid == 0) nb_mbar_wait(wbar, 0);   // never exit under a copy in flight
  if (warp == 0) nb_tmem_dealloc(tm, 256);
}

// ----------------------------------------------------------------------------- the first edge layer's node halves
// PQ = true  (forward):  P = h W1[:, h_row]^T + b1 ; Q = h W1[:, h_col]^T      one A operand, two products, two outputs
// PQ = false (backward): gh += gP W1[:, h_row] + gQ W1[:, h_col]               two A operands, one accumulated output
// The same tile scheme as above with 32 KB of weight images: 192 of 256 TMEM columns, two CTAs per SM.  (The generic
// k_gemm64_tc ran these as two-job / two-source launches through shared-memory A tiles: 21 us per launch at 51 200 rows.)
struct NbEgnoPairArgs {
  int rows;
  const unsigned char* img;   // W1 h_row | W1 h_col
  const float *A0, *A1;       // [rows][64]  (PQ: A1 unused)
  const float* bias;          // PQ: b1 (added to the first output)
  float *O0, *O1;             // PQ: P, Q ; else O0 = gh (read-modify-write), O1 unused
};
#define NB_EPR_W_BYTES (2 * 2 * NB_TC_TILE_BYTES(64))
#define NB_EPR_SMEM (NB_EPR_W_BYTES + NB_H * 4 + 64 + 1024)

template <bool PQ>
__global__ void __launch_bounds__(NB_THREADS, 2) k_egno_pair(NbEgnoPairArgs a) {
  NB_PDL_ENTER();
  extern __shared__ __align__(1024) unsigned char nb_smraw[];
  unsigned char* base = nb_smraw + ((1024u - (nb_smem_u32(nb_smraw) & 1023u)) & 1023u);
  float* sbias = reinterpret_cast<float*>(base + NB_EPR_W_BYTES);
  uint64_t* bar = reinterpret_cast<uint64_t*>(sbias + NB_H);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, hf = warp >> 2;
  const int row = 32 * q + lane, cb = 32 * hf;
  const int ntiles = (a.rows + NB_TILE - 1) / NB_TILE;
  const uint32_t lane_base = (uint32_t)(32 * q) << 16;
  const uint32_t mine = lane_base + 16u * (uint32_t)hf;
  float v[32];
  {
    const int64_t gr0 = (int64_t)blockIdx.x * NB_TILE + row;
    nb_enf_load32(a.A0 + gr0 * NB_H + cb, (int)blockIdx.x < ntiles && gr0 < a.rows, v);
  }
  uint64_t* wbar = bar + 2;   // weight images have landed
  if (tid == 0) {
    nb_mbar_init(bar, 1);
    nb_mbar_init(wbar, 1);
    nb_mbar_fence_init();
    nb_bulk_g2s(base, a.img, (uint32_t)NB_EPR_W_BYTES, wbar);
  }
  if (tid < NB_H) sbias[tid] = (PQ && a.bias) ? __ldg(a.bias + tid) : 0.f;
  if (warp == 0) nb_tmem_alloc(tmem_slot, 256);
  nb_fence_async_smem();
  nb_tc_fence_before();
  __syncthreads();
  nb_tc_fence_after();
  const uint32_t tm = *tmem_slot;
  const uint32_t d1 = tm + lane_base + (uint32_t)cb;
  const uint32_t a0h = tm + 128, a0l = tm + 160, a1h = tm + 192, a1l = tm + 224;
  const uint32_t idesc = PQ ? nb_idesc_bf16(128, 64, 0, 0) : nb_idesc_bf16(128, 64, 0, 1);
  const uint32_t sW = nb_smem_u32(base);
  uint32_t phase = 0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t gr = (int64_t)tile * NB_TILE + row;
    const bool live = gr < a.rows;
    const int64_t off = gr * NB_H + cb;
    if (tile != (int)blockIdx.x) nb_enf_load32(a.A0 + off, live, v);
    nb_store32_ta(nullptr, nullptr, row, hf, v, a0h + mine, a0l + mine);
    if (!PQ) {
      nb_enf_load32(a.A1 + off, live, v);
      nb_store32_ta(nullptr, nullptr, row, hf, v, a1h + mine, a1l + mine);
    }
    nb_tmem_st_wait();
    nb_tc_fence_before();
    __syncthreads();
    if (NB_ISSUER(0)) {
      if (tile == (int)blockIdx.x) nb_mbar_wait(wbar, 0);
      nb_tc_fence_after();
      if (PQ) {
        nb_issue_w3_ta(tm, a0h, a0l, NB_ENF_WH(0), NB_ENF_WL(0), false, idesc, 0u);
        nb_issue_w3_ta(tm + 64, a0h, a0l, NB_ENF_WH(1), NB_ENF_WL(1), false, idesc, 0u);
      } else {
        nb_issue_w3_ta(tm, a0h, a0l, NB_ENF_WH(0), NB_ENF_WL(0), true, idesc, 0u);
        nb_issue_w3_ta(tm, a1h, a1l, NB_ENF_WH(1), NB_ENF_WL(1), true, idesc, 1u);
      }
      nb_mma_commit(bar);
    }
    float r[32];
    if (!PQ) nb_enf_load32(a.O0 + off, live, r);   // the accumulate target, requested under the MMAs
    nb_mbar_wait(bar, phase);
    phase ^= 1;
    nb_tc_fence_after();
    nb_tmem_ld32(d1, v);
    if (PQ) {
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] += sbias[cb + i];
      nb_enf_store32(a.O0 + off, live, v);
      nb_tmem_ld32(d1 + 64, v);
      nb_enf_store32(a.O1 + off, live, v);
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] += r[i];
      nb_enf_store32(a.O0 + off, live, v);
    }
    nb_tc_fence_before();
  }
  if ((int)blockIdx.x >= ntiles && tid == 0) nb_mbar_wait(wbar, 0);   // never exit under a copy in flight
  nb_tc_fence_before();
  __syncthreads();
  if (warp == 0) nb_tmem_dealloc(tm, 256);
}
#endif  // NB_EMU
