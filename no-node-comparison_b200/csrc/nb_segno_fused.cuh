// nb_segno_fused.cuh — SEGNO's T second-order integration sub-steps fused into ONE kernel (forward).
//
// Reference: SEGNO.forward_step (SEGNO/models/model.py:95-102) calls the weight-shared SEGNO_GCL T times
// (gcl.py:111-119).  Here a CTA owns a unit of G trajectories (G*N <= 27 nodes) for the whole call: the node state
// (h, x, v) lives in shared memory across all T sub-steps, every weight matrix is staged once as a split-bf16
// operand tile, and each sub-step runs on the tensor cores end to end:
//
//   P|Q      = h W1[:, h_row]^T + b1 | h W1[:, h_col]^T          node MMA (M = 64)        -> node tile
//   per 128-edge tile: gather -> SiLU -> W2 -> SiLU -> W3 -> phi_x head -> scatter           (as k_edge_fwd_sel)
//   a        = clamp-per-edge mean force ; v += a/T ; x += v/T                              (gcl.py:100-102,116-117)
//   U5       = [h, M] W5^T + b5 ; h <- h + SiLU(U5) W6^T + b6                               node MMAs (gcl.py:89-94)
//
// When `saved` is given, the per-sub-step state the (unfused) backward needs — h_k, M_k, U5_k, x_k — is written
// in the layout of nb_segno_forward's saved buffer; nothing else reaches HBM between sub-steps.
#pragma once
#ifndef NB_EMU
#include "nb_edge_sel.cuh"

struct NbSegnoFusedArgs {
  NbEdgeGeom g;       // NGT = B, clamp_edge = 1
  int T, recurrent;
  float inv_T, cw;
  const float *W1, *b1;   // edge_mlp.0 [64][ldw1]: cols h_row | h_col | radial | edge_attr
  int ldw1, col_rad, col_ef;
  const float *W2, *b2, *W3, *b3, *w4, *b4;   // edge_mlp.2, coord_mlp.0, coord_mlp.2
  const float *W5, *b5, *W6, *b6;             // node_mlp.0 [64][128], node_mlp.2 [64][64]
  const float *h_in, *x_in, *v_in;            // [B*N][64], [B*N][3], [B*N][3]
  const float* ef;                            // [B*EPG][nef]
  float *h_out, *x_out, *v_out;
  float* saved;                               // nullable; [T][iter_stride]: h | M | U5 | x  (each [B*N] rows)
  int64_t iter_stride;
};

// shared memory map (bytes after 1024-alignment)
#define NB_FS_W 0                                            // 14 weight pieces x 8 KB: W2 W3 W1r W1c W5a W5b W6 (hi, lo)
#define NB_FS_T (14 * NB_TC_TILE_BYTES(64))                  // activation tile hi/lo      2 x 16 KB
#define NB_FS_SEL (NB_FS_T + 2 * NB_TC_TILE_BYTES(128))      // selector                   16 KB
#define NB_FS_NT (NB_FS_SEL + NB_TC_TILE_BYTES(128))         // node tile hi/lo            2 x 8 KB
#define NB_FS_F (NB_FS_NT + 2 * NB_TC_TILE_BYTES(64))        // force tile hi/lo           2 x 2 KB
#define NB_FS_HN (NB_FS_F + 2 * NB_TILE * 16)                // h tile hi/lo (64 rows)     2 x 8 KB
#define NB_FS_UN (NB_FS_HN + 2 * NB_TC_TILE_BYTES(64))       // M / SiLU(U5) tile hi/lo    2 x 8 KB
#define NB_FS_FL (NB_FS_UN + 2 * NB_TC_TILE_BYTES(64))
#define NB_FS_NFLOAT (28 * NB_H + 2 * 32 * 3 + 6 * NB_H)
#define NB_SEGNO_FUSED_SMEM(RU) (NB_FS_FL + NB_FS_NFLOAT * 4 + (RU) * 4 + 64 + 1024)
#define NB_FS_TMEM_COLS 512  // [0,64) pre | [64,128) M sums | [128,136) F sums | [192,256) P / U5 / dh | [256,320) Q |
                             // [448,480) hi, [480,512) lo pieces of the A operand (z1, then m) as packed bf16 pairs

#define NB_FS_WH(p) (Wt + (2 * (p)) * NB_TC_TILE_BYTES(64))
#define NB_FS_WL(p) (Wt + (2 * (p) + 1) * NB_TC_TILE_BYTES(64))
#define NB_FS_SWH(p) (sW + (2 * (p)) * NB_TC_TILE_BYTES(64))
#define NB_FS_SWL(p) (sW + (2 * (p) + 1) * NB_TC_TILE_BYTES(64))

// 512 threads (thread = row x 16 columns, as in k_edge_bwd_sel): the staged weights fill the shared memory, so there is one
// CTA per SM either way and 16 warps are what hides the latencies of the SiLU stages; the two 64-deep products of an
// edge tile read their activation operand from tensor memory (z1 has no shared-memory copy; m keeps one for the scatter).
// Measured against the first version (256 threads, 32 columns per thread, shared-memory A operands): 396 -> 378 us per
// launch at B = 256, N = 20, T = 10 — the kernel is bound by its ~16 dependent MMA round trips per sub-step, not by the
// CUDA-core stages.

// 16 consecutive fp32 values of row r (column quarter cq) -> split pieces into this thread's TMEM lane and, when `hi`
// is given, into the shared-memory tiles
__device__ __forceinline__ void nb_fs_store16(unsigned char* hi, unsigned char* lo, int r, int cq, const float* v, uint32_t ta_hi,
                                              uint32_t ta_lo) {
  uint32_t h0[4], l0[4], h1[4], l1[4];
  nb_split8(v, h0, l0);
  nb_split8(v + 8, h1, l1);
  if (hi) {
    const uint32_t o0 = nb_tc_chunk_off(r, 2 * cq), o1 = nb_tc_chunk_off(r, 2 * cq + 1);
    *reinterpret_cast<uint4*>(hi + o0) = make_uint4(h0[0], h0[1], h0[2], h0[3]);
    *reinterpret_cast<uint4*>(hi + o1) = make_uint4(h1[0], h1[1], h1[2], h1[3]);
    *reinterpret_cast<uint4*>(lo + o0) = make_uint4(l0[0], l0[1], l0[2], l0[3]);
    *reinterpret_cast<uint4*>(lo + o1) = make_uint4(l1[0], l1[1], l1[2], l1[3]);
  }
  nb_tmem_st44(ta_hi, h0, h1);
  nb_tmem_st44(ta_lo, l0, l1);
}
__device__ __forceinline__ void nb_fs_stage_w(unsigned char* hi, unsigned char* lo, const float* __restrict__ W, int ldw, int tid) {
  const int o = tid >> 3, j = tid & 7;   // 64 x 8 chunks = 512 threads
  float v[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __ldg(W + (int64_t)o * ldw + 8 * j + i);
  nb_tc_store8(hi, lo, o, j, v);
}

__global__ void __launch_bounds__(NB_SB_THREADS, 1) k_segno_fused_fwd(NbSegnoFusedArgs a) {
  NB_PDL_ENTER();
  constexpr int NT = NB_SB_THREADS;
  extern __shared__ __align__(1024) unsigned char nb_smraw[];
  unsigned char* base = nb_smraw + ((1024u - (nb_smem_u32(nb_smraw) & 1023u)) & 1023u);
  unsigned char* Wt = base + NB_FS_W;  // piece p (hi at 2p, lo at 2p+1): 0 W2, 1 W3, 2 W1r, 3 W1c, 4 W5a, 5 W5b, 6 W6
  unsigned char* Th = base + NB_FS_T;
  unsigned char* Tl = Th + NB_TC_TILE_BYTES(128);
  unsigned char* Sel = base + NB_FS_SEL;
  unsigned char* Nh = base + NB_FS_NT;
  unsigned char* Nl = Nh + NB_TC_TILE_BYTES(64);
  unsigned char* Fh = base + NB_FS_F;
  unsigned char* Fl = Fh + NB_TILE * 16;
  unsigned char* Hh = base + NB_FS_HN;
  unsigned char* Hl = Hh + NB_TC_TILE_BYTES(64);
  unsigned char* Uh = base + NB_FS_UN;
  unsigned char* Ul = Uh + NB_TC_TILE_BYTES(64);
  float* fl = reinterpret_cast<float*>(base + NB_FS_FL);
  float* hs = fl;                    // [28][64] node state h (fp32), G*N <= 27
  float* xs = hs + 28 * NB_H;        // [32][3]
  float* vs = xs + 32 * 3;           // [32][3]
  float* vb1 = vs + 32 * 3;
  float* vb2 = vb1 + NB_H;
  float* vb3 = vb2 + NB_H;
  float* vw4 = vb3 + NB_H;
  float* vb5 = vw4 + NB_H;
  float* vb6 = vb5 + NB_H;
  // [4][128] partial dots of the phi_x head: lives in the first 2 KB of the M / SiLU(U5) tile, which is idle during the
  // edge tiles (rows 0..15 of its hi piece; they are rewritten by the read-out (d) before the node MMAs read them, and a
  // node row beyond the unit's nodes only ever feeds accumulator rows nobody reads) — with its own 2 KB the kernel does
  // not fit the 227 KB of a CTA at G * N = 27
  float* cpart = reinterpret_cast<float*>(Uh);
  uint32_t* rowinfo = reinterpret_cast<uint32_t*>(vb6 + NB_H);
  const NbEdgeGeom g = a.g;
  const int RU = g.G * g.EPG, GN = g.G * g.N;
  uint64_t* bar = reinterpret_cast<uint64_t*>(rowinfo + RU + (RU & 1));
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, cq = warp >> 2;
  const int row = 32 * q + lane;
  const int cb = 16 * cq;
  const int nl = 16 * q + lane;      // node owned in the M = 64 accumulators (lanes < 16 only)
  const bool nown = lane < 16;

  nb_fs_stage_w(NB_FS_WH(0), NB_FS_WL(0), a.W2, NB_H, tid);
  nb_fs_stage_w(NB_FS_WH(1), NB_FS_WL(1), a.W3, NB_H, tid);
  nb_fs_stage_w(NB_FS_WH(2), NB_FS_WL(2), a.W1, a.ldw1, tid);
  nb_fs_stage_w(NB_FS_WH(3), NB_FS_WL(3), a.W1 + NB_H, a.ldw1, tid);
  nb_fs_stage_w(NB_FS_WH(4), NB_FS_WL(4), a.W5, 2 * NB_H, tid);
  nb_fs_stage_w(NB_FS_WH(5), NB_FS_WL(5), a.W5 + NB_H, 2 * NB_H, tid);
  nb_fs_stage_w(NB_FS_WH(6), NB_FS_WL(6), a.W6, NB_H, tid);
  // zero: node tile, h tile, U tile (rows beyond the unit's nodes must stay finite zeros)
  for (int idx = tid; idx < 2 * NB_TC_TILE_BYTES(64) / 16; idx += NT) reinterpret_cast<uint4*>(Nh)[idx] = make_uint4(0u, 0u, 0u, 0u);
  for (int idx = tid; idx < 4 * NB_TC_TILE_BYTES(64) / 16; idx += NT) reinterpret_cast<uint4*>(Hh)[idx] = make_uint4(0u, 0u, 0u, 0u);
  nb_sel_build_rowinfo(rowinfo, g, tid, NT);
  if (tid < NB_H) {
    vb1[tid] = __ldg(a.b1 + tid);
    vb2[tid] = __ldg(a.b2 + tid);
    vb3[tid] = __ldg(a.b3 + tid);
    vw4[tid] = __ldg(a.w4 + tid);
    vb5[tid] = __ldg(a.b5 + tid);
    vb6[tid] = __ldg(a.b6 + tid);
  }
  if (tid == 0) {
    nb_mbar_init(bar, 1);
    nb_mbar_fence_init();
  }
  if (warp == 0) nb_tmem_alloc(tmem_slot, NB_FS_TMEM_COLS);
  __syncthreads();
  if (tid < 10 * 8) {  // weight rows of the node tile (w_rad, w_ef)
    int k = tid >> 3, j = tid & 7;
    int f = (k >> 1) - 1;
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int c = 8 * j + i;
      v[i] = f < 0 ? __ldg(a.W1 + (int64_t)c * a.ldw1 + a.col_rad)
                   : (f < g.nef ? __ldg(a.W1 + (int64_t)c * a.ldw1 + a.col_ef + f) : 0.f);
    }
    nb_tc_store8(Nh, Nl, NB_SEL_XC0 + k, j, v);
  }
  nb_fence_async_smem();
  nb_tc_fence_before();
  __syncthreads();
  nb_tc_fence_after();
  const uint32_t tm = *tmem_slot;
  const uint32_t lane_base = (uint32_t)(32 * q) << 16;
  const uint32_t tm_mine = tm + lane_base + (uint32_t)cb;
  const uint32_t ta_h = tm + 448, ta_l = tm + 480;
  const uint32_t ta_hm = ta_h + lane_base + 8u * (uint32_t)cq, ta_lm = ta_l + lane_base + 8u * (uint32_t)cq;
  const uint32_t idesc_fwd = nb_idesc_bf16(128, 64, 0, 0);
  const uint32_t idesc_gat = nb_idesc_bf16(128, 64, 0, 1);
  const uint32_t idesc_sc = nb_idesc_bf16(64, 64, 1, 1);
  const uint32_t idesc_sc8 = nb_idesc_bf16(64, 8, 1, 1);
  const uint32_t idesc_node = nb_idesc_bf16(64, 64, 0, 0);   // node rows x W^T, M = 64
  const uint32_t sTh = nb_smem_u32(Th), sTl = nb_smem_u32(Tl), sSel = nb_smem_u32(Sel), sNh = nb_smem_u32(Nh),
                 sNl = nb_smem_u32(Nl), sFh = nb_smem_u32(Fh), sFl = nb_smem_u32(Fl), sHh = nb_smem_u32(Hh),
                 sHl = nb_smem_u32(Hl), sUh = nb_smem_u32(Uh), sUl = nb_smem_u32(Ul), sW = nb_smem_u32(Wt);
  const float b4 = __ldg(a.b4);
  const float cnt = (float)(g.N - 1 > 1 ? g.N - 1 : 1);
  const int64_t Nn = (int64_t)g.NGT * g.N;
  uint32_t phase = 0;

  for (int u = blockIdx.x; u < g.n_units; u += gridDim.x) {
    const int gt0 = u * g.G;
    const int ngt = min(g.G, g.NGT - gt0);
    const int R = ngt * g.EPG;
    const int nnode = ngt * g.N;
    const int64_t node0 = (int64_t)gt0 * g.N;
    // ---- load the unit's state (nnode * 16 <= 432 float4, nnode * 3 <= 81 scalars: one each per thread)
    if (tid < nnode * 16) nb_st4(hs + tid * 4, nb_ld4(a.h_in + node0 * NB_H + tid * 4));
    if (tid < nnode * 3) {
      xs[tid] = __ldg(a.x_in + node0 * 3 + tid);
      vs[tid] = __ldg(a.v_in + node0 * 3 + tid);
    }
    __syncthreads();

    for (int it = 0; it < a.T; ++it) {
      float* sv = a.saved ? a.saved + (int64_t)it * a.iter_stride : nullptr;  // h | M | U5 | x
      // ---- (a) h tile <- split(h) ; save h_k, x_k
      if (tid < nnode * 8) {
        int n = tid >> 3, j = tid & 7;
        float4 p0 = nb_ld4(hs + n * NB_H + 8 * j), p1 = nb_ld4(hs + n * NB_H + 8 * j + 4);
        float v[8] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w};
        nb_tc_store8(Hh, Hl, n, j, v);
        if (sv) {
          nb_st4(sv + (node0 + n) * NB_H + 8 * j, p0);
          nb_st4(sv + (node0 + n) * NB_H + 8 * j + 4, p1);
        }
      }
      if (sv && tid >= NT - nnode * 3) {
        const int idx = tid - (NT - nnode * 3);
        sv[3 * Nn * NB_H + node0 * 3 + idx] = xs[idx];
      }
      nb_fence_async_smem();
      nb_tc_fence_before();
      __syncthreads();
      // ---- (b) P = h W1r^T, Q = h W1c^T -> node tile rows [0, GN) and [GN, 2 GN)
      if (NB_ISSUER(0)) {
        nb_tc_fence_after();
        nb_issue_w3(tm + 192, sHh, sHl, NB_FS_SWH(2), NB_FS_SWL(2), false, idesc_node, 0u);
        nb_issue_w3(tm + 256, sHh, sHl, NB_FS_SWH(3), NB_FS_SWL(3), false, idesc_node, 0u);
        nb_mma_commit(bar);
      }
      // (the products are read out inside the first edge tile, after its geometry and edge-feature loads have been
      //  issued: those do not depend on P / Q, so their latency hides under the MMAs)

      // ---- (c) edge tiles
      for (int r0 = 0; r0 < R; r0 += NB_TILE) {
        const int nv = min(NB_TILE, R - r0);
        const bool valid = row < nv;
        float dx = 0.f, dy = 0.f, dz = 0.f, r2 = 0.f;
        float e[NB_MAX_EF];
#pragma unroll
        for (int f = 0; f < NB_MAX_EF; ++f) e[f] = 0.f;
        int li = 0, lj = 0;
        if (valid) {
          const uint32_t ri = rowinfo[r0 + row];
          li = ri & 0xff;
          lj = (ri >> 8) & 0xff;
          const int lg = ri >> 16;
          dx = xs[li * 3 + 0] - xs[lj * 3 + 0];
          dy = xs[li * 3 + 1] - xs[lj * 3 + 1];
          dz = xs[li * 3 + 2] - xs[lj * 3 + 2];
          r2 = dx * dx + dy * dy + dz * dz;
          if (cq == 1) {  // only the selector's second half carries the scalars
            const int64_t eoff = ((int64_t)((gt0 + lg) % g.B) * g.EPG + (r0 + row - lg * g.EPG)) * g.nef;
#pragma unroll
            for (int f = 0; f < NB_MAX_EF; ++f)
              if (f < g.nef) e[f] = __ldg(a.ef + eoff + f);
          }
        }
        if (r0 > 0) {  // the scatter MMAs of the previous tile have consumed Sel / T / F
          nb_mbar_wait(bar, phase);
          phase ^= 1;
          nb_tc_fence_after();
        } else {       // (b) read-out: P + b1 and Q rows of the unit's nodes -> node tile
          nb_mbar_wait(bar, phase);
          phase ^= 1;
          nb_tc_fence_after();
          float v[16];
          nb_tmem_ld16(tm + lane_base + 192 + (uint32_t)cb, v);
          if (nown && nl < nnode) {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] += vb1[cb + i];
            nb_tc_store8(Nh, Nl, nl, 2 * cq, v);
            nb_tc_store8(Nh, Nl, nl, 2 * cq + 1, v + 8);
          }
          nb_tmem_ld16(tm + lane_base + 256 + (uint32_t)cb, v);
          if (nown && nl < nnode) {
            nb_tc_store8(Nh, Nl, GN + nl, 2 * cq, v);
            nb_tc_store8(Nh, Nl, GN + nl, 2 * cq + 1, v + 8);
          }
          nb_tc_fence_before();
          // (the selector write below is followed by fence + __syncthreads before the gather reads the node tile)
        }
        if (cq < 2) nb_sel_write_row(Sel, row, cq, valid, li, GN + lj, r2, e);
        nb_fence_async_smem();
        nb_tc_fence_before();
        __syncthreads();
        if (NB_ISSUER(0)) {
          nb_tc_fence_after();
          nb_issue_gather(tm, sSel, sNh, sNl, 4, idesc_gat, 0u);
          nb_mma_commit(bar);
        }
        nb_mbar_wait(bar, phase);
        phase ^= 1;
        nb_tc_fence_after();
        {
          float v[16];
          nb_tmem_ld16(tm_mine, v);
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = nb_silu(v[i]);
          nb_fs_store16(nullptr, nullptr, row, cq, v, ta_hm, ta_lm);  // z1 is only ever an A operand
          nb_tmem_st_wait();
        }
        nb_tc_fence_before();
        __syncthreads();
        if (NB_ISSUER(0)) {
          nb_tc_fence_after();
          nb_issue_w3_ta(tm, ta_h, ta_l, NB_FS_SWH(0), NB_FS_SWL(0), false, idesc_fwd, 0u);
          nb_mma_commit(bar);
        }
        nb_mbar_wait(bar, phase);
        phase ^= 1;
        nb_tc_fence_after();
        {
          float v[16];
          nb_tmem_ld16(tm_mine, v);
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = nb_silu(v[i] + vb2[cb + i]);
          nb_fs_store16(Th, Tl, row, cq, v, ta_hm, ta_lm);  // shared-memory copy: B operand of the scatter
          nb_tmem_st_wait();
        }
        nb_fence_async_smem();
        nb_tc_fence_before();
        __syncthreads();
        if (NB_ISSUER(0)) {
          nb_tc_fence_after();
          nb_issue_w3_ta(tm, ta_h, ta_l, NB_FS_SWH(1), NB_FS_SWL(1), false, idesc_fwd, 0u);
          nb_mma_commit(bar);
          nb_issue_scatter(tm + 64, sSel, sTh, sTl, idesc_sc, r0 > 0 ? 1u : 0u);  // M_i += Sel^T m
        }
        nb_mbar_wait(bar, phase);
        phase ^= 1;
        nb_tc_fence_after();
        {
          float v[16];
          nb_tmem_ld16(tm_mine, v);
          float cp = 0.f;
#pragma unroll
          for (int i = 0; i < 16; ++i) cp = fmaf(vw4[cb + i], nb_silu(v[i] + vb3[cb + i]), cp);
          cpart[cq * NB_TILE + row] = cp;
        }
        nb_tc_fence_before();
        __syncthreads();
        if (cq == 0) {
          float c = (cpart[row] + cpart[NB_TILE + row]) + (cpart[2 * NB_TILE + row] + cpart[3 * NB_TILE + row]) + b4;
          float fx = dx * c, fy = dy * c, fz = dz * c;
          if (g.clamp_edge) {
            fx = fminf(fmaxf(fx, -100.f), 100.f);
            fy = fminf(fmaxf(fy, -100.f), 100.f);
            fz = fminf(fmaxf(fz, -100.f), 100.f);
          }
          const uint32_t px = nb_pack_split(fx), py = nb_pack_split(fy), pz = nb_pack_split(fz);
          *reinterpret_cast<uint4*>(Fh + row * 16) = make_uint4((px & 0xffffu) | (py << 16), pz & 0xffffu, 0u, 0u);
          *reinterpret_cast<uint4*>(Fl + row * 16) = make_uint4((px >> 16) | (py & 0xffff0000u), pz >> 16, 0u, 0u);
        }
        nb_fence_async_smem();
        __syncthreads();
        if (NB_ISSUER(0)) {
          nb_tc_fence_after();
          nb_issue_scatter8(tm + 128, sSel, sFh, sFl, idesc_sc8, r0 > 0 ? 1u : 0u);
          nb_mma_commit(bar);
        }
      }
      // ---- (d) unit read-out: M_i -> U tile (+ saved), Fsum_i -> integrator
      nb_mbar_wait(bar, phase);
      phase ^= 1;
      nb_tc_fence_after();
      {
        float v[16];
        nb_tmem_ld16(tm + lane_base + 64 + (uint32_t)cb, v);
        if (nown && nl < nnode) {
          nb_tc_store8(Uh, Ul, nl, 2 * cq, v);
          nb_tc_store8(Uh, Ul, nl, 2 * cq + 1, v + 8);
          if (sv) {
            float* dst = sv + Nn * NB_H + (node0 + nl) * NB_H + cb;
#pragma unroll
            for (int k = 0; k < 4; ++k) nb_st4(dst + 4 * k, make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]));
          }
        }
        float f4[4];
        nb_tmem_ld4(tm + lane_base + 128, f4);
        if (cq == 0 && nown && nl < nnode) {
#pragma unroll
          for (int d = 0; d < 3; ++d) {
            const float acc = f4[d] / cnt * a.cw;             // gcl.py:101-102
            const float vn = vs[nl * 3 + d] + acc * a.inv_T;  // gcl.py:116
            vs[nl * 3 + d] = vn;
            xs[nl * 3 + d] = xs[nl * 3 + d] + vn * a.inv_T;   // gcl.py:117
          }
        }
      }
      nb_fence_async_smem();
      nb_tc_fence_before();
      __syncthreads();
      // ---- (e) U5 = [h, M] W5^T + b5 ; h <- h + SiLU(U5) W6^T + b6
      if (NB_ISSUER(0)) {
        nb_tc_fence_after();
        nb_issue_w3(tm + 192, sHh, sHl, NB_FS_SWH(4), NB_FS_SWL(4), false, idesc_node, 0u);
        nb_issue_w3(tm + 192, sUh, sUl, NB_FS_SWH(5), NB_FS_SWL(5), false, idesc_node, 1u);
        nb_mma_commit(bar);
      }
      nb_mbar_wait(bar, phase);
      phase ^= 1;
      nb_tc_fence_after();
      {
        float v[16];
        nb_tmem_ld16(tm + lane_base + 192 + (uint32_t)cb, v);
        if (nown && nl < nnode) {
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] += vb5[cb + i];
          if (sv) {
            float* dst = sv + 2 * Nn * NB_H + (node0 + nl) * NB_H + cb;
#pragma unroll
            for (int k = 0; k < 4; ++k) nb_st4(dst + 4 * k, make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]));
          }
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = nb_silu(v[i]);
          nb_tc_store8(Uh, Ul, nl, 2 * cq, v);
          nb_tc_store8(Uh, Ul, nl, 2 * cq + 1, v + 8);
        }
      }
      nb_fence_async_smem();
      nb_tc_fence_before();
      __syncthreads();
      if (NB_ISSUER(0)) {
        nb_tc_fence_after();
        nb_issue_w3(tm + 192, sUh, sUl, NB_FS_SWH(6), NB_FS_SWL(6), false, idesc_node, 0u);
        nb_mma_commit(bar);
      }
      nb_mbar_wait(bar, phase);
      phase ^= 1;
      nb_tc_fence_after();
      {
        float v[16];
        nb_tmem_ld16(tm + lane_base + 192 + (uint32_t)cb, v);
        if (nown && nl < nnode) {
          float* hp = hs + nl * NB_H + cb;
#pragma unroll
          for (int i = 0; i < 16; ++i) hp[i] = (a.recurrent ? hp[i] : 0.f) + (v[i] + vb6[cb + i]);
        }
      }
      nb_tc_fence_before();
      __syncthreads();
    }
    // ---- write the unit's final state
    if (tid < nnode * 16) nb_st4(a.h_out + node0 * NB_H + tid * 4, nb_ld4(hs + tid * 4));
    if (tid < nnode * 3) {
      a.x_out[node0 * 3 + tid] = xs[tid];
      a.v_out[node0 * 3 + tid] = vs[tid];
    }
    __syncthreads();
  }
  nb_tc_fence_before();
  __syncthreads();
  if (warp == 0) nb_tmem_dealloc(tm, NB_FS_TMEM_COLS);
}

// ----------------------------------------------------------------------------- node-level backward between two edge sweeps
// SEGNO's backward walks the T sub-steps in reverse; between the edge-tile backward of sub-step k and that of sub-step
// k - 1 the node-level chain is (gcl.py:78-94 backwards; all products are data gradients, g_in = g_out W):
//   gh      = gh_k + gP_k W1[:, h_row] + gQ_k W1[:, h_col]          dL/dh entering sub-step k - 1 (edge_mlp.0's h halves)
//   GU5     = (gh W6) * SiLU'(U5_{k-1})                              node_mlp.2 backwards, through the activation
//   gh_{k-1} = GU5 W5[:, :64] (+ gh: residual) ;  gM = GU5 W5[:, 64:]  node_mlp.0 backwards: the h and the M halves
// followed by the integrator's backward (k_segno_integ_bwd).  These were four launches on the critical path of every
// sub-step (three k_gemm64_tc launches of 40 tiles each + the integrator); here they are ONE: a CTA owns a 128-row tile,
// stages the five pre-split weight images once (80 KB), and chains the three products through tensor memory — each
// result is split in registers and written back as the A operand of the next product, so nothing but the tensors the
// weight-gradient reduction needs later (gh, GU5) and the edge kernel's inputs (gM) goes to HBM.
// TMEM: [0,64) D1 | [64,128) D3 (h half) | [128,192) D3 (M half) | [192,256) A0 hi|lo | [256,320) A1 hi|lo.
struct NbSegnoNodeBwdArgs {
  int rows, recurrent;
  const unsigned char* img;   // 5 images, 16 KB each: W1 h_row | W1 h_col | W5 h half | W5 M half | W6  (segno_weight_images)
  const float *gP, *gQ;       // [rows][64], sub-step k  (unused by the HEAD instantiation: gh = gh_in as it is)
  float* gh_k;                // in: gh_k (partial) ; out: gh (total)
  const float* gh_in;         // HEAD only: dL/dh of the call's output (read-only; null = zero)
  const float* U5;            // [rows][64] pre-activations of sub-step k - 1
  float *GU5, *gh_km1, *gM;   // out, sub-step k - 1
  // integrator backward of sub-step k - 1 (gcl.py:101-102,116-117)
  int64_t n3;
  int N;
  float inv_T, cw;
  const float *gx, *gv;
  float *gv_out, *gFsum;
};
#define NB_SNB_SMEM (5 * 2 * NB_TC_TILE_BYTES(64) + 64 + 1024)

__device__ __forceinline__ void nb_snb_load32(const float* p, bool live, float (&v)[32]) {
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float4 t = live ? nb_ld4(p + 4 * k) : make_float4(0.f, 0.f, 0.f, 0.f);
    v[4 * k] = t.x; v[4 * k + 1] = t.y; v[4 * k + 2] = t.z; v[4 * k + 3] = t.w;
  }
}
__device__ __forceinline__ void nb_snb_store32(float* p, bool live, const float (&v)[32]) {
  if (!live) return;
#pragma unroll
  for (int k = 0; k < 8; ++k) nb_st4(p + 4 * k, make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]));
}

// HEAD: the first sub-step of the sweep — no edge gradients yet, gh = gh_in as it is (the first product is skipped)
template <bool HEAD>
__global__ void __launch_bounds__(NB_THREADS, 1) k_segno_node_bwd(NbSegnoNodeBwdArgs a) {
  NB_PDL_ENTER();
  extern __shared__ __align__(1024) unsigned char nb_smraw[];
  unsigned char* base = nb_smraw + ((1024u - (nb_smem_u32(nb_smraw) & 1023u)) & 1023u);
  uint64_t* bar = reinterpret_cast<uint64_t*>(base + 5 * 2 * NB_TC_TILE_BYTES(64));
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, hf = warp >> 2;
  const int row = 32 * q + lane, cb = 32 * hf;
  const int ntiles = (a.rows + NB_TILE - 1) / NB_TILE;
  // the first tile's rows are requested before anything else, the 80 KB of weight images in batches of ten independent
  // 16-byte loads per thread: the kernel is a latency chain, so every load that can be in flight early is
  float v[32], r[32], u[32];
  {
    const int64_t gr0 = (int64_t)blockIdx.x * NB_TILE + row;
    const bool live0 = (int)blockIdx.x < ntiles && gr0 < a.rows;
    if (!HEAD) {
      nb_snb_load32(a.gP + gr0 * NB_H + cb, live0, v);
      nb_snb_load32(a.gQ + gr0 * NB_H + cb, live0, u);
      nb_snb_load32(a.gh_k + gr0 * NB_H + cb, live0, r);
    } else {
      nb_snb_load32(a.gh_in + gr0 * NB_H + cb, live0 && a.gh_in, r);
    }
  }
  uint64_t* wbar = bar + 2;   // weight images have landed (one TMA bulk copy, see nb_bulk_g2s)
  if (tid == 0) {
    nb_mbar_init(bar, 1);
    nb_mbar_init(wbar, 1);
    nb_mbar_fence_init();
    nb_bulk_g2s(base, a.img, (uint32_t)(5 * 2 * NB_TC_TILE_BYTES(64)), wbar);
  }
  if (warp == 0) nb_tmem_alloc(tmem_slot, 512);
  {  // integrator backward: independent element-wise work, issued while the weight copies are in flight
    const float cnt = (float)(a.N - 1 > 1 ? a.N - 1 : 1);
    for (int64_t i = (int64_t)blockIdx.x * NB_THREADS + tid; i < a.n3; i += (int64_t)gridDim.x * NB_THREADS) {
      const float gxi = a.gx ? a.gx[i] : 0.f;
      const float gvt = (a.gv ? a.gv[i] : 0.f) + gxi * a.inv_T;
      a.gv_out[i] = gvt;
      a.gFsum[i] = gvt * a.inv_T * a.cw / cnt;
    }
  }
  nb_fence_async_smem();
  nb_tc_fence_before();
  __syncthreads();
  nb_tc_fence_after();
  const uint32_t tm = *tmem_slot;
  const uint32_t lane_base = (uint32_t)(32 * q) << 16;
  const uint32_t d1 = tm + lane_base + (uint32_t)cb;
  const uint32_t a0h = tm + 192, a0l = tm + 224, a1h = tm + 256, a1l = tm + 288;
  const uint32_t mine = lane_base + 16u * (uint32_t)hf;
  const uint32_t idesc_mn = nb_idesc_bf16(128, 64, 0, 1);
  const uint32_t sW = nb_smem_u32(base);
#define NB_SNB_WH(i) (sW + (uint32_t)(i) * 2u * (uint32_t)NB_TC_TILE_BYTES(64))
#define NB_SNB_WL(i) (NB_SNB_WH(i) + (uint32_t)NB_TC_TILE_BYTES(64))
  uint32_t phase = 0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t gr = (int64_t)tile * NB_TILE + row;
    const bool live = gr < a.rows;
    const int64_t off = gr * NB_H + cb;
    if (tile != (int)blockIdx.x) {   // (the first tile's rows are already in registers)
      if (!HEAD) {
        nb_snb_load32(a.gP + off, live, v);
        nb_snb_load32(a.gQ + off, live, u);
        nb_snb_load32(a.gh_k + off, live, r);
      } else {
        nb_snb_load32(a.gh_in + off, live && a.gh_in, r);
      }
    }
    if (!HEAD) {
      nb_store32_ta(nullptr, nullptr, row, hf, v, a0h + mine, a0l + mine);
      nb_store32_ta(nullptr, nullptr, row, hf, u, a1h + mine, a1l + mine);
      nb_tmem_st_wait();
      nb_tc_fence_before();
      __syncthreads();
      if (NB_ISSUER(0)) {
        if (tile == (int)blockIdx.x) nb_mbar_wait(wbar, 0);
        nb_tc_fence_after();
        nb_issue_w3_ta(tm, a0h, a0l, NB_SNB_WH(0), NB_SNB_WL(0), true, idesc_mn, 0u);
        nb_issue_w3_ta(tm, a1h, a1l, NB_SNB_WH(1), NB_SNB_WL(1), true, idesc_mn, 1u);
        nb_mma_commit(bar);
      }
      nb_snb_load32(a.U5 + off, live, u);   // requested under the MMAs
      nb_mbar_wait(bar, phase);
      phase ^= 1;
      nb_tc_fence_after();
      // ---- gh = gh_k + gP W1r + gQ W1c
      nb_tmem_ld32(d1, v);
#pragma unroll
      for (int i = 0; i < 32; ++i) r[i] += v[i];
      nb_snb_store32(a.gh_k + off, live, r);
    } else {
      nb_snb_load32(a.U5 + off, live, u);
    }
    nb_store32_ta(nullptr, nullptr, row, hf, r, a0h + mine, a0l + mine);
    nb_tmem_st_wait();
    nb_tc_fence_before();
    __syncthreads();
    if (NB_ISSUER(0)) {
      if (HEAD && tile == (int)blockIdx.x) nb_mbar_wait(wbar, 0);
      nb_tc_fence_after();
      nb_issue_w3_ta(tm, a0h, a0l, NB_SNB_WH(4), NB_SNB_WL(4), true, idesc_mn, 0u);
      nb_mma_commit(bar);
    }
    nb_mbar_wait(bar, phase);
    phase ^= 1;
    nb_tc_fence_after();
    // ---- GU5 = (gh W6) * SiLU'(U5)
    nb_tmem_ld32(d1, v);
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = live ? v[i] * nb_dsilu(u[i]) : 0.f;
    nb_snb_store32(a.GU5 + off, live, v);
    nb_store32_ta(nullptr, nullptr, row, hf, v, a0h + mine, a0l + mine);
    nb_tmem_st_wait();
    nb_tc_fence_before();
    __syncthreads();
    if (NB_ISSUER(0)) {
      nb_tc_fence_after();
      nb_issue_w3_ta(tm + 64, a0h, a0l, NB_SNB_WH(2), NB_SNB_WL(2), true, idesc_mn, 0u);
      nb_issue_w3_ta(tm + 128, a0h, a0l, NB_SNB_WH(3), NB_SNB_WL(3), true, idesc_mn, 0u);
      nb_mma_commit(bar);
    }
    nb_mbar_wait(bar, phase);
    phase ^= 1;
    nb_tc_fence_after();
    // ---- gh_{k-1} = GU5 W5a (+ gh) ; gM = GU5 W5b
    nb_tmem_ld32(d1 + 64, v);
    if (a.recurrent) {
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] += r[i];
    }
    nb_snb_store32(a.gh_km1 + off, live, v);
    nb_tmem_ld32(d1 + 128, v);
    nb_snb_store32(a.gM + off, live, v);
    nb_tc_fence_before();
  }
  if ((int)blockIdx.x >= ntiles && tid == 0) nb_mbar_wait(wbar, 0);   // never exit under a copy in flight
  nb_tc_fence_before();
  __syncthreads();
  if (warp == 0) nb_tmem_dealloc(tm, 512);
}
#endif  // NB_EMU
