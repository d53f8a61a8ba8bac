// nb_edge.cuh — the fused E_GCL edge tile (forward, and backward with edge-tile recompute).
//
// Replaces, per layer / integration sub-step, the reference's gather + cat + 4 Linear + scatter
// chain (EGNO/model/basic.py:168-175,182 ; SEGNO/models/models/gcl.py:104-109,74-83,97-102,87):
//
//   rij = x_i - x_j ; r2 = |rij|^2
//   z1  = SiLU(P_i + Q_j + w_rad r2 + W_ef e_ij)        P = W1[:,h_row] h + b1, Q = W1[:,h_col] h  (per node)
//   m   = SiLU(W2 z1 + b2)                              phi_e
//   c   = w4 . SiLU(W3 m + b3) + b4                     phi_x
//   M_i = sum_j m_ij ;  Fsum_i = sum_j rij c            (SEGNO clamps rij c to +-100 per edge first)
//
// Nothing per-edge ever reaches HBM: the [E,131] concat of the reference (510 MB at cfg3) is replaced
// by the per-node pre-projections P, Q, and the receiver reductions run over the contiguous N-1 edge
// rows of each receiver inside the tile — deterministic, no atomics.
//
// Work decomposition: a *unit* is G consecutive graph-instances (graph-time pairs, index gt = t*B + b,
// node index gt*N + i, the reference's t-major order).  Its G*N*(N-1) edge rows are processed in tiles
// of 128 rows by one CTA; row r of the unit is edge (i -> j) of local graph lg with
//   lg = r / (N(N-1)),  rem = r % (N(N-1)),  i = rem / (N-1),  jj = rem % (N-1),  j = jj + (jj >= i)
// i.e. exactly the canonical edge order of dataset_simple.py:64-71, so `r / (N-1)` is the receiver's
// node index inside the unit.  Edge features are shared across time: index ((gt % B)*N(N-1) + rem).
#pragma once
#include "nb_common.cuh"

struct NbEdgeW {
  const float* W1;  // first edge layer [64][ldw1]; only the radial / edge-feature columns are read here
  int ldw1, col_rad, col_ef;
  const float *W2, *b2, *W3, *b3, *w4, *b4;
};

struct NbEdgeGeom {
  int N, EPG, NGT, B, G, n_units, nef;
  int clamp_edge;  // SEGNO: clamp(rij*c, +-100) per edge before the mean (gcl.py:100)
  int blk, nI, nJ, IB, JB;  // selector kernels, N > 27: a graph is walked in (IB receivers x JB senders) blocks, one tile each
  int multi;                // EGNO num_inputs > 1: edge features are per input frame, [L][B*EPG][nef]
  int tmap[NB_MAX_T];       // frame t -> input index (EGNO/utils.py:115-131)
};
// graph index into the edge-feature array of graph-instance gt = t*B + b  (shared across time unless `multi`)
__device__ __forceinline__ int nb_ef_graph(const NbEdgeGeom& g, int gt) {
  const int b = gt % g.B;
  return g.multi ? g.tmap[gt / g.B] * g.B + b : b;
}

struct NbEdgeFwdArgs {
  NbEdgeGeom g;
  NbEdgeW w;
  const float* x;   // [NGT*N][3]
  const float* P;   // [NGT*N][64]
  const float* Q;   // [NGT*N][64]
  const float* ef;  // [B*EPG][nef]
  float* M;         // [NGT*N][64]
  float* Fsum;      // [NGT*N][3]
};

// shared-memory row arrays of one tile (128 rows)
struct NbRowInfo {
  int* rI;     // receiver node (global)
  int* rJ;     // sender node (global)
  float* rR2;  // |rij|^2
  float* rD;   // [3][128] rij
  float* rE;   // [NB_MAX_EF][128]
};

__device__ __forceinline__ void nb_row_setup(const NbEdgeGeom& g, const float* __restrict__ x,
                                             const float* __restrict__ ef, int gt0, int r0, int nv, int tid,
                                             const NbRowInfo& ri) {
  if (tid < NB_TILE) {
    int ni, nj;
    float dx = 0.f, dy = 0.f, dz = 0.f;
    float e[NB_MAX_EF];
#pragma unroll
    for (int f = 0; f < NB_MAX_EF; ++f) e[f] = 0.f;
    if (tid < nv) {
      int r = r0 + tid;
      int lg = r / g.EPG, rem = r - lg * g.EPG;
      int i = rem / (g.N - 1), jj = rem - i * (g.N - 1);
      int j = jj + (jj >= i ? 1 : 0);
      int gt = gt0 + lg;
      ni = gt * g.N + i;
      nj = gt * g.N + j;
      dx = __ldg(x + (int64_t)ni * 3 + 0) - __ldg(x + (int64_t)nj * 3 + 0);
      dy = __ldg(x + (int64_t)ni * 3 + 1) - __ldg(x + (int64_t)nj * 3 + 1);
      dz = __ldg(x + (int64_t)ni * 3 + 2) - __ldg(x + (int64_t)nj * 3 + 2);
      int64_t eoff = ((int64_t)nb_ef_graph(g, gt) * g.EPG + rem) * g.nef;
#pragma unroll
      for (int f = 0; f < NB_MAX_EF; ++f)
        if (f < g.nef) e[f] = __ldg(ef + eoff + f);
    } else {
      ni = nj = gt0 * g.N;  // padded row: valid address, zero geometry; its results are never reduced
    }
    ri.rI[tid] = ni;
    ri.rJ[tid] = nj;
    ri.rD[tid] = dx;
    ri.rD[NB_TILE + tid] = dy;
    ri.rD[2 * NB_TILE + tid] = dz;
    ri.rR2[tid] = dx * dx + dy * dy + dz * dz;
#pragma unroll
    for (int f = 0; f < NB_MAX_EF; ++f) ri.rE[f * NB_TILE + tid] = e[f];
  }
}

// pre-activation of the first edge layer for the thread's 4 columns of row `row`
__device__ __forceinline__ float4 nb_pre1(const float* __restrict__ P, const float* __restrict__ Q,
                                          const NbRowInfo& ri, int row, int tx, const float4& wr,
                                          const float4 (&we)[NB_MAX_EF], int nef) {
  float4 p = nb_ld4(P + (int64_t)ri.rI[row] * NB_H + tx * 4);
  float4 q = nb_ld4(Q + (int64_t)ri.rJ[row] * NB_H + tx * 4);
  float r2 = ri.rR2[row];
  float4 v = make_float4(p.x + q.x, p.y + q.y, p.z + q.z, p.w + q.w);
  v.x = fmaf(wr.x, r2, v.x);
  v.y = fmaf(wr.y, r2, v.y);
  v.z = fmaf(wr.z, r2, v.z);
  v.w = fmaf(wr.w, r2, v.w);
#pragma unroll
  for (int f = 0; f < NB_MAX_EF; ++f)
    if (f < nef) {
      float e = ri.rE[f * NB_TILE + row];
      v.x = fmaf(we[f].x, e, v.x);
      v.y = fmaf(we[f].y, e, v.y);
      v.z = fmaf(we[f].z, e, v.z);
      v.w = fmaf(we[f].w, e, v.w);
    }
  return v;
}

__device__ __forceinline__ void nb_load_w1_slices(const NbEdgeW& w, int nef, int tx, float4& wr,
                                                  float4 (&we)[NB_MAX_EF]) {
  const float* W1 = w.W1;
  int c = tx * 4;
  wr = make_float4(__ldg(W1 + (int64_t)(c + 0) * w.ldw1 + w.col_rad), __ldg(W1 + (int64_t)(c + 1) * w.ldw1 + w.col_rad),
                   __ldg(W1 + (int64_t)(c + 2) * w.ldw1 + w.col_rad), __ldg(W1 + (int64_t)(c + 3) * w.ldw1 + w.col_rad));
#pragma unroll
  for (int f = 0; f < NB_MAX_EF; ++f) {
    we[f] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (f < nef)
      we[f] = make_float4(
          __ldg(W1 + (int64_t)(c + 0) * w.ldw1 + w.col_ef + f), __ldg(W1 + (int64_t)(c + 1) * w.ldw1 + w.col_ef + f),
          __ldg(W1 + (int64_t)(c + 2) * w.ldw1 + w.col_ef + f), __ldg(W1 + (int64_t)(c + 3) * w.ldw1 + w.col_ef + f));
  }
}

#define NB_EDGE_FWD_SMEM_FLOATS (2 * NB_H * NB_H + 3 * NB_H + NB_TILE * NB_LDA + NB_TILE * (2 + 1 + 3 + NB_MAX_EF + 1))

__global__ void __launch_bounds__(NB_THREADS) k_edge_fwd(NbEdgeFwdArgs a) {
  NB_PDL_ENTER();
  NB_DYN_SMEM(sm);
  float* W2t = sm;                  // [k][o]
  float* W3t = W2t + NB_H * NB_H;   // [k][o]
  float* vb2 = W3t + NB_H * NB_H;
  float* vb3 = vb2 + NB_H;
  float* vw4 = vb3 + NB_H;
  float* As = vw4 + NB_H;           // [128][68]
  NbRowInfo ri;
  ri.rI = reinterpret_cast<int*>(As + NB_TILE * NB_LDA);
  ri.rJ = ri.rI + NB_TILE;
  ri.rR2 = reinterpret_cast<float*>(ri.rJ + NB_TILE);
  ri.rD = ri.rR2 + NB_TILE;
  ri.rE = ri.rD + 3 * NB_TILE;
  float* rC = ri.rE + NB_MAX_EF * NB_TILE;

  const NbEdgeGeom g = a.g;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;

  nb_stage_b(W2t, a.w.W2, 1, NB_H, 1.f, tid);  // Bs[k][o] = W2[o][k]
  nb_stage_b(W3t, a.w.W3, 1, NB_H, 1.f, tid);
  if (tid < NB_H) {
    vb2[tid] = __ldg(a.w.b2 + tid);
    vb3[tid] = __ldg(a.w.b3 + tid);
    vw4[tid] = __ldg(a.w.w4 + tid);
  }
  float4 wr, we[NB_MAX_EF];
  nb_load_w1_slices(a.w, g.nef, tx, wr, we);
  const float b4 = __ldg(a.w.b4);
  __syncthreads();
  const float4 b2v = nb_ld4(vb2 + tx * 4), b3v = nb_ld4(vb3 + tx * 4), w4v = nb_ld4(vw4 + tx * 4);
  const int Nm1 = g.N - 1;

  for (int u = blockIdx.x; u < g.n_units; u += gridDim.x) {
    const int gt0 = u * g.G;
    const int ngt = min(g.G, g.NGT - gt0);
    const int R = ngt * g.EPG;
    const int64_t node0 = (int64_t)gt0 * g.N;
    for (int r0 = 0; r0 < R; r0 += NB_TILE) {
      const int nv = min(NB_TILE, R - r0);
      // 1. per-row geometry
      nb_row_setup(g, a.x, a.ef, gt0, r0, nv, tid, ri);
      __syncthreads();
      // 2. z1 = SiLU(pre1) -> As
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        int row = ty + 16 * q;
        float4 v = nb_pre1(a.P, a.Q, ri, row, tx, wr, we, g.nef);
        nb_st4(As + row * NB_LDA + tx * 4, make_float4(nb_silu(v.x), nb_silu(v.y), nb_silu(v.z), nb_silu(v.w)));
      }
      __syncthreads();
      // 3. pre2 = z1 W2^T
      float acc[8][4];
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.f;
      nb_tile_gemm<8>(As, W2t, acc, ty, tx);
      __syncthreads();
      // 4. m = SiLU(pre2 + b2) -> As
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        int row = ty + 16 * q;
        nb_st4(As + row * NB_LDA + tx * 4,
               make_float4(nb_silu(acc[q][0] + b2v.x), nb_silu(acc[q][1] + b2v.y), nb_silu(acc[q][2] + b2v.z),
                           nb_silu(acc[q][3] + b2v.w)));
      }
      __syncthreads();
      // 5a. M_i += sum over the receiver's rows inside this tile (receiver s = unit row / (N-1))
      const int s0 = r0 / Nm1, s1 = (r0 + nv - 1) / Nm1;
      {
        const int c = tid & 63, part = tid >> 6;
        for (int s = s0 + part; s <= s1; s += 4) {
          int ra = max(s * Nm1, r0), rb = min((s + 1) * Nm1, r0 + nv);
          float sum = 0.f;
          for (int r = ra; r < rb; ++r) sum += As[(r - r0) * NB_LDA + c];
          float* dst = a.M + (node0 + s) * NB_H + c;
          if (s * Nm1 >= r0) *dst = sum;  // first tile touching this receiver
          else *dst += sum;               // continuation from the previous tile (same CTA, after a barrier)
        }
      }
      // 5b. pre3 = m W3^T ; c = w4 . SiLU(pre3 + b3) + b4
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.f;
      nb_tile_gemm<8>(As, W3t, acc, ty, tx);
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        float cp = w4v.x * nb_silu(acc[q][0] + b3v.x) + w4v.y * nb_silu(acc[q][1] + b3v.y) +
                   w4v.z * nb_silu(acc[q][2] + b3v.z) + w4v.w * nb_silu(acc[q][3] + b3v.w);
        cp = nb_reduce_tx(cp);
        if (tx == 0) rC[ty + 16 * q] = cp + b4;
      }
      __syncthreads();
      // 6. Fsum_i += sum_j rij * c
      for (int idx = tid; idx < (s1 - s0 + 1) * 3; idx += NB_THREADS) {
        int s = s0 + idx / 3, d = idx % 3;
        int ra = max(s * Nm1, r0), rb = min((s + 1) * Nm1, r0 + nv);
        float sum = 0.f;
        for (int r = ra; r < rb; ++r) {
          float f = ri.rD[d * NB_TILE + (r - r0)] * rC[r - r0];
          if (g.clamp_edge) f = fminf(fmaxf(f, -100.f), 100.f);
          sum += f;
        }
        float* dst = a.Fsum + (node0 + s) * 3 + d;
        if (s * Nm1 >= r0) *dst = sum;
        else *dst += sum;
      }
      __syncthreads();
    }
  }
}

// ============================================================================= backward
// Partial-sum slice written by each CTA (reduced by k_finalize):
#define NB_EB_GW2 0
#define NB_EB_GW3 (NB_H * NB_H)
#define NB_EB_GB2 (2 * NB_H * NB_H)
#define NB_EB_GB3 (NB_EB_GB2 + NB_H)
#define NB_EB_GW4 (NB_EB_GB3 + NB_H)
#define NB_EB_GWR (NB_EB_GW4 + NB_H)
#define NB_EB_GWE (NB_EB_GWR + NB_H)                 // [NB_MAX_EF][64]
#define NB_EB_GB4 (NB_EB_GWE + NB_MAX_EF * NB_H)     // 1 (+63 pad)
#define NB_EB_PLEN (NB_EB_GB4 + NB_H)

struct NbEdgeBwdArgs {
  NbEdgeGeom g;
  NbEdgeW w;
  const float* x;
  const float* P;
  const float* Q;
  const float* ef;
  const float* gM;     // [NGT*N][64]
  const float* gFsum;  // [NGT*N][3]
  float* gP;           // [NGT*N][64]  overwritten
  float* gQ;           // [NGT*N][64]  overwritten
  float* gx;           // [NGT*N][3]   accumulated into
  float* partial;      // [gridDim.x][NB_EB_PLEN]
  // EGRAD instantiations only: dL/d(edge features) of every replicated edge row, [NGT*EPG][nef], row gt*EPG + e_local
  // (overwritten, one plain store per row and feature)
  float* gef;
};

#define NB_EDGE_BWD_SMEM_FLOATS(GN) \
  (4 * NB_H * NB_H + 4 * NB_H + 3 * NB_TILE * NB_LDA + NB_TILE * (2 + 1 + 3 + NB_MAX_EF + 3 + 3) + (GN) * (NB_H + 3))

// EGRAD: also dL/de = W_e^T g1 per edge row into a.gef (false: the kernel without input gradients, unchanged)
template <bool EGRAD>
__global__ void __launch_bounds__(NB_THREADS) k_edge_bwd(NbEdgeBwdArgs a) {
  NB_PDL_ENTER();
  NB_DYN_SMEM(sm);
  float* W2t = sm;                 // [k][o]  (forward recompute)
  float* W3t = W2t + NB_H * NB_H;
  float* W2n = W3t + NB_H * NB_H;  // [o][k]  (data gradients)
  float* W3n = W2n + NB_H * NB_H;
  float* vb2 = W3n + NB_H * NB_H;
  float* vb3 = vb2 + NB_H;
  float* vw4 = vb3 + NB_H;
  float* vwr = vw4 + NB_H;
  float* Z1s = vwr + NB_H;                 // z1 tile
  float* Ms = Z1s + NB_TILE * NB_LDA;      // m tile
  float* Gs = Ms + NB_TILE * NB_LDA;       // gradient tile (g3 -> g2 -> g1)
  NbRowInfo ri;
  ri.rI = reinterpret_cast<int*>(Gs + NB_TILE * NB_LDA);
  ri.rJ = ri.rI + NB_TILE;
  ri.rR2 = reinterpret_cast<float*>(ri.rJ + NB_TILE);
  ri.rD = ri.rR2 + NB_TILE;
  ri.rE = ri.rD + 3 * NB_TILE;
  float* rGF = ri.rE + NB_MAX_EF * NB_TILE;  // [3][128] dL/dFsum of the row's receiver
  float* rG = rGF + 3 * NB_TILE;             // [3][128] dL/drij
  float* gQacc = rG + 3 * NB_TILE;           // [G*N][64]
  float* gxacc = gQacc + a.g.G * a.g.N * NB_H;  // [G*N][3]

  const NbEdgeGeom g = a.g;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int wk = tid & 15, wo = tid >> 4;  // weight-gradient mapping

  nb_stage_b(W2t, a.w.W2, 1, NB_H, 1.f, tid);
  nb_stage_b(W3t, a.w.W3, 1, NB_H, 1.f, tid);
  nb_stage_b(W2n, a.w.W2, NB_H, 1, 1.f, tid);
  nb_stage_b(W3n, a.w.W3, NB_H, 1, 1.f, tid);
  if (tid < NB_H) {
    vb2[tid] = __ldg(a.w.b2 + tid);
    vb3[tid] = __ldg(a.w.b3 + tid);
    vw4[tid] = __ldg(a.w.w4 + tid);
    vwr[tid] = __ldg(a.w.W1 + (int64_t)tid * a.w.ldw1 + a.w.col_rad);
  }
  float4 wr, we[NB_MAX_EF];
  nb_load_w1_slices(a.w, g.nef, tx, wr, we);
  const float b4 = __ldg(a.w.b4);
  __syncthreads();
  const float4 b2v = nb_ld4(vb2 + tx * 4), b3v = nb_ld4(vb3 + tx * 4), w4v = nb_ld4(vw4 + tx * 4);
  const int Nm1 = g.N - 1;

  // per-thread accumulators that live across the whole kernel
  float gW2[4][4], gW3[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
    gW2[i][0] = gW2[i][1] = gW2[i][2] = gW2[i][3] = gW3[i][0] = gW3[i][1] = gW3[i][2] = gW3[i][3] = 0.f;
  float gb2[4] = {0.f, 0.f, 0.f, 0.f}, gb3[4] = {0.f, 0.f, 0.f, 0.f}, gw4[4] = {0.f, 0.f, 0.f, 0.f};
  float gwr[4] = {0.f, 0.f, 0.f, 0.f};
  float gwe[NB_MAX_EF][4];
#pragma unroll
  for (int f = 0; f < NB_MAX_EF; ++f) gwe[f][0] = gwe[f][1] = gwe[f][2] = gwe[f][3] = 0.f;
  float gb4 = 0.f;

  for (int u = blockIdx.x; u < g.n_units; u += gridDim.x) {
    const int gt0 = u * g.G;
    const int ngt = min(g.G, g.NGT - gt0);
    const int R = ngt * g.EPG;
    const int nnode = ngt * g.N;
    const int64_t node0 = (int64_t)gt0 * g.N;
    for (int idx = tid; idx < nnode * NB_H; idx += NB_THREADS) gQacc[idx] = 0.f;
    for (int idx = tid; idx < nnode * 3; idx += NB_THREADS) gxacc[idx] = 0.f;
    // (the barrier after row setup orders these writes before their first use)

    for (int r0 = 0; r0 < R; r0 += NB_TILE) {
      const int nv = min(NB_TILE, R - r0);
      // 1. per-row geometry + the receiver's dL/dFsum
      nb_row_setup(g, a.x, a.ef, gt0, r0, nv, tid, ri);
      if (tid < NB_TILE) {
        int64_t ni = (tid < nv) ? (node0 + (r0 + tid) / Nm1) : node0;
        float sc = (tid < nv) ? 1.f : 0.f;
        rGF[tid] = sc * __ldg(a.gFsum + ni * 3 + 0);
        rGF[NB_TILE + tid] = sc * __ldg(a.gFsum + ni * 3 + 1);
        rGF[2 * NB_TILE + tid] = sc * __ldg(a.gFsum + ni * 3 + 2);
      }
      __syncthreads();
      // 2. recompute z1 (+ SiLU' kept in registers)
      float d1[8][4], d2[8][4], acc[8][4];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        int row = ty + 16 * q;
        float4 v = nb_pre1(a.P, a.Q, ri, row, tx, wr, we, g.nef);
        float4 z;
        nb_silu_grad(v.x, z.x, d1[q][0]);
        nb_silu_grad(v.y, z.y, d1[q][1]);
        nb_silu_grad(v.z, z.z, d1[q][2]);
        nb_silu_grad(v.w, z.w, d1[q][3]);
        nb_st4(Z1s + row * NB_LDA + tx * 4, z);
      }
      __syncthreads();
      // 3. recompute m
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.f;
      nb_tile_gemm<8>(Z1s, W2t, acc, ty, tx);
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        int row = ty + 16 * q;
        float4 mv;
        nb_silu_grad(acc[q][0] + b2v.x, mv.x, d2[q][0]);
        nb_silu_grad(acc[q][1] + b2v.y, mv.y, d2[q][1]);
        nb_silu_grad(acc[q][2] + b2v.z, mv.z, d2[q][2]);
        nb_silu_grad(acc[q][3] + b2v.w, mv.w, d2[q][3]);
        nb_st4(Ms + row * NB_LDA + tx * 4, mv);
      }
      __syncthreads();
      // 4. recompute phi_x, start the backward: g3 = dL/dpre3
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.f;
      nb_tile_gemm<8>(Ms, W3t, acc, ty, tx);
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        int row = ty + 16 * q;
        float z3[4], d3[4];
        nb_silu_grad(acc[q][0] + b3v.x, z3[0], d3[0]);
        nb_silu_grad(acc[q][1] + b3v.y, z3[1], d3[1]);
        nb_silu_grad(acc[q][2] + b3v.z, z3[2], d3[2]);
        nb_silu_grad(acc[q][3] + b3v.w, z3[3], d3[3]);
        float c = nb_reduce_tx(w4v.x * z3[0] + w4v.y * z3[1] + w4v.z * z3[2] + w4v.w * z3[3]) + b4;
        float rx = ri.rD[row], ry = ri.rD[NB_TILE + row], rz = ri.rD[2 * NB_TILE + row];
        float gfx = rGF[row], gfy = rGF[NB_TILE + row], gfz = rGF[2 * NB_TILE + row];
        if (g.clamp_edge) {  // clamp(rij*c) passes gradient only inside [-100, 100]
          float fx = rx * c, fy = ry * c, fz = rz * c;
          if (!(fx >= -100.f && fx <= 100.f)) gfx = 0.f;
          if (!(fy >= -100.f && fy <= 100.f)) gfy = 0.f;
          if (!(fz >= -100.f && fz <= 100.f)) gfz = 0.f;
        }
        float gc = rx * gfx + ry * gfy + rz * gfz;  // dL/dc   (0 for padded rows: rGF == 0)
        if (tx == 0) {
          rG[row] = c * gfx;  // dL/drij through f = rij * c
          rG[NB_TILE + row] = c * gfy;
          rG[2 * NB_TILE + row] = c * gfz;
          gb4 += gc;
        }
        float g3[4] = {gc * w4v.x * d3[0], gc * w4v.y * d3[1], gc * w4v.z * d3[2], gc * w4v.w * d3[3]};
#pragma unroll
        for (int c4 = 0; c4 < 4; ++c4) {
          gw4[c4] = fmaf(gc, z3[c4], gw4[c4]);
          gb3[c4] += g3[c4];
        }
        nb_st4(Gs + row * NB_LDA + tx * 4, make_float4(g3[0], g3[1], g3[2], g3[3]));
      }
      __syncthreads();
      // 5. dW3 += g3^T m ;  gm = g3 W3 + gM_i ;  g2 = gm * SiLU'(pre2)
      nb_tile_wgrad(Gs, Ms, nv, gW3, wo, wk);
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.f;
      nb_tile_gemm<8>(Gs, W3n, acc, ty, tx);
      __syncthreads();
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        int row = ty + 16 * q;
        float4 gm = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row < nv) gm = nb_ld4(a.gM + (int64_t)ri.rI[row] * NB_H + tx * 4);
        float g2[4] = {(acc[q][0] + gm.x) * d2[q][0], (acc[q][1] + gm.y) * d2[q][1], (acc[q][2] + gm.z) * d2[q][2],
                       (acc[q][3] + gm.w) * d2[q][3]};
        if (row >= nv) g2[0] = g2[1] = g2[2] = g2[3] = 0.f;
#pragma unroll
        for (int c4 = 0; c4 < 4; ++c4) gb2[c4] += g2[c4];
        nb_st4(Gs + row * NB_LDA + tx * 4, make_float4(g2[0], g2[1], g2[2], g2[3]));
      }
      __syncthreads();
      // 6. dW2 += g2^T z1 ;  gz1 = g2 W2 ;  g1 = gz1 * SiLU'(pre1)
      nb_tile_wgrad(Gs, Z1s, nv, gW2, wo, wk);
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.f;
      nb_tile_gemm<8>(Gs, W2n, acc, ty, tx);
      __syncthreads();
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        int row = ty + 16 * q;
        float g1[4] = {acc[q][0] * d1[q][0], acc[q][1] * d1[q][1], acc[q][2] * d1[q][2], acc[q][3] * d1[q][3]};
        float r2 = ri.rR2[row];
#pragma unroll
        for (int c4 = 0; c4 < 4; ++c4) gwr[c4] = fmaf(g1[c4], r2, gwr[c4]);
#pragma unroll
        for (int f = 0; f < NB_MAX_EF; ++f)
          if (f < g.nef) {
            float e = ri.rE[f * NB_TILE + row];
#pragma unroll
            for (int c4 = 0; c4 < 4; ++c4) gwe[f][c4] = fmaf(g1[c4], e, gwe[f][c4]);
          }
        // dL/dr2 = w_rad . g1 ;  dL/drij += 2 rij dL/dr2
        float gr2 = nb_reduce_tx(wr.x * g1[0] + wr.y * g1[1] + wr.z * g1[2] + wr.w * g1[3]);
        if (tx == 0) {
          rG[row] = fmaf(2.f * ri.rD[row], gr2, rG[row]);
          rG[NB_TILE + row] = fmaf(2.f * ri.rD[NB_TILE + row], gr2, rG[NB_TILE + row]);
          rG[2 * NB_TILE + row] = fmaf(2.f * ri.rD[2 * NB_TILE + row], gr2, rG[2 * NB_TILE + row]);
        }
        if constexpr (EGRAD) {  // dL/de_f = w_ef[f] . g1: the unit's rows are the replicated rows gt0*EPG + r
#pragma unroll
          for (int f = 0; f < NB_MAX_EF; ++f)
            if (f < g.nef) {
              const float ge = nb_reduce_tx(we[f].x * g1[0] + we[f].y * g1[1] + we[f].z * g1[2] + we[f].w * g1[3]);
              if (tx == 0 && row < nv) a.gef[((int64_t)gt0 * g.EPG + r0 + row) * g.nef + f] = ge;
            }
        }
        nb_st4(Gs + row * NB_LDA + tx * 4, make_float4(g1[0], g1[1], g1[2], g1[3]));
      }
      __syncthreads();
      // 7. node-level reductions of g1 (receiver rows -> gP, sender rows -> gQ) and of dL/drij -> gx
      const int s0 = r0 / Nm1, s1 = (r0 + nv - 1) / Nm1;  // receivers (unit-local node ids) touched by the tile
      {
        const int c = tid & 63, part = tid >> 6;
        for (int s = s0 + part; s <= s1; s += 4) {
          int ra = max(s * Nm1, r0), rb = min((s + 1) * Nm1, r0 + nv);
          float sum = 0.f;
          for (int r = ra; r < rb; ++r) sum += Gs[(r - r0) * NB_LDA + c];
          float* dst = a.gP + (node0 + s) * NB_H + c;
          if (s * Nm1 >= r0) *dst = sum;
          else *dst += sum;
        }
        const int v0 = (s0 / g.N) * g.N, v1 = (s1 / g.N + 1) * g.N;  // senders of the touched graphs
        for (int v = v0 + part; v < v1; v += 4) {
          int lg = v / g.N, j = v - lg * g.N;
          int sa = max(s0, lg * g.N), sb = min(s1, lg * g.N + g.N - 1);
          float sum = 0.f;
          for (int s = sa; s <= sb; ++s) {
            int i = s - lg * g.N;
            if (i == j) continue;
            int r = s * Nm1 + (j < i ? j : j - 1);
            if (r < r0 || r >= r0 + nv) continue;
            sum += Gs[(r - r0) * NB_LDA + c];
          }
          gQacc[v * NB_H + c] += sum;
        }
      }
      {
        const int v0 = (s0 / g.N) * g.N, v1 = (s1 / g.N + 1) * g.N;
        for (int idx = tid; idx < (v1 - v0) * 3; idx += NB_THREADS) {
          int v = v0 + idx / 3, d = idx % 3;
          int lg = v / g.N, j = v - lg * g.N;
          float sum = 0.f;
          // as receiver: + dL/drij over its rows in this tile
          if (v >= s0 && v <= s1) {
            int ra = max(v * Nm1, r0), rb = min((v + 1) * Nm1, r0 + nv);
            for (int r = ra; r < rb; ++r) sum += rG[d * NB_TILE + (r - r0)];
          }
          // as sender: - dL/drij over rows (i -> v)
          int sa = max(s0, lg * g.N), sb = min(s1, lg * g.N + g.N - 1);
          for (int s = sa; s <= sb; ++s) {
            int i = s - lg * g.N;
            if (i == j) continue;
            int r = s * Nm1 + (j < i ? j : j - 1);
            if (r < r0 || r >= r0 + nv) continue;
            sum -= rG[d * NB_TILE + (r - r0)];
          }
          gxacc[v * 3 + d] += sum;
        }
      }
      __syncthreads();
    }
    // unit epilogue: sender sums and coordinate gradients of this unit's nodes
    for (int idx = tid; idx < nnode * NB_H; idx += NB_THREADS) a.gQ[node0 * NB_H + idx] = gQacc[idx];
    for (int idx = tid; idx < nnode * 3; idx += NB_THREADS) a.gx[node0 * 3 + idx] += gxacc[idx];
    __syncthreads();
  }

  // ---- CTA epilogue: reduce the column accumulators over the 16 ty groups, write the partial slice
  float* out = a.partial + (int64_t)blockIdx.x * NB_EB_PLEN;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    nb_st4(out + NB_EB_GW2 + (wo * 4 + i) * NB_H + wk * 4, make_float4(gW2[i][0], gW2[i][1], gW2[i][2], gW2[i][3]));
    nb_st4(out + NB_EB_GW3 + (wo * 4 + i) * NB_H + wk * 4, make_float4(gW3[i][0], gW3[i][1], gW3[i][2], gW3[i][3]));
  }
  float* red = Gs;  // [16][64] scratch (all tile work is done)
  const int nvec = 4 + NB_MAX_EF;
  for (int vsel = 0; vsel < nvec; ++vsel) {
    float4 val;
    if (vsel == 0) val = make_float4(gb2[0], gb2[1], gb2[2], gb2[3]);
    else if (vsel == 1) val = make_float4(gb3[0], gb3[1], gb3[2], gb3[3]);
    else if (vsel == 2) val = make_float4(gw4[0], gw4[1], gw4[2], gw4[3]);
    else if (vsel == 3) val = make_float4(gwr[0], gwr[1], gwr[2], gwr[3]);
    else {
      int f = vsel - 4;
      val = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int ff = 0; ff < NB_MAX_EF; ++ff)
        if (ff == f) val = make_float4(gwe[ff][0], gwe[ff][1], gwe[ff][2], gwe[ff][3]);
    }
    __syncthreads();
    nb_st4(red + ty * NB_H + tx * 4, val);
    __syncthreads();
    if (tid < NB_H) {
      float s = 0.f;
      for (int t = 0; t < 16; ++t) s += red[t * NB_H + tid];
      int off = vsel == 0 ? NB_EB_GB2 : vsel == 1 ? NB_EB_GB3 : vsel == 2 ? NB_EB_GW4 : vsel == 3 ? NB_EB_GWR
                                                                                           : NB_EB_GWE + (vsel - 4) * NB_H;
      out[off + tid] = s;
    }
  }
  __syncthreads();
  if (tx == 0) red[ty] = gb4;
  __syncthreads();
  if (tid < NB_H) {
    float s = 0.f;
    if (tid == 0)
      for (int t = 0; t < 16; ++t) s += red[t];
    out[NB_EB_GB4 + tid] = s;
  }
}
