// nb_edge_sel.cuh — fused E_GCL edge tiles with ALL gathers and scatters on the tensor cores.
//
// Same math and unit / tile decomposition as nb_edge.cuh.  What changes is how per-node data reaches
// the edge rows and how per-edge data is reduced back onto nodes: both go through a one-hot *selector* tile
//
//     Sel[row][col]   (128 edge rows x 64 columns, bf16, exact 0/1 entries plus a few split scalars)
//       col li          (0 <= li < GN)         1 iff the row's receiver is local node li
//       col GN + lj                            1 iff the row's sender   is local node lj
//       cols 54..63                            r2_hi, r2_lo, e0_hi, e0_lo, ... e3_hi, e3_lo   (split-bf16 scalars)
//
// and a per-unit node tile  NT[k][0:64]  (rows: P of the unit's nodes | Q of the unit's nodes | w_rad, w_ef rows):
//
//     pre1      = Sel  . NT                      P_i + Q_j + w_rad r2 + W_ef e        (gather  = MMA, A K-major)
//     gm       += Sel  . gM_unit                 broadcast of dL/dM_i onto the rows   (gather  = MMA)
//     M_i, ...  = Sel^T . m                      receiver / sender sums               (scatter = MMA, A MN-major)
//     gP|gQ|gw  = Sel^T . g1 ,  gx = Sel^T . rG
//
// One-hot products are exact, so the only rounding is the 2-piece bf16 split of the gathered / reduced operand
// (2^-17 relative), the same as every other operand of these kernels.  The unit-level accumulators live in TMEM
// across the tiles of a unit and are read out once per unit: no per-edge global gather, no shared-memory reduction
// loops, no atomics; bitwise deterministic.
//
// Units.  N <= 27: a unit is G whole graph-instances (G*N <= 27 nodes: 2 G N + 10 selector columns <= 64), walked in
// the canonical edge order, accumulators read out once per unit.  N > 27: a graph-instance is walked in blocks of
// (IB receivers) x (JB senders) = one tile of IB*JB <= 128 rows each (selector columns: IB receivers | JB senders |
// scalars, IB + JB <= 54; the host picks the pair that minimises the number of tiles, e.g. 5 x 25 for N = 100); the
// read-out of a tile adds onto global memory (M_i / gP_i over the sender blocks, gQ_j over the receiver blocks); all
// blocks of a graph-instance belong to one CTA, in a fixed order, so there are still no atomics and no races.
#pragma once
#ifndef NB_EMU
#include "nb_edge.cuh"
#include "nb_tc.cuh"

#define NB_SEL_MAX_GN 27
#define NB_SEL_XC0 54  // first scalar column of the selector / first weight row of the node tile

// stage a [64][64] fp32 weight matrix (row-major, row = output unit) as a split-bf16 operand tile
__device__ __forceinline__ void nb_tc_stage_weight(unsigned char* hi, unsigned char* lo, const float* __restrict__ W,
                                                   int tid) {
  for (int idx = tid; idx < 64 * 8; idx += NB_THREADS) {
    int o = idx >> 3, j = idx & 7;
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __ldg(W + o * NB_H + 8 * j + i);
    nb_tc_store8(hi, lo, o, j, v);
  }
}

// fp32 [128][64] scratch with 16-byte chunks XOR-swizzled by (row & 7): conflict-free for row-owner writes and
// for column-owner reads
__device__ __forceinline__ float* nb_scratch_chunk(float* S, int r, int j4) { return S + r * NB_H + ((j4 ^ (r & 7)) << 2); }
__device__ __forceinline__ float nb_scratch_get(const float* S, int r, int c) {
  return S[r * NB_H + ((((c >> 2) ^ (r & 7))) << 2) + (c & 3)];
}

// one unit of work of a selector kernel (see "Units" above)
struct NbSelUnit {
  int R;               // edge rows (blocked mode: 128, validity per row)
  int gt0;             // first graph-instance
  int recv0, nrecv;    // global node index of receiver slot 0, slots in use
  int send0, nsend;    // same for the senders
  int RC;              // selector column / node-tile row of sender slot 0
  int I0, J0;          // blocked mode: first receiver / sender index inside the graph
  bool first_j, last_j;  // blocked mode: first / last sender block of this receiver block
  bool first_i, last_i;  //               first / last receiver block of this graph-instance
};
template <bool BLK>
__device__ __forceinline__ NbSelUnit nb_sel_unit(const NbEdgeGeom& g, int uo, int sub) {
  NbSelUnit U;
  if (!BLK) {
    U.gt0 = uo * g.G;
    const int ngt = min(g.G, g.NGT - U.gt0);
    U.R = ngt * g.EPG;
    U.recv0 = U.send0 = U.gt0 * g.N;
    U.nrecv = U.nsend = ngt * g.N;
    U.RC = g.G * g.N;
    U.I0 = U.J0 = 0;
    U.first_j = U.last_j = U.first_i = U.last_i = true;
  } else {
    const int ib = sub / g.nJ, jb = sub - ib * g.nJ;
    U.gt0 = uo;
    U.R = NB_TILE;
    U.I0 = ib * g.IB;
    U.J0 = jb * g.JB;
    U.recv0 = uo * g.N + U.I0;
    U.nrecv = min(g.IB, g.N - U.I0);
    U.send0 = uo * g.N + U.J0;
    U.nsend = min(g.JB, g.N - U.J0);
    U.RC = g.IB;
    U.first_j = jb == 0;
    U.last_j = jb == g.nJ - 1;
    U.first_i = ib == 0;
    U.last_i = ib == g.nI - 1;
  }
  return U;
}
// row r of the unit -> receiver / sender slots, graph-instance, edge index inside the graph; false for padding rows
template <bool BLK>
__device__ __forceinline__ bool nb_sel_row(const NbEdgeGeom& g, const NbSelUnit& U, const uint32_t* rowinfo, int r, int& li,
                                           int& lj, int& gt, int& rem) {
  if (!BLK) {
    if (r >= U.R) return false;
    const uint32_t ri = rowinfo[r];
    li = ri & 0xff;
    lj = (ri >> 8) & 0xff;
    const int lg = ri >> 16;
    gt = U.gt0 + lg;
    rem = r - lg * g.EPG;
    return true;
  }
  li = r / g.JB;
  lj = r - li * g.JB;
  const int i = U.I0 + li, j = U.J0 + lj;
  gt = U.gt0;
  rem = i * (g.N - 1) + (j < i ? j : j - 1);
  return li < U.nrecv && lj < U.nsend && i != j;
}

// ----------------------------------------------------------------------------- cheap descriptor arithmetic
// 64-bit shared-memory descriptors as (lo, hi) halves: hi is a per-layout constant, lo = address field + LBO field;
// advancing a k-step is one 32-bit add on lo.
#define NB_DESC_HI_SW128 (((1024u >> 4) & 0x3FFFu) | (1u << 14) | (2u << 29))
#define NB_DESC_HI_NOSW (((128u >> 4) & 0x3FFFu) | (1u << 14))
__device__ __forceinline__ uint32_t nb_desc_lo_k(uint32_t addr) { return ((addr >> 4) & 0x3FFFu) | ((16u >> 4) << 16); }      // K-major SW128
__device__ __forceinline__ uint32_t nb_desc_lo_mn(uint32_t addr) { return ((addr >> 4) & 0x3FFFu) | ((8192u >> 4) << 16); }  // MN-major SW128
__device__ __forceinline__ uint32_t nb_desc_lo_n8(uint32_t addr) { return ((addr >> 4) & 0x3FFFu) | ((128u >> 4) << 16); }   // dense [rows][8]
#define NB_KSTEP_K 2u     // 32 bytes  >> 4
#define NB_KSTEP_MN 128u  // 2048 bytes >> 4
#define NB_KSTEP_N8 16u   // 256 bytes >> 4

__device__ __forceinline__ void nb_mma2(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                        uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
      "}" ::"r"(tmem_d),
      "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}

// the three split passes of a 64-deep product, A K-major [128][64], B = weight tile (K-major: W^T product, MN-major: W product)
__device__ __forceinline__ void nb_issue_w3(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, uint32_t w_hi, uint32_t w_lo,
                                            bool w_mn, uint32_t idesc, uint32_t acc0) {
  const uint32_t bstep = w_mn ? NB_KSTEP_MN : NB_KSTEP_K;
  uint32_t acc = acc0;
#pragma unroll
  for (int pass = 0; pass < 3; ++pass) {
    const uint32_t a = nb_desc_lo_k(pass == 1 ? a_lo : a_hi);
    const uint32_t b = w_mn ? nb_desc_lo_mn(pass == 2 ? w_lo : w_hi) : nb_desc_lo_k(pass == 2 ? w_lo : w_hi);
#pragma unroll
    for (int s = 0; s < 4; ++s) {
      nb_mma2(tmem_d, a + NB_KSTEP_K * s, NB_DESC_HI_SW128, b + bstep * s, NB_DESC_HI_SW128, idesc, acc);
      acc = 1u;
    }
  }
}

// the same product with the activation operand in tensor memory (hi pieces at columns ta_hi .., lo pieces at ta_lo ..,
// 8 columns per k-step): only the 2 KB weight slice of a k-step is fetched from shared memory
__device__ __forceinline__ void nb_issue_w3_ta(uint32_t tmem_d, uint32_t ta_hi, uint32_t ta_lo, uint32_t w_hi, uint32_t w_lo,
                                               bool w_mn, uint32_t idesc, uint32_t acc0) {
  const uint32_t bstep = w_mn ? NB_KSTEP_MN : NB_KSTEP_K;
  uint32_t acc = acc0;
#pragma unroll
  for (int pass = 0; pass < 3; ++pass) {
    const uint32_t a = pass == 1 ? ta_lo : ta_hi;
    const uint32_t b = w_mn ? nb_desc_lo_mn(pass == 2 ? w_lo : w_hi) : nb_desc_lo_k(pass == 2 ? w_lo : w_hi);
#pragma unroll
    for (int s = 0; s < 4; ++s) {
      nb_mma_bf16_ta(tmem_d, a + 8u * s, b + bstep * s, NB_DESC_HI_SW128, idesc, acc);
      acc = 1u;
    }
  }
}
// 16 consecutive fp32 values of row r (column quarter cq) -> split bf16 pieces into the shared-memory tiles (chunks
// 2 cq, 2 cq + 1: the side MMAs' copy) and into this thread's TMEM lane (8 packed columns each: the A operand's copy)
__device__ __forceinline__ void nb_store16_ta(unsigned char* hi, unsigned char* lo, int r, int cq, const float* v,
                                              uint32_t ta_hi, uint32_t ta_lo) {
  uint32_t h0[4], l0[4], h1[4], l1[4];
  nb_split8(v, h0, l0);
  nb_split8(v + 8, h1, l1);
  const uint32_t o0 = nb_tc_chunk_off(r, 2 * cq), o1 = nb_tc_chunk_off(r, 2 * cq + 1);
  *reinterpret_cast<uint4*>(hi + o0) = make_uint4(h0[0], h0[1], h0[2], h0[3]);
  *reinterpret_cast<uint4*>(hi + o1) = make_uint4(h1[0], h1[1], h1[2], h1[3]);
  *reinterpret_cast<uint4*>(lo + o0) = make_uint4(l0[0], l0[1], l0[2], l0[3]);
  *reinterpret_cast<uint4*>(lo + o1) = make_uint4(l1[0], l1[1], l1[2], l1[3]);
  nb_tmem_st44(ta_hi, h0, h1);
  nb_tmem_st44(ta_lo, l0, l1);
}

// 32 consecutive fp32 values of row r (column half hf) -> this thread's TMEM lane (2 x 8 packed columns per piece) and,
// when `hi` is given, the shared-memory tiles (chunks 4 hf .. 4 hf + 3)
__device__ __forceinline__ void nb_store32_ta(unsigned char* hi, unsigned char* lo, int r, int hf, const float* v, uint32_t ta_hi,
                                              uint32_t ta_lo) {
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    uint32_t h0[4], l0[4], h1[4], l1[4];
    nb_split8(v + 16 * k, h0, l0);
    nb_split8(v + 16 * k + 8, h1, l1);
    if (hi) {
      const uint32_t o0 = nb_tc_chunk_off(r, 4 * hf + 2 * k), o1 = nb_tc_chunk_off(r, 4 * hf + 2 * k + 1);
      *reinterpret_cast<uint4*>(hi + o0) = make_uint4(h0[0], h0[1], h0[2], h0[3]);
      *reinterpret_cast<uint4*>(hi + o1) = make_uint4(h1[0], h1[1], h1[2], h1[3]);
      *reinterpret_cast<uint4*>(lo + o0) = make_uint4(l0[0], l0[1], l0[2], l0[3]);
      *reinterpret_cast<uint4*>(lo + o1) = make_uint4(l1[0], l1[1], l1[2], l1[3]);
    }
    nb_tmem_st44(ta_hi + 8u * k, h0, h1);
    nb_tmem_st44(ta_lo + 8u * k, l0, l1);
  }
}

// gather: D[128 x 64] (+)= Sel[128 x 16 ksteps] . (Nh + Nl),  Sel K-major, node tile MN-major (K = node-tile rows)
__device__ __forceinline__ void nb_issue_gather(uint32_t tmem_d, uint32_t sel, uint32_t n_hi, uint32_t n_lo, int ksteps,
                                                uint32_t idesc, uint32_t acc0) {
  uint32_t acc = acc0;
  const uint32_t a = nb_desc_lo_k(sel);
#pragma unroll
  for (int pass = 0; pass < 2; ++pass) {
    const uint32_t b = nb_desc_lo_mn(pass ? n_lo : n_hi);
#pragma unroll
    for (int s = 0; s < 4; ++s)
      if (s < ksteps) {
        nb_mma2(tmem_d, a + NB_KSTEP_K * s, NB_DESC_HI_SW128, b + NB_KSTEP_MN * s, NB_DESC_HI_SW128, idesc, acc);
        acc = 1u;
      }
  }
}

// scatter: D[64 x 64] (+)= Sel^T . (Vh + Vl),  Sel MN-major (M = selector columns, K = 128 rows), V MN-major [128][64]
__device__ __forceinline__ void nb_issue_scatter(uint32_t tmem_d, uint32_t sel, uint32_t v_hi, uint32_t v_lo,
                                                 uint32_t idesc, uint32_t acc0) {
  uint32_t acc = acc0;
  const uint32_t a = nb_desc_lo_mn(sel);
#pragma unroll
  for (int pass = 0; pass < 2; ++pass) {
    const uint32_t b = nb_desc_lo_mn(pass ? v_lo : v_hi);
#pragma unroll
    for (int s = 0; s < 8; ++s) {
      nb_mma2(tmem_d, a + NB_KSTEP_MN * s, NB_DESC_HI_SW128, b + NB_KSTEP_MN * s, NB_DESC_HI_SW128, idesc, acc);
      acc = 1u;
    }
  }
}
// scatter of a dense [128][8] tile: D[64 x 8] (+)= Sel^T . (Vh + Vl)
__device__ __forceinline__ void nb_issue_scatter8(uint32_t tmem_d, uint32_t sel, uint32_t v_hi, uint32_t v_lo,
                                                  uint32_t idesc, uint32_t acc0) {
  uint32_t acc = acc0;
  const uint32_t a = nb_desc_lo_mn(sel);
#pragma unroll
  for (int pass = 0; pass < 2; ++pass) {
    const uint32_t b = nb_desc_lo_n8(pass ? v_lo : v_hi);
#pragma unroll
    for (int s = 0; s < 8; ++s) {
      nb_mma2(tmem_d, a + NB_KSTEP_MN * s, NB_DESC_HI_SW128, b + NB_KSTEP_N8 * s, NB_DESC_HI_NOSW, idesc, acc);
      acc = 1u;
    }
  }
}

// 16 / 8 / 4 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void nb_tmem_ld4(uint32_t taddr, float (&v)[4]) {
  uint32_t r[4];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(taddr)
               : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 4; ++i) v[i] = __uint_as_float(r[i]);
}

// ----------------------------------------------------------------------------- row bookkeeping
// rowinfo[r] for unit-local row r:  li | lj << 8 | lg << 16   (built once per CTA; every unit has the same structure)
__device__ __forceinline__ void nb_sel_build_rowinfo(uint32_t* rowinfo, const NbEdgeGeom& g, int tid, int nthreads) {
  const int R = g.blk ? 0 : g.G * g.EPG;
  for (int r = tid; r < R; r += nthreads) {
    int lg = r / g.EPG, rem = r - lg * g.EPG;
    int i = rem / (g.N - 1), jj = rem - i * (g.N - 1);
    int j = jj + (jj >= i ? 1 : 0);
    rowinfo[r] = (uint32_t)(lg * g.N + i) | ((uint32_t)(lg * g.N + j) << 8) | ((uint32_t)lg << 16);
  }
}

__device__ __forceinline__ uint32_t nb_pack_split(float v) {  // (hi, lo) bf16 pieces of v in one 32-bit word
  __nv_bfloat16 h = __float2bfloat16_rn(v);
  __nv_bfloat16 l = __float2bfloat16_rn(v - __bfloat162float(h));
  return (uint32_t)__bfloat16_as_ushort(h) | ((uint32_t)__bfloat16_as_ushort(l) << 16);
}

// this thread's half (hf) of selector row `row`: 4 chunks of 16 bytes, then the two one-hot entries
__device__ __forceinline__ void nb_sel_write_row(unsigned char* Sel, int row, int hf, bool valid, int li, int cj,
                                                 float r2, const float (&e)[NB_MAX_EF]) {
  const uint4 z = make_uint4(0u, 0u, 0u, 0u);
  unsigned char* rp = Sel + row * NB_TC_ROW_BYTES;
  const int sw = row & 7;
  if (hf == 0) {
#pragma unroll
    for (int c = 0; c < 4; ++c) *reinterpret_cast<uint4*>(rp + ((c ^ sw) << 4)) = z;
  } else {
    *reinterpret_cast<uint4*>(rp + ((4 ^ sw) << 4)) = z;
    *reinterpret_cast<uint4*>(rp + ((5 ^ sw) << 4)) = z;
    uint4 c6 = z, c7 = z;
    if (valid) {
      c6.w = nb_pack_split(r2);  // columns 54, 55
      c7.x = nb_pack_split(e[0]);
      c7.y = nb_pack_split(e[1]);
      c7.z = nb_pack_split(e[2]);
      c7.w = nb_pack_split(e[3]);
    }
    *reinterpret_cast<uint4*>(rp + ((6 ^ sw) << 4)) = c6;
    *reinterpret_cast<uint4*>(rp + ((7 ^ sw) << 4)) = c7;
  }
  if (valid) {  // same thread, after its own zero fill: program order
    if ((li >> 5) == hf) *reinterpret_cast<unsigned short*>(rp + (((li >> 3) ^ sw) << 4) + (li & 7) * 2) = 0x3F80;
    if ((cj >> 5) == hf) *reinterpret_cast<unsigned short*>(rp + (((cj >> 3) ^ sw) << 4) + (cj & 7) * 2) = 0x3F80;
  }
}

// general unit: rows [0, nrecv) <- P of the receiver list, rows [RC, RC + nsend) <- Q of the sender list
__device__ __forceinline__ void nb_sel_stage_unit(unsigned char* Nh, unsigned char* Nl, const float* __restrict__ P,
                                                  const float* __restrict__ Q, const NbSelUnit& U, int tid, int nthreads,
                                                  bool with_recv = true) {
  const int total = (U.nrecv + U.nsend) * 8;
  for (int idx = tid + (with_recv ? 0 : U.nrecv * 8); idx < total; idx += nthreads) {
    const int n = idx >> 3, j = idx & 7;
    const bool snd = n >= U.nrecv;
    const float* src = snd ? Q + (int64_t)(U.send0 + n - U.nrecv) * NB_H + 8 * j : P + (int64_t)(U.recv0 + n) * NB_H + 8 * j;
    float4 a = nb_ld4(src), b = nb_ld4(src + 4);
    float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    nb_tc_store8(Nh, Nl, snd ? U.RC + n - U.nrecv : n, j, v);
  }
}

// TMEM lane of accumulator row i for M = 64 MMAs; thread (warp quarter q, lane < 16) owns row 16 q + lane
// ----------------------------------------------------------------------------- forward
// shared memory (bytes after 1024-alignment)
#define NB_SF_W 0                                   // W2 hi/lo, W3 hi/lo       4 x 8 KB
#define NB_SF_T (4 * NB_TC_TILE_BYTES(64))          // activation tile hi/lo    2 x 16 KB
#define NB_SF_SEL (NB_SF_T + 2 * NB_TC_TILE_BYTES(128))   // selector          16 KB
#define NB_SF_NT (NB_SF_SEL + NB_TC_TILE_BYTES(128))      // node tile hi/lo   2 x 8 KB
#define NB_SF_F (NB_SF_NT + 2 * NB_TC_TILE_BYTES(64))     // force tile hi/lo  2 x 2 KB  ([128][8] bf16)
#define NB_SF_FL (NB_SF_F + 2 * NB_TILE * 16)
#define NB_SF_NFLOAT (3 * NB_H + 2 * NB_TILE + 2 * 32 * 3)
#define NB_EDGE_FWD_SEL_SMEM(RU) (NB_SF_FL + NB_SF_NFLOAT * 4 + (RU) * 4 + 64 + 1024)
#define NB_SF_TMEM_COLS 256  // [0,64) pre-activations | [64,128) M accumulators | [128,136) Fsum accumulators |
                             // [192,224) hi, [224,256) lo pieces of the A operand (z1, then m) as packed bf16 pairs

// SiLU of the forward tile: elements whose index i satisfies (i % NB_FWD_FMA_DEN) < NB_FWD_FMA_NUM take their reciprocal
// on the FMA pipe (nb_sigmoid_fma), the rest on the MUFU.  Measured on B200 (tools/ab_variants.py, cfg3, same box,
// alternating): 0/1 -> 188.9 us per launch, 1/2 -> 188.6, 2/3 -> 193.4, 1/1 -> 201.3: halving the MUFU load buys
// nothing (XU was 53 % of peak, the tile is bound by its dependent chain at two CTAs per SM, and the seven extra FMA-pipe
// instructions per element cost issue slots), so the default stays 0 / 1; the variant remains as a build-time switch.
#ifndef NB_FWD_FMA_NUM
#define NB_FWD_FMA_NUM 0
#define NB_FWD_FMA_DEN 1
#endif
#define NB_FWD_SILU(i, x) ((((i) % NB_FWD_FMA_DEN) < NB_FWD_FMA_NUM) ? nb_silu_fma(x) : nb_silu(x))

template <bool BLK>
__global__ void __launch_bounds__(NB_THREADS, 2) k_edge_fwd_sel(NbEdgeFwdArgs a) {
  NB_PDL_ENTER();
  extern __shared__ __align__(1024) unsigned char nb_smraw[];
  unsigned char* base = nb_smraw + ((1024u - (nb_smem_u32(nb_smraw) & 1023u)) & 1023u);
  unsigned char* W2h = base + NB_SF_W;
  unsigned char* W2l = W2h + NB_TC_TILE_BYTES(64);
  unsigned char* W3h = W2l + NB_TC_TILE_BYTES(64);
  unsigned char* W3l = W3h + NB_TC_TILE_BYTES(64);
  unsigned char* Th = base + NB_SF_T;
  unsigned char* Tl = Th + NB_TC_TILE_BYTES(128);
  unsigned char* Sel = base + NB_SF_SEL;
  unsigned char* Nh = base + NB_SF_NT;
  unsigned char* Nl = Nh + NB_TC_TILE_BYTES(64);
  unsigned char* Fh = base + NB_SF_F;
  unsigned char* Fl = Fh + NB_TILE * 16;
  float* fl = reinterpret_cast<float*>(base + NB_SF_FL);
  float* vb2 = fl;
  float* vb3 = vb2 + NB_H;
  float* vw4 = vb3 + NB_H;
  float* cpart = vw4 + NB_H;         // [2][128]
  float* xs = cpart + 2 * NB_TILE;   // [32][3] positions of the unit's receivers
  float* xq = xs + 32 * 3;           // [32][3] positions of the unit's senders
  uint32_t* rowinfo = reinterpret_cast<uint32_t*>(xq + 32 * 3);
  const NbEdgeGeom g = a.g;
  const int RU = BLK ? 0 : g.G * g.EPG;
  uint64_t* bar = reinterpret_cast<uint64_t*>(rowinfo + RU + (RU & 1));
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, hf = warp >> 2;
  const int row = 32 * q + lane;
  const int cb = 32 * hf;

  nb_tc_stage_weight(W2h, W2l, a.w.W2, tid);
  nb_tc_stage_weight(W3h, W3l, a.w.W3, tid);
  for (int idx = tid; idx < 2 * NB_TC_TILE_BYTES(64) / 16; idx += NB_THREADS)
    reinterpret_cast<uint4*>(Nh)[idx] = make_uint4(0u, 0u, 0u, 0u);
  nb_sel_build_rowinfo(rowinfo, g, tid, NB_THREADS);
  if (tid < NB_H) {
    vb2[tid] = __ldg(a.w.b2 + tid);
    vb3[tid] = __ldg(a.w.b3 + tid);
    vw4[tid] = __ldg(a.w.w4 + tid);
  }
  if (tid == 0) {
    nb_mbar_init(bar, 1);
    nb_mbar_fence_init();
  }
  if (warp == 0) nb_tmem_alloc(tmem_slot, NB_SF_TMEM_COLS);
  __syncthreads();
  // weight rows of the node tile: 54,55 <- w_rad ; 56 + 2f, 57 + 2f <- w_ef[f]
  for (int idx = tid; idx < 10 * 8; idx += NB_THREADS) {
    int k = idx >> 3, j = idx & 7;
    int f = (k >> 1) - 1;  // -1: radial
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int c = 8 * j + i;
      v[i] = f < 0 ? __ldg(a.w.W1 + (int64_t)c * a.w.ldw1 + a.w.col_rad)
                   : (f < g.nef ? __ldg(a.w.W1 + (int64_t)c * a.w.ldw1 + a.w.col_ef + f) : 0.f);
    }
    nb_tc_store8(Nh, Nl, NB_SEL_XC0 + k, j, v);
  }
  nb_fence_async_smem();
  nb_tc_fence_before();
  __syncthreads();
  nb_tc_fence_after();
  const uint32_t tm = *tmem_slot;
  const uint32_t tm_mine = tm + ((uint32_t)(32 * q) << 16) + (uint32_t)cb;
  // the two 64-deep products read their activation operand from tensor memory (see the backward kernel's note)
  const uint32_t ta_h = tm + 192, ta_l = tm + 224;
  const uint32_t ta_hm = ta_h + ((uint32_t)(32 * q) << 16) + 16u * (uint32_t)hf, ta_lm = ta_l + ((uint32_t)(32 * q) << 16) + 16u * (uint32_t)hf;
  const uint32_t idesc_fwd = nb_idesc_bf16(128, 64, 0, 0);  // A K-major, B K-major (W^T)
  const uint32_t idesc_gat = nb_idesc_bf16(128, 64, 0, 1);  // A K-major, B MN-major
  const uint32_t idesc_sc = nb_idesc_bf16(64, 64, 1, 1);    // Sel^T . tile
  const uint32_t idesc_sc8 = nb_idesc_bf16(64, 8, 1, 1);
  const uint32_t sTh = nb_smem_u32(Th), sTl = nb_smem_u32(Tl), sSel = nb_smem_u32(Sel), sNh = nb_smem_u32(Nh),
                 sNl = nb_smem_u32(Nl), sFh = nb_smem_u32(Fh), sFl = nb_smem_u32(Fl), sW2h = nb_smem_u32(W2h),
                 sW2l = nb_smem_u32(W2l), sW3h = nb_smem_u32(W3h), sW3l = nb_smem_u32(W3l);
  const float b4 = __ldg(a.w.b4);
  uint32_t phase = 0;

  const int n_outer = BLK ? g.NGT : g.n_units, n_sub = BLK ? g.nI * g.nJ : 1;
  for (int uo = blockIdx.x; uo < n_outer; uo += gridDim.x)
  for (int sub = 0; sub < n_sub; ++sub) {
    const NbSelUnit U = nb_sel_unit<BLK>(g, uo, sub);
    const int R = U.R;
    // every MMA of the previous unit has completed (its read-out waited for the last commit)
    {  // positions of the receiver and (blocked mode: distinct) sender lists: at most one per thread, loaded before the
       // node-tile staging below so that the unit pays one memory round trip
      const int n3r = U.nrecv * 3, n3 = n3r + (BLK ? U.nsend * 3 : 0);
      const int t_x = tid + (U.first_j ? 0 : n3r);
      float xv = 0.f;
      if (t_x < n3) xv = t_x < n3r ? __ldg(a.x + (int64_t)U.recv0 * 3 + t_x) : __ldg(a.x + (int64_t)U.send0 * 3 + (t_x - n3r));
      nb_sel_stage_unit(Nh, Nl, a.P, a.Q, U, tid, NB_THREADS, U.first_j);
      if (t_x < n3) {
        if (t_x < n3r) xs[t_x] = xv;
        else xq[t_x - n3r] = xv;
      }
    }
    const float* xsnd = BLK ? xq : xs;  // whole-graph units: senders = receivers
    __syncthreads();

    for (int r0 = 0; r0 < R; r0 += NB_TILE) {
      // ---- geometry + selector row
      float dx = 0.f, dy = 0.f, dz = 0.f, r2 = 0.f;
      float e[NB_MAX_EF];
#pragma unroll
      for (int f = 0; f < NB_MAX_EF; ++f) e[f] = 0.f;
      int li = 0, lj = 0, gt = 0, rem = 0;
      const bool valid = nb_sel_row<BLK>(g, U, rowinfo, r0 + row, li, lj, gt, rem);
      if (valid) {
        dx = xs[li * 3 + 0] - xsnd[lj * 3 + 0];
        dy = xs[li * 3 + 1] - xsnd[lj * 3 + 1];
        dz = xs[li * 3 + 2] - xsnd[lj * 3 + 2];
        r2 = dx * dx + dy * dy + dz * dz;
        const int64_t eoff = ((int64_t)nb_ef_graph(g, gt) * g.EPG + rem) * g.nef;
#pragma unroll
        for (int f = 0; f < NB_MAX_EF; ++f)
          if (f < g.nef) e[f] = __ldg(a.ef + eoff + f);
      }
      // the scatter MMAs of the previous tile read Sel / T / F: they were issued before, and therefore complete
      // before, the MMA whose commit this CTA waited for last  -> Sel may be rewritten only after that wait; the
      // last wait of a tile (stage 3) precedes the scatter issue, so wait for the scatters here.
      if (r0 > 0) {
        nb_mbar_wait(bar, phase);
        phase ^= 1;
        nb_tc_fence_after();
      }
      nb_sel_write_row(Sel, row, hf, valid, li, U.RC + lj, r2, e);
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
      // ---- z1 = SiLU(pre1) -> tile
      {
        float v[32];
        nb_tmem_ld32(tm_mine, v);
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = NB_FWD_SILU(i, v[i]);
        nb_store32_ta(nullptr, nullptr, row, hf, v, ta_hm, ta_lm);  // z1 is only ever an A operand: no shared-memory copy
        nb_tmem_st_wait();
      }
      nb_tc_fence_before();
      __syncthreads();
      if (NB_ISSUER(0)) {
        nb_tc_fence_after();
        nb_issue_w3_ta(tm, ta_h, ta_l, sW2h, sW2l, false, idesc_fwd, 0u);
        nb_mma_commit(bar);
      }
      nb_mbar_wait(bar, phase);
      phase ^= 1;
      nb_tc_fence_after();
      // ---- m = SiLU(pre2 + b2) -> tile
      {
        float v[32];
        nb_tmem_ld32(tm_mine, v);
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = NB_FWD_SILU(i, v[i] + vb2[cb + i]);
        nb_store32_ta(Th, Tl, row, hf, v, ta_hm, ta_lm);  // shared-memory copy: B operand of the scatter M_i += Sel^T m
        nb_tmem_st_wait();
      }
      nb_fence_async_smem();
      nb_tc_fence_before();
      __syncthreads();
      if (NB_ISSUER(0)) {
        nb_tc_fence_after();
        nb_issue_w3_ta(tm, ta_h, ta_l, sW3h, sW3l, false, idesc_fwd, 0u);
        nb_mma_commit(bar);
        // M_i += Sel^T m  (runs underneath the phi_x epilogue)
        nb_issue_scatter(tm + 64, sSel, sTh, sTl, idesc_sc, (r0 > 0 || !U.first_j) ? 1u : 0u);
      }
      nb_mbar_wait(bar, phase);
      phase ^= 1;
      nb_tc_fence_after();
      // ---- c = w4 . SiLU(pre3 + b3) + b4 ; F = rij c -> force tile
      {
        float v[32];
        nb_tmem_ld32(tm_mine, v);
        float cp = 0.f;
#pragma unroll
        for (int i = 0; i < 32; ++i) cp = fmaf(vw4[cb + i], NB_FWD_SILU(i, v[i] + vb3[cb + i]), cp);
        cpart[hf * NB_TILE + row] = cp;
      }
      nb_tc_fence_before();
      __syncthreads();
      if (hf == 0) {
        float c = cpart[row] + cpart[NB_TILE + row] + b4;
        float fx = dx * c, fy = dy * c, fz = dz * c;  // 0 for padded rows
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
        nb_issue_scatter8(tm + 128, sSel, sFh, sFl, idesc_sc8, (r0 > 0 || !U.first_j) ? 1u : 0u);
        nb_mma_commit(bar);  // waited for at the top of the next tile / at the unit read-out
      }
    }
    // ---- unit read-out: M_i and Fsum_i of the unit's nodes (accumulator row i <-> TMEM lane (i % 16) + 32 (i / 16))
    nb_mbar_wait(bar, phase);
    phase ^= 1;
    nb_tc_fence_after();
    if (U.last_j) {  // blocked mode: the receivers' accumulators collect all sender blocks in TMEM first
      const int nl = 16 * q + lane;
      float v[32];
      nb_tmem_ld32(tm + ((uint32_t)(32 * q) << 16) + 64 + (uint32_t)cb, v);
      if (lane < 16 && nl < U.nrecv) {
        float* dst = a.M + (int64_t)(U.recv0 + nl) * NB_H + cb;
#pragma unroll
        for (int k = 0; k < 8; ++k) nb_st4(dst + 4 * k, make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]));
      }
      float f4[4];
      nb_tmem_ld4(tm + ((uint32_t)(32 * q) << 16) + 128, f4);
      if (hf == 0 && lane < 16 && nl < U.nrecv) {
        float* dst = a.Fsum + (int64_t)(U.recv0 + nl) * 3;
        dst[0] = f4[0];
        dst[1] = f4[1];
        dst[2] = f4[2];
      }
    }
    nb_tc_fence_before();
    __syncthreads();
  }
  nb_tc_fence_before();
  __syncthreads();
  if (warp == 0) nb_tmem_dealloc(tm, NB_SF_TMEM_COLS);
}

// ----------------------------------------------------------------------------- forward, three tiles in flight
// Whole-graph units of at least three tiles (G = 1, N = 17 .. 27), one CTA per SM.  The tile of k_edge_fwd_sel is a
// dependent chain of four MMA round trips; at two CTAs per SM an SM has two such chains and no pipe is saturated.  Here
// the CTA runs three chains: warp group g (warps 4g .. 4g + 3, one thread per tile row, all 64 columns) walks tiles
// g, g + 3, ... of each unit with its own selector / activation / force tiles and TMEM columns, and warp 12 issues every
// MMA from one thread.  The issuer serves the groups stage by stage in tile order (gathers of a round of three tiles,
// then their W2 products, then W3 + M scatter, then the F scatters), so the M / Fsum scatters of a unit are issued, and
// run, in tile order with tile 0 clearing the accumulators: the per-row arithmetic and the accumulation order are
// those of k_edge_fwd_sel<false>, and M / Fsum are bitwise equal to it.
//   groups -> issuer: ready[g] (one arrival after the group's named barrier);  issuer -> group: done[g] (tcgen05.commit)
// Unit boundaries overlap the next unit's tiles: the node tile and positions are double-buffered (each thread stages its
// share of the next unit's rows while its first tile of the current unit waits for W2; ntfull[b] counts 384 arrivals),
// and the group holding a unit's last tile reads the accumulators out while the other groups start the next unit; the
// issuer holds the next unit's first M scatter until that read-out has arrived on accfree.
//
// TMEM columns: group g: [128 g, 128 g + 64) pre-activations | [128 g + 64, +32) hi, [128 g + 96, +32) lo pieces of the
//               A operand;  [384, 448) M accumulators | [448, 456) Fsum accumulators
#define NB_F3_GROUPS 3
#define NB_F3_THREADS (128 * NB_F3_GROUPS + 32)
#define NB_F3_ISSUER_WARP (4 * NB_F3_GROUPS)
#define NB_F3_W 0                                    // W2 hi/lo, W3 hi/lo                4 x 8 KB
#define NB_F3_NT (4 * NB_TC_TILE_BYTES(64))          // node tile hi/lo, two buffers      4 x 8 KB
#define NB_F3_GRP (NB_F3_NT + 4 * NB_TC_TILE_BYTES(64))
#define NB_F3_GRP_BYTES (3 * NB_TC_TILE_BYTES(128) + 2 * NB_TILE * 16)  // per group: Sel | T hi | T lo | F hi | F lo
#define NB_F3_FL (NB_F3_GRP + NB_F3_GROUPS * NB_F3_GRP_BYTES)
#define NB_F3_NFLOAT (3 * NB_H + 2 * 32 * 3)
#define NB_EDGE_FWD_SEL3_SMEM(RU) (NB_F3_FL + NB_F3_NFLOAT * 4 + (RU) * 4 + 16 * 8 + 1024)
#define NB_F3_TMEM_COLS 512
#define NB_F3_TM_M 384
#define NB_F3_TM_F 448

__device__ __forceinline__ void nb_named_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void nb_mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(nb_smem_u32(bar)) : "memory");
}

__global__ void __launch_bounds__(NB_F3_THREADS, 1) k_edge_fwd_sel3(NbEdgeFwdArgs a) {
  NB_PDL_ENTER();
  extern __shared__ __align__(1024) unsigned char nb_smraw[];
  unsigned char* base = nb_smraw + ((1024u - (nb_smem_u32(nb_smraw) & 1023u)) & 1023u);
  unsigned char* W2h = base + NB_F3_W;
  unsigned char* W2l = W2h + NB_TC_TILE_BYTES(64);
  unsigned char* W3h = W2l + NB_TC_TILE_BYTES(64);
  unsigned char* W3l = W3h + NB_TC_TILE_BYTES(64);
  unsigned char* NT = base + NB_F3_NT;  // buffer b: hi at NT + 2 b x 8 KB, lo 8 KB above
  float* fl = reinterpret_cast<float*>(base + NB_F3_FL);
  float* vb2 = fl;
  float* vb3 = vb2 + NB_H;
  float* vw4 = vb3 + NB_H;
  float* xsb = vw4 + NB_H;  // [2][32][3] positions of the unit's nodes, one buffer per node-tile buffer
  uint32_t* rowinfo = reinterpret_cast<uint32_t*>(xsb + 2 * 32 * 3);
  const NbEdgeGeom g = a.g;
  const int RU = g.G * g.EPG;
  uint64_t* bars = reinterpret_cast<uint64_t*>(rowinfo + RU + (RU & 1));
  uint64_t* ready = bars;       // [3]
  uint64_t* done = bars + 3;    // [3]
  uint64_t* ntfull = bars + 6;  // [2]
  uint64_t* accfree = bars + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);
  constexpr int NC = 128 * NB_F3_GROUPS;  // compute threads

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int grp = warp >> 2, q = warp & 3;
  const int row = 32 * q + lane;

  if (tid < NB_THREADS) {
    nb_tc_stage_weight(W2h, W2l, a.w.W2, tid);
    nb_tc_stage_weight(W3h, W3l, a.w.W3, tid);
  }
  for (int idx = tid; idx < 4 * NB_TC_TILE_BYTES(64) / 16; idx += NB_F3_THREADS)
    reinterpret_cast<uint4*>(NT)[idx] = make_uint4(0u, 0u, 0u, 0u);
  nb_sel_build_rowinfo(rowinfo, g, tid, NB_F3_THREADS);
  if (tid < NB_H) {
    vb2[tid] = __ldg(a.w.b2 + tid);
    vb3[tid] = __ldg(a.w.b3 + tid);
    vw4[tid] = __ldg(a.w.w4 + tid);
  }
  if (tid == 0) {
    for (int i = 0; i < NB_F3_GROUPS; ++i) {
      nb_mbar_init(ready + i, 1);
      nb_mbar_init(done + i, 1);
    }
    nb_mbar_init(ntfull, NC);
    nb_mbar_init(ntfull + 1, NC);
    nb_mbar_init(accfree, 128);
    nb_mbar_fence_init();
  }
  if (warp == 0) nb_tmem_alloc(tmem_slot, NB_F3_TMEM_COLS);
  __syncthreads();
  // weight rows of both node-tile buffers: 54,55 <- w_rad ; 56 + 2f, 57 + 2f <- w_ef[f]
  for (int idx = tid; idx < 2 * 10 * 8; idx += NB_F3_THREADS) {
    const int b = idx / 80, k = (idx % 80) >> 3, j = idx & 7;
    const int f = (k >> 1) - 1;  // -1: radial
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int c = 8 * j + i;
      v[i] = f < 0 ? __ldg(a.w.W1 + (int64_t)c * a.w.ldw1 + a.w.col_rad)
                   : (f < g.nef ? __ldg(a.w.W1 + (int64_t)c * a.w.ldw1 + a.w.col_ef + f) : 0.f);
    }
    unsigned char* nh = NT + 2 * b * NB_TC_TILE_BYTES(64);
    nb_tc_store8(nh, nh + NB_TC_TILE_BYTES(64), NB_SEL_XC0 + k, j, v);
  }
  // the CTA's first unit -> buffer 0
  if (blockIdx.x < g.n_units) {
    const NbSelUnit U = nb_sel_unit<false>(g, blockIdx.x, 0);
    nb_sel_stage_unit(NT, NT + NB_TC_TILE_BYTES(64), a.P, a.Q, U, tid, NB_F3_THREADS);
    if (tid < U.nrecv * 3) xsb[tid] = __ldg(a.x + (int64_t)U.recv0 * 3 + tid);
  }
  nb_fence_async_smem();
  nb_tc_fence_before();
  __syncthreads();
  nb_tc_fence_after();
  const uint32_t tm = *tmem_slot;
  const uint32_t idesc_fwd = nb_idesc_bf16(128, 64, 0, 0);  // A K-major, B K-major (W^T)
  const uint32_t idesc_gat = nb_idesc_bf16(128, 64, 0, 1);  // A K-major, B MN-major
  const uint32_t idesc_sc = nb_idesc_bf16(64, 64, 1, 1);    // Sel^T . tile
  const uint32_t idesc_sc8 = nb_idesc_bf16(64, 8, 1, 1);

  if (warp == NB_F3_ISSUER_WARP) {
    // ---------------------------------------------------------------- MMA issuer
    if (nb_elect_one()) {
      const uint32_t sW2h = nb_smem_u32(W2h), sW2l = nb_smem_u32(W2l), sW3h = nb_smem_u32(W3h), sW3l = nb_smem_u32(W3l);
      const uint32_t sGrp = nb_smem_u32(base + NB_F3_GRP);
      uint32_t ph_ready = 0;  // bit g: phase of ready[g]
      int k = 0;
      for (int uo = blockIdx.x; uo < g.n_units; uo += gridDim.x, ++k) {
        const int ntl = (nb_sel_unit<false>(g, uo, 0).R + NB_TILE - 1) / NB_TILE;
        const uint32_t sNh = nb_smem_u32(NT + 2 * (k & 1) * NB_TC_TILE_BYTES(64)), sNl = sNh + NB_TC_TILE_BYTES(64);
        if (k > 0) nb_mbar_wait(ntfull + (k & 1), ((k - 1) >> 1) & 1);
        for (int t0 = 0; t0 < ntl; t0 += NB_F3_GROUPS) {
          const int ng = min(NB_F3_GROUPS, ntl - t0);
#pragma unroll 1
          for (int st = 0; st < 4; ++st)
#pragma unroll 1
            for (int gi = 0; gi < ng; ++gi) {
              const uint32_t sSel = sGrp + gi * NB_F3_GRP_BYTES, sTh = sSel + NB_TC_TILE_BYTES(128),
                             sTl = sTh + NB_TC_TILE_BYTES(128), sFh = sTl + NB_TC_TILE_BYTES(128), sFl = sFh + NB_TILE * 16;
              const uint32_t tg = tm + 128u * gi;
              const uint32_t acc = (t0 + gi > 0) ? 1u : 0u;
              nb_mbar_wait(ready + gi, (ph_ready >> gi) & 1u);
              ph_ready ^= 1u << gi;
              nb_tc_fence_after();
              if (st == 0) {
                nb_issue_gather(tg, sSel, sNh, sNl, 4, idesc_gat, 0u);
              } else if (st == 1) {
                nb_issue_w3_ta(tg, tg + 64, tg + 96, sW2h, sW2l, false, idesc_fwd, 0u);
              } else if (st == 2) {
                nb_issue_w3_ta(tg, tg + 64, tg + 96, sW3h, sW3l, false, idesc_fwd, 0u);
                nb_mma_commit(done + gi);
                if (t0 + gi == 0 && k > 0) {  // the previous unit's accumulators have been read out
                  nb_mbar_wait(accfree, (k - 1) & 1);
                  nb_tc_fence_after();
                }
                nb_issue_scatter(tm + NB_F3_TM_M, sSel, sTh, sTl, idesc_sc, acc);  // runs underneath the phi_x head
                continue;
              } else {
                nb_issue_scatter8(tm + NB_F3_TM_F, sSel, sFh, sFl, idesc_sc8, acc);
              }
              nb_mma_commit(done + gi);
            }
        }
      }
    }
    __syncwarp();
  } else {
    // ---------------------------------------------------------------- tile groups
    unsigned char* Sel = base + NB_F3_GRP + grp * NB_F3_GRP_BYTES;
    unsigned char* Th = Sel + NB_TC_TILE_BYTES(128);
    unsigned char* Tl = Th + NB_TC_TILE_BYTES(128);
    unsigned char* Fh = Tl + NB_TC_TILE_BYTES(128);
    unsigned char* Fl = Fh + NB_TILE * 16;
    const uint32_t lq = (uint32_t)(32 * q) << 16;
    const uint32_t tpre = tm + lq + 128u * grp;  // this thread's row of the group's pre-activations
    const uint32_t ta_h = tpre + 64, ta_l = tpre + 96;
    const float b4 = __ldg(a.w.b4);
    uint32_t phase = 0;
    bool pend = false;  // the group's last F scatter has not been waited for
    int k = 0;
    for (int uo = blockIdx.x; uo < g.n_units; uo += gridDim.x, ++k) {
      const NbSelUnit U = nb_sel_unit<false>(g, uo, 0);
      const int R = U.R, ntl = (R + NB_TILE - 1) / NB_TILE;
      const int b = k & 1;
      if (k > 0) nb_mbar_wait(ntfull + b, ((k - 1) >> 1) & 1);
      const float* xs = xsb + b * 96;
      for (int t = grp; t < ntl; t += NB_F3_GROUPS) {
        const int r0 = t * NB_TILE;
        // ---- geometry + selector row
        float dx = 0.f, dy = 0.f, dz = 0.f, r2 = 0.f;
        float e[NB_MAX_EF];
#pragma unroll
        for (int f = 0; f < NB_MAX_EF; ++f) e[f] = 0.f;
        int li = 0, lj = 0, gt = 0, rem = 0;
        const bool valid = nb_sel_row<false>(g, U, rowinfo, r0 + row, li, lj, gt, rem);
        if (valid) {
          dx = xs[li * 3 + 0] - xs[lj * 3 + 0];
          dy = xs[li * 3 + 1] - xs[lj * 3 + 1];
          dz = xs[li * 3 + 2] - xs[lj * 3 + 2];
          r2 = dx * dx + dy * dy + dz * dz;
          const int64_t eoff = ((int64_t)nb_ef_graph(g, gt) * g.EPG + rem) * g.nef;
#pragma unroll
          for (int f = 0; f < NB_MAX_EF; ++f)
            if (f < g.nef) e[f] = __ldg(a.ef + eoff + f);
        }
        if (pend) {  // the group's previous scatters read Sel / T / F
          nb_mbar_wait(done + grp, phase);
          phase ^= 1;
          nb_tc_fence_after();
        }
        nb_sel_write_row(Sel, row, 0, valid, li, U.RC + lj, r2, e);
        nb_sel_write_row(Sel, row, 1, valid, li, U.RC + lj, r2, e);
        nb_fence_async_smem();
        nb_tc_fence_before();
        nb_named_sync(1 + grp, 128);
        if (row == 0) nb_mbar_arrive(ready + grp);
        nb_mbar_wait(done + grp, phase);
        phase ^= 1;
        nb_tc_fence_after();
        // ---- z1 = SiLU(pre1) -> A operand
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          float v[32];
          nb_tmem_ld32(tpre + 32 * hf, v);
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = NB_FWD_SILU(i, v[i]);
          nb_store32_ta(nullptr, nullptr, row, hf, v, ta_h + 16 * hf, ta_l + 16 * hf);
        }
        nb_tmem_st_wait();
        nb_tc_fence_before();
        nb_named_sync(1 + grp, 128);
        if (row == 0) nb_mbar_arrive(ready + grp);
        if (t == grp && uo + (int)gridDim.x < g.n_units) {
          // this thread's share of the next unit's node tile and positions, underneath the W2 product; the other
          // buffer's last readers (the previous unit's gathers and geometry) finished before this group's gather did
          const NbSelUnit Un = nb_sel_unit<false>(g, uo + gridDim.x, 0);
          unsigned char* nh = NT + 2 * (b ^ 1) * NB_TC_TILE_BYTES(64);
          const float xv = tid < Un.nrecv * 3 ? __ldg(a.x + (int64_t)Un.recv0 * 3 + tid) : 0.f;
          nb_sel_stage_unit(nh, nh + NB_TC_TILE_BYTES(64), a.P, a.Q, Un, tid, NC);
          if (tid < Un.nrecv * 3) xsb[(b ^ 1) * 96 + tid] = xv;
          nb_fence_async_smem();
          nb_mbar_arrive(ntfull + (b ^ 1));
        }
        nb_mbar_wait(done + grp, phase);
        phase ^= 1;
        nb_tc_fence_after();
        // ---- m = SiLU(pre2 + b2) -> A operand and the scatter's B operand
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          float v[32];
          nb_tmem_ld32(tpre + 32 * hf, v);
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = NB_FWD_SILU(i, v[i] + vb2[32 * hf + i]);
          nb_store32_ta(Th, Tl, row, hf, v, ta_h + 16 * hf, ta_l + 16 * hf);
        }
        nb_tmem_st_wait();
        nb_fence_async_smem();
        nb_tc_fence_before();
        nb_named_sync(1 + grp, 128);
        if (row == 0) nb_mbar_arrive(ready + grp);
        nb_mbar_wait(done + grp, phase);
        phase ^= 1;
        nb_tc_fence_after();
        // ---- c = w4 . SiLU(pre3 + b3) + b4 (two 32-term chains, as k_edge_fwd_sel) ; F = rij c -> force tile
        float cp[2];
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          float v[32];
          nb_tmem_ld32(tpre + 32 * hf, v);
          cp[hf] = 0.f;
#pragma unroll
          for (int i = 0; i < 32; ++i) cp[hf] = fmaf(vw4[32 * hf + i], NB_FWD_SILU(i, v[i] + vb3[32 * hf + i]), cp[hf]);
        }
        {
          const float c = cp[0] + cp[1] + b4;
          float fx = dx * c, fy = dy * c, fz = dz * c;  // 0 for padded rows
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
        nb_tc_fence_before();
        nb_named_sync(1 + grp, 128);
        if (row == 0) nb_mbar_arrive(ready + grp);
        pend = true;
      }
      if (grp == (ntl - 1) % NB_F3_GROUPS) {
        // ---- unit read-out (accumulator row i <-> TMEM lane (i % 16) + 32 (i / 16)); the last F scatter completes
        // after every other scatter of the unit
        nb_mbar_wait(done + grp, phase);
        phase ^= 1;
        pend = false;
        nb_tc_fence_after();
        const int nl = 16 * q + lane;
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          float v[32];
          nb_tmem_ld32(tm + lq + NB_F3_TM_M + 32 * hf, v);
          if (lane < 16 && nl < U.nrecv) {
            float* dst = a.M + (int64_t)(U.recv0 + nl) * NB_H + 32 * hf;
#pragma unroll
            for (int j = 0; j < 8; ++j) nb_st4(dst + 4 * j, make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
          }
        }
        float f4[4];
        nb_tmem_ld4(tm + lq + NB_F3_TM_F, f4);
        if (lane < 16 && nl < U.nrecv) {
          float* dst = a.Fsum + (int64_t)(U.recv0 + nl) * 3;
          dst[0] = f4[0];
          dst[1] = f4[1];
          dst[2] = f4[2];
        }
        nb_tc_fence_before();
        nb_mbar_arrive(accfree);
      }
    }
    if (pend) {
      nb_mbar_wait(done + grp, phase);
      nb_tc_fence_after();
    }
  }
  nb_tc_fence_before();
  __syncthreads();
  if (warp == 0) nb_tmem_dealloc(tm, NB_F3_TMEM_COLS);
}

// ----------------------------------------------------------------------------- backward
// 512 threads: thread (warp w, lane l) owns row 32 (w & 3) + l and the 16 columns of quarter (w >> 2).
//   S1  selector row (for the scatters); pre1 = P_i + Q_j + w_rad r2 + W_e e summed in fp32 from shared-memory
//       copies of the unit's P / Q rows (no gather MMA, no round trip); z1, SiLU'(pre1) parked in TMEM -> MMA 1   pre2
//   S2  m,  SiLU'(pre2) parked in TMEM                 -> MMA 2   pre3
//   S3  phi_x head, g3                                 -> dgrad 3                 | side: dW3, db3
//   S4  g2 = (gm + gM_i) SiLU'(pre2), gM_i from smem   -> dgrad 2                 | side: dW2, db2
//   S5  g1 = gz1 SiLU'(pre1), dL/drij                  ->                           side: gP|gQ|gw += Sel^T g1, gx += Sel^T rG
// One elected lane of warp 0 issues every MMA: first the critical-path ones (mbarrier `bar`), then the side ones
// (`bar2`) -- the tensor pipe runs them in issue order, so the side MMAs execute underneath the next stage's CUDA-core
// work and never ahead of the MMA the CTA is waiting for.
//
// TMEM columns: [0,64) pre1 -> SiLU'(pre1) | [64,128) pre2 -> SiLU'(pre2) | [128,192) pre3 -> gm -> gz1 |
//               [192,256) dW3 | [256,320) dW2 | [320,328) db3 | [328,336) db2 | [336,400) node sums | [400,408) x sums |
//               [448,480) hi pieces, [480,512) lo pieces of the current A operand (z1 -> m -> g3 -> g2; packed bf16 pairs)
// The four critical products read their activation operand from tensor memory (nb_issue_w3_ta): a 128x64x16 MMA with both
// operands in shared memory is bound by the 6 KB operand fetch (~85 cycles measured, tools/stage_clocks.py and the
// timed modes of k_tc_selftest), not by the tensor pipe (32 cycles).  The shared-memory copies stay: the weight-gradient
// and scatter MMAs need the activations as MN-major / B operands, which cannot come from tensor memory.
#define NB_SB_THREADS 512
#define NB_SB_W 0
#define NB_SB_TZ (4 * NB_TC_TILE_BYTES(64))
#define NB_SB_TM (NB_SB_TZ + 2 * NB_TC_TILE_BYTES(128))
#define NB_SB_TG (NB_SB_TM + 2 * NB_TC_TILE_BYTES(128))
#define NB_SB_SEL (NB_SB_TG + 2 * NB_TC_TILE_BYTES(128))
#define NB_SB_NT (NB_SB_SEL + NB_TC_TILE_BYTES(128))
#define NB_SB_GM (NB_SB_NT + 2 * NB_TC_TILE_BYTES(64))
#define NB_SB_ONES (NB_SB_GM + 2 * NB_TC_TILE_BYTES(64))
#define NB_SB_RG (NB_SB_ONES + NB_TILE * 16)
#define NB_SB_FL (NB_SB_RG + 2 * NB_TILE * 16)
#define NB_SB_NFLOAT (4 * NB_H + 4 * NB_TILE + 3 * 32 * 3 + 10 * NB_H + NB_H * 4 + NB_MAX_EF * NB_H)
#define NB_SB_QLD 68  // row stride of the sender rows: lanes of a warp read 16 B of DIFFERENT rows at the same column offset
#define NB_EDGE_BWD_SEL_SMEM(RU) (NB_SB_FL + NB_SB_NFLOAT * 4 + (RU) * 4 + 64 + 1024)
#define NB_SB_GXACC(N) (((N) * 3 + 3) / 4 * 4)
#define NB_EDGE_BWD_SEL_BLK_EXTRA(N) ((32 * NB_H + (N) * NB_H + NB_SB_GXACC(N)) * 4)
#define NB_SB_TMEM_COLS 512

__device__ __forceinline__ void nb_tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void nb_tmem_st16_nowait(uint32_t taddr, const float (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
      "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
      "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
      "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
      : "memory");
}

// dW (+)= G^T A  (both MN-major, K = 128 rows, three split passes) and db (+)= G^T 1
__device__ __forceinline__ void nb_issue_wgrad(uint32_t tmem_w, uint32_t tmem_b, uint32_t g_hi, uint32_t g_lo, uint32_t a_hi,
                                               uint32_t a_lo, uint32_t ones, uint32_t idesc_wg, uint32_t idesc_bs,
                                               uint32_t acc0) {
  uint32_t acc = acc0;
#pragma unroll
  for (int pass = 0; pass < 3; ++pass) {
    const uint32_t ga = nb_desc_lo_mn(pass == 1 ? g_lo : g_hi);
    const uint32_t ab = nb_desc_lo_mn(pass == 2 ? a_lo : a_hi);
#pragma unroll
    for (int s = 0; s < 8; ++s) {
      nb_mma2(tmem_w, ga + NB_KSTEP_MN * s, NB_DESC_HI_SW128, ab + NB_KSTEP_MN * s, NB_DESC_HI_SW128, idesc_wg, acc);
      acc = 1u;
    }
  }
  acc = acc0;
  const uint32_t ob = nb_desc_lo_n8(ones);
#pragma unroll
  for (int pass = 0; pass < 2; ++pass) {
    const uint32_t ga = nb_desc_lo_mn(pass ? g_lo : g_hi);
#pragma unroll
    for (int s = 0; s < 8; ++s) {
      nb_mma2(tmem_b, ga + NB_KSTEP_MN * s, NB_DESC_HI_SW128, ob + NB_KSTEP_N8 * s, NB_DESC_HI_NOSW, idesc_bs, acc);
      acc = 1u;
    }
  }
}

// Optional per-stage cycle counters of CTA 0 (profiling builds only: -DNB_STAGE_CLOCKS, tools/stage_clocks.py)
#ifdef NB_STAGE_CLOCKS
__device__ long long nb_dbg_clk[32];
#define NB_CLK(i)                                   \
  if (dbg_on) {                                     \
    const long long t_now = clock64();              \
    dbg_acc[i] += t_now - dbg_last;                 \
    dbg_last = t_now;                               \
  }
#else
#define NB_CLK(i)
#endif

// dW | db (+)= G^T [A | 1]: the bias column sums ride in the weight-gradient MMAs as a second MN block of the B operand
// (N = 72: the 64 columns of A, then 8 columns of an all-ones SW128 tile `lbo` bytes above a_hi) for the passes
// (g_hi, a_hi), (g_lo, a_hi); the pass (g_hi, a_lo) stays N = 64.  24 MMAs instead of 24 + 16 (an N = 8 MMA costs 23 cycles).
__device__ __forceinline__ void nb_issue_wgrad_fold(uint32_t tmem_w, uint32_t g_hi, uint32_t g_lo, uint32_t a_hi, uint32_t a_lo,
                                                    uint32_t lbo, uint32_t idesc64, uint32_t idesc72, uint32_t acc0) {
  uint32_t acc = acc0;
  const uint32_t b72 = ((a_hi >> 4) & 0x3FFFu) | ((lbo >> 4) << 16);
#pragma unroll
  for (int pass = 0; pass < 3; ++pass) {
    const uint32_t ga = nb_desc_lo_mn(pass == 1 ? g_lo : g_hi);
    const uint32_t ab = pass == 2 ? nb_desc_lo_mn(a_lo) : b72;
#pragma unroll
    for (int s = 0; s < 8; ++s) {
      nb_mma2(tmem_w, ga + NB_KSTEP_MN * s, NB_DESC_HI_SW128, ab + NB_KSTEP_MN * s, NB_DESC_HI_SW128, pass == 2 ? idesc64 : idesc72, acc);
      acc = 1u;
    }
  }
}
// gP | gQ | gw | x sums (+)= Sel^T [g1 | rG]: the [128][8] dL/dr tile rides as the second MN block of the B operand
// (N = 72); its hi / lo pieces live in logical chunks 1 / 2 of the all-ones tile (whose chunk 0 serves the bias fold), so
// the second block starts lbo_* bytes above the g1 piece of the pass.  16 MMAs instead of 16 + 16.
__device__ __forceinline__ void nb_issue_scatter_fold(uint32_t tmem_d, uint32_t sel, uint32_t v_hi, uint32_t v_lo, uint32_t lbo_hi,
                                                      uint32_t lbo_lo, uint32_t idesc72, uint32_t acc0) {
  uint32_t acc = acc0;
  const uint32_t a = nb_desc_lo_mn(sel);
#pragma unroll
  for (int pass = 0; pass < 2; ++pass) {
    const uint32_t b = (((pass ? v_lo : v_hi) >> 4) & 0x3FFFu) | (((pass ? lbo_lo : lbo_hi) >> 4) << 16);
#pragma unroll
    for (int s = 0; s < 8; ++s) {
      nb_mma2(tmem_d, a + NB_KSTEP_MN * s, NB_DESC_HI_SW128, b + NB_KSTEP_MN * s, NB_DESC_HI_SW128, idesc72, acc);
      acc = 1u;
    }
  }
}
#define NB_SB_ONES64_BYTES NB_TC_TILE_BYTES(128)  // whole-graph units only: all-ones SW128 tile (second MN block of the fold)

// EGRAD: S5 also forms dL/de = W_e^T g1 per edge row (a.gef); false is the kernel without input gradients, unchanged
template <bool BLK, bool EGRAD>
__global__ void __launch_bounds__(NB_SB_THREADS, 1) k_edge_bwd_sel(NbEdgeBwdArgs a) {
  NB_PDL_ENTER();
#ifdef NB_STAGE_CLOCKS
  __shared__ long long dbg_acc[32];
  const bool dbg_on = blockIdx.x == 0 && threadIdx.x == 0;
  const long long dbg_t0 = clock64();
  unsigned long long dbg_g0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(dbg_g0));
  long long dbg_last = 0;
  if (dbg_on) {
    for (int i = 0; i < 32; ++i) dbg_acc[i] = 0;
    dbg_last = clock64();
  }
#endif
  extern __shared__ __align__(1024) unsigned char nb_smraw[];
  unsigned char* base = nb_smraw + ((1024u - (nb_smem_u32(nb_smraw) & 1023u)) & 1023u);
  unsigned char* W2h = base + NB_SB_W;
  unsigned char* W2l = W2h + NB_TC_TILE_BYTES(64);
  unsigned char* W3h = W2l + NB_TC_TILE_BYTES(64);
  unsigned char* W3l = W3h + NB_TC_TILE_BYTES(64);
  unsigned char* Tzh = base + NB_SB_TZ;
  unsigned char* Tzl = Tzh + NB_TC_TILE_BYTES(128);
  unsigned char* Tmh = base + NB_SB_TM;
  unsigned char* Tml = Tmh + NB_TC_TILE_BYTES(128);
  unsigned char* Tgh = base + NB_SB_TG;
  unsigned char* Tgl = Tgh + NB_TC_TILE_BYTES(128);
  unsigned char* Sel = base + NB_SB_SEL;
  float* Pf = reinterpret_cast<float*>(base + NB_SB_NT);  // [receivers][64] fp32: P rows of the unit (P includes b1)
  float* Qf = Pf + (BLK ? a.g.IB : a.g.G * a.g.N) * NB_H; // [senders][NB_SB_QLD] fp32: Q rows; receivers + senders <= 54: 14.7 KB
  float* gMs = reinterpret_cast<float*>(base + NB_SB_GM);  // [32][64] fp32: dL/dM_i of the unit's receivers (added in S4)
  float* epart = gMs + 32 * NB_H;  // EGRAD only: [NB_MAX_EF][4][128] quarter sums of dL/de, the unused second half of NB_SB_GM
  unsigned char* ones = base + NB_SB_ONES;
  unsigned char* RGh = base + NB_SB_RG;
  unsigned char* RGl = RGh + NB_TILE * 16;
  float* scratch = reinterpret_cast<float*>(Tzh);  // fp32 [128][64] view, CTA epilogue only
  constexpr bool FOLD = !BLK;  // bias sums folded into the weight-gradient MMAs (needs 16 KB the blocked walk does not have)
  unsigned char* ones64 = base + NB_SB_FL;  // FOLD only
  float* fl = reinterpret_cast<float*>(base + NB_SB_FL + (FOLD ? NB_SB_ONES64_BYTES : 0));
  float* vb2 = fl;
  float* vb3 = vb2 + NB_H;
  float* vw4 = vb3 + NB_H;
  float* vwr = vw4 + NB_H;
  float* cpart = vwr + NB_H;          // [4][128]
  float* xs = cpart + 4 * NB_TILE;    // [32][3] positions of the unit's receivers
  float* xq = xs + 32 * 3;            // [32][3] positions of the unit's senders
  float* gfs = xq + 32 * 3;           // [32][3] dL/dFsum of the unit's receivers
  float* gwacc = gfs + 32 * 3;        // [10][64]: rows 0,1 w_rad (hi, lo piece) ; 2 + 2f, 3 + 2f w_ef[f]
  float* gxst = gwacc + 10 * NB_H;    // [64][4]
  float* Wef = gxst + NB_H * 4;       // [NB_MAX_EF][64] edge-feature columns of W1
  // blocked mode: per-graph accumulators, so that nothing is read-modified-written in global memory per tile
  float* gPacc = Wef + NB_MAX_EF * NB_H;                   // [32][64]  receivers of the current receiver block
  float* gQacc = gPacc + (BLK ? 32 * NB_H : 0);            // [N][64]   all senders of the graph-instance
  float* gxacc = gQacc + (BLK ? a.g.N * NB_H : 0);         // [N][3] (+ pad)
  uint32_t* rowinfo = reinterpret_cast<uint32_t*>(gxacc + (BLK ? NB_SB_GXACC(a.g.N) : 0));
  const NbEdgeGeom g = a.g;
  const int RU = BLK ? 0 : g.G * g.EPG;
  uint64_t* bar = reinterpret_cast<uint64_t*>(rowinfo + RU + (RU & 1));
  uint64_t* bar2 = bar + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar2 + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, cq = warp >> 2;
  const int row = 32 * q + lane;
  const int cb = 16 * cq;

  for (int idx = tid; idx < 64 * 8; idx += NB_SB_THREADS) {
    int o = idx >> 3, j = idx & 7;
    float v2[8], v3[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      v2[i] = __ldg(a.w.W2 + o * NB_H + 8 * j + i);
      v3[i] = __ldg(a.w.W3 + o * NB_H + 8 * j + i);
    }
    nb_tc_store8(W2h, W2l, o, j, v2);
    nb_tc_store8(W3h, W3l, o, j, v3);
  }
  for (int idx = tid; idx < 4 * NB_TC_TILE_BYTES(64) / 16; idx += NB_SB_THREADS)  // P / Q rows + gM rows (contiguous)
    reinterpret_cast<uint4*>(Pf)[idx] = make_uint4(0u, 0u, 0u, 0u);
  for (int idx = tid; idx < NB_MAX_EF * NB_H; idx += NB_SB_THREADS) {
    const int f = idx >> 6, c = idx & 63;
    Wef[idx] = f < g.nef ? __ldg(a.w.W1 + (int64_t)c * a.w.ldw1 + a.w.col_ef + f) : 0.f;
  }
  nb_sel_build_rowinfo(rowinfo, g, tid, NB_SB_THREADS);
  if (tid < NB_TILE) {
    uint32_t one2 = 0x3F803F80u;  // bf16 (1.0, 1.0)
    *reinterpret_cast<uint4*>(ones + tid * 16) = make_uint4(one2, one2, one2, one2);
  }
  if (FOLD)
    for (int idx = tid; idx < (int)(NB_SB_ONES64_BYTES / 16); idx += NB_SB_THREADS)
      reinterpret_cast<uint4*>(ones64)[idx] = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
  if (tid < NB_H) {
    vb2[tid] = __ldg(a.w.b2 + tid);
    vb3[tid] = __ldg(a.w.b3 + tid);
    vw4[tid] = __ldg(a.w.w4 + tid);
    vwr[tid] = __ldg(a.w.W1 + (int64_t)tid * a.w.ldw1 + a.w.col_rad);
  }
  for (int idx = tid; idx < 10 * NB_H; idx += NB_SB_THREADS) gwacc[idx] = 0.f;
  if (tid == 0) {
    nb_mbar_init(bar, 1);
    nb_mbar_init(bar2, 1);
    nb_mbar_fence_init();
  }
  if (warp == 0) nb_tmem_alloc(tmem_slot, NB_SB_TMEM_COLS);
  __syncthreads();
  nb_fence_async_smem();
  nb_tc_fence_before();
  __syncthreads();
  nb_tc_fence_after();
  const uint32_t tm = *tmem_slot;
  const uint32_t lane_base = (uint32_t)(32 * q) << 16;
  const uint32_t t1 = tm + lane_base + 0 + (uint32_t)cb;    // pre1 / SiLU'(pre1)
  const uint32_t t2 = tm + lane_base + 64 + (uint32_t)cb;   // pre2 / SiLU'(pre2)
  const uint32_t t3 = tm + lane_base + 128 + (uint32_t)cb;  // pre3 / gm / gz1
  const uint32_t ta_h = tm + 448, ta_l = tm + 480;            // A operand in tensor memory (issuer's view)
  const uint32_t ta_hm = ta_h + lane_base + 8u * (uint32_t)cq, ta_lm = ta_l + lane_base + 8u * (uint32_t)cq;  // this thread's slice
  const uint32_t idesc_fwd = nb_idesc_bf16(128, 64, 0, 0);
  const uint32_t idesc_dg = nb_idesc_bf16(128, 64, 0, 1);   // also the gathers
  const uint32_t idesc_wg = nb_idesc_bf16(64, 64, 1, 1);    // also the 64-wide scatters
  const uint32_t idesc_bs = nb_idesc_bf16(64, 8, 1, 1);
  const uint32_t idesc_wg72 = nb_idesc_bf16(64, 72, 1, 1);
  // TMEM columns of the weight-gradient accumulators: dW3 | db3 | dW2 | db2 contiguous when folded
  constexpr uint32_t cW3 = 192, cW2 = FOLD ? 264 : 256, cB3 = FOLD ? 256 : 320, cB2 = 328;
  const uint32_t sOnes64 = nb_smem_u32(ones64);
  const uint32_t sTzh = nb_smem_u32(Tzh), sTzl = nb_smem_u32(Tzl), sTmh = nb_smem_u32(Tmh), sTml = nb_smem_u32(Tml),
                 sTgh = nb_smem_u32(Tgh), sTgl = nb_smem_u32(Tgl), sSel = nb_smem_u32(Sel), sOnes = nb_smem_u32(ones),
                 sRGh = nb_smem_u32(RGh), sRGl = nb_smem_u32(RGl), sW2h = nb_smem_u32(W2h), sW2l = nb_smem_u32(W2l),
                 sW3h = nb_smem_u32(W3h), sW3l = nb_smem_u32(W3l);
  const float b4 = __ldg(a.w.b4);
  uint32_t phase = 0, phase2 = 0;
  uint32_t wacc = 0;

  float gw4acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) gw4acc[i] = 0.f;
  float gb4acc = 0.f;

  const int n_outer = BLK ? g.NGT : g.n_units, n_sub = BLK ? g.nI * g.nJ : 1;
  for (int uo = blockIdx.x; uo < n_outer; uo += gridDim.x)
  for (int sub = 0; sub < n_sub; ++sub) {
    const NbSelUnit U = nb_sel_unit<BLK>(g, uo, sub);
    const int R = U.R;
    NB_CLK(0)
    // every MMA of the previous unit has completed (the read-out waited for the last side commit)
    // unit staging: every global load is issued before the first dependent store (one memory round trip, not three).
    // (nrecv + nsend) * 8 <= 432 node-tile tasks and nrecv * 8 <= 256 gM tasks: at most one of each per thread.
    {
      const int n_nt = (U.nrecv + U.nsend) * 8, n_gm = U.first_j ? U.nrecv * 8 : 0;
      const int t_nt = tid + (U.first_j ? 0 : U.nrecv * 8);          // receivers change with the receiver block only
      const bool do_nt = t_nt < n_nt, do_gm = tid < n_gm;
      const int n3r = U.nrecv * 3, n3 = n3r + (BLK ? U.nsend * 3 : 0);
      const int t_x = tid + (U.first_j ? 0 : n3r);
      float4 p0 = make_float4(0.f, 0.f, 0.f, 0.f), p1 = p0, m0 = p0, m1 = p0;
      float xv = 0.f, gv = 0.f;
      int nt_row = 0;
      if (do_nt) {
        const int n = t_nt >> 3, j = t_nt & 7;
        const bool snd = n >= U.nrecv;
        const float* src = snd ? a.Q + (int64_t)(U.send0 + n - U.nrecv) * NB_H + 8 * j : a.P + (int64_t)(U.recv0 + n) * NB_H + 8 * j;
        p0 = nb_ld4(src);
        p1 = nb_ld4(src + 4);
        nt_row = snd ? U.RC + n - U.nrecv : n;
      }
      if (do_gm) {
        const float* src = a.gM + (int64_t)(U.recv0 + (tid >> 3)) * NB_H + 8 * (tid & 7);
        m0 = nb_ld4(src);
        m1 = nb_ld4(src + 4);
      }
      if (t_x < n3) {
        if (t_x < n3r) {
          xv = __ldg(a.x + (int64_t)U.recv0 * 3 + t_x);
          gv = __ldg(a.gFsum + (int64_t)U.recv0 * 3 + t_x);
        } else {
          xv = __ldg(a.x + (int64_t)U.send0 * 3 + (t_x - n3r));
        }
      }
      if (BLK && U.first_i && U.first_j)
        for (int idx = tid; idx < g.N * 3; idx += NB_SB_THREADS) gxacc[idx] = 0.f;
      if (do_nt) {  // nt_row: receivers [0, nrecv), senders [RC, RC + nsend)
        float* dst = nt_row < U.RC ? Pf + nt_row * NB_H + 8 * (t_nt & 7) : Qf + (nt_row - U.RC) * NB_SB_QLD + 8 * (t_nt & 7);
        nb_st4(dst, p0);
        nb_st4(dst + 4, p1);
      }
      if (do_gm) {
        nb_st4(gMs + (tid >> 3) * NB_H + 8 * (tid & 7), m0);
        nb_st4(gMs + (tid >> 3) * NB_H + 8 * (tid & 7) + 4, m1);
      }
      if (t_x < n3) {
        if (t_x < n3r) {
          xs[t_x] = xv;
          gfs[t_x] = gv;
        } else {
          xq[t_x - n3r] = xv;
        }
      }
    }
    const float* xsnd = BLK ? xq : xs;  // whole-graph units: senders = receivers
    __syncthreads();
    NB_CLK(1)

    for (int r0 = 0; r0 < R; r0 += NB_TILE) {
      // ---- T0: geometry + selector row
      float dx = 0.f, dy = 0.f, dz = 0.f, r2 = 0.f, gfx = 0.f, gfy = 0.f, gfz = 0.f;
      float e[NB_MAX_EF];
#pragma unroll
      for (int f = 0; f < NB_MAX_EF; ++f) e[f] = 0.f;
      int li = 0, lj = 0, gt = 0, rem = 0;
      const bool valid = nb_sel_row<BLK>(g, U, rowinfo, r0 + row, li, lj, gt, rem);
      if (valid) {
        dx = xs[li * 3 + 0] - xsnd[lj * 3 + 0];
        dy = xs[li * 3 + 1] - xsnd[lj * 3 + 1];
        dz = xs[li * 3 + 2] - xsnd[lj * 3 + 2];
        r2 = dx * dx + dy * dy + dz * dz;
        gfx = gfs[li * 3 + 0];
        gfy = gfs[li * 3 + 1];
        gfz = gfs[li * 3 + 2];
        {
          const int64_t eoff = ((int64_t)nb_ef_graph(g, gt) * g.EPG + rem) * g.nef;
#pragma unroll
          for (int f = 0; f < NB_MAX_EF; ++f)
            if (f < g.nef) e[f] = __ldg(a.ef + eoff + f);
        }
      }
      NB_CLK(2)
      if (r0 > 0) {  // the side MMAs of the previous tile (dW2, scatters) have consumed Sel, Tz, Tm, Tg, rG
        nb_mbar_wait(bar2, phase2);
        phase2 ^= 1;
        nb_tc_fence_after();
      }
      NB_CLK(3)
      if (cq < 2) nb_sel_write_row(Sel, row, cq, valid, li, U.RC + lj, r2, e);  // consumed by the scatters of S5
      // ---- S1: pre1 in fp32 from the unit's P / Q rows; z1 -> tile, SiLU'(pre1) -> TMEM
      {
        float v[16], d[16];
        const float* pr = Pf + (valid ? li : 0) * NB_H + cb;
        const float* qr = Qf + (valid ? lj : 0) * NB_SB_QLD + cb;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float4 pp = nb_ld4(pr + 4 * k), qq = nb_ld4(qr + 4 * k), wr = nb_ld4(vwr + cb + 4 * k);
          v[4 * k + 0] = fmaf(r2, wr.x, pp.x + qq.x);
          v[4 * k + 1] = fmaf(r2, wr.y, pp.y + qq.y);
          v[4 * k + 2] = fmaf(r2, wr.z, pp.z + qq.z);
          v[4 * k + 3] = fmaf(r2, wr.w, pp.w + qq.w);
        }
#pragma unroll
        for (int f = 0; f < NB_MAX_EF; ++f)
          if (f < g.nef) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float4 we = nb_ld4(Wef + f * NB_H + cb + 4 * k);
              v[4 * k + 0] = fmaf(e[f], we.x, v[4 * k + 0]);
              v[4 * k + 1] = fmaf(e[f], we.y, v[4 * k + 1]);
              v[4 * k + 2] = fmaf(e[f], we.z, v[4 * k + 2]);
              v[4 * k + 3] = fmaf(e[f], we.w, v[4 * k + 3]);
            }
          }
        if (!valid) {  // padded rows: pre1 = 0 (what their all-zero selector row used to gather)
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = 0.f;
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) nb_silu_grad(v[i], v[i], d[i]);
        nb_tmem_st16_nowait(t1, d);
        nb_store16_ta(Tzh, Tzl, row, cq, v, ta_hm, ta_lm);
        nb_tmem_st_wait();  // one wait for the parked SiLU' values and the A operand
      }
      nb_fence_async_smem();
      nb_tc_fence_before();
      __syncthreads();
      NB_CLK(7)
      if (NB_ISSUER(0)) {
        nb_tc_fence_after();
        nb_issue_w3_ta(tm + 64, ta_h, ta_l, sW2h, sW2l, false, idesc_fwd, 0u);
        nb_mma_commit(bar);
      }
      NB_CLK(8)
      nb_mbar_wait(bar, phase);
      phase ^= 1;
      nb_tc_fence_after();
      NB_CLK(9)
      // ---- S2: m -> tile, SiLU'(pre2) -> TMEM
      {
        float v[16], d[16];
        nb_tmem_ld16(t2, v);
#pragma unroll
        for (int i = 0; i < 16; ++i) nb_silu_grad(v[i] + vb2[cb + i], v[i], d[i]);
        nb_tmem_st16_nowait(t2, d);
        nb_store16_ta(Tmh, Tml, row, cq, v, ta_hm, ta_lm);
        nb_tmem_st_wait();
      }
      nb_fence_async_smem();
      nb_tc_fence_before();
      __syncthreads();
      NB_CLK(10)
      if (NB_ISSUER(0)) {
        nb_tc_fence_after();
        nb_issue_w3_ta(tm + 128, ta_h, ta_l, sW3h, sW3l, false, idesc_fwd, 0u);
        nb_mma_commit(bar);
      }
      NB_CLK(11)
      nb_mbar_wait(bar, phase);
      phase ^= 1;
      nb_tc_fence_after();
      NB_CLK(12)
      // ---- S3: phi_x head, g3 = dL/dpre3
      float rgx, rgy, rgz;
      {
        float v[16], d[16];
        nb_tmem_ld16(t3, v);
        float cp = 0.f;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          nb_silu_grad(v[i] + vb3[cb + i], v[i], d[i]);  // v = z3
          cp = fmaf(vw4[cb + i], v[i], cp);
        }
        cpart[cq * NB_TILE + row] = cp;
        nb_tc_fence_before();
        __syncthreads();
        const float cval = (cpart[row] + cpart[NB_TILE + row]) + (cpart[2 * NB_TILE + row] + cpart[3 * NB_TILE + row]) + b4;
        if (g.clamp_edge) {  // clamp(rij * c) passes gradient only inside [-100, 100]
          float fx = dx * cval, fy = dy * cval, fz = dz * cval;
          if (!(fx >= -100.f && fx <= 100.f)) gfx = 0.f;
          if (!(fy >= -100.f && fy <= 100.f)) gfy = 0.f;
          if (!(fz >= -100.f && fz <= 100.f)) gfz = 0.f;
        }
        const float gc = dx * gfx + dy * gfy + dz * gfz;  // 0 for padded rows
        rgx = cval * gfx;
        rgy = cval * gfy;
        rgz = cval * gfz;
        if (cq == 0) gb4acc += gc;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          gw4acc[i] = fmaf(gc, v[i], gw4acc[i]);
          v[i] = gc * vw4[cb + i] * d[i];  // g3
        }
        nb_store16_ta(Tgh, Tgl, row, cq, v, ta_hm, ta_lm);
        nb_tmem_st_wait();
      }
      nb_fence_async_smem();
      nb_tc_fence_before();
      __syncthreads();
      NB_CLK(13)
      if (NB_ISSUER(0)) {
        nb_tc_fence_after();
        nb_issue_w3_ta(tm + 128, ta_h, ta_l, sW3h, sW3l, true, idesc_dg, 0u);        // gm = g3 W3  (+ gM_i: added in S4)
        nb_mma_commit(bar);
        NB_CLK(14)
        if (FOLD) nb_issue_wgrad_fold(tm + cW3, sTgh, sTgl, sTmh, sTml, sOnes64 - sTmh, idesc_wg, idesc_wg72, wacc);
        else nb_issue_wgrad(tm + cW3, tm + cB3, sTgh, sTgl, sTmh, sTml, sOnes, idesc_wg, idesc_bs, wacc);  // dW3, db3
        nb_mma_commit(bar2);
      }
      NB_CLK(15)
      nb_mbar_wait(bar, phase);
      phase ^= 1;
      nb_tc_fence_after();
      NB_CLK(16)
      // ---- S4: g2 = (gm + gM_i) * SiLU'(pre2)    (padded rows: gm = 0 and the gathered gM = 0)
      {
        float v[16], d[16];
        nb_tmem_ld16(t3, v);
        nb_tmem_ld16(t2, d);
        {  // + dL/dM of the row's receiver, straight from shared memory (exact; 4 gather MMAs less on the critical path)
          int li4 = 0, lj4, gt4, rem4;
          const bool ok4 = nb_sel_row<BLK>(g, U, rowinfo, r0 + row, li4, lj4, gt4, rem4);
          const float* gmr = gMs + (ok4 ? li4 : 0) * NB_H + cb;
          const float msk = ok4 ? 1.f : 0.f;  // padded rows: g2 = 0 (their SiLU' values are arbitrary)
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float4 gq = nb_ld4(gmr + 4 * k);
            v[4 * k + 0] = fmaf(msk, gq.x, v[4 * k + 0]);
            v[4 * k + 1] = fmaf(msk, gq.y, v[4 * k + 1]);
            v[4 * k + 2] = fmaf(msk, gq.z, v[4 * k + 2]);
            v[4 * k + 3] = fmaf(msk, gq.w, v[4 * k + 3]);
          }
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] *= d[i];
        NB_CLK(17)
        nb_mbar_wait(bar2, phase2);  // dW3 / db3 have consumed the g3 and m tiles
        phase2 ^= 1;
        NB_CLK(18)
        nb_store16_ta(Tgh, Tgl, row, cq, v, ta_hm, ta_lm);
        nb_tmem_st_wait();
      }
      nb_fence_async_smem();
      nb_tc_fence_before();
      __syncthreads();
      NB_CLK(19)
      if (NB_ISSUER(0)) {
        nb_tc_fence_after();
        nb_issue_w3_ta(tm + 128, ta_h, ta_l, sW2h, sW2l, true, idesc_dg, 0u);  // gz1 = g2 W2
        nb_mma_commit(bar);
        NB_CLK(20)
        if (FOLD) nb_issue_wgrad_fold(tm + cW2, sTgh, sTgl, sTzh, sTzl, sOnes64 - sTzh, idesc_wg, idesc_wg72, wacc);
        else nb_issue_wgrad(tm + cW2, tm + cB2, sTgh, sTgl, sTzh, sTzl, sOnes, idesc_wg, idesc_bs, wacc);  // dW2, db2
      }
      wacc = 1;
      NB_CLK(21)
      nb_mbar_wait(bar, phase);
      phase ^= 1;
      nb_tc_fence_after();
      NB_CLK(22)
      // ---- S5: g1 = gz1 * SiLU'(pre1) -> the (free) m tile ; dL/drij -> rG tile
      {
        float v[16], d[16];
        nb_tmem_ld16(t3, v);
        nb_tmem_ld16(t1, d);
        float gr2 = 0.f;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          v[i] *= d[i];
          gr2 = fmaf(vwr[cb + i], v[i], gr2);  // dL/dr2 = w_rad . g1
        }
        cpart[cq * NB_TILE + row] = gr2;
        if constexpr (EGRAD) {  // dL/de_f = w_ef[f] . g1: this quarter's 16 columns
#pragma unroll
          for (int f = 0; f < NB_MAX_EF; ++f)
            if (f < g.nef) {
              float ge = 0.f;
#pragma unroll
              for (int i = 0; i < 16; ++i) ge = fmaf(Wef[f * NB_H + cb + i], v[i], ge);
              epart[(f * 4 + cq) * NB_TILE + row] = ge;
            }
        }
        nb_tc_store8(Tmh, Tml, row, 2 * cq, v);
        nb_tc_store8(Tmh, Tml, row, 2 * cq + 1, v + 8);
      }
      nb_tc_fence_before();
      __syncthreads();
      if (cq == 0) {
        const float gr2 = 2.f * ((cpart[row] + cpart[NB_TILE + row]) + (cpart[2 * NB_TILE + row] + cpart[3 * NB_TILE + row]));
        const uint32_t px = nb_pack_split(fmaf(dx, gr2, rgx)), py = nb_pack_split(fmaf(dy, gr2, rgy)),
                       pz = nb_pack_split(fmaf(dz, gr2, rgz));
        const uint4 rh = make_uint4((px & 0xffffu) | (py << 16), pz & 0xffffu, 0u, 0u);
        const uint4 rl = make_uint4((px >> 16) | (py & 0xffff0000u), pz >> 16, 0u, 0u);
        if (FOLD) {  // logical chunks 1 (hi) and 2 (lo) of this row of the all-ones tile
          *reinterpret_cast<uint4*>(ones64 + nb_tc_chunk_off(row, 1)) = rh;
          *reinterpret_cast<uint4*>(ones64 + nb_tc_chunk_off(row, 2)) = rl;
        } else {
          *reinterpret_cast<uint4*>(RGh + row * 16) = rh;
          *reinterpret_cast<uint4*>(RGl + row * 16) = rl;
        }
        if constexpr (EGRAD) {  // the four quarters in a fixed order; one plain store per replicated row and feature
          int li5 = 0, lj5, gt5 = 0, rem5 = 0;
          if (nb_sel_row<BLK>(g, U, rowinfo, r0 + row, li5, lj5, gt5, rem5)) {
            float* dst = a.gef + ((int64_t)gt5 * g.EPG + rem5) * g.nef;
#pragma unroll
            for (int f = 0; f < NB_MAX_EF; ++f)
              if (f < g.nef) {
                const float* ep = epart + f * 4 * NB_TILE + row;
                dst[f] = (ep[0] + ep[NB_TILE]) + (ep[2 * NB_TILE] + ep[3 * NB_TILE]);
              }
          }
        }
      }
      nb_fence_async_smem();
      __syncthreads();
      NB_CLK(23)
      if (NB_ISSUER(0)) {
        nb_tc_fence_after();
        const uint32_t uacc = r0 > 0 ? 1u : 0u;
        if (FOLD) {  // [gP | gQ | gw partials | x sums] += Sel^T [g1 | rG]: accumulator columns [336, 408)
          nb_issue_scatter_fold(tm + 336, sSel, sTmh, sTml, sOnes64 + 16 - sTmh, sOnes64 + 32 - sTml, idesc_wg72, uacc);
        } else {
          nb_issue_scatter(tm + 336, sSel, sTmh, sTml, idesc_wg, uacc);    // gP | gQ | gw partials += Sel^T g1
          nb_issue_scatter8(tm + 400, sSel, sRGh, sRGl, idesc_bs, uacc);   // x sums += Sel^T rG
        }
        nb_mma_commit(bar2);  // also covers dW2 / db2; waited for at the top of the next tile / at the read-out
      }
      NB_CLK(24)
    }
    // ---- unit read-out (accumulator row i <-> TMEM lane (i % 16) + 32 (i / 16): thread (q, lane < 16) owns row 16 q + lane)
    nb_mbar_wait(bar2, phase2);
    phase2 ^= 1;
    nb_tc_fence_after();
    NB_CLK(25)
    float gx_old = 0.f;  // whole-graph units: issued here, consumed after the read-out's barrier (latency hidden)
    if (!BLK && tid < U.nrecv * 3) gx_old = a.gx[(int64_t)U.recv0 * 3 + tid];
    {
      const int i = 16 * q + lane;
      float v[16];
      nb_tmem_ld16(tm + lane_base + 336 + (uint32_t)cb, v);
      if (lane < 16) {
        const bool is_recv = i < U.nrecv, is_send = i >= U.RC && i < U.RC + U.nsend;
        if (is_recv || is_send) {
          float* dst = is_recv ? a.gP + (int64_t)(U.recv0 + i) * NB_H + cb : a.gQ + (int64_t)(U.send0 + i - U.RC) * NB_H + cb;
          if (!BLK) {
#pragma unroll
            for (int k = 0; k < 4; ++k) nb_st4(dst + 4 * k, make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]));
          } else {
            // this thread is the only one that ever touches this accumulator slice: gP collects the sender blocks of
            // the receiver block, gQ the receiver blocks of the graph-instance; global memory is written once
            float* acc = is_recv ? gPacc + i * NB_H + cb : gQacc + (U.J0 + i - U.RC) * NB_H + cb;
            const bool first = is_recv ? U.first_j : U.first_i, last = is_recv ? U.last_j : U.last_i;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              float4 o = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
              if (!first) {
                const float4 old = nb_ld4(acc + 4 * k);
                o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w;
              }
              nb_st4(last ? dst + 4 * k : acc + 4 * k, o);
            }
          }
        } else if (i >= NB_SEL_XC0) {
          float* dst = gwacc + (i - NB_SEL_XC0) * NB_H + cb;  // exclusive owner of these 16 accumulators
#pragma unroll
          for (int k = 0; k < 16; ++k) dst[k] += v[k];
        }
      }
      float f4[4];
      nb_tmem_ld4(tm + lane_base + 400, f4);
      if (cq == 0 && lane < 16) {
        gxst[i * 4 + 0] = f4[0];
        gxst[i * 4 + 1] = f4[1];
        gxst[i * 4 + 2] = f4[2];
      }
    }
    nb_tc_fence_before();
    __syncthreads();
    // dL/dx: + receiver sums - sender sums
    if (!BLK) {  // one node list
      if (tid < U.nrecv * 3) {  // nrecv * 3 <= 81 < blockDim.x
        const int n = tid / 3, dd = tid - 3 * n;
        a.gx[(int64_t)U.recv0 * 3 + tid] = gx_old + (gxst[n * 4 + dd] - gxst[(U.RC + n) * 4 + dd]);
      }
    } else {       // two lists that may overlap: two passes, into the per-graph accumulator
      for (int idx = tid; idx < U.nrecv * 3; idx += NB_SB_THREADS) {
        int n = idx / 3, dd = idx - 3 * n;
        gxacc[U.I0 * 3 + idx] += gxst[n * 4 + dd];
      }
      __syncthreads();
      for (int idx = tid; idx < U.nsend * 3; idx += NB_SB_THREADS) {
        int n = idx / 3, dd = idx - 3 * n;
        gxacc[U.J0 * 3 + idx] -= gxst[(U.RC + n) * 4 + dd];
      }
      if (U.last_i && U.last_j) {
        __syncthreads();
        for (int idx = tid; idx < g.N * 3; idx += NB_SB_THREADS) a.gx[(int64_t)U.gt0 * g.N * 3 + idx] += gxacc[idx];
      }
    }
    __syncthreads();
  }

  NB_CLK(26)
#ifdef NB_STAGE_CLOCKS
  if (dbg_on)
    for (int i = 0; i < 32; ++i) nb_dbg_clk[i] += dbg_acc[i];
#endif
  // ---- CTA epilogue: weight-gradient accumulators (TMEM), register / shared accumulators -> this CTA's partial slice
  float* out = a.partial + (int64_t)blockIdx.x * NB_EB_PLEN;
  nb_tc_fence_after();
  {
    float v[16];
    const int o = 16 * q + lane;
    nb_tmem_ld16(tm + lane_base + 192 + (uint32_t)cb, v);  // dW3[o][cb..]
    if (lane < 16 && wacc) {
#pragma unroll
      for (int k = 0; k < 4; ++k) nb_st4(out + NB_EB_GW3 + o * NB_H + cb + 4 * k, make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]));
    }
    nb_tmem_ld16(tm + lane_base + cW2 + (uint32_t)cb, v);  // dW2[o][cb..]
    if (lane < 16 && wacc) {
#pragma unroll
      for (int k = 0; k < 4; ++k) nb_st4(out + NB_EB_GW2 + o * NB_H + cb + 4 * k, make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]));
    }
    float b3v[4], b2v[4];
    nb_tmem_ld4(tm + lane_base + cB3, b3v);  // db3 / db2: every column of the 8-wide block holds the sum
    nb_tmem_ld4(tm + lane_base + cB2, b2v);
    if (lane < 16 && cq == 0 && wacc) {
      out[NB_EB_GB3 + o] = b3v[0];
      out[NB_EB_GB2 + o] = b2v[0];
    }
  }
  if (!wacc) {  // a CTA that processed no tile contributes zeros
    for (int idx = tid; idx < 2 * NB_H * NB_H + 2 * NB_H; idx += NB_SB_THREADS) out[idx] = 0.f;
  }
  // dw4: sum of the per-row accumulators over the 128 rows (through an fp32 scratch over the z1 tile); db4 likewise
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 4; ++k)
    nb_st4(nb_scratch_chunk(scratch, row, (cb >> 2) + k),
           make_float4(gw4acc[4 * k], gw4acc[4 * k + 1], gw4acc[4 * k + 2], gw4acc[4 * k + 3]));
  if (cq == 0) cpart[row] = gb4acc;
  __syncthreads();
  {
    const int rc = tid & 63, rpart = tid >> 6;  // column, part (0..7): 16 rows each
    float sacc = 0.f;
    for (int r = rpart * 16; r < rpart * 16 + 16; ++r) sacc += nb_scratch_get(scratch, r, rc);
    float* red = reinterpret_cast<float*>(Tmh);  // [8][64]
    red[rpart * NB_H + rc] = sacc;
    __syncthreads();
    if (tid < NB_H) {
      float t = 0.f;
#pragma unroll
      for (int p = 0; p < 8; ++p) t += red[p * NB_H + tid];
      out[NB_EB_GW4 + tid] = t;
      out[NB_EB_GWR + tid] = gwacc[tid] + gwacc[NB_H + tid];
#pragma unroll
      for (int f = 0; f < NB_MAX_EF; ++f) out[NB_EB_GWE + f * NB_H + tid] = gwacc[(2 + 2 * f) * NB_H + tid] + gwacc[(3 + 2 * f) * NB_H + tid];
      float t4 = 0.f;
      if (tid == 0)
        for (int r = 0; r < NB_TILE; ++r) t4 += cpart[r];
      out[NB_EB_GB4 + tid] = t4;
    }
  }
  nb_tc_fence_before();
  __syncthreads();
  if (warp == 0) nb_tmem_dealloc(tm, NB_SB_TMEM_COLS);
#ifdef NB_STAGE_CLOCKS
  if (threadIdx.x == 0) {  // whole-CTA cycles: [27] max over CTAs and launches, [28] sum over CTAs; [29] the same span in ns
    const long long dt = clock64() - dbg_t0;
    unsigned long long g1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g1));
    atomicMax((unsigned long long*)&nb_dbg_clk[27], (unsigned long long)dt);
    atomicAdd((unsigned long long*)&nb_dbg_clk[28], (unsigned long long)dt);
    atomicAdd((unsigned long long*)&nb_dbg_clk[29], g1 - dbg_g0);  // [28] / [29] = effective SM clock in GHz
  }
#endif
}
#endif  // NB_EMU
