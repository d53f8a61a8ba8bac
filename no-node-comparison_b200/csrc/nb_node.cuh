// nb_node.cuh — node-level kernels: 64-wide tiled GEMM with fused epilogues, weight-gradient
// reduction, partial-sum finalisation, and the row-wise update kernels of EGNO / SEGNO.
//
// Node-level work is ~1/(N-1) of the edge work (SURVEY.md §8), HBM-light and expressed through a
// small set of generic kernels; the fused edge tile lives in nb_edge.cuh.
#pragma once
#include "nb_common.cuh"

// ============================================================================= gemm64
// out[r][0:64] = epi( sum_s  act_s(A_s[r][0:64]) @ B_s  + bias ) (+ R[r]) , B_s[k][n] = W_s[k*sk + n*sn] * scale_s
struct NbGemmSrc {
  const float* A;
  int lda;
  int a_silu;  // apply SiLU to A while loading (A holds pre-activations)
  const float* W;
  int64_t sk, sn;
  float scale;
  int kmax;    // valid k of this source (<= 64; operand rows beyond it are taken as zero)
  // tcgen05 kernel only: a pre-split copy of the 64 x 64 weight block in the shared-memory tile layout (8 KB of hi
  // pieces, then 8 KB of lo pieces, SW128; tile row = the block's row, tile column = its column), written once per call by
  // k_weight_images.  A CTA then stages its B operand with 1 024 coalesced 16-byte copies instead of 4 096 strided scalar
  // loads.  img_mn = 1: the product uses the block transposed (dgrad), i.e. reads the same image as an MN-major operand.
  const unsigned char* img;
  int img_mn;
  // segmented rows (seg_rows > 0): logical row r of A lives in block r / seg_rows at offset r % seg_rows, blocks seg_a
  // floats apart (the same tensor of all SEGNO sub-steps, stored one block per sub-step)
  int seg_rows;
  int64_t seg_a;
};
__device__ __forceinline__ const float* nb_seg_row(const float* base, int ld, int seg_rows, int64_t seg_stride, int64_t r) {
  if (seg_rows <= 0) return base + r * ld;
  const int64_t sgm = r / seg_rows;
  return base + sgm * seg_stride + (r - sgm * seg_rows) * ld;
}
enum { NB_EPI_NONE = 0, NB_EPI_SILU = 1, NB_EPI_MUL_DSILU = 2 };
struct NbGemmArgs {
  int rows;
  int nsrc;
  NbGemmSrc src[2];
  const float* bias;  // [64] or null
  int epi;
  const float* U;  // NB_EPI_MUL_DSILU: out = acc * silu'(U[r][c])
  int ldu;
  const float* R;  // residual added after the epilogue (nullable)
  int ldr;
  float* out;
  int ldo;
  int accumulate;  // out += result
  float* out_pre;  // optional: pre-activation (acc + bias) stored here
  int ldp;
};

#define NB_MAX_GEMM_JOBS 4
struct NbGemmBatch {
  int njobs;
  NbGemmArgs job[NB_MAX_GEMM_JOBS];
};

// blockIdx.y selects the job; blockIdx.x the 128-row tile (CTAs past a job's last tile exit)
__global__ void __launch_bounds__(NB_THREADS) k_gemm64(NbGemmBatch batch) {
  NB_PDL_ENTER();
  const NbGemmArgs& a = batch.job[blockIdx.y];
  if ((int)blockIdx.x * NB_TILE >= a.rows) return;
  NB_DYN_SMEM(sm);
  float* As = sm;                     // [128][68]
  float* Bs = sm + NB_TILE * NB_LDA;  // [64][64]
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int r0 = blockIdx.x * NB_TILE;
  const int nv = min(NB_TILE, a.rows - r0);
  float acc[8][4];
#pragma unroll
  for (int q = 0; q < 8; ++q) acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.f;

  for (int s = 0; s < a.nsrc; ++s) {
    if (s > 0) __syncthreads();
    nb_stage_b(Bs, a.src[s].W, a.src[s].sk, a.src[s].sn, a.src[s].scale, tid, a.src[s].kmax);
    const float* A = a.src[s].A;
    const int lda = a.src[s].lda;
    const int asilu = a.src[s].a_silu;
    for (int idx = tid; idx < NB_TILE * 16; idx += NB_THREADS) {
      int r = idx >> 4, c4 = idx & 15;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < nv) {
        v = nb_ld4(nb_seg_row(A, lda, a.src[s].seg_rows, a.src[s].seg_a, r0 + r) + c4 * 4);
        if (asilu) {
          v.x = nb_silu(v.x);
          v.y = nb_silu(v.y);
          v.z = nb_silu(v.z);
          v.w = nb_silu(v.w);
        }
      }
      nb_st4(As + r * NB_LDA + c4 * 4, v);
    }
    __syncthreads();
    nb_tile_gemm<8>(As, Bs, acc, ty, tx);
  }

  float4 bias = make_float4(0.f, 0.f, 0.f, 0.f);
  if (a.bias) bias = make_float4(__ldg(a.bias + tx * 4), __ldg(a.bias + tx * 4 + 1), __ldg(a.bias + tx * 4 + 2),
                                 __ldg(a.bias + tx * 4 + 3));
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    int r = ty + 16 * q;
    if (r >= nv) continue;
    int64_t gr = r0 + r;
    float4 v = make_float4(acc[q][0] + bias.x, acc[q][1] + bias.y, acc[q][2] + bias.z, acc[q][3] + bias.w);
    if (a.out_pre) nb_st4(a.out_pre + gr * a.ldp + tx * 4, v);
    if (a.epi == NB_EPI_SILU) {
      v.x = nb_silu(v.x);
      v.y = nb_silu(v.y);
      v.z = nb_silu(v.z);
      v.w = nb_silu(v.w);
    } else if (a.epi == NB_EPI_MUL_DSILU) {
      float4 u = nb_ld4(a.U + gr * a.ldu + tx * 4);
      v.x *= nb_dsilu(u.x);
      v.y *= nb_dsilu(u.y);
      v.z *= nb_dsilu(u.z);
      v.w *= nb_dsilu(u.w);
    }
    if (a.R) {
      float4 rr = nb_ld4(a.R + gr * a.ldr + tx * 4);
      v.x += rr.x;
      v.y += rr.y;
      v.z += rr.z;
      v.w += rr.w;
    }
    if (a.out) {
      float* o = a.out + gr * a.ldo + tx * 4;
      if (a.accumulate) {
        float4 old = nb_ld4(o);
        v.x += old.x;
        v.y += old.y;
        v.z += old.z;
        v.w += old.w;
      }
      nb_st4(o, v);
    }
  }
}

// ============================================================================= wgrad64
// partial[cta][o*64 + k] = sum over this CTA's rows of  sum_p scale_p * G_p[r][o] * act_p(A_p[r][k])
// partial[cta][4096 + o]  = column sums of G_0 (bias gradient), when colsum != 0
#define NB_WGRAD_PLEN (NB_H * NB_H + NB_H)
struct NbWgradPair {
  const float* G;
  int ldg;
  const float* A;
  int lda;
  int a_silu;
  float scale;
  // segmented operands (seg_rows > 0): logical row r lives in segment r / seg_rows at offset r % seg_rows; segments
  // are seg_g / seg_a floats apart.  Lets ONE reduction run over the same tensor of all SEGNO sub-steps (stored one
  // block per sub-step) instead of one small reduction per sub-step.
  int seg_rows;
  int64_t seg_g, seg_a;
};
#define nb_wg_row nb_seg_row
struct NbWgradArgs {
  int rows;
  int npair;
  NbWgradPair pair[2];
  int colsum;
  float* partial;  // [gridDim.x][NB_WGRAD_PLEN]
};

#define NB_MAX_WGRAD_JOBS 12
struct NbWgradBatch {
  int njobs;
  NbWgradArgs job[NB_MAX_WGRAD_JOBS];
};

// blockIdx.y selects the job; each job owns gridDim.x partial slices
__global__ void __launch_bounds__(NB_THREADS) k_wgrad64(NbWgradBatch batch) {
  NB_PDL_ENTER();
  const NbWgradArgs& a = batch.job[blockIdx.y];
  NB_DYN_SMEM(sm);
  float* Gs = sm;                     // [128][68]
  float* As = sm + NB_TILE * NB_LDA;  // [128][68]
  const int tid = threadIdx.x, wk = tid & 15, wo = tid >> 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
  float csum = 0.f;
  const int ntiles = (a.rows + NB_TILE - 1) / NB_TILE;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int r0 = tile * NB_TILE;
    const int nv = min(NB_TILE, a.rows - r0);
    for (int p = 0; p < a.npair; ++p) {
      __syncthreads();
      const NbWgradPair pr = a.pair[p];
      for (int idx = tid; idx < nv * 16; idx += NB_THREADS) {
        int r = idx >> 4, c4 = idx & 15;
        float4 g = nb_ld4(nb_wg_row(pr.G, pr.ldg, pr.seg_rows, pr.seg_g, r0 + r) + c4 * 4);
        float4 v = nb_ld4(nb_wg_row(pr.A, pr.lda, pr.seg_rows, pr.seg_a, r0 + r) + c4 * 4);
        if (pr.a_silu) {
          v.x = nb_silu(v.x);
          v.y = nb_silu(v.y);
          v.z = nb_silu(v.z);
          v.w = nb_silu(v.w);
        }
        g.x *= pr.scale;
        g.y *= pr.scale;
        g.z *= pr.scale;
        g.w *= pr.scale;
        nb_st4(Gs + r * NB_LDA + c4 * 4, g);
        nb_st4(As + r * NB_LDA + c4 * 4, v);
      }
      __syncthreads();
      nb_tile_wgrad(Gs, As, nv, acc, wo, wk);
      if (a.colsum && p == 0 && tid < NB_H) {
        float s = 0.f;
        for (int r = 0; r < nv; ++r) s += Gs[r * NB_LDA + tid];
        csum += s;
      }
    }
  }
  float* out = a.partial + (int64_t)blockIdx.x * NB_WGRAD_PLEN;
#pragma unroll
  for (int i = 0; i < 4; ++i)
    nb_st4(out + (wo * 4 + i) * NB_H + wk * 4, make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]));
  if (tid < NB_H) out[NB_H * NB_H + tid] = a.colsum ? csum : 0.f;
}

// ============================================================================= finalize
// dst[seg.dst_off + o*so + k*si] (=|+=) sum_p partial[p][e],  e = seg.start + o*inner + k
// One launch finalises a batch of reductions (blockIdx.y = job).  A block handles 32 consecutive elements: lane =
// element (coalesced 128-byte reads of each partial slice), warp w sums the slices p = w, w+8, ...; the 8 warp sums
// meet in shared memory in a fixed order (deterministic).
#define NB_MAX_SEG 8
#define NB_MAX_FIN_JOBS 16
struct NbFinSeg {
  int start, count, inner;
  int64_t dst_off, so, si;
  int klimit;  // > 0: only k < klimit is written (results narrower than the 64-wide accumulator rows)
};
struct NbFinArgs {
  const float* partial;
  int nparts, plen, nseg, total;
  NbFinSeg seg[NB_MAX_SEG];
  float* dst;
  int accumulate;
};
struct NbFinBatch {
  int njobs;
  NbFinArgs job[NB_MAX_FIN_JOBS];
};

__global__ void __launch_bounds__(256) k_finalize(NbFinBatch batch) {
  NB_PDL_ENTER();
  __shared__ float red[8][33];
  const NbFinArgs& a = batch.job[blockIdx.y];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int idx = blockIdx.x * 32 + lane;
  if (blockIdx.x * 32 >= a.total) return;
  // locate the segment of flat element idx (segments are listed back to back in `total` space)
  int s = 0, base = 0;
  const bool act = idx < a.total;
  if (act) {
    while (s < a.nseg - 1 && idx >= base + a.seg[s].count) {
      base += a.seg[s].count;
      ++s;
    }
  }
  const int l = idx - base;
  const int e = a.seg[s].start + l;
  float sum = 0.f;
  if (act) {
    // 4 independent partial sums per warp keep 4 loads in flight; combined in a fixed order (deterministic)
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    int p = warp;
    for (; p + 24 < a.nparts; p += 32) {
      s0 += a.partial[(int64_t)p * a.plen + e];
      s1 += a.partial[(int64_t)(p + 8) * a.plen + e];
      s2 += a.partial[(int64_t)(p + 16) * a.plen + e];
      s3 += a.partial[(int64_t)(p + 24) * a.plen + e];
    }
    for (; p < a.nparts; p += 8) s0 += a.partial[(int64_t)p * a.plen + e];
    sum = (s0 + s1) + (s2 + s3);
  }
  red[warp][lane] = sum;
  __syncthreads();
  if (warp == 0 && act) {
    float t = red[0][lane];
#pragma unroll
    for (int w = 1; w < 8; ++w) t += red[w][lane];
    const NbFinSeg sg = a.seg[s];
    int o = l / sg.inner, k = l - o * sg.inner;
    if (sg.klimit <= 0 || k < sg.klimit) {
      float* d = a.dst + sg.dst_off + (int64_t)o * sg.so + (int64_t)k * sg.si;
      if (a.accumulate) t += *d;
      *d = t;
    }
  }
}

// ============================================================================= embedding
// out[t][k][o] = sum_f W[o][f] * in_f + b[o];  in = [ nodes[k][0:F0] | sin(ts*freq) | cos(ts*freq) ],
// ts = timesteps[(k mod B)][t]  -- the reference's `k mod B` broadcast quirk (egno.py:66).  D == 0: no time part.
struct NbEmbedArgs {
  int T, Nn0, B, F0, D;  // D = time_emb_dim (even), 0 for SEGNO
  const float* nodes;    // [Nn0][F0]
  const int64_t* tsteps; // [B][T]
  const float* W;        // [64][F0 + D]
  const float* bias;     // [64]
  float* out;            // [T*Nn0][64]
  float freq[32];        // D/2 frequencies
  float* table;          // [T][B][D] sinusoidal embedding of timesteps[b][t] (k_time_table), read by the kernels below
  // EGNO num_inputs = L > 1 (egno.py:42-47,59-61,68-70): node features per input frame, a second embedding of the
  // input times; frame t reads input tmap[t]
  int L;                       // 0 / 1: single input
  const int64_t* tsteps_in;    // [B][L]
  float* table_in;             // [T][B][D]: embedding of timesteps_in[b][tmap[t]]
  int tmap[NB_MAX_T];
};

// table[t][b][j] = sin(ts * freq[j]) (j < D/2) | cos(ts * freq[j - D/2]),  ts = timesteps[b][t]   (layer_no.py:8-17)
__device__ __forceinline__ float nb_time_emb(const NbEmbedArgs& a, int j, float ts) {
  const int half = a.D >> 1;
  const float arg = ts * a.freq[j < half ? j : j - half];
  return j < half ? sinf(arg) : cosf(arg);
}
__global__ void __launch_bounds__(256) k_time_table(NbEmbedArgs a, int input_times) {
  NB_PDL_ENTER();
  const int total = a.T * a.B * a.D;
  float* tab = input_times ? a.table_in : a.table;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int j = idx % a.D, tb = idx / a.D, b = tb % a.B, t = tb / a.B;
    const float ts = input_times ? (float)__ldg(a.tsteps_in + (int64_t)b * a.L + a.tmap[t])
                                 : (float)__ldg(a.tsteps + (int64_t)b * a.T + t);
    tab[idx] = nb_time_emb(a, j, ts);
  }
}
// the same table from fp32 times (`timesteps.float()` of a floating-point tensor): integral values give the int64
// kernel's table bit for bit, since (float)int64 is exact below 2^24
__global__ void __launch_bounds__(256) k_time_table_f(NbEmbedArgs a, const float* __restrict__ ts_out,
                                                      const float* __restrict__ ts_in, int input_times) {
  NB_PDL_ENTER();
  const int total = a.T * a.B * a.D;
  float* tab = input_times ? a.table_in : a.table;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int j = idx % a.D, tb = idx / a.D, b = tb % a.B, t = tb / a.B;
    const float ts = input_times ? __ldg(ts_in + (int64_t)b * a.L + a.tmap[t]) : __ldg(ts_out + (int64_t)b * a.T + t);
    tab[idx] = nb_time_emb(a, j, ts);
  }
}

// dL/dtimes through the sinusoidal embeddings, from G = dL/d(embedding output) [T][Nn0][64] and W = W_emb [64][ldw]:
//   gt_out[b][t] = sum_j (Gs[t][b] . W[:, c_out + j]) demb_j/dt,   Gs[t][b] = sum over the nodes k = b mod B of G[t][k]
// (the `k mod B` broadcast of egno.py:66,69), with d sin(t f)/dt = f cos(t f) and d cos(t f)/dt = -f sin(t f);
// c_out = F0 for one input frame, F0 + D for several, whose input-time columns c_in = F0 give gt_in[b][l] as the same
// sum over the frames t with tmap[t] = l.  One CTA per trajectory b; every sum runs in a fixed order (no atomics).
// gt_out and gt_in are nullable.
constexpr int NB_TGRAD_THREADS = 256;
__global__ void __launch_bounds__(NB_TGRAD_THREADS) k_time_grad(NbEmbedArgs a, const float* __restrict__ ts_out,
                                                                const float* __restrict__ ts_in,
                                                                const float* __restrict__ G, const float* __restrict__ W,
                                                                int ldw, float* __restrict__ gt_out,
                                                                float* __restrict__ gt_in) {
  NB_PDL_ENTER();
  __shared__ float gs[NB_MAX_T * NB_H];   // Gs[t][:] of this trajectory
  __shared__ float q[NB_MAX_T * 128];     // [t][in-time columns | out-time columns] terms of the sums over j
  __shared__ float pin[NB_MAX_T];         // per-frame input-time sums
  const int b = blockIdx.x, tid = threadIdx.x, D = a.D, T = a.T, N = a.Nn0 / a.B;
  const bool multi = a.L > 1;
  const int ncol = multi ? 2 * D : D, c0 = a.F0;
  for (int i = tid; i < T * NB_H; i += NB_TGRAD_THREADS) {
    const int t = i / NB_H, c = i % NB_H;
    const float* g = G + ((int64_t)t * a.Nn0 + b) * NB_H + c;
    float s = 0.f;
    for (int n = 0; n < N; ++n) s += __ldg(g + (int64_t)n * a.B * NB_H);
    gs[i] = s;
  }
  __syncthreads();
  for (int i = tid; i < T * ncol; i += NB_TGRAD_THREADS) {
    const int t = i / ncol, j = i % ncol;
    const float* gt = gs + t * NB_H;
    float p = 0.f;
#pragma unroll 8
    for (int c = 0; c < NB_H; ++c) p = fmaf(gt[c], __ldg(W + (int64_t)c * ldw + c0 + j), p);
    const bool in = multi && j < D;
    const int jj = multi && !in ? j - D : j, half = D >> 1;
    const float ts = in ? __ldg(ts_in + (int64_t)b * a.L + a.tmap[t]) : __ldg(ts_out + (int64_t)b * T + t);
    const float f = a.freq[jj < half ? jj : jj - half], arg = ts * f;
    q[t * 128 + j] = p * (jj < half ? f * cosf(arg) : -f * sinf(arg));
  }
  __syncthreads();
  const int warp = tid >> 5, lane = tid & 31;
  for (int t = warp; t < T; t += NB_TGRAD_THREADS / 32) {
    const float* qt = q + t * 128;
    float so = 0.f, si = 0.f;
    for (int j = lane; j < D; j += 32) {
      so += qt[(multi ? D : 0) + j];
      if (multi) si += qt[j];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      so += __shfl_xor_sync(0xffffffffu, so, o);
      si += __shfl_xor_sync(0xffffffffu, si, o);
    }
    if (lane == 0) {
      if (gt_out) gt_out[(int64_t)b * T + t] = so;
      pin[t] = si;
    }
  }
  if (!multi || !gt_in) return;
  __syncthreads();
  if (tid < a.L) {
    float s = 0.f;
    for (int t = 0; t < T; ++t)
      if (a.tmap[t] == tid) s += pin[t];
    gt_in[(int64_t)b * a.L + tid] = s;
  }
}

// feature f of the embedding input of node k at frame t: [ nodes | (emb of the input time) | emb of the output time ]
__device__ __forceinline__ float nb_embed_feature(const NbEmbedArgs& a, int t, int k, int f) {
  const bool multi = a.L > 1;
  if (f < a.F0) return __ldg(a.nodes + ((int64_t)(multi ? a.tmap[t] : 0) * a.Nn0 + k) * a.F0 + f);
  f -= a.F0;
  const int64_t tb = ((int64_t)t * a.B + (k % a.B)) * a.D;   // the `k mod B` broadcast of egno.py:66,69
  if (multi) {
    if (f < a.D) return __ldg(a.table_in + tb + f);
    f -= a.D;
  }
  return __ldg(a.table + tb + f);
}

// ein[row][0:64] = [ nodes | time embedding | zeros ]: the embedding Linear and its weight gradient then run through
// the 64-wide GEMM / weight-gradient kernels (tcgen05 on the GPU).  One thread per (row, 4 columns).
__global__ void __launch_bounds__(256) k_embed_inputs(NbEmbedArgs a, float* __restrict__ ein, int foff) {
  NB_PDL_ENTER();
  const int F = a.F0 + a.D * (a.L > 1 ? 2 : 1) - foff;   // features foff .. foff + 63 of the input row
  const int64_t total = (int64_t)a.T * a.Nn0 * 16;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = idx >> 4;
    const int c0 = (int)(idx & 15) * 4;
    const int t = (int)(row / a.Nn0), k = (int)(row % a.Nn0);
    float v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = c0 + i < F ? nb_embed_feature(a, t, k, foff + c0 + i) : 0.f;
    nb_st4(ein + row * NB_H + c0, make_float4(v[0], v[1], v[2], v[3]));
  }
}

__global__ void __launch_bounds__(256) k_embed_fwd(NbEmbedArgs a) {
  NB_PDL_ENTER();
  NB_DYN_SMEM(sm);
  const int F = a.F0 + a.D;
  float* Ws = sm;              // [F][64] transposed
  float* ins = sm + F * NB_H;  // [4][F]
  const int tid = threadIdx.x, o = tid & 63, lr = tid >> 6;
  for (int idx = tid; idx < F * NB_H; idx += 256) {
    int oo = idx / F, f = idx - oo * F;
    Ws[f * NB_H + oo] = __ldg(a.W + idx);
  }
  const float b = __ldg(a.bias + o);
  const int64_t rows = (int64_t)a.T * a.Nn0;
  for (int64_t rb = (int64_t)blockIdx.x * 4; rb < rows; rb += (int64_t)gridDim.x * 4) {
    __syncthreads();
    for (int idx = tid; idx < 4 * F; idx += 256) {
      int rr = idx / F, f = idx - rr * F;
      int64_t row = rb + rr;
      ins[idx] = row < rows ? nb_embed_feature(a, (int)(row / a.Nn0), (int)(row % a.Nn0), f) : 0.f;
    }
    __syncthreads();
    int64_t row = rb + lr;
    if (row < rows) {
      float s = b;
      for (int f = 0; f < F; ++f) s = fmaf(ins[lr * F + f], Ws[f * NB_H + o], s);
      a.out[row * NB_H + o] = s;
    }
  }
}

// gW[o][f] = sum_rows g[row][o] * in_f(row);  gb[o] = sum_rows g[row][o]
// partial[cta][o*F + f], partial[cta][64*F + o]
struct NbEmbedBwdArgs {
  NbEmbedArgs e;
  const float* g;  // [T*Nn0][64]
  float* partial;  // [grid][64*F + 64]
};

__global__ void __launch_bounds__(256) k_embed_bwd(NbEmbedBwdArgs a) {
  NB_PDL_ENTER();
  NB_DYN_SMEM(sm);
  const int F = a.e.F0 + a.e.D;
  float* ins = sm;            // [32][F]
  float* gs = sm + 32 * F;    // [32][64]
  const int tid = threadIdx.x, o = tid & 63, fg = tid >> 6;  // 4 feature groups
  const int fper = (F + 3) / 4;
  float acc[16];  // fper <= 16  (F <= 64)
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = 0.f;
  float bsum = 0.f;
  const int64_t rows = (int64_t)a.e.T * a.e.Nn0;
  for (int64_t rb = (int64_t)blockIdx.x * 32; rb < rows; rb += (int64_t)gridDim.x * 32) {
    __syncthreads();
    for (int idx = tid; idx < 32 * F; idx += 256) {
      int rr = idx / F, f = idx - rr * F;
      int64_t row = rb + rr;
      ins[idx] = row < rows ? nb_embed_feature(a.e, (int)(row / a.e.Nn0), (int)(row % a.e.Nn0), f) : 0.f;
    }
    for (int idx = tid; idx < 32 * NB_H; idx += 256) {
      int rr = idx >> 6;
      int64_t row = rb + rr;
      gs[idx] = row < rows ? a.g[row * NB_H + (idx & 63)] : 0.f;
    }
    __syncthreads();
    for (int rr = 0; rr < 32; ++rr) {
      float gv = gs[rr * NB_H + o];
      if (fg == 0) bsum += gv;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        int f = fg * fper + i;
        if (i < fper && f < F) acc[i] = fmaf(gv, ins[rr * F + f], acc[i]);
      }
    }
  }
  float* out = a.partial + (int64_t)blockIdx.x * (NB_H * F + NB_H);
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    int f = fg * fper + i;
    if (i < fper && f < F) out[o * F + f] = acc[i];
  }
  if (fg == 0) out[NB_H * F + o] = bsum;
}

// ============================================================================= small row-wise kernels
// frame t of the T output frames is fed by input tmap[t] (all zeros for a single input)
struct NbFrameMap {
  int L;
  int m[NB_MAX_T];
};
// dst[t][k][0:3] = src[tmap[t]][k][0:3]
__global__ void __launch_bounds__(256) k_replicate3(const float* __restrict__ src, float* __restrict__ dst, int n3,
                                                    int T, NbFrameMap fm) {
  NB_PDL_ENTER();
  int64_t total = (int64_t)n3 * T;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x)
    dst[i] = src[(int64_t)fm.m[i / n3] * n3 + i % n3];
}
// dst[l][k] = sum over the frames t fed by input l of src[t][k]
__global__ void __launch_bounds__(256) k_sum_over_t(const float* __restrict__ src, float* __restrict__ dst, int n3,
                                                    int T, NbFrameMap fm) {
  NB_PDL_ENTER();
  const int64_t total = (int64_t)n3 * fm.L;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int l = (int)(idx / n3), i = (int)(idx - (int64_t)l * n3);
    float s = 0.f;
    for (int t = 0; t < T; ++t)
      if (fm.m[t] == l) s += src[(int64_t)t * n3 + i];
    dst[idx] = s;
  }
}

// ----------------------------------------------------------------------------- input gradients (nb_*_backward_ex)
// dst[i] = sum over the slices s = 0 .. nslices-1, in that order, of src[s * n + i]
__global__ void __launch_bounds__(256) k_sum_slices(const float* __restrict__ src, float* __restrict__ dst, int64_t n,
                                                    int nslices) {
  NB_PDL_ENTER();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int k = 0; k < nslices; ++k) s += src[(int64_t)k * n + i];
    dst[i] = s;
  }
}
// the embedding's input gradient: out[r][f] = sum_c g[r][c] W[c][f] for the first F0 of the ldw input columns
__global__ void __launch_bounds__(256) k_embed_input_grad(const float* __restrict__ g, const float* __restrict__ W, int ldw,
                                                          int F0, int64_t rows, float* __restrict__ out) {
  NB_PDL_ENTER();
  const int64_t total = rows * F0;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = idx / F0;
    const int f = (int)(idx - r * F0);
    const float* gr = g + r * NB_H;
    float s = 0.f;
#pragma unroll 8
    for (int c = 0; c < NB_H; ++c) s = fmaf(gr[c], __ldg(W + (int64_t)c * ldw + f), s);
    out[idx] = s;
  }
}
// EGNO loc_mean: x1 = x0 + conv(x0 - mean) with the mean added back, so one layer contributes
// dL/dmean = sum_t (dL/dx1[t] - dL/dx0[t]); layers accumulate in the order of the backward sweep
__global__ void __launch_bounds__(256) k_loc_mean_grad(const float* __restrict__ gx1, const float* __restrict__ gx0,
                                                       float* __restrict__ g_mean, int n3, int T, int accumulate) {
  NB_PDL_ENTER();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n3; i += (int64_t)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int t = 0; t < T; ++t) s += gx1[(int64_t)t * n3 + i] - gx0[(int64_t)t * n3 + i];
    g_mean[i] = accumulate ? g_mean[i] + s : s;
  }
}

// EGNO coordinate update (basic.py:172-178):  s = w2 . SiLU(UV) + b2 ;  x' = x + s v + clamp(Fsum/(N-1), +-100)
struct NbXupdArgs {
  int64_t rows;
  int N;
  const float *x, *v, *UV, *w2, *b2, *Fsum;
  float* x_out;
  // backward
  const float *gx, *gv;  // incoming [rows,3]
  float *gv_out, *gFsum, *GUV;
  float* partial;  // [grid][65]: gw2[64], gb2
};

__global__ void __launch_bounds__(256) k_egno_xupd_fwd(NbXupdArgs a) {
  NB_PDL_ENTER();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float w0 = __ldg(a.w2 + 2 * lane), w1 = __ldg(a.w2 + 2 * lane + 1), b2 = __ldg(a.b2);
  const float cnt = (float)(a.N - 1 > 1 ? a.N - 1 : 1);
  for (int64_t row = (int64_t)blockIdx.x * 8 + warp; row < a.rows; row += (int64_t)gridDim.x * 8) {
    const float2 uv = *reinterpret_cast<const float2*>(a.UV + row * NB_H + 2 * lane);  // one 256-byte row per warp load
    float s = w0 * nb_silu(uv.x) + w1 * nb_silu(uv.y);
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) s += __shfl_xor_sync(0xffffffffu, s, m);
    s += b2;
    if (lane < 3) {
      float f = a.Fsum[row * 3 + lane] / cnt;
      f = fminf(fmaxf(f, -100.f), 100.f);
      a.x_out[row * 3 + lane] = a.x[row * 3 + lane] + s * a.v[row * 3 + lane] + f;
    }
  }
}

__global__ void __launch_bounds__(256) k_egno_xupd_bwd(NbXupdArgs a) {
  NB_PDL_ENTER();
  __shared__ float red[8][65];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float w0 = __ldg(a.w2 + 2 * lane), w1 = __ldg(a.w2 + 2 * lane + 1), b2 = __ldg(a.b2);
  const float cnt = (float)(a.N - 1 > 1 ? a.N - 1 : 1);
  float gw0 = 0.f, gw1 = 0.f, gb = 0.f;
  for (int64_t row = (int64_t)blockIdx.x * 8 + warp; row < a.rows; row += (int64_t)gridDim.x * 8) {
    float z0, d0, z1, d1;
    const float2 uv = *reinterpret_cast<const float2*>(a.UV + row * NB_H + 2 * lane);  // lane owns columns 2l, 2l+1
    nb_silu_grad(uv.x, z0, d0);
    nb_silu_grad(uv.y, z1, d1);
    float s = w0 * z0 + w1 * z1;
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) s += __shfl_xor_sync(0xffffffffu, s, m);
    s += b2;
    float gxl = lane < 3 ? a.gx[row * 3 + lane] : 0.f;
    float vl = lane < 3 ? a.v[row * 3 + lane] : 0.f;
    float gs = gxl * vl;
    gs += __shfl_xor_sync(0xffffffffu, gs, 1);
    gs += __shfl_xor_sync(0xffffffffu, gs, 2);
    gs = __shfl_sync(0xffffffffu, gs, 0);  // lanes 0..3 hold the sum (lane 3 contributes 0)
    if (lane < 3) {
      float gvin = a.gv ? a.gv[row * 3 + lane] : 0.f;
      a.gv_out[row * 3 + lane] = gvin + s * gxl;
      float f = a.Fsum[row * 3 + lane] / cnt;
      a.gFsum[row * 3 + lane] = (f >= -100.f && f <= 100.f) ? gxl / cnt : 0.f;
    }
    *reinterpret_cast<float2*>(a.GUV + row * NB_H + 2 * lane) = make_float2(gs * w0 * d0, gs * w1 * d1);
    gw0 = fmaf(gs, z0, gw0);
    gw1 = fmaf(gs, z1, gw1);
    gb += gs;
  }
  red[warp][2 * lane] = gw0;
  red[warp][2 * lane + 1] = gw1;
  if (lane == 0) red[warp][64] = gb;
  __syncthreads();
  if (threadIdx.x < 65) {
    float s = 0.f;
    for (int w = 0; w < 8; ++w) s += red[w][threadIdx.x];
    a.partial[(int64_t)blockIdx.x * 65 + threadIdx.x] = s;
  }
}

// SEGNO integrator (gcl.py:101-102,116-117):  a = Fsum/(N-1) * cw ; v' = v + a/T ; x' = x + v'/T
struct NbIntegArgs {
  int64_t n3;  // rows*3
  int N;
  float inv_T, cw;
  const float *x, *v, *Fsum;
  float *x_out, *v_out;
  const float *gx, *gv;         // backward in
  float *gx_out, *gv_out, *gFsum;  // backward out (gx_out may alias gx)
};
__global__ void __launch_bounds__(256) k_segno_integ_fwd(NbIntegArgs a) {
  NB_PDL_ENTER();
  const float cnt = (float)(a.N - 1 > 1 ? a.N - 1 : 1);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.n3; i += (int64_t)gridDim.x * blockDim.x) {
    float acc = a.Fsum[i] / cnt * a.cw;
    float vn = a.v[i] + acc * a.inv_T;
    a.v_out[i] = vn;
    a.x_out[i] = a.x[i] + vn * a.inv_T;
  }
}
__global__ void __launch_bounds__(256) k_segno_integ_bwd(NbIntegArgs a) {
  NB_PDL_ENTER();
  const float cnt = (float)(a.N - 1 > 1 ? a.N - 1 : 1);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.n3; i += (int64_t)gridDim.x * blockDim.x) {
    float gxi = a.gx ? a.gx[i] : 0.f;
    float gvt = (a.gv ? a.gv[i] : 0.f) + gxi * a.inv_T;
    a.gx_out[i] = gxi;
    a.gv_out[i] = gvt;
    a.gFsum[i] = gvt * a.inv_T * a.cw / cnt;
  }
}

// Canonical fully connected edge list check (dataset_simple.py:64-71, :101-111).
__global__ void __launch_bounds__(256) k_check_edges(const int64_t* __restrict__ row, const int64_t* __restrict__ col,
                                                     int64_t E, int B, int N, int* flag) {
  NB_PDL_ENTER();
  const int64_t epg = (int64_t)N * (N - 1);
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x) {
    int64_t b = e / epg, rem = e - b * epg;
    int64_t i = rem / (N - 1), jj = rem - i * (N - 1);
    int64_t j = jj + (jj >= i ? 1 : 0);
    if (row[e] != b * N + i || col[e] != b * N + j) atomicCAS(flag, 0, (int)(e % 2147483646) + 1);
  }
}

// ============================================================================= fused Adam over the flat buffers
// torch.optim.Adam semantics (amsgrad = False, maximize = False): g += wd p; m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2;
// p -= lr / (1 - b1^t) * m / (sqrt(v) / sqrt(1 - b2^t) + eps).  The step counter lives on the device (k_adam_tick), so
// the pair of launches is CUDA-graph capturable; parameters and gradients are ONE flat buffer each (the layout of the
// C ABI), so one launch updates the whole model.
__global__ void k_adam_tick(float* step) {
  NB_PDL_ENTER(); *step += 1.0f; }

#define NB_MAX_PEERS 8
struct NbAdamArgs {
  int64_t n;
  float* p;
  const float* g;
  float *m, *v;
  const float* step;   // already incremented
  double lr, beta1, beta2, eps, weight_decay;   // hyper-parameters in double, like the Python scalars torch uses
  float grad_scale;    // gradients are multiplied by it first (data parallel: 1 / world over the summed bucket)
  // Data parallel over peer memory (npeer > 0): the gradient is the SUM over the ranks' flat gradient buffers, read in
  // place through NVLink / NVSwitch (peer[r] = rank r's buffer as mapped into this process), in rank order on every rank
  // so that the replicas stay bit-identical: the all-reduce and the optimizer update are one kernel, no collective call.
  const float* peer[NB_MAX_PEERS];
  int npeer;
};
__global__ void __launch_bounds__(256) k_adam(NbAdamArgs a) {
  NB_PDL_ENTER();
  const double t = (double)*a.step;
  const double bc1 = 1.0 - pow(a.beta1, t), bc2 = 1.0 - pow(a.beta2, t);
  const float step_size = (float)(a.lr / bc1), bc2_sqrt = (float)sqrt(bc2);
  const float b1 = (float)a.beta1, b2 = (float)a.beta2, omb1 = (float)(1.0 - a.beta1), omb2 = (float)(1.0 - a.beta2);
  const float eps = (float)a.eps, wd = (float)a.weight_decay;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += (int64_t)gridDim.x * blockDim.x) {
    const float p = a.p[i];
    float gsum;
    if (a.npeer > 0) {
      float pg[NB_MAX_PEERS];
#pragma unroll
      for (int r = 0; r < NB_MAX_PEERS; ++r) pg[r] = r < a.npeer ? a.peer[r][i] : 0.f;   // all loads in flight together
      gsum = pg[0];
#pragma unroll
      for (int r = 1; r < NB_MAX_PEERS; ++r) gsum += pg[r];
    } else {
      gsum = a.g[i];
    }
    const float g = fmaf(wd, p, gsum * a.grad_scale);  // grad.add(param, alpha=weight_decay)
    const float m = fmaf(omb1, g - a.m[i], a.m[i]);      // exp_avg.lerp_(grad, 1 - beta1)
    const float v = fmaf(omb2 * g, g, b2 * a.v[i]);      // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
    a.m[i] = m;
    a.v[i] = v;
    a.p[i] = p - step_size * (m / (sqrtf(v) / bc2_sqrt + eps));   // param.addcdiv_(exp_avg, denom, value=-step_size)
    (void)b1;
  }
}
