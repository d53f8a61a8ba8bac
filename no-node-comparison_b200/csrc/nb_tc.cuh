// nb_tc.cuh — tcgen05 / TMEM / mbarrier building blocks (sm_100a inline PTX) for the 64-wide MLP tiles.
//
// Numerics: operands are split into two bf16 pieces, x = b1 + b2 (+ O(2^-18 x)), and every product is evaluated as
// b1*c1 + b2*c1 + b1*c2 with fp32 accumulation in TMEM ("fp32-accumulated split-BF16", SURVEY.md §7): three
// kind::f16 MMAs per logical fp32 MMA, ~1e-5 relative error per product, at 1.5x the tensor time of one TF32 pass
// and half the shared-memory bytes of a TF32 hi/lo split.
//
// One physical tile layout serves every operand role.  A tile is [rows][64] bf16, 128 bytes per row, with the
// canonical 128-byte swizzle (16-byte chunk index XOR (row & 7)); tile bases are 1024-byte aligned.
//   * K-major operand   (K = the 64 columns):  k-step s (16 elements) starts at byte 32*s of each row;
//                                              SBO = 1024 B between 8-row groups.
//   * MN-major operand  (MN = the 64 columns, K = rows): k-step s covers rows 16 s .. 16 s + 15, start = 2048 * s;
//                                              SBO = 1024 B between 8-row K groups; one 128-byte MN block (LBO unused).
// For 16-bit types these two canonical layouts (cute::UMMA::Layout_K_SW128_Atom / Layout_MN_SW128_Atom) coincide
// physically, which is what lets the backward reuse one copy of m, z1, g and W for recompute, dgrad and wgrad.
#pragma once
#ifndef NB_EMU
#include <cuda_bf16.h>
#include "nb_common.cuh"

#define NB_TC_ROW_BYTES 128            // 64 bf16
#define NB_TC_TILE_BYTES(rows) ((rows) * NB_TC_ROW_BYTES)

__device__ __forceinline__ uint32_t nb_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ----------------------------------------------------------------------------- mbarrier
__device__ __forceinline__ void nb_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(nb_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void nb_mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void nb_mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t a = nb_smem_u32(bar);
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "DONE:\n\t"
      "}" ::"r"(a),
      "r"(parity)
      : "memory");
}

// ----------------------------------------------------------------------------- TMEM
__device__ __forceinline__ void nb_tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(nb_smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void nb_tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // the allocating warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void nb_tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void nb_tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// generic-proxy shared-memory writes -> visible to the async proxy (tensor core operand reads)
// One lane of a fully converged warp (call under a warp-uniform condition only).  MMAs issued under
// `if (warp == W && nb_elect_one())` compile to back-to-back UTCHMMA; under `if (tid == 0)` the compiler wraps every
// single MMA in an ELECT / BRA.U.ANY loop (about ten instructions per MMA, all on the critical path of the issuing warp).
__device__ __forceinline__ bool nb_elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}
#define NB_ISSUER(w) (warp == (w) && nb_elect_one())

// One thread hands a contiguous global -> shared copy (16-byte aligned, a multiple of 16 bytes) to the TMA engine
// (cp.async.bulk, UBLKCP in SASS); `bar` (initialised with count 1) completes when all `bytes` have landed.  The weight
// images of the node kernels are stored in global memory in their shared-memory tile layout, so a whole set of tiles is
// one such copy: no register staging, and the copy runs underneath the first tile's row loads.  The data is written and
// (by tcgen05.mma) read through the async proxy: the reader only has to wait for the barrier.
__device__ __forceinline__ void nb_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  const uint32_t b = nb_smem_u32(bar);
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(nb_smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(b)
               : "memory");
}
__device__ __forceinline__ void nb_fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// 32 lanes x 32 consecutive fp32 columns: thread l of warp w reads TMEM lane 32*(w%4)+l
__device__ __forceinline__ void nb_tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// store 32 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void nb_tmem_st32(uint32_t taddr, const float (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
      "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
      "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
      "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15])),
      "r"(__float_as_uint(v[16])), "r"(__float_as_uint(v[17])), "r"(__float_as_uint(v[18])), "r"(__float_as_uint(v[19])),
      "r"(__float_as_uint(v[20])), "r"(__float_as_uint(v[21])), "r"(__float_as_uint(v[22])), "r"(__float_as_uint(v[23])),
      "r"(__float_as_uint(v[24])), "r"(__float_as_uint(v[25])), "r"(__float_as_uint(v[26])), "r"(__float_as_uint(v[27])),
      "r"(__float_as_uint(v[28])), "r"(__float_as_uint(v[29])), "r"(__float_as_uint(v[30])), "r"(__float_as_uint(v[31]))
      : "memory");
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// ----------------------------------------------------------------------------- descriptors
// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) |
// version=1 [46,48) | layout_type [61,64) (2 = SWIZZLE_128B)
__device__ __forceinline__ uint64_t nb_make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// K-major view of a [rows][64] bf16 tile, k-step s (16 columns)
__device__ __forceinline__ uint64_t nb_desc_kmajor(uint32_t tile_addr, int s) {
  return nb_make_desc(tile_addr + 32 * s, 16, 1024);
}
// MN-major view (MN = the 64 columns, K = rows), k-step s (rows 16 s ..)
__device__ __forceinline__ uint64_t nb_desc_mnmajor(uint32_t tile_addr, int s) {
  return nb_make_desc(tile_addr + 2048 * s, 8192, 1024);
}
// dense [rows][8] bf16 tile (16 bytes per row, no swizzle) as an MN-major operand with MN = 8, K = rows:
// canonical INTERLEAVE layout ((8,1),(8,k)) : 8x8 core matrices of 128 contiguous bytes, K groups LBO = 128 B apart.
__device__ __forceinline__ uint64_t nb_desc_mn8_noswizzle(uint32_t tile_addr, int s) {
  uint64_t d = 0;
  d |= (uint64_t)(((tile_addr + 256 * s) >> 4) & 0x3FFF);
  d |= (uint64_t)((128 >> 4) & 0x3FFF) << 16;   // LBO: stride between 8-row K groups
  d |= (uint64_t)((128 >> 4) & 0x3FFF) << 32;   // SBO: stride between MN blocks (single block: unused)
  d |= (uint64_t)1 << 46;
  return d;                                      // layout_type 0 = SWIZZLE_NONE
}
// instruction descriptor (cute::UMMA::InstrDescriptor), kind::f16, bf16 x bf16 -> f32
__host__ __device__ constexpr uint32_t nb_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) /*c=f32*/ | (1u << 7) /*a=bf16*/ | (1u << 10) /*b=bf16*/ | ((uint32_t)a_mn_major << 15) |
         ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem], issued by ONE thread
__device__ __forceinline__ void nb_mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]: the A operand (M = 128 rows on the 128 lanes, K-major: the 16 bf16 of a k-step packed
// two per 32-bit column, 8 columns per k-step) is read from tensor memory instead of shared memory.  A 128x64x16 MMA
// with both operands in shared memory is bound by the operand fetch (6 KB per MMA), not by the tensor pipe.
__device__ __forceinline__ void nb_mma_bf16_ta(uint32_t tmem_d, uint32_t tmem_a, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 db;\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t"
      "}" ::"r"(tmem_d),
      "r"(tmem_a), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void nb_tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// split 8 consecutive fp32 values into packed bf16 pairs: hi[i] = (v[2i], v[2i+1]) leading pieces, lo[i] = the remainders
__device__ __forceinline__ void nb_split8(const float* v, uint32_t (&hi)[4], uint32_t (&lo)[4]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __nv_bfloat162 b1 = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    float2 f1 = __bfloat1622float2(b1);
    __nv_bfloat162 b2 = __floats2bfloat162_rn(v[2 * i] - f1.x, v[2 * i + 1] - f1.y);
    hi[i] = *reinterpret_cast<uint32_t*>(&b1);
    lo[i] = *reinterpret_cast<uint32_t*>(&b2);
  }
}
// 8 consecutive 32-bit columns of this thread's TMEM lane <- two groups of 4 packed words
__device__ __forceinline__ void nb_tmem_st44(uint32_t taddr, const uint32_t (&a)[4], const uint32_t (&b)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(a[0]),
               "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3])
               : "memory");
}

// all MMAs issued so far by this thread arrive on `bar` when complete (implies fence::before_thread_sync)
__device__ __forceinline__ void nb_mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(nb_smem_u32(bar)) : "memory");
}

// ----------------------------------------------------------------------------- split-bf16 tile stores
// byte offset of the 16-byte chunk j (8 bf16, columns 8j..8j+7) of row r inside a swizzled tile
__device__ __forceinline__ uint32_t nb_tc_chunk_off(int r, int j) { return (uint32_t)r * NB_TC_ROW_BYTES + (uint32_t)((j ^ (r & 7)) << 4); }

// split 8 consecutive fp32 values into their bf16 pieces and store chunk j of row r into the hi / lo tiles
__device__ __forceinline__ void nb_tc_store8(unsigned char* hi, unsigned char* lo, int r, int j, const float* v) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __nv_bfloat162 b1 = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    float2 f1 = __bfloat1622float2(b1);
    __nv_bfloat162 b2 = __floats2bfloat162_rn(v[2 * i] - f1.x, v[2 * i + 1] - f1.y);
    h[i] = *reinterpret_cast<uint32_t*>(&b1);
    l[i] = *reinterpret_cast<uint32_t*>(&b2);
  }
  uint32_t off = nb_tc_chunk_off(r, j);
  *reinterpret_cast<uint4*>(hi + off) = make_uint4(h[0], h[1], h[2], h[3]);
  *reinterpret_cast<uint4*>(lo + off) = make_uint4(l[0], l[1], l[2], l[3]);
}

// Issue the three split passes of one logical 64-deep (K-major A) or rows-deep (MN-major) product.
//   a_mn / b_mn: operand views;  ksteps: 4 for K = 64 columns, rows/16 for K = rows.
__device__ __forceinline__ void nb_tc_issue3(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, int a_mn, uint32_t b_hi,
                                             uint32_t b_lo, int b_mn, int ksteps, uint32_t idesc, bool accumulate) {
  uint32_t acc = accumulate ? 1u : 0u;
#pragma unroll 1
  for (int pass = 0; pass < 3; ++pass) {
    uint32_t a = pass == 1 ? a_lo : a_hi;
    uint32_t b = pass == 2 ? b_lo : b_hi;
    for (int s = 0; s < ksteps; ++s) {
      uint64_t ad = a_mn ? nb_desc_mnmajor(a, s) : nb_desc_kmajor(a, s);
      uint64_t bd = b_mn ? nb_desc_mnmajor(b, s) : nb_desc_kmajor(b, s);
      nb_mma_bf16(tmem_d, ad, bd, idesc, acc);
      acc = 1u;
    }
  }
}

// ============================================================================= self test
// mode 0: D[128x64] = A[128x64] * W^T      (A K-major, B = W[o][k] K-major)        forward form
// mode 1: D[128x64] = A[128x64] * W        (A K-major, B = W[o][k] MN-major)       data-gradient form
// mode 3: D[ 64x 8] = A^T * ones[128x8]  (column sums; dense no-swizzle B operand)
// mode 2: D[ 64x64] = A^T * G              (A = A[r][c] MN-major (M = c), B = G[r][c] MN-major (N = c), K = 128 rows)
// mode 4 / 5: modes 0 / 1 with the A operand in tensor memory (nb_mma_bf16_ta)
// mode 6 .. 9: modes 0 .. 3 (shared-memory A), timed like 4 / 5
// mode 10: D[64 x 72] = A^T * [G | 1]: the weight-gradient form with the bias column sums folded in as a second MN block
//          of the B operand (N = 72: 64 columns of G, then 8 columns of an all-ones SW128 tile LBO bytes further on);
//          hi*hi + lo*hi with N = 72, hi*lo with N = 64.  Dump: columns 0..63 of the accumulator, then out[8192 + 64 l + c]
//          = columns 64..71 (c < 8) of lane l
// out: raw dump of the 128 TMEM lanes x 64 columns; modes >= 4 append out[8192] = cycles of one 12-MMA group (issue ->
//      commit observed), out[8193] = cycles of four groups issued back to back
__global__ void __launch_bounds__(128) k_tc_selftest(int mode, const float* __restrict__ A, const float* __restrict__ W,
                                                     float* __restrict__ out) {
  NB_PDL_ENTER();
  extern __shared__ __align__(1024) unsigned char tsm[];
  unsigned char* base = (unsigned char*)(((uintptr_t)tsm + 1023) & ~(uintptr_t)1023);
  unsigned char* a_hi = base;
  unsigned char* a_lo = a_hi + NB_TC_TILE_BYTES(128);
  unsigned char* b_hi = a_lo + NB_TC_TILE_BYTES(128);
  unsigned char* b_lo = b_hi + NB_TC_TILE_BYTES(128);
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_base;
  const int tid = threadIdx.x, warp = tid >> 5;
  if (tid == 0) {
    nb_mbar_init(&bar, 1);
    nb_mbar_fence_init();
  }
  if (warp == 0) nb_tmem_alloc(&tmem_base, 128);
  const bool fold = mode == 10;
  if (fold) mode = 2;
  const bool timed = mode >= 4, a_tmem = mode == 4 || mode == 5;
  if (mode >= 6) mode -= 6;
  // operand tiles: this thread owns row `tid`
  {
    const float* ar = A + (size_t)tid * 64;
    for (int j = 0; j < 8; ++j) nb_tc_store8(a_hi, a_lo, tid, j, ar + 8 * j);
    const int brows = (mode == 2) ? 128 : 64;
    if (mode == 3) {  // ones[128][8] bf16
      uint32_t one2 = 0x3F803F80u;
      *reinterpret_cast<uint4*>(b_hi + tid * 16) = make_uint4(one2, one2, one2, one2);
    } else if (tid < brows) {
      const float* wr = W + (size_t)tid * 64;
      for (int j = 0; j < 8; ++j) nb_tc_store8(b_hi, b_lo, tid, j, wr + 8 * j);
    }
  }
  unsigned char* ones_t = b_lo + NB_TC_TILE_BYTES(128);  // mode 10 only (the host sizes shared memory for it)
  if (fold) {
    const uint32_t one2 = 0x3F803F80u;
    for (int c = 0; c < 8; ++c) *reinterpret_cast<uint4*>(ones_t + tid * NB_TC_ROW_BYTES + 16 * c) = make_uint4(one2, one2, one2, one2);
  }
  nb_fence_async_smem();
  nb_tc_fence_before();
  __syncthreads();
  nb_tc_fence_after();
  const uint32_t tm = tmem_base;
  if (fold) {
    if (tid == 0) {
      const uint32_t sah = nb_smem_u32(a_hi), sal = nb_smem_u32(a_lo), sbh = nb_smem_u32(b_hi), sbl = nb_smem_u32(b_lo);
      const uint32_t lbo = nb_smem_u32(ones_t) - sbh;  // second MN block of the B operand: the ones tile
      uint32_t acc = 0;
      for (int pass = 0; pass < 3; ++pass)
        for (int s = 0; s < 8; ++s) {
          const uint64_t ad = nb_desc_mnmajor(pass == 1 ? sal : sah, s);
          const uint64_t bd = pass == 2 ? nb_desc_mnmajor(sbl, s) : nb_make_desc(sbh + 2048 * s, lbo, 1024);
          nb_mma_bf16(tm, ad, bd, pass == 2 ? nb_idesc_bf16(64, 64, 1, 1) : nb_idesc_bf16(64, 72, 1, 1), acc);
          acc = 1;
        }
      nb_mma_commit(&bar);
    }
    nb_mbar_wait(&bar, 0);
    nb_tc_fence_after();
    float v8[4];
    const uint32_t la = tm + ((uint32_t)(warp * 32) << 16);
    for (int h = 0; h < 2; ++h) {
      uint32_t r[4];
      asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(la + 64 + 4 * h) : "memory");
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      for (int i = 0; i < 4; ++i) v8[i] = __uint_as_float(r[i]);
      for (int i = 0; i < 4; ++i) out[8192 + (size_t)tid * 64 + 4 * h + i] = v8[i];
    }
  } else
  if (a_tmem) {  // A row `tid` -> TMEM lane tid, columns [64, 96) hi pieces, [96, 128) lo pieces
    const float* ar = A + (size_t)tid * 64;
    const uint32_t la = tm + ((uint32_t)(warp * 32) << 16);
    for (int ks = 0; ks < 4; ++ks) {  // k-step ks = columns 16 ks .. 16 ks + 15 = 8 packed words
      uint32_t h0[4], l0[4], h1[4], l1[4];
      nb_split8(ar + 16 * ks, h0, l0);
      nb_split8(ar + 16 * ks + 8, h1, l1);
      nb_tmem_st44(la + 64 + 8 * ks, h0, h1);
      nb_tmem_st44(la + 96 + 8 * ks, l0, l1);
    }
    nb_tmem_st_wait();
    nb_tc_fence_before();
    __syncthreads();
    nb_tc_fence_after();
    mode -= 4;
  }
  if (timed) {
    long long c1 = 0, c4 = 0;
    const uint32_t idesc = mode == 0 ? nb_idesc_bf16(128, 64, 0, 0) : nb_idesc_bf16(128, 64, 0, 1);
    const uint32_t sah = nb_smem_u32(a_hi), sal = nb_smem_u32(a_lo), sbh = nb_smem_u32(b_hi), sbl = nb_smem_u32(b_lo);
    uint32_t ph = 0;
    for (int rep = 0; rep < 2; ++rep) {
      const int groups = rep == 0 ? 4 : 1;   // the single group last: its result is the one dumped
      long long t0 = 0;
      if (warp == 0 && nb_elect_one()) {
        t0 = clock64();
        for (int gi = 0; gi < groups; ++gi) {
          uint32_t acc = 0;
          if (mode == 2) {
            nb_tc_issue3(tm, sah, sal, 1, sbh, sbl, 1, 8, nb_idesc_bf16(64, 64, 1, 1), false);
          } else if (mode == 3) {
            for (int pass = 0; pass < 2; ++pass)
              for (int s = 0; s < 8; ++s) {
                nb_mma_bf16(tm, nb_desc_mnmajor(pass ? sal : sah, s), nb_desc_mn8_noswizzle(sbh, s), nb_idesc_bf16(64, 8, 1, 1), acc);
                acc = 1;
              }
          } else
          for (int pass = 0; pass < 3; ++pass)
            for (int s = 0; s < 4; ++s) {
              const uint32_t bt = pass == 2 ? sbl : sbh;
              const uint64_t bd = mode == 0 ? nb_desc_kmajor(bt, s) : nb_desc_mnmajor(bt, s);
              if (a_tmem)
                nb_mma_bf16_ta(tm, tm + (pass == 1 ? 96u : 64u) + 8u * s, (uint32_t)bd, (uint32_t)(bd >> 32), idesc, acc);
              else
                nb_mma_bf16(tm, nb_desc_kmajor(pass == 1 ? sal : sah, s), bd, idesc, acc);
              acc = 1;
            }
        }
        nb_mma_commit(&bar);
      }
      nb_mbar_wait(&bar, ph);
      ph ^= 1;
      nb_tc_fence_after();
      if (tid == 0) {
        const long long dt = clock64() - t0;
        if (rep == 0) c4 = dt; else c1 = dt;
      }
      nb_tc_fence_before();
      __syncthreads();
    }
    if (tid == 0) {
      out[8192] = (float)c1;
      out[8193] = (float)c4;
    }
  } else
  if (tid == 0) {
    if (mode == 0)
      nb_tc_issue3(tm, nb_smem_u32(a_hi), nb_smem_u32(a_lo), 0, nb_smem_u32(b_hi), nb_smem_u32(b_lo), 0, 4,
                   nb_idesc_bf16(128, 64, 0, 0), false);
    else if (mode == 1)
      nb_tc_issue3(tm, nb_smem_u32(a_hi), nb_smem_u32(a_lo), 0, nb_smem_u32(b_hi), nb_smem_u32(b_lo), 1, 4,
                   nb_idesc_bf16(128, 64, 0, 1), false);
    else if (mode == 2)
      nb_tc_issue3(tm, nb_smem_u32(a_hi), nb_smem_u32(a_lo), 1, nb_smem_u32(b_hi), nb_smem_u32(b_lo), 1, 8,
                   nb_idesc_bf16(64, 64, 1, 1), false);
    else {  // mode 3: column sums  D[64 x 8] = A^T * ones[128 x 8]  (ones tile: dense, no swizzle, exact in bf16)
      uint32_t acc = 0;
      for (int pass = 0; pass < 2; ++pass)
        for (int s = 0; s < 8; ++s) {
          nb_mma_bf16(tm, nb_desc_mnmajor(nb_smem_u32(pass ? a_lo : a_hi), s), nb_desc_mn8_noswizzle(nb_smem_u32(b_hi), s),
                      nb_idesc_bf16(64, 8, 1, 1), acc);
          acc = 1;
        }
    }
    nb_mma_commit(&bar);
  }
  if (!timed && !fold) nb_mbar_wait(&bar, 0);
  nb_tc_fence_after();
  float v[32];
  const uint32_t lane_addr = tm + ((uint32_t)(warp * 32) << 16);
  nb_tmem_ld32(lane_addr, v);
  for (int i = 0; i < 32; ++i) out[(size_t)tid * 64 + i] = v[i];
  nb_tmem_ld32(lane_addr + 32, v);
  for (int i = 0; i < 32; ++i) out[(size_t)tid * 64 + 32 + i] = v[i];
  nb_tc_fence_before();
  __syncthreads();
  if (warp == 0) nb_tmem_dealloc(tm, 128);
}
#endif  // NB_EMU
