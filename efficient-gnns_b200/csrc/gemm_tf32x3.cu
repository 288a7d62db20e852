// fp32-faithful dense GEMM on the 5th-gen tensor cores (tcgen05 / TMEM / TMA), sm_100a only.
//
//   C[M,N] = A[M,K] · B[N,K]^T (+ bias[N])          all fp32 in HBM, fp32 accumulation in TMEM
//
// The reference computes its dense contractions (GCNConv's X·W, nn.Linear, the backward dX = dY·W^T;
// arxiv_pyg/gnn.py:47,52 via PyG) in fp32 and the parity bar is 1e-5, which a single TF32 pass (10-bit
// mantissa) cannot meet.  So every product is evaluated with the 3xTF32 split
//        a·b ≈ a_hi·b_hi + a_lo·b_hi + a_hi·b_lo ,   x_hi = x rounded to tf32 (cvt.rna),
//                                                    x_lo = (x - x_hi) rounded to tf32,
// three tcgen05.mma.kind::tf32 instructions per K-step into the same TMEM accumulator.  The dropped terms
// are O(2^-22) relative.  B (the small weight matrix) arrives pre-split from b200gnn_split_tf32_f32; A (the
// big activation matrix) is split on the fly in shared memory, so HBM only ever sees one fp32 copy of it.
//
// Structure (one persistent CTA per SM, 384 threads):
//   warp 0      TMA producer: cp.async.bulk.tensor 128x32 fp32 boxes (128B swizzle) of A, B_hi, B_lo
//   warp 1      MMA issuer  : one elected thread, 12 tcgen05.mma per stage, tcgen05.commit -> mbarriers
//   warp 2      TMEM allocator (256 columns = two 128x128 fp32 accumulators, double buffered)
//   warps 4-7   splitter    : A tile -> (A_hi in place, A_lo) in smem, fence.proxy.async, arrive
//   warps 8-11  epilogue    : tcgen05.ld 32x32b.x32 -> registers -> (+bias) -> 128-bit global stores
// Three pipelines: smem stages (TMA -> split -> MMA -> free), TMEM accumulators (MMA <-> epilogue), tiles.
#include <cuda.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace b200gnn {
namespace gemm {
using namespace tc;

constexpr int BM = 128, BK = 32, UMMA_K = 8;
constexpr int ACC_STAGES = 2;
constexpr int THREADS = 384;
constexpr int TILE_BYTES = BM * BK * 4;                 // 16 KB: one 128 x 32 fp32 A tile
constexpr int BAR_BYTES = 256;
constexpr int EPI_LD = 36;                              // floats per staged row (144 B: 16-byte aligned, conflict-free)
constexpr int EPI_BYTES = 4 * 32 * EPI_LD * 4;          // one 32x32 staging block per epilogue warp
constexpr int STAT_MAX_N = 256;                         // fused column statistics: output width limit
constexpr int STAT_BYTES = 4 * 2 * STAT_MAX_N * 4;      // per epilogue warp: [2][STAT_MAX_N] column accumulators
constexpr int XY_SLOT_BYTES = 2 * 32 * 32 * 4;          // one 32x32 fp32 block of Xout + the same block of Y
constexpr int XY_BYTES = 4 * 2 * XY_SLOT_BYTES;         // 4 epilogue warps x 2 slots (stat_mode 2 with TMA-staged operands)
constexpr int XY_BAR_OFF = 192;                         // byte offset of the 8 Xout/Y mbarriers inside the barrier block

// Tile shape: BN_T output columns per tile (the UMMA N) and the number of smem stages that fit.
//   Wide  <128, 3>: 3 x 64 KB stages, 2 x 128 TMEM columns.
//   Narrow <48, 4>: for N <= 48 (the 40-class logits): the B tiles shrink to 6 KB, one more stage fits (the narrow
//                   GEMM is bound by the DRAM latency of A, so depth is what it needs) and the MMAs do 3/8 of the work.
template <int BN_T, int NSTAGE, int EXTRA = 0>
struct Cfg {
  static constexpr int EXTRA_BYTES = EXTRA;
  static constexpr int BN = BN_T, STAGES = NSTAGE;
  static constexpr int B_TILE_BYTES = BN_T * BK * 4;
  static constexpr int STAGE_BYTES = 2 * TILE_BYTES + 2 * B_TILE_BYTES;          // A_hi, A_lo, B_hi, B_lo
  static constexpr int ACC_HALF = BN_T <= 64 ? 64 : 128;                          // TMEM columns of one accumulator
  // Two accumulators per stage: [0, ACC_HALF) collects a_hi·b_hi, [ACC_HALF, 2·ACC_HALF) the two correction terms.
  // The tensor core ROUNDS ITS fp32 ACCUMULATOR TOWARDS ZERO on every accumulate (tools/probe_accum.py: -2.7e-8 relative
  // per MMA, i.e. -2.6e-6 after the 96 MMAs of a K=256 contraction, against 1e-7 for an fp32 FMA chain); the loss depends
  // on how many times the LARGE accumulator is updated, not on what is added.  Keeping the 2^-11-sized correction terms
  // in their own accumulator takes two of every three updates off the large one; the epilogue adds the pair (RN) once.
  static constexpr int ACC_STRIDE = 2 * ACC_HALF;
  static constexpr int TMEM_COLS = ACC_STAGES * ACC_STRIDE;                       // 256 or 512 (power of two)
  static constexpr int SMEM_BYTES = NSTAGE * STAGE_BYTES + BAR_BYTES + EPI_BYTES + STAT_BYTES + EXTRA + 1024;  // + alignment slack
  static_assert(B_TILE_BYTES % 1024 == 0 && BN_T % 16 == 0 && BN_T <= 256, "tile shape");
  static_assert(SMEM_BYTES <= 232448, "shared memory");
};

// K-major, 128B-swizzled operand tile: rows of 128 B, 8-row groups 1024 B apart.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);        // start address  (bits 0-13)
  d |= (uint64_t)1 << 16;                          // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;                // stride byte offset = 1024 B (bits 32-45)
  d |= (uint64_t)1 << 46;                          // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                          // SWIZZLE_128B
  return d;
}

// tcgen05 instruction descriptor: D=f32, A=B=tf32, both K-major, M=128, N=BN.
template <int BN>
__device__ __forceinline__ uint32_t make_idesc() {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

struct Params {
  float* C;
  const float* bias;
  int64_t ldc;
  int32_t M, N, K;
  int32_t accumulate;   // C += A·B^T (+bias) instead of C = ...
  // Fused R->C layout exchange of the multi-GPU engine (hybrid.py): output columns [q*kc, (q+1)*kc) go to rank q's
  // [N, kc] buffer Cp[q] at rows row_off + m — the epilogue stores straight into the consumers' memory over NVLink
  // (peer mappings), so the exchange costs no kernel of its own and overlaps the GEMM tile by tile.  n_peer = 0: off.
  float* Cp[16];
  int32_t n_peer, kc;
  int64_t row_off;
  int32_t bcast;        // 1: every Cp[q] receives ALL columns at rows row_off + m (fused all-gather of a narrow result)
  // Fused row passes (§8 f1): column reductions over the rows of the OUTPUT, taken in the epilogue while the tile is in
  // registers, so the separate full sweeps over C disappear.  Each epilogue warp keeps [2][N] running column sums in shared
  // memory over all tiles of its CTA and stores them once to stat_partial[(cta*4 + warp)][2][N] (fixed order: deterministic).
  //   stat_mode 1: (sum c, sum c^2) — the BatchNorm batch statistics of the layer output (forward);
  //   stat_mode 2: C is dOut of BN->ReLU->dropout (arxiv_pyg/gnn.py:48-50): the epilogue forms
  //                dz = dOut * [Xout > 0] / (1-p), STORES dz in place of dOut and reduces (sum dz, sum dz*xhat),
  //                xhat = (Y - mean) * invstd — pass 1 of the BatchNorm backward.
  int32_t stat_mode;
  float* stat_partial;
  const float* bn_x;    // Xout [M, ldc]  (post-dropout activation: > 0 <=> ReLU-active and kept)
  const float* bn_y;    // Y    [M, ldc]  (BatchNorm input)
  const float* bn_mean;
  const float* bn_invstd;
  float inv_keep;
};

// stat_mode 2: the pieces of Xout / Y one epilogue lane needs for a 32-column chunk (8 rows x 4 columns: rows it*4 + lane/8
// of the warp's 32-row quarter, columns 4*(lane%8)...) — the same row segments its stores cover.
__device__ __forceinline__ void load_bn_chunk(const Params& p, int tile, int c, int num_n, int BN, int q, int lane,
                                              float4 (&x)[8], float4 (&y)[8]) {
  const int m0 = (tile / num_n) * BM, col = (tile % num_n) * BN + c * 32;
  if (col + 32 > p.N) return;
  const int sub = lane >> 3, cq = (lane & 7) * 4;
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    const int grow = m0 + q * 32 + it * 4 + sub;
    if (grow < p.M) {
      const size_t o = (size_t)grow * p.ldc + col + cq;
      x[it] = __ldg(reinterpret_cast<const float4*>(p.bn_x + o));
      y[it] = __ldg(reinterpret_cast<const float4*>(p.bn_y + o));
    }
  }
}

// STAT: 0 plain, 1 / 2 the fused column reductions (Params::stat_mode); PEER: the output goes to peer buffers (Params::Cp).
// Compile-time so that each instantiation carries only its own epilogue (the epilogue is the hot loop of the narrow-K GEMMs).
template <class C, int STAT, bool PEER>
__global__ void __launch_bounds__(THREADS, 1)
gemm_tf32x3_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmBhi,
                   const __grid_constant__ CUtensorMap tmBlo, const __grid_constant__ CUtensorMap tmX,
                   const __grid_constant__ CUtensorMap tmY, const Params p) {
  constexpr bool BNB = STAT >= 2;        // BatchNorm-backward epilogue; STAT == 3: its Xout / Y blocks arrive by TMA
  constexpr bool XYTMA = STAT == 3;
  constexpr int BN = C::BN, STAGES = C::STAGES, STAGE_BYTES = C::STAGE_BYTES, B_TILE_BYTES = C::B_TILE_BYTES;
  constexpr int TMEM_COLS = C::TMEM_COLS, ACC_STRIDE = C::ACC_STRIDE, ACC_HALF = C::ACC_HALF;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* full = bars;                      // TMA landed            [STAGES]
  uint64_t* split = bars + STAGES;            // A_hi/A_lo written     [STAGES]
  uint64_t* empty = bars + 2 * STAGES;        // MMAs done with stage  [STAGES]
  uint64_t* acc_full = bars + 3 * STAGES;     // accumulator ready     [ACC_STAGES]
  uint64_t* acc_empty = acc_full + ACC_STAGES;  // accumulator drained [ACC_STAGES]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + ACC_STAGES);
  float* epi_smem = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES + BAR_BYTES);
  float* stat_smem = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES + BAR_BYTES + EPI_BYTES);
  uint8_t* xy_smem = smem + STAGES * STAGE_BYTES + BAR_BYTES + EPI_BYTES + STAT_BYTES;
  uint64_t* xy_full = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES + XY_BAR_OFF);   // [4 warps][2 slots]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&split[s], 128); mbar_init(&empty[s], 1); }
    for (int a = 0; a < ACC_STAGES; ++a) { mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], 128); }
    if (XYTMA)
      for (int i = 0; i < 8; ++i) mbar_init(&xy_full[i], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "n"(TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int num_m = (p.M + BM - 1) / BM, num_n = (p.N + BN - 1) / BN;
  const int num_tiles = num_m * num_n;
  const int num_kb = (p.K + BK - 1) / BK;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int s = 0; uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m0 = (tile / num_n) * BM, n0 = (tile % num_n) * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty[s], ph ^ 1);
          uint8_t* st = smem + s * STAGE_BYTES;
          mbar_expect_tx(&full[s], TILE_BYTES + 2 * B_TILE_BYTES);
          tma_load_2d(&tmA, &full[s], st, kb * BK, m0);
          tma_load_2d(&tmBhi, &full[s], st + 2 * TILE_BYTES, kb * BK, n0);
          tma_load_2d(&tmBlo, &full[s], st + 2 * TILE_BYTES + B_TILE_BYTES, kb * BK, n0);
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      const uint32_t idesc = make_idesc<BN>();
      int s = 0; uint32_t ph = 0; int a = 0; uint32_t aph = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        mbar_wait(&acc_empty[a], aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(a * ACC_STRIDE);
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full[s], ph);
          mbar_wait(&split[s], ph);
          tc_fence_after();
          const uint32_t st = smem_u32(smem + s * STAGE_BYTES);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            const uint32_t koff = k * UMMA_K * 4;  // 32 B per K-step inside the 128 B swizzle atom
            const uint64_t a_hi = make_smem_desc(st + koff), a_lo = make_smem_desc(st + TILE_BYTES + koff);
            const uint64_t b_hi = make_smem_desc(st + 2 * TILE_BYTES + koff);
            const uint64_t b_lo = make_smem_desc(st + 2 * TILE_BYTES + B_TILE_BYTES + koff);
            mma_tf32(d_tmem + ACC_HALF, a_lo, b_hi, idesc, (kb | k) != 0);   // correction accumulator
            mma_tf32(d_tmem + ACC_HALF, a_hi, b_lo, idesc, 1);
            mma_tf32(d_tmem, a_hi, b_hi, idesc, (kb | k) != 0);              // main accumulator
          }
          mma_commit(&empty[s]);                       // frees the smem stage once these MMAs retire
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
        mma_commit(&acc_full[a]);                      // accumulator complete -> epilogue
        if (++a == ACC_STAGES) { a = 0; aph ^= 1; }
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ------------------------------------------------------------------ splitter: A -> (A_hi, A_lo)
    const int t = threadIdx.x - 128;
    int s = 0; uint32_t ph = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full[s], ph);
        uint4* hi = reinterpret_cast<uint4*>(smem + s * STAGE_BYTES);
        uint4* lo = reinterpret_cast<uint4*>(smem + s * STAGE_BYTES + TILE_BYTES);
#pragma unroll
        for (int i = 0; i < TILE_BYTES / 16 / 128; ++i) {
          const int o = i * 128 + t;
          const uint4 v = hi[o];
          uint4 h, l;
          split4(v, h, l);
          hi[o] = h;
          lo[o] = l;
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> tensor-core reads
        mbar_arrive(&split[s]);
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp >= 8) {
    // ------------------------------------------------------------------ epilogue
    const int q = warp & 3;                         // TMEM lane quarter this warp may access
    int a = 0; uint32_t aph = 0;
    const bool vec_ok = PEER ? true : ((p.ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 15) == 0));
    float* stat = stat_smem + (warp - 8) * (2 * STAT_MAX_N);     // this warp's [2][N] column accumulators
    if (STAT) {
      for (int i = lane; i < 2 * p.N; i += 32) stat[i] = 0.f;
      __syncwarp();
    }
    constexpr int NCHUNK = (BN + 31) / 32;
    // stat_mode 2 reads Xout and Y next to every output element; neither depends on the accumulator.
    //   STAT == 2: register path — the lane's pieces of a chunk are requested at the top of the chunk (latency overlaps the
    //              wait for the MMAs and the TMEM loads; one chunk = 32 KB per SM in flight, all the registers allow);
    //   STAT == 3: (N % 128 == 0) each warp keeps TWO chunks of Xout / Y in flight in shared memory through TMA
    //              ({32 x 32} boxes, one mbarrier per slot, refilled by lane 0 as soon as the chunk has been consumed):
    //              twice the bytes in flight and no register cost — the narrow-K input-gradient GEMM is bound by exactly that.
    uint8_t* xy = xy_smem + (warp - 8) * (2 * XY_SLOT_BYTES);
    uint64_t* xyb = xy_full + (warp - 8) * 2;
    int n_mine = 0;                                  // chunks this CTA will process (XYTMA: all chunks are whole)
    if (XYTMA) {
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) n_mine += NCHUNK;
      if (lane == 0)
        for (int g = 0; g < 2 && g < n_mine; ++g) {
          const int t = blockIdx.x + (g / NCHUNK) * gridDim.x, cc = g % NCHUNK;
          mbar_expect_tx(&xyb[g], XY_SLOT_BYTES);
          tma_load_2d(&tmX, &xyb[g], xy + g * XY_SLOT_BYTES, (t % num_n) * BN + cc * 32, (t / num_n) * BM + q * 32);
          tma_load_2d(&tmY, &xyb[g], xy + g * XY_SLOT_BYTES + XY_SLOT_BYTES / 2, (t % num_n) * BN + cc * 32, (t / num_n) * BM + q * 32);
        }
    }
    int g_chunk = 0;                                 // running chunk index of this warp (XYTMA slot = g & 1, phase = (g >> 1) & 1)
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int m0 = (tile / num_n) * BM, n0 = (tile % num_n) * BN;
      const int row = m0 + q * 32 + lane;
#pragma unroll 1
      for (int c = 0; c < NCHUNK; ++c, ++g_chunk) { // a partial last chunk reads spare columns of the accumulator's stride
        float4 xr[8], yr[8];
        if (STAT == 2) load_bn_chunk(p, tile, c, num_n, BN, q, lane, xr, yr);
        if (c == 0) {
          mbar_wait(&acc_full[a], aph);
          tc_fence_after();
        }
        uint32_t r[32];
        {
          uint32_t rc[32];
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * ACC_STRIDE + c * 32), r);
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * ACC_STRIDE + ACC_HALF + c * 32), rc);
#pragma unroll
          for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) + __uint_as_float(rc[j]));
        }
        const int col0 = n0 + c * 32;
        if (vec_ok && col0 + 32 <= p.N) {
          // Transpose the warp's 32x32 block through shared memory so that global stores are whole 128-byte row
          // segments (4 rows x 128 B per instruction) instead of 32 scattered 16-byte pieces.
          float* tile = epi_smem + (warp - 8) * (32 * EPI_LD);
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            *reinterpret_cast<float4*>(tile + lane * EPI_LD + j) =
                make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]), __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
          __syncwarp();
          const float* xs = reinterpret_cast<const float*>(xy + (g_chunk & 1) * XY_SLOT_BYTES);   // [32 rows][32 floats]
          const float* ys = xs + 32 * 32;
          if (XYTMA) mbar_wait(&xyb[g_chunk & 1], (uint32_t)((g_chunk >> 1) & 1));
          const int sub = lane >> 3, cq = (lane & 7) * 4;     // 4 rows per instruction, 8 lanes x float4 per row
          float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
          if (p.bias) b4 = make_float4(__ldg(p.bias + col0 + cq), __ldg(p.bias + col0 + cq + 1), __ldg(p.bias + col0 + cq + 2),
                                       __ldg(p.bias + col0 + cq + 3));
          float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f), q4 = s4, mu4 = s4, is4 = s4;
          if (BNB) {
            mu4 = __ldg(reinterpret_cast<const float4*>(p.bn_mean + col0 + cq));
            is4 = __ldg(reinterpret_cast<const float4*>(p.bn_invstd + col0 + cq));
          }
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            const int rr = it * 4 + sub;
            const int grow = m0 + q * 32 + rr;
            float4 v = *reinterpret_cast<const float4*>(tile + rr * EPI_LD + cq);
            v.x += b4.x; v.y += b4.y; v.z += b4.z; v.w += b4.w;
            if (PEER && grow < p.M && p.bcast) {
              for (int q = 0; q < p.n_peer; ++q)
                *reinterpret_cast<float4*>(p.Cp[q] + (size_t)(p.row_off + grow) * p.ldc + col0 + cq) = v;
            } else if (grow < p.M) {
              float4* dst;
              if (PEER) {                           // a 32-column chunk never straddles two ranks (kc % 32 == 0)
                const int q = col0 / p.kc;
                dst = reinterpret_cast<float4*>(p.Cp[q] + (size_t)(p.row_off + grow) * p.kc + (col0 - q * p.kc) + cq);
              } else {
                dst = reinterpret_cast<float4*>(p.C + (size_t)grow * p.ldc + col0 + cq);
              }
              if (!PEER && p.accumulate) { const float4 o = *dst; v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w; }
              if (STAT == 1) {
                vstat(s4, q4, v);
              } else if (BNB) {
                const float4 x = XYTMA ? *reinterpret_cast<const float4*>(xs + rr * 32 + cq) : xr[it];
                const float4 y = XYTMA ? *reinterpret_cast<const float4*>(ys + rr * 32 + cq) : yr[it];
                v.x = x.x > 0.f ? v.x * p.inv_keep : 0.f; v.y = x.y > 0.f ? v.y * p.inv_keep : 0.f;
                v.z = x.z > 0.f ? v.z * p.inv_keep : 0.f; v.w = x.w > 0.f ? v.w * p.inv_keep : 0.f;
                s4.x += v.x; s4.y += v.y; s4.z += v.z; s4.w += v.w;
                q4.x = fmaf(v.x, (y.x - mu4.x) * is4.x, q4.x); q4.y = fmaf(v.y, (y.y - mu4.y) * is4.y, q4.y);
                q4.z = fmaf(v.z, (y.z - mu4.z) * is4.z, q4.z); q4.w = fmaf(v.w, (y.w - mu4.w) * is4.w, q4.w);
              }
              *dst = v;
            }
          }
          if (STAT) {
            // 4 row sub-groups (lane >> 3) hold the same columns: fold them, lanes 0-7 add into the warp's accumulators
#pragma unroll
            for (int d = 8; d <= 16; d <<= 1) {
              s4.x += __shfl_xor_sync(0xffffffffu, s4.x, d); s4.y += __shfl_xor_sync(0xffffffffu, s4.y, d);
              s4.z += __shfl_xor_sync(0xffffffffu, s4.z, d); s4.w += __shfl_xor_sync(0xffffffffu, s4.w, d);
              q4.x += __shfl_xor_sync(0xffffffffu, q4.x, d); q4.y += __shfl_xor_sync(0xffffffffu, q4.y, d);
              q4.z += __shfl_xor_sync(0xffffffffu, q4.z, d); q4.w += __shfl_xor_sync(0xffffffffu, q4.w, d);
            }
            if (lane < 8) {
              float4* ps = reinterpret_cast<float4*>(stat + col0 + cq);
              float4* pq = reinterpret_cast<float4*>(stat + p.N + col0 + cq);
              float4 a0 = *ps, a1 = *pq;
              a0.x += s4.x; a0.y += s4.y; a0.z += s4.z; a0.w += s4.w;
              a1.x += q4.x; a1.y += q4.y; a1.z += q4.z; a1.w += q4.w;
              *ps = a0; *pq = a1;
            }
          }
          __syncwarp();
          if (XYTMA && lane == 0 && g_chunk + 2 < n_mine) {      // the slot has been read by every lane: refill it
            const int g = g_chunk + 2, t = blockIdx.x + (g / NCHUNK) * gridDim.x, cc = g % NCHUNK;
            uint8_t* dst = xy + (g & 1) * XY_SLOT_BYTES;
            mbar_expect_tx(&xyb[g & 1], XY_SLOT_BYTES);
            tma_load_2d(&tmX, &xyb[g & 1], dst, (t % num_n) * BN + cc * 32, (t / num_n) * BM + q * 32);
            tma_load_2d(&tmY, &xyb[g & 1], dst + XY_SLOT_BYTES / 2, (t % num_n) * BN + cc * 32, (t / num_n) * BM + q * 32);
          }
        } else if (PEER && row < p.M && col0 < p.N && p.bcast) {
          for (int q = 0; q < p.n_peer; ++q) {
            float* dst = p.Cp[q] + (size_t)(p.row_off + row) * p.ldc + col0;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (col0 + j < p.N) dst[j] = __uint_as_float(r[j]) + (p.bias ? __ldg(p.bias + col0 + j) : 0.f);
          }
        } else if (row < p.M && col0 < p.N) {
          float* dst = p.C + (size_t)row * p.ldc + col0;
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (col0 + j < p.N) dst[j] = __uint_as_float(r[j]) + (p.bias ? __ldg(p.bias + col0 + j) : 0.f) + (p.accumulate ? dst[j] : 0.f);
        }
      }
      tc_fence_before();
      mbar_arrive(&acc_empty[a]);
      if (++a == ACC_STAGES) { a = 0; aph ^= 1; }
    }
    if (STAT) {
      __syncwarp();
      float* out = p.stat_partial + (size_t)(blockIdx.x * 4 + (warp - 8)) * 2 * p.N;
      for (int i = lane; i < 2 * p.N; i += 32) out[i] = stat[i];
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS));
  }
}

// hi/lo split of a small matrix (weights), optionally transposed: out[c][r] when transpose.
__global__ void __launch_bounds__(256) split_tf32_kernel(const float* __restrict__ W, int64_t rows, int64_t cols,
                                                         int transpose, float* __restrict__ hi, float* __restrict__ lo) {
  const int64_t n = rows * cols;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / cols, c = i - r * cols;
    uint32_t h, l;
    split1(__float_as_uint(W[i]), h, l);
    const int64_t o = transpose ? c * rows + r : i;
    hi[o] = __uint_as_float(h);
    lo[o] = __uint_as_float(l);
  }
}

// [rows, cols] fp32 row-major with leading dimension ld -> boxes of 32 columns x box_rows rows, 128B swizzle, zero OOB fill
static bool make_map(CUtensorMap* m, const float* base, int64_t rows, int64_t cols, int64_t ld, int box_rows, bool swizzle = true) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <class C, int STAT = 0, bool PEER = false>
static int launch(const float* A, int64_t lda, const float* B_hi, const float* B_lo, int64_t ldb, const Params& p,
                  cudaStream_t stream) {
  CUtensorMap tA, tBh, tBl, tX, tY;
  if (!make_map(&tA, A, p.M, p.K, lda, BM) || !make_map(&tBh, B_hi, p.N, p.K, ldb, C::BN) ||
      !make_map(&tBl, B_lo, p.N, p.K, ldb, C::BN))
    return B200GNN_ERR_UNSUPPORTED;
  tX = tA; tY = tA;                                  // placeholders unless the epilogue stages Xout / Y through TMA
  if (STAT == 3 && (!make_map(&tX, p.bn_x, p.M, p.N, p.ldc, 32, false) || !make_map(&tY, p.bn_y, p.M, p.N, p.ldc, 32, false)))
    return B200GNN_ERR_UNSUPPORTED;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  static bool attr_set[64] = {};                    // per device and instantiation; idempotent if two threads race
  if (dev >= 0 && dev < 64 && !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(gemm_tf32x3_kernel<C, STAT, PEER>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES);
    if (e != cudaSuccess) { set_cuda_error(e); return B200GNN_ERR_CUDA; }
    attr_set[dev] = true;
  }
  const int tiles = ((p.M + BM - 1) / BM) * ((p.N + C::BN - 1) / C::BN);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int grid = tiles < sms ? tiles : sms;
  gemm_tf32x3_kernel<C, STAT, PEER><<<grid, THREADS, C::SMEM_BYTES, stream>>>(tA, tBh, tBl, tX, tY, p);
  return check_launch();
}

// ---------------------------------------------------------------------------------------------------------------------
// Grouped form: G row ranges of one A / C pair, each with its own B (and K, bias), in one launch — the per-node-type
// weights of an R-GCN layer.  Same pipeline as gemm_tf32x3_kernel with the plain / bias / accumulate epilogue only; the
// tile scheduler maps a tile to (group, m-tile, n-tile) through the prefix table tile0, so no tile straddles two groups
// and each group's tiles do exactly the arithmetic a launch of the plain kernel on that group would do.  A group with
// K = 0 has no MMAs: its tiles store the bias alone (the caller leaves such groups out in accumulate mode).
// The tensor maps travel in the kernel parameters (~6.6 KB, large kernel parameters), so a launch needs no upload and
// captures into a CUDA graph.
constexpr int MAX_GROUPS = 16;

struct GroupMaps { CUtensorMap a, bhi, blo; };

struct GroupedParams {
  GroupMaps map[MAX_GROUPS];
  const float* bias[MAX_GROUPS];
  int64_t row0[MAX_GROUPS];
  int32_t rows[MAX_GROUPS], K[MAX_GROUPS];
  int32_t tile0[MAX_GROUPS + 1];          // first tile of each group; tile0[n_groups] = total tiles
  float* C;
  int64_t ldc;
  int32_t N, n_groups, accumulate;
};

template <class C>
__global__ void __launch_bounds__(THREADS, 1) gemm_grouped_kernel(const __grid_constant__ GroupedParams p) {
  constexpr int BN = C::BN, STAGES = C::STAGES, STAGE_BYTES = C::STAGE_BYTES, B_TILE_BYTES = C::B_TILE_BYTES;
  constexpr int TMEM_COLS = C::TMEM_COLS, ACC_STRIDE = C::ACC_STRIDE, ACC_HALF = C::ACC_HALF;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* full = bars;
  uint64_t* split = bars + STAGES;
  uint64_t* empty = bars + 2 * STAGES;
  uint64_t* acc_full = bars + 3 * STAGES;
  uint64_t* acc_empty = acc_full + ACC_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + ACC_STAGES);
  float* epi_smem = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES + BAR_BYTES);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&split[s], 128); mbar_init(&empty[s], 1); }
    for (int a = 0; a < ACC_STAGES; ++a) { mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "n"(TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int num_n = (p.N + BN - 1) / BN;
  const int num_tiles = p.tile0[p.n_groups];
  // tile -> (group, first row inside the group, first column)
  auto locate = [&](int tile, int& g, int& m0, int& n0) {
    g = 0;
    while (tile >= p.tile0[g + 1]) ++g;
    const int lt = tile - p.tile0[g];
    m0 = (lt / num_n) * BM;
    n0 = (lt % num_n) * BN;
  };

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int s = 0; uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        int g, m0, n0;
        locate(tile, g, m0, n0);
        const int num_kb = (p.K[g] + BK - 1) / BK;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty[s], ph ^ 1);
          uint8_t* st = smem + s * STAGE_BYTES;
          mbar_expect_tx(&full[s], TILE_BYTES + 2 * B_TILE_BYTES);
          tma_load_2d(&p.map[g].a, &full[s], st, kb * BK, m0);
          tma_load_2d(&p.map[g].bhi, &full[s], st + 2 * TILE_BYTES, kb * BK, n0);
          tma_load_2d(&p.map[g].blo, &full[s], st + 2 * TILE_BYTES + B_TILE_BYTES, kb * BK, n0);
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      const uint32_t idesc = make_idesc<BN>();
      int s = 0; uint32_t ph = 0; int a = 0; uint32_t aph = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        int g, m0, n0;
        locate(tile, g, m0, n0);
        const int num_kb = (p.K[g] + BK - 1) / BK;
        if (num_kb == 0) continue;                     // bias-only tile: no accumulator
        mbar_wait(&acc_empty[a], aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(a * ACC_STRIDE);
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full[s], ph);
          mbar_wait(&split[s], ph);
          tc_fence_after();
          const uint32_t st = smem_u32(smem + s * STAGE_BYTES);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            const uint32_t koff = k * UMMA_K * 4;
            const uint64_t a_hi = make_smem_desc(st + koff), a_lo = make_smem_desc(st + TILE_BYTES + koff);
            const uint64_t b_hi = make_smem_desc(st + 2 * TILE_BYTES + koff);
            const uint64_t b_lo = make_smem_desc(st + 2 * TILE_BYTES + B_TILE_BYTES + koff);
            mma_tf32(d_tmem + ACC_HALF, a_lo, b_hi, idesc, (kb | k) != 0);
            mma_tf32(d_tmem + ACC_HALF, a_hi, b_lo, idesc, 1);
            mma_tf32(d_tmem, a_hi, b_hi, idesc, (kb | k) != 0);
          }
          mma_commit(&empty[s]);
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
        mma_commit(&acc_full[a]);
        if (++a == ACC_STAGES) { a = 0; aph ^= 1; }
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ------------------------------------------------------------------ splitter: A -> (A_hi, A_lo)
    const int t = threadIdx.x - 128;
    int s = 0; uint32_t ph = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      int g, m0, n0;
      locate(tile, g, m0, n0);
      const int num_kb = (p.K[g] + BK - 1) / BK;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full[s], ph);
        uint4* hi = reinterpret_cast<uint4*>(smem + s * STAGE_BYTES);
        uint4* lo = reinterpret_cast<uint4*>(smem + s * STAGE_BYTES + TILE_BYTES);
#pragma unroll
        for (int i = 0; i < TILE_BYTES / 16 / 128; ++i) {
          const int o = i * 128 + t;
          const uint4 v = hi[o];
          uint4 h, l;
          split4(v, h, l);
          hi[o] = h;
          lo[o] = l;
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_arrive(&split[s]);
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp >= 8) {
    // ------------------------------------------------------------------ epilogue (plain / bias / accumulate)
    const int q = warp & 3;
    int a = 0; uint32_t aph = 0;
    const bool vec_ok = (p.ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 15) == 0);
    constexpr int NCHUNK = (BN + 31) / 32;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      int g, m0, n0;
      locate(tile, g, m0, n0);
      const bool mma = p.K[g] > 0;
      const int M = p.rows[g];
      const float* bias = p.bias[g];
      float* Cg = p.C + p.row0[g] * p.ldc;
      const int row = m0 + q * 32 + lane;
#pragma unroll 1
      for (int c = 0; c < NCHUNK; ++c) {
        uint32_t r[32];
        if (mma) {
          if (c == 0) {
            mbar_wait(&acc_full[a], aph);
            tc_fence_after();
          }
          uint32_t rc[32];
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * ACC_STRIDE + c * 32), r);
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * ACC_STRIDE + ACC_HALF + c * 32), rc);
#pragma unroll
          for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) + __uint_as_float(rc[j]));
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) r[j] = 0u;
        }
        const int col0 = n0 + c * 32;
        if (vec_ok && col0 + 32 <= p.N) {
          float* tl = epi_smem + (warp - 8) * (32 * EPI_LD);
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            *reinterpret_cast<float4*>(tl + lane * EPI_LD + j) =
                make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]), __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
          __syncwarp();
          const int sub = lane >> 3, cq = (lane & 7) * 4;
          float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
          if (bias) b4 = make_float4(__ldg(bias + col0 + cq), __ldg(bias + col0 + cq + 1), __ldg(bias + col0 + cq + 2),
                                     __ldg(bias + col0 + cq + 3));
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            const int rr = it * 4 + sub;
            const int grow = m0 + q * 32 + rr;
            float4 v = *reinterpret_cast<const float4*>(tl + rr * EPI_LD + cq);
            v.x += b4.x; v.y += b4.y; v.z += b4.z; v.w += b4.w;
            if (grow < M) {
              float4* dst = reinterpret_cast<float4*>(Cg + (size_t)grow * p.ldc + col0 + cq);
              if (p.accumulate) { const float4 o = *dst; v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w; }
              *dst = v;
            }
          }
          __syncwarp();
        } else if (row < M && col0 < p.N) {
          float* dst = Cg + (size_t)row * p.ldc + col0;
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (col0 + j < p.N) dst[j] = __uint_as_float(r[j]) + (bias ? __ldg(bias + col0 + j) : 0.f) + (p.accumulate ? dst[j] : 0.f);
        }
      }
      if (mma) {
        tc_fence_before();
        mbar_arrive(&acc_empty[a]);
        if (++a == ACC_STAGES) { a = 0; aph ^= 1; }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS));
  }
}

template <class C>
static int launch_grouped(const float* A, int64_t lda, const b200gnn_gemm_group* groups, int32_t n_groups, GroupedParams& p,
                          cudaStream_t stream) {
  const int num_n = (p.N + C::BN - 1) / C::BN;
  int64_t tiles = 0;
  int ng = 0;
  for (int i = 0; i < n_groups; ++i) {
    const b200gnn_gemm_group& gr = groups[i];
    if (gr.rows == 0 || (gr.K == 0 && p.accumulate)) continue;     // nothing to store
    if (gr.K > 0 && (!make_map(&p.map[ng].a, A + gr.row0 * lda, gr.rows, gr.K, lda, BM) ||
                     !make_map(&p.map[ng].bhi, gr.B_hi, p.N, gr.K, gr.ldb, C::BN) ||
                     !make_map(&p.map[ng].blo, gr.B_lo, p.N, gr.K, gr.ldb, C::BN)))
      return B200GNN_ERR_UNSUPPORTED;
    p.bias[ng] = gr.bias; p.row0[ng] = gr.row0; p.rows[ng] = (int32_t)gr.rows; p.K[ng] = (int32_t)gr.K;
    p.tile0[ng] = (int32_t)tiles;
    tiles += ((gr.rows + BM - 1) / BM) * num_n;
    ++ng;
  }
  if (tiles >= INT32_MAX) return B200GNN_ERR_BAD_ARG;
  p.n_groups = ng;
  p.tile0[ng] = (int32_t)tiles;
  if (tiles == 0) return B200GNN_OK;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  static bool attr_set[64] = {};
  if (dev >= 0 && dev < 64 && !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(gemm_grouped_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES);
    if (e != cudaSuccess) { set_cuda_error(e); return B200GNN_ERR_CUDA; }
    attr_set[dev] = true;
  }
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int grid = tiles < sms ? (int)tiles : sms;
  gemm_grouped_kernel<C><<<grid, THREADS, C::SMEM_BYTES, stream>>>(p);
  return check_launch();
}

}  // namespace gemm
}  // namespace b200gnn

using namespace b200gnn;

extern "C" int b200gnn_split_tf32_f32(const float* W, int64_t rows, int64_t cols, int transpose, float* hi, float* lo,
                                      void* stream) {
  if (!W || !hi || !lo || rows <= 0 || cols <= 0) return B200GNN_ERR_BAD_ARG;
  const int64_t n = rows * cols;
  int grid = (int)((n + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  gemm::split_tf32_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(W, rows, cols, transpose, hi, lo);
  return check_launch();
}

static int g_bnbwd_variant = 0;   // A/B knob: 0 automatic, 2 force the register path of the BatchNorm-backward epilogue
extern "C" void b200gnn_gemm_set_bnbwd_variant(int v) { g_bnbwd_variant = v; }

static int gemm_dispatch(const float* A, int64_t lda, const float* B_hi, const float* B_lo, int64_t ldb, float* C, int64_t ldc,
                         int64_t M, int64_t N, int64_t K, const float* bias, int accumulate, void* stream,
                         const gemm::Params* st = nullptr) {
  if (!A || !B_hi || !B_lo || !C || M <= 0 || N <= 0 || K <= 0 || lda < K || ldb < K || ldc < N ||
      M >= INT32_MAX || N >= INT32_MAX || K >= INT32_MAX)
    return B200GNN_ERR_BAD_ARG;
  // TMA: 16-byte aligned bases and row pitches
  if (lda % 4 || ldb % 4 || !aligned_to(A, 16) || !aligned_to(B_hi, 16) || !aligned_to(B_lo, 16))
    return B200GNN_ERR_UNSUPPORTED;
  gemm::Params p{};
  p.C = C; p.bias = bias; p.ldc = ldc; p.M = (int32_t)M; p.N = (int32_t)N; p.K = (int32_t)K; p.accumulate = accumulate ? 1 : 0;
  p.n_peer = 0; p.kc = 0; p.row_off = 0; p.bcast = 0;
  if (st) {
    // fused column statistics: whole 32-column chunks through the vectorised epilogue only
    if (N % 32 || N > gemm::STAT_MAX_N || N <= 48 || ldc % 4 || !aligned_to(C, 16) || !st->stat_partial) return B200GNN_ERR_UNSUPPORTED;
    p.stat_mode = st->stat_mode; p.stat_partial = st->stat_partial; p.bn_x = st->bn_x; p.bn_y = st->bn_y;
    p.bn_mean = st->bn_mean; p.bn_invstd = st->bn_invstd; p.inv_keep = st->inv_keep;
    if (p.stat_mode == 1) return gemm::launch<gemm::Cfg<128, 3>, 1>(A, lda, B_hi, B_lo, ldb, p, (cudaStream_t)stream);
    // BatchNorm-backward epilogue: Xout / Y staged through TMA (two chunks in flight per warp) when every chunk is whole
    if (N % 128 == 0 && g_bnbwd_variant != 2)
      return gemm::launch<gemm::Cfg<128, 2, gemm::XY_BYTES>, 3>(A, lda, B_hi, B_lo, ldb, p, (cudaStream_t)stream);
    return gemm::launch<gemm::Cfg<128, 3>, 2>(A, lda, B_hi, B_lo, ldb, p, (cudaStream_t)stream);
  }
  if (N <= 48) return gemm::launch<gemm::Cfg<48, 4>>(A, lda, B_hi, B_lo, ldb, p, (cudaStream_t)stream);
  return gemm::launch<gemm::Cfg<128, 3>>(A, lda, B_hi, B_lo, ldb, p, (cudaStream_t)stream);
}

// Slots of the statistics partial buffer the fused GEMMs below fill: [slots][2][N] floats.
extern "C" int64_t b200gnn_gemm_stat_slots(int64_t M, int64_t N) {
  if (M <= 0 || N <= 0) return B200GNN_ERR_BAD_ARG;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int64_t tiles = ((M + gemm::BM - 1) / gemm::BM) * ((N + 127) / 128);
  return 4 * (tiles < sms ? tiles : sms);
}

// C = A · B^T + bias (or C += A · B^T when accumulate: the second GEMM of a SAGEConv, lin_l(mean) + lin_r(x)) with the BatchNorm
// batch statistics of the FINAL C taken in the epilogue: partial[slots][2][N] receives per-slot (sum, sum of squares) over the rows — the input of b200gnn_bn_finalize_f32 (replaces b200gnn_col_stats_f32's sweep over C).
extern "C" int b200gnn_gemm_tf32x3_stats_f32(const float* A, int64_t lda, const float* B_hi, const float* B_lo, int64_t ldb,
                                             float* C, int64_t ldc, int64_t M, int64_t N, int64_t K, const float* bias,
                                             int accumulate, float* partial, int64_t slots, void* stream) {
  if (!partial || slots < b200gnn_gemm_stat_slots(M, N) || (accumulate && bias)) return B200GNN_ERR_BAD_ARG;
  gemm::Params st{};
  st.stat_mode = 1; st.stat_partial = partial;
  return gemm_dispatch(A, lda, B_hi, B_lo, ldb, C, ldc, M, N, K, bias, accumulate, stream, &st);
}

// The input-gradient GEMM of a layer that follows BatchNorm -> ReLU -> dropout (arxiv_pyg/gnn.py:48-50), with pass 1 of that
// block's backward in its epilogue:  dOut = A · B^T (+ C when accumulate);  dz = dOut * [Xout > 0] / (1-p) is what is STORED
// to C, and partial[slots][2][N] receives per-slot (sum dz, sum dz * xhat), xhat = (Y - mean) * invstd.  Follow with
// b200gnn_bn_act_bwd_apply_f32(dOut = C, Xout = NULL, ...).  Xout, Y: [M, ldc] like C.
extern "C" int b200gnn_gemm_tf32x3_bnbwd_f32(const float* A, int64_t lda, const float* B_hi, const float* B_lo, int64_t ldb,
                                             float* C, int64_t ldc, int64_t M, int64_t N, int64_t K, int accumulate,
                                             const float* Xout, const float* Y, const float* mean, const float* invstd, float p_drop,
                                             float* partial, int64_t slots, void* stream) {
  if (!partial || !Xout || !Y || !mean || !invstd || p_drop < 0.f || p_drop >= 1.f || slots < b200gnn_gemm_stat_slots(M, N))
    return B200GNN_ERR_BAD_ARG;
  if (!aligned_to(Xout, 16) || !aligned_to(Y, 16) || !aligned_to(mean, 16) || !aligned_to(invstd, 16)) return B200GNN_ERR_UNSUPPORTED;
  gemm::Params st{};
  st.stat_mode = 2; st.stat_partial = partial; st.bn_x = Xout; st.bn_y = Y; st.bn_mean = mean; st.bn_invstd = invstd;
  st.inv_keep = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
  return gemm_dispatch(A, lda, B_hi, B_lo, ldb, C, ldc, M, N, K, nullptr, accumulate, stream, &st);
}

extern "C" int b200gnn_gemm_tf32x3_f32(const float* A, int64_t lda, const float* B_hi, const float* B_lo, int64_t ldb,
                                       float* C, int64_t ldc, int64_t M, int64_t N, int64_t K, const float* bias,
                                       void* stream) {
  return gemm_dispatch(A, lda, B_hi, B_lo, ldb, C, ldc, M, N, K, bias, 0, stream);
}

// C += A · B^T (same kernel; the epilogue adds the tile it is about to overwrite).  Used by the chunked G-CRD backward.
extern "C" int b200gnn_gemm_tf32x3_acc_f32(const float* A, int64_t lda, const float* B_hi, const float* B_lo, int64_t ldb,
                                           float* C, int64_t ldc, int64_t M, int64_t N, int64_t K, void* stream) {
  return gemm_dispatch(A, lda, B_hi, B_lo, ldb, C, ldc, M, N, K, nullptr, 1, stream);
}

// C[row0_g + m, :N] (+)= A[row0_g + m, :K_g] · B_g^T (+ bias_g) for every group g, one launch (see gemm_grouped_kernel).
extern "C" int b200gnn_gemm_tf32x3_grouped_f32(const float* A, int64_t lda, float* C, int64_t ldc, int64_t N,
                                               const b200gnn_gemm_group* groups, int32_t n_groups, int accumulate,
                                               void* stream) {
  if (!A || !C || !groups || n_groups < 0 || n_groups > gemm::MAX_GROUPS || N <= 0 || N >= INT32_MAX || ldc < N || lda <= 0)
    return B200GNN_ERR_BAD_ARG;
  for (int i = 0; i < n_groups; ++i) {
    const b200gnn_gemm_group& g = groups[i];
    if (g.row0 < 0 || g.rows < 0 || g.rows >= INT32_MAX || g.K < 0 || g.K > lda || g.K >= INT32_MAX)
      return B200GNN_ERR_BAD_ARG;
    if (g.K > 0 && (!g.B_hi || !g.B_lo || g.ldb < g.K)) return B200GNN_ERR_BAD_ARG;
    if (g.K % 4 || (g.K > 0 && (g.ldb % 4 || !aligned_to(g.B_hi, 16) || !aligned_to(g.B_lo, 16)))) return B200GNN_ERR_UNSUPPORTED;
  }
  if (lda % 4 || !aligned_to(A, 16)) return B200GNN_ERR_UNSUPPORTED;
  gemm::GroupedParams p{};
  p.C = C; p.ldc = ldc; p.N = (int32_t)N; p.accumulate = accumulate ? 1 : 0;
  if (N <= 48) return gemm::launch_grouped<gemm::Cfg<48, 4>>(A, lda, groups, n_groups, p, (cudaStream_t)stream);
  return gemm::launch_grouped<gemm::Cfg<128, 3>>(A, lda, groups, n_groups, p, (cudaStream_t)stream);
}

// C = A · B^T (+bias) with the output SCATTERED BY COLUMN BLOCK to `world` destination buffers: columns [q*kc, (q+1)*kc)
// -> C_ptrs[q][(row_off + m) * kc + ...] (each an [*, kc] row-major matrix; for the multi-GPU engine these are the ranks'
// C-layout buffers, peer-mapped).  kc = N / world must be a multiple of 32.  C_ptrs: HOST array of `world` device pointers.
extern "C" int b200gnn_gemm_tf32x3_scatter_f32(const float* A, int64_t lda, const float* B_hi, const float* B_lo, int64_t ldb,
                                               float* const* C_ptrs, int32_t world, int64_t row_off, int64_t M, int64_t N, int64_t K,
                                               const float* bias, void* stream) {
  if (!A || !B_hi || !B_lo || !C_ptrs || world <= 0 || world > 16 || M <= 0 || N <= 0 || K <= 0 || lda < K || ldb < K || row_off < 0 ||
      M >= INT32_MAX || N >= INT32_MAX || K >= INT32_MAX)
    return B200GNN_ERR_BAD_ARG;
  if (N % world || (N / world) % 32 || N <= 48) return B200GNN_ERR_UNSUPPORTED;
  if (lda % 4 || ldb % 4 || !aligned_to(A, 16) || !aligned_to(B_hi, 16) || !aligned_to(B_lo, 16)) return B200GNN_ERR_UNSUPPORTED;
  gemm::Params p{};
  p.C = nullptr; p.bias = bias; p.ldc = N; p.M = (int32_t)M; p.N = (int32_t)N; p.K = (int32_t)K; p.accumulate = 0;
  p.n_peer = world; p.kc = (int32_t)(N / world); p.row_off = row_off; p.bcast = 0;
  for (int q = 0; q < world; ++q) {
    if (!C_ptrs[q] || !aligned_to(C_ptrs[q], 16)) return B200GNN_ERR_BAD_ARG;
    p.Cp[q] = C_ptrs[q];
  }
  return gemm::launch<gemm::Cfg<128, 3>, 0, true>(A, lda, B_hi, B_lo, ldb, p, (cudaStream_t)stream);
}

// C = A · B^T (+bias) stored to EVERY destination buffer C_ptrs[q] (row pitch ldc floats) at rows row_off + m: the row
// all-gather of a narrow result (the multi-GPU engine's [N, 40] logits operand) fused into the GEMM epilogue.
extern "C" int b200gnn_gemm_tf32x3_bcast_f32(const float* A, int64_t lda, const float* B_hi, const float* B_lo, int64_t ldb,
                                             float* const* C_ptrs, int32_t world, int64_t row_off, int64_t ldc, int64_t M, int64_t N,
                                             int64_t K, const float* bias, void* stream) {
  if (!A || !B_hi || !B_lo || !C_ptrs || world <= 0 || world > 16 || M <= 0 || N <= 0 || K <= 0 || lda < K || ldb < K || ldc < N ||
      row_off < 0 || M >= INT32_MAX || N >= INT32_MAX || K >= INT32_MAX)
    return B200GNN_ERR_BAD_ARG;
  if (lda % 4 || ldb % 4 || ldc % 4 || !aligned_to(A, 16) || !aligned_to(B_hi, 16) || !aligned_to(B_lo, 16)) return B200GNN_ERR_UNSUPPORTED;
  gemm::Params p{};
  p.C = C_ptrs[0]; p.bias = bias; p.ldc = ldc; p.M = (int32_t)M; p.N = (int32_t)N; p.K = (int32_t)K; p.accumulate = 0;
  p.n_peer = world; p.kc = (int32_t)N; p.row_off = row_off; p.bcast = 1;
  for (int q = 0; q < world; ++q) {
    if (!C_ptrs[q] || !aligned_to(C_ptrs[q], 16)) return B200GNN_ERR_BAD_ARG;
    p.Cp[q] = C_ptrs[q];
  }
  if (N <= 48) return gemm::launch<gemm::Cfg<48, 4>, 0, true>(A, lda, B_hi, B_lo, ldb, p, (cudaStream_t)stream);
  return gemm::launch<gemm::Cfg<128, 3>, 0, true>(A, lda, B_hi, B_lo, ldb, p, (cudaStream_t)stream);
}
