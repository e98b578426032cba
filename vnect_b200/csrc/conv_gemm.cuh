// Implicit-GEMM convolution for sm_100a: TMA (tiled, 5-D, zero OOB fill = SAME padding) -> 128B-swizzled smem
// -> tcgen05.mma (fp16 operands, fp32 accumulators in TMEM) -> fused epilogue (bias / folded BN / residual / ReLU).
//
// GEMM view: D[M = pixels, N = Cout] = A[M, K] * B[N, K]^T with K = taps * Cin. Activations are NHWC fp16, so A is
// K-major straight out of HBM; weights are pre-packed [Cout][tap][Cin] (K-major). One K block = one filter tap x
// BLOCK_K channels = ONE TMA box whose W/H origin is shifted by the tap offset; out-of-image rows/cols are zero
// filled by the TMA unit, which is exactly TF 'SAME' padding for stride-1 convs (SURVEY.md App. A.2).
//
// Every conv of src/vnect_model.py:27-214 (reference) maps onto this one kernel:
//   1x1 convs           flat rows (M = n*H*W), 1 tap
//   3x3 convs           9 taps: halo patches or spatial tiles tw x th (<=128 px) of one image, or flat rows (im2col)
//   4x4/2 transposed    4 output phases, each a 2x2-tap conv (SURVEY.md App. A.2), epilogue scatters to (2y+py, 2x+px)
//
// Warp roles (256 threads, persistent over tiles): warp 0 = TMA producer, warp 1 = MMA issuer (one thread),
// warp 2 = TMEM allocator, warps 4-7 = epilogue (TMEM lane quarter = warp % 4). TMEM accumulators are double
// buffered so the epilogue of tile i overlaps the MMAs of tile i+1.
#pragma once
#include "ptx.cuh"

namespace vnect {

constexpr int kBlockM = 128;
constexpr int kGemmThreads = 256;      // 4 control warps + 4 epilogue warps
constexpr int kGemmThreadsTma = 384;   // TMA epilogues: two epilogue warpgroups working on alternate 64-column chunks
constexpr int kSmemBudget = 227 * 1024;

enum EpiKind : int {
  EPI_PLANAR_F32 = 1,  // fp32 channel-planar [n][c][OH][OW] (heat-map / location-map output, read by the post-process)
  EPI_DECONV_HEAD = 2, // fused res5c head: BN(folded)+ReLU on cols 0-127, deltas on 128-190, bone lengths -> 191-211
  EPI_TMA = 3,         // fp16 NHWC through swizzled smem staging + TMA tensor store (coalesced, clipped), bias (+ReLU)
  EPI_TMA_RES = 4      // same, plus the residual tile prefetched by TMA (warp 3) while the MMAs run
};

constexpr int kEpiChunkBytes = kBlockM * 128;  // one 64-column fp16 chunk of a tile: 128 rows x 128 B
constexpr int kOutStages = 1;   // per epilogue warpgroup (two groups alternate, so each ring needs one slot)
constexpr int kEpiGroups = 2;
constexpr int kResStages = 4;

struct ConvGemmParams {
  // ---- tiling of the GEMM rows
  int mode;  // 0 = flat rows, 1 = spatial tiles
  int M;     // valid rows (flat)
  int NB, H, W;
  int tw, th, tiles_x, tiles_y;
  int num_m_tiles, num_n_tiles;
  int phases;            // 1, or 4 for the transposed conv
  int taps, cblocks;     // K loop = taps * cblocks blocks of BLOCK_K ...
  int cblocks2;          // ... followed by cblocks2 blocks read from a SECOND activation tensor (1x1, same rows):
                         // a projection shortcut folded into the block's last conv as extra K (W = [W_2c | W_1])
  int b_rows_per_phase;  // padded Cout
  signed char tap_dx[16], tap_dy[16];  // [phase * taps + tap]
  uint32_t stage_tx_bytes;
  uint32_t res_tx_bytes;  // bytes of one residual chunk box (EPI_TMA_RES)
  int reverse;            // 1: walk the tiles from last to first.  Consecutive layers alternate, so a layer starts on
                          // the part of its input that the previous layer wrote last and that is still in L2
  int in_stride;          // 1, or 2: the conv samples its input at every second pixel (TMA element strides)
  int res_stride;         // 1, or 2: residual read at every second pixel of a 2H x 2W tensor
  // ---- epilogue
  int n_valid;    // valid output columns
  int relu_cols;  // ReLU on columns < relu_cols (multiple of 32)
  const float* bias;
  void* out;
  int ldc;
  int OH, OW;    // output grid
  int oys, oxs;  // output pixel = (y*oys + py, x*oxs + px)
  int im2col;    // 1: flat-row 3x3 conv whose A operand comes through an im2col tensor map (tap_dx / tap_dy = filter offsets 0..2)
};

// CG = 2: CTA pair (cluster of two SMs) working on one 256-row x BLOCK_N tile with tcgen05.mma.cta_group::2.  Each CTA
// stages its own 128 rows of A and only HALF of the B tile, so the MMA reads (128 + BLOCK_N/2) smem rows per K step
// instead of (128 + BLOCK_N): the single-CTA MMA rate is bound by exactly that operand traffic (~57 B/clk measured).
// BRES: the whole weight matrix of the layer (<= kMaxResidentKBlocks K blocks, one N tile) is loaded into smem once
// per CTA and stays there; the pipeline stages then carry activations only.  For the 64-channel 3x3 convs this cuts
// the L2->SM traffic per tile from 9 x 24 KB to 9 x 16 KB, and those layers are bound by exactly that traffic.
constexpr int kMaxResidentKBlocks = 9;
// HALO (3x3 stride-1 convs at 92x92 / 46x46): instead of one TMA box per filter tap (nine boxes that fetch the same
// pixels nine times: measured 9.5x the input bytes in L2->SM traffic, and as many smem writes competing with the
// MMA's operand reads for the 128 B/clk shared-memory port), ONE (8+2) x (16+2) pixel patch per 64-channel block is
// loaded and all nine taps read it in place: the A descriptor of tap (ky, kx) starts (ky * 10 + kx) pixels = that
// many 128-byte rows into the patch, its 8-row groups are one patch row (10 px = 1280 B) apart.  tcgen05 applies the
// 128B swizzle to absolute smem address bits, so a start that is not 1024-byte aligned and a stride that is not a
// multiple of 1024 read exactly what the TMA wrote (measured: selftest `probe`, base_offset 0, every shift / pitch).
// The weight tiles have their own ring (filled by warp 3) or are resident (BRES); the patch ring reuses the
// residual-prefetch barriers, which a 3x3 conv never needs.
constexpr int kHaloTW = 8, kHaloTH = 16;                  // output tile: 8 x 16 pixels = 128 GEMM rows, m = ly * 8 + lx
constexpr int kHaloPW = kHaloTW + 2, kHaloPH = kHaloTH + 2;
constexpr int kHaloPatchTx = kHaloPW * kHaloPH * 128;      // bytes one patch load delivers (OOB pixels are zero-filled)
constexpr int kHaloABytes = ((kHaloPatchTx + 1023) / 1024) * 1024;
template <int BLOCK_N, int EPI, int CG = 1, bool BRES = false, bool HALO = false>
struct GemmCfg {
  static constexpr int BLOCK_K = 64;  // fp16 elements per 128-byte swizzled smem row
  static constexpr int A_BYTES = kBlockM * 128;
  static constexpr int B_BYTES = (BLOCK_N / CG) * 128;
  // ring stage: A + B tiles; activations only with resident weights; weight tiles only in HALO mode (the patches have
  // their own ring); HALO + BRES streams nothing through it (one dummy stage keeps the barrier arrays non-empty)
  static constexpr int STAGE_BYTES = HALO ? (BRES ? 1024 : B_BYTES) : (BRES ? A_BYTES : A_BYTES + B_BYTES);
  static constexpr int BRES_BYTES = BRES ? kMaxResidentKBlocks * B_BYTES : 0;
  static constexpr int HALO_STAGES = HALO ? (BRES ? 4 : 3) : 0;  // <= kResStages (shares those barriers)
  static constexpr int HALO_BYTES = HALO_STAGES * kHaloABytes;
  static constexpr int EPI_BYTES = (EPI == EPI_TMA)          ? kEpiGroups * kOutStages * kEpiChunkBytes
                                   : (EPI == EPI_TMA_RES)    ? (kEpiGroups * kOutStages + kResStages) * kEpiChunkBytes
                                   : (EPI == EPI_PLANAR_F32) ? BLOCK_N * kBlockM * 4  // [column][row] fp32 transpose tile
                                                             : 0;
  // two epilogue warpgroups: the TMA epilogues (alternate 64-column chunks) and the deconv head (features / deltas)
  static constexpr int THREADS = (EPI == EPI_TMA || EPI == EPI_TMA_RES || EPI == EPI_DECONV_HEAD) ? kGemmThreadsTma : kGemmThreads;
  static constexpr int STAGES_RAW = (kSmemBudget - 1024 - 512 - EPI_BYTES - BRES_BYTES - HALO_BYTES) / STAGE_BYTES;
  static constexpr int STAGES_MAX = HALO ? (BRES ? 1 : 16) : 8;
  static constexpr int STAGES = STAGES_RAW > STAGES_MAX ? STAGES_MAX : STAGES_RAW;
  static constexpr uint32_t TMEM_COLS = (2 * BLOCK_N <= 32)    ? 32
                                        : (2 * BLOCK_N <= 64)  ? 64
                                        : (2 * BLOCK_N <= 128) ? 128
                                        : (2 * BLOCK_N <= 256) ? 256
                                                               : 512;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + BRES_BYTES + HALO_BYTES + EPI_BYTES + 1024 /*align slack*/ + 512 /*barriers*/;
  static_assert(STAGES >= 2 || (HALO && BRES), "pipeline needs at least two stages");
  static_assert(!HALO || EPI == EPI_TMA, "the halo-patch path is the plain 3x3 conv: EPI_TMA");
  static_assert(2 * STAGES + 5 + 2 * kResStages + 2 <= 64, "barriers must fit their 512-byte region");
  static_assert(2 * BLOCK_N <= 512, "two accumulator stages must fit TMEM");
  static_assert(BLOCK_N % 32 == 0 && BLOCK_N >= 32 && BLOCK_N <= 256, "epilogue walks 32-column chunks");
  static_assert(CG == 1 || CG == 2, "a CTA pair at most");
  static_assert(CG == 1 || (BLOCK_N / 2) % 8 == 0, "each CTA of a pair stages whole 8-row swizzle atoms of B");
  static_assert((EPI != EPI_TMA && EPI != EPI_TMA_RES) || BLOCK_N % 64 == 0, "TMA epilogue walks 64-column chunks");
};

__device__ __forceinline__ uint32_t pack_half2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

// fp32 pair -> packed fp16 with ReLU folded into the conversion (lo = a, hi = b)
__device__ __forceinline__ uint32_t pack_half2_relu(float a, float b) {
  uint32_t d;
  asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
  return d;
}

template <int BLOCK_N, int EPI, int CG = 1, bool BRES = false, bool HALO = false>
__global__ void __launch_bounds__((EPI == EPI_TMA || EPI == EPI_TMA_RES || EPI == EPI_DECONV_HEAD) ? kGemmThreadsTma : kGemmThreads, 1)
conv_gemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                 const __grid_constant__ CUtensorMap tmap_out, const __grid_constant__ CUtensorMap tmap_res,
                 const __grid_constant__ CUtensorMap tmap_a2, const __grid_constant__ ConvGemmParams p) {
  using Cfg = GemmCfg<BLOCK_N, EPI, CG, BRES, HALO>;
  static_assert(!BRES || CG == 1, "resident weights are a single-CTA variant");
  constexpr bool kTmaEpi = (EPI == EPI_TMA || EPI == EPI_TMA_RES);
  constexpr int BLOCK_K = Cfg::BLOCK_K;
  constexpr int STAGES = Cfg::STAGES;
  constexpr uint32_t IDESC = make_idesc_f16(kBlockM * CG, BLOCK_N, false);
  // CTA pair: rank 0 leads (issues the MMAs, owns full_bar / tmem_empty); a pair takes GEMM rows 256 at a time
  const int cta_rank = (CG == 2) ? static_cast<int>(cluster_ctarank()) : 0;
  const int worker = blockIdx.x / CG, n_workers = gridDim.x / CG;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* b_res = smem + STAGES * Cfg::STAGE_BYTES;                            // BRES: k_iters x B_BYTES, resident
  uint8_t* halo = b_res + Cfg::BRES_BYTES;                                      // HALO: patch ring, HALO_STAGES x 23 KB
  uint8_t* out_stage = halo + Cfg::HALO_BYTES;                                  // 2 groups x kOutStages x 16 KB
  uint8_t* res_stage = out_stage + kEpiGroups * kOutStages * kEpiChunkBytes;    // kResStages x 16 KB (EPI_TMA_RES)
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES + Cfg::BRES_BYTES + Cfg::HALO_BYTES + Cfg::EPI_BYTES);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + STAGES;
  uint64_t* tmem_full = bars + 2 * STAGES;
  uint64_t* tmem_empty = bars + 2 * STAGES + 2;
  uint64_t* res_full = bars + 2 * STAGES + 4;
  uint64_t* res_empty = bars + 2 * STAGES + 4 + kResStages;
  uint64_t* bres_full = bars + 2 * STAGES + 4 + 2 * kResStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 5 + 2 * kResStages);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    if (p.cblocks2 > 0) tma_prefetch_desc(&tmap_a2);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      // one arrive per epilogue warp that reads the accumulator: both groups when a tile has >= 2 chunks
      mbar_init(&tmem_empty[s], CG * (((kTmaEpi && BLOCK_N >= 128) || EPI == EPI_DECONV_HEAD) ? 8 : 4));
    }
    for (int s = 0; s < kResStages; ++s) {
      mbar_init(&res_full[s], 1);
      mbar_init(&res_empty[s], 1);
    }
    mbar_init(bres_full, 1);
    if constexpr (kTmaEpi) tma_prefetch_desc(&tmap_out);
    if constexpr (EPI == EPI_TMA_RES) tma_prefetch_desc(&tmap_res);
    fence_barrier_init();
  }
  if (warp == 2) {
    if constexpr (CG == 2) tmem_alloc_pair<Cfg::TMEM_COLS>(tmem_slot);
    else tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();  // orders the TMEM allocator's smem write of the base address before everybody's read of it
  if constexpr (CG == 2) cluster_sync_all();  // the peer's barriers must be initialised before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // PDL: everything above (barrier init, descriptor prefetch, TMEM allocation) may overlap the previous layer's tail;
  // from here on this kernel reads what the previous one wrote.
  pdl_launch_dependents();
  pdl_wait();

  const int m_units = (p.num_m_tiles + CG - 1) / CG;  // with an odd tile count the last pair's second half is all
                                                      // out of bounds: zero-filled loads, fully clipped stores
  const int total_tiles = p.phases * m_units * p.num_n_tiles;
  const int k_iters = p.taps * p.cblocks + p.cblocks2;

  // NOTE on the single-lane roles below: the whole warp runs each loop converged and only the issuing instructions are
  // predicated on one elected lane.  Loop state then stays warp-uniform, so ptxas keeps descriptors, coordinates and
  // barrier addresses in uniform registers; with the loop inside `if (elect_one())` every UTMALDG / UTCHMMA needed
  // ~7 R2UR moves and the issue rate, not the tensor pipe, bounded small-N layers.
  if (warp == 0) {
    // ================================================================ TMA producer
    const bool issuer = elect_one();
    {
      if constexpr (BRES) {  // weights are constants: no dependency on the previous layer, but pdl_wait came first anyway
        if (issuer && worker < total_tiles) {
          mbar_arrive_expect_tx(bres_full, static_cast<uint32_t>(k_iters) * Cfg::B_BYTES);
          for (int kb = 0; kb < k_iters; ++kb)
            tma_load_2d(b_res + kb * Cfg::B_BYTES, &tmap_b, bres_full, kb * BLOCK_K, 0);
        }
        __syncwarp();
      }
      int stage = 0;
      uint32_t phase = 0;
      for (int it = worker; it < total_tiles; it += n_workers) {
        const int tile = p.reverse ? total_tiles - 1 - it : it;
        const int n_tile = tile % p.num_n_tiles;
        const int rest = tile / p.num_n_tiles;
        const int m_tile = (rest % m_units) * CG + cta_rank;
        const int ph = rest / m_units;
        int cx, cy, cn;
        if (p.mode == 0) {
          cx = m_tile * kBlockM;
          cy = 0;
          cn = 0;
        } else {
          const int per_img = p.tiles_x * p.tiles_y;
          cn = m_tile / per_img;
          const int t2 = m_tile - cn * per_img;
          cy = (t2 / p.tiles_x) * p.th;
          cx = (t2 % p.tiles_x) * p.tw;
        }
        if constexpr (HALO) {
          // one (8+2) x (16+2) pixel patch per 64-channel block; `stage` / `phase` walk the PATCH ring here
          for (int cb = 0; cb < p.cblocks; ++cb) {
            mbar_wait(&res_empty[stage], phase ^ 1);
            if (issuer) {
              uint8_t* sa = halo + stage * kHaloABytes;
              if constexpr (CG == 2) {
                if (cta_rank == 0) mbar_arrive_expect_tx(&res_full[stage], 2 * kHaloPatchTx);
                tma_load_5d_pair(sa, &tmap_a, &res_full[stage], cb * BLOCK_K, cx - 1, cy - 1, 0, cn);
              } else {
                mbar_arrive_expect_tx(&res_full[stage], kHaloPatchTx);
                tma_load_5d(sa, &tmap_a, &res_full[stage], cb * BLOCK_K, cx - 1, cy - 1, 0, cn);
              }
            }
            __syncwarp();
            if (++stage == Cfg::HALO_STAGES) {
              stage = 0;
              phase ^= 1;
            }
          }
          continue;
        }
        const int b_row = ph * p.b_rows_per_phase + n_tile * BLOCK_N + cta_rank * (BLOCK_N / CG);
        // im2col: the tile is 128 consecutive output pixels of the batch; base pixel of the first one (SAME padding 1)
        int iw = 0, ih = 0, in_ = 0;
        if (p.im2col) {
          const int px0 = m_tile * kBlockM;
          in_ = px0 / (p.H * p.W);
          const int rem = px0 - in_ * p.H * p.W;
          ih = rem / p.W;
          iw = (rem - ih * p.W) * p.in_stride - 1;  // in_stride 2: the conv is evaluated at every second pixel of its input
          ih = ih * p.in_stride - 1;
        }
        for (int t = 0; t < p.taps; ++t) {
          const int ti = ph * p.taps + t;
          const int ax = cx * p.in_stride + p.tap_dx[ti], ay = cy * p.in_stride + p.tap_dy[ti];
          for (int cb = 0; cb < p.cblocks; ++cb) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            if (issuer) {
              uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
              if constexpr (CG == 2) {  // both CTAs' bytes are counted on the leader's barrier
                if (cta_rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * p.stage_tx_bytes);
                if (p.im2col) tma_load_im2col_4d_pair(sa, &tmap_a, &full_bar[stage], cb * BLOCK_K, iw, ih, in_, p.tap_dx[ti], p.tap_dy[ti]);
                else tma_load_5d_pair(sa, &tmap_a, &full_bar[stage], cb * BLOCK_K, ax, ay, 0, cn);
                tma_load_2d_pair(sa + Cfg::A_BYTES, &tmap_b, &full_bar[stage], (t * p.cblocks + cb) * BLOCK_K, b_row);
              } else {
                mbar_arrive_expect_tx(&full_bar[stage], p.stage_tx_bytes);
                if (p.im2col) tma_load_im2col_4d(sa, &tmap_a, &full_bar[stage], cb * BLOCK_K, iw, ih, in_, p.tap_dx[ti], p.tap_dy[ti]);
                else tma_load_5d(sa, &tmap_a, &full_bar[stage], cb * BLOCK_K, ax, ay, 0, cn);
                if constexpr (!BRES)
                  tma_load_2d(sa + Cfg::A_BYTES, &tmap_b, &full_bar[stage], (t * p.cblocks + cb) * BLOCK_K, b_row);
              }
            }
            __syncwarp();
            if (++stage == STAGES) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
        for (int cb = 0; cb < p.cblocks2; ++cb) {  // folded projection shortcut: second A tensor, 1x1
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (issuer) {
            uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
            if constexpr (CG == 2) {
              if (cta_rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * p.stage_tx_bytes);
              tma_load_5d_pair(sa, &tmap_a2, &full_bar[stage], cb * BLOCK_K, cx, cy, 0, cn);
              tma_load_2d_pair(sa + Cfg::A_BYTES, &tmap_b, &full_bar[stage], (p.taps * p.cblocks + cb) * BLOCK_K, b_row);
            } else {
              mbar_arrive_expect_tx(&full_bar[stage], p.stage_tx_bytes);
              tma_load_5d(sa, &tmap_a2, &full_bar[stage], cb * BLOCK_K, cx, cy, 0, cn);
              tma_load_2d(sa + Cfg::A_BYTES, &tmap_b, &full_bar[stage], (p.taps * p.cblocks + cb) * BLOCK_K, b_row);
            }
          }
          __syncwarp();
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
      if constexpr (CG == 2) {
        // drain: the leader's multicast commits still arrive on this CTA's empty barriers after the last load was
        // issued; do not let the CTA retire (and its smem be reused) before every slot has been released
        constexpr int kRing = HALO ? Cfg::HALO_STAGES : STAGES;
        uint64_t* ring_empty = HALO ? res_empty : empty_bar;
        for (int s2 = 0; s2 < kRing; ++s2) {
          mbar_wait(&ring_empty[stage], phase ^ 1);
          if (++stage == kRing) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================================================================ MMA issuer (one elected lane issues)
    const bool issuer = elect_one();
    if (cta_rank == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      [[maybe_unused]] int astage = 0;        // HALO: patch ring position
      [[maybe_unused]] uint32_t aphase = 0;
      if constexpr (BRES) {
        if (worker < total_tiles) mbar_wait(bres_full, 0);
      }
      for (int tile = worker; tile < total_tiles; tile += n_workers) {
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * BLOCK_N);
        if constexpr (HALO) {
          // K order: channel block outermost, then the nine taps of the resident patch (all plans of a layer use this
          // same order, so results do not depend on the plan)
          for (int cb = 0; cb < p.cblocks; ++cb) {
            mbar_wait(&res_full[astage], aphase);
            tc_fence_after();
            const uint32_t patch = smem_u32(halo + astage * kHaloABytes);
#pragma unroll 1
            for (int t = 0; t < 9; ++t) {
              const int ky = t / 3, kx = t - 3 * ky;
              const uint64_t a_desc = make_kmajor_desc_sbo(patch + static_cast<uint32_t>((ky * kHaloPW + kx) * 128), kHaloPW * 128);
              uint64_t b_desc;
              if constexpr (BRES) {
                b_desc = make_kmajor_desc<128>(smem_u32(b_res + (t * p.cblocks + cb) * Cfg::B_BYTES));
              } else {
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                b_desc = make_kmajor_desc<128>(smem_u32(smem + stage * Cfg::STAGE_BYTES));
              }
              if (issuer) {
#pragma unroll
                for (int k = 0; k < BLOCK_K / 16; ++k) {
                  if constexpr (CG == 2) umma_f16_pair(d_tmem, a_desc + 2 * k, b_desc + 2 * k, IDESC, (cb | t | k) != 0 ? 1u : 0u);
                  else umma_f16(d_tmem, a_desc + 2 * k, b_desc + 2 * k, IDESC, (cb | t | k) != 0 ? 1u : 0u);
                }
                if constexpr (!BRES) {
                  if constexpr (CG == 2) umma_commit_pair(&empty_bar[stage]);
                  else umma_commit(&empty_bar[stage]);
                }
              }
              __syncwarp();
              if constexpr (!BRES) {
                if (++stage == STAGES) {
                  stage = 0;
                  phase ^= 1;
                }
              }
            }
            if (issuer) {  // the patch may be overwritten once these MMAs have read it
              if constexpr (CG == 2) umma_commit_pair(&res_empty[astage]);
              else umma_commit(&res_empty[astage]);
            }
            __syncwarp();
            if (++astage == Cfg::HALO_STAGES) {
              astage = 0;
              aphase ^= 1;
            }
          }
        } else
        for (int kb = 0; kb < k_iters; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + stage * Cfg::STAGE_BYTES);
          const uint64_t a_desc = make_kmajor_desc<128>(a_addr);
          const uint64_t b_desc = BRES ? make_kmajor_desc<128>(smem_u32(b_res + kb * Cfg::B_BYTES))
                                       : make_kmajor_desc<128>(a_addr + Cfg::A_BYTES);
          if (issuer) {
#pragma unroll
            for (int k = 0; k < BLOCK_K / 16; ++k) {  // +32 B per K step = +2 in the descriptor's (addr >> 4) field
              if constexpr (CG == 2) umma_f16_pair(d_tmem, a_desc + 2 * k, b_desc + 2 * k, IDESC, (kb | k) != 0 ? 1u : 0u);
              else umma_f16(d_tmem, a_desc + 2 * k, b_desc + 2 * k, IDESC, (kb | k) != 0 ? 1u : 0u);
            }
            // frees the smem slot (in both CTAs of a pair) once these MMAs have read it
            if constexpr (CG == 2) umma_commit_pair(&empty_bar[stage]);
            else umma_commit(&empty_bar[stage]);
          }
          __syncwarp();
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (issuer) {  // accumulator complete -> epilogue (of both CTAs of a pair)
          if constexpr (CG == 2) umma_commit_pair(&tmem_full[acc]);
          else umma_commit(&tmem_full[acc]);
        }
        __syncwarp();
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else if (warp == 3) {
    // ================================================================ HALO: weight-tile producer (its own ring, so the
    // next patch never queues behind nine weight tiles in one warp's program order)
    if constexpr (HALO && !BRES) {
      const bool issuer = elect_one();
      int stage = 0;
      uint32_t phase = 0;
      for (int it = worker; it < total_tiles; it += n_workers) {
        const int tile = p.reverse ? total_tiles - 1 - it : it;
        const int n_tile = tile % p.num_n_tiles;
        const int b_row = n_tile * BLOCK_N + cta_rank * (BLOCK_N / CG);
        for (int cb = 0; cb < p.cblocks; ++cb)
          for (int t = 0; t < 9; ++t) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            if (issuer) {
              uint8_t* sb = smem + stage * Cfg::STAGE_BYTES;
              if constexpr (CG == 2) {
                if (cta_rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * Cfg::B_BYTES);
                tma_load_2d_pair(sb, &tmap_b, &full_bar[stage], (t * p.cblocks + cb) * BLOCK_K, b_row);
              } else {
                mbar_arrive_expect_tx(&full_bar[stage], Cfg::B_BYTES);
                tma_load_2d(sb, &tmap_b, &full_bar[stage], (t * p.cblocks + cb) * BLOCK_K, b_row);
              }
            }
            __syncwarp();
            if (++stage == STAGES) {
              stage = 0;
              phase ^= 1;
            }
          }
      }
      if constexpr (CG == 2) {
        for (int s2 = 0; s2 < STAGES; ++s2) {  // drain, as in the patch producer
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
    // ================================================================ residual prefetcher (EPI_TMA_RES only)
    if constexpr (EPI == EPI_TMA_RES) {
      const bool issuer = elect_one();
      {
        uint32_t ctr = 0;
        for (int it = worker; it < total_tiles; it += n_workers) {
          const int tile = p.reverse ? total_tiles - 1 - it : it;
          const int n_tile = tile % p.num_n_tiles;
          const int m_tile = ((tile / p.num_n_tiles) % m_units) * CG + cta_rank;
          int cx, cy, cn;
          if (p.mode == 0) {
            cx = m_tile * kBlockM; cy = 0; cn = 0;
          } else {
            const int per_img = p.tiles_x * p.tiles_y;
            cn = m_tile / per_img;
            const int t2 = m_tile - cn * per_img;
            cy = (t2 / p.tiles_x) * p.th;
            cx = (t2 % p.tiles_x) * p.tw;
          }
          for (int c0 = 0; c0 < BLOCK_N; c0 += 64, ++ctr) {
            const int rb = ctr % kResStages;
            mbar_wait(&res_empty[rb], ((ctr / kResStages) & 1) ^ 1);
            if (issuer) {
              mbar_arrive_expect_tx(&res_full[rb], p.res_tx_bytes);
              tma_load_5d(res_stage + rb * kEpiChunkBytes, &tmap_res, &res_full[rb], n_tile * BLOCK_N + c0,
                          cx * p.res_stride, cy * p.res_stride, 0, cn);
            }
            __syncwarp();
          }
        }
      }
    }
  } else if (warp >= 4 && kTmaEpi) {
    // ================================================================ epilogue through smem staging + TMA store
    // Two warpgroups (warps 4-7 and 8-11) take alternate 64-column chunks of the global chunk sequence, each with its
    // own staging ring, so one group's TMEM load / barrier / store latencies hide behind the other's arithmetic.
    constexpr int CH = BLOCK_N / 64;  // chunks per tile
    const int grp = (warp - 4) >> 2;
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const bool leader = (threadIdx.x == 128 + grp * 128);
    const uint32_t row_off = static_cast<uint32_t>(r) * 128u;
    const uint32_t sw = static_cast<uint32_t>(r & 7);
    uint8_t* my_out = out_stage + grp * kOutStages * kEpiChunkBytes;
    int acc = 0;
    uint32_t acc_phase = 0, ctr = 0, mine = 0;
    for (int it = worker; it < total_tiles; it += n_workers) {
      const int tile = p.reverse ? total_tiles - 1 - it : it;
      const int n_tile = tile % p.num_n_tiles;
      const int m_tile = ((tile / p.num_n_tiles) % m_units) * CG + cta_rank;
      int cx, cy, cn;
      if (p.mode == 0) {
        cx = m_tile * kBlockM; cy = 0; cn = 0;
      } else {
        const int per_img = p.tiles_x * p.tiles_y;
        cn = m_tile / per_img;
        const int t2 = m_tile - cn * per_img;
        cy = (t2 / p.tiles_x) * p.th;
        cx = (t2 % p.tiles_x) * p.tw;
      }
      const int col_base = n_tile * BLOCK_N;
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(acc * BLOCK_N);
      bool waited = false;
#pragma unroll 1
      for (int c = 0; c < CH; ++c, ++ctr) {
        if ((ctr & 1u) != static_cast<uint32_t>(grp)) continue;
        const int c0 = c * 64;
        if (!waited) {
          mbar_wait(&tmem_full[acc], acc_phase);
          tc_fence_after();
          waited = true;
        }
        // the chunk's 64 bias values, two per lane, requested BEFORE the accumulator is read so that their latency hides
        // behind the TMEM load (a per-use __ldg put ~16 % of the epilogue warps' stall samples on the bias adds)
        float bias_lo = 0.f, bias_hi = 0.f;
        if (p.bias != nullptr) {
          bias_lo = __ldg(p.bias + col_base + c0 + lane);
          bias_hi = __ldg(p.bias + col_base + c0 + 32 + lane);
        }
        uint32_t v[64];
        tmem_ld_32x32(t_row + c0, *reinterpret_cast<uint32_t(*)[32]>(&v[0]));
        tmem_ld_32x32(t_row + c0 + 32, *reinterpret_cast<uint32_t(*)[32]>(&v[32]));
        tmem_ld_wait();
        if (c + 2 >= CH) {  // this group's last chunk of the tile: its share of the accumulator has been read
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if constexpr (CG == 2) mbar_arrive_leader(&tmem_empty[acc]);
            else mbar_arrive(&tmem_empty[acc]);
          }
        }
        const int rb = ctr % kResStages;
        uint8_t* ostage = my_out + (mine % kOutStages) * kEpiChunkBytes;
        ++mine;
        const uint8_t* rstage = res_stage + rb * kEpiChunkBytes;
        if constexpr (EPI == EPI_TMA_RES) mbar_wait(&res_full[rb], (ctr / kResStages) & 1);
        if (leader) bulk_wait_group_read<kOutStages - 1>();  // the store that last used `ostage` has read it
        named_bar_sync(1 + grp, 128);
        const int col0 = col_base + c0;
        const bool relu = col0 < p.relu_cols;
#pragma unroll
        for (int j = 0; j < 8; ++j) {  // 8 x 16 B = this row's 64 output channels
          float f[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) f[e] = __uint_as_float(v[8 * j + e]);
#pragma unroll
          for (int e = 0; e < 8; ++e)  // column 8j+e of the chunk: lane (8j+e) & 31 of the low / high half holds its bias
            f[e] += __shfl_sync(0xffffffffu, j < 4 ? bias_lo : bias_hi, (8 * j + e) & 31);
          const uint32_t off = row_off + ((static_cast<uint32_t>(j) ^ sw) << 4);  // 128B swizzle, as the TMA unit does
          if constexpr (EPI == EPI_TMA_RES) {
            const uint4 rv = *reinterpret_cast<const uint4*>(rstage + off);
            const __half2* h = reinterpret_cast<const __half2*>(&rv);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 t = __half22float2(h[e]);
              f[2 * e] += t.x;
              f[2 * e + 1] += t.y;
            }
          }
          uint4 o;
          if (relu) {
            o.x = pack_half2_relu(f[0], f[1]);
            o.y = pack_half2_relu(f[2], f[3]);
            o.z = pack_half2_relu(f[4], f[5]);
            o.w = pack_half2_relu(f[6], f[7]);
          } else {
            o.x = pack_half2(f[0], f[1]);
            o.y = pack_half2(f[2], f[3]);
            o.z = pack_half2(f[4], f[5]);
            o.w = pack_half2(f[6], f[7]);
          }
          *reinterpret_cast<uint4*>(ostage + off) = o;
        }
        fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the TMA (async proxy)
        named_bar_sync(1 + grp, 128);
        if (leader) {
          tma_store_5d(&tmap_out, ostage, col0, cx, cy, 0, cn);
          bulk_commit_group();
          if constexpr (EPI == EPI_TMA_RES) mbar_arrive(&res_empty[rb]);
        }
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (leader) bulk_wait_group<0>();  // all tensor stores complete before the CTA retires its smem
  } else if (warp >= 4) {
    // ================================================================ epilogue (4 warps = 128 TMEM lanes = 128 rows)
    const int q = warp & 3;
    const int r = q * 32 + lane;  // row of the tile owned by this thread
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int it = worker; it < total_tiles; it += n_workers) {
      const int tile = p.reverse ? total_tiles - 1 - it : it;
      const int n_tile = tile % p.num_n_tiles;
      const int rest = tile / p.num_n_tiles;
      const int m_tile = (rest % m_units) * CG + cta_rank;
      const int ph = rest / m_units;
      bool valid;
      int n, y, x;
      if (p.mode == 0) {
        const int m = m_tile * kBlockM + r;
        valid = m < p.M;
        const int hw = p.H * p.W;
        n = m / hw;
        const int rem = m - n * hw;
        y = rem / p.W;
        x = rem - y * p.W;
      } else {
        const int per_img = p.tiles_x * p.tiles_y;
        n = m_tile / per_img;
        const int t2 = m_tile - n * per_img;
        const int ly = r / p.tw, lx = r - ly * p.tw;
        y = (t2 / p.tiles_x) * p.th + ly;
        x = (t2 % p.tiles_x) * p.tw + lx;
        valid = (ly < p.th) && (y < p.H) && (x < p.W) && (n < p.NB);
      }
      const int oy = y * p.oys + (ph >> 1), ox = x * p.oxs + (ph & 1);
      const size_t pix = (static_cast<size_t>(n) * p.OH + oy) * p.OW + ox;
      const int col_base = n_tile * BLOCK_N;

      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(acc * BLOCK_N);

      float bone[21];
      if constexpr (EPI == EPI_DECONV_HEAD) {
#pragma unroll
        for (int j = 0; j < 21; ++j) bone[j] = 0.f;
      }

      // deconv head: warps 4-7 take the 128 feature columns, warps 8-11 the 63 deltas + bone lengths
      [[maybe_unused]] const int head_grp = (warp - 4) >> 2;
#pragma unroll
      for (int c0 = 0; c0 < BLOCK_N; c0 += 32) {
        if constexpr (EPI == EPI_DECONV_HEAD) {
          if ((c0 >= 128) != (head_grp == 1)) continue;
        }
        uint32_t v[32];
        tmem_ld_32x32(t_row + c0, v);
        tmem_ld_wait();
        const int col0 = col_base + c0;
        float f[32];
        if (p.bias != nullptr) {
          const float4* bp = reinterpret_cast<const float4*>(p.bias + col0);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 b = __ldg(bp + j);
            f[4 * j + 0] = __uint_as_float(v[4 * j + 0]) + b.x;
            f[4 * j + 1] = __uint_as_float(v[4 * j + 1]) + b.y;
            f[4 * j + 2] = __uint_as_float(v[4 * j + 2]) + b.z;
            f[4 * j + 3] = __uint_as_float(v[4 * j + 3]) + b.w;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
        }
        if constexpr (EPI == EPI_PLANAR_F32) {
          // transpose through smem: one scalar store per (thread, plane) straight to HBM kept a single warp per
          // scheduler busy with ~1500 dependent instructions per tile; [column][row] staging, then 16-byte stores
          float* st = reinterpret_cast<float*>(out_stage);
#pragma unroll
          for (int j = 0; j < 32; ++j) st[(c0 + j) * kBlockM + r] = f[j];
        } else {
          if (valid) {
            if (col0 < p.relu_cols) {
#pragma unroll
              for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
            }
            if constexpr (EPI == EPI_DECONV_HEAD) {
              // columns 128..190 are the 63 (dx, dy, dz) deltas; bone_j = sqrt(dx_j^2 + dy_j^2 + dz_j^2)
              // (reference: src/vnect_model.py:198-205)
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const int c = c0 + j;  // compile-time after unrolling (single N tile)
                if (c >= 128 && c < 191) bone[(c - 128) % 21] += f[j] * f[j];
              }
            }
            uint4* op = reinterpret_cast<uint4*>(reinterpret_cast<__half*>(p.out) + pix * p.ldc + col0);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint4 o;
              o.x = pack_half2(f[8 * j + 0], f[8 * j + 1]);
              o.y = pack_half2(f[8 * j + 2], f[8 * j + 3]);
              o.z = pack_half2(f[8 * j + 4], f[8 * j + 5]);
              o.w = pack_half2(f[8 * j + 6], f[8 * j + 7]);
              op[j] = o;
            }
          }
        }
      }
      if constexpr (EPI == EPI_PLANAR_F32) {
        // flat rows only (1x1 conv): row m = n * hw + rem, planes are [n][column][hw]; hw % 4 == 0
        named_bar_sync(1, 128);
        const float* st = reinterpret_cast<const float*>(out_stage);
        float* o = reinterpret_cast<float*>(p.out);
        const int hw = p.H * p.W;
        const int m0 = m_tile * kBlockM + 4 * lane;
        if (m0 < p.M) {
          const int n0 = m0 / hw;
          float* obase = o + static_cast<size_t>(n0) * p.n_valid * hw + (m0 - n0 * hw);
          for (int c = q; c < p.n_valid; c += 4)
            *reinterpret_cast<float4*>(obase + static_cast<size_t>(c) * hw) =
                *reinterpret_cast<const float4*>(st + c * kBlockM + 4 * lane);
        }
        named_bar_sync(1, 128);  // the staging tile may be overwritten by the next tile
      }
      if constexpr (EPI == EPI_DECONV_HEAD) {
        if (valid && head_grp == 1) {
          __half* o = reinterpret_cast<__half*>(p.out) + pix * p.ldc;
          float b[26];
#pragma unroll
          for (int j = 0; j < 21; ++j) b[j] = sqrtf(bone[j]);
          b[21] = b[22] = b[23] = b[24] = b[25] = 0.f;
          o[191] = __float2half_rn(b[0]);  // overwrites the zero pad column written by the generic store above
          uint4* op = reinterpret_cast<uint4*>(o + 192);
#pragma unroll
          for (int j = 0; j < 3; ++j) {
            uint4 w;
            w.x = pack_half2(b[1 + 8 * j + 0], b[1 + 8 * j + 1]);
            w.y = pack_half2(b[1 + 8 * j + 2], b[1 + 8 * j + 3]);
            w.z = pack_half2(b[1 + 8 * j + 4], b[1 + 8 * j + 5]);
            w.w = (j < 2) ? pack_half2(b[1 + 8 * j + 6], b[1 + 8 * j + 7]) : 0u;
            op[j] = w;
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (CG == 2) mbar_arrive_leader(&tmem_empty[acc]);
        else mbar_arrive(&tmem_empty[acc]);
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  }

  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all();  // neither CTA may retire while its partner can still signal it
  else __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    if constexpr (CG == 2) tmem_dealloc_pair<Cfg::TMEM_COLS>(tmem_base);
    else tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

}  // namespace vnect
