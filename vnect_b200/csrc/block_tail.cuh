// Tail of a bottleneck block fused with the head of the next one (reference: src/vnect_model.py:38-51 + 44, 58-66,
// 70-76, ... -- `resNx_branch2c` [+ `branch1`] + add + ReLU, then `resN(x+1)_branch2a` + ReLU):
//
//     X[m, :]  = relu( A[m, :K1] * W^T + bias (+ R[m, :]) )        fp16, written to HBM (the block output)
//     Y[m, :]  = relu( fp16(X[m, :]) * W2^T + bias2 )              fp16, written to HBM (the next block's 1x1 reduce)
//
// Unfused, the reduce conv re-reads X from HBM right after it was written (0.6 ms of a 3.6 ms forward batch, all of it
// HBM-bound at res2 / res3).  Here every 64-channel chunk of X that the epilogue stages in shared memory for its TMA
// store -- a 128B-swizzled [128 px x 64 ch] tile, i.e. exactly one K block of a K-major A operand -- is also fed to
// the tensor cores as the A operand of the second GEMM; W2 streams through its own small ring.  X is read back by
// nobody but the residual / projection path of the next block.
//
// One CTA pair (tcgen05 cta_group::2) owns 256 GEMM rows and walks ALL output-channel tiles of those rows (256 columns
// each), so the second accumulator sees the whole K = Cout.  TMEM: columns [0, 256) main accumulator (single
// buffered), [256, 512) two second accumulators.  K order of the second GEMM is channel order,
// the same as the stand-alone reduce conv, so both plans give bit-identical results.
//
// Scheduling (the first version serialised everything and ran 2x slower than the two kernels it replaces):
//   * every epilogue warpgroup owns TWO staging tiles, so staging chunk c+2 never waits for the second GEMM on chunk c;
//   * the MMA warp issues the second-GEMM work two chunks behind the main GEMM, across tile AND unit boundaries: the
//     main accumulator is refilled as soon as it has been read, while the last two chunks are still being staged;
//   * the second accumulator of a unit is drained after the epilogue has staged its first chunk of the NEXT unit.
//
// Warp roles (384 threads): 0 = TMA producer of the main GEMM (A rows + half of the W tile), 1 = MMA issuer (leader
// CTA), 2 = TMEM allocator, then producer of the W2 tiles, 3 = residual prefetcher, 4-7 / 8-11 = two epilogue
// warpgroups on alternate 64-column chunks (each owns one staging tile).
#pragma once
#include "conv_gemm.cuh"

namespace vnect {

constexpr int kTailBlockN = 256;

struct BlockTailParams {
  ConvGemmParams g;      // rows / tiling / main epilogue (mode, M, tiles, cblocks, cblocks2, bias, relu_cols, strides)
  const float* bias2;    // [N2]
  int n2_k_chunks;       // Cout / 64: K blocks of the second GEMM (= 4 * g.num_n_tiles)
};

template <int N2, bool RES>
struct TailCfg {
  static constexpr int A_BYTES = kBlockM * 128;
  static constexpr int B_BYTES = (kTailBlockN / 2) * 128;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int W2_STAGES = 4;
  static constexpr int W2_BYTES = (N2 / 2) * 128;
  static constexpr int OUT_BUFS = 2;                                   // staging tiles per epilogue group
  static constexpr int OUT_BYTES = kEpiGroups * OUT_BUFS * kEpiChunkBytes;
  static constexpr int RES_STAGES = RES ? 4 : 0;
  static constexpr int RES_BYTES = RES_STAGES * kEpiChunkBytes;
  static constexpr int STAGES_RAW = (kSmemBudget - 1024 - 512 - OUT_BYTES - RES_BYTES - W2_STAGES * W2_BYTES) / STAGE_BYTES;
  static constexpr int STAGES = STAGES_RAW > 6 ? 6 : STAGES_RAW;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + W2_STAGES * W2_BYTES + OUT_BYTES + RES_BYTES + 1024 + 512;
  static_assert(STAGES >= 2, "pipeline needs at least two stages");
  static_assert(N2 == 64 || N2 == 128, "second GEMM width");
  static_assert(kTailBlockN + 2 * N2 <= 512, "accumulators must fit TMEM");
};

template <int N2, bool RES>
__global__ void __launch_bounds__(kGemmThreadsTma, 1)
block_tail_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                  const __grid_constant__ CUtensorMap tmap_out, const __grid_constant__ CUtensorMap tmap_res,
                  const __grid_constant__ CUtensorMap tmap_a2, const __grid_constant__ CUtensorMap tmap_w2,
                  const __grid_constant__ CUtensorMap tmap_out2, const __grid_constant__ BlockTailParams bp) {
  using Cfg = TailCfg<N2, RES>;
  constexpr int STAGES = Cfg::STAGES;
  constexpr int BLOCK_N = kTailBlockN;
  constexpr int BLOCK_K = 64;
  constexpr int CH = BLOCK_N / 64;   // main chunks per output-channel tile
  constexpr int CH2 = N2 / 64;       // chunks of the second accumulator
  constexpr int W2S = Cfg::W2_STAGES;
  constexpr int RS = Cfg::RES_STAGES > 0 ? Cfg::RES_STAGES : 1;
  constexpr int A2 = 2;              // second accumulators (double buffered)
  constexpr uint32_t IDESC = make_idesc_f16(2 * kBlockM, BLOCK_N, false);
  constexpr uint32_t IDESC2 = make_idesc_f16(2 * kBlockM, N2, false);
  const ConvGemmParams& p = bp.g;
  const int cta_rank = static_cast<int>(cluster_ctarank());
  const int worker = blockIdx.x / 2, n_workers = gridDim.x / 2;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* w2_ring = smem + STAGES * Cfg::STAGE_BYTES;
  uint8_t* out_stage = w2_ring + W2S * Cfg::W2_BYTES;      // [group][buffer] x 16 KB
  uint8_t* res_stage = out_stage + Cfg::OUT_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(res_stage + Cfg::RES_BYTES);
  uint64_t* full_bar = bars;                       // [STAGES]
  uint64_t* empty_bar = full_bar + STAGES;         // [STAGES]
  uint64_t* tmem_full = empty_bar + STAGES;        // main accumulator complete
  uint64_t* tmem_empty = tmem_full + 1;            // main accumulator read (8 epilogue warps x 2 CTAs)
  uint64_t* acc2_full = tmem_empty + 1;            // [2]
  uint64_t* acc2_empty = acc2_full + 2;            // [2]
  uint64_t* res_full = acc2_empty + 2;             // [4]
  uint64_t* res_empty = res_full + 4;              // [4]
  uint64_t* w2_full = res_empty + 4;               // [4]
  uint64_t* w2_empty = w2_full + 4;                // [4]
  uint64_t* chunk_ready = w2_empty + 4;            // [group * 2 + buffer]: the staging tile holds a chunk of X (both CTAs)
  uint64_t* chunk_free = chunk_ready + 4;          // [group * 2 + buffer]: the second GEMM has read it
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(chunk_free + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    tma_prefetch_desc(&tmap_out);
    tma_prefetch_desc(&tmap_w2);
    tma_prefetch_desc(&tmap_out2);
    if (p.cblocks2 > 0) tma_prefetch_desc(&tmap_a2);
    if constexpr (RES) tma_prefetch_desc(&tmap_res);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tmem_full, 1);
    mbar_init(tmem_empty, 2 * 8);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&acc2_full[s], 1);
      mbar_init(&acc2_empty[s], 2 * (CH2 >= 2 ? 8 : 4));
    }
    for (int s = 0; s < 4; ++s) {
      mbar_init(&res_full[s], 1);
      mbar_init(&res_empty[s], 1);
      mbar_init(&w2_full[s], 1);
      mbar_init(&w2_empty[s], 1);
      mbar_init(&chunk_ready[s], 2);  // one arrive per CTA of the pair
      mbar_init(&chunk_free[s], 1);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_pair<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();  // orders the TMEM allocator's smem write of the base address before everybody's read of it
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();

  const int m_units = (p.num_m_tiles + 1) / 2;
  const int NT = p.num_n_tiles;
  const int k_iters = p.cblocks + p.cblocks2;
  const int jobs_per_unit = CH * NT;

  auto tile_coords = [&](int unit, int* cx, int* cy, int* cn) {
    const int m_tile = unit * 2 + cta_rank;
    if (p.mode == 0) {
      *cx = m_tile * kBlockM; *cy = 0; *cn = 0;
    } else {
      const int per_img = p.tiles_x * p.tiles_y;
      *cn = m_tile / per_img;
      const int t2 = m_tile - *cn * per_img;
      *cy = (t2 / p.tiles_x) * p.th;
      *cx = (t2 % p.tiles_x) * p.tw;
    }
  };

  if (warp == 0) {
    // ================================================================ main-GEMM producer
    const bool issuer = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    for (int it = worker; it < m_units; it += n_workers) {
      const int unit = p.reverse ? m_units - 1 - it : it;
      int cx, cy, cn;
      tile_coords(unit, &cx, &cy, &cn);
      for (int nt = 0; nt < NT; ++nt) {
        const int b_row = nt * BLOCK_N + cta_rank * (BLOCK_N / 2);
        for (int kb = 0; kb < k_iters; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (issuer) {
            uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
            if (cta_rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * p.stage_tx_bytes);
            if (kb < p.cblocks) tma_load_5d_pair(sa, &tmap_a, &full_bar[stage], kb * BLOCK_K, cx * p.in_stride, cy * p.in_stride, 0, cn);
            else tma_load_5d_pair(sa, &tmap_a2, &full_bar[stage], (kb - p.cblocks) * BLOCK_K, cx, cy, 0, cn);
            tma_load_2d_pair(sa + Cfg::A_BYTES, &tmap_b, &full_bar[stage], kb * BLOCK_K, b_row);
          }
          __syncwarp();
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
    for (int s2 = 0; s2 < STAGES; ++s2) {  // drain: the leader's multicast commits still arrive on our empty barriers
      mbar_wait(&empty_bar[stage], phase ^ 1);
      if (++stage == STAGES) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else if (warp == 1) {
    // ================================================================ MMA issuer (leader CTA)
    const bool issuer = elect_one();
    if (cta_rank == 0) {
      int stage = 0;
      uint32_t phase = 0;
      uint32_t tiles = 0;   // main tiles issued so far
      uint32_t jobs = 0;    // chunks fed to the second GEMM so far (global order: unit, tile, chunk)
      int ws = 0;
      uint32_t wphase = 0;
      // second GEMM on global chunk `jobs`: A = staging tile (group, buffer) of that chunk, B = next W2 tile
      auto chain_one = [&]() {
        const uint32_t s = jobs;
        const uint32_t cu = s / static_cast<uint32_t>(jobs_per_unit);         // unit (local count) of this chunk
        const uint32_t j = s - cu * static_cast<uint32_t>(jobs_per_unit);     // K block of the second GEMM
        const uint32_t g = s & 1u, m = s >> 1, b = m & 1u;                    // group, its main-chunk count, its buffer
        const uint32_t a2 = cu % A2;
        mbar_wait(&w2_full[ws], wphase);
        mbar_wait(&chunk_ready[g * 2 + b], (m >> 1) & 1u);
        if (j == 0) mbar_wait(&acc2_empty[a2], ((cu / A2) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t d_acc2 = tmem_base + BLOCK_N + a2 * N2;
        const uint64_t a_desc = make_kmajor_desc<128>(smem_u32(out_stage + (g * 2 + b) * kEpiChunkBytes));
        const uint64_t b_desc = make_kmajor_desc<128>(smem_u32(w2_ring + ws * Cfg::W2_BYTES));
        if (issuer) {
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_f16_pair(d_acc2, a_desc + 2 * k, b_desc + 2 * k, IDESC2, (j | k) != 0 ? 1u : 0u);
          umma_commit_pair(&w2_empty[ws]);
          umma_commit_pair(&chunk_free[g * 2 + b]);
          if (j + 1 == static_cast<uint32_t>(jobs_per_unit)) umma_commit_pair(&acc2_full[a2]);
        }
        __syncwarp();
        ++jobs;
        if (++ws == W2S) {
          ws = 0;
          wphase ^= 1;
        }
      };
      for (int it = worker; it < m_units; it += n_workers) {
        for (int nt = 0; nt < NT; ++nt) {
          mbar_wait(tmem_empty, (tiles & 1u) ^ 1u);
          tc_fence_after();
          for (int kb = 0; kb < k_iters; ++kb) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            const uint32_t a_addr = smem_u32(smem + stage * Cfg::STAGE_BYTES);
            const uint64_t a_desc = make_kmajor_desc<128>(a_addr);
            const uint64_t b_desc = make_kmajor_desc<128>(a_addr + Cfg::A_BYTES);
            if (issuer) {
#pragma unroll
              for (int k = 0; k < 4; ++k) umma_f16_pair(tmem_base, a_desc + 2 * k, b_desc + 2 * k, IDESC, (kb | k) != 0 ? 1u : 0u);
              umma_commit_pair(&empty_bar[stage]);
            }
            __syncwarp();
            if (++stage == STAGES) {
              stage = 0;
              phase ^= 1;
            }
          }
          if (issuer) umma_commit_pair(tmem_full);
          __syncwarp();
          ++tiles;
          // the second GEMM runs two chunks behind: everything up to chunk 1 of the tile just issued
          while (jobs + 2 < CH * tiles) chain_one();
        }
      }
      while (jobs < CH * tiles) chain_one();
    }
  } else if (warp == 2) {
    // ================================================================ W2 producer ([N2/2 rows of this CTA] x 64 K per chunk)
    const bool issuer = elect_one();
    int ws = 0;
    uint32_t wphase = 0;
    for (int it = worker; it < m_units; it += n_workers) {
      for (int j = 0; j < bp.n2_k_chunks; ++j) {
        mbar_wait(&w2_empty[ws], wphase ^ 1);
        if (issuer) {
          if (cta_rank == 0) mbar_arrive_expect_tx(&w2_full[ws], 2 * Cfg::W2_BYTES);
          tma_load_2d_pair(w2_ring + ws * Cfg::W2_BYTES, &tmap_w2, &w2_full[ws], j * BLOCK_K, cta_rank * (N2 / 2));
        }
        __syncwarp();
        if (++ws == W2S) {
          ws = 0;
          wphase ^= 1;
        }
      }
    }
    for (int s2 = 0; s2 < W2S; ++s2) {  // drain
      mbar_wait(&w2_empty[ws], wphase ^ 1);
      if (++ws == W2S) {
        ws = 0;
        wphase ^= 1;
      }
    }
  } else if (warp == 3) {
    // ================================================================ residual prefetcher
    if constexpr (RES) {
      const bool issuer = elect_one();
      uint32_t ctr = 0;
      for (int it = worker; it < m_units; it += n_workers) {
        const int unit = p.reverse ? m_units - 1 - it : it;
        int cx, cy, cn;
        tile_coords(unit, &cx, &cy, &cn);
        for (int nt = 0; nt < NT; ++nt)
          for (int c0 = 0; c0 < BLOCK_N; c0 += 64, ++ctr) {
            const int rb = ctr % RS;
            mbar_wait(&res_empty[rb], ((ctr / RS) & 1) ^ 1);
            if (issuer) {
              mbar_arrive_expect_tx(&res_full[rb], p.res_tx_bytes);
              tma_load_5d(res_stage + rb * kEpiChunkBytes, &tmap_res, &res_full[rb], nt * BLOCK_N + c0,
                          cx * p.res_stride, cy * p.res_stride, 0, cn);
            }
            __syncwarp();
          }
      }
    }
  } else {
    // ================================================================ epilogue: two warpgroups on alternate chunks
    const int grp = (warp - 4) >> 2;
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const bool leader = (threadIdx.x == 128 + grp * 128);
    const uint32_t row_off = static_cast<uint32_t>(r) * 128u;
    const uint32_t sw = static_cast<uint32_t>(r & 7);
    uint8_t* my_stage = out_stage + grp * Cfg::OUT_BUFS * kEpiChunkBytes;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    uint32_t tiles = 0, res_ctr = 0;
    uint32_t m = 0;                       // main chunks staged by this group so far; chunk m uses buffer m & 1
    // per staging buffer (kept in scalars: indexing small arrays by a run-time buffer number puts them in local memory)
    uint32_t m_last0 = 0, m_last1 = 0;              // last main chunk staged into the buffer ...
    bool chained0 = false, chained1 = false;        // ... and whether its second-GEMM read has not been waited for yet
    uint32_t store_seq = 0, last_store0 = 0, last_store1 = 0;
    bool stored0 = false, stored1 = false;

    // fp32 x 64 (+ bias, + residual) -> relu? -> fp16 into a swizzled staging tile
    // bias_lo / bias_hi: this lane's two of the chunk's 64 bias values (columns lane and 32 + lane), loaded by the caller
    // before the TMEM read so their latency is hidden; distributed by shuffles here
    auto stage_chunk = [&](uint8_t* ostage, const uint32_t (&v)[64], float bias_lo, float bias_hi, bool relu, const uint8_t* rstage) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float f[8];
#pragma unroll
        for (int e = 0; e < 8; ++e)
          f[e] = __uint_as_float(v[8 * j + e]) + __shfl_sync(0xffffffffu, j < 4 ? bias_lo : bias_hi, (8 * j + e) & 31);
        const uint32_t off = row_off + ((static_cast<uint32_t>(j) ^ sw) << 4);
        if (rstage != nullptr) {
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
          o.x = pack_half2_relu(f[0], f[1]); o.y = pack_half2_relu(f[2], f[3]);
          o.z = pack_half2_relu(f[4], f[5]); o.w = pack_half2_relu(f[6], f[7]);
        } else {
          o.x = pack_half2(f[0], f[1]); o.y = pack_half2(f[2], f[3]);
          o.z = pack_half2(f[4], f[5]); o.w = pack_half2(f[6], f[7]);
        }
        *reinterpret_cast<uint4*>(ostage + off) = o;
      }
    };
    // buffer b may be rewritten once the second GEMM has read its last chained content and its last TMA store has
    // read it (the store of the OTHER buffer may still be in flight)
    auto acquire = [&](int b) {
      const bool chained = b ? chained1 : chained0;
      if (chained) {
        mbar_wait(&chunk_free[grp * 2 + b], ((b ? m_last1 : m_last0) >> 1) & 1u);
        if (b) chained1 = false; else chained0 = false;
      }
      if (leader && (b ? stored1 : stored0)) {
        if (store_seq - (b ? last_store1 : last_store0) <= 1) bulk_wait_group_read<0>();
        else bulk_wait_group_read<1>();
      }
      named_bar_sync(1 + grp, 128);
    };
    auto note_store = [&](int b) {
      ++store_seq;
      if (b) { last_store1 = store_seq; stored1 = true; } else { last_store0 = store_seq; stored0 = true; }
    };
    // second accumulator of local unit `du` -> Y (bias2, ReLU), through the staging tile the next main chunk will use
    auto drain_acc2 = [&](uint32_t du, int cx, int cy, int cn) {
      if (grp >= CH2) return;
      const uint32_t a2 = du % A2;
      mbar_wait(&acc2_full[a2], (du / A2) & 1u);
      tc_fence_after();
      const int b = m & 1u;
      uint8_t* ostage = my_stage + b * kEpiChunkBytes;
#pragma unroll 1
      for (int e = grp; e < CH2; e += 2) {
        const float bias_lo = __ldg(bp.bias2 + e * 64 + lane), bias_hi = __ldg(bp.bias2 + e * 64 + 32 + lane);
        uint32_t v[64];
        tmem_ld_32x32(t_lane + BLOCK_N + a2 * N2 + e * 64, *reinterpret_cast<uint32_t(*)[32]>(&v[0]));
        tmem_ld_32x32(t_lane + BLOCK_N + a2 * N2 + e * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&v[32]));
        tmem_ld_wait();
        if (e + 2 >= CH2) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_leader(&acc2_empty[a2]);
        }
        acquire(b);
        stage_chunk(ostage, v, bias_lo, bias_hi, true, nullptr);
        fence_proxy_async_smem();
        named_bar_sync(1 + grp, 128);
        if (leader) {
          tma_store_5d(&tmap_out2, ostage, e * 64, cx, cy, 0, cn);
          bulk_commit_group();
        }
        note_store(b);
      }
    };

    bool drain_due = false;
    uint32_t drain_unit = 0, units = 0;
    int dcx = 0, dcy = 0, dcn = 0;
    for (int it = worker; it < m_units; it += n_workers) {
      const int unit = p.reverse ? m_units - 1 - it : it;
      int cx, cy, cn;
      tile_coords(unit, &cx, &cy, &cn);
      for (int nt = 0; nt < NT; ++nt) {
        mbar_wait(tmem_full, tiles & 1u);
        tc_fence_after();
#pragma unroll 1
        for (int c = grp; c < CH; c += 2) {
          const int c0 = c * 64;
          const int col0 = nt * BLOCK_N + c0;
          float bias_lo = 0.f, bias_hi = 0.f;
          if (p.bias != nullptr) {
            bias_lo = __ldg(p.bias + col0 + lane);
            bias_hi = __ldg(p.bias + col0 + 32 + lane);
          }
          uint32_t v[64];
          tmem_ld_32x32(t_lane + c0, *reinterpret_cast<uint32_t(*)[32]>(&v[0]));
          tmem_ld_32x32(t_lane + c0 + 32, *reinterpret_cast<uint32_t(*)[32]>(&v[32]));
          tmem_ld_wait();
          if (c + 2 >= CH) {  // this group's share of the main accumulator has been read
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_leader(tmem_empty);
          }
          const uint8_t* rstage = nullptr;
          uint32_t rb = 0;
          if constexpr (RES) {
            const uint32_t ctr = res_ctr + static_cast<uint32_t>(c);
            rb = ctr % RS;
            mbar_wait(&res_full[rb], (ctr / RS) & 1);
            rstage = res_stage + rb * kEpiChunkBytes;
          }
          const int b = m & 1u;
          uint8_t* ostage = my_stage + b * kEpiChunkBytes;
          acquire(b);
          stage_chunk(ostage, v, bias_lo, bias_hi, col0 < p.relu_cols, rstage);
          fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the TMA store and to the tensor cores
          named_bar_sync(1 + grp, 128);
          if (leader) {
            tma_store_5d(&tmap_out, ostage, col0, cx, cy, 0, cn);
            bulk_commit_group();
            if constexpr (RES) mbar_arrive(&res_empty[rb]);
            mbar_arrive_leader(&chunk_ready[grp * 2 + b]);  // this CTA's half of the chunk is in place
          }
          note_store(b);
          if (b) { m_last1 = m; chained1 = true; } else { m_last0 = m; chained0 = true; }
          ++m;
          if (drain_due) {  // the previous unit's second accumulator, now that this unit is under way
            drain_acc2(drain_unit, dcx, dcy, dcn);
            drain_due = false;
          }
        }
        res_ctr += CH;
        ++tiles;
      }
      drain_due = true;
      drain_unit = units++;
      dcx = cx; dcy = cy; dcn = cn;
    }
    if (drain_due) drain_acc2(drain_unit, dcx, dcy, dcn);
    if (leader) bulk_wait_group<0>();
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_pair<512>(tmem_base);
  }
}

}  // namespace vnect
