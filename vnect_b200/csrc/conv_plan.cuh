// Host side of the implicit-GEMM convolution: tensor-map construction, tile-shape choice and launch.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdio>
#include <cstring>
#include <string>

#include "conv_gemm.cuh"
#include "block_tail.cuh"
#include "stem_roll.cuh"

namespace vnect {

// ---------------------------------------------------------------------------------------------------------------
// cuTensorMapEncodeTiled is fetched through the runtime so the library has no link-time dependency on libcuda
// (it must dlopen on a CPU-only box for the symbol-export test).
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<PFN_encodeTiled>(p);
  return fn;
}

typedef CUresult (*PFN_encodeIm2col)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                     const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*,
                                     CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                     CUtensorMapFloatOOBfill);

// NHWC fp16 activation [NB, H, W, C] as an im2col tensor map of a 3x3 'SAME' stride-1 conv: a load delivers 128
// consecutive output pixels (walking on across rows and images) x 64 channels at one filter offset, 128B-swizzled.
// Base pixels run over [-1, W - 2] x [-1, H - 2] (lower corner -pad, upper corner pad - (filter - 1)), in steps of
// `stride` (element strides of the map) for a conv evaluated at every stride-th pixel of the [NB, H, W, C] tensor: a
// load still delivers 128 pixels (measured with a probe: W = 14, stride 2 -> 7 pixels per row, then the next row).
inline bool encode_tmap_im2col_3x3(CUtensorMap* m, const void* ptr, int NB, int H, int W, int C, std::string* err, int stride = 1) {
  static PFN_encodeIm2col fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &p, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess) {
      if (err) *err = "cuTensorMapEncodeIm2col entry point unavailable";
      return false;
    }
    fn = reinterpret_cast<PFN_encodeIm2col>(p);
  }
  const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)NB};
  const cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)C * 2 * W, (cuuint64_t)C * 2 * W * H};
  const int lower[2] = {-1, -1}, upper[2] = {-1, -1};
  const cuuint32_t estr[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
  const CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(ptr), dims, strides, lower, upper, 64, kBlockM,
                        estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    if (err) *err = "cuTensorMapEncodeIm2col failed (" + std::to_string((int)r) + ")";
    return false;
  }
  return true;
}

// swz_bytes: 128 (every GEMM operand and output tile) or 0 (the stem's raw strips)
inline bool encode_tmap(CUtensorMap* m, const void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                        const uint32_t* box, int swz_bytes, std::string* err, const uint32_t* elem_strides = nullptr) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) {
    if (err) *err = "cuTensorMapEncodeTiled entry point unavailable";
    return false;
  }
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  if (elem_strides)
    for (int i = 0; i < rank; ++i) estr[i] = elem_strides[i];
  const CUtensorMapSwizzle sw = swz_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, rank, const_cast<void*>(ptr), dims, strides_bytes, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    if (err) {
      char buf[256];
      snprintf(buf, sizeof buf,
               "cuTensorMapEncodeTiled failed (%d): rank %d dims[%llu %llu %llu ...] box[%u %u %u ...] stride0 %llu",
               (int)r, rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
               (unsigned long long)(rank > 2 ? dims[2] : 0), box[0], rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0,
               (unsigned long long)strides_bytes[0]);
      *err = buf;
    }
    return false;
  }
  return true;
}

// ---------------------------------------------------------------------------------------------------------------
enum ConvKind : int { CONV_1x1 = 0, CONV_3x3 = 1, CONV_DECONV4 = 2 };

struct ConvSpec {
  int kind = CONV_1x1;
  int NB = 1, H = 1, W = 1;    // GEMM-row grid (= conv output grid before the phase scatter)
  const __half* in = nullptr;  // NHWC fp16 activation [NB,H,W,cin_pad]
  int cin_pad = 64;            // channels per pixel of `in` (multiple of 64)
  const __half* w = nullptr;  // packed [phases * n_pad][taps * cin_pad] fp16, K-major
  int n_pad = 64;             // padded Cout (multiple of block_n)
  int n_valid = 64;
  int block_n = 64;
  const float* bias = nullptr;  // [n_pad] fp32 or null
  int relu_cols = 0;
  const __half* residual = nullptr;
  int ldr = 0;
  void* out = nullptr;
  int ldc = 0;
  int epi = EPI_TMA;
  // stride-2 sampling (the stride-2 1x1 convs of res3a/res4a only read even pixels of res2c/res3d, so those two
  // blocks are computed at even pixels only): the conv reads `in` [NB, in_stride*H, in_stride*W, cin_pad] at every
  // in_stride-th pixel; the residual is [NB, res_stride*H, res_stride*W, ldr] read likewise. 1x1 convs with a
  // strided operand use spatial tiles.
  int in_stride = 1;
  int res_stride = 1;
  // folded projection shortcut (1x1 convs only): a second activation tensor [NB,H,W,cin2_pad] whose channels extend
  // the K dimension; `w` is then [n_pad][cin_pad + cin2_pad]
  const __half* in2 = nullptr;
  int cin2_pad = 0;
  // fused block tail (block_tail.cuh): this 1x1 conv (+ residual / folded shortcut) also feeds a second 1x1 conv
  // Y = relu(out * W2^T + bias2) of n2 output channels; w2 is [n2][n_pad] fp16 K-major, out2 NHWC [.., n2] on the
  // same pixel grid as `out`.  Needs block_n = 256 (CTA pairs) and n2 = 64 with EPI_TMA or n2 = 128 with EPI_TMA_RES.
  const __half* w2 = nullptr;
  const float* bias2 = nullptr;
  void* out2 = nullptr;
  int n2 = 0;
};

struct ConvLaunch {
  CUtensorMap tmap_a, tmap_b, tmap_out, tmap_res, tmap_a2, tmap_w2, tmap_out2;
  ConvGemmParams p;
  const float* bias2 = nullptr;
  int n2 = 0;  // > 0: fused block tail (block_tail_kernel)
  int block_n = 0, epi = 0, grid = 0, cg = 1, b_resident = 0, halo = 0;
  size_t smem = 0;
  double flops = 0;  // algorithmic: 2 * valid rows * n_valid * taps * real Cin is tracked by the caller; this is GEMM work
};

// persistent grid: one CTA (or CTA pair) per SM (pair of SMs), never more workers than tiles
inline int conv_grid(const ConvGemmParams& p, int cg, int num_sms) {
  const int units = p.phases * ((p.num_m_tiles + cg - 1) / cg) * p.num_n_tiles;
  const int workers = num_sms / cg;
  return cg * (units < workers ? units : workers);
}

// fused block tail: one CTA pair per 256-row unit, walking all output-channel tiles of its rows
inline int tail_grid(const ConvGemmParams& p, int num_sms) {
  const int units = (p.num_m_tiles + 1) / 2;
  const int workers = num_sms / 2;
  return 2 * (units < workers ? units : workers);
}

inline void choose_tile(int H, int W, int* tw_out, int* th_out) {
  int best_tiles = 1 << 30, btw = 1, bth = 1;
  for (int tw = 1; tw <= (W < 128 ? W : 128); ++tw) {
    int th = 128 / tw;
    if (th > H) th = H;
    if (th < 1) continue;
    int tiles = ((W + tw - 1) / tw) * ((H + th - 1) / th);
    if (tiles < best_tiles || (tiles == best_tiles && tw > btw)) {
      best_tiles = tiles;
      btw = tw;
      bth = th;
    }
  }
  *tw_out = btw;
  *th_out = bth;
}

// The halo-patch kernel works on fixed 8 x 16 pixel tiles; use it where that tiling wastes at most ~10 % more GEMM rows
// than the free-form tile (92x92, 46x46, 56x56, 64x64 grids: yes; 23x23 and 28x28: no, those layers are tensor-bound)
inline bool halo_tiling_ok(int H, int W) {
  int tw, th;
  choose_tile(H, W, &tw, &th);
  const int free_tiles = ((W + tw - 1) / tw) * ((H + th - 1) / th);
  const int halo_tiles = ((W + kHaloTW - 1) / kHaloTW) * ((H + kHaloTH - 1) / kHaloTH);
  return halo_tiles * 10 <= free_tiles * 11;
}

// How a conv runs, from its shape, output tile width and epilogue.  build_conv applies these rules to every conv, so
// the library and the self-test build exactly the configurations that have a kernel.
struct ConvPath {
  // CTA pairs (tcgen05 cta_group::2) pay off where the MMA's smem operand reads are the limit: N >= 128 tiles
  // (measured 5-8 % on the tensor-bound layers, nothing at N = 64)
  int cg;
  // 64-channel convs whose whole weight matrix fits kMaxResidentKBlocks K blocks keep it resident in smem: the 3x3s of
  // res2 are bound by L2->SM traffic (158 -> 135 us), the 1x1 256->64 convs gain a few percent.  Those 3x3s run on
  // spatial tiles, one shifted box per tap, where the halo tiling does not apply (stride 2, small grids).
  int b_resident;
  // stride-1 3x3 convs on the larger grids read one halo patch per channel block instead of nine shifted boxes
  // (conv_gemm.cuh HALO)
  int halo;
  // the other 3x3 convs (23 x 23 at box size 368: five 23 x 5 tiles fill 529 of 640 GEMM rows; stride-2 ones included,
  // res3d's 3x3 at 46 -> 23: 31 -> 27 us) and the transposed conv (114 -> 103 us per 128 forwards) run on flat pixel
  // rows through an im2col tensor map: every row of a 128-row tile is a real pixel.  Same K order, so the same results.
  int im2col;
};

inline ConvPath conv_path(const ConvSpec& s) {
  ConvPath r;
  r.cg = s.block_n >= 128 ? 2 : 1;
  const int taps = s.kind == CONV_3x3 ? 9 : 1;
  r.b_resident = s.kind != CONV_DECONV4 && s.block_n == 64 && s.n_pad == 64 && s.epi == EPI_TMA && !s.in2 &&
                 taps * s.cin_pad / 64 <= kMaxResidentKBlocks;
  r.halo = s.kind == CONV_3x3 && s.in_stride == 1 && s.epi == EPI_TMA && s.block_n <= 128 && halo_tiling_ok(s.H, s.W);
  r.im2col = s.kind == CONV_DECONV4 || (s.kind == CONV_3x3 && !r.halo && !r.b_resident);
  return r;
}

// cudaFuncSetAttribute is per device (context): remember, per kernel instantiation, which devices of this process
// already carry the opt-in.  One bit per device ordinal; a process holds at most one handle per GPU of an 8-GPU box.
template <typename Kern>
inline cudaError_t ensure_dyn_smem(Kern kern, int bytes, unsigned long long* done_mask) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const unsigned long long bit = 1ull << (dev & 63);
  if (__atomic_load_n(done_mask, __ATOMIC_ACQUIRE) & bit) return cudaSuccess;
  e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) return e;
  __atomic_fetch_or(done_mask, bit, __ATOMIC_RELEASE);
  return cudaSuccess;
}

// One conv_gemm_kernel instantiation with its launch shape
typedef void (*ConvKernelFn)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, ConvGemmParams);
struct ConvKernel {
  ConvKernelFn fn = nullptr;
  int threads = 0, smem = 0, cg = 1;
  unsigned long long* smem_done = nullptr;  // ensure_dyn_smem's device mask of this instantiation
};

template <int BLOCK_N, int EPI, int CG, bool BRES = false, bool HALO = false>
inline ConvKernel conv_kernel() {
  using Cfg = GemmCfg<BLOCK_N, EPI, CG, BRES, HALO>;
  static unsigned long long done = 0;
  return {conv_gemm_kernel<BLOCK_N, EPI, CG, BRES, HALO>, Cfg::THREADS, Cfg::SMEM_BYTES, CG, &done};
}

// The instantiations the plans launch (see conv_path); any other combination has no kernel (fn == nullptr)
inline ConvKernel find_conv_kernel(const ConvLaunch& L) {
  const int bn = L.block_n, epi = L.epi, cg = L.cg;
  if (epi == EPI_TMA && cg == 1 && bn == 64) {
    if (L.halo) return L.b_resident ? conv_kernel<64, EPI_TMA, 1, true, true>() : conv_kernel<64, EPI_TMA, 1, false, true>();
    return L.b_resident ? conv_kernel<64, EPI_TMA, 1, true>() : conv_kernel<64, EPI_TMA, 1>();
  }
  if (L.b_resident) return {};
  if (epi == EPI_TMA && cg == 2 && bn == 128) return L.halo ? conv_kernel<128, EPI_TMA, 2, false, true>() : conv_kernel<128, EPI_TMA, 2>();
  if (L.halo) return {};
  if (epi == EPI_TMA && cg == 2 && bn == 256) return conv_kernel<256, EPI_TMA, 2>();
  if (epi == EPI_TMA_RES && cg == 1 && bn == 64) return conv_kernel<64, EPI_TMA_RES, 1>();
  if (epi == EPI_TMA_RES && cg == 2 && bn == 256) return conv_kernel<256, EPI_TMA_RES, 2>();
  if (epi == EPI_PLANAR_F32 && cg == 1 && bn == 96) return conv_kernel<96, EPI_PLANAR_F32, 1>();
  if (epi == EPI_DECONV_HEAD && cg == 2 && bn == 192) return conv_kernel<192, EPI_DECONV_HEAD, 2>();
  return {};
}

// fused block tails: a 64-wide second conv after a folded projection, a 128-wide one after a residual add
inline bool tail_supported(int n2, int epi) { return (n2 == 64 && epi == EPI_TMA) || (n2 == 128 && epi == EPI_TMA_RES); }

inline bool build_conv(const ConvSpec& s, int num_sms, ConvLaunch* L, std::string* err) {
  memset(L, 0, sizeof(*L));
  ConvGemmParams& p = L->p;
  constexpr int block_k = 64;
  const ConvPath path = conv_path(s);
  L->block_n = s.block_n;
  L->epi = s.epi;
  L->cg = path.cg;
  L->b_resident = path.b_resident;
  L->halo = path.halo;
  if (s.cin_pad % 64 != 0 || s.cin2_pad % 64 != 0) {
    if (err) *err = "input channels must be padded to multiples of 64";
    return false;
  }
  if (s.n_pad % s.block_n != 0) {
    if (err) *err = "n_pad must be a multiple of block_n";
    return false;
  }
  if (s.kind == CONV_DECONV4 && s.in_stride != 1) {
    if (err) *err = "the transposed conv reads every input pixel";
    return false;
  }
  p.NB = s.NB;
  p.H = s.H;
  p.W = s.W;
  p.M = s.NB * s.H * s.W;
  p.phases = 1;
  p.b_rows_per_phase = s.n_pad;
  p.num_n_tiles = s.n_pad / s.block_n;
  p.n_valid = s.n_valid;
  p.relu_cols = s.relu_cols;
  p.bias = s.bias;
  p.out = s.out;
  p.ldc = s.ldc;
  p.OH = s.H;
  p.OW = s.W;
  p.oys = p.oxs = 1;
  p.in_stride = s.in_stride;
  p.res_stride = s.res_stride;
  const bool spatial1 = s.kind == CONV_1x1 && (s.in_stride != 1 || s.res_stride != 1);
  uint32_t estr[5] = {1, (uint32_t)s.in_stride, (uint32_t)s.in_stride, 1, 1};

  uint64_t dims[5], strides[4];
  uint32_t box[5];
  int k_total;
  if ((s.kind == CONV_1x1 && !spatial1) || path.im2col) {  // flat pixel rows
    p.mode = 0;
    p.cblocks = s.cin_pad / block_k;
    p.num_m_tiles = (p.M + kBlockM - 1) / kBlockM;
    p.tw = kBlockM;
    p.th = 1;
    p.tiles_x = p.tiles_y = 1;
    // for im2col, dims / box describe the A tile for the byte count below; the map is built by encode_tmap_im2col_3x3
    dims[0] = s.cin_pad; dims[1] = p.M; dims[2] = 1; dims[3] = 1; dims[4] = 1;
    strides[0] = (uint64_t)s.cin_pad * 2;
    strides[1] = strides[2] = strides[3] = (uint64_t)s.cin_pad * 2 * p.M;
    box[0] = block_k; box[1] = kBlockM; box[2] = 1; box[3] = 1; box[4] = 1;
    if (s.kind == CONV_1x1) {
      p.taps = 1;
      p.cblocks2 = s.cin2_pad / block_k;
    } else if (s.kind == CONV_3x3) {
      p.im2col = 1;
      p.taps = 9;
      for (int ky = 0; ky < 3; ++ky)
        for (int kx = 0; kx < 3; ++kx) {  // filter offsets from the base pixel, not displacements from the output pixel
          p.tap_dy[ky * 3 + kx] = (signed char)ky;
          p.tap_dx[ky * 3 + kx] = (signed char)kx;
        }
    } else {
      // 4x4 stride-2 'SAME' transposed conv: output (2j+py, 2i+px); per axis, phase 0 uses kernel taps {1,3} at
      // input offsets {0,-1}, phase 1 uses taps {0,2} at offsets {+1,0} (SURVEY.md App. A.2): each phase is a 2x2-tap
      // conv inside the same 3x3 neighbourhood. Tap order here must match pack_deconv_weights(): tap = a*2 + b with a
      // the row choice, b the column choice.
      p.im2col = 1;
      p.taps = 4;
      p.phases = 4;
      p.oys = p.oxs = 2;
      p.OH = 2 * s.H;
      p.OW = 2 * s.W;
      for (int ph = 0; ph < 4; ++ph) {
        const int py = ph >> 1, px = ph & 1;
        for (int a = 0; a < 2; ++a)
          for (int b = 0; b < 2; ++b) {
            const int dy = py == 0 ? (a == 0 ? 0 : -1) : (a == 0 ? 1 : 0);
            const int dx = px == 0 ? (b == 0 ? 0 : -1) : (b == 0 ? 1 : 0);
            p.tap_dy[ph * 4 + a * 2 + b] = (signed char)(dy + 1);
            p.tap_dx[ph * 4 + a * 2 + b] = (signed char)(dx + 1);
          }
      }
    }
    k_total = p.taps * s.cin_pad + s.cin2_pad;
  } else {  // spatial tiles: halo-patch or resident-weight 3x3 convs, 1x1 convs with a strided operand
    p.mode = 1;
    if (path.halo) {
      p.tw = kHaloTW;
      p.th = kHaloTH;
    } else {
      choose_tile(s.H, s.W, &p.tw, &p.th);
    }
    p.tiles_x = (s.W + p.tw - 1) / p.tw;
    p.tiles_y = (s.H + p.th - 1) / p.th;
    p.num_m_tiles = s.NB * p.tiles_x * p.tiles_y;
    p.cblocks = s.cin_pad / block_k;
    if (spatial1) {
      p.taps = 1;
      p.tap_dx[0] = p.tap_dy[0] = 0;
    } else {
      p.taps = 9;
      for (int ky = 0; ky < 3; ++ky)
        for (int kx = 0; kx < 3; ++kx) {
          p.tap_dy[ky * 3 + kx] = (signed char)(ky - 1);
          p.tap_dx[ky * 3 + kx] = (signed char)(kx - 1);
        }
    }
    dims[0] = s.cin_pad; dims[1] = (uint64_t)s.W * s.in_stride; dims[2] = (uint64_t)s.H * s.in_stride; dims[3] = 1; dims[4] = s.NB;
    strides[0] = (uint64_t)s.cin_pad * 2;
    strides[1] = strides[0] * dims[1];
    strides[2] = strides[1] * dims[2];
    strides[3] = strides[2];
    box[0] = block_k; box[1] = p.tw * s.in_stride; box[2] = p.th * s.in_stride; box[3] = 1; box[4] = 1;
    if (path.halo) {  // the A box is the whole patch: tile + one pixel of halo on every side
      box[1] = kHaloPW;
      box[2] = kHaloPH;
    }
    k_total = p.taps * s.cin_pad;
  }
  const int a_stride = p.im2col ? 1 : s.in_stride;  // an im2col load is 128 pixels whatever the stride
  // per CTA: its A rows plus its share of the B tile (half of it in a CTA pair; nothing when the weights are resident)
  p.stage_tx_bytes = (uint32_t)(box[0] * (box[1] / a_stride) * (box[2] / a_stride) * 2 +
                                (path.b_resident ? 0u : (uint32_t)(s.block_n / path.cg) * block_k * 2));
  if (path.halo) p.stage_tx_bytes = 0;  // patch / weight-tile byte counts are compile-time constants of the HALO kernel
  if (p.im2col) {
    if (!encode_tmap_im2col_3x3(&L->tmap_a, s.in, s.NB, s.H * s.in_stride, s.W * s.in_stride, s.cin_pad, err, s.in_stride)) return false;
  } else if (!encode_tmap(&L->tmap_a, s.in, 5, dims, strides, box, 128, err, a_stride != 1 ? estr : nullptr)) return false;
  uint64_t bd[2] = {(uint64_t)k_total, (uint64_t)p.phases * s.n_pad};
  uint64_t bs[1] = {(uint64_t)k_total * 2};
  uint32_t bb[2] = {(uint32_t)block_k, (uint32_t)(s.block_n / path.cg)};
  if (!encode_tmap(&L->tmap_b, s.w, 2, bd, bs, bb, 128, err)) return false;
  L->tmap_out = L->tmap_a;  // placeholders for the epilogues that do not use them
  L->tmap_res = L->tmap_a;
  L->tmap_a2 = L->tmap_a;
  if (s.in2) {
    if (p.mode != 0 || s.kind != CONV_1x1) {
      if (err) *err = "a folded shortcut needs a flat 1x1 conv";
      return false;
    }
    uint64_t d2[5] = {(uint64_t)s.cin2_pad, (uint64_t)p.M, 1, 1, 1};
    uint64_t s2[4] = {(uint64_t)s.cin2_pad * 2, (uint64_t)s.cin2_pad * 2 * p.M, (uint64_t)s.cin2_pad * 2 * p.M,
                      (uint64_t)s.cin2_pad * 2 * p.M};
    if (!encode_tmap(&L->tmap_a2, s.in2, 5, d2, s2, box, 128, err)) return false;
  }
  if (s.epi == EPI_PLANAR_F32 && (p.mode != 0 || (s.H * s.W) % 4 != 0)) {
    if (err) *err = "the planar epilogue needs a flat 1x1 conv whose plane size is a multiple of 4";
    return false;
  }
  if (s.epi == EPI_TMA || s.epi == EPI_TMA_RES) {
    // output (and residual) tiles leave / enter through swizzled smem in 64-channel chunks: same row tiling as A
    if (s.kind == CONV_DECONV4 || s.ldc % 8 != 0) {
      if (err) *err = "TMA epilogue needs a plain NHWC output";
      return false;
    }
    uint64_t od[5], os[4];
    uint32_t ob[5];
    auto act_map = [&](const void* ptr, int ld, CUtensorMap* m, int stride) {
      uint32_t es[5] = {1, (uint32_t)stride, (uint32_t)stride, 1, 1};
      if (p.mode == 0) {
        od[0] = ld; od[1] = p.M; od[2] = 1; od[3] = 1; od[4] = 1;
        os[0] = (uint64_t)ld * 2; os[1] = os[2] = os[3] = (uint64_t)ld * 2 * p.M;
        ob[0] = 64; ob[1] = kBlockM; ob[2] = 1; ob[3] = 1; ob[4] = 1;
      } else {
        od[0] = ld; od[1] = (uint64_t)s.W * stride; od[2] = (uint64_t)s.H * stride; od[3] = 1; od[4] = s.NB;
        os[0] = (uint64_t)ld * 2; os[1] = os[0] * od[1]; os[2] = os[1] * od[2]; os[3] = os[2];
        ob[0] = 64; ob[1] = p.tw * stride; ob[2] = p.th * stride; ob[3] = 1; ob[4] = 1;
      }
      return encode_tmap(m, ptr, 5, od, os, ob, 128, err, stride != 1 ? es : nullptr);
    };
    if (!act_map(s.out, s.ldc, &L->tmap_out, 1)) return false;
    L->tmap_out2 = L->tmap_out;
    L->tmap_w2 = L->tmap_b;
    if (s.out2 != nullptr) {
      if (s.block_n != kTailBlockN || s.kind != CONV_1x1 || p.mode != 0 || !tail_supported(s.n2, s.epi) || !s.w2 || !s.bias2) {
        if (err) *err = "a fused block tail needs a flat 1x1 conv with 256-column tiles and a 64-wide (EPI_TMA) or 128-wide (EPI_TMA_RES) second conv";
        return false;
      }
      if (!act_map(s.out2, s.n2, &L->tmap_out2, 1)) return false;
      uint64_t wd[2] = {(uint64_t)s.n_pad, (uint64_t)s.n2};
      uint64_t ws[1] = {(uint64_t)s.n_pad * 2};
      uint32_t wb[2] = {64, (uint32_t)(s.n2 / 2)};
      if (!encode_tmap(&L->tmap_w2, s.w2, 2, wd, ws, wb, 128, err)) return false;
      L->n2 = s.n2;
      L->bias2 = s.bias2;
    }
    if (s.epi == EPI_TMA_RES) {
      if (!s.residual) {
        if (err) *err = "EPI_TMA_RES without a residual";
        return false;
      }
      if (!act_map(s.residual, s.ldr, &L->tmap_res, s.res_stride)) return false;
      p.res_tx_bytes = (ob[1] / s.res_stride) * (ob[2] / s.res_stride) * 128;
    }
  } else if (s.residual) {
    if (err) *err = "only the EPI_TMA_RES epilogue adds a residual";
    return false;
  }
  if (s.out2 != nullptr && L->n2 == 0) {
    if (err) *err = "a fused block tail needs a TMA epilogue";
    return false;
  }
  if (L->n2 == 0 && find_conv_kernel(*L).fn == nullptr) {
    if (err) {
      char buf[160];
      snprintf(buf, sizeof buf, "no conv kernel for a %d-column tile with epilogue %d (cg %d, resident %d, halo %d)", s.block_n,
               s.epi, path.cg, path.b_resident, path.halo);
      *err = buf;
    }
    return false;
  }
  L->grid = L->n2 ? tail_grid(p, num_sms) : conv_grid(p, path.cg, num_sms);
  L->flops = 2.0 * p.phases * (double)p.M * s.n_pad * k_total + 2.0 * (double)p.M * s.n_pad * L->n2;
  return true;
}

// Launch with programmatic stream serialization (PDL): the kernel may start while its predecessor drains; each of our
// kernels calls pdl_wait() before it touches the predecessor's output.
template <typename Kern, typename... Args>
inline cudaError_t launch_pdl_cluster(Kern kern, dim3 grid, dim3 block, size_t smem, cudaStream_t st, int cluster_x,
                                      Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (cluster_x > 1) {
    attr[1].id = cudaLaunchAttributeClusterDimension;
    attr[1].val.clusterDim.x = cluster_x;
    attr[1].val.clusterDim.y = 1;
    attr[1].val.clusterDim.z = 1;
    cfg.numAttrs = 2;
  }
  return cudaLaunchKernelEx(&cfg, kern, args...);
}
template <typename Kern, typename... Args>
inline cudaError_t launch_pdl(Kern kern, dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  return launch_pdl_cluster(kern, grid, block, smem, st, 1, args...);
}

template <int N2, bool RES>
inline cudaError_t launch_one_tail(const ConvLaunch& L, cudaStream_t st) {
  using Cfg = TailCfg<N2, RES>;
  static unsigned long long done = 0;
  auto kern = block_tail_kernel<N2, RES>;
  if (cudaError_t e = ensure_dyn_smem(kern, Cfg::SMEM_BYTES, &done); e != cudaSuccess) return e;
  BlockTailParams bp;
  bp.g = L.p;
  bp.bias2 = L.bias2;
  bp.n2_k_chunks = L.p.num_n_tiles * (kTailBlockN / 64);
  return launch_pdl_cluster(kern, dim3(L.grid), dim3(kGemmThreadsTma), Cfg::SMEM_BYTES, st, 2, L.tmap_a, L.tmap_b,
                            L.tmap_out, L.tmap_res, L.tmap_a2, L.tmap_w2, L.tmap_out2, bp);
}

inline cudaError_t launch_conv(const ConvLaunch& L, cudaStream_t st) {
  if (L.n2) {
    if (L.n2 == 64 && L.epi == EPI_TMA) return launch_one_tail<64, false>(L, st);
    if (L.n2 == 128 && L.epi == EPI_TMA_RES) return launch_one_tail<128, true>(L, st);
    return cudaErrorInvalidConfiguration;
  }
  const ConvKernel k = find_conv_kernel(L);
  if (k.fn == nullptr) return cudaErrorInvalidConfiguration;
  if (cudaError_t e = ensure_dyn_smem(k.fn, k.smem, k.smem_done); e != cudaSuccess) return e;
  return launch_pdl_cluster(k.fn, dim3(L.grid), dim3(k.threads), k.smem, st, k.cg, L.tmap_a, L.tmap_b, L.tmap_out,
                            L.tmap_res, L.tmap_a2, L.p);
}

// ---------------------------------------------------------------------------------------------------------------
// conv1 + pool1 fused (stem_roll.cuh)
struct StemPoolLaunch {
  StemRollParams r;
  int grid = 0;
  int cg = 1;          // 2: CTA pairs (stem_roll_kernel<., 2>), the two x tiles of a segment on the two CTAs
  CUtensorMap tmap_x;  // pairs: the stem input as [16-byte units][8 halves], strips are boxes of 132 units
};

// [64][224] K-major (k = ky*32 + kx*4 + c) -> the rolling kernel's stacked weights: rows (ky = 6, 4, 2, 0) x 64 couts for
// even input rows, then rows (ky = 5, 3, 1) x 64 couts for odd ones; every row is the 32 K values (64 B) of one row tap
// in the 64B-swizzled K-major UMMA layout (16-byte chunk index ^= (row >> 1) & 3)
inline void pack_stem_stacked(const __half* kmajor, __half* out) {
  __half* even = out;
  __half* odd = out + kRollWEvenBytes / 2;
  for (int n = 0; n < 64; ++n)
    for (int k = 0; k < 32; ++k) {
      const int c = k >> 3, e = k & 7;
      for (int g = 0; g < 4; ++g) {
        const int row = g * 64 + n;
        even[row * 32 + ((c ^ ((row >> 1) & 3)) << 3) + e] = kmajor[n * 224 + (6 - 2 * g) * 32 + k];
      }
      for (int g = 0; g < 3; ++g) {
        const int row = g * 64 + n;
        odd[row * 32 + ((c ^ ((row >> 1) & 3)) << 3) + e] = kmajor[n * 224 + (5 - 2 * g) * 32 + k];
      }
    }
}

// Per-rank weight tables of the CTA-pair kernel (stem_roll.cuh): out = [rank][kPairWBytes]; entry (g, cnt) of a parity
// holds rows [64 g + 32 cnt rank, + 32 cnt) of that parity's stack, 64B-swizzled like pack_stem_stacked
inline void pack_stem_pair(const __half* kmajor, __half* out) {
  for (int rank = 0; rank < 2; ++rank)
    for (int parity = 0; parity < 2; ++parity) {
      const int ng = parity ? 3 : 4;
      __half* pbase = out + (size_t)rank * (kPairWBytes / 2) + (parity ? kPairWEvenBytes / 2 : 0);
      for (int g = 0; g < ng; ++g)
        for (int cnt = 1; cnt <= ng - g; ++cnt) {
          __half* entry = pbase + (size_t)pair_w_units(ng, g, cnt) * (kPairUnitBytes / 2);
          for (int r = 0; r < 32 * cnt; ++r) {
            const int srow = 64 * g + 32 * cnt * rank + r;
            const int gg = srow / 64, n = srow % 64;
            const int ky = (parity ? 5 : 6) - 2 * gg;
            for (int k = 0; k < 32; ++k) {
              const int c = k >> 3, e = k & 7;
              entry[r * 32 + ((c ^ ((r >> 1) & 3)) << 3) + e] = kmajor[n * 224 + ky * 32 + k];
            }
          }
        }
    }
}

// segment length (pooled rows) of the rolling kernel: fewest (waves x input rows per item); a segment re-reads 6
// input rows of its upper neighbour, so longer is cheaper until the last wave goes idle
inline void stem_roll_set_batch(StemRollParams& r, int nb, int num_sms, int* grid) {
  int best_rows = r.PH;
  long best_cost = -1;
  for (int rows = 1; rows <= r.PH; ++rows) {
    const int segs = (r.PH + rows - 1) / rows;
    const long items = (long)nb * segs * r.n_xt;
    const long waves = (items + num_sms - 1) / num_sms;
    const long cost = waves * (4 * rows + 7);
    if (best_cost < 0 || cost <= best_cost) {
      best_cost = cost;
      best_rows = rows;
    }
  }
  r.seg_rows = best_rows;
  r.segs_per_image = (r.PH + best_rows - 1) / best_rows;
  r.num_items = nb * r.segs_per_image * r.n_xt;
  *grid = r.num_items < num_sms ? r.num_items : num_sms;
  *grid &= ~1;  // CTA pairs need an even grid (n_xt == 2 makes the item count even); harmless otherwise unless 1
  if (*grid == 0) *grid = 1;
}

// w_pair: pack_stem_pair's tables, used when the box splits into two x tiles (CTA pairs); x1_halves: allocated size of
// the stem input
inline bool build_stem_pool(const __half* x1, int S, int rows_per_parity, int row_pitch, const __half* w_stacked,
                            const float* bias, __half* pooled_out, int nb, int num_sms, StemPoolLaunch* L,
                            std::string* err, const __half* w_pair, size_t x1_halves) {
  memset(L, 0, sizeof(*L));
  L->cg = 1;
  StemRollParams& r = L->r;
  r.vw = S / 2 + 3;
  if (row_pitch * 2 != r.vw * 16 || S % 16 != 0) {
    if (err) *err = "stem row pitch must be (S/2+3)*16 bytes and S a multiple of 16";
    return false;
  }
  r.x1 = reinterpret_cast<const uint8_t*>(x1);
  r.plane_bytes = (int64_t)rows_per_parity * row_pitch * 2;
  r.w = reinterpret_cast<const uint8_t*>(w_stacked);
  r.bias = bias;
  r.out = pooled_out;
  r.CH = r.CW = S / 2;
  r.PH = r.PW = S / 4;
  int pb = 0;
  while (pb < r.PW) {  // x tiles: 128 conv columns each, pooled columns split where a 3-wide window would cross
    if (r.n_xt == kMaxXTiles) {
      if (err) *err = "box size too large for the rolling stem";
      return false;
    }
    int x0 = 2 * pb < r.CW - kBlockM ? 2 * pb : r.CW - kBlockM;
    if (x0 < 0) x0 = 0;
    const int pe = x0 + kBlockM >= r.CW ? r.PW : (x0 + kBlockM - 3) / 2 + 1;
    r.xt_x0[r.n_xt] = x0;
    r.xt_pb[r.n_xt] = pb;
    r.xt_pe[r.n_xt] = pe;
    ++r.n_xt;
    pb = pe;
  }
  if (r.n_xt == 2 && x1_halves >= 8 && num_sms >= 2) {
    const uint64_t dims[2] = {8, (uint64_t)(x1_halves / 8)};
    const uint64_t strides[1] = {16};
    const uint32_t box[2] = {8, (uint32_t)(kRollStripLoad / 16)};
    if (!encode_tmap(&L->tmap_x, x1, 2, dims, strides, box, 0, err)) return false;
    L->cg = 2;
    r.w = reinterpret_cast<const uint8_t*>(w_pair);
    r.x1_units = (int64_t)(x1_halves / 8);
  }
  stem_roll_set_batch(r, nb, num_sms, &L->grid);
  return true;
}

inline void stem_pool_set_batch(StemPoolLaunch& L, int nb, int num_sms) { stem_roll_set_batch(L.r, nb, num_sms, &L.grid); }

// DBG = true: the cycle-counter variant (stem_roll.cuh), launched by the self-test only
template <bool DBG = false>
inline cudaError_t launch_stem_pool(const StemPoolLaunch& L, cudaStream_t st) {
  static unsigned long long done[2] = {0, 0};
  auto go = [&](auto kern, unsigned long long* mask) -> cudaError_t {
    if (cudaError_t e = ensure_dyn_smem(kern, StemRollSmem::BYTES, mask); e != cudaSuccess) return e;
    return launch_pdl_cluster(kern, dim3(L.grid), dim3(kRollThreads), StemRollSmem::BYTES, st, L.cg, L.r, L.tmap_x);
  };
  return L.cg == 2 ? go(stem_roll_kernel<DBG, 2>, &done[1]) : go(stem_roll_kernel<DBG, 1>, &done[0]);
}

}  // namespace vnect
