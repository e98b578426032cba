// Bandwidth-bound kernels around the CNN: bit-exact OpenCV-style preprocessing (K1), the bbox tracker and the
// fused post-process (K8: multi-scale average -> x8 upsample argmax -> 1-euro filters -> location-map gather).
//
// Reference semantics being restated (XinArkh/VNect): src/estimator.py:70-81 and src/utils.py:13-21,82-150 (K1),
// src/estimator.py:105-142 + src/utils.py:58-79,153-219 + src/OneEuroFilter.py:13-75
// (K8).  Arithmetic that has to be bit-faithful uses explicit round-to-nearest intrinsics so that nvcc cannot
// contract a*b+c into an FMA where OpenCV / CPython do not (and uses FMA where OpenCV+IPP does: the float64 x8
// upsample; see oracle/prepost.py).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "ptx.cuh"

namespace vnect {

constexpr int kJoints = 21;
constexpr int kRootJoint = 14;
constexpr int kMaxScales = 4;
constexpr int kMaxHm = 64;  // heat-map side limit (46 @368, 56 @448)

// ---------------------------------------------------------------------------------------------------------------
// OpenCV INTER_LINEAR coordinate rule (SURVEY.md App. C.1): f = float((d + 0.5) * inv_scale - 0.5) in double, then
// i = floor(f), f -= i in float.  reset=true (x axis): clamp i into [0, src-1] and zero f at the borders.
__device__ __forceinline__ void cv_linear_coord(int d, double inv_scale, int src, bool reset, int* i_out,
                                                float* f_out) {
  const double fd = __dsub_rn(__dmul_rn(__dadd_rn((double)d, 0.5), inv_scale), 0.5);
  float f = __double2float_rn(fd);
  int i = (int)floorf(f);
  f = __fsub_rn(f, (float)i);
  if (reset) {
    if (i < 0) { i = 0; f = 0.f; }
    if (i >= src - 1) { i = src - 1; f = 0.f; }
  }
  *i_out = i;
  *f_out = f;
}

__device__ __forceinline__ int cv_coef(float f) { return __float2int_rn(__fmul_rn(f, 2048.f)); }

// One output pixel (3 channels) of cv2.resize(u8, INTER_LINEAR): 11-bit fixed point, vertical pass
// (((b0*(T0>>4))>>16) + ((b1*(T1>>4))>>16) + 2) >> 2.   `src` reads the source pixels (BgrSrc / Yuv420Src below).
template <class Src>
__device__ __forceinline__ void cv_resize_u8_px(const Src& src, int sh, int sw, int dy, int dx, double inv_scale,
                                                int out[3]) {
  int ix, iy;
  float fx, fy;
  cv_linear_coord(dx, inv_scale, sw, true, &ix, &fx);
  cv_linear_coord(dy, inv_scale, sh, false, &iy, &fy);
  const int a0 = cv_coef(__fsub_rn(1.f, fx)), a1 = cv_coef(fx);
  const int b0 = cv_coef(__fsub_rn(1.f, fy)), b1 = cv_coef(fy);
  const int ix1 = min(ix + 1, sw - 1);
  const int y0 = min(max(iy, 0), sh - 1), y1 = min(max(iy + 1, 0), sh - 1);
  const auto r0 = src.at(y0, 0);
  const auto r1 = src.at(y1, 0);
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const int t0 = src.get(r0, ix, c) * a0 + src.get(r0, ix1, c) * a1;
    const int t1 = src.get(r1, ix, c) * a0 + src.get(r1, ix1, c) * a1;
    out[c] = (((b0 * (t0 >> 4)) >> 16) + ((b1 * (t1 >> 4)) >> 16) + 2) >> 2;
  }
}

// Channel c (0 B, 1 G, 2 R) of cv2.cvtColor(COLOR_YUV2BGR_NV12 / _I420) of one pixel: BT.601 limited range in OpenCV's
// 20-bit fixed point.  Every intermediate stays below 6e8 in magnitude, so int32 is exact.
__device__ __forceinline__ int yuv_to_bgr(int Y, int U, int V, int c) {
  const int uu = U - 128, vv = V - 128, half = 1 << 19;
  const int y = max(0, Y - 16) * 1220542;
  const int uv = c == 0 ? half + 2116026 * uu : c == 1 ? half - 852492 * vv - 409993 * uu : half + 1673527 * vv;
  return min(max((y + uv) >> 20, 0), 255);
}

// Per-frame crop + squarify geometry of the tracked-stream path (run_estimator.py:100 crop, utils.py:107-120 squarify).
struct FrameGeom {
  int x, y, w, h;           // crop box inside the full frame
  int dh, dw;               // scaled content size (cvRound(h*scaler), cvRound(w*scaler))
  int off_x, off_y;         // placement inside the S x S box (utils.py:82-104)
  int mode;                 // 0 bilinear, 1 exact 2x decimation (INTER_AREA)
  int orient;               // VNECT_ORIENT_* of the frame (frame_geometry_oriented_kernel; 0 elsewhere)
  double scaler, inv_scale;
};

struct SquarifyParams {
  int n_frames, H, W;       // raw frames (when geoms != nullptr: the FULL frame size, crops come from geoms)
  int64_t pitch, frame_stride;
  int S;                    // box size
  int dh, dw;               // scaled content size (cvRound(H*scaler), cvRound(W*scaler))
  int off_x, off_y;         // placement inside the box (utils.py:82-104)
  double inv_scale;         // 1 / scaler
  int mode;                 // 0 = bilinear, 1 = exact 2x decimation (OpenCV switches INTER_LINEAR to INTER_AREA)
  const FrameGeom* geoms;   // optional per-frame geometry (tracked streams); overrides the uniform fields above
  // YUV 4:2:0 sources only (`pitch` is then the luma pitch): chroma planes relative to a frame's start
  int64_t uv_pitch, u_offset, v_offset;
  int uv_step;              // bytes between horizontally adjacent chroma samples: 2 (NV12) or 1 (I420)
};

// One frame of a mixed-size batch: the device copy of a vnect_frame (include/vnect_b200.h; same layout, 48 bytes).
// `data` is the frame's first byte (BGR) or the first byte of its luma plane (YUV), height x width its FULL size,
// `pitch` the BGR or luma row pitch; YUV chroma planes are addressed relative to `data`.
struct FrameDesc {
  const uint8_t* data;
  int height, width;
  int64_t pitch, uv_pitch, u_offset, v_offset;
};

// Source pixels of squarify_kernel, one type per input format.  Coordinates count from the crop origin set by crop()
// (the frame's top-left corner when there is none):
//   at(y, x)         a handle on pixel (y, x)
//   below(q, step)   the handle one row below q when step is true, q otherwise
//   get(q, dx, c)    channel c (0 B, 1 G, 2 R) of the pixel dx columns right of q
struct BgrSrc {
  const uint8_t* p;
  int64_t pitch;
  __device__ __forceinline__ BgrSrc(const uint8_t* frame, const SquarifyParams& sp) : p(frame), pitch(sp.pitch) {}
  __device__ __forceinline__ BgrSrc(const FrameDesc& f, const SquarifyParams&) : p(f.data), pitch(f.pitch) {}
  __device__ __forceinline__ void crop(int x, int y) { p += (int64_t)y * pitch + (int64_t)x * 3; }
  __device__ __forceinline__ void crop(const FrameGeom& g) { crop(g.x, g.y); }
  __device__ __forceinline__ const uint8_t* at(int y, int x) const { return p + (int64_t)y * pitch + (int64_t)x * 3; }
  __device__ __forceinline__ const uint8_t* below(const uint8_t* q, bool step) const { return q + (step ? pitch : 0); }
  __device__ __forceinline__ int get(const uint8_t* q, int dx, int c) const { return q[dx * 3 + c]; }
};

// NV12 (uv_step 2) and I420 (uv_step 1), converted per tap.  One chroma pair covers a 2x2 luma block of the FULL frame,
// so the chroma row and column come from full-frame coordinates, not crop-relative ones (a crop box may be odd).
struct Yuv420Src {
  const uint8_t *luma, *u, *v;
  int64_t pitch, uv_pitch;
  int uv_step, x0, y0;
  __device__ __forceinline__ Yuv420Src(const uint8_t* frame, const SquarifyParams& sp)
      : luma(frame), u(frame + sp.u_offset), v(frame + sp.v_offset), pitch(sp.pitch), uv_pitch(sp.uv_pitch),
        uv_step(sp.uv_step), x0(0), y0(0) {}
  __device__ __forceinline__ Yuv420Src(const FrameDesc& f, const SquarifyParams& sp)
      : luma(f.data), u(f.data + f.u_offset), v(f.data + f.v_offset), pitch(f.pitch), uv_pitch(f.uv_pitch),
        uv_step(sp.uv_step), x0(0), y0(0) {}
  __device__ __forceinline__ void crop(int x, int y) { x0 = x; y0 = y; }
  __device__ __forceinline__ void crop(const FrameGeom& g) { crop(g.x, g.y); }
  __device__ __forceinline__ int2 at(int y, int x) const { return make_int2(x0 + x, y0 + y); }  // full-frame (x, y)
  __device__ __forceinline__ int2 below(int2 q, bool step) const { return make_int2(q.x, q.y + (step ? 1 : 0)); }
  __device__ __forceinline__ int get(int2 q, int dx, int c) const {
    const int fx = q.x + dx;
    const int64_t ci = (int64_t)(q.y >> 1) * uv_pitch + (int64_t)(fx >> 1) * uv_step;
    return yuv_to_bgr(luma[(int64_t)q.y * pitch + fx], u[ci], v[ci], c);
  }
};

// Source of a frame of a mixed-size batch.  squarify_kernel's frame pointer `in + n * frame_stride` is then entry n of
// the device frame table (in = the table, frame_stride = sizeof(FrameDesc)), which gives the frame's own address,
// pitches and chroma layout; its crop and size come from SquarifyParams::geoms (frame_geometry_kernel).
template <class Base>
struct FrameTableSrc : Base {
  __device__ __forceinline__ FrameTableSrc(const uint8_t* entry, const SquarifyParams& sp)
      : Base(*reinterpret_cast<const FrameDesc*>(entry), sp) {}
};

// Frame orientation VNECT_ORIENT_* (include/vnect_b200.h) as an index map.  Oriented pixel (yo, xo) of a stored H x W
// frame is stored pixel (ys, xs): ys comes from xo for the codes that swap the sides (1, 3, 6, 7), from yo otherwise,
// and is H-1-(that) for codes 1, 2, 5, 7; xs comes from the other one and is W-1-(that) for codes 2, 3, 4, 7.  The map
// is affine, stored = origin + yo * (step per oriented row) + xo * (step per oriented column), and sends every 2x2
// block of an even-sided frame to a 2x2 block, so 4:2:0 chroma at (ys >> 1, xs >> 1) is that of the oriented frame.
__device__ __forceinline__ bool orient_swaps(int o) { return (0xCA >> o) & 1; }
__device__ __forceinline__ bool orient_rev_y(int o) { return (0xA6 >> o) & 1; }
__device__ __forceinline__ bool orient_rev_x(int o) { return (0x9C >> o) & 1; }

// squarify_kernel source of an oriented frame of a mixed-size batch (through FrameTableSrc): the crop box and the
// pixel coordinates are the oriented frame's, FrameGeom::orient is the code, the FrameDesc the frame as stored.
template <class Base>
struct Oriented;

// BGR: a handle is the stored pixel's byte pointer; one oriented row / column is `sy` / `sx` bytes (signed), e.g.
// (pitch, 3) for identity and (3, -pitch) for ROT90_CW.
template <>
struct Oriented<BgrSrc> {
  const uint8_t *frame, *p;
  int64_t pitch, sy, sx;
  int H, W;
  __device__ __forceinline__ Oriented(const FrameDesc& f, const SquarifyParams&)
      : frame(f.data), p(f.data), pitch(f.pitch), sy(f.pitch), sx(3), H(f.height), W(f.width) {}
  __device__ __forceinline__ void crop(const FrameGeom& g) {
    const int o = g.orient;
    const bool ry = orient_rev_y(o), rx = orient_rev_x(o);
    const int64_t dy = ry ? -pitch : pitch, dx = rx ? -3 : 3;
    if (orient_swaps(o)) { sy = dx; sx = dy; } else { sy = dy; sx = dx; }
    p = frame + (ry ? (int64_t)(H - 1) * pitch : 0) + (rx ? (int64_t)(W - 1) * 3 : 0) + (int64_t)g.y * sy +
        (int64_t)g.x * sx;
  }
  __device__ __forceinline__ const uint8_t* at(int y, int x) const { return p + (int64_t)y * sy + (int64_t)x * sx; }
  __device__ __forceinline__ const uint8_t* below(const uint8_t* q, bool step) const { return q + (step ? sy : 0); }
  __device__ __forceinline__ int get(const uint8_t* q, int dx, int c) const { return q[dx * sx + c]; }
};

// YUV 4:2:0: a handle is the stored full-frame (x, y); `ey` / `ex` are the stored (x, y) steps of one oriented row /
// column.  Luma and chroma are read at the stored coordinates, like Yuv420Src.
template <>
struct Oriented<Yuv420Src> : Yuv420Src {
  int H, W;
  int2 org, ey, ex;
  __device__ __forceinline__ Oriented(const FrameDesc& f, const SquarifyParams& sp)
      : Yuv420Src(f, sp), H(f.height), W(f.width), org(make_int2(0, 0)), ey(make_int2(0, 1)), ex(make_int2(1, 0)) {}
  __device__ __forceinline__ void crop(const FrameGeom& g) {
    const int o = g.orient;
    const bool ry = orient_rev_y(o), rx = orient_rev_x(o);
    const int2 dy = make_int2(0, ry ? -1 : 1), dx = make_int2(rx ? -1 : 1, 0);
    if (orient_swaps(o)) { ey = dx; ex = dy; } else { ey = dy; ex = dx; }
    org = make_int2((rx ? W - 1 : 0) + g.y * ey.x + g.x * ex.x, (ry ? H - 1 : 0) + g.y * ey.y + g.x * ex.y);
  }
  __device__ __forceinline__ int2 at(int y, int x) const {
    return make_int2(org.x + y * ey.x + x * ex.x, org.y + y * ey.y + x * ex.y);
  }
  __device__ __forceinline__ int2 below(int2 q, bool step) const {
    return step ? make_int2(q.x + ey.x, q.y + ey.y) : q;
  }
  __device__ __forceinline__ int get(int2 q, int dx, int c) const {
    const int xs = q.x + dx * ex.x, ys = q.y + dx * ex.y;
    const int64_t ci = (int64_t)(ys >> 1) * uv_pitch + (int64_t)(xs >> 1) * uv_step;
    return yuv_to_bgr(luma[(int64_t)ys * pitch + xs], u[ci], v[ci], c);
  }
};

// utils.img_scale_squarify geometry (utils.py:107-120) for box (x, y, w, h) -- same arithmetic as the host version
__device__ __forceinline__ FrameGeom make_frame_geom(int x, int y, int w, int h, int S) {
  FrameGeom g;
  g.x = x; g.y = y; g.w = w; g.h = h;
  g.scaler = __ddiv_rn((double)S, (double)max(h, w));
  g.dw = __double2int_rn(__dmul_rn((double)w, g.scaler));
  g.dh = __double2int_rn(__dmul_rn((double)h, g.scaler));
  g.off_x = g.off_y = 0;
  if (g.dh > g.dw) g.off_x = S / 2 - g.dw / 2;
  else g.off_y = S / 2 - g.dh / 2;
  g.inv_scale = __ddiv_rn(1.0, g.scaler);
  g.mode = (g.inv_scale == 2.0) ? 1 : 0;
  g.orient = 0;
  return g;
}

// numpy slicing frame[y:y+h, x:x+w] clips a tracked box to the FH x FW frame (run_estimator.py:100); keep at least
// 2x2 pixels
__device__ __forceinline__ int4 clip_box(int4 b, int FH, int FW) {
  b.x = min(max(b.x, 0), FW - 2);
  b.y = min(max(b.y, 0), FH - 2);
  b.z = max(min(b.z, FW - b.x), 2);
  b.w = max(min(b.w, FH - b.y), 2);
  return b;
}

// boxes: [max_streams] int4 (x, y, w, h); one thread per frame
__global__ void track_geometry_kernel(const int4* __restrict__ boxes, const int* __restrict__ stream_ids, int n, int S,
                                      int FH, int FW, FrameGeom* __restrict__ geoms, int* __restrict__ boxes_used) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int4 b = clip_box(boxes[stream_ids[i]], FH, FW);
  geoms[i] = make_frame_geom(b.x, b.y, b.z, b.w, S);
  boxes_used[4 * i + 0] = b.x; boxes_used[4 * i + 1] = b.y; boxes_used[4 * i + 2] = b.z; boxes_used[4 * i + 3] = b.w;
}

// Geometry of a mixed-size batch, one thread per frame, from each frame's own size: the stream's tracked box clipped
// to that frame when `boxes` is set (boxes_used records it), otherwise the whole frame, box (0, 0, W_i, H_i).
__global__ void frame_geometry_kernel(const FrameDesc* __restrict__ frames, const int4* __restrict__ boxes,
                                      const int* __restrict__ stream_ids, int n, int S, FrameGeom* __restrict__ geoms,
                                      int* __restrict__ boxes_used) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int FH = frames[i].height, FW = frames[i].width;
  int4 b = make_int4(0, 0, FW, FH);
  if (boxes != nullptr) {
    b = clip_box(boxes[stream_ids[i]], FH, FW);
    boxes_used[4 * i + 0] = b.x; boxes_used[4 * i + 1] = b.y; boxes_used[4 * i + 2] = b.z; boxes_used[4 * i + 3] = b.w;
  }
  geoms[i] = make_frame_geom(b.x, b.y, b.z, b.w, S);
}

// frame_geometry_kernel for a batch with oriented frames (orient[i]: frame i's VNECT_ORIENT_* code): box, clip and
// geometry are those of the oriented frame, whose sides are the stored ones swapped for codes 1, 3, 6 and 7.
__global__ void frame_geometry_oriented_kernel(const FrameDesc* __restrict__ frames, const int* __restrict__ orient,
                                               const int4* __restrict__ boxes, const int* __restrict__ stream_ids,
                                               int n, int S, FrameGeom* __restrict__ geoms,
                                               int* __restrict__ boxes_used) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int o = orient[i];
  const bool swap = orient_swaps(o);
  const int FH = swap ? frames[i].width : frames[i].height, FW = swap ? frames[i].height : frames[i].width;
  int4 b = make_int4(0, 0, FW, FH);
  if (boxes != nullptr) {
    b = clip_box(boxes[stream_ids[i]], FH, FW);
    boxes_used[4 * i + 0] = b.x; boxes_used[4 * i + 1] = b.y; boxes_used[4 * i + 2] = b.z; boxes_used[4 * i + 3] = b.w;
  }
  FrameGeom g = make_frame_geom(b.x, b.y, b.z, b.w, S);
  g.orient = o;
  geoms[i] = g;
}

// utils.img_scale_squarify (utils.py:107-120): resize so the longer side is S, centre on black.  out: u8 [n,S,S,3].
// Src is the source format: BgrSrc, or Yuv420Src, which makes this cv2.cvtColor(YUV2BGR) followed by the squarify.
// Output pixel (n, y, x) of squarify_tiled_kernel, element i = (n * S + y) * S + x of `out`: squarify_kernel's loop
// body, restated because routing squarify_kernel through it changes that kernel's SASS.
template <class Src>
__device__ __forceinline__ void squarify_px(const uint8_t* __restrict__ in, uint8_t* __restrict__ out,
                                            const SquarifyParams& p, int n, int y, int x, int64_t i) {
  int H = p.H, W = p.W, dh = p.dh, dw = p.dw, off_x = p.off_x, off_y = p.off_y, mode = p.mode;
  double inv_scale = p.inv_scale;
  Src src(in + (int64_t)n * p.frame_stride, p);
  if (p.geoms != nullptr) {
    const FrameGeom g = p.geoms[n];
    H = g.h; W = g.w; dh = g.dh; dw = g.dw; off_x = g.off_x; off_y = g.off_y; mode = g.mode; inv_scale = g.inv_scale;
    src.crop(g);
  }
  int v[3] = {0, 0, 0};
  const int sy = y - off_y, sx = x - off_x;
  if (sy >= 0 && sy < dh && sx >= 0 && sx < dw) {
    if (mode == 0) {
      cv_resize_u8_px(src, H, W, sy, sx, inv_scale, v);
    } else {
      // OpenCV resizeAreaFast (exact 2x): full 2x2 blocks are (sum + 2) >> 2; where an odd source side leaves a
      // partial block (e.g. 736x735 -> dw = cvRound(367.5) = 368), only the in-range pixels are averaged:
      // saturate_cast<uchar>((float)sum / count), i.e. float division then round-half-even.
      const auto r0 = src.at(2 * sy, 2 * sx);
      const bool col2 = 2 * sx + 1 < W, row2 = 2 * sy + 1 < H;
      const auto r1 = src.below(r0, row2);
      if (col2 && row2) {
#pragma unroll
        for (int c = 0; c < 3; ++c)
          v[c] = (src.get(r0, 0, c) + src.get(r0, 1, c) + src.get(r1, 0, c) + src.get(r1, 1, c) + 2) >> 2;
      } else {
        const int count = (col2 ? 2 : 1) * (row2 ? 2 : 1);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          int sum = src.get(r0, 0, c);
          if (col2) sum += src.get(r0, 1, c);
          if (row2) sum += src.get(r1, 0, c);
          v[c] = __float2int_rn(__fdiv_rn((float)sum, (float)count));
        }
      }
    }
  }
  uint8_t* o = out + i * 3;
  o[0] = (uint8_t)v[0];
  o[1] = (uint8_t)v[1];
  o[2] = (uint8_t)v[2];
}

template <class Src>
__global__ void squarify_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, SquarifyParams p) {
  const int64_t total = (int64_t)p.n_frames * p.S * p.S;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int x = (int)(i % p.S);
    const int y = (int)((i / p.S) % p.S);
    const int n = (int)(i / ((int64_t)p.S * p.S));
    int H = p.H, W = p.W, dh = p.dh, dw = p.dw, off_x = p.off_x, off_y = p.off_y, mode = p.mode;
    double inv_scale = p.inv_scale;
    Src src(in + (int64_t)n * p.frame_stride, p);
    if (p.geoms != nullptr) {
      const FrameGeom g = p.geoms[n];
      H = g.h; W = g.w; dh = g.dh; dw = g.dw; off_x = g.off_x; off_y = g.off_y; mode = g.mode; inv_scale = g.inv_scale;
      src.crop(g);
    }
    int v[3] = {0, 0, 0};
    const int sy = y - off_y, sx = x - off_x;
    if (sy >= 0 && sy < dh && sx >= 0 && sx < dw) {
      if (mode == 0) {
        cv_resize_u8_px(src, H, W, sy, sx, inv_scale, v);
      } else {
        // OpenCV resizeAreaFast (exact 2x): full 2x2 blocks are (sum + 2) >> 2; where an odd source side leaves a
        // partial block (e.g. 736x735 -> dw = cvRound(367.5) = 368), only the in-range pixels are averaged:
        // saturate_cast<uchar>((float)sum / count), i.e. float division then round-half-even.
        const auto r0 = src.at(2 * sy, 2 * sx);
        const bool col2 = 2 * sx + 1 < W, row2 = 2 * sy + 1 < H;
        const auto r1 = src.below(r0, row2);
        if (col2 && row2) {
#pragma unroll
          for (int c = 0; c < 3; ++c)
            v[c] = (src.get(r0, 0, c) + src.get(r0, 1, c) + src.get(r1, 0, c) + src.get(r1, 1, c) + 2) >> 2;
        } else {
          const int count = (col2 ? 2 : 1) * (row2 ? 2 : 1);
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            int sum = src.get(r0, 0, c);
            if (col2) sum += src.get(r0, 1, c);
            if (row2) sum += src.get(r1, 0, c);
            v[c] = __float2int_rn(__fdiv_rn((float)sum, (float)count));
          }
        }
      }
    }
    uint8_t* o = out + i * 3;
    o[0] = (uint8_t)v[0];
    o[1] = (uint8_t)v[1];
    o[2] = (uint8_t)v[2];
  }
}

// squarify_kernel with each warp on an 8 x 4 (rows x columns) tile of output pixels instead of 32 consecutive pixels
// of one row.  For the orientations that swap the sides, one oriented column is one stored row: a warp's taps then
// fall on 4 stored rows, 8 adjacent pixels each, instead of 32 stored rows one pixel each.  S is a multiple of 16, so
// the tiles cover the box exactly.
template <class Src>
__global__ void squarify_tiled_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, SquarifyParams p) {
  const int tx = p.S / 4, per_frame = tx * (p.S / 8);
  const int64_t tiles = (int64_t)p.n_frames * per_frame;
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x / 32);
  for (int64_t t = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / 32; t < tiles; t += warps) {
    const int n = (int)(t / per_frame), r = (int)(t - (int64_t)n * per_frame);
    const int y = (r / tx) * 8 + (lane >> 2), x = (r % tx) * 4 + (lane & 3);
    squarify_px<Src>(in, out, p, n, y, x, ((int64_t)n * p.S + y) * p.S + x);
  }
}

constexpr int kMaxBox = 512;

// Per pyramid scale: the OpenCV coordinate / fixed-point coefficient of every destination column and row, computed
// once on the host with the same arithmetic as cv_linear_coord / cv_coef (the scales are fixed at vnect_create).
struct PyramidTable {
  uint2 xt[kMaxBox];   // x axis (index clamp + f reset): .x = 4*ix | 4*ix1 << 16 (byte offsets into a staged row of 4-byte
                       // pixels), .y = a0 | a1 << 16 (11-bit fixed-point weights)
  short4 yt[kMaxBox];  // y axis (rows clamped, f kept): .x/.y = the two source rows, .z/.w = weights
};

constexpr int kPyrRows = 8;       // output rows per block
constexpr int kPyrThreads = 256;

struct PyramidParams {
  int n_frames, S, n_scales;
  int64_t sq_pitch, sq_frame_stride;  // square u8 input (may alias the raw frames when they are already S x S)
  int R[kMaxScales];                  // resized side cvRound(S*s); == S for s >= 1 (identity)
  int pad0[kMaxScales];               // (S - R) / 2
  unsigned int r_magic[kMaxScales];   // floor(2^32 / R) + 1: i / R == umulhi(i, r_magic) for the indices used here
  unsigned int q_magic;               // the same for S / 4
  double inv_scale[kMaxScales];       // 1 / s
  const PyramidTable* tables;         // [n_scales], device
  const uint32_t* lut;                // [256]: fp16(float32(v) / 255 - 0.4) in the low half of a word, for every 8-bit value
  // stem layout: [forward][parity][rows_per_parity][row_pitch] halves, pixel (y, x) lives at padded (y+2, x+2)
  int rows_per_parity, row_pitch;
  int full;                           // also write the black surround of the shrunken scales (see below)
};

__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {  // plain shared-memory load from a 32-bit shared address
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}

// 12 source bytes = 4 BGR pixels as three words -> four words with one pixel in the low three bytes of each
__device__ __forceinline__ uint4 expand_bgr4(uint32_t w0, uint32_t w1, uint32_t w2) {
  return make_uint4(w0, __funnelshift_r(w0, w1, 24), __funnelshift_r(w1, w2, 16), w2 >> 8);
}
__device__ __forceinline__ void load_bgr4(const uint8_t* s, bool aligned, uint32_t* w0, uint32_t* w1, uint32_t* w2) {
  if (aligned) {
    *w0 = __ldg(reinterpret_cast<const uint32_t*>(s));
    *w1 = __ldg(reinterpret_cast<const uint32_t*>(s) + 1);
    *w2 = __ldg(reinterpret_cast<const uint32_t*>(s) + 2);
  } else {
    *w0 = s[0] | (s[1] << 8) | (s[2] << 16) | ((uint32_t)s[3] << 24);
    *w1 = s[4] | (s[5] << 8) | (s[6] << 16) | ((uint32_t)s[7] << 24);
    *w2 = s[8] | (s[9] << 8) | (s[10] << 16) | ((uint32_t)s[11] << 24);
  }
}

// estimator.gen_input_batch (estimator.py:70-81): per scale shrink + zero pad (utils.py:123-150), then
// float32(u8)/255 - 0.4, stored as fp16 in the parity-split padded NHWC4 layout the stem conv's TMA reads.
//
// grid = (ceil(S / 8), n_frames * n_scales forwards); a block writes 8 output rows of one forward.
//  * scale 1: pure conversion, four pixels (12 source bytes as three aligned words, 32 output bytes) per thread;
//  * shrunken scale: only the R x R picture is computed.  Its black surround is the same constant for every frame
//    (fp16(0/255 - 0.4)), lives in a slot of x1 that always holds this scale, and is therefore written ONCE
//    (`full`, at start-up and after vnect_forward has overwritten the buffer): 51 % of a 0.7-scale forward's bytes.
//    The source rows the block's 8 output rows sample (~8/s + 2) are staged in shared memory as 4-byte pixels, so a
//    tap is one aligned word, the horizontal pass of a row is two byte permutes + three dp2a (weights as a 16-bit
//    pair), and every source byte leaves L2 once per block;
//  * the normalisation is a 256-entry table built on the host (an IEEE division per channel was a third of the first
//    version's instructions; rebuilding the table in every block was most of the second's).
__global__ void __launch_bounds__(kPyrThreads) pyramid_kernel(const uint8_t* __restrict__ sq, __half* __restrict__ x1,
                                                              const __grid_constant__ PyramidParams p) {
  extern __shared__ __align__(16) uint8_t s_px[];  // staged source rows, 4 bytes per pixel
  __shared__ __align__(16) uint32_t s_lut[256];
  __shared__ uint2 s_xt[kMaxBox];  // this scale's column entries
  struct RowInfo { int r0, r1; unsigned int b0, b1; int out; int pad[3]; };
  __shared__ __align__(16) RowInfo s_row[kPyrRows];
  pdl_launch_dependents();
  const int tid = threadIdx.x;
  s_lut[tid] = p.lut[tid];  // kPyrThreads == 256
  pdl_wait();  // x1 may still be read by the previous batch's stem kernel; sq comes from the copy / squarify before us
  const int S = p.S;
  const int fwd = blockIdx.y;
  const int frame = fwd / p.n_scales, si = fwd - frame * p.n_scales;
  const int R = p.R[si], pad0 = p.pad0[si];
  const uint8_t* src = sq + (int64_t)frame * p.sq_frame_stride;
  const int y0 = blockIdx.x * kPyrRows, y1 = min(y0 + kPyrRows, S);
  __half* x1f = x1 + (int64_t)fwd * 2 * p.rows_per_parity * p.row_pitch;
  // output row y starts at padded row y + 2, padded column 2 (8 halves); offset in halves from x1f
  auto out_row = [&](int y) -> int {
    const int pr = y + 2;
    return ((pr & 1) * p.rows_per_parity + (pr >> 1)) * p.row_pitch + 8;
  };
  const bool aligned = ((reinterpret_cast<uintptr_t>(src) | (uintptr_t)p.sq_pitch) & 3) == 0;
  const int qpr = S >> 2;  // 4-pixel groups per row (S is a multiple of 16)
  const int pitch = (int)p.sq_pitch;  // a frame's rows are less than 2 GB apart
  // flat index i = tid + k * 256 over rows of `w` items as (row, column), advanced without a division per step
  const int step_rows_q = kPyrThreads / qpr, step_cols_q = kPyrThreads - step_rows_q * qpr;
  if (R == S) {
    __syncthreads();
    const uint8_t* src0 = src + (int64_t)y0 * p.sq_pitch;
    const int rows = y1 - y0;
    int ly = (int)__umulhi((unsigned int)tid, p.q_magic), qx = tid - ly * qpr;
    for (; ly < rows; ly += step_rows_q, qx += step_cols_q) {
      if (qx >= qpr) { qx -= qpr; if (++ly >= rows) break; }
      uint32_t w0, w1, w2;
      load_bgr4(src0 + (ly * pitch + qx * 12), aligned, &w0, &w1, &w2);
      uint4 o0, o1;  // the fourth half of a pixel is fp16 zero = the empty high half of a table word
      o0.x = s_lut[w0 & 0xff] | (s_lut[(w0 >> 8) & 0xff] << 16);
      o0.y = s_lut[(w0 >> 16) & 0xff];
      o0.z = s_lut[w0 >> 24] | (s_lut[w1 & 0xff] << 16);
      o0.w = s_lut[(w1 >> 8) & 0xff];
      o1.x = s_lut[(w1 >> 16) & 0xff] | (s_lut[w1 >> 24] << 16);
      o1.y = s_lut[w2 & 0xff];
      o1.z = s_lut[(w2 >> 8) & 0xff] | (s_lut[(w2 >> 16) & 0xff] << 16);
      o1.w = s_lut[w2 >> 24];
      uint4* o = reinterpret_cast<uint4*>(x1f + (out_row(y0 + ly) + qx * 16));
      o[0] = o0;
      o[1] = o1;
    }
    return;
  }
  const PyramidTable* __restrict__ T = p.tables + si;
  const int ry0 = max(y0, pad0) - pad0, ry1 = min(y1, pad0 + R) - pad0;  // picture rows of this block
  if (ry0 < ry1) {
    // stage the source rows [s_lo, s_hi] (the row entries are non-decreasing), expanded to one word per pixel
    const int s_lo = T->yt[ry0].x, s_hi = T->yt[ry1 - 1].y;
    const int rb = S * 4;
    {
      const uint8_t* src0 = src + (int64_t)s_lo * p.sq_pitch;
      const int rows = s_hi - s_lo + 1;
      int r = (int)__umulhi((unsigned int)tid, p.q_magic), qx = tid - r * qpr;
      for (; r < rows; r += step_rows_q, qx += step_cols_q) {
        if (qx >= qpr) { qx -= qpr; if (++r >= rows) break; }
        uint32_t w0, w1, w2;
        load_bgr4(src0 + (r * pitch + qx * 12), aligned, &w0, &w1, &w2);
        *reinterpret_cast<uint4*>(s_px + r * rb + qx * 16) = expand_bgr4(w0, w1, w2);
      }
    }
    for (int i = tid; i < R; i += kPyrThreads) s_xt[i] = T->xt[i];
    if (tid < ry1 - ry0) {
      const short4 yt = T->yt[ry0 + tid];
      RowInfo ri;
      ri.r0 = (yt.x - s_lo) * rb;
      ri.r1 = (yt.y - s_lo) * rb;
      // (b * (t >> 4)) >> 16 as the high word of (b << 16) * (t >> 4): all operands are non-negative
      ri.b0 = (unsigned int)yt.z << 16;
      ri.b1 = (unsigned int)yt.w << 16;
      ri.out = out_row(ry0 + tid + pad0) + pad0 * 4;
      ri.pad[0] = ri.pad[1] = ri.pad[2] = 0;
      s_row[tid] = ri;
    }
    __syncthreads();
    const int rows = ry1 - ry0;
    const int step_rows = kPyrThreads / R, step_cols = kPyrThreads - step_rows * R;
    const uint32_t px_base = smem_u32(s_px), lut_base = smem_u32(s_lut);
    int ly = (int)__umulhi((unsigned int)tid, p.r_magic[si]), rx = tid - ly * R;
    for (; ly < rows; ly += step_rows, rx += step_cols) {
      if (rx >= R) { rx -= R; if (++ly >= rows) break; }
      const RowInfo ri = s_row[ly];
      const uint2 xt = s_xt[rx];
      const uint32_t c0 = px_base + (xt.x & 0xffff), c1 = px_base + (xt.x >> 16);
      const uint32_t p00 = lds_u32(c0 + ri.r0), p01 = lds_u32(c1 + ri.r0);
      const uint32_t p10 = lds_u32(c0 + ri.r1), p11 = lds_u32(c1 + ri.r1);
      // horizontal pass: t = v(x0) * a0 + v(x1) * a1 per channel, the two bytes of a channel side by side
      const uint32_t q0 = __byte_perm(p00, p01, 0x5140), q0r = __byte_perm(p00, p01, 0x0062);
      const uint32_t q1 = __byte_perm(p10, p11, 0x5140), q1r = __byte_perm(p10, p11, 0x0062);
      const uint32_t t0[3] = {__dp2a_lo(xt.y, q0, 0u), __dp2a_hi(xt.y, q0, 0u), __dp2a_lo(xt.y, q0r, 0u)};
      const uint32_t t1[3] = {__dp2a_lo(xt.y, q1, 0u), __dp2a_hi(xt.y, q1, 0u), __dp2a_lo(xt.y, q1r, 0u)};
      uint32_t e[3];  // table word of channel c: its address is base + 4 * ((sum + 2) >> 2) = (base + 2 + sum) & ~3
#pragma unroll
      for (int c = 0; c < 3; ++c)
        e[c] = lds_u32((lut_base + 2u + __umulhi(ri.b0, t0[c] >> 4) + __umulhi(ri.b1, t1[c] >> 4)) & ~3u);
      uint2 o;
      o.x = e[0] | (e[1] << 16);
      o.y = e[2];
      *reinterpret_cast<uint2*>(x1f + (ri.out + rx * 4)) = o;
    }
  } else {
    __syncthreads();  // s_lut
  }
  if (p.full) {  // the black surround: float32(0) / 255 - 0.4
    uint2 o;
    o.x = s_lut[0] | (s_lut[0] << 16);
    o.y = s_lut[0];
    const int npx = (y1 - y0) * S;
    for (int i = tid; i < npx; i += kPyrThreads) {
      const int ly = i / S, x = i - ly * S, y = y0 + ly;
      const bool inside = y >= pad0 && y < pad0 + R && x >= pad0 && x < pad0 + R;
      if (!inside) *reinterpret_cast<uint2*>(x1f + out_row(y) + x * 4) = o;
    }
  }
}

// Operator-level entry (vnect_forward): float32 NHWC [n,S,S,3] -> stem layout (fp16).
__global__ void f32_to_stem_kernel(const float* __restrict__ in, __half* __restrict__ x1, int n, int S,
                                   int rows_per_parity, int row_pitch) {
  const int64_t total = (int64_t)n * S * S;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int x = (int)(i % S);
    const int y = (int)((i / S) % S);
    const int fwd = (int)(i / ((int64_t)S * S));
    __half h[4];
    h[0] = __float2half_rn(in[i * 3 + 0]);
    h[1] = __float2half_rn(in[i * 3 + 1]);
    h[2] = __float2half_rn(in[i * 3 + 2]);
    h[3] = __float2half_rn(0.f);
    const int pr = y + 2, pc = x + 2;
    __half* o = x1 + (((int64_t)fwd * 2 + (pr & 1)) * rows_per_parity + (pr >> 1)) * row_pitch + pc * 4;
    *reinterpret_cast<uint2*>(o) = *reinterpret_cast<const uint2*>(h);
  }
}

// Inverse of the above for tests: stem layout -> float32 NHWC [n,S,S,3].
__global__ void stem_to_f32_kernel(const __half* __restrict__ x1, float* __restrict__ out, int n, int S,
                                   int rows_per_parity, int row_pitch) {
  const int64_t total = (int64_t)n * S * S;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int x = (int)(i % S);
    const int y = (int)((i / S) % S);
    const int fwd = (int)(i / ((int64_t)S * S));
    const int pr = y + 2, pc = x + 2;
    const __half* o = x1 + (((int64_t)fwd * 2 + (pr & 1)) * rows_per_parity + (pr >> 1)) * row_pitch + pc * 4;
    out[i * 3 + 0] = __half2float(o[0]);
    out[i * 3 + 1] = __half2float(o[1]);
    out[i * 3 + 2] = __half2float(o[2]);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// K8: fused post-process.
struct ScaleTable {  // per pyramid scale: where output cell c of the cropped, 1/s-resized map samples the raw map
  short i0[kMaxHm], i1[kMaxHm];      // x axis (index clamp + f reset)
  float a0[kMaxHm], a1[kMaxHm];
  short j0[kMaxHm], j1[kMaxHm];      // y axis (rows clamped, f kept)
  float b0[kMaxHm], b1[kMaxHm];
  int4 rowpk[kMaxHm];                 // the y-axis entries again, one 16-byte load: (j0*hs, j1*hs, bits of b0, bits of b1)
  int identity;                       // s == 1: plain copy
  int row_lo, row_hi;                 // raw rows the cropped resize ever reads (only those are staged on chip)
};

struct FilterCfg { double freq, mincutoff, beta, dcutoff; };

// One scalar 1-euro filter (OneEuroFilter.py:41-75).
struct FilterState {
  double prev;      // last raw value (LowPassFilter.__y of the x filter); float32-valued for 3D filters
  double s_x, s_dx; // smoothed value / smoothed derivative
  double lasttime, freq;
  int has_prev, has_time;
};

__device__ __forceinline__ double oef_alpha(double freq, double cutoff) {
  const double te = __ddiv_rn(1.0, freq);
  const double tau = __ddiv_rn(1.0, __dmul_rn(6.283185307179586, cutoff));  // 2*math.pi is exact doubling
  return __ddiv_rn(1.0, __dadd_rn(1.0, __ddiv_rn(tau, te)));
}

// x_is_f32: numpy-1.x ("legacy") promotion for the float32 3D joints -- the raw difference is float32.
// The host validates t > lasttime before anything is launched (a repeated timestamp is the reference's
// ZeroDivisionError, an earlier one its LowPassFilter ValueError: alpha leaves (0, 1]), so freq stays positive here.
__device__ __forceinline__ double oef_step(FilterState& st, const FilterCfg& cfg, double x, double t, bool x_is_f32) {
  if (st.has_time && st.lasttime != 0.0 && t != 0.0) st.freq = __ddiv_rn(1.0, __dsub_rn(t, st.lasttime));
  st.lasttime = t;
  st.has_time = 1;
  double dx = 0.0;
  if (st.has_prev) {
    const double diff = x_is_f32 ? (double)__fsub_rn((float)x, (float)st.prev) : __dsub_rn(x, st.prev);
    dx = __dmul_rn(diff, st.freq);
  }
  const double a_d = oef_alpha(st.freq, cfg.dcutoff);
  const double edx = st.has_prev ? __dadd_rn(__dmul_rn(a_d, dx), __dmul_rn(__dsub_rn(1.0, a_d), st.s_dx)) : dx;
  const double cutoff = __dadd_rn(cfg.mincutoff, __dmul_rn(cfg.beta, fabs(edx)));
  const double a = oef_alpha(st.freq, cutoff);
  const double s = st.has_prev ? __dadd_rn(__dmul_rn(a, x), __dmul_rn(__dsub_rn(1.0, a), st.s_x)) : x;
  st.prev = x;
  st.s_x = s;
  st.s_dx = edx;
  st.has_prev = 1;
  return s;
}

struct PostParams {
  int n_frames, n_scales, hs, S;  // hs = S / 8
  const float* maps;              // planar [n_frames*n_scales][84][hs][hs]
  const ScaleTable* tables;       // [n_scales]
  const int* stream_ids;          // [n_frames]
  const double* t2d;              // [n_frames]
  const double* t3d;
  FilterState* st2d;              // [max_streams][21][2]
  FilterState* st3d;              // [max_streams][21][3]
  FilterCfg cfg2d, cfg3d;
  int filters_on;
  int scores_off;                 // SCORES: the [n_frames][21] float64 scores start this many ints after raw_argmax (in
                                  // the padding before `scaler`, so the parameter block is that of the other kernels)
  double scaler;                  // box px per input px (S / max(H, W))
  int off_x, off_y;
  const FrameGeom* geoms;         // optional per-frame geometry (tracked streams): scaler, offsets and the crop origin
  double* j2_box;                 // [n_frames][21][2] scratch: filtered 2D joints in box pixels (also an output tap)
  float* j3_raw;                  // [n_frames][21][3] scratch: x100 location-map samples before root subtraction
  int* raw_argmax;                // [n_frames][21][2] unfiltered argmax (row, col), a tap for parity tests
  unsigned int* frame_counter;    // [n_frames]: zero between launches (the last block of a frame puts it back to zero)
  double* out2d;                  // [n_frames][21][2]
  float* out3d;                   // [n_frames][21][3]
  double* packed;                 // optional [n_frames][21][5] = (row, col, x, y, z): the layout the multi-GPU gather moves
  unsigned int* nonfinite;        // counts (frame, joint) blocks that met a NaN / Inf in the CNN's maps (fp16 overflow guard)
  unsigned int* nonfinite_flag;   // host-visible (mapped pinned) word of the submitting lane: set to 1 in that case
  double* prep3;                  // [n_frames][21][3][3] scratch: clock-only part (freq, te, alpha_d) of every 3D filter step,
                                  // computed by the joint's own block while it is otherwise idle, used by the frame's tail
  // shared-memory plan of one block (post_smem_plan, host): which raw cells of every scale's heat-map plane are staged
  // and where.  An identity scale needs its whole plane, a resized one only the rows its centre crop samples.
  int identity_mask;              // bit sc: scale sc is a plain copy
  int plane_start[kMaxScales];    // first raw cell staged
  int plane_len[kMaxScales];      // cells staged
  int plane_off[kMaxScales];      // where, in floats from the start of the dynamic shared memory (multiple of 4)
  int sum_off;                    // float32 plane of per-cell sums over the scales
  int alias_scale;                // the sums overwrite this (identity) scale's staged plane in place; -1: own plane
  int smem_floats;                // dynamic shared memory, in floats
  int y_split;                    // the sum pass starts on rows [0, y_split) while the rest is still in flight
  int plane_split[kMaxScales];    // staged cells (from plane_start) that rows [0, y_split) need
  unsigned long long* trace;      // optional [blocks][16] globaltimer readings at the phase boundaries (VNECT_B200_POST_TRACE)
};

// Host side of the plan above.  `rows_lo/hi` per scale come from the ScaleTable.
inline void post_smem_plan(PostParams& p, const ScaleTable* host_tables, int y_split) {
  const int cells = p.hs * p.hs;
  const bool vec = (cells & 3) == 0;  // 16-byte cp.async needs 16-byte aligned plane starts
  int off = 0;
  p.identity_mask = 0;
  p.alias_scale = -1;
  for (int sc = 0; sc < kMaxScales; ++sc) { p.plane_start[sc] = p.plane_len[sc] = p.plane_off[sc] = p.plane_split[sc] = 0; }
  for (int sc = 0; sc < p.n_scales; ++sc) {
    const ScaleTable& T = host_tables[sc];
    int start = 0, end = cells;
    if (T.identity) {
      p.identity_mask |= 1 << sc;
      if (p.alias_scale < 0) p.alias_scale = sc;
    } else {
      start = T.row_lo * p.hs;
      end = (T.row_hi + 1) * p.hs;
      if (vec) { start &= ~3; end = (end + 3) & ~3; }
      if (end > cells) end = cells;
    }
    p.plane_start[sc] = start;
    p.plane_len[sc] = end - start;
    p.plane_off[sc] = off;
    int split = end - start;
    if (y_split > 0 && y_split < p.hs) {
      const int last = T.identity ? y_split * p.hs : (T.j1[y_split - 1] + 1) * p.hs;  // first raw cell rows < y_split never read
      split = last - start;
      if (vec) split = (split + 3) & ~3;
      if (split > end - start) split = end - start;
      if (split < 0) split = 0;
    }
    p.plane_split[sc] = split;
    off += (end - start + 3) & ~3;
  }
  if (p.alias_scale >= 0) {
    p.sum_off = p.plane_off[p.alias_scale];
  } else {
    p.sum_off = off;
    off += (cells + 3) & ~3;
  }
  p.smem_floats = off;
  p.y_split = (y_split > 0 && y_split < p.hs) ? y_split : p.hs;
}

constexpr int kPostMaxThreads = 512;
constexpr int kPostMaxWarps = kPostMaxThreads / 32;
constexpr int kQuadPar = 32;   // up to this many: one thread per cell / per candidate
constexpr int kQuadCap = 192;  // survivor quads kept in the list; more than that (flat maps) takes the full scan

// threads per (frame, joint) block: `rows` heat-map rows per pass, one thread per cell of those rows
inline int post_threads(int hs, int rows) {
  int t = (rows * hs + 31) & ~31;
  if (t > kPostMaxThreads) t = kPostMaxThreads;
  if (t < 64) t = 64;  // hs <= kMaxHm = 64 cells per row; the gather uses up to 12 * kMaxScales = 48 threads
  return t;
}

// 1/s-resized (float32, cv2 arithmetic: separate mul/add) + cropped value of raw planar map `m` at cell (y, x).
__device__ __forceinline__ float scaled_cell(const float* __restrict__ m, int hs, const ScaleTable& T, int y, int x) {
  if (T.identity) return __ldg(m + y * hs + x);
  const float* r0 = m + T.j0[y] * hs;
  const float* r1 = m + T.j1[y] * hs;
  const int x0 = T.i0[x], x1 = T.i1[x];
  const float a0 = T.a0[x], a1 = T.a1[x];
  const float t0 = __fadd_rn(__fmul_rn(__ldg(r0 + x0), a0), __fmul_rn(__ldg(r0 + x1), a1));
  const float t1 = __fadd_rn(__fmul_rn(__ldg(r1 + x0), a0), __fmul_rn(__ldg(r1 + x1), a1));
  return __fadd_rn(__fmul_rn(t0, T.b0[y]), __fmul_rn(t1, T.b1[y]));
}

// Candidate k (0 .. 2*hs-1) of the x8 upsample along one axis: destination index d, source cell i, fraction f.
// Between two source cell centres the EXACT bilinear upsample is affine, so its maximum over the 8 samples of a segment
// sits at the first (f = 1/16) or last (f = 15/16) one; d = 0 stands for the exactly-tied samples 0..3 and
// d = 8*(hs-1)+4 for the last four (SURVEY.md App. C.4), where the first index wins like np.argmax.  The ROUNDED
// upsample is not monotonic on a quad whose corners agree to ~1e-11 relative: an interior sample can then beat or tie
// (at an earlier index) both ends, so step D rescans every sample of the quads near the best candidate.
__device__ __forceinline__ void upsample_candidate(int k, int hs, int* d, int* i, double* f) {
  if (k == 0) { *d = 0; *i = 0; *f = 0.0; return; }
  if (k == 2 * hs - 1) { *d = 8 * (hs - 1) + 4; *i = hs - 1; *f = 0.0; return; }
  const int r = (k - 1) >> 1;
  if ((k - 1) & 1) { *d = 8 * r + 11; *i = r; *f = 0.9375; }
  else             { *d = 8 * r + 4;  *i = r; *f = 0.0625; }
}

// Sample j along one axis of the quad whose first cell is q: the samples with source cell q (d = 8q+4 .. 8q+11,
// f = 1/16 .. 15/16), plus d = 0 (f = 0) ahead of them for q = 0; the last cell has the one sample d = 8(hs-1)+4.
// An axis has 9, 8 or 1 of them (upsample_axis_len); together the quads cover every sample exactly once.
__device__ __forceinline__ int upsample_axis_len(int q, int hs) { return q == hs - 1 ? 1 : q == 0 ? 9 : 8; }
__device__ __forceinline__ void upsample_sample(int q, int j, int hs, int* d, double* f) {
  if (q == hs - 1) { *d = 8 * q + 4; *f = 0.0; return; }
  if (q == 0) {
    if (j == 0) { *d = 0; *f = 0.0; return; }
    --j;
  }
  *d = 8 * q + 4 + j;
  *f = (double)(2 * j + 1) * 0.0625;
}

// OpenCV+IPP's float64 x8 upsample at fractions (fy, fx) inside the source quad (s00 s01 / s10 s11): fma per axis
__device__ __forceinline__ double upsample_quad(double s00, double s01, double s10, double s11, double fy, double fx) {
  const double h0 = __fma_rn(__dsub_rn(s01, s00), fx, s00);
  const double h1 = __fma_rn(__dsub_rn(s11, s10), fx, s10);
  return __fma_rn(__dsub_rn(h1, h0), fy, h0);
}

// Rounding of upsample_quad against the exact bilinear value, relative to M = the largest |corner|: each difference
// errs by <= u * 2M (u = 2^-53), each row fma by <= 2uM + u(M + 2uM), the column step adds <= 2uM + uM: in all
// < 6.01 uM.  The window 2e = 2^-49 M (e = 8uM) keeps a further ~4uM for the rounding of `best - 2e` itself.
// A sample's exact value is at most its quad's best exact candidate (the exact upsample is affine per axis), so a
// sample that ties or beats the best COMPUTED candidate B lies in a quad whose best computed candidate is >= B - 2e.
// A quad with four equal corners rounds every sample to that value; its first sample is a candidate already.
__device__ __forceinline__ bool quad_needs_scan(double e00, double e01, double e10, double e11, double cand, double b) {
  const double m = fmax(fmax(fabs(e00), fabs(e01)), fmax(fabs(e10), fabs(e11)));
  return !(e00 == e01 && e00 == e10 && e00 == e11) && cand >= b - m * 0x1p-49;
}

__device__ __forceinline__ void cp_async_16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_but_one() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

// The part of a 1-euro step that depends on the clock only (OneEuroFilter.py:64-67 and the derivative's alpha,
// :69-70): it can run while the value is still being computed.  Same operations as oef_step, in the same order.
struct FilterPrep { double freq, te, a_d; };
__device__ __forceinline__ FilterPrep oef_prepare(const FilterState& st, const FilterCfg& cfg, double t) {
  FilterPrep f;
  f.freq = st.freq;
  if (st.has_time && st.lasttime != 0.0 && t != 0.0) f.freq = __ddiv_rn(1.0, __dsub_rn(t, st.lasttime));
  f.te = __ddiv_rn(1.0, f.freq);
  const double tau = __ddiv_rn(1.0, __dmul_rn(6.283185307179586, cfg.dcutoff));
  f.a_d = __ddiv_rn(1.0, __dadd_rn(1.0, __ddiv_rn(tau, f.te)));
  return f;
}
__device__ __forceinline__ double oef_finish(FilterState& st, const FilterCfg& cfg, const FilterPrep& f, double x, double t,
                                             bool x_is_f32) {
  st.freq = f.freq;
  st.lasttime = t;
  st.has_time = 1;
  double dx = 0.0;
  if (st.has_prev) {
    const double diff = x_is_f32 ? (double)__fsub_rn((float)x, (float)st.prev) : __dsub_rn(x, st.prev);
    dx = __dmul_rn(diff, st.freq);
  }
  const double edx = st.has_prev ? __dadd_rn(__dmul_rn(f.a_d, dx), __dmul_rn(__dsub_rn(1.0, f.a_d), st.s_dx)) : dx;
  const double cutoff = __dadd_rn(cfg.mincutoff, __dmul_rn(cfg.beta, fabs(edx)));
  const double tau = __ddiv_rn(1.0, __dmul_rn(6.283185307179586, cutoff));
  const double a = __ddiv_rn(1.0, __dadd_rn(1.0, __ddiv_rn(tau, f.te)));
  const double sm = st.has_prev ? __dadd_rn(__dmul_rn(a, x), __dmul_rn(__dsub_rn(1.0, a), st.s_x)) : x;
  st.prev = x;
  st.s_x = sm;
  st.s_dx = edx;
  st.has_prev = 1;
  return sm;
}

// ---- step E's location-map gather and rescale, shared by postprocess_kernel and sequence_filter_kernel
// utils.hm_pt_interp_bilinear (utils.py:58-79) at a filtered joint (py, px) in box pixels: the heat-map cells around it
// and the UNCLAMPED bilinear weights (a point below 3.5 extrapolates, one at or above 8(hs-1)+3.5 gives exactly 0).
struct GatherPoint {
  double sx, sy;
  int x0, y0, x1, y1;
};
__device__ __forceinline__ GatherPoint gather_point(double py, double px, int hs) {
  GatherPoint g;
  g.sx = __dsub_rn(__dmul_rn(__dadd_rn(px, 0.5), 0.125), 0.5);  // / 8 exactly
  g.sy = __dsub_rn(__dmul_rn(__dadd_rn(py, 0.5), 0.125), 0.5);
  int x0 = (int)g.sx, y0 = (int)g.sy;  // truncation toward zero, like int()
  x0 = min(max(x0, 0), hs - 1);        // memory safety only: filtered joints stay inside the box
  y0 = min(max(y0, 0), hs - 1);
  g.x0 = x0; g.y0 = y0;
  g.x1 = min(x0 + 1, hs - 1); g.y1 = min(y0 + 1, hs - 1);
  return g;
}

// gather_value and gather_combine are sequence_filter_kernel's; postprocess_kernel keeps the same arithmetic inline,
// since routing it through them changes that kernel's SASS at MASK = -1.
// Item i (0 .. 12*NS-1) of a joint's gather: scale i % NS of cell (i / NS) & 3 (bit 1: row y1, bit 0: column x1) of
// location map i / (4*NS) (x, y, z), resampled like the heat maps.
template <int NS>
__device__ __forceinline__ float gather_value(const PostParams& p, int hs, int cells, int frame, int joint, int i,
                                             const GatherPoint& g) {
  const int sc = i % NS;
  const int cell = (i / NS) & 3;
  const int map = i / (4 * NS);
  const float* m = p.maps + ((size_t)(frame * NS + sc) * 84 + kJoints * (1 + map) + joint) * cells;
  return scaled_cell(m, hs, p.tables[sc], (cell & 2) ? g.y1 : g.y0, (cell & 1) ? g.x1 : g.x0);
}

// Map `map`'s 4 cells x NS scales (items[(map * 4 + cell) * NS + sc], as gather_value numbers them) -> the x100 sample in mm:
// float64 sum over the scales in order, / NS, bilinear with the weights of `g`, float32 store.
template <int NS>
__device__ __forceinline__ float gather_combine(const float* items, int map, const GatherPoint& g) {
  double v[4];
#pragma unroll
  for (int cell = 0; cell < 4; ++cell) {
    double acc = 0.0;
    for (int sc = 0; sc < NS; ++sc) acc = __dadd_rn(acc, (double)items[(map * 4 + cell) * NS + sc]);
    // an exact scaling for 1, 2 or 4 scales, bit-identical to the division
    v[cell] = NS == 1 ? acc : NS == 2 ? __dmul_rn(acc, 0.5) : NS == 4 ? __dmul_rn(acc, 0.25) : __ddiv_rn(acc, (double)NS);
  }
  const double wx1 = __dsub_rn((double)g.x1, g.sx), wx0 = __dsub_rn(g.sx, (double)g.x0);
  const double wy1 = __dsub_rn((double)g.y1, g.sy), wy0 = __dsub_rn(g.sy, (double)g.y0);
  const double value0 = __dadd_rn(__dmul_rn(wx1, v[0]), __dmul_rn(wx0, v[1]));
  const double value1 = __dadd_rn(__dmul_rn(wx1, v[2]), __dmul_rn(wx0, v[3]));
  const double val = __dadd_rn(__dmul_rn(wy1, value0), __dmul_rn(wy0, value1));
  return __double2float_rn(__dmul_rn(val, 100.0));
}

// Coordinate c (0 row, 1 col) of a filtered joint in box pixels -> input pixels (estimator.py:138-139; + the crop
// origin for tracked streams, run_estimator.py:104-105).
__device__ __forceinline__ double rescale_joint(const PostParams& p, int frame, int c, double jb) {
  double off = (c == 0) ? (double)p.off_y : (double)p.off_x, scaler = p.scaler;
  double v2;
  if (p.geoms != nullptr) {
    const FrameGeom g = p.geoms[frame];
    off = (c == 0) ? (double)g.off_y : (double)g.off_x;
    scaler = g.scaler;
    v2 = __ddiv_rn(__dsub_rn(jb, off), scaler);
    v2 = __dadd_rn(v2, (c == 0) ? (double)g.y : (double)g.x);
  } else {
    v2 = __ddiv_rn(__dsub_rn(jb, off), scaler);
  }
  return v2;
}

// grid = n_frames * 21 blocks; block (frame, joint), thread = one cell of the `rpp` heat-map rows a pass covers.
//
//  A. the raw heat-map planes of every scale go to shared memory with 16-byte cp.async (the only HBM traffic that
//     scales with the map: 4 * hs * hs bytes per scale);
//  B. one float32 pass: cv2-exact resized value of every scale, float32 sum over the scales per cell, the largest
//     cell.  The float32 sum differs from the reference's float64 accumulation by < n_scales * 2^-24 relative;
//  C. a lower bound on the maximum of the x8 upsample from the 4 x 4 upsample candidates around the largest cell; every
//     cell below (bound - 1e-6 * largest |sum|) provably cannot belong to the source quad of the argmax (an upsampled
//     value is a convex combination of its quad), so only the quads around the few remaining cells survive;
//  D. the survivors are evaluated EXACTLY as the reference does (float64 accumulation over the scales, /= n,
//     OpenCV+IPP's fma upsample), ties to the first index like np.argmax: first their candidates (upsample_candidate),
//     then every sample of the quads whose best candidate is within the rounding window of the block's best one
//     (quad_needs_scan; usually just the winning quad).  Pruning only removes samples that cannot win, so the result
//     equals the exhaustive float64 scan bit for bit; if more than kQuadCap quads survive (flat or saturated maps)
//     every quad that passes the same test is evaluated in place;
//  E. 2D 1-euro filters, location-map gather at the FILTERED point, and -- in the last block of the frame to arrive --
//     root subtraction, 3D filters and the rescale to input pixels.
#define POST_TRACE(i) do { if (p.trace != nullptr && threadIdx.x == 0) p.trace[(size_t)blockIdx.x * 16 + (i)] = globaltimer_ns(); } while (0)
// RAW_ONLY: steps A-D only, ending with raw_argmax (the argmax launch of a sequence call, sequence_filter_kernel does
// the rest); no filter state, scratch or frame counter is touched.
// SCORES: step D's best value -- the reference's upsampled float64 heat-map at the raw argmax, i.e. the joint's
// confidence -- goes to p.scores as well.
template <int NS, int MASK, bool RAW_ONLY = false, bool SCORES = false>  // MASK >= 0: the identity mask (PostParams::identity_mask) is this compile-time constant
__global__ void __launch_bounds__(kPostMaxThreads, 2) postprocess_kernel(const __grid_constant__ PostParams p) {
  extern __shared__ float4 s_dyn4[];
  float* s_dyn = reinterpret_cast<float*>(s_dyn4);
  __shared__ int4 s_rowpk[NS][kMaxHm];  // y-axis resize entries as byte offsets: (j0*hs*4, j1*hs*4, b0, b1)
  __shared__ int4 s_colpk[NS][kMaxHm];  // x-axis entries: (i0*4, i1*4, a0, a1) -- the exact path looks them up per quad
  __shared__ float s_wmax[kPostMaxWarps], s_wmin[kPostMaxWarps], s_wamax[kPostMaxWarps];
  __shared__ int s_widx[kPostMaxWarps];
  __shared__ double s_bval[kPostMaxWarps];
  __shared__ int s_bidx[kPostMaxWarps];
  __shared__ unsigned short s_quads[kQuadCap];
  __shared__ int s_nq;
  __shared__ double s_pt[2];
  __shared__ float s_gather[12 * kMaxScales];
  __shared__ int s_is_last;
  __shared__ __align__(16) FilterState s_st2[2];
  __shared__ double s_t2;
  __shared__ double s_exact[kQuadPar * 4];
  __shared__ double s_prep[2][3];
  __shared__ __align__(16) FilterState s_st3[3];
  __shared__ double s_t3;
  __shared__ int s_sid;

  const int frame = blockIdx.x / kJoints;
  const int joint = blockIdx.x - frame * kJoints;
  const int hs = p.hs, S = p.S;
  constexpr int ns = NS;  // p.n_scales
  const int idmask = MASK >= 0 ? MASK : p.identity_mask;
  const int cells = hs * hs, nc = 2 * hs;
  const int tid = threadIdx.x, nthreads = blockDim.x;
  const int warp_id = tid >> 5, lane_id = tid & 31, nwarps = nthreads >> 5;
  const int rpp = nthreads / hs;          // rows per pass (host guarantees nthreads >= hs)
  const bool act = tid < rpp * hs;
  const int ro = tid / hs, x = tid - ro * hs;
  POST_TRACE(0);
  if (p.trace != nullptr && tid == 0) p.trace[(size_t)blockIdx.x * 16 + 11] = (unsigned long long)clock64();

  // per-thread column entries of the resize tables, the row entries to shared memory (static data: may be read before
  // the predecessor has finished)
  int cx0[NS], cx1[NS];
  float ca0[NS], ca1[NS];
#pragma unroll
  for (int sc = 0; sc < NS; ++sc) {
    cx0[sc] = cx1[sc] = 0;
    ca0[sc] = ca1[sc] = 0.f;
    if (!((idmask >> sc) & 1)) {
      const ScaleTable& T = p.tables[sc];
      cx0[sc] = T.i0[x] * 4; cx1[sc] = T.i1[x] * 4;  // byte offsets inside a row
      ca0[sc] = T.a0[x]; ca1[sc] = T.a1[x];
      for (int i = tid; i < hs; i += nthreads) {
        int4 rp = T.rowpk[i];
        rp.x *= 4; rp.y *= 4;
        s_rowpk[sc][i] = rp;
        s_colpk[sc][i] = make_int4(T.i0[i] * 4, T.i1[i] * 4, __float_as_int(T.a0[i]), __float_as_int(T.a1[i]));
      }
    }
  }
  if (tid == 0) s_nq = 0;
  pdl_launch_dependents();
  pdl_wait();  // the maps come from the last conv
  POST_TRACE(1);

  // ---- A. stage the planes, in two cp.async groups: what rows [0, y_split) of the sum pass read, then the rest
  const char* pl[NS];  // byte pointer such that pl[sc] + 4 * (absolute raw cell) is that cell
#pragma unroll
  for (int part = 0; part < 2; ++part) {
#pragma unroll
    for (int sc = 0; sc < NS; ++sc) {
      const float* g = p.maps + ((size_t)(frame * ns + sc) * 84 + joint) * cells + p.plane_start[sc];
      float* d = s_dyn + p.plane_off[sc];
      const int lo = part == 0 ? 0 : p.plane_split[sc], hi = part == 0 ? p.plane_split[sc] : p.plane_len[sc];
      if ((cells & 3) == 0) {
        for (int i = lo + tid * 4; i < hi; i += nthreads * 4) cp_async_16(d + i, g + i);
      } else {
        for (int i = lo + tid; i < hi; i += nthreads) d[i] = __ldg(g + i);
      }
      pl[sc] = reinterpret_cast<const char*>(d - p.plane_start[sc]);
    }
    if (part == 0) {
      // the two 2D filters of this joint: state fetched now, used after the argmax
      static_assert(sizeof(FilterState) == 48, "three 16-byte pieces per filter state");
      if (tid < 6 && !RAW_ONLY && p.filters_on) {
        const int sid = p.stream_ids[frame];
        cp_async_16(reinterpret_cast<char*>(s_st2) + tid * 16,
                    reinterpret_cast<const char*>(p.st2d + ((size_t)sid * kJoints + joint) * 2) + tid * 16);
        if (tid == 0) { s_sid = sid; s_t2 = p.t2d[frame]; s_t3 = p.t3d[frame]; }
      } else if (tid < 15 && !RAW_ONLY && p.filters_on) {  // this joint's three 3D filter states (144 contiguous bytes)
        const int sid = p.stream_ids[frame];
        cp_async_16(reinterpret_cast<char*>(s_st3) + (tid - 6) * 16,
                    reinterpret_cast<const char*>(p.st3d + ((size_t)sid * kJoints + joint) * 3) + (tid - 6) * 16);
      }
    }
    cp_async_commit();
  }

  // ---- B. float32 sums over the scales (estimator.py:105-129 in float32), largest cell
  float* s_sum = s_dyn + p.sum_off;
  float tmax = -INFINITY, tmin = INFINITY, tvmax = 0.f, chk = 0.f;
  int ty = 0;
  auto sum_rows = [&](int y_begin, int y_end) {  // y_begin is a multiple of rpp
#pragma unroll 2
    for (int y = y_begin + ro; y < y_end; y += rpp) {
      const int cb = (y * hs + x) * 4;
      float s = 0.f;
#pragma unroll
      for (int sc = 0; sc < NS; ++sc) {
        float v;
        if ((idmask >> sc) & 1) {
          v = *reinterpret_cast<const float*>(pl[sc] + cb);
        } else {  // cv2 float32 resize arithmetic: separate multiplies and adds
          const int4 rp = s_rowpk[sc][y];
          const char* c0 = pl[sc] + cx0[sc];
          const char* c1 = pl[sc] + cx1[sc];
          const float t0 = __fadd_rn(__fmul_rn(*reinterpret_cast<const float*>(c0 + rp.x), ca0[sc]),
                                     __fmul_rn(*reinterpret_cast<const float*>(c1 + rp.x), ca1[sc]));
          const float t1 = __fadd_rn(__fmul_rn(*reinterpret_cast<const float*>(c0 + rp.y), ca0[sc]),
                                     __fmul_rn(*reinterpret_cast<const float*>(c1 + rp.y), ca1[sc]));
          v = __fadd_rn(__fmul_rn(t0, __int_as_float(rp.z)), __fmul_rn(t1, __int_as_float(rp.w)));
        }
        s = sc == 0 ? v : __fadd_rn(s, v);
        if (NS > 2) tvmax = fmaxf(tvmax, fabsf(v));  // partial sums of three or more terms can exceed the final |s|
      }
      *reinterpret_cast<float*>(reinterpret_cast<char*>(s_sum) + cb) = s;  // may overwrite pl[alias_scale]'s cell: this thread was its only reader
      chk = __fmaf_rn(s, 0.f, chk);  // NaN as soon as one s is NaN or Inf (a non-finite v always makes s non-finite)
      if (s > tmax) { tmax = s; ty = y; }
      tmin = fminf(tmin, s);
    }
  };
  cp_async_wait_but_one();
  __syncthreads();
  POST_TRACE(2);
  if (act) sum_rows(0, p.y_split);
  cp_async_wait_all();
  __syncthreads();
  if (act) sum_rows(p.y_split, hs);
  const int bad = chk != chk;
  POST_TRACE(3);
  float bmax = tmax, bmin = tmin, bvmax = tvmax;
  int bidx = ty * hs + x;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bmax, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bidx, o);
    if (ov > bmax) { bmax = ov; bidx = oi; }
    bmin = fminf(bmin, __shfl_xor_sync(0xffffffffu, bmin, o));
    if (NS > 2) bvmax = fmaxf(bvmax, __shfl_xor_sync(0xffffffffu, bvmax, o));
  }
  if (lane_id == 0) { s_wmax[warp_id] = bmax; s_widx[warp_id] = bidx; s_wmin[warp_id] = bmin; s_wamax[warp_id] = bvmax; }
  // fp16 activations overflow at 65504: an Inf / NaN anywhere in the CNN almost surely reaches the maps.  Count it (the
  // host turns a non-zero count into an error) instead of returning joints computed from garbage.
  const int any_bad = __syncthreads_or(bad);
  if (any_bad && tid == 0 && p.nonfinite != nullptr) {
    atomicAdd(p.nonfinite, 1u);
    if (p.nonfinite_flag != nullptr) *reinterpret_cast<volatile unsigned int*>(p.nonfinite_flag) = 1u;
  }
  bmax = s_wmax[0]; bidx = s_widx[0]; bmin = s_wmin[0]; bvmax = s_wamax[0];
  for (int w = 1; w < nwarps; ++w) {
    if (s_wmax[w] > bmax) { bmax = s_wmax[w]; bidx = s_widx[w]; }
    bmin = fminf(bmin, s_wmin[w]);
    bvmax = fmaxf(bvmax, s_wamax[w]);
  }
  const float bamax = fmaxf(fmaxf(fabsf(bmax), fabsf(bmin)), bvmax);  // largest |s| (and |v| for three or more scales)
  POST_TRACE(4);

  // ---- C. bound from the 4 x 4 candidates around the largest cell (every warp computes the same value)
  float thr;
  {
    const int r0 = bidx / hs, c0 = bidx - r0 * hs;
    const int ky0 = max(2 * r0 - 1, 0), kx0 = max(2 * c0 - 1, 0);
    const int ky = min(ky0 + ((lane_id >> 2) & 3), nc - 1), kx = min(kx0 + (lane_id & 3), nc - 1);
    int dy, dx, iy, ix;
    double fy, fx;
    upsample_candidate(ky, hs, &dy, &iy, &fy);
    upsample_candidate(kx, hs, &dx, &ix, &fx);
    const int iy1 = min(iy + 1, hs - 1), ix1 = min(ix + 1, hs - 1);
    double v = upsample_quad((double)s_sum[iy * hs + ix], (double)s_sum[iy * hs + ix1], (double)s_sum[iy1 * hs + ix],
                             (double)s_sum[iy1 * hs + ix1], fy, fx);
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    // margin: the float32 summation errs by < 2^-24 |s| at two scales and by < (n-1) * 2^-24 * n * max|v| per cell at
    // n >= 3 (on both sides of the comparison: 1.5e-6 * max|v| at n = 4), the upsample's own rounding by 1e-16
    thr = any_bad ? -INFINITY : __double2float_rd(v - (double)bamax * (1e-6 * ns));
  }
  // Cells that may belong to the argmax's quad -> the (up to four) quads around each, filtered once more: every
  // candidate of a quad has fractions in [0, 15/16] on both axes and the upsample is affine in each, so its largest
  // candidate is at most the largest of the four corner values of that box -- a far tighter cap than the quad's largest
  // cell (with random-init maps the plain cell test left 20 quads per joint in the median, 170 at worst).  A quad is
  // listed by the first of its cells (row-major) that passed the cell test.
  if (act && tmax >= thr) {
    unsigned long long rows = 0;  // bit k: this thread's k-th cell passes (hs <= 64 rows)
    int k = 0;
#pragma unroll 4
    for (int y = ro; y < hs; y += rpp, ++k) rows |= (unsigned long long)(s_sum[y * hs + x] >= thr) << k;
    while (rows) {
      const int y = ro + (__ffsll((long long)rows) - 1) * rpp;
      rows &= rows - 1;
      for (int qy = max(y - 1, 0); qy <= y; ++qy)
        for (int qx = max(x - 1, 0); qx <= x; ++qx) {
          const int qy1 = min(qy + 1, hs - 1), qx1 = min(qx + 1, hs - 1);
          const float s00 = s_sum[qy * hs + qx], s01 = s_sum[qy * hs + qx1], s10 = s_sum[qy1 * hs + qx], s11 = s_sum[qy1 * hs + qx1];
          // an earlier cell of the quad passed the cell test too: that one lists it
          const bool first = (qy == y && qx == x) || (qy == y && !(s00 >= thr)) ||
                             (qy != y && qx == x && !(s00 >= thr) && !(s01 >= thr && qx1 != qx)) ||
                             (qy != y && qx != x && !(s00 >= thr) && !(s01 >= thr) && !(s10 >= thr));
          if (!first) continue;
          const float f = 0.9375f;
          const float h0 = fmaf(s01 - s00, f, s00), h1 = fmaf(s11 - s10, f, s10);
          const float cap = fmaxf(fmaxf(s00, h0), fmaxf(fmaf(s10 - s00, f, s00), fmaf(h1 - h0, f, h0)));
          // float32 evaluation of the cap: a few 2^-24 relative, far inside the margin already taken off thr
          if (!(cap >= thr)) continue;
          const int slot = atomicAdd(&s_nq, 1);
          if (slot < kQuadCap) s_quads[slot] = (unsigned short)(qy * hs + qx);
        }
    }
  }
  __syncthreads();
  POST_TRACE(5);

  // ---- D. exact float64 evaluation of the survivors (utils.py:153-175 on estimator.py:105-129's hm_avg)
  auto exact_cell = [&](int y, int xx) -> double {
    const int c = y * hs + xx;
    double acc = 0.0;
#pragma unroll
    for (int sc = 0; sc < NS; ++sc) {
      {
        float v;
        if ((idmask >> sc) & 1) {
          // the staged plane of alias_scale now holds the sums: its raw value comes from L2
          v = sc == p.alias_scale ? __ldg(p.maps + ((size_t)(frame * ns + sc) * 84 + joint) * cells + c)
                                  : *reinterpret_cast<const float*>(pl[sc] + c * 4);
        } else {
          const int4 rp = s_rowpk[sc][y], cp = s_colpk[sc][xx];
          const char* r0 = pl[sc] + rp.x;
          const char* r1 = pl[sc] + rp.y;
          const float a0 = __int_as_float(cp.z), a1 = __int_as_float(cp.w);
          const float t0 = __fadd_rn(__fmul_rn(*reinterpret_cast<const float*>(r0 + cp.x), a0), __fmul_rn(*reinterpret_cast<const float*>(r0 + cp.y), a1));
          const float t1 = __fadd_rn(__fmul_rn(*reinterpret_cast<const float*>(r1 + cp.x), a0), __fmul_rn(*reinterpret_cast<const float*>(r1 + cp.y), a1));
          v = __fadd_rn(__fmul_rn(t0, __int_as_float(rp.z)), __fmul_rn(t1, __int_as_float(rp.w)));
        }
        acc = __dadd_rn(acc, (double)v);
      }
    }
    // hm_avg /= len(scales): for 1, 2 or 4 scales the quotient is an exact scaling, bit-identical to the division
    return ns == 1 ? acc : ns == 2 ? __dmul_rn(acc, 0.5) : ns == 4 ? __dmul_rn(acc, 0.25) : __ddiv_rn(acc, (double)ns);
  };
  double best = -INFINITY;
  int best_idx = 0x7fffffff;
  auto take = [&](double v, int idx) {
    if (v > best || (v == best && idx < best_idx)) { best = v; best_idx = idx; }
  };
  auto warp_best = [&]() {  // (best, best_idx) of the warp in every lane
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ov = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, best_idx, o);
      if (ov > best || (ov == best && oi < best_idx)) { best = ov; best_idx = oi; }
    }
  };
  // samples first, first + step, ... (row-major) of every sample of quad (qy, qx)
  auto scan_quad = [&](int qy, int qx, double e00, double e01, double e10, double e11, int first, int step) {
    const int nx = upsample_axis_len(qx, hs), n = upsample_axis_len(qy, hs) * nx;
    for (int i = first; i < n; i += step) {
      const int jy = i / nx;
      int dy, dx;
      double fy, fx;
      upsample_sample(qy, jy, hs, &dy, &fy);
      upsample_sample(qx, i - jy * nx, hs, &dx, &fx);
      take(upsample_quad(e00, e01, e10, e11, fy, fx), dy * S + dx);
    }
  };
  // quad = cells (qy, qy+1) x (qx, qx+1), clamped; its axis candidates: cell 0: k = 0..2, cell i: k = 2i+1, 2i+2, the
  // last cell: k = 2*hs-1.  First look (b = -INFINITY): the candidates; returns whether the quad is within the window
  // of this thread's best so far, a superset of the quads within the window of the block's best.  Second look (b = the
  // block's best candidate): the candidates again, and every sample if the quad is within the window of b.
  auto eval_quad = [&](int qy, int qx, double b) -> bool {
    const int qy1 = min(qy + 1, hs - 1), qx1 = min(qx + 1, hs - 1);
    const double e00 = exact_cell(qy, qx);
    const double e01 = qx1 == qx ? e00 : exact_cell(qy, qx1);
    const double e10 = qy1 == qy ? e00 : exact_cell(qy1, qx);
    const double e11 = qy1 == qy ? e01 : (qx1 == qx ? e10 : exact_cell(qy1, qx1));
    const int ky_lo = qy == 0 ? 0 : 2 * qy + 1, ky_hi = qy == hs - 1 ? nc - 1 : 2 * qy + 2;
    const int kx_lo = qx == 0 ? 0 : 2 * qx + 1, kx_hi = qx == hs - 1 ? nc - 1 : 2 * qx + 2;
    double cand = -INFINITY;
    for (int ky = ky_lo; ky <= ky_hi; ++ky) {
      int dy, iy;
      double fy;
      upsample_candidate(ky, hs, &dy, &iy, &fy);
      for (int kx = kx_lo; kx <= kx_hi; ++kx) {
        int dx, ix;
        double fx;
        upsample_candidate(kx, hs, &dx, &ix, &fx);
        const double v = upsample_quad(e00, e01, e10, e11, fy, fx);
        cand = fmax(cand, v);
        take(v, dy * S + dx);
      }
    }
    if (b == -INFINITY) return quad_needs_scan(e00, e01, e10, e11, cand, best);
    if (quad_needs_scan(e00, e01, e10, e11, cand, b)) scan_quad(qy, qx, e00, e01, e10, e11, 0, 1);
    return false;
  };
  const int nq = s_nq;
  const bool one_warp = nq <= kQuadPar;  // the usual case: a handful of quads
  if (p.trace != nullptr && tid == 0) p.trace[(size_t)blockIdx.x * 16 + 13] = (unsigned long long)nq;
  // Five lanes of warp 1 advance the clock-only part (four dependent divisions, ~0.5 us each here) of this joint's two 2D
  // and three 3D filter steps while warp 0 evaluates the quads; the 3D ones go to global scratch for the frame's tail.
  if (!RAW_ONLY && p.filters_on && tid >= 32 && tid < 37) {
    const int k = tid - 32;
    if (k < 2) {
      const FilterPrep f = oef_prepare(s_st2[k], p.cfg2d, s_t2);
      s_prep[k][0] = f.freq; s_prep[k][1] = f.te; s_prep[k][2] = f.a_d;
    } else {
      const FilterPrep f = oef_prepare(s_st3[k - 2], p.cfg3d, s_t3);
      double* o = p.prep3 + ((size_t)(frame * kJoints + joint) * 3 + (k - 2)) * 3;
      o[0] = f.freq; o[1] = f.te; o[2] = f.a_d;
    }
  }
  unsigned second = 0;  // bit k: the k-th quad this thread evaluated needs a second look (k < hs / rpp <= 32)
  if (one_warp) {
    // every cell of every surviving quad on its own thread, then every candidate on its own lane of warp 0
    for (int i = tid; i < nq * 4; i += nthreads) {
      const int q = s_quads[i >> 2];
      const int qy = q / hs, qx = q - qy * hs;
      s_exact[i] = exact_cell(min(qy + ((i >> 1) & 1), hs - 1), min(qx + (i & 1), hs - 1));
    }
    __syncthreads();
    if (p.trace != nullptr && tid == 0) p.trace[(size_t)blockIdx.x * 16 + 14] = globaltimer_ns();
    if (warp_id == 0) {
      // candidate slot -> its value; returns false for the slots a border quad does not have
      auto candidate = [&](int i, double* v, int* idx) -> bool {
        const int qi = i / 9, slot = i - qi * 9;
        const int q = s_quads[qi];
        const int qy = q / hs, qx = q - qy * hs;
        const int ky = (qy == 0 ? 0 : 2 * qy + 1) + slot / 3, kx = (qx == 0 ? 0 : 2 * qx + 1) + slot % 3;
        if (ky > (qy == hs - 1 ? nc - 1 : 2 * qy + 2) || kx > (qx == hs - 1 ? nc - 1 : 2 * qx + 2)) return false;
        int dy, dx, iy, ix;
        double fy, fx;
        upsample_candidate(ky, hs, &dy, &iy, &fy);
        upsample_candidate(kx, hs, &dx, &ix, &fx);
        *v = upsample_quad(s_exact[qi * 4], s_exact[qi * 4 + 1], s_exact[qi * 4 + 2], s_exact[qi * 4 + 3], fy, fx);
        *idx = dy * S + dx;
        return true;
      };
      for (int i = lane_id; i < nq * 9; i += 32) {
        double v;
        int idx;
        if (candidate(i, &v, &idx)) take(v, idx);
      }
      warp_best();
      // the quads within the window of the best candidate (bit qi), then all their samples on the lanes of the warp
      unsigned scan = 0;
      for (int i = lane_id; i < nq * 9; i += 32) {
        double v;
        int idx;
        const int qi = i / 9;
        if (candidate(i, &v, &idx) &&
            quad_needs_scan(s_exact[qi * 4], s_exact[qi * 4 + 1], s_exact[qi * 4 + 2], s_exact[qi * 4 + 3], v, best))
          scan |= 1u << qi;
      }
      scan = __reduce_or_sync(0xffffffffu, scan);
      if (scan) {
        do {
          const int qi = __ffs(scan) - 1;
          scan &= scan - 1;
          const int q = s_quads[qi];
          const int qy = q / hs;
          scan_quad(qy, q - qy * hs, s_exact[qi * 4], s_exact[qi * 4 + 1], s_exact[qi * 4 + 2], s_exact[qi * 4 + 3],
                    lane_id, 32);
        } while (scan);
        warp_best();
      }
      if (lane_id == 0) { s_bval[0] = best; s_bidx[0] = best_idx; }
    }
  } else {
    if (nq <= kQuadCap) {
      for (int i = tid, k = 0; i < nq; i += nthreads, ++k) {
        const int q = s_quads[i];
        const int qy = q / hs;
        if (eval_quad(qy, q - qy * hs, -INFINITY)) second |= 1u << k;
      }
    } else if (act) {
      for (int y = ro, k = 0; y < hs; y += rpp, ++k) {
        const int y1 = min(y + 1, hs - 1), x1 = min(x + 1, hs - 1);
        const float m4 = fmaxf(fmaxf(s_sum[y * hs + x], s_sum[y * hs + x1]), fmaxf(s_sum[y1 * hs + x], s_sum[y1 * hs + x1]));
        if (m4 >= thr && eval_quad(y, x, -INFINITY)) second |= 1u << k;
      }
    }
    warp_best();
    if (lane_id == 0) { s_bval[warp_id] = best; s_bidx[warp_id] = best_idx; }
    if (__syncthreads_or(second != 0)) {  // block-uniform
      double b = s_bval[0];
      for (int w = 1; w < nwarps; ++w) b = fmax(b, s_bval[w]);
      __syncthreads();  // every warp has read s_bval
      while (second) {
        const int k = __ffs(second) - 1;
        second &= second - 1;
        if (nq <= kQuadCap) {
          const int q = s_quads[tid + k * nthreads];
          const int qy = q / hs;
          eval_quad(qy, q - qy * hs, b);
        } else {
          eval_quad(ro + k * rpp, x, b);
        }
      }
      warp_best();
      if (lane_id == 0) { s_bval[warp_id] = best; s_bidx[warp_id] = best_idx; }
      __syncthreads();
    }
  }
  POST_TRACE(6);

  // ---- E. 2D filters, then the location-map gather at the FILTERED point (estimator.py:132-134)
  if (tid < 32) {
    if (!one_warp) {
      best = s_bval[0]; best_idx = s_bidx[0];
      for (int w = 1; w < nwarps; ++w)
        if (s_bval[w] > best || (s_bval[w] == best && s_bidx[w] < best_idx)) { best = s_bval[w]; best_idx = s_bidx[w]; }
    }
    const int row = best_idx / S, col = best_idx - row * S;
    double coord = (tid == 0) ? (double)row : (double)col;
    if (SCORES && tid == 0) reinterpret_cast<double*>(p.raw_argmax + p.scores_off)[frame * kJoints + joint] = best;
    if (tid < 2) {
      p.raw_argmax[(frame * kJoints + joint) * 2 + tid] = (tid == 0) ? row : col;
      if (!RAW_ONLY && p.filters_on) {
        FilterState st2 = s_st2[tid];
        const FilterPrep f = {s_prep[tid][0], s_prep[tid][1], s_prep[tid][2]};
        coord = oef_finish(st2, p.cfg2d, f, coord, s_t2, false);
        p.st2d[((size_t)s_sid * kJoints + joint) * 2 + tid] = st2;
      }
      if (!RAW_ONLY) p.j2_box[(frame * kJoints + joint) * 2 + tid] = coord;
    }
    const double py = __shfl_sync(0xffffffffu, coord, 0), px = __shfl_sync(0xffffffffu, coord, 1);
    if (tid == 0) { s_pt[0] = py; s_pt[1] = px; }
    POST_TRACE(7);
  }
  if (RAW_ONLY) return;
  __syncthreads();
  // utils.hm_pt_interp_bilinear (utils.py:58-79) on the three averaged location maps.  The 3 maps x 4 cells x n_scales
  // resampled values are fetched by 12*n_scales threads at once (the first version walked them serially in 3 threads
  // and the dependent global loads dominated the kernel); the float64 arithmetic and its order are unchanged.
  {
    const double py = s_pt[0], px = s_pt[1];
    const GatherPoint g = gather_point(py, px, hs);
    // rescale to input pixels: two lanes of warp 1, beside the gather of warp 0
    if (tid >= 32 && tid < 34) {
      const int c = tid - 32;
      const double v2 = rescale_joint(p, frame, c, c == 0 ? py : px);
      p.out2d[(frame * kJoints + joint) * 2 + c] = v2;
      if (p.packed != nullptr) p.packed[(frame * kJoints + joint) * 5 + c] = v2;
    }
    const int items = 12 * ns;
    if (tid < items) {
      const int sc = tid % ns;
      const int cell = (tid / ns) & 3;
      const int map = tid / (4 * ns);
      const float* m = p.maps + ((size_t)(frame * ns + sc) * 84 + kJoints * (1 + map) + joint) * cells;
      const float gv = scaled_cell(m, hs, p.tables[sc], (cell & 2) ? g.y1 : g.y0, (cell & 1) ? g.x1 : g.x0);
      s_gather[tid] = gv;
      if (!(fabsf(gv) <= 3.4028234e38f) && p.nonfinite != nullptr) {
        atomicAdd(p.nonfinite, 1u);
        if (p.nonfinite_flag != nullptr) *reinterpret_cast<volatile unsigned int*>(p.nonfinite_flag) = 1u;
      }
    }
    __syncthreads();
    if (tid < 3) {  // gather_combine's arithmetic, kept inline: through the function the MASK = -1 SASS changes
      double v[4];
#pragma unroll
      for (int cell = 0; cell < 4; ++cell) {
        double acc = 0.0;
        for (int sc = 0; sc < ns; ++sc) acc = __dadd_rn(acc, (double)s_gather[(tid * 4 + cell) * ns + sc]);
        // an exact scaling for 1, 2 or 4 scales, bit-identical to the division
        v[cell] = ns == 1 ? acc : ns == 2 ? __dmul_rn(acc, 0.5) : ns == 4 ? __dmul_rn(acc, 0.25) : __ddiv_rn(acc, (double)ns);
      }
      const double wx1 = __dsub_rn((double)g.x1, g.sx), wx0 = __dsub_rn(g.sx, (double)g.x0);
      const double wy1 = __dsub_rn((double)g.y1, g.sy), wy0 = __dsub_rn(g.sy, (double)g.y0);
      const double value0 = __dadd_rn(__dmul_rn(wx1, v[0]), __dmul_rn(wx0, v[1]));
      const double value1 = __dadd_rn(__dmul_rn(wx1, v[2]), __dmul_rn(wx0, v[3]));
      const double val = __dadd_rn(__dmul_rn(wy1, value0), __dmul_rn(wy0, value1));
      p.j3_raw[(frame * kJoints + joint) * 3 + tid] = __double2float_rn(__dmul_rn(val, 100.0));  // mm, float32 store
    }
  }

  // ---- per-frame tail in the last block to arrive
  POST_TRACE(8);
  __threadfence();
  __syncthreads();
  if (tid == 0) s_is_last = (atomicAdd(&p.frame_counter[frame], 1u) == kJoints - 1);
  __syncthreads();
  POST_TRACE(9);
  if (!s_is_last) return;
  __threadfence();
  if (tid == 0) p.frame_counter[frame] = 0;  // ready for the next launch (no memset node between the conv and this kernel)
  for (int i = tid; i < kJoints * 3; i += nthreads) {
    const int j = i / 3, c = i - j * 3;
    const volatile float* raw = p.j3_raw + frame * kJoints * 3;
    float v = __fsub_rn(raw[j * 3 + c], raw[kRootJoint * 3 + c]);  // joints_3d -= joints_3d[14] (utils.py:218)
    if (p.filters_on) {
      const size_t si = ((size_t)p.stream_ids[frame] * kJoints + j) * 3 + c;
      FilterState st = p.st3d[si];
      const volatile double* pr = p.prep3 + ((size_t)(frame * kJoints + j) * 3 + c) * 3;  // written by joint j's block
      const FilterPrep f = {pr[0], pr[1], pr[2]};
      v = __double2float_rn(oef_finish(st, p.cfg3d, f, (double)v, p.t3d[frame], true));
      p.st3d[si] = st;
    }
    p.out3d[(frame * kJoints + j) * 3 + c] = v;
    if (p.packed != nullptr) p.packed[(frame * kJoints + j) * 5 + 2 + c] = (double)v;
  }
  POST_TRACE(10);
  if (p.trace != nullptr && tid == 0) p.trace[(size_t)blockIdx.x * 16 + 12] = (unsigned long long)clock64();
}
#undef POST_TRACE

// ---------------------------------------------------------------------------------------------------------------
// Sequence calls: a stream id may appear several times in one call, its frames consecutive in time in call order.
// postprocess_kernel<NS, MASK, true> gives every frame's raw argmax (it depends on no other frame); this kernel then
// walks each stream's frames in order through everything that carries state from one frame to the next.  Segment
// table (host: stage_sequence_meta): seg[0] = number of distinct streams n_seg, seg[1 .. n_seg+1] = where each stream's
// frames start in the frame list seg[n_seg + 2 ..], which holds the frame indices of every stream in call order.
// grid = n_frames blocks (the surplus ones return), so the launch does not depend on the composition; block b = the
// b-th distinct stream.  Same arithmetic as postprocess_kernel's step E and frame tail:
//   1. 42 threads, one per (joint, axis), walk the 2D filters and write j2_box, out2d (and packed); 63 other threads
//      walk the clock-only part (FilterPrep) of the 3D filters ahead, into prep3;
//   2. all threads gather the three location maps at the filtered points of every (frame, joint), into j3_raw;
//   3. 63 threads, one per (joint, axis), subtract the root and walk the 3D filters: out3d (and packed).
constexpr int kSeqThreads = 512;
template <int NS>
__global__ void __launch_bounds__(kSeqThreads) sequence_filter_kernel(const __grid_constant__ PostParams p,
                                                                      const int* __restrict__ seg) {
  const int n_seg = seg[0];
  if ((int)blockIdx.x >= n_seg) return;
  const int lo = seg[1 + blockIdx.x], hi = seg[2 + blockIdx.x];
  const int* fr = seg + 2 + n_seg;
  const int sid = p.stream_ids[fr[lo]];
  const int tid = threadIdx.x;
  if (tid < 2 * kJoints) {
    const int joint = tid >> 1, c = tid & 1;
    FilterState st;
    FilterPrep pr;
    if (p.filters_on) {
      st = p.st2d[((size_t)sid * kJoints + joint) * 2 + c];
      pr = oef_prepare(st, p.cfg2d, p.t2d[fr[lo]]);
    }
    for (int k = lo; k < hi; ++k) {
      const int f = fr[k], i = (f * kJoints + joint) * 2 + c;
      double coord = (double)p.raw_argmax[i];
      if (p.filters_on) {
        const double t = p.t2d[f];
        FilterPrep nx = pr;
        if (k + 1 < hi) {  // the next step's clock-only part: independent of this step's value chain
          FilterState clk = st;
          clk.freq = pr.freq; clk.lasttime = t; clk.has_time = 1;
          nx = oef_prepare(clk, p.cfg2d, p.t2d[fr[k + 1]]);
        }
        coord = oef_finish(st, p.cfg2d, pr, coord, t, false);
        pr = nx;
      }
      p.j2_box[i] = coord;
      const double v2 = rescale_joint(p, f, c, coord);
      p.out2d[i] = v2;
      if (p.packed != nullptr) p.packed[(f * kJoints + joint) * 5 + c] = v2;
    }
    if (p.filters_on) p.st2d[((size_t)sid * kJoints + joint) * 2 + c] = st;
  } else if (tid >= 64 && tid < 64 + 3 * kJoints && p.filters_on) {
    const int k3 = tid - 64, joint = k3 / 3, c = k3 - joint * 3;
    FilterState clk = p.st3d[((size_t)sid * kJoints + joint) * 3 + c];
    for (int k = lo; k < hi; ++k) {
      const int f = fr[k];
      const double t = p.t3d[f];
      const FilterPrep pr = oef_prepare(clk, p.cfg3d, t);
      double* o = p.prep3 + ((size_t)(f * kJoints + joint) * 3 + c) * 3;
      o[0] = pr.freq; o[1] = pr.te; o[2] = pr.a_d;
      clk.freq = pr.freq; clk.lasttime = t; clk.has_time = 1;
    }
  }
  __syncthreads();
  // 2. gather: one thread per (frame, joint, map), its 4 cells x NS scales loaded at once
  for (int item = tid; item < (hi - lo) * kJoints * 3; item += blockDim.x) {
    const int k = lo + item / (kJoints * 3), r = item - (k - lo) * (kJoints * 3);
    const int joint = r / 3, map = r - joint * 3;
    const int f = fr[k];
    const GatherPoint g = gather_point(p.j2_box[(f * kJoints + joint) * 2], p.j2_box[(f * kJoints + joint) * 2 + 1], p.hs);
    float v4[4 * NS];
    bool bad = false;
#pragma unroll
    for (int i = 0; i < 4 * NS; ++i) {
      v4[i] = gather_value<NS>(p, p.hs, p.hs * p.hs, f, joint, map * 4 * NS + i, g);
      bad |= !(fabsf(v4[i]) <= 3.4028234e38f);
    }
    if (bad && p.nonfinite != nullptr) {
      atomicAdd(p.nonfinite, 1u);
      if (p.nonfinite_flag != nullptr) *reinterpret_cast<volatile unsigned int*>(p.nonfinite_flag) = 1u;
    }
    p.j3_raw[(f * kJoints + joint) * 3 + map] = gather_combine<NS>(v4, 0, g);
  }
  __syncthreads();
  // 3. root subtraction (utils.py:218) and the 3D filters in frame order
  if (tid < 3 * kJoints) {
    const int joint = tid / 3, c = tid - joint * 3;
    FilterState st;
    if (p.filters_on) st = p.st3d[((size_t)sid * kJoints + joint) * 3 + c];
    for (int k = lo; k < hi; ++k) {
      const int f = fr[k];
      const float* raw = p.j3_raw + f * kJoints * 3;
      float v = __fsub_rn(raw[joint * 3 + c], raw[kRootJoint * 3 + c]);
      if (p.filters_on) {
        const double* pr = p.prep3 + ((size_t)(f * kJoints + joint) * 3 + c) * 3;
        const FilterPrep fp = {pr[0], pr[1], pr[2]};
        v = __double2float_rn(oef_finish(st, p.cfg3d, fp, (double)v, p.t3d[f], true));
      }
      p.out3d[(f * kJoints + joint) * 3 + c] = v;
      if (p.packed != nullptr) p.packed[(f * kJoints + joint) * 5 + 2 + c] = (double)v;
    }
    if (p.filters_on) p.st3d[((size_t)sid * kJoints + joint) * 3 + c] = st;
  }
}

// Bounding-box tracker of the reference's video loop (run_estimator.py:110-119), one warp per frame:
//   buffer_x = 0.8 * (x_max - x_min + 1);  buffer_y = 0.2 * (y_max - y_min + 1)
//   x, y = max(int(x_min - buffer_x / 2), 0), max(int(y_min - buffer_y / 2), 0)
//   w, h = int(min(x_max - x_min + buffer_x, W_img - x)), int(min(y_max - y_min + buffer_y, H_img - y))
// joints2d are full-frame (row, col) coordinates; float64 arithmetic without FMA, int() truncates toward zero.
__device__ __forceinline__ void track_box_update(const double* __restrict__ joints2d, const int* __restrict__ stream_ids,
                                                 int frame, int FH, int FW, int4* __restrict__ boxes) {
  const int lane = threadIdx.x;
  double ymin = INFINITY, ymax = -INFINITY, xmin = INFINITY, xmax = -INFINITY;
  if (lane < kJoints) {
    ymin = ymax = joints2d[(frame * kJoints + lane) * 2 + 0];
    xmin = xmax = joints2d[(frame * kJoints + lane) * 2 + 1];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ymin = fmin(ymin, __shfl_xor_sync(0xffffffffu, ymin, o));
    ymax = fmax(ymax, __shfl_xor_sync(0xffffffffu, ymax, o));
    xmin = fmin(xmin, __shfl_xor_sync(0xffffffffu, xmin, o));
    xmax = fmax(xmax, __shfl_xor_sync(0xffffffffu, xmax, o));
  }
  if (lane == 0) {
    const double buffer_x = __dmul_rn(0.8, __dadd_rn(__dsub_rn(xmax, xmin), 1.0));
    const double buffer_y = __dmul_rn(0.2, __dadd_rn(__dsub_rn(ymax, ymin), 1.0));
    const int x = max((int)__dsub_rn(xmin, __ddiv_rn(buffer_x, 2.0)), 0);
    const int y = max((int)__dsub_rn(ymin, __ddiv_rn(buffer_y, 2.0)), 0);
    const int w = (int)fmin(__dadd_rn(__dsub_rn(xmax, xmin), buffer_x), (double)(FW - x));
    const int h = (int)fmin(__dadd_rn(__dsub_rn(ymax, ymin), buffer_y), (double)(FH - y));
    boxes[stream_ids[frame]] = make_int4(x, y, w, h);
  }
}

__global__ void track_update_kernel(const double* __restrict__ joints2d, const int* __restrict__ stream_ids, int n,
                                    int FH, int FW, int4* __restrict__ boxes) {
  track_box_update(joints2d, stream_ids, blockIdx.x, FH, FW, boxes);
}

// the same for a mixed-size batch: frame f's box is clipped to its own full-frame size frames[f]
__global__ void track_update_frames_kernel(const double* __restrict__ joints2d, const int* __restrict__ stream_ids,
                                           const FrameDesc* __restrict__ frames, int4* __restrict__ boxes) {
  const int f = blockIdx.x;
  track_box_update(joints2d, stream_ids, f, frames[f].height, frames[f].width, boxes);
}

// the same with oriented frames: the box is clamped to the oriented frame's sides (W_img, H_img of the frame the
// joints are in)
__global__ void track_update_frames_oriented_kernel(const double* __restrict__ joints2d,
                                                    const int* __restrict__ stream_ids,
                                                    const FrameDesc* __restrict__ frames,
                                                    const int* __restrict__ orient, int4* __restrict__ boxes) {
  const int f = blockIdx.x;
  const bool swap = orient_swaps(orient[f]);
  track_box_update(joints2d, stream_ids, f, swap ? frames[f].width : frames[f].height,
                   swap ? frames[f].height : frames[f].width, boxes);
}

// The box update of a call in which some stream recovers lost people (vnect_set_track_recovery), with or without
// oriented frames (orient == nullptr: all identity).  Frame f's mean score m = (((s0 + s1) + s2) + ... + s20) / 21, in
// float64 without FMA (Python's sum(scores) / 21), against the stream's threshold min_mean[f] taken at submission:
// below a positive threshold the stream's next crop is its whole frame, the box vnect_reset_stream leaves; otherwise
// the reference's box update runs unchanged.
__global__ void track_update_frames_recover_kernel(const double* __restrict__ joints2d,
                                                   const int* __restrict__ stream_ids,
                                                   const FrameDesc* __restrict__ frames,
                                                   const int* __restrict__ orient, const double* __restrict__ scores,
                                                   const double* __restrict__ min_mean, int4* __restrict__ boxes) {
  const int f = blockIdx.x;
  int lost = 0;
  if (threadIdx.x == 0) {
    const double tau = min_mean[f];
    double acc = 0.0;
    for (int j = 0; j < kJoints; ++j) acc = __dadd_rn(acc, scores[f * kJoints + j]);
    lost = tau > 0.0 && __ddiv_rn(acc, (double)kJoints) < tau;
  }
  if (__shfl_sync(0xffffffffu, lost, 0)) {
    if (threadIdx.x == 0) boxes[stream_ids[f]] = make_int4(0, 0, 1 << 30, 1 << 30);
    return;
  }
  const bool swap = orient != nullptr && orient_swaps(orient[f]);
  track_box_update(joints2d, stream_ids, f, swap ? frames[f].width : frames[f].height,
                   swap ? frames[f].height : frames[f].width, boxes);
}

// vnect_track_set_boxes: up to kSeedBoxes seeded boxes travel in the kernel's parameters, so the caller's arrays are
// free once the launch returns and the write lands in stream order between the tracked calls around it.  Ids are
// distinct (checked on the host), so one thread per box writes without conflicts.
constexpr int kSeedBoxes = 64;
struct BoxSeeds {
  int4 box[kSeedBoxes];  // (x, y, w, h)
  int stream_id[kSeedBoxes];
  int n;
};

__global__ void track_seed_boxes_kernel(const __grid_constant__ BoxSeeds s, int4* __restrict__ boxes) {
  const int i = threadIdx.x;
  if (i < s.n) boxes[s.stream_id[i]] = s.box[i];
}

// ---------------------------------------------------------------------------------------------------------------
// Joints2Angles (reference: src/joints2angles.py:60-110): eight arm angles of a robot from the 3D joints -- the step
// right after the hot path for the robot use case (SURVEY.md section 8f row 4).  One thread per frame.  The reference
// mixes float32 (joint differences, their cross product, their norms) and float64 (everything touched by the integer
// list [0, 1, 0]); the same types are used here, dot products are accumulated left to right.  numpy's dot goes through
// BLAS (unspecified order / FMA) and its arccos through libm, so parity is to a tolerance, not bit-exact.
struct Vec3f { float x, y, z; };
struct Vec3d { double x, y, z; };
__device__ __forceinline__ Vec3f sub3f(const float* a, const float* b) {
  return {__fsub_rn(a[0], b[0]), __fsub_rn(a[1], b[1]), __fsub_rn(a[2], b[2])};
}
__device__ __forceinline__ Vec3f cross3f(Vec3f a, Vec3f b) {  // np.cross on float32: separate products, then subtract
  return {__fsub_rn(__fmul_rn(a.y, b.z), __fmul_rn(a.z, b.y)), __fsub_rn(__fmul_rn(a.z, b.x), __fmul_rn(a.x, b.z)),
          __fsub_rn(__fmul_rn(a.x, b.y), __fmul_rn(a.y, b.x))};
}
__device__ __forceinline__ float dot3f(Vec3f a, Vec3f b) {
  return __fadd_rn(__fadd_rn(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)), __fmul_rn(a.z, b.z));
}
__device__ __forceinline__ double dot3d(Vec3d a, Vec3d b) {
  return __dadd_rn(__dadd_rn(__dmul_rn(a.x, b.x), __dmul_rn(a.y, b.y)), __dmul_rn(a.z, b.z));
}
__device__ __forceinline__ Vec3d widen(Vec3f a) { return {(double)a.x, (double)a.y, (double)a.z}; }
__device__ __forceinline__ double clamp_acos(double c) { return acos(c); }  // np.arccos: NaN outside [-1, 1], like acos

struct AnglesParams {
  const float* joints3d;   // [n][21][3]
  const int* stream_ids;   // [n]
  const double* t;         // [n] clock readings, or nullptr = no filtering (Joints2Angles(filter=False))
  FilterState* st;         // [max_streams][8]
  double* angles;          // [n][8] radians: s0_l, s1_l, e0_l, e1_l, s0_r, s1_r, e0_r, e1_r
  int n;
};

__global__ void joints2angles_kernel(AnglesParams p) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n) return;
  const float* j = p.joints3d + (size_t)i * kJoints * 3;
  const float *sh_l = j + 5 * 3, *el_l = j + 6 * 3, *wr_l = j + 7 * 3, *sh_r = j + 2 * 3, *el_r = j + 3 * 3, *wr_r = j + 4 * 3;
  const Vec3f s2e_l = sub3f(el_l, sh_l), e2w_l = sub3f(wr_l, el_l);
  const Vec3f s2e_r = sub3f(el_r, sh_r), e2w_r = sub3f(wr_r, el_r);
  const Vec3f v1_l = sub3f(sh_r, sh_l);
  const Vec3f v1_r = {-v1_l.x, -v1_l.y, -v1_l.z};
  const Vec3d down = {0.0, 1.0, 0.0};
  // cross(a, [0, 1, 0]) in float64 = (-a.z, 0, a.x) up to the sign of zero
  const Vec3d v3_l = {-(double)s2e_l.z, 0.0, (double)s2e_l.x}, v3_r = {-(double)s2e_r.z, 0.0, (double)s2e_r.x};
  const Vec3f v4_l = cross3f(s2e_l, e2w_l), v4_r = cross3f(s2e_r, e2w_r);
  auto norm_f = [](Vec3f a) { return (double)__fsqrt_rn(dot3f(a, a)); };   // float32 norm, promoted when multiplied
  auto norm_d = [](Vec3d a) { return __dsqrt_rn(dot3d(a, a)); };
  // cal_angle(v1, v2) = arccos(dot / (|v1| * |v2|)) with numpy's result types
  auto ang_fd = [&](Vec3f a, Vec3d b) { return clamp_acos(__ddiv_rn(dot3d(widen(a), b), __dmul_rn(norm_f(a), norm_d(b)))); };
  auto ang_dd_f = [&](Vec3d a, Vec3f b) { return clamp_acos(__ddiv_rn(dot3d(a, widen(b)), __dmul_rn(norm_d(a), norm_f(b)))); };
  auto ang_ff = [&](Vec3f a, Vec3f b) {  // all float32: float32 cosine, float32 arccos
    const float c = __fdiv_rn(dot3f(a, b), __fmul_rn(__fsqrt_rn(dot3f(a, a)), __fsqrt_rn(dot3f(b, b))));
    return (double)acosf(c);
  };
  const double kPi = 3.141592653589793;
  double a[8];
  a[0] = __dsub_rn(__ddiv_rn(__dmul_rn(kPi, 3.0), 4.0), ang_fd(v1_l, v3_l));   // s0_l
  a[1] = __dsub_rn(__ddiv_rn(kPi, 2.0), ang_dd_f(down, s2e_l));               // s1_l
  a[2] = -ang_dd_f(v3_l, v4_l);                                                // e0_l
  a[3] = ang_ff(s2e_l, e2w_l);                                                 // e1_l (float32 in the reference)
  a[4] = __dsub_rn(__ddiv_rn(kPi, 4.0), ang_fd(v1_r, v3_r));                   // s0_r
  a[5] = __dsub_rn(__ddiv_rn(kPi, 2.0), ang_dd_f(down, s2e_r));               // s1_r
  a[6] = ang_dd_f(v3_r, v4_r);                                                 // e0_r
  a[7] = ang_ff(s2e_r, e2w_r);                                                 // e1_r (float32)
  a[0] = __dsub_rn(a[0], __ddiv_rn(kPi, 4.0));   // the script's final pose offsets (joints2angles.py:101-105)
  a[3] = -a[3];
  a[4] = __dadd_rn(a[4], __ddiv_rn(kPi, 4.0));
  a[5] = -a[5];
  if (p.t != nullptr) {
    const FilterCfg cfg = {120.0, 0.5, 0.5, 1.0};  // joints2angles.py:35-41
    FilterState* st = p.st + (size_t)p.stream_ids[i] * 8;
    for (int k = 0; k < 8; ++k) {
      FilterState s = st[k];
      a[k] = oef_step(s, cfg, a[k], p.t[i], false);
      st[k] = s;
    }
  }
  for (int k = 0; k < 8; ++k) p.angles[(size_t)i * 8 + k] = a[k];
}

// Debug scan (vnect_check_finite): values of an fp16 activation tensor that are NaN / Inf or saturated (|x| >= 65504).
__global__ void count_nonfinite_kernel(const __half* __restrict__ x, size_t n, unsigned long long* __restrict__ out) {
  unsigned long long c = 0;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float v = __half2float(x[i]);
    c += !(fabsf(v) < 65504.f);
  }
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}

// VNectEstimator.joint_filter (estimator.py:83-95) on explicit values: 21*dim scalar filters of one stream.
// is_f32: the caller's array is float32 (the reference's joints_3d), so the raw difference and the stored result are.
__global__ void joint_filter_kernel(FilterState* st, FilterCfg cfg, double* values, double t, int dim, int is_f32) {
  const int i = threadIdx.x;
  if (i >= kJoints * dim) return;
  FilterState s = st[i];
  const double v = oef_step(s, cfg, values[i], t, is_f32 != 0);
  values[i] = is_f32 ? (double)__double2float_rn(v) : v;
  st[i] = s;
}

}  // namespace vnect
