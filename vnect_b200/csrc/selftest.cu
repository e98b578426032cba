// GPU self-test of the tcgen05 implicit-GEMM convolution kernel against a naive direct convolution written with
// plain CUDA loops (test infrastructure only; never linked into libvnect_b200.so).
//   build: make -C vnect_b200/csrc selftest      run (on a B200): build/selftest
#include <cmath>
#include <cstdlib>
#include <string>
#include <vector>

#include "conv_plan.cuh"

using namespace vnect;

#define CK(x)                                                                              \
  do {                                                                                     \
    cudaError_t e_ = (x);                                                                  \
    if (e_ != cudaSuccess) {                                                               \
      printf("CUDA error %s at %s:%d: %s\n", #x, __FILE__, __LINE__, cudaGetErrorString(e_)); \
      exit(2);                                                                             \
    }                                                                                      \
  } while (0)

struct NaiveGeom {
  int NB, H, W, cin_pad, n_pad, taps, phases, k_total;
  int stem;  // 1: the 7x7/2 stem conv on the parity-split padded input [NB][2][stem_rpp][stem_pitch], row taps dy / dp
  int stem_rpp, stem_pitch;
  int in_stride;
  signed char dx[16], dy[16], dp[16];
};

// raw fp32 accumulators acc[ph][m][col]
__global__ void naive_acc_kernel(const __half* __restrict__ in, const __half* __restrict__ w, float* __restrict__ acc,
                                 NaiveGeom g, const __half* __restrict__ in2 = nullptr, int cin2 = 0) {
  const long long total = (long long)g.phases * g.NB * g.H * g.W * g.n_pad;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int col = (int)(i % g.n_pad);
    long long r = i / g.n_pad;
    const int x = (int)(r % g.W);
    r /= g.W;
    const int y = (int)(r % g.H);
    r /= g.H;
    const int n = (int)(r % g.NB);
    const int ph = (int)(r / g.NB);
    const __half* wrow = w + ((size_t)ph * g.n_pad + col) * g.k_total;
    float s = 0.f;
    for (int t = 0; t < g.taps; ++t) {
      const int ti = ph * g.taps + t;
      if (g.stem) {
        const int row = y + g.dy[ti];
        if (row < 0 || row >= g.stem_rpp) continue;
        const __half* a = in + (((size_t)n * 2 + g.dp[ti]) * g.stem_rpp + row) * g.stem_pitch + (size_t)x * 8;
        for (int c = 0; c < 32; ++c) s += __half2float(a[c]) * __half2float(wrow[t * 32 + c]);
      } else {
        const int IH = g.H * g.in_stride, IW = g.W * g.in_stride;
        const int yy = y * g.in_stride + g.dy[ti], xx = x * g.in_stride + g.dx[ti];
        if (yy < 0 || yy >= IH || xx < 0 || xx >= IW) continue;
        const __half* a = in + (((size_t)n * IH + yy) * IW + xx) * g.cin_pad;
        for (int c = 0; c < g.cin_pad; ++c) s += __half2float(a[c]) * __half2float(wrow[(size_t)t * g.cin_pad + c]);
      }
    }
    if (in2) {  // folded 1x1 shortcut: extra K from a second tensor on the same pixel
      const __half* a2 = in2 + (((size_t)n * g.H + y) * g.W + x) * cin2;
      for (int c = 0; c < cin2; ++c) s += __half2float(a2[c]) * __half2float(wrow[(size_t)g.taps * g.cin_pad + c]);
    }
    acc[i] = s;
  }
}

static uint32_t rng_state = 12345u;
static float frand() {
  rng_state = rng_state * 1664525u + 1013904223u;
  return ((rng_state >> 8) & 0xFFFF) / 32768.0f - 1.0f;
}

// build_conv picks the kernel path (CTA pairs, resident weights, halo patches, im2col) from the shape, block_n and
// epilogue, as it does for the library's plans; every result line names the path taken
struct Case {
  const char* name;
  int kind, NB, H, W, cin_pad, n_pad, n_valid, block_n, epi;
  bool bias, residual;
  int relu_cols;
  int in_stride = 1, res_stride = 1;
  int cin2 = 0;  // folded shortcut: second input tensor with cin2 channels (1x1 only)
  int n2 = 0;    // > 0: fused block tail, second 1x1 conv of n2 channels on this conv's output (block_tail.cuh)
};

// reference of the chained conv, from the fp16 X the kernel under test wrote: y[m][col] = relu(sum_c X[m][c] * W2[col][c] + b2[col])
__global__ void naive_chain_kernel(const __half* __restrict__ x, const __half* __restrict__ w2, const float* __restrict__ b2,
                                   float* __restrict__ y, long long rows, int cout, int n2) {
  const long long total = rows * n2;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int col = (int)(i % n2);
    const long long m = i / n2;
    const __half* xr = x + m * cout;
    const __half* wr = w2 + (size_t)col * cout;
    float s = 0.f;
    for (int c = 0; c < cout; ++c) s += __half2float(xr[c]) * __half2float(wr[c]);
    y[i] = fmaxf(s + b2[col], 0.f);
  }
}

static int run_case(const Case& c, int num_sms, bool timing) {
  ConvSpec s;
  s.kind = c.kind;
  s.NB = c.NB;
  s.H = c.H;
  s.W = c.W;
  s.cin_pad = c.cin_pad;
  s.n_pad = c.n_pad;
  s.n_valid = c.n_valid;
  s.block_n = c.block_n;
  s.epi = c.epi;
  s.relu_cols = c.relu_cols;
  s.in_stride = c.in_stride;
  s.res_stride = c.res_stride;
  const int phases = c.kind == CONV_DECONV4 ? 4 : 1;
  const int taps = c.kind == CONV_1x1 ? 1 : c.kind == CONV_3x3 ? 9 : 4;
  const int k_total = taps * c.cin_pad + c.cin2;
  const size_t in_elems = (size_t)c.NB * c.H * c.W * c.cin_pad * c.in_stride * c.in_stride;
  std::vector<__half> h_in(in_elems), h_w((size_t)phases * c.n_pad * k_total);
  for (auto& v : h_in) v = __float2half(frand());
  const float wscale = 1.0f / sqrtf((float)k_total);
  for (auto& v : h_w) v = __float2half(frand() * wscale * 2.f);
  std::vector<float> h_bias(c.n_pad);
  for (auto& v : h_bias) v = frand() * 0.5f;

  int OH = c.H, OW = c.W;
  if (c.kind == CONV_DECONV4) { OH = 2 * c.H; OW = 2 * c.W; }
  const int ldc = c.epi == EPI_DECONV_HEAD ? 256 : c.n_pad;
  const size_t out_elems = c.epi == EPI_PLANAR_F32 ? (size_t)c.NB * c.n_valid * OH * OW : (size_t)c.NB * OH * OW * ldc;
  const size_t out_bytes = out_elems * (c.epi == EPI_PLANAR_F32 ? 4 : 2);
  const int ldr = c.n_pad;
  std::vector<__half> h_res;
  if (c.residual) {
    h_res.resize((size_t)c.NB * c.H * c.W * ldr * c.res_stride * c.res_stride);
    for (auto& v : h_res) v = __float2half(frand());
  }

  __half* d_in2 = nullptr;
  std::vector<__half> h_in2;
  if (c.cin2) {
    h_in2.resize((size_t)c.NB * c.H * c.W * c.cin2);
    for (auto& v : h_in2) v = __float2half(frand());
    CK(cudaMalloc(&d_in2, h_in2.size() * 2));
    CK(cudaMemcpy(d_in2, h_in2.data(), h_in2.size() * 2, cudaMemcpyHostToDevice));
  }
  __half *d_in, *d_w, *d_res = nullptr;
  float *d_bias, *d_acc;
  void* d_out;
  CK(cudaMalloc(&d_in, in_elems * 2));
  CK(cudaMalloc(&d_w, h_w.size() * 2));
  CK(cudaMalloc(&d_bias, c.n_pad * 4));
  CK(cudaMalloc(&d_out, out_bytes));
  CK(cudaMemset(d_out, 0, out_bytes));
  const size_t acc_elems = (size_t)phases * c.NB * c.H * c.W * c.n_pad;
  CK(cudaMalloc(&d_acc, acc_elems * 4));
  CK(cudaMemcpy(d_in, h_in.data(), in_elems * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_w, h_w.data(), h_w.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_bias, h_bias.data(), c.n_pad * 4, cudaMemcpyHostToDevice));
  if (c.residual) {
    CK(cudaMalloc(&d_res, h_res.size() * 2));
    CK(cudaMemcpy(d_res, h_res.data(), h_res.size() * 2, cudaMemcpyHostToDevice));
  }
  __half *d_w2 = nullptr, *d_out2 = nullptr;
  float* d_bias2 = nullptr;
  if (c.n2) {
    std::vector<__half> h_w2((size_t)c.n2 * c.n_pad);
    std::vector<float> h_b2(c.n2);
    const float w2s = 2.0f / sqrtf((float)c.n_pad);
    for (auto& v : h_w2) v = __float2half(frand() * w2s);
    for (auto& v : h_b2) v = frand() * 0.5f;
    CK(cudaMalloc(&d_w2, h_w2.size() * 2));
    CK(cudaMalloc(&d_bias2, c.n2 * 4));
    CK(cudaMalloc(&d_out2, (size_t)c.NB * c.H * c.W * c.n2 * 2));
    CK(cudaMemset(d_out2, 0xff, (size_t)c.NB * c.H * c.W * c.n2 * 2));
    CK(cudaMemcpy(d_w2, h_w2.data(), h_w2.size() * 2, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_bias2, h_b2.data(), c.n2 * 4, cudaMemcpyHostToDevice));
    s.w2 = d_w2; s.bias2 = d_bias2; s.out2 = d_out2; s.n2 = c.n2;
  }
  s.in = d_in;
  s.in2 = d_in2;
  s.cin2_pad = c.cin2;
  s.w = d_w;
  s.bias = c.bias ? d_bias : nullptr;
  s.residual = d_res;
  s.ldr = ldr;
  s.out = d_out;
  s.ldc = ldc;

  ConvLaunch L;
  std::string err;
  if (!build_conv(s, num_sms, &L, &err)) {
    printf("[%s] build_conv FAILED: %s\n", c.name, err.c_str());
    return 1;
  }
  CK(launch_conv(L, 0));
  cudaError_t se = cudaDeviceSynchronize();
  if (se != cudaSuccess) {
    printf("[%s] kernel FAILED: %s\n", c.name, cudaGetErrorString(se));
    exit(3);  // context is gone
  }

  NaiveGeom g;
  memset(&g, 0, sizeof g);
  g.NB = c.NB; g.H = c.H; g.W = c.W; g.cin_pad = c.cin_pad; g.n_pad = c.n_pad;
  g.in_stride = c.in_stride;
  g.taps = taps; g.phases = phases; g.k_total = k_total;
  memcpy(g.dx, L.p.tap_dx, 16); memcpy(g.dy, L.p.tap_dy, 16);
  if (L.p.im2col)  // the launch holds filter offsets from the base pixel (0..2); the reference wants displacements (-1..1)
    for (int t = 0; t < 16; ++t) { g.dx[t] = (signed char)(g.dx[t] - 1); g.dy[t] = (signed char)(g.dy[t] - 1); }
  naive_acc_kernel<<<1184, 256>>>(d_in, d_w, d_acc, g, d_in2, c.cin2);
  CK(cudaDeviceSynchronize());
  std::vector<float> h_acc(acc_elems);
  CK(cudaMemcpy(h_acc.data(), d_acc, acc_elems * 4, cudaMemcpyDeviceToHost));
  std::vector<uint8_t> h_out(out_bytes);
  CK(cudaMemcpy(h_out.data(), d_out, out_bytes, cudaMemcpyDeviceToHost));
  const __half* o16 = reinterpret_cast<const __half*>(h_out.data());
  const float* o32 = reinterpret_cast<const float*>(h_out.data());

  double max_err = 0;
  long long bad = 0, checked = 0;
  auto check = [&](float got, float exp) {
    const float tol = 3e-3f * fabsf(exp) + 3e-3f;
    const float e = fabsf(got - exp);
    if (!(e <= tol)) {
      if (bad < 5) printf("   mismatch got %f exp %f\n", got, exp);
      ++bad;
    }
    if (e > max_err) max_err = e;
    ++checked;
  };
  for (int ph = 0; ph < phases; ++ph)
    for (int n = 0; n < c.NB; ++n)
      for (int y = 0; y < c.H; ++y)
        for (int x = 0; x < c.W; ++x) {
          const size_t m = ((size_t)n * c.H + y) * c.W + x;
          const float* a = &h_acc[((size_t)ph * c.NB * c.H * c.W + m) * c.n_pad];
          int oy, ox;
          if (c.kind == CONV_DECONV4) {
            oy = 2 * y + (ph >> 1); ox = 2 * x + (ph & 1);
          } else {
            oy = y; ox = x;
          }
          const size_t pix = ((size_t)n * OH + oy) * OW + ox;
          float bone[21] = {0};
          for (int col = 0; col < c.n_pad; ++col) {
            float v = a[col] + (c.bias ? h_bias[col] : 0.f);
            if (c.residual) {
              const size_t rm = ((size_t)n * c.H * c.res_stride + (size_t)y * c.res_stride) * c.W * c.res_stride + (size_t)x * c.res_stride;
              v += __half2float(h_res[rm * ldr + col]);
            }
            if (col < c.relu_cols) v = fmaxf(v, 0.f);
            if (c.epi == EPI_PLANAR_F32) {
              if (col < c.n_valid) check(o32[((size_t)n * c.n_valid + col) * OH * OW + (size_t)oy * OW + ox], v);
            } else if (c.epi == EPI_DECONV_HEAD) {
              if (col < 191) check(__half2float(o16[pix * ldc + col]), v);
              if (col >= 128 && col < 191) bone[(col - 128) % 21] += v * v;
            } else {
              check(__half2float(o16[pix * ldc + col]), v);
            }
          }
          if (c.epi == EPI_DECONV_HEAD) {
            for (int j = 0; j < 21; ++j) check(__half2float(o16[pix * ldc + 191 + j]), sqrtf(bone[j]));
            for (int j = 212; j < 216; ++j) check(__half2float(o16[pix * ldc + j]), 0.f);
          }
        }
  if (c.n2) {  // the chained conv against a naive evaluation on the X this kernel wrote
    const long long rows = (long long)c.NB * c.H * c.W;
    float* d_y;
    CK(cudaMalloc(&d_y, rows * c.n2 * 4));
    naive_chain_kernel<<<1184, 256>>>(reinterpret_cast<const __half*>(d_out), d_w2, d_bias2, d_y, rows, c.n_pad, c.n2);
    CK(cudaDeviceSynchronize());
    std::vector<float> h_y((size_t)rows * c.n2);
    std::vector<__half> h_o2((size_t)rows * c.n2);
    CK(cudaMemcpy(h_y.data(), d_y, h_y.size() * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(h_o2.data(), d_out2, h_o2.size() * 2, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < h_y.size(); ++i) check(__half2float(h_o2[i]), h_y[i]);
    cudaFree(d_y);
  }
  printf("[%s] path=%s%s%s%sn%d/cg%d tiles=%d grid=%d tile=%dx%d checked=%lld bad=%lld max_abs_err=%.3e  %s\n", c.name,
         L.n2 ? "tail " : "", L.b_resident ? "resident " : "", L.halo ? "halo " : "", L.p.im2col ? "im2col " : "",
         L.block_n, L.cg, L.p.phases * L.p.num_m_tiles * L.p.num_n_tiles, L.grid, L.p.tw, L.p.th, checked, bad, max_err,
         bad == 0 ? "PASS" : "FAIL");

  if (timing && bad == 0) {
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    for (int i = 0; i < 3; ++i) CK(launch_conv(L, 0));
    CK(cudaEventRecord(e0));
    const int reps = 20;
    for (int i = 0; i < reps; ++i) CK(launch_conv(L, 0));
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    const double us = ms * 1000.0 / reps;
    printf("   timing: %.2f us/launch, %.1f TFLOP/s (GEMM flops incl. padding)\n", us, L.flops / us * 1e-6);
  }
  cudaFree(d_in); cudaFree(d_w); cudaFree(d_bias); cudaFree(d_out); cudaFree(d_acc);
  if (d_res) cudaFree(d_res);
  if (d_in2) cudaFree(d_in2);
  if (d_w2) { cudaFree(d_w2); cudaFree(d_bias2); cudaFree(d_out2); }
  return bad == 0 ? 0 : 1;
}

// fused conv1 + pool1 against naive conv + host max-pool
static int run_stem_pool(int NB, int S, int num_sms) {
  const bool roll = true;
  const int OH = S / 2, PH = S / 4, vw = OH + 3, rpp = OH + 3, pitch = vw * 8;
  const size_t in_elems = (size_t)NB * 2 * rpp * pitch + 8192;
  std::vector<__half> h_in(in_elems), h_w((size_t)64 * 224), h_ws((size_t)64 * 224);
  for (auto& v : h_in) v = __float2half(frand());
  for (auto& v : h_w) v = __float2half(frand() * 0.15f);
  pack_stem_stacked(h_w.data(), h_ws.data());
  std::vector<__half> h_wp((size_t)kPairWBytes);
  pack_stem_pair(h_w.data(), h_wp.data());
  std::vector<float> h_bias(64);
  for (auto& v : h_bias) v = frand() * 0.5f;
  __half *d_in, *d_w, *d_ws, *d_wp, *d_out;
  CK(cudaMalloc(&d_ws, h_ws.size() * 2));
  CK(cudaMemcpy(d_ws, h_ws.data(), h_ws.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMalloc(&d_wp, h_wp.size() * 2));
  CK(cudaMemcpy(d_wp, h_wp.data(), h_wp.size() * 2, cudaMemcpyHostToDevice));
  float *d_bias, *d_acc;
  CK(cudaMalloc(&d_in, in_elems * 2));
  CK(cudaMalloc(&d_w, h_w.size() * 2));
  CK(cudaMalloc(&d_bias, 64 * 4));
  CK(cudaMemcpy(d_in, h_in.data(), in_elems * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_w, h_w.data(), h_w.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_bias, h_bias.data(), 64 * 4, cudaMemcpyHostToDevice));
  const size_t out_elems = (size_t)NB * PH * PH * 64;
  CK(cudaMalloc(&d_out, out_elems * 2));
  CK(cudaMemset(d_out, 0xff, out_elems * 2));
  StemPoolLaunch L;
  std::string err;
  if (!build_stem_pool(d_in, S, rpp, pitch, d_ws, d_bias, d_out, NB, num_sms, &L, &err, d_wp, in_elems)) {
    printf("[stem_pool] build FAILED: %s\n", err.c_str());
    return 1;
  }
  unsigned long long* d_dbg;
  CK(cudaMalloc(&d_dbg, 8 * sizeof(unsigned long long)));
  CK(cudaMemset(d_dbg, 0, 8 * sizeof(unsigned long long)));
  L.r.dbg = d_dbg;
  CK(launch_stem_pool<true>(L, 0));
  cudaError_t se = cudaDeviceSynchronize();
  if (se != cudaSuccess) {
    printf("[stem_pool] kernel FAILED: %s\n", cudaGetErrorString(se));
    exit(3);
  }
  NaiveGeom g;
  memset(&g, 0, sizeof g);
  g.stem = 1; g.NB = NB; g.H = OH; g.W = OH; g.n_pad = 64; g.taps = 7; g.phases = 1;
  g.k_total = 224; g.stem_rpp = rpp; g.stem_pitch = pitch; g.in_stride = 1;
  for (int ky = 0; ky < 7; ++ky) { g.dy[ky] = (signed char)(ky >> 1); g.dx[ky] = 0; g.dp[ky] = (signed char)(ky & 1); }
  const size_t acc_elems = (size_t)NB * OH * OH * 64;
  CK(cudaMalloc(&d_acc, acc_elems * 4));
  naive_acc_kernel<<<1184, 256>>>(d_in, d_w, d_acc, g);
  CK(cudaDeviceSynchronize());
  std::vector<float> h_acc(acc_elems);
  std::vector<__half> h_out(out_elems);
  CK(cudaMemcpy(h_acc.data(), d_acc, acc_elems * 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(h_out.data(), d_out, out_elems * 2, cudaMemcpyDeviceToHost));
  long long bad = 0, checked = 0;
  double max_err = 0;
  for (int n = 0; n < NB; ++n)
    for (int py = 0; py < PH; ++py)
      for (int px = 0; px < PH; ++px)
        for (int c = 0; c < 64; ++c) {
          float exp = -1e30f;
          for (int a = 0; a < 3; ++a)
            for (int b = 0; b < 3; ++b) {
              const int y = 2 * py + a, x = 2 * px + b;
              if (y >= OH || x >= OH) continue;
              exp = fmaxf(exp, fmaxf(h_acc[(((size_t)n * OH + y) * OH + x) * 64 + c] + h_bias[c], 0.f));
            }
          const float got = __half2float(h_out[(((size_t)n * PH + py) * PH + px) * 64 + c]);
          const float e = fabsf(got - exp);
          if (!(e <= 3e-3f * fabsf(exp) + 3e-3f)) {
            if (bad < 5) printf("   mismatch n%d py%d px%d c%d got %f exp %f\n", n, py, px, c, got, exp);
            ++bad;
          }
          if (e > max_err) max_err = e;
          ++checked;
        }
  {
    unsigned long long h_dbg[8];
    CK(cudaMemcpy(h_dbg, d_dbg, sizeof h_dbg, cudaMemcpyDeviceToHost));
    const double items0 = (double)((L.r.num_items + L.grid - 1) / L.grid);
    if (!roll) printf("   CTA0 epilogue cycles per band: wait-MMA %.0f, drain %.0f, barrier %.0f, pool %.0f\n", h_dbg[0] / items0,
           h_dbg[1] / items0, h_dbg[2] / items0, h_dbg[3] / items0);
    if (roll) printf("   CTA0 epilogue cycles: wait-MMA %llu, drain %llu, pool %llu, total %llu\n", h_dbg[0], h_dbg[1], h_dbg[2], h_dbg[3]);
    if (roll) printf("   CTA0 MMA warp cycles: wait-strips %llu, wait-slot %llu, total %llu\n", h_dbg[4], h_dbg[5], h_dbg[6]);
    L.r.dbg = nullptr;
  }
  printf("[stem_roll rolling conv1+pool1 S=%d nb=%d cg=%d] items=%d grid=%d x-tiles=%d seg_rows=%d checked=%lld bad=%lld max_abs_err=%.3e  %s\n",
         S, NB, L.cg, L.r.num_items, L.grid, L.r.n_xt, L.r.seg_rows, checked, bad, max_err, bad == 0 ? "PASS" : "FAIL");
  if (bad == 0) {
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    for (int i = 0; i < 3; ++i) CK(launch_stem_pool(L, 0));
    CK(cudaEventRecord(e0));
    for (int i = 0; i < 20; ++i) CK(launch_stem_pool(L, 0));
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    printf("   timing: %.2f us/launch\n", ms * 1000.0 / 20);
  }
  cudaFree(d_in); cudaFree(d_w); cudaFree(d_ws); cudaFree(d_bias); cudaFree(d_out); cudaFree(d_acc);
  return bad == 0 ? 0 : 1;
}

// ---------------------------------------------------------------------------------------------------------------
// Descriptor probe: how does tcgen05.mma address a 128B-swizzled K-major A operand whose start address is NOT aligned
// to the 1024-byte swizzle atom and whose 8-row groups are `pitch` rows apart?  (The halo-patch 3x3 convolution reads
// its nine filter taps from ONE shared-memory patch by shifting the descriptor's start address by whole pixels.)
// Rows are written exactly as the TMA unit writes a dense box: 16-byte chunk c of row r lands at
// r*128 + ((c ^ (r & 7)) << 4) from a 1024-aligned base.  Logical A row m of the MMA is patch row
// shift + (m / 8) * pitch + (m % 8).  bo = 1 sets the descriptor's base-offset field to (start >> 7) & 7.
__global__ void __launch_bounds__(128, 1) desc_probe_kernel(const __half* __restrict__ a_rows, int n_rows,
                                                             const __half* __restrict__ b_rows, float* __restrict__ d,
                                                             int shift, int pitch, int bo) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sa = smem;                                   // n_rows x 128 B
  uint8_t* sb = smem + ((n_rows * 128 + 1023) / 1024) * 1024;  // 64 x 128 B
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x;
  for (int i = tid; i < n_rows * 8; i += 128) {
    const int r = i >> 3, c = i & 7;
    *reinterpret_cast<uint4*>(sa + r * 128 + ((c ^ (r & 7)) << 4)) = *reinterpret_cast<const uint4*>(a_rows + r * 64 + c * 8);
  }
  for (int i = tid; i < 64 * 8; i += 128) {
    const int r = i >> 3, c = i & 7;
    *reinterpret_cast<uint4*>(sb + r * 128 + ((c ^ (r & 7)) << 4)) = *reinterpret_cast<const uint4*>(b_rows + r * 64 + c * 8);
  }
  if (tid == 0) {
    mbar_init(&bar, 1);
    fence_barrier_init();
  }
  if (tid < 32) tmem_alloc<64>(&tmem_slot);
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;
  if (tid == 0) {
    const uint32_t a_addr = smem_u32(sa) + shift * 128;
    uint64_t a_desc = 0;
    a_desc |= static_cast<uint64_t>((a_addr & 0x3FFFF) >> 4);
    a_desc |= static_cast<uint64_t>(1) << 16;
    a_desc |= static_cast<uint64_t>((pitch * 128) >> 4) << 32;
    a_desc |= 1ull << 46;
    if (bo) a_desc |= static_cast<uint64_t>((a_addr >> 7) & 7) << 49;
    a_desc |= 2ull << 61;
    const uint64_t b_desc = make_kmajor_desc<128>(smem_u32(sb));
    constexpr uint32_t IDESC = make_idesc_f16(128, 64, false);
    for (int k = 0; k < 4; ++k) umma_f16(tmem, a_desc + 2 * k, b_desc + 2 * k, IDESC, k ? 1u : 0u);
    umma_commit(&bar);
  }
  mbar_wait(&bar, 0);
  tc_fence_after();
  {
    const int warp = tid >> 5;
    uint32_t v[32];
    for (int c0 = 0; c0 < 64; c0 += 32) {
      tmem_ld_32x32(tmem + (static_cast<uint32_t>(warp * 32) << 16) + c0, v);
      tmem_ld_wait();
      for (int j = 0; j < 32; ++j) d[tid * 64 + c0 + j] = __uint_as_float(v[j]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (tid < 32) tmem_dealloc<64>(tmem);
}

static void run_desc_probe() {
  const int n_rows = 288;
  std::vector<__half> h_a((size_t)n_rows * 64), h_b((size_t)64 * 64);
  for (auto& v : h_a) v = __float2half(frand());
  for (auto& v : h_b) v = __float2half(frand());
  __half *d_a, *d_b;
  float* d_d;
  CK(cudaMalloc(&d_a, h_a.size() * 2));
  CK(cudaMalloc(&d_b, h_b.size() * 2));
  CK(cudaMalloc(&d_d, 128 * 64 * 4));
  CK(cudaMemcpy(d_a, h_a.data(), h_a.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_b, h_b.data(), h_b.size() * 2, cudaMemcpyHostToDevice));
  const int smem = n_rows * 128 + 64 * 128 + 3072;
  CK(cudaFuncSetAttribute(desc_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  printf("[desc probe] SW128 K-major A operand read at a shifted start; rows = patch[shift + (m/8)*pitch + m%%8]\n");
  const int shifts[] = {0, 1, 3, 8, 11, 21};
  const int pitches[] = {8, 10, 16};
  for (int pitch : pitches)
    for (int shift : shifts)
      for (int bo = 0; bo < 2; ++bo) {
        if (shift + 15 * pitch + 8 > n_rows) continue;
        CK(cudaMemset(d_d, 0, 128 * 64 * 4));
        desc_probe_kernel<<<1, 128, smem>>>(d_a, n_rows, d_b, d_d, shift, pitch, bo);
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) {
          printf("   pitch %2d shift %2d base_offset %d: kernel error %s\n", pitch, shift, bo, cudaGetErrorString(e));
          exit(4);
        }
        std::vector<float> h_d(128 * 64);
        CK(cudaMemcpy(h_d.data(), d_d, h_d.size() * 4, cudaMemcpyDeviceToHost));
        int bad = 0;
        double max_err = 0;
        for (int m = 0; m < 128; ++m) {
          const int row = shift + (m / 8) * pitch + (m % 8);
          for (int n = 0; n < 64; ++n) {
            double acc = 0;
            for (int k = 0; k < 64; ++k) acc += (double)__half2float(h_a[(size_t)row * 64 + k]) * __half2float(h_b[(size_t)n * 64 + k]);
            const double err = fabs(acc - h_d[m * 64 + n]);
            if (err > max_err) max_err = err;
            if (err > 2e-3) ++bad;
          }
        }
        printf("   pitch %2d shift %2d base_offset %d: %s (bad %d, max_err %.3e)\n", pitch, shift, bo, bad ? "MISMATCH" : "match", bad, max_err);
      }
  cudaFree(d_a); cudaFree(d_b); cudaFree(d_d);
}

int main(int argc, char** argv) {
  int dev = 0;
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, dev));
  printf("device: %s, SMs %d, cc %d.%d\n", prop.name, prop.multiProcessorCount, prop.major, prop.minor);
  const int sms = prop.multiProcessorCount;
  const bool big = argc > 1 && atoi(argv[1]) > 0;
  if (argc > 1 && strcmp(argv[1], "probe") == 0) {
    run_desc_probe();
    return 0;
  }
  if (argc > 1 && strcmp(argv[1], "stem") == 0) {  // the fused conv1 + pool1 kernel only
    int f = 0;
    f += run_stem_pool(2, 368, sms);
    f += run_stem_pool(3, 448, sms);
    f += run_stem_pool(1, 64, sms);
    f += run_stem_pool(1, 512, sms);
    f += run_stem_pool(32, 368, sms);
    f += run_stem_pool(128, 368, sms);
    printf(f ? "SELFTEST FAILED (%d failing cases)\n" : "SELFTEST PASSED (%d failing cases)\n", f);
    return f ? 1 : 0;
  }
  // single-CTA tiles are 64 columns wide, as on the latency plans; the PAIR loop below reruns every TMA-epilogue case
  // with the throughput plans' tile (256 columns from Cout 256, else 128) on CTA pairs
  std::vector<Case> cases = {
      {"1x1 64->64 relu 92x92", CONV_1x1, 2, 92, 92, 64, 64, 64, 64, EPI_TMA, true, false, 64},
      {"1x1 64->256 lin 92x92", CONV_1x1, 2, 92, 92, 64, 256, 256, 64, EPI_TMA, true, false, 0},
      {"TMARES 1x1 64->256 +res relu 92x92", CONV_1x1, 2, 92, 92, 64, 256, 256, 64, EPI_TMA_RES, true, true, 256},
      {"TMARES 1x1 256->1024 +res relu 23x23", CONV_1x1, 7, 23, 23, 256, 1024, 1024, 64, EPI_TMA_RES, true, true, 1024},
      {"TMARES 1x1 128->512 +res relu 46x46", CONV_1x1, 3, 46, 46, 128, 512, 512, 64, EPI_TMA_RES, true, true, 512},
      {"3x3 64->64 relu 92x92", CONV_3x3, 2, 92, 92, 64, 64, 64, 64, EPI_TMA, true, false, 64},
      {"3x3 256->256 relu 23x23", CONV_3x3, 3, 23, 23, 256, 256, 256, 64, EPI_TMA, true, false, 256},
      {"3x3 128->128 relu 46x46", CONV_3x3, 1, 46, 46, 128, 128, 128, 64, EPI_TMA, true, false, 128},
      {"3x3 256->128 relu 23x23", CONV_3x3, 3, 23, 23, 256, 128, 128, 64, EPI_TMA, true, false, 128},
      {"S2 3x3 64->64 relu 92->46", CONV_3x3, 2, 46, 46, 64, 64, 64, 64, EPI_TMA, true, false, 64, 2, 1},
      {"S2 3x3 128->128 relu 46->23", CONV_3x3, 3, 23, 23, 128, 128, 128, 64, EPI_TMA, true, false, 128, 2, 1},
      {"S2RES 1x1 64->256 +res(92) relu 46x46", CONV_1x1, 2, 46, 46, 64, 256, 256, 64, EPI_TMA_RES, true, true, 256, 1, 2},
      {"S2RES 1x1 128->512 +res(46) relu 23x23", CONV_1x1, 3, 23, 23, 128, 512, 512, 64, EPI_TMA_RES, true, true, 512, 1, 2},
      {"FOLD 1x1 64(+64)->256 relu 92x92", CONV_1x1, 2, 92, 92, 64, 256, 256, 64, EPI_TMA, true, false, 256, 1, 1, 64},
      {"FOLD 1x1 128(+256)->512 relu 46x46", CONV_1x1, 3, 46, 46, 128, 512, 512, 64, EPI_TMA, true, false, 512, 1, 1, 256},
      {"FOLD 1x1 512(+1024)->1024 relu 23x23", CONV_1x1, 5, 23, 23, 512, 1024, 1024, 64, EPI_TMA, true, false, 1024, 1, 1, 1024},
      {"deconv4x4s2 256->192 head 23x23", CONV_DECONV4, 2, 23, 23, 256, 192, 191, 192, EPI_DECONV_HEAD, true, false, 128},
      {"1x1 128->84 planar f32 46x46", CONV_1x1, 2, 46, 46, 128, 96, 84, 96, EPI_PLANAR_F32, false, false, 0},
  };
  int fails = 0;
  for (const auto& c : cases) fails += run_case(c, sms, true);
  // the same layers on CTA pairs (odd tile counts included: 2x92x92 1x1 = 133 tiles)
  std::vector<std::string> pair_names;
  pair_names.reserve(cases.size());
  for (const auto& c : cases) {
    if ((c.epi != EPI_TMA && c.epi != EPI_TMA_RES) || c.n_pad < 128) continue;
    Case c2 = c;
    pair_names.push_back(std::string("PAIR ") + c.name);
    c2.name = pair_names.back().c_str();
    c2.block_n = c.n_pad >= 256 ? 256 : 128;
    fails += run_case(c2, sms, true);
  }
  {  // resident weights on spatial tiles: the 64-channel 3x3 convs on small grids (no halo tiling), and a 1x1
    Case r1 = {"BRES 3x3 64->64 relu 23x23", CONV_3x3, 2, 23, 23, 64, 64, 64, 64, EPI_TMA, true, false, 64};
    Case r2 = {"BRES 3x3 64->64 relu 17x9", CONV_3x3, 3, 17, 9, 64, 64, 64, 64, EPI_TMA, true, false, 64};
    Case r3 = {"BRES 1x1 256->64 relu 92x92", CONV_1x1, 2, 92, 92, 256, 64, 64, 64, EPI_TMA, true, false, 64};
    for (Case* c : {&r1, &r2, &r3}) fails += run_case(*c, sms, true);
  }
  {  // halo-patch 3x3 convs: every instantiation, image sizes that are / are not multiples of the 8 x 16 tile
    Case h1 = {"HALO BRES 3x3 64->64 relu 92x92", CONV_3x3, 2, 92, 92, 64, 64, 64, 64, EPI_TMA, true, false, 64};
    Case h2 = {"HALO BRES 3x3 64->64 relu 46x46", CONV_3x3, 3, 46, 46, 64, 64, 64, 64, EPI_TMA, true, false, 64};
    Case h3 = {"HALO PAIR 3x3 128->128 relu 46x46", CONV_3x3, 3, 46, 46, 128, 128, 128, 128, EPI_TMA, true, false, 128};
    Case h5 = {"HALO 3x3 128->128 relu 46x46 bn64", CONV_3x3, 1, 46, 46, 128, 128, 128, 64, EPI_TMA, true, false, 128};
    Case h6 = {"HALO PAIR 3x3 256->128 relu 46x46 (head)", CONV_3x3, 2, 46, 46, 256, 128, 128, 128, EPI_TMA, true, false, 128};
    Case h7 = {"HALO PAIR 3x3 128->128 lin 56x56", CONV_3x3, 1, 56, 56, 128, 128, 128, 128, EPI_TMA, true, false, 0};
    Case h8 = {"HALO BRES 3x3 64->64 relu 13x15", CONV_3x3, 3, 13, 15, 64, 64, 64, 64, EPI_TMA, true, false, 64};
    for (Case* c : {&h1, &h2, &h3, &h5, &h6, &h7, &h8}) fails += run_case(*c, sms, true);
  }
  {  // fused block tails: both (N2, residual) instantiations, odd unit counts
    Case t2 = {"TAIL FOLD 1x1 64(+64)->256 relu 92x92 > 64", CONV_1x1, 2, 92, 92, 64, 256, 256, 256, EPI_TMA, true, false, 256, 1, 1, 64, 64};
    Case t3 = {"TAIL 1x1 128->512 +res relu 46x46 > 128", CONV_1x1, 3, 46, 46, 128, 512, 512, 256, EPI_TMA_RES, true, true, 512, 1, 1, 0, 128};
    for (Case* c : {&t2, &t3}) fails += run_case(*c, sms, true);
  }
  {  // 3x3 / transposed convs on flat pixel rows through the im2col tensor map (single CTAs, pairs, odd tile counts)
    Case a = {"IM2COL 3x3 256->256 relu 23x23 n64", CONV_3x3, 3, 23, 23, 256, 256, 256, 64, EPI_TMA, true, false, 256};
    Case b = {"IM2COL PAIR 3x3 256->256 relu 23x23", CONV_3x3, 3, 23, 23, 256, 256, 256, 256, EPI_TMA, true, false, 256};
    Case c = {"IM2COL PAIR 3x3 512->512 relu 23x23 (odd tile count)", CONV_3x3, 5, 23, 23, 512, 512, 512, 256, EPI_TMA, true, false, 512};
    Case d = {"IM2COL 3x3 128->128 relu 13x9 n64", CONV_3x3, 2, 13, 9, 128, 128, 128, 64, EPI_TMA, true, false, 128};
    Case g = {"IM2COL PAIR deconv4x4s2 256->192 head 23x23", CONV_DECONV4, 3, 23, 23, 256, 192, 191, 192, EPI_DECONV_HEAD, true, false, 128};
    for (Case* k : {&a, &b, &c, &d, &g}) fails += run_case(*k, sms, true);
  }
  fails += run_stem_pool(2, 368, sms);
  fails += run_stem_pool(2, 448, sms);
  fails += run_stem_pool(1, 64, sms);
  fails += run_stem_pool(1, 512, sms);
  if (big) {
    fails += run_stem_pool(32, 368, sms);
    fails += run_stem_pool(128, 368, sms);
    std::vector<Case> bigc = {
        {"BIG TMARES 1x1 64->256 +res 92x92 nb32", CONV_1x1, 32, 92, 92, 64, 256, 256, 256, EPI_TMA_RES, true, true, 256},
        {"BIG TMA 1x1 64->256 92x92 nb32", CONV_1x1, 32, 92, 92, 64, 256, 256, 256, EPI_TMA, true, false, 0},
        {"BIG TMA 3x3 64->64 92x92 nb32", CONV_3x3, 32, 92, 92, 64, 64, 64, 64, EPI_TMA, true, false, 64},
        {"BIG TMARES 1x1 256->1024 +res 23x23 nb128", CONV_1x1, 128, 23, 23, 256, 1024, 1024, 256, EPI_TMA_RES, true, true, 1024},
        {"BIG TMA 1x1 1024->256 23x23 nb128", CONV_1x1, 128, 23, 23, 1024, 256, 256, 256, EPI_TMA, true, false, 256},
        {"BIG TMA 1x1 512->128 46x46 nb128", CONV_1x1, 128, 46, 46, 512, 128, 128, 128, EPI_TMA, true, false, 128},
        {"BIG TMARES 1x1 128->512 +res 46x46 nb128", CONV_1x1, 128, 46, 46, 128, 512, 512, 256, EPI_TMA_RES, true, true, 512},
        {"BIG TMARES 1x1 64->256 +res 92x92 nb128", CONV_1x1, 128, 92, 92, 64, 256, 256, 256, EPI_TMA_RES, true, true, 256},
        {"BRES BIG 1x1 256->64 92x92 nb128", CONV_1x1, 128, 92, 92, 256, 64, 64, 64, EPI_TMA, true, false, 64},
        // fused block tails at full batch (compare: the unfused 2c kernels above + the stand-alone reduce convs)
        {"BIG TAIL 1x1 128->512 +res 46x46 nb128 > 128", CONV_1x1, 128, 46, 46, 128, 512, 512, 256, EPI_TMA_RES, true, true, 512, 1, 1, 0, 128},
        {"BIG TAIL FOLD 1x1 64(+64)->256 92x92 nb128 > 64", CONV_1x1, 128, 92, 92, 64, 256, 256, 256, EPI_TMA, true, false, 256, 1, 1, 64, 64},
        // halo patches, full batch
        {"BIG HALO BRES 3x3 64->64 92x92 nb128", CONV_3x3, 128, 92, 92, 64, 64, 64, 64, EPI_TMA, true, false, 64},
        {"BIG HALO PAIR 3x3 128->128 46x46 nb128", CONV_3x3, 128, 46, 46, 128, 128, 128, 128, EPI_TMA, true, false, 128},
        {"BIG HALO PAIR 3x3 256->128 46x46 nb128 (head)", CONV_3x3, 128, 46, 46, 256, 128, 128, 128, EPI_TMA, true, false, 128},
        // resident weights on spatial tiles and im2col, full batch
        {"BIG BRES S2 3x3 64->64 92->46 nb128", CONV_3x3, 128, 46, 46, 64, 64, 64, 64, EPI_TMA, true, false, 64, 2, 1},
        {"BIG IM2COL PAIR 3x3 256->256 23x23 nb128", CONV_3x3, 128, 23, 23, 256, 256, 256, 256, EPI_TMA, true, false, 256},
        {"BIG IM2COL PAIR 3x3 512->512 23x23 nb128", CONV_3x3, 128, 23, 23, 512, 512, 512, 256, EPI_TMA, true, false, 512},
        {"BIG IM2COL S2 PAIR 3x3 128->128 46->23 nb128", CONV_3x3, 128, 23, 23, 128, 128, 128, 128, EPI_TMA, true, false, 128, 2, 1},
        {"BIG IM2COL PAIR deconv4x4s2 256->192 head 23x23 nb128", CONV_DECONV4, 128, 23, 23, 256, 192, 191, 192, EPI_DECONV_HEAD, true, false, 128},
    };
    for (const auto& c : bigc) fails += run_case(c, sms, true);
  }
  printf("SELFTEST %s (%d failing cases)\n", fails == 0 ? "PASSED" : "FAILED", fails);
  return fails == 0 ? 0 : 1;
}
