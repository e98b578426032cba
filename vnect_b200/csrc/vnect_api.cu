// C ABI of the B200-native VNect hot path (see include/vnect_b200.h): handle, weight ingest, plan, entry points.
#include "vnect_b200.h"

#include <cmath>
#include <cstdarg>
#include <cstddef>
#include <cstdlib>
#include <cstring>
#include <tuple>
#include <map>
#include <algorithm>
#include <set>
#include <string>
#include <vector>

#include "conv_plan.cuh"
#include "prepost_kernels.cuh"

using namespace vnect;

namespace {

struct Act {
  __half* p = nullptr;
  int H = 0, W = 0, C = 0;
  int row_px = 0;       // row pitch in pixels (== W except for conv1's virtual layout)
  int64_t img_px = 0;   // image stride in pixels (== H*W except for conv1)
};

struct Step {
  int kind = 0;  // 0 = implicit-GEMM conv (conv_gemm_kernel), 3 = fused conv1 + pool1 (stem_roll_kernel)
  std::string name;
  ConvLaunch launch;
  StemPoolLaunch stem_pool;
};

struct HostVar {
  std::vector<float> data;
  std::vector<int64_t> shape;
};

}  // namespace

struct vnect_handle {
  vnect_config cfg{};
  int S = 368, hs = 46, n_scales = 1, cap_fw = 1, num_sms = 148;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  bool finalized = false;
  std::string err;
  long long launches = 0;
  std::map<std::string, HostVar> vars;
  std::vector<void*> allocs;
  std::map<std::string, Act> acts;
  std::vector<Step> steps;
  int conv_steps = 0;
  // stem input
  __half* x1 = nullptr;
  int stem_rpp = 0, stem_pitch = 0;
  // output maps, planar fp32 [cap_fw][84][hs][hs]
  float* maps = nullptr;
  // pre/post buffers
  size_t d_frames_bytes = 0;
  uint8_t* d_sq = nullptr;
  float* d_f32_in = nullptr;  // vnect_forward staging [cap_fw][S][S][3]
  ScaleTable* d_tables = nullptr;
  unsigned long long* d_post_trace = nullptr;  // VNECT_B200_POST_TRACE=1: phase timestamps of the last post-process launch
  std::vector<ScaleTable> h_tables;  // host copy: the post-process block's shared-memory plan is derived from it
  PyramidTable* d_pyr_tables = nullptr;
  uint32_t* d_norm_lut = nullptr;
  int pyr_src_rows = 1;         // most source rows a pyramid block stages
  bool x1_surround_ok = false;  // the constant surround of the shrunken scales is in place in every slot of x1
  FilterState *d_st2d = nullptr, *d_st3d = nullptr;
  double* d_j2_box = nullptr;
  float* d_j3_raw = nullptr;
  int* d_raw_argmax = nullptr;
  double* d_scores = nullptr;  // [max_frames][21] after d_raw_argmax's [max_frames][21][2] (PostParams::scores_off)
  unsigned int* d_counter = nullptr;
  double* d_prep3 = nullptr;   // [max_frames][21][3][3]: see PostParams::prep3
  double* d_filter_scratch = nullptr;
  // Two submission lanes: each owns its input staging, per-call meta (pinned host + device) and result buffers, so
  // the H2D copy of batch k+1 (copy stream) overlaps the kernels of batch k (compute stream).
  struct Lane {
    uint8_t* d_frames = nullptr;
    int* d_stream_ids = nullptr;
    double *d_t2d = nullptr, *d_t3d = nullptr;
    double* d_out2d = nullptr;
    float* d_out3d = nullptr;
    int* h_stream_ids = nullptr;
    double *h_t2d = nullptr, *h_t3d = nullptr;
    void* h_meta = nullptr;               // pinned block behind h_stream_ids / h_t2d / h_t3d (one H2D copy per call)
    size_t meta_bytes = 0;                // ids | t2d | t3d: what a uniform call copies
    // mixed-size calls: [max_frames] frame descriptors after the ids and timestamps in the same block (copied with
    // them), and the per-frame geometry the device derives from them.  Per lane: lane 1's table is written on the
    // copy stream while lane 0's kernels still read theirs.
    size_t table_off = 0;
    FrameDesc *h_table = nullptr, *d_table = nullptr;
    FrameGeom* d_geoms = nullptr;         // [max_frames]
    // sequence calls: the segment table of sequence_filter_kernel (n_seg, [max_frames + 1] starts, [max_frames] frame
    // indices) after the frame table, copied with it
    size_t seg_off = 0;
    int *h_seg = nullptr, *d_seg = nullptr;
    // calls with oriented frames: each frame's VNECT_ORIENT_* code ([max_frames]) after the segment table, copied with
    // the rest (a call takes its streams' codes at submission)
    size_t orient_off = 0;
    int *h_orient = nullptr, *d_orient = nullptr;
    // tracked calls with a recovering stream: each frame's threshold ([max_frames], vnect_set_track_recovery) after the
    // orientation codes, copied with the rest (a call takes its streams' thresholds at submission)
    size_t recover_off = 0;
    double *h_recover = nullptr, *d_recover = nullptr;
    unsigned int* h_nonfinite = nullptr;  // pinned + device-visible: set by the post-process when a batch of this lane met NaN / Inf maps
    cudaEvent_t copy_done = nullptr, done = nullptr;
    bool pending = false;
  } lanes[2];
  Lane* cur = &lanes[0];
  cudaStream_t copy_stream = nullptr;
  std::vector<unsigned int> seen_stamp;  // duplicate stream ids within a call (stage_frame_meta)
  unsigned int seen_epoch = 0;
  std::vector<int> seq_slot;             // stage_sequence_meta: a stream's segment in the current call
  std::vector<double> seq_t2d, seq_t3d;  // stage_sequence_meta: a stream's last timestamps as the call's frames advance
  unsigned device_calls = 0;
  // tracked streams (run_estimator.py:100-119): per-stream crop box on the device, per-call frame geometry
  int4* d_boxes = nullptr;         // [max_streams] (x, y, w, h)
  FrameGeom* d_geoms = nullptr;    // [max_frames]
  int* d_boxes_used = nullptr;     // [max_frames][4]
  std::vector<int32_t> orient;     // [max_streams] VNECT_ORIENT_* per stream (vnect_set_orientations), host only
  std::vector<double> recover;     // [max_streams] least mean score of a tracked frame (vnect_set_track_recovery), 0 = off
  double* score_req = nullptr;     // vnect_request_scores: where the next result-producing call writes its scores
  // CUDA graphs of the kernel sequence of one estimate call, keyed by everything baked into the kernel parameters.
  // First use of a key runs directly (warm-up), the second captures, later ones replay: ~50 launches -> 1.
  // (lane + tracked, n_frames, H, W, pitch, frame_stride, frames, out2d, out3d, format, uv_pitch, u_offset, v_offset).
  // Mixed-size calls read sizes and addresses from the lane's device table, so only (4 + lane + 2 * tracked, n_frames,
  // out2d, out3d, format) is set in their key: one graph serves every composition of a batch.
  typedef std::tuple<int, int, int, int, long long, long long, const void*, const void*, const void*, int, long long,
                     long long, long long> GraphKey;
  struct GraphEntry {
    cudaGraphExec_t exec = nullptr;
    long long launches = 0;
    bool unusable = false;
    unsigned long long last_use = 0;
  };
  static constexpr size_t kMaxGraphs = 16;  // a video loop changes its crop size every frame: bound the cache (LRU)
  unsigned long long graph_clock = 0;
  std::map<GraphKey, GraphEntry> graphs;
  bool use_graphs = true;
  std::vector<double> last_t2d, last_t3d;  // host mirror of the filters' last timestamps (NaN = none yet)
  PyramidParams pyr{};
  double* d_packed = nullptr;  // caller-owned device buffer [max_frames][21][5] (vnect_set_packed_results) or null
  FilterState* d_st_ang = nullptr;      // [max_streams][8] one-euro filters of Joints2Angles (joints2angles.py:35-42)
  std::vector<double> last_t_ang;
  float* d_ang_in = nullptr;            // [max_frames][21][3]
  double* d_ang_t = nullptr;            // [max_frames]
  int* d_ang_ids = nullptr;
  double* d_ang_out = nullptr;          // [max_frames][8]
  unsigned int* d_nonfinite = nullptr;  // (frame, joint) blocks whose maps held NaN / Inf since the last check
  unsigned long long* d_scan = nullptr; // vnect_check_finite scratch
};

// Every entry point runs on the handle's device and leaves the caller's current device as it found it: function
// attributes, streams and allocations are per device, and a process may hold one handle per GPU.
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) switched = (cudaSetDevice(dev) == cudaSuccess);
  }
  ~DeviceGuard() {
    if (switched) cudaSetDevice(prev);
  }
};
#define ON_DEVICE(h) DeviceGuard device_guard_((h)->cfg.device)

static int fail(vnect_t* h, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (h) h->err = buf;
  return code;
}

#define CU(h, call)                                                                                       \
  do {                                                                                                    \
    cudaError_t e_ = (call);                                                                              \
    if (e_ != cudaSuccess) return fail(h, VNECT_E_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

template <typename T>
static int dev_alloc(vnect_t* h, T** p, size_t count, bool zero = true) {
  void* q = nullptr;
  CU(h, cudaMalloc(&q, count * sizeof(T) + 256));
  if (zero) CU(h, cudaMemset(q, 0, count * sizeof(T) + 256));
  h->allocs.push_back(q);
  *p = reinterpret_cast<T*>(q);
  return VNECT_OK;
}

static inline int grid_for(int64_t total, int threads, int sms) {
  int64_t b = (total + threads - 1) / threads;
  int64_t cap = (int64_t)sms * 16;
  return (int)(b < cap ? (b < 1 ? 1 : b) : cap);
}

// ------------------------------------------------------------------------------------------------ weights
static const char* kBnVars[4] = {"gamma", "beta", "moving_mean", "moving_variance"};

struct ConvDef {
  std::string scope;
  int k, cin, cout;
};

static std::vector<ConvDef> conv_defs() {
  std::vector<ConvDef> d;
  d.reserve(64);
  auto add = [&](const std::string& s, int k, int ci, int co) { d.push_back({s, k, ci, co}); };
  auto block = [&](const std::string& pre, int cin, int mid, int cout, bool proj, const std::string& suf) {
    if (proj) add(pre + "_branch1" + suf, 1, cin, cout);
    add(pre + "_branch2a" + suf, 1, cin, mid);
    add(pre + "_branch2b" + suf, 3, mid, mid);
    add(pre + "_branch2c" + suf, 1, mid, cout);
  };
  add("conv1", 7, 3, 64);
  block("res2a", 64, 64, 256, true, "");
  block("res2b", 256, 64, 256, false, "");
  block("res2c", 256, 64, 256, false, "");
  block("res3a", 256, 128, 512, true, "");
  for (const char* b : {"res3b", "res3c", "res3d"}) block(b, 512, 128, 512, false, "");
  block("res4a", 512, 256, 1024, true, "");
  for (const char* b : {"res4b", "res4c", "res4d", "res4e", "res4f"}) block(b, 1024, 256, 1024, false, "");
  block("res5a", 1024, 512, 1024, true, "_new");
  add("res5b_branch2a_new", 1, 1024, 256);
  add("res5b_branch2b_new", 3, 256, 128);
  add("res5b_branch2c_new", 1, 128, 256);
  add("res5c_branch2b", 3, 212, 128);
  return d;
}

static bool expected_shape(const std::string& name, std::vector<int64_t>* shape) {
  const size_t slash = name.find('/');
  if (slash == std::string::npos) return false;
  const std::string scope = name.substr(0, slash), leaf = name.substr(slash + 1);
  if (scope == "bn5c_branch2a") {
    for (const char* v : kBnVars)
      if (leaf == v) {
        *shape = {128};
        return true;
      }
    return false;
  }
  if (leaf == "kernel") {
    if (scope == "res5c_branch1a") { *shape = {4, 4, 63, 256}; return true; }
    if (scope == "res5c_branch2a") { *shape = {4, 4, 128, 256}; return true; }
    if (scope == "res5c_branch2c") { *shape = {1, 1, 128, 84}; return true; }
    return false;
  }
  for (const ConvDef& c : conv_defs())
    if (scope == c.scope) {
      if (leaf == "weights") { *shape = {c.k, c.k, c.cin, c.cout}; return true; }
      if (leaf == "biases") { *shape = {c.cout}; return true; }
    }
  return false;
}

static std::vector<__half> to_half(const std::vector<float>& v) {
  std::vector<__half> o(v.size());
  for (size_t i = 0; i < v.size(); ++i) o[i] = __float2half_rn(v[i]);
  return o;
}

// HWIO [k,k,cin,cout] -> [n_pad][k*k*cin_pad], K-major per output channel, zero padded
static std::vector<float> pack_conv(const HostVar& w, int k, int cin, int cout, int cin_pad, int n_pad) {
  std::vector<float> b((size_t)n_pad * k * k * cin_pad, 0.f);
  for (int ky = 0; ky < k; ++ky)
    for (int kx = 0; kx < k; ++kx)
      for (int ci = 0; ci < cin; ++ci)
        for (int co = 0; co < cout; ++co)
          b[(size_t)co * k * k * cin_pad + (size_t)(ky * k + kx) * cin_pad + ci] =
              w.data[(((size_t)ky * k + kx) * cin + ci) * cout + co];
  return b;
}

// stem: [64][7 rows][8 px][4 ch] (px 7 and ch 3 are zero)
static std::vector<float> pack_stem(const HostVar& w) {
  std::vector<float> b((size_t)64 * 224, 0.f);
  for (int ky = 0; ky < 7; ++ky)
    for (int kx = 0; kx < 7; ++kx)
      for (int c = 0; c < 3; ++c)
        for (int co = 0; co < 64; ++co) b[(size_t)co * 224 + ky * 32 + kx * 4 + c] = w.data[((ky * 7 + kx) * 3 + c) * 64 + co];
  return b;
}

// Both transposed convs + folded batch norm as 4 phase GEMMs: [4 phases][192 cols][4 taps][256 ch].
// cols 0-127 = res5c_branch2a * bn scale, 128-190 = res5c_branch1a, 191 = 0.  TF kernel layout [kh,kw,out,in].
static std::vector<float> pack_deconv(const HostVar& w2a, const HostVar& w1a, const std::vector<float>& bn_scale) {
  std::vector<float> b((size_t)4 * 192 * 1024, 0.f);
  for (int ph = 0; ph < 4; ++ph) {
    const int py = ph >> 1, px = ph & 1;
    for (int a = 0; a < 2; ++a)
      for (int bb = 0; bb < 2; ++bb) {
        const int ky = py == 0 ? (a == 0 ? 1 : 3) : (a == 0 ? 0 : 2);
        const int kx = px == 0 ? (bb == 0 ? 1 : 3) : (bb == 0 ? 0 : 2);
        for (int col = 0; col < 191; ++col)
          for (int ci = 0; ci < 256; ++ci) {
            float v;
            if (col < 128)
              v = w2a.data[(((size_t)ky * 4 + kx) * 128 + col) * 256 + ci] * bn_scale[col];
            else
              v = w1a.data[(((size_t)ky * 4 + kx) * 63 + (col - 128)) * 256 + ci];
            b[((size_t)ph * 192 + col) * 1024 + (size_t)(a * 2 + bb) * 256 + ci] = v;
          }
      }
  }
  return b;
}

template <typename T>
static int upload(vnect_t* h, const std::vector<T>& v, T** out) {
  int rc = dev_alloc(h, out, v.size(), false);
  if (rc) return rc;
  CU(h, cudaMemcpy(*out, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  return VNECT_OK;
}

// ------------------------------------------------------------------------------------------------ plan
static int new_act(vnect_t* h, const std::string& name, int H, int W, int C) {
  Act a;
  a.H = H; a.W = W; a.C = C; a.row_px = W; a.img_px = (int64_t)H * W;
  int rc = dev_alloc(h, &a.p, (size_t)h->cap_fw * H * W * C, true);
  if (rc) return rc;
  h->acts[name] = a;
  return VNECT_OK;
}

struct ConvOpts {
  bool relu = true;
  std::string residual;  // act name or empty
  int in_stride = 1;     // 2: compute the conv at even input pixels only (output grid is half-size)
  int res_stride = 1;    // 2: the residual is a full-size tensor read at even pixels
  // fused block tail (block_tail.cuh): scope of the NEXT block's 1x1 reduce conv, computed from this conv's output
  // while it is still in shared memory; its output activation is created under that scope's name
  std::string chain_scope;
  int chain_cout = 0;
};

// uploads the chained conv's weights ([n2][cout] K-major fp16) and bias, creates its output activation
static int attach_chain(vnect_t* h, ConvSpec& s, const ConvOpts& o, int cout, int OH, int OW) {
  const HostVar& w = h->vars.at(o.chain_scope + "/weights");
  const HostVar& b = h->vars.at(o.chain_scope + "/biases");
  __half* dw = nullptr;
  float* db = nullptr;
  int rc = upload(h, to_half(pack_conv(w, 1, cout, o.chain_cout, cout, o.chain_cout)), &dw);
  if (rc) return rc;
  if ((rc = upload(h, b.data, &db))) return rc;
  if ((rc = new_act(h, o.chain_scope, OH, OW, o.chain_cout))) return rc;
  s.w2 = dw;
  s.bias2 = db;
  s.n2 = o.chain_cout;
  s.out2 = h->acts.at(o.chain_scope).p;
  return VNECT_OK;
}

// The block tail is fused with the next block's reduce conv on the throughput plans (256-column tiles on CTA pairs).
// Measured at batch 128 (profiles/r02_gpu_check_tail.log): the fused tail beats the two kernels it replaces where the
// pair is HBM-bound -- res2a (224 vs 262 us), res2c (78 vs 101), res3b / res3c (137 vs 172) -- and loses where the
// second accumulator is 256 wide (single-buffered TMEM, res3d / res4* / res5a: 120 vs 107 us) or the main GEMM carries a
// folded projection with a 128-wide second conv (res3a: 165 vs 161).
static bool can_chain(const ConvSpec& s, const ConvOpts& o, int cout) {
  if (o.chain_scope.empty() || s.block_n != kTailBlockN || cout % kTailBlockN != 0) return false;
  return o.chain_cout == 64 || (o.chain_cout == 128 && s.residual != nullptr);
}

// Output-channel tile.  Throughput plans (many forwards) use the widest tile; latency plans (a handful of forwards, e.g.
// the drop-in estimator: one frame x n_scales) use 64-wide tiles so that 4x more CTAs share each layer's serial K loop.
static int pick_block_n(int n, int cap_fw) {
  if (cap_fw <= 8) return 64;
  return n >= 256 ? 256 : n >= 128 ? 128 : 64;
}

static int add_conv(vnect_t* h, const std::string& scope, int k, const std::string& in, const std::string& out,
                    int cin, int cout, const ConvOpts& o) {
  const Act& ai = h->acts.at(in);
  const HostVar& w = h->vars.at(scope + "/weights");
  const HostVar& b = h->vars.at(scope + "/biases");
  const int cin_pad = ai.C;
  __half* dw = nullptr;
  float* db = nullptr;
  int rc = upload(h, to_half(pack_conv(w, k, cin, cout, cin_pad, cout)), &dw);
  if (rc) return rc;
  rc = upload(h, b.data, &db);
  if (rc) return rc;
  const int OH = ai.H / o.in_stride, OW = ai.W / o.in_stride;
  rc = new_act(h, out, OH, OW, cout);
  if (rc) return rc;
  ConvSpec s;
  s.kind = k == 1 ? CONV_1x1 : CONV_3x3;
  s.NB = h->cap_fw; s.H = OH; s.W = OW;
  s.in = ai.p; s.cin_pad = cin_pad; s.in_stride = o.in_stride;
  s.w = dw; s.n_pad = cout; s.n_valid = cout; s.block_n = pick_block_n(cout, h->cap_fw);
  s.bias = db; s.relu_cols = o.relu ? cout : 0;
  if (!o.residual.empty()) {
    const Act& r = h->acts.at(o.residual);
    if (r.H != OH * o.res_stride || r.W != OW * o.res_stride || r.C != cout)
      return fail(h, VNECT_E_INVALID, "residual shape mismatch at %s", scope.c_str());
    s.residual = r.p; s.ldr = r.C; s.res_stride = o.res_stride;
  }
  // outputs leave through swizzled smem + TMA tensor stores; residual tiles are prefetched by TMA
  s.out = h->acts.at(out).p; s.ldc = cout;
  s.epi = s.residual ? EPI_TMA_RES : EPI_TMA;  // resident weights, halo patches or im2col: conv_path() in build_conv
  Step st;
  st.kind = 0; st.name = scope;
  if (k == 1 && can_chain(s, o, cout)) {
    if ((rc = attach_chain(h, s, o, cout, OH, OW))) return rc;
    st.name = scope + ">" + o.chain_scope;
  }
  std::string err;
  if (!build_conv(s, h->num_sms, &st.launch, &err)) return fail(h, VNECT_E_CUDA, "%s: %s", scope.c_str(), err.c_str());
  h->steps.push_back(st);
  return VNECT_OK;
}

// Last conv of a projection block with the shortcut folded in (vnect_model.py:32-41, 64-73, 106-115, 168-177):
//   relu(W_2c * b + bias_2c + W_1 * x + bias_1) == relu([W_2c | W_1] * [b ; x] + (bias_2c + bias_1))
// one GEMM whose K runs over the 3x3's output and then over the block input; the branch1 tensor never exists.
static int add_proj_tail(vnect_t* h, const std::string& scope2c, const std::string& scope1, const std::string& in_b,
                         const std::string& in_x, const std::string& out, int mid, int cin, int cout,
                         const ConvOpts& o = ConvOpts()) {
  const Act& ab = h->acts.at(in_b);
  const Act& ax = h->acts.at(in_x);
  if (ab.H != ax.H || ab.W != ax.W || ab.C != mid || ax.C != cin)
    return fail(h, VNECT_E_INVALID, "projection fold shape mismatch at %s", scope2c.c_str());
  const HostVar& w2 = h->vars.at(scope2c + "/weights");
  const HostVar& w1 = h->vars.at(scope1 + "/weights");
  const HostVar& b2 = h->vars.at(scope2c + "/biases");
  const HostVar& b1 = h->vars.at(scope1 + "/biases");
  const int K = mid + cin;
  std::vector<float> w((size_t)cout * K), bias(cout);
  for (int co = 0; co < cout; ++co) {
    for (int ci = 0; ci < mid; ++ci) w[(size_t)co * K + ci] = w2.data[(size_t)ci * cout + co];
    for (int ci = 0; ci < cin; ++ci) w[(size_t)co * K + mid + ci] = w1.data[(size_t)ci * cout + co];
    bias[co] = b2.data[co] + b1.data[co];
  }
  __half* dw = nullptr;
  float* db = nullptr;
  int rc = upload(h, to_half(w), &dw);
  if (rc) return rc;
  if ((rc = upload(h, bias, &db))) return rc;
  if ((rc = new_act(h, out, ab.H, ab.W, cout))) return rc;
  ConvSpec s;
  s.kind = CONV_1x1;
  s.NB = h->cap_fw; s.H = ab.H; s.W = ab.W;
  s.in = ab.p; s.cin_pad = mid; s.in2 = ax.p; s.cin2_pad = cin;
  s.w = dw; s.n_pad = cout; s.n_valid = cout; s.block_n = pick_block_n(cout, h->cap_fw);
  s.bias = db; s.relu_cols = cout;
  s.out = h->acts.at(out).p; s.ldc = cout; s.epi = EPI_TMA;
  Step st;
  st.kind = 0; st.name = scope2c + "+" + scope1;
  if (can_chain(s, o, cout)) {
    if ((rc = attach_chain(h, s, o, cout, ab.H, ab.W))) return rc;
    st.name += ">" + o.chain_scope;
  }
  std::string err;
  if (!build_conv(s, h->num_sms, &st.launch, &err)) return fail(h, VNECT_E_CUDA, "%s: %s", st.name.c_str(), err.c_str());
  h->steps.push_back(st);
  return VNECT_OK;
}

// bottleneck block (reference: src/vnect_model.py:31-177); `a_override` replaces the 3x3's input (the res2c wiring,
// :56).  even_only: the block's output feeds nothing but stride-2 1x1 convs (res2c -> res3a, res3d -> res4a), so
// the 3x3, the last 1x1 and the residual add are evaluated at even pixels only -- same values, a quarter of the work.
static int add_block(vnect_t* h, const std::string& pre, const std::string& in, int cin, int mid, int cout, bool proj,
                     const std::string& suf, bool even_only, const std::string& a_override = "",
                     const std::string& chain_scope = "", int chain_cout = 0) {
  int rc;
  ConvOpts relu;
  std::string a = a_override;
  if (a.empty()) {
    a = pre + "_branch2a" + suf;
    if (!h->acts.count(a)) {  // otherwise the previous block's fused tail has already computed it
      rc = add_conv(h, a, 1, in, a, cin, mid, relu);
      if (rc) return rc;
    }
  }
  ConvOpts mid3; mid3.in_stride = even_only ? 2 : 1;
  rc = add_conv(h, pre + "_branch2b" + suf, 3, a, pre + "_branch2b" + suf, mid, mid, mid3);
  if (rc) return rc;
  ConvOpts last; last.relu = true;
  last.chain_scope = chain_scope; last.chain_cout = chain_cout;
  if (proj)
    return add_proj_tail(h, pre + "_branch2c" + suf, pre + "_branch1" + suf, pre + "_branch2b" + suf, in, pre, mid, cin, cout, last);
  // the residual is read at the pixels this block is evaluated at: stride 2 into a full-size input, stride 1 when the
  // input itself is already an even-pixel tensor (res2c reading res2b)
  last.residual = in;
  last.res_stride = h->acts.at(in).H / h->acts.at(pre + "_branch2b" + suf).H;
  return add_conv(h, pre + "_branch2c" + suf, 1, pre + "_branch2b" + suf, pre, mid, cout, last);
}

static void set_batch(ConvLaunch& L, int nb, int sms) {
  ConvGemmParams& p = L.p;
  p.NB = nb;
  p.M = nb * p.H * p.W;
  p.num_m_tiles = p.mode == 0 ? (p.M + kBlockM - 1) / kBlockM : nb * p.tiles_x * p.tiles_y;
  L.grid = L.n2 ? tail_grid(p, sms) : conv_grid(p, L.cg, sms);
}

// cv2 INTER_LINEAR coordinate rule on the host, identical arithmetic to cv_linear_coord (double -> float)
static void host_linear_coord(int d, double inv_scale, int src, bool reset, int* i_out, float* f_out) {
  const double fd = ((double)d + 0.5) * inv_scale - 0.5;
  float f = (float)fd;
  int i = (int)std::floor(f);
  f = f - (float)i;
  if (reset) {
    if (i < 0) { i = 0; f = 0.f; }
    if (i >= src - 1) { i = src - 1; f = 0.f; }
  }
  *i_out = i;
  *f_out = f;
}

static inline int cv_round_host(double v) { return (int)std::nearbyint(v); }

static int build_tables(vnect_t* h) {
  std::vector<ScaleTable> t(h->n_scales);
  const int hs = h->hs;
  for (int s = 0; s < h->n_scales; ++s) {
    ScaleTable& T = t[s];
    memset(&T, 0, sizeof T);
    const double sc = h->cfg.scales[s];
    // estimator.py:112-120: rescale = 1.0 / s; cv2.resize(fx = fy = rescale); centre crop of hs cells
    const double rescale = 1.0 / sc;
    const int R = cv_round_host(hs * rescale);
    // cv::resize copies the source when the destination size equals the source size, so every scale whose resized
    // map keeps hs cells (s > hs / (hs + 0.5), not only s = 1) is a plain copy, not a resample with inv = s
    if (R == hs) {
      T.identity = 1;
      continue;
    }
    const double inv = 1.0 / rescale;
    const int crop0 = R / 2 - hs / 2;
    for (int c = 0; c < hs; ++c) {
      int i;
      float f;
      host_linear_coord(c + crop0, inv, hs, true, &i, &f);
      T.i0[c] = (short)i;
      T.i1[c] = (short)std::min(i + 1, hs - 1);
      T.a0[c] = 1.f - f;
      T.a1[c] = f;
      host_linear_coord(c + crop0, inv, hs, false, &i, &f);
      T.j0[c] = (short)std::min(std::max(i, 0), hs - 1);
      T.j1[c] = (short)std::min(std::max(i + 1, 0), hs - 1);
      T.b0[c] = 1.f - f;
      T.b1[c] = f;
      int b0_bits, b1_bits;
      memcpy(&b0_bits, &T.b0[c], 4);
      memcpy(&b1_bits, &T.b1[c], 4);
      T.rowpk[c] = make_int4(T.j0[c] * hs, T.j1[c] * hs, b0_bits, b1_bits);
    }
    T.row_lo = hs - 1;
    T.row_hi = 0;
    for (int c = 0; c < hs; ++c) {
      T.row_lo = std::min<int>(T.row_lo, T.j0[c]);
      T.row_hi = std::max<int>(T.row_hi, T.j1[c]);
    }
  }
  h->h_tables = t;
  return upload(h, t, &h->d_tables);
}

constexpr size_t kPyrMaxSmem = 160 * 1024;  // dynamic shared memory of pyramid_kernel's staged source rows

// The pyramid's per-scale geometry (h->pyr: R, pad0, 1 / s, the magic divisors) and resize tables, and the most source
// rows one block stages (h->pyr_src_rows).  Host arithmetic only: vnect_create refuses a scale list whose staged rows
// do not fit in kPyrMaxSmem before anything is allocated.
static void pyramid_tables(vnect_t* h, std::vector<PyramidTable>* ptab_out) {
  const int S = h->S;
  PyramidParams& py = h->pyr;
  py.S = S; py.n_scales = h->n_scales;
  std::vector<PyramidTable>& ptab = *ptab_out;
  ptab.assign(h->n_scales, PyramidTable{});
  h->pyr_src_rows = 1;
  for (int i = 0; i < h->n_scales; ++i) {
    const double sc = h->cfg.scales[i];
    py.R[i] = sc < 1.0 ? cv_round_host(S * sc) : S;  // estimator.py:77: only scales < 1 are resized
    py.pad0[i] = (S - py.R[i]) / 2;
    py.inv_scale[i] = 1.0 / sc;
    for (int d = 0; d < py.R[i] && py.R[i] != S; ++d) {  // same arithmetic as cv_linear_coord / cv_coef on the device
      int ix, iy;
      float fx, fy;
      host_linear_coord(d, py.inv_scale[i], S, true, &ix, &fx);
      host_linear_coord(d, py.inv_scale[i], S, false, &iy, &fy);
      const unsigned int a0 = (unsigned int)std::nearbyint((1.f - fx) * 2048.f), a1 = (unsigned int)std::nearbyint(fx * 2048.f);
      ptab[i].xt[d].x = (unsigned int)(4 * ix) | ((unsigned int)(4 * std::min(ix + 1, S - 1)) << 16);
      ptab[i].xt[d].y = a0 | (a1 << 16);
      ptab[i].yt[d].x = (short)std::min(std::max(iy, 0), S - 1);
      ptab[i].yt[d].y = (short)std::min(std::max(iy + 1, 0), S - 1);
      ptab[i].yt[d].z = (short)std::nearbyint((1.f - fy) * 2048.f);
      ptab[i].yt[d].w = (short)std::nearbyint(fy * 2048.f);
    }
    py.r_magic[i] = (unsigned int)((1ull << 32) / (unsigned long long)py.R[i]) + 1u;
    // source rows one block of kPyrRows output rows samples
    for (int y0 = 0; y0 < py.R[i] && py.R[i] != S; y0 += 1) {
      const int y1 = std::min(y0 + kPyrRows, py.R[i]) - 1;
      h->pyr_src_rows = std::max(h->pyr_src_rows, ptab[i].yt[y1].y - ptab[i].yt[y0].x + 1);
    }
  }
  py.q_magic = (unsigned int)((1ull << 32) / (unsigned long long)(S / 4)) + 1u;
}

static int alloc_prepost(vnect_t* h, const std::vector<PyramidTable>& ptab) {
  const int S = h->S, nb = h->cap_fw;
  int rc;
  // stem input: parity-split, zero-padded NHWC4 (zeros are written once here and never touched again)
  h->stem_rpp = S / 2 + 3;
  h->stem_pitch = (S + 6) * 4;
  // + slack: the last strip of the last image reads a few KB past its parity plane (stem_roll.cuh)
  if ((rc = dev_alloc(h, &h->x1, (size_t)nb * 2 * h->stem_rpp * h->stem_pitch + 16384, true))) return rc;
  if ((rc = dev_alloc(h, &h->maps, (size_t)nb * 84 * h->hs * h->hs, true))) return rc;
  const int mf = h->cfg.max_frames, ms = h->cfg.max_streams;
  h->d_frames_bytes = (size_t)mf * h->cfg.max_input_h * h->cfg.max_input_w * 3;
  CU(h, cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
  for (auto& L : h->lanes) {
    if ((rc = dev_alloc(h, &L.d_frames, h->d_frames_bytes))) return rc;
    {  // ids | t2d | t3d in one block on both sides: one H2D copy per call
      const size_t off_t2 = ((size_t)mf * sizeof(int) + 15) & ~size_t(15), off_t3 = off_t2 + (size_t)mf * sizeof(double);
      L.meta_bytes = off_t3 + (size_t)mf * sizeof(double);
      L.table_off = (L.meta_bytes + 15) & ~size_t(15);
      L.seg_off = L.table_off + (size_t)mf * sizeof(FrameDesc);
      L.orient_off = L.seg_off + (size_t)(2 * mf + 2) * sizeof(int);
      L.recover_off = (L.orient_off + (size_t)mf * sizeof(int) + 7) & ~size_t(7);
      const size_t block = L.recover_off + (size_t)mf * sizeof(double);
      uint8_t* d_meta = nullptr;
      if ((rc = dev_alloc(h, &d_meta, block))) return rc;
      L.d_stream_ids = reinterpret_cast<int*>(d_meta);
      L.d_t2d = reinterpret_cast<double*>(d_meta + off_t2);
      L.d_t3d = reinterpret_cast<double*>(d_meta + off_t3);
      L.d_table = reinterpret_cast<FrameDesc*>(d_meta + L.table_off);
      L.d_seg = reinterpret_cast<int*>(d_meta + L.seg_off);
      L.d_orient = reinterpret_cast<int*>(d_meta + L.orient_off);
      L.d_recover = reinterpret_cast<double*>(d_meta + L.recover_off);
      CU(h, cudaMallocHost(&L.h_meta, block));
      memset(L.h_meta, 0, block);
      L.h_stream_ids = reinterpret_cast<int*>(L.h_meta);
      L.h_t2d = reinterpret_cast<double*>(static_cast<uint8_t*>(L.h_meta) + off_t2);
      L.h_t3d = reinterpret_cast<double*>(static_cast<uint8_t*>(L.h_meta) + off_t3);
      L.h_table = reinterpret_cast<FrameDesc*>(static_cast<uint8_t*>(L.h_meta) + L.table_off);
      L.h_seg = reinterpret_cast<int*>(static_cast<uint8_t*>(L.h_meta) + L.seg_off);
      L.h_orient = reinterpret_cast<int*>(static_cast<uint8_t*>(L.h_meta) + L.orient_off);
      L.h_recover = reinterpret_cast<double*>(static_cast<uint8_t*>(L.h_meta) + L.recover_off);
    }
    if ((rc = dev_alloc(h, &L.d_geoms, mf))) return rc;
    if ((rc = dev_alloc(h, &L.d_out2d, (size_t)mf * kJoints * 2))) return rc;
    if ((rc = dev_alloc(h, &L.d_out3d, (size_t)mf * kJoints * 3))) return rc;
    CU(h, cudaHostAlloc(&L.h_nonfinite, sizeof(unsigned int), cudaHostAllocMapped));
    *L.h_nonfinite = 0;
    CU(h, cudaEventCreateWithFlags(&L.copy_done, cudaEventDisableTiming));
    CU(h, cudaEventCreateWithFlags(&L.done, cudaEventDisableTiming));
  }
  if ((rc = dev_alloc(h, &h->d_sq, (size_t)mf * S * S * 3))) return rc;
  if ((rc = dev_alloc(h, &h->d_f32_in, (size_t)nb * S * S * 3))) return rc;
  if ((rc = build_tables(h))) return rc;
  if ((rc = dev_alloc(h, &h->d_st2d, (size_t)ms * kJoints * 2))) return rc;
  if ((rc = dev_alloc(h, &h->d_st3d, (size_t)ms * kJoints * 3))) return rc;
  if ((rc = dev_alloc(h, &h->d_j2_box, (size_t)mf * kJoints * 2))) return rc;
  if ((rc = dev_alloc(h, &h->d_j3_raw, (size_t)mf * kJoints * 3))) return rc;
  // the raw argmax, then the scores of a SCORES post-process; both are per call and ordered on the handle's stream
  if ((rc = dev_alloc(h, &h->d_raw_argmax, (size_t)mf * kJoints * 4))) return rc;
  h->d_scores = reinterpret_cast<double*>(h->d_raw_argmax + (size_t)mf * kJoints * 2);
  if ((rc = dev_alloc(h, &h->d_counter, mf))) return rc;
  if ((rc = dev_alloc(h, &h->d_prep3, (size_t)mf * kJoints * 9))) return rc;
  if (getenv("VNECT_B200_POST_TRACE") && (rc = dev_alloc(h, &h->d_post_trace, (size_t)mf * kJoints * 16))) return rc;
  if ((rc = dev_alloc(h, &h->d_filter_scratch, 64))) return rc;
  if ((rc = dev_alloc(h, &h->d_st_ang, (size_t)ms * 8))) return rc;
  if ((rc = dev_alloc(h, &h->d_ang_in, (size_t)mf * kJoints * 3))) return rc;
  if ((rc = dev_alloc(h, &h->d_ang_t, mf))) return rc;
  if ((rc = dev_alloc(h, &h->d_ang_ids, mf))) return rc;
  if ((rc = dev_alloc(h, &h->d_ang_out, (size_t)mf * 8))) return rc;
  h->last_t_ang.assign(ms, NAN);
  if ((rc = dev_alloc(h, &h->d_nonfinite, 1))) return rc;
  if ((rc = dev_alloc(h, &h->d_scan, 1))) return rc;
  if ((rc = dev_alloc(h, &h->d_boxes, ms))) return rc;
  if ((rc = dev_alloc(h, &h->d_geoms, mf))) return rc;
  if ((rc = dev_alloc(h, &h->d_boxes_used, (size_t)mf * 4))) return rc;
  h->orient.assign(ms, VNECT_ORIENT_IDENTITY);
  h->recover.assign(ms, 0.0);
  h->last_t2d.assign(ms, NAN);
  h->last_t3d.assign(ms, NAN);
  PyramidParams& py = h->pyr;
  py.rows_per_parity = h->stem_rpp; py.row_pitch = h->stem_pitch;
  if ((rc = upload(h, ptab, &h->d_pyr_tables))) return rc;
  py.tables = h->d_pyr_tables;
  // float32(v) / 255 - 0.4 -> fp16 (estimator.py:81 in float32, then the operand precision of the stem)
  std::vector<uint32_t> lut(256);
  for (int v = 0; v < 256; ++v) {
    const __half hv = __float2half_rn((float)v / 255.f - 0.4f);
    unsigned short bits;
    memcpy(&bits, &hv, 2);
    lut[v] = bits;
  }
  if ((rc = upload(h, lut, &h->d_norm_lut))) return rc;
  py.lut = h->d_norm_lut;
  py.full = 0;
  return VNECT_OK;
}

// ------------------------------------------------------------------------------------------------ C ABI
extern "C" {

const char* vnect_version(void) { return "vnect_b200 0.1 (sm_100a; fp16 operands, fp32 accumulate)"; }

const char* vnect_last_error(vnect_t* h) { return h ? h->err.c_str() : "null handle"; }

int vnect_create(vnect_t** out, const vnect_config* cfg) {
  if (!out || !cfg) return VNECT_E_INVALID;
  *out = nullptr;
  vnect_t* h = new vnect_handle();
  *out = h;  // returned even on failure so the caller can read the error, then destroy
  h->cfg = *cfg;
  if (cfg->box_size < 64 || cfg->box_size % 16 != 0 || cfg->box_size / 8 > kMaxHm || cfg->box_size > kMaxBox)
    return fail(h, VNECT_E_INVALID, "box_size %d must be a multiple of 16 in [64, %d]", cfg->box_size, kMaxHm * 8);
  if (cfg->n_scales < 1 || cfg->n_scales > kMaxScales) return fail(h, VNECT_E_INVALID, "n_scales out of range");
  for (int i = 0; i < cfg->n_scales; ++i)
    if (!(cfg->scales[i] > 0.0 && cfg->scales[i] <= 1.0))
      return fail(h, VNECT_E_INVALID, "scale %g not in (0, 1]", cfg->scales[i]);
  if (cfg->max_frames < 1 || cfg->max_streams < 1) return fail(h, VNECT_E_INVALID, "max_frames/max_streams must be >= 1");
  h->S = cfg->box_size;
  h->hs = h->S / 8;
  h->n_scales = cfg->n_scales;
  h->cap_fw = cfg->max_frames * cfg->n_scales;
  std::vector<PyramidTable> ptab;
  pyramid_tables(h, &ptab);
  if ((size_t)h->pyr_src_rows * h->S * 4 > kPyrMaxSmem)
    return fail(h, VNECT_E_INVALID, "pyramid scale too small: a block stages %d source rows (%zu bytes, at most %zu)",
                h->pyr_src_rows, (size_t)h->pyr_src_rows * h->S * 4, kPyrMaxSmem);
  if (h->cfg.max_input_h <= 0) h->cfg.max_input_h = h->S;
  if (h->cfg.max_input_w <= 0) h->cfg.max_input_w = h->S;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(h, VNECT_E_CUDA, "no CUDA device: this library has no CPU path");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(h, VNECT_E_INVALID, "device %d not in [0, %d)", cfg->device, ndev);
  ON_DEVICE(h);  // the caller's current device is restored on return
  cudaDeviceProp prop;
  CU(h, cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10) return fail(h, VNECT_E_CUDA, "device %s is sm_%d%d; this library is built for sm_100a only", prop.name, prop.major, prop.minor);
  h->num_sms = prop.multiProcessorCount;
  CU(h, cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  h->own_stream = true;
  h->use_graphs = getenv("VNECT_B200_NO_GRAPH") == nullptr;
  int rc = alloc_prepost(h, ptab);
  if (rc) return rc;
  return vnect_reset_stream(h, -1);
}

int vnect_set_weight(vnect_t* h, const char* tf_name, const float* data, const int64_t* shape, int32_t rank) {
  if (!h || !tf_name || !data || !shape) return fail(h, VNECT_E_INVALID, "null argument");
  if (h->finalized) return fail(h, VNECT_E_INVALID, "weights are frozen after vnect_finalize");
  std::vector<int64_t> want;
  if (!expected_shape(tf_name, &want)) return fail(h, VNECT_E_WEIGHT, "unknown variable '%s'", tf_name);
  if ((int)want.size() != rank) return fail(h, VNECT_E_WEIGHT, "'%s': rank %d, expected %zu", tf_name, rank, want.size());
  size_t n = 1;
  for (int i = 0; i < rank; ++i) {
    if (shape[i] != want[i]) return fail(h, VNECT_E_WEIGHT, "'%s': dim %d is %lld, expected %lld", tf_name, i, (long long)shape[i], (long long)want[i]);
    n *= (size_t)shape[i];
  }
  HostVar& v = h->vars[tf_name];
  v.data.assign(data, data + n);
  v.shape = want;
  return VNECT_OK;
}

int vnect_finalize(vnect_t* h) {
  if (!h) return VNECT_E_INVALID;
  if (h->finalized) return fail(h, VNECT_E_INVALID, "already finalized");
  ON_DEVICE(h);
  // every variable of the graph must be present (the reference restores all 109 from the checkpoint)
  for (const ConvDef& c : conv_defs())
    for (const char* leaf : {"/weights", "/biases"})
      if (!h->vars.count(c.scope + leaf)) return fail(h, VNECT_E_WEIGHT, "missing variable %s%s", c.scope.c_str(), leaf);
  for (const char* k : {"res5c_branch1a/kernel", "res5c_branch2a/kernel", "res5c_branch2c/kernel"})
    if (!h->vars.count(k)) return fail(h, VNECT_E_WEIGHT, "missing variable %s", k);
  for (const char* v : kBnVars)
    if (!h->vars.count(std::string("bn5c_branch2a/") + v)) return fail(h, VNECT_E_WEIGHT, "missing variable bn5c_branch2a/%s", v);

  const int S = h->S, nb = h->cap_fw;
  int rc;
  {  // conv1 + pool1 (vnect_model.py:27-29) fused: rolling raw-strip implicit GEMM + max-pool (stem_roll.cuh)
    std::vector<__half> wk = to_half(pack_stem(h->vars.at("conv1/weights"))), ws(wk.size());
    pack_stem_stacked(wk.data(), ws.data());
    std::vector<__half> wp((size_t)kPairWBytes);  // two ranks x kPairWBytes / 2 halves
    pack_stem_pair(wk.data(), wp.data());
    __half *dws = nullptr, *dwp = nullptr;
    float* db = nullptr;
    if ((rc = upload(h, ws, &dws))) return rc;
    if ((rc = upload(h, wp, &dwp))) return rc;
    if ((rc = upload(h, h->vars.at("conv1/biases").data, &db))) return rc;
    if ((rc = new_act(h, "pool1", S / 4, S / 4, 64))) return rc;
    Step st;
    st.kind = 3; st.name = "conv1+pool1";
    std::string err;
    if (!build_stem_pool(h->x1, S, h->stem_rpp, h->stem_pitch, dws, db, h->acts.at("pool1").p, nb, h->num_sms, &st.stem_pool, &err,
                         dwp, (size_t)nb * 2 * h->stem_rpp * h->stem_pitch + 16384))
      return fail(h, VNECT_E_CUDA, "conv1+pool1: %s", err.c_str());
    h->steps.push_back(st);
  }
  // each block's tail also computes the next block's 1x1 reduce conv (block_tail.cuh) where the plan allows
  if ((rc = add_block(h, "res2a", "pool1", 64, 64, 256, true, "", false, "", "res2b_branch2a", 64))) return rc;
  // res2b's output feeds nothing but the residual add of res2c: res2c's 3x3 reads res2b_branch2a (vnect_model.py:56) and
  // res2c_branch2a is dead.  res2c is evaluated at even pixels only (below), so res2b's 3x3, last 1x1 and add are too.
  if ((rc = add_block(h, "res2b", "res2a", 256, 64, 256, false, "", true))) return rc;
  // res2c: its output only feeds stride-2 1x1 convs -> even pixels only; the stride-2 reduce of res3a is then a plain
  // 1x1 conv on the compact tensor and can ride on res2c's tail
  if ((rc = add_block(h, "res2c", "res2b", 256, 64, 256, false, "", true, "res2b_branch2a", "res3a_branch2a", 128))) return rc;
  if ((rc = add_block(h, "res3a", "res2c", 256, 128, 512, true, "", false, "", "res3b_branch2a", 128))) return rc;
  if ((rc = add_block(h, "res3b", "res3a", 512, 128, 512, false, "", false, "", "res3c_branch2a", 128))) return rc;
  if ((rc = add_block(h, "res3c", "res3b", 512, 128, 512, false, "", false, "", "res3d_branch2a", 128))) return rc;
  if ((rc = add_block(h, "res3d", "res3c", 512, 128, 512, false, "", true, "", "res4a_branch2a", 256))) return rc;
  if ((rc = add_block(h, "res4a", "res3d", 512, 256, 1024, true, "", false, "", "res4b_branch2a", 256))) return rc;
  {
    const char* names[] = {"res4b", "res4c", "res4d", "res4e", "res4f"};
    std::string prev = "res4a";
    for (int i = 0; i < 5; ++i) {
      // res4f feeds res5a_branch2a_new (512 channels: too wide for the second accumulator) -> not chained
      const std::string next = i < 4 ? std::string(names[i + 1]) + "_branch2a" : std::string();
      if ((rc = add_block(h, names[i], prev, 1024, 256, 1024, false, "", false, "", next, next.empty() ? 0 : 256))) return rc;
      prev = names[i];
    }
  }
  if ((rc = add_block(h, "res5a", "res4f", 1024, 512, 1024, true, "_new", false, "", "res5b_branch2a_new", 256))) return rc;
  ConvOpts relu;
  if (!h->acts.count("res5b_branch2a_new") &&
      (rc = add_conv(h, "res5b_branch2a_new", 1, "res5a", "res5b_branch2a_new", 1024, 256, relu))) return rc;
  if ((rc = add_conv(h, "res5b_branch2b_new", 3, "res5b_branch2a_new", "res5b_branch2b_new", 256, 128, relu))) return rc;
  if ((rc = add_conv(h, "res5b_branch2c_new", 1, "res5b_branch2b_new", "res5b_branch2c_new", 128, 256, relu))) return rc;
  {  // res5c head: two transposed convs + BN + ReLU + bone lengths + concat (vnect_model.py:188-209), one kernel
    const HostVar& g = h->vars.at("bn5c_branch2a/gamma");
    const HostVar& be = h->vars.at("bn5c_branch2a/beta");
    const HostVar& mu = h->vars.at("bn5c_branch2a/moving_mean");
    const HostVar& var = h->vars.at("bn5c_branch2a/moving_variance");
    std::vector<float> scale(128), bias(192, 0.f);
    for (int c = 0; c < 128; ++c) {
      scale[c] = g.data[c] / std::sqrt(var.data[c] + 0.001f);  // tc.layers.batch_norm epsilon default
      bias[c] = be.data[c] - mu.data[c] * scale[c];
    }
    __half* dw = nullptr;
    float* db = nullptr;
    rc = upload(h, to_half(pack_deconv(h->vars.at("res5c_branch2a/kernel"), h->vars.at("res5c_branch1a/kernel"), scale)), &dw);
    if (rc) return rc;
    if ((rc = upload(h, bias, &db))) return rc;
    if ((rc = new_act(h, "res5c_branch2a_feat", S / 8, S / 8, 256))) return rc;
    const Act& ai = h->acts.at("res5b_branch2c_new");
    ConvSpec s;
    s.kind = CONV_DECONV4;
    s.NB = nb; s.H = ai.H; s.W = ai.W; s.in = ai.p; s.cin_pad = 256;
    s.w = dw; s.n_pad = 192; s.n_valid = 191; s.block_n = 192; s.bias = db; s.relu_cols = 128;
    s.out = h->acts.at("res5c_branch2a_feat").p; s.ldc = 256; s.epi = EPI_DECONV_HEAD;
    Step st;
    st.kind = 0; st.name = "res5c_deconv_head";
    std::string err;
    if (!build_conv(s, h->num_sms, &st.launch, &err)) return fail(h, VNECT_E_CUDA, "deconv head: %s", err.c_str());
    h->steps.push_back(st);
  }
  if ((rc = add_conv(h, "res5c_branch2b", 3, "res5c_branch2a_feat", "res5c_branch2b", 212, 128, relu))) return rc;
  {  // res5c_branch2c: 1x1 128 -> 84, no bias, linear (vnect_model.py:213); channel-planar fp32 for the post-process
    const HostVar& w = h->vars.at("res5c_branch2c/kernel");
    __half* dw = nullptr;
    rc = upload(h, to_half(pack_conv(w, 1, 128, 84, 128, 96)), &dw);
    if (rc) return rc;
    const Act& ai = h->acts.at("res5c_branch2b");
    ConvSpec s;
    s.kind = CONV_1x1;
    s.NB = nb; s.H = ai.H; s.W = ai.W; s.in = ai.p; s.cin_pad = 128;
    s.w = dw; s.n_pad = 96; s.n_valid = 84; s.block_n = 96; s.bias = nullptr; s.relu_cols = 0;
    s.out = h->maps; s.ldc = 0; s.epi = EPI_PLANAR_F32;
    Step st;
    st.kind = 0; st.name = "res5c_branch2c";
    std::string err;
    if (!build_conv(s, h->num_sms, &st.launch, &err)) return fail(h, VNECT_E_CUDA, "res5c_branch2c: %s", err.c_str());
    h->steps.push_back(st);
  }
  h->conv_steps = 0;
  h->conv_steps = (int)h->steps.size();
  // ping-pong tile order: layer i walks its tiles in the opposite direction of layer i-1, so it starts on the data
  // that is still in the 126 MB L2 (the pyramid kernel writes forwards in ascending order, hence the stem reverses)
  for (size_t i = 0; i < h->steps.size(); ++i) {
    const int rev = i % 2 == 0 ? 1 : 0;
    if (h->steps[i].kind == 0) h->steps[i].launch.p.reverse = rev;
    else h->steps[i].stem_pool.r.reverse = rev;
  }

  h->vars.clear();  // host copies no longer needed
  h->finalized = true;
  CU(h, cudaDeviceSynchronize());
  return VNECT_OK;
}

}  // extern "C"

// run the CNN on the first n forwards of x1 (already filled), on the handle's stream
static int run_forward(vnect_t* h, int n, cudaEvent_t* layer_events = nullptr) {
  int ei = 0;
  for (Step& st : h->steps) {
    if (layer_events) CU(h, cudaEventRecord(layer_events[ei++], h->stream));
    if (st.kind == 0) {
      set_batch(st.launch, n, h->num_sms);
      CU(h, launch_conv(st.launch, h->stream));
    } else {
      stem_pool_set_batch(st.stem_pool, n, h->num_sms);
      CU(h, launch_stem_pool(st.stem_pool, h->stream));
    }
    ++h->launches;
  }
  if (layer_events) CU(h, cudaEventRecord(layer_events[ei++], h->stream));
  return VNECT_OK;
}

constexpr int kFmtBGR = 0;  // packed BGR24; the YUV formats are VNECT_FMT_NV12 / VNECT_FMT_I420

// Where the pixels of each frame of a batch are, in device memory, for any input format.
struct FrameSource {
  int format = kFmtBGR;
  int64_t pitch = 0;         // bytes between BGR rows, or between luma rows
  int64_t frame_stride = 0;  // bytes between frames
  int64_t uv_pitch = 0, u_offset = 0, v_offset = 0;  // YUV: chroma rows, chroma planes relative to a frame's start
  bool table = false;  // mixed sizes: every frame's address, size and layout come from the current lane's d_table
};

static FrameSource table_source(int format) {
  FrameSource s;
  s.format = format;
  s.table = true;
  return s;
}

static FrameSource bgr_source(int64_t pitch, int64_t frame_stride) {
  FrameSource s;
  s.pitch = pitch;
  s.frame_stride = frame_stride;
  return s;
}

static FrameSource yuv_source(const vnect_yuv_layout& l) {
  FrameSource s;
  s.format = l.format;
  s.pitch = l.y_pitch;
  s.frame_stride = l.frame_stride;
  s.uv_pitch = l.uv_pitch;
  s.u_offset = l.u_offset;
  s.v_offset = l.v_offset;
  return s;
}

// cv2's contiguous layout of a [3H/2][W] YUV 4:2:0 frame (what the host paths stage on the device)
static vnect_yuv_layout packed_yuv_layout(int format, int H, int W) {
  vnect_yuv_layout l{};
  l.format = format;
  l.y_pitch = W;
  l.uv_pitch = format == VNECT_FMT_NV12 ? W : W / 2;
  l.u_offset = (int64_t)H * W;
  l.v_offset = format == VNECT_FMT_NV12 ? l.u_offset + 1 : l.u_offset + (int64_t)(H / 2) * (W / 2);
  l.frame_stride = (int64_t)H * W * 3 / 2;
  return l;
}

struct Geometry {
  double scaler;
  int dh, dw, off_x, off_y, mode;
  bool alias;  // BGR frames already are S x S: the pyramid reads them directly
};

// utils.img_scale_squarify geometry (utils.py:82-120).  YUV frames never alias: the squarify stage converts them.
static Geometry squarify_geometry(int S, int H, int W, int format = kFmtBGR) {
  Geometry g;
  g.scaler = (double)S / (double)std::max(H, W);
  g.dw = cv_round_host(W * g.scaler);
  g.dh = cv_round_host(H * g.scaler);
  g.off_x = g.off_y = 0;
  if (g.dh > g.dw) g.off_x = S / 2 - g.dw / 2;
  else g.off_y = S / 2 - g.dh / 2;
  g.mode = (1.0 / g.scaler == 2.0) ? 1 : 0;  // OpenCV turns exact 2x INTER_LINEAR decimation into INTER_AREA
  g.alias = (format == kFmtBGR && H == S && W == S);
  return g;
}

// device frames -> x1 (stem layout) for n_frames * n_scales forwards
static int launch_pyramid(vnect_t* h, const uint8_t* sq, int64_t sq_pitch, int64_t sq_stride, int n_frames, bool full_surround) {
  const int S = h->S;
  PyramidParams py = h->pyr;
  py.n_frames = n_frames; py.sq_pitch = sq_pitch; py.sq_frame_stride = sq_stride;
  py.full = full_surround ? 1 : 0;
  const size_t smem = (size_t)h->pyr_src_rows * S * 4;  // staged source rows, one word per pixel (vnect_create: <= kPyrMaxSmem)
  static unsigned long long done = 0;
  CU(h, ensure_dyn_smem(pyramid_kernel, kPyrMaxSmem, &done));
  CU(h, launch_pdl(pyramid_kernel, dim3((S + kPyrRows - 1) / kPyrRows, n_frames * h->n_scales), dim3(kPyrThreads), smem,
                   h->stream, sq, h->x1, py));
  ++h->launches;
  return VNECT_OK;
}

// The surround of every shrunken scale is a per-slot constant of x1: written here for all slots, once, and again only
// after vnect_forward has put caller-supplied images into the buffer.  Never part of a captured graph.
static int ensure_surround(vnect_t* h) {
  if (h->x1_surround_ok) return VNECT_OK;
  const int S = h->S;
  int rc = launch_pyramid(h, h->d_sq, (int64_t)S * 3, (int64_t)S * S * 3, h->cfg.max_frames, true);
  if (rc) return rc;
  h->x1_surround_ok = true;
  return VNECT_OK;
}

static int run_preprocess(vnect_t* h, const uint8_t* dev_frames, int n_frames, int H, int W, const FrameSource& src,
                          const Geometry& g, bool tracked = false, bool oriented = false) {
  const int S = h->S;
  int rc0 = ensure_surround(h);
  if (rc0) return rc0;
  if (src.table) {  // per-frame geometry from each frame's own size, then squarify through the lane's table
    vnect_handle::Lane* L = h->cur;
    if (oriented)
      frame_geometry_oriented_kernel<<<(n_frames + 63) / 64, 64, 0, h->stream>>>(
          L->d_table, L->d_orient, tracked ? h->d_boxes : nullptr, L->d_stream_ids, n_frames, S, L->d_geoms,
          h->d_boxes_used);
    else
      frame_geometry_kernel<<<(n_frames + 63) / 64, 64, 0, h->stream>>>(L->d_table, tracked ? h->d_boxes : nullptr,
                                                                        L->d_stream_ids, n_frames, S, L->d_geoms,
                                                                        h->d_boxes_used);
    CU(h, cudaGetLastError());
    ++h->launches;
    SquarifyParams sp{};  // nothing size- or address-dependent: one captured graph serves every composition
    sp.geoms = L->d_geoms;
    sp.n_frames = n_frames; sp.S = S;
    sp.frame_stride = sizeof(FrameDesc);
    sp.uv_step = src.format == VNECT_FMT_NV12 ? 2 : 1;
    const int64_t total = (int64_t)n_frames * S * S;
    const uint8_t* table = reinterpret_cast<const uint8_t*>(L->d_table);
    const int grid = grid_for(total, 256, h->num_sms);
    if (oriented && src.format == kFmtBGR)
      squarify_tiled_kernel<FrameTableSrc<Oriented<BgrSrc>>><<<grid, 256, 0, h->stream>>>(table, h->d_sq, sp);
    else if (oriented)
      squarify_tiled_kernel<FrameTableSrc<Oriented<Yuv420Src>>><<<grid, 256, 0, h->stream>>>(table, h->d_sq, sp);
    else if (src.format == kFmtBGR)
      squarify_kernel<FrameTableSrc<BgrSrc>><<<grid, 256, 0, h->stream>>>(table, h->d_sq, sp);
    else
      squarify_kernel<FrameTableSrc<Yuv420Src>><<<grid, 256, 0, h->stream>>>(table, h->d_sq, sp);
    CU(h, cudaGetLastError());
    ++h->launches;
    return launch_pyramid(h, h->d_sq, (int64_t)S * 3, (int64_t)S * S * 3, n_frames, false);
  }
  const uint8_t* sq = dev_frames;
  int64_t sq_pitch = src.pitch, sq_stride = src.frame_stride;
  if (tracked) {
    track_geometry_kernel<<<(n_frames + 63) / 64, 64, 0, h->stream>>>(h->d_boxes, h->cur->d_stream_ids, n_frames, S, H, W,
                                                                      h->d_geoms, h->d_boxes_used);
    CU(h, cudaGetLastError());
    ++h->launches;
  }
  if (!g.alias || tracked) {
    SquarifyParams sp;
    sp.geoms = tracked ? h->d_geoms : nullptr;
    sp.n_frames = n_frames; sp.H = H; sp.W = W; sp.pitch = src.pitch; sp.frame_stride = src.frame_stride; sp.S = S;
    sp.dh = g.dh; sp.dw = g.dw; sp.off_x = g.off_x; sp.off_y = g.off_y; sp.inv_scale = 1.0 / g.scaler; sp.mode = g.mode;
    sp.uv_pitch = src.uv_pitch; sp.u_offset = src.u_offset; sp.v_offset = src.v_offset;
    sp.uv_step = src.format == VNECT_FMT_NV12 ? 2 : 1;
    const int64_t total = (int64_t)n_frames * S * S;
    if (src.format == kFmtBGR)
      squarify_kernel<BgrSrc><<<grid_for(total, 256, h->num_sms), 256, 0, h->stream>>>(dev_frames, h->d_sq, sp);
    else
      squarify_kernel<Yuv420Src><<<grid_for(total, 256, h->num_sms), 256, 0, h->stream>>>(dev_frames, h->d_sq, sp);
    CU(h, cudaGetLastError());
    ++h->launches;
    sq = h->d_sq; sq_pitch = (int64_t)S * 3; sq_stride = (int64_t)S * S * 3;
  }
  if (int rc = launch_pyramid(h, sq, sq_pitch, sq_stride, n_frames, false)) return rc;
  return VNECT_OK;
}

// validates ids / timestamps on the host exactly where the reference would raise, then stages them to the device
// waits until the lane's previous submission has fully completed (its pinned meta and device buffers are reusable)
static int lane_acquire(vnect_t* h, int lane) {
  h->cur = &h->lanes[lane];
  if (h->cur->pending) {
    CU(h, cudaEventSynchronize(h->cur->done));
    h->cur->pending = false;
    if (*reinterpret_cast<volatile unsigned int*>(h->cur->h_nonfinite) != 0) {  // the batch that just completed produced NaN / Inf maps: fail loudly, once
      unsigned int n = 0;  // error path only: the count lives on the device
      cudaStreamSynchronize(h->stream);
      cudaMemcpy(&n, h->d_nonfinite, sizeof n, cudaMemcpyDeviceToHost);
      *h->cur->h_nonfinite = 0;
      cudaMemset(h->d_nonfinite, 0, sizeof(unsigned int));
      return fail(h, VNECT_E_NUMERIC, "non-finite values in the CNN output maps (%u joint blocks): fp16 activations "
                  "overflow at 65504 -- are the weights normalised? (vnect_check_finite names the first layer)", n);
    }
  }
  return VNECT_OK;
}

// The post-process itself raises the lane's host-visible flag (PostParams::nonfinite_flag, a mapped pinned word) when
// it meets NaN / Inf maps, so no device -> host copy of a counter sits in the stream after every batch.
static int snapshot_nonfinite(vnect_t*) { return VNECT_OK; }

// table_frames > 0: the lane's frame table (already written to its pinned block) travels in the same copy.
// oriented: so do the frames' orientation codes, taken from their streams now (a call with oriented frames always
// carries its table); recover: so do the frames' recovery thresholds (a tracked call with a recovering stream always
// carries its table)
static int stage_frame_meta(vnect_t* h, int n_frames, const int32_t* stream_ids, const double* t2d, const double* t3d,
                            cudaStream_t copy_on, int table_frames = 0, bool oriented = false, bool recover = false) {
  if (n_frames < 1 || n_frames > h->cfg.max_frames) return fail(h, VNECT_E_INVALID, "n_frames %d not in [1, %d]", n_frames, h->cfg.max_frames);
  h->seen_stamp.resize(h->cfg.max_streams, 0);
  const unsigned int stamp = ++h->seen_epoch;
  for (int i = 0; i < n_frames; ++i) {
    const int sid = stream_ids ? stream_ids[i] : i;
    if (sid < 0 || sid >= h->cfg.max_streams) return fail(h, VNECT_E_INVALID, "stream id %d not in [0, %d)", sid, h->cfg.max_streams);
    const bool dup = h->seen_stamp[sid] == stamp;
    h->seen_stamp[sid] = stamp;
    if (dup) return fail(h, VNECT_E_INVALID, "stream id %d appears twice in one call (frames of a stream are sequential)", sid);
    if (h->cfg.filters) {
      if (!t2d || !t3d) return fail(h, VNECT_E_INVALID, "timestamps required when filters are on");
      // OneEuroFilter.py:65-66: freq = 1.0 / (timestamp - lasttime) when both are truthy
      if (h->last_t2d[sid] == h->last_t2d[sid] && h->last_t2d[sid] != 0.0 && t2d[i] != 0.0 && t2d[i] == h->last_t2d[sid])
        return fail(h, VNECT_E_ZERO_DT, "float division by zero (stream %d: repeated 2D timestamp %.17g)", sid, t2d[i]);
      if (h->last_t3d[sid] == h->last_t3d[sid] && h->last_t3d[sid] != 0.0 && t3d[i] != 0.0 && t3d[i] == h->last_t3d[sid])
        return fail(h, VNECT_E_ZERO_DT, "float division by zero (stream %d: repeated 3D timestamp %.17g)", sid, t3d[i]);
      // an EARLIER timestamp makes freq negative and every alpha leave (0, 1]: LowPassFilter raises ValueError
      // (OneEuroFilter.py:21-22).  Refused here, before any filter state is touched.
      if (h->last_t2d[sid] == h->last_t2d[sid] && h->last_t2d[sid] != 0.0 && t2d[i] != 0.0 && t2d[i] < h->last_t2d[sid])
        return fail(h, VNECT_E_INVALID, "alpha should be in (0.0, 1.0] (stream %d: 2D timestamp %.17g earlier than the previous %.17g)", sid, t2d[i], h->last_t2d[sid]);
      if (h->last_t3d[sid] == h->last_t3d[sid] && h->last_t3d[sid] != 0.0 && t3d[i] != 0.0 && t3d[i] < h->last_t3d[sid])
        return fail(h, VNECT_E_INVALID, "alpha should be in (0.0, 1.0] (stream %d: 3D timestamp %.17g earlier than the previous %.17g)", sid, t3d[i], h->last_t3d[sid]);
    }
  }
  for (int i = 0; i < n_frames; ++i) {
    const int sid = stream_ids ? stream_ids[i] : i;
    h->cur->h_stream_ids[i] = sid;
    h->cur->h_t2d[i] = t2d ? t2d[i] : 0.0;
    h->cur->h_t3d[i] = t3d ? t3d[i] : 0.0;
    if (oriented) h->cur->h_orient[i] = h->orient[sid];
    if (recover) h->cur->h_recover[i] = h->recover[sid];
    if (h->cfg.filters) {
      h->last_t2d[sid] = t2d[i];
      h->last_t3d[sid] = t3d[i];
    }
  }
  const size_t bytes = recover ? h->cur->recover_off + (size_t)n_frames * sizeof(double)
                       : oriented ? h->cur->orient_off + (size_t)n_frames * sizeof(int)
                       : table_frames > 0 ? h->cur->table_off + (size_t)table_frames * sizeof(FrameDesc)
                                          : h->cur->meta_bytes;
  CU(h, cudaMemcpyAsync(h->cur->d_stream_ids, h->cur->h_meta, bytes, cudaMemcpyHostToDevice, copy_on));
  return VNECT_OK;
}

// stage_frame_meta for a sequence call: a stream id may repeat, its frames being consecutive in time in call order.
// Every frame's timestamps are checked against its stream's previous reading -- the one before the call, then the
// call's own earlier frames -- with stage_frame_meta's rules and messages, and only once the whole call has passed is
// anything recorded.  The segment table of sequence_filter_kernel goes to the lane's pinned block after the frame
// table, and ids, timestamps, table and segments travel in one copy.
static int stage_sequence_meta(vnect_t* h, int n_frames, const int32_t* stream_ids, const double* t2d,
                               const double* t3d, cudaStream_t copy_on, bool oriented = false) {
  if (n_frames < 1 || n_frames > h->cfg.max_frames) return fail(h, VNECT_E_INVALID, "n_frames %d not in [1, %d]", n_frames, h->cfg.max_frames);
  if (!stream_ids) return fail(h, VNECT_E_INVALID, "a sequence call needs stream ids");
  if (h->cfg.filters && (!t2d || !t3d)) return fail(h, VNECT_E_INVALID, "timestamps required when filters are on");
  const int ms = h->cfg.max_streams;
  h->seen_stamp.resize(ms, 0);
  h->seq_slot.resize(ms, 0);
  h->seq_t2d.resize(ms, NAN);
  h->seq_t3d.resize(ms, NAN);
  const unsigned int stamp = ++h->seen_epoch;
  vnect_handle::Lane* L = h->cur;
  int* starts = L->h_seg + 1;
  int n_seg = 0;
  for (int i = 0; i < n_frames; ++i) {
    const int sid = stream_ids[i];
    if (sid < 0 || sid >= ms) return fail(h, VNECT_E_INVALID, "stream id %d not in [0, %d)", sid, ms);
    if (h->seen_stamp[sid] != stamp) {
      h->seen_stamp[sid] = stamp;
      h->seq_slot[sid] = n_seg;
      starts[n_seg++] = 0;
      h->seq_t2d[sid] = h->last_t2d[sid];
      h->seq_t3d[sid] = h->last_t3d[sid];
    }
    ++starts[h->seq_slot[sid]];
    if (h->cfg.filters) {
      const double l2 = h->seq_t2d[sid], l3 = h->seq_t3d[sid];
      if (l2 == l2 && l2 != 0.0 && t2d[i] != 0.0 && t2d[i] == l2)
        return fail(h, VNECT_E_ZERO_DT, "float division by zero (stream %d: repeated 2D timestamp %.17g)", sid, t2d[i]);
      if (l3 == l3 && l3 != 0.0 && t3d[i] != 0.0 && t3d[i] == l3)
        return fail(h, VNECT_E_ZERO_DT, "float division by zero (stream %d: repeated 3D timestamp %.17g)", sid, t3d[i]);
      if (l2 == l2 && l2 != 0.0 && t2d[i] != 0.0 && t2d[i] < l2)
        return fail(h, VNECT_E_INVALID, "alpha should be in (0.0, 1.0] (stream %d: 2D timestamp %.17g earlier than the previous %.17g)", sid, t2d[i], l2);
      if (l3 == l3 && l3 != 0.0 && t3d[i] != 0.0 && t3d[i] < l3)
        return fail(h, VNECT_E_INVALID, "alpha should be in (0.0, 1.0] (stream %d: 3D timestamp %.17g earlier than the previous %.17g)", sid, t3d[i], l3);
      h->seq_t2d[sid] = t2d[i];
      h->seq_t3d[sid] = t3d[i];
    }
  }
  // counts -> starts (exclusive prefix sum), then the frame list, each stream's frames in call order
  L->h_seg[0] = n_seg;
  for (int b = 0, acc = 0; b <= n_seg; ++b) {
    const int c = b < n_seg ? starts[b] : 0;
    starts[b] = acc;
    acc += c;
  }
  int* list = L->h_seg + 2 + n_seg;
  for (int i = 0; i < n_frames; ++i) {
    const int sid = stream_ids[i];
    list[starts[h->seq_slot[sid]]++] = i;
  }
  for (int b = n_seg; b > 0; --b) starts[b] = starts[b - 1];  // the fill advanced each start to the next one's
  starts[0] = 0;
  for (int i = 0; i < n_frames; ++i) {
    const int sid = stream_ids[i];
    L->h_stream_ids[i] = sid;
    L->h_t2d[i] = t2d ? t2d[i] : 0.0;
    L->h_t3d[i] = t3d ? t3d[i] : 0.0;
    if (oriented) L->h_orient[i] = h->orient[sid];
    if (h->cfg.filters) {
      h->last_t2d[sid] = h->seq_t2d[sid];
      h->last_t3d[sid] = h->seq_t3d[sid];
    }
  }
  const size_t bytes = oriented ? L->orient_off + (size_t)n_frames * sizeof(int)
                                : L->seg_off + (size_t)(2 + n_seg + n_frames) * sizeof(int);
  CU(h, cudaMemcpyAsync(L->d_stream_ids, L->h_meta, bytes, cudaMemcpyHostToDevice, copy_on));
  return VNECT_OK;
}

// The SCORES instantiations of postprocess_kernel: `launch` as run_postprocess defines it.
template <bool RAW_ONLY, class Launch>
static cudaError_t launch_post_scores(Launch& launch, int n_scales, bool mask1) {
  static unsigned long long done[2][kMaxScales] = {{0, 0, 0, 0}, {0, 0, 0, 0}};
  switch (n_scales) {
    case 1: return mask1 ? launch(postprocess_kernel<1, 1, RAW_ONLY, true>, &done[0][0])
                         : launch(postprocess_kernel<1, -1, RAW_ONLY, true>, &done[1][0]);
    case 2: return mask1 ? launch(postprocess_kernel<2, 1, RAW_ONLY, true>, &done[0][1])
                         : launch(postprocess_kernel<2, -1, RAW_ONLY, true>, &done[1][1]);
    case 3: return mask1 ? launch(postprocess_kernel<3, 1, RAW_ONLY, true>, &done[0][2])
                         : launch(postprocess_kernel<3, -1, RAW_ONLY, true>, &done[1][2]);
    default: return mask1 ? launch(postprocess_kernel<4, 1, RAW_ONLY, true>, &done[0][3])
                          : launch(postprocess_kernel<4, -1, RAW_ONLY, true>, &done[1][3]);
  }
}

// geoms: per-frame geometry (tracked streams, mixed sizes), which overrides scaler and the offsets.
// seq_seg: a sequence call's device segment table (stage_sequence_meta): the argmax-only instantiation, then
// sequence_filter_kernel walks each stream's frames in order.
// scores: the SCORES instantiation, which also writes every joint's score to d_scores.
static int run_postprocess(vnect_t* h, int n_frames, double scaler, int off_x, int off_y, double* dev_out2d,
                           float* dev_out3d, const FrameGeom* geoms = nullptr, bool guard = true,
                           const int* seq_seg = nullptr, bool scores = false) {
  PostParams p;
  p.geoms = geoms;
  p.n_frames = n_frames; p.n_scales = h->n_scales; p.hs = h->hs; p.S = h->S;
  p.maps = h->maps; p.tables = h->d_tables;
  p.stream_ids = h->cur->d_stream_ids; p.t2d = h->cur->d_t2d; p.t3d = h->cur->d_t3d;
  p.st2d = h->d_st2d; p.st3d = h->d_st3d;
  p.cfg2d = {30.0, 1.7, 0.3, 0.4};  // estimator.py:34-39
  p.cfg3d = {30.0, 0.8, 0.4, 0.4};  // estimator.py:40-45
  p.filters_on = h->cfg.filters;
  p.scaler = scaler; p.off_x = off_x; p.off_y = off_y;
  p.j2_box = h->d_j2_box; p.j3_raw = h->d_j3_raw; p.raw_argmax = h->d_raw_argmax;
  p.frame_counter = h->d_counter;
  p.prep3 = h->d_prep3;
  p.out2d = dev_out2d; p.out3d = dev_out3d;
  p.packed = h->d_packed;
  p.nonfinite = guard ? h->d_nonfinite : nullptr;  // caller-supplied maps (vnect_postprocess) are taken as they are
  p.nonfinite_flag = nullptr;
  if (guard) CU(h, cudaHostGetDevicePointer(reinterpret_cast<void**>(&p.nonfinite_flag), h->cur->h_nonfinite, 0));
  // Threads per (frame, joint) block = the cells of `rows` heat-map rows.  A full batch is bound by instruction issue
  // summed over all blocks (two rows: every lane busy at hs = 46); a few frames leave most SMs empty, so wider blocks
  // shorten each block's own chain instead.
  const int rows = n_frames >= 48 ? 2 : n_frames >= 12 ? 4 : 8;
  const int threads = post_threads(h->hs, rows);
  const int rpp = threads / h->hs;
  post_smem_plan(p, h->h_tables.data(), (h->hs / 2 / rpp) * rpp);
  p.trace = h->d_post_trace;
  p.scores_off = h->cfg.max_frames * kJoints * 2;
  const size_t smem = (size_t)p.smem_floats * sizeof(float);
  static unsigned long long done[kMaxScales] = {0, 0, 0, 0};
  auto launch = [&](auto kern, unsigned long long* mask) -> cudaError_t {
    if (cudaError_t e = ensure_dyn_smem(kern, 96 * 1024, mask); e != cudaSuccess) return e;
    return launch_pdl(kern, dim3(n_frames * kJoints), dim3(threads), smem, h->stream, p);
  };
  // the usual pyramid (scale 1.0 first, smaller ones after) gets its identity mask as a compile-time constant
  static unsigned long long done1[kMaxScales] = {0, 0, 0, 0};
  if (seq_seg != nullptr) {
    static unsigned long long done_raw[2][kMaxScales] = {{0, 0, 0, 0}, {0, 0, 0, 0}};
    if (scores) {
      CU(h, launch_post_scores<true>(launch, h->n_scales, p.identity_mask == 1));
    } else if (p.identity_mask == 1) {
      switch (h->n_scales) {
        case 1: CU(h, launch(postprocess_kernel<1, 1, true>, &done_raw[0][0])); break;
        case 2: CU(h, launch(postprocess_kernel<2, 1, true>, &done_raw[0][1])); break;
        case 3: CU(h, launch(postprocess_kernel<3, 1, true>, &done_raw[0][2])); break;
        default: CU(h, launch(postprocess_kernel<4, 1, true>, &done_raw[0][3])); break;
      }
    } else {
      switch (h->n_scales) {
        case 1: CU(h, launch(postprocess_kernel<1, -1, true>, &done_raw[1][0])); break;
        case 2: CU(h, launch(postprocess_kernel<2, -1, true>, &done_raw[1][1])); break;
        case 3: CU(h, launch(postprocess_kernel<3, -1, true>, &done_raw[1][2])); break;
        default: CU(h, launch(postprocess_kernel<4, -1, true>, &done_raw[1][3])); break;
      }
    }
    ++h->launches;
    // one block per distinct stream; n_frames blocks whatever the composition, so one graph serves them all
    switch (h->n_scales) {
      case 1: sequence_filter_kernel<1><<<n_frames, kSeqThreads, 0, h->stream>>>(p, seq_seg); break;
      case 2: sequence_filter_kernel<2><<<n_frames, kSeqThreads, 0, h->stream>>>(p, seq_seg); break;
      case 3: sequence_filter_kernel<3><<<n_frames, kSeqThreads, 0, h->stream>>>(p, seq_seg); break;
      default: sequence_filter_kernel<4><<<n_frames, kSeqThreads, 0, h->stream>>>(p, seq_seg); break;
    }
    CU(h, cudaGetLastError());
    ++h->launches;
    return VNECT_OK;
  }
  if (scores) {
    CU(h, launch_post_scores<false>(launch, h->n_scales, p.identity_mask == 1));
  } else if (p.identity_mask == 1) {
    switch (h->n_scales) {
      case 1: CU(h, launch(postprocess_kernel<1, 1>, &done1[0])); break;
      case 2: CU(h, launch(postprocess_kernel<2, 1>, &done1[1])); break;
      case 3: CU(h, launch(postprocess_kernel<3, 1>, &done1[2])); break;
      default: CU(h, launch(postprocess_kernel<4, 1>, &done1[3])); break;
    }
  } else {
    switch (h->n_scales) {
      case 1: CU(h, launch(postprocess_kernel<1, -1>, &done[0])); break;
      case 2: CU(h, launch(postprocess_kernel<2, -1>, &done[1])); break;
      case 3: CU(h, launch(postprocess_kernel<3, -1>, &done[2])); break;
      default: CU(h, launch(postprocess_kernel<4, -1>, &done[3])); break;
    }
  }
  ++h->launches;
  return VNECT_OK;
}

extern "C" {

int vnect_forward(vnect_t* h, const float* nhwc, int32_t n, float* hm, float* xm, float* ym, float* zm) {
  if (!h || !h->finalized) return fail(h, VNECT_E_INVALID, "handle not finalized");
  ON_DEVICE(h);
  if (!nhwc || !hm || !xm || !ym || !zm) return fail(h, VNECT_E_INVALID, "null buffer");
  if (n < 1 || n > h->cap_fw) return fail(h, VNECT_E_INVALID, "n %d not in [1, %d]", n, h->cap_fw);
  const int S = h->S, hs = h->hs;
  const size_t in_elems = (size_t)n * S * S * 3;
  CU(h, cudaMemcpyAsync(h->d_f32_in, nhwc, in_elems * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  h->x1_surround_ok = false;  // caller-supplied images replace whole slots of x1
  f32_to_stem_kernel<<<grid_for((int64_t)n * S * S, 256, h->num_sms), 256, 0, h->stream>>>(h->d_f32_in, h->x1, n, S, h->stem_rpp, h->stem_pitch);
  CU(h, cudaGetLastError());
  ++h->launches;
  int rc = run_forward(h, n);
  if (rc) return rc;
  std::vector<float> planar((size_t)n * 84 * hs * hs);
  CU(h, cudaMemcpyAsync(planar.data(), h->maps, planar.size() * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaStreamSynchronize(h->stream));
  float* outs[4] = {hm, xm, ym, zm};
  const size_t plane = (size_t)hs * hs;
  for (int i = 0; i < n; ++i)
    for (int m = 0; m < 4; ++m)
      for (int j = 0; j < kJoints; ++j) {
        const float* src = planar.data() + ((size_t)i * 84 + m * kJoints + j) * plane;
        float* dst = outs[m] + (size_t)i * plane * kJoints + j;
        for (size_t px = 0; px < plane; ++px) dst[px * kJoints] = src[px];
      }
  return VNECT_OK;
}

}  // extern "C"

// Runs direct() -- the kernel sequence of one batch -- as a CUDA graph cached under `key`: the first use of a key runs
// directly (warm-up), the second captures, later ones replay.
template <class F>
static int run_graphed(vnect_t* h, const vnect_handle::GraphKey& key, F direct) {
  auto it = h->graphs.find(key);
  if (it == h->graphs.end()) {
    if (h->graphs.size() >= vnect_handle::kMaxGraphs) {  // evict the least recently used entry
      auto victim = h->graphs.begin();
      for (auto g = h->graphs.begin(); g != h->graphs.end(); ++g)
        if (g->second.last_use < victim->second.last_use) victim = g;
      if (victim->second.exec) cudaGraphExecDestroy(victim->second.exec);
      h->graphs.erase(victim);
    }
    h->graphs[key].last_use = ++h->graph_clock;
    return direct();  // warm-up run: sets function attributes, exercises every launch configuration
  }
  vnect_handle::GraphEntry& e = it->second;
  e.last_use = ++h->graph_clock;
  if (e.unusable) return direct();
  if (!e.exec) {
    const long long before = h->launches;
    if (cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
      cudaGetLastError();
      e.unusable = true;  // e.g. the legacy default stream cannot be captured
      return direct();
    }
    const int rc = direct();
    cudaGraph_t graph = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(h->stream, &graph);
    e.launches = h->launches - before;
    h->launches = before;
    if (rc != VNECT_OK || ce != cudaSuccess || graph == nullptr) {
      if (graph) cudaGraphDestroy(graph);
      cudaGetLastError();
      e.unusable = true;
      return rc != VNECT_OK ? rc : direct();
    }
    const cudaError_t ie = cudaGraphInstantiate(&e.exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ie != cudaSuccess) {
      cudaGetLastError();
      e.exec = nullptr;
      e.unusable = true;
      return direct();
    }
  }
  CU(h, cudaGraphLaunch(e.exec, h->stream));
  h->launches += e.launches;
  return VNECT_OK;
}

extern "C" {

// pre-process -> CNN -> post-process for one batch, as a replayed CUDA graph when possible
// oriented (table calls only): the lane carries its frames' orientation codes
// scores: the post-process writes every joint's score to d_scores (the caller copies them out)
// recover (tracked table calls only): the lane carries its frames' recovery thresholds, and the box update checks
// each frame's mean score against them (it implies scores)
static int run_pipeline(vnect_t* h, int lane, const uint8_t* dev_frames, int n_frames, int H, int W,
                        const FrameSource& src, double* out2d, float* out3d, bool tracked = false,
                        bool sequence = false, bool oriented = false, bool scores = false, bool recover = false) {
  scores = scores || recover;
  // the kernel choices the key does not otherwise carry: the SCORES post-process and the recovering box update
  const int variant = (scores ? 16 : 0) + (recover ? 32 : 0);
  if (src.table) {  // sizes, addresses and geometry live in the lane's device tables, not in kernel parameters
    if (int rc = ensure_surround(h)) return rc;
    auto direct = [&]() -> int {
      int rc;
      if ((rc = run_preprocess(h, nullptr, n_frames, 0, 0, src, Geometry{}, tracked, oriented))) return rc;
      if ((rc = run_forward(h, n_frames * h->n_scales))) return rc;
      if ((rc = run_postprocess(h, n_frames, 1.0, 0, 0, out2d, out3d, h->cur->d_geoms, true,
                                sequence ? h->cur->d_seg : nullptr, scores)))
        return rc;
      if (tracked) {
        if (recover)
          track_update_frames_recover_kernel<<<n_frames, 32, 0, h->stream>>>(
              out2d, h->cur->d_stream_ids, h->cur->d_table, oriented ? h->cur->d_orient : nullptr, h->d_scores,
              h->cur->d_recover, h->d_boxes);
        else if (oriented)
          track_update_frames_oriented_kernel<<<n_frames, 32, 0, h->stream>>>(out2d, h->cur->d_stream_ids, h->cur->d_table,
                                                                              h->cur->d_orient, h->d_boxes);
        else
          track_update_frames_kernel<<<n_frames, 32, 0, h->stream>>>(out2d, h->cur->d_stream_ids, h->cur->d_table, h->d_boxes);
        CU(h, cudaGetLastError());
        ++h->launches;
      }
      return VNECT_OK;
    };
    if (!h->use_graphs) return direct();
    // sequence calls (8 + lane) read their segment table from the lane's device block as well; so do calls with
    // oriented frames their codes (the third field), so every composition of orientations replays one graph
    const vnect_handle::GraphKey key(variant + (sequence ? 8 + lane : 4 + lane + (tracked ? 2 : 0)), n_frames,
                                     oriented ? 1 : 0, 0, 0, 0, nullptr, out2d, out3d, src.format, 0, 0, 0);
    return run_graphed(h, key, direct);
  }
  const Geometry g = squarify_geometry(h->S, H, W, src.format);
  if (int rc = ensure_surround(h)) return rc;
  auto direct = [&]() -> int {
    int rc;
    if ((rc = run_preprocess(h, dev_frames, n_frames, H, W, src, g, tracked))) return rc;
    if ((rc = run_forward(h, n_frames * h->n_scales))) return rc;
    if ((rc = run_postprocess(h, n_frames, g.scaler, g.off_x, g.off_y, out2d, out3d, tracked ? h->d_geoms : nullptr, true,
                              nullptr, scores)))
      return rc;
    if (tracked) {
      track_update_kernel<<<n_frames, 32, 0, h->stream>>>(out2d, h->cur->d_stream_ids, n_frames, H, W, h->d_boxes);
      CU(h, cudaGetLastError());
      ++h->launches;
    }
    return VNECT_OK;
  };
  if (!h->use_graphs) return direct();
  // the format and the chroma layout are baked into the squarify launch as much as the pointers are
  const vnect_handle::GraphKey key(variant + lane + (tracked ? 2 : 0), n_frames, H, W, (long long)src.pitch,
                                   (long long)src.frame_stride, dev_frames, out2d, out3d, src.format,
                                   (long long)src.uv_pitch, (long long)src.u_offset, (long long)src.v_offset);
  return run_graphed(h, key, direct);
}

// Checks a YUV 4:2:0 layout of H x W frames (include/vnect_b200.h) before anything is launched or staged.
static int check_yuv_layout(vnect_t* h, const vnect_yuv_layout* l, int H, int W) {
  if (!l) return fail(h, VNECT_E_INVALID, "null layout");
  if ((l->format != VNECT_FMT_NV12 && l->format != VNECT_FMT_I420) || l->reserved != 0)
    return fail(h, VNECT_E_INVALID, "unknown YUV format %d (reserved %d)", l->format, l->reserved);
  if (H < 2 || W < 2 || (H & 1) || (W & 1))
    return fail(h, VNECT_E_INVALID, "YUV 4:2:0 frame %dx%d: H and W must be even and at least 2", H, W);
  const bool nv12 = l->format == VNECT_FMT_NV12;
  if (l->y_pitch < W || l->uv_pitch < (nv12 ? W : W / 2))
    return fail(h, VNECT_E_INVALID, "pitch smaller than a row (y_pitch %lld, uv_pitch %lld, W %d)", (long long)l->y_pitch,
                (long long)l->uv_pitch, W);
  if (l->u_offset < 0 || l->v_offset < 0) return fail(h, VNECT_E_INVALID, "negative chroma offset");
  const int64_t luma_end = (int64_t)(H - 1) * l->y_pitch + W;
  if (l->u_offset < luma_end || l->v_offset < luma_end)
    return fail(h, VNECT_E_INVALID, "chroma plane overlaps the luma plane (offsets %lld / %lld, luma ends at %lld)",
                (long long)l->u_offset, (long long)l->v_offset, (long long)luma_end);
  if (nv12 && l->v_offset != l->u_offset + 1) return fail(h, VNECT_E_INVALID, "NV12 needs v_offset == u_offset + 1");
  return VNECT_OK;
}

static int check_host_frame_size(vnect_t* h, int H, int W) {
  if (H < 2 || W < 2 || H > h->cfg.max_input_h || W > h->cfg.max_input_w)
    return fail(h, VNECT_E_INVALID, "frame %dx%d outside [2, max_input %dx%d]", H, W, h->cfg.max_input_h, h->cfg.max_input_w);
  return VNECT_OK;
}

// one host frame described by `src` -> dst in the layout stage_frames packs it in (BGR: 3W-byte rows, YUV: cv2's
// contiguous [3H/2][W] layout), on the copy stream
static int stage_frame(vnect_t* h, uint8_t* dst, const uint8_t* f, int H, int W, const FrameSource& src) {
  if (src.format == kFmtBGR) {
    CU(h, cudaMemcpy2DAsync(dst, (size_t)W * 3, f, src.pitch, (size_t)W * 3, H, cudaMemcpyHostToDevice, h->copy_stream));
    return VNECT_OK;
  }
  // per plane: luma, then the interleaved U/V plane (NV12) or the U and the V plane (I420)
  const vnect_yuv_layout l = packed_yuv_layout(src.format, H, W);
  const int64_t uv_row = src.format == VNECT_FMT_NV12 ? W : W / 2;
  CU(h, cudaMemcpy2DAsync(dst, l.y_pitch, f, src.pitch, W, H, cudaMemcpyHostToDevice, h->copy_stream));
  CU(h, cudaMemcpy2DAsync(dst + l.u_offset, l.uv_pitch, f + src.u_offset, src.uv_pitch, uv_row, H / 2, cudaMemcpyHostToDevice, h->copy_stream));
  if (src.format == VNECT_FMT_I420)
    CU(h, cudaMemcpy2DAsync(dst + l.v_offset, l.uv_pitch, f + src.v_offset, src.uv_pitch, uv_row, H / 2, cudaMemcpyHostToDevice, h->copy_stream));
  return VNECT_OK;
}

// host frames described by `src` -> the current lane's d_frames, tightly packed (BGR: 3 bytes per pixel, YUV: cv2's
// contiguous layout, 1.5), on the copy stream; `packed` describes them there
// how stage_frames packs H x W frames of `format` on the device
static FrameSource packed_source(int format, int H, int W) {
  return format == kFmtBGR ? bgr_source((int64_t)W * 3, (int64_t)W * 3 * H) : yuv_source(packed_yuv_layout(format, H, W));
}

static int stage_frames(vnect_t* h, const uint8_t* frames, int n_frames, int H, int W, const FrameSource& src,
                        FrameSource* packed) {
  uint8_t* d = h->cur->d_frames;
  *packed = packed_source(src.format, H, W);
  if (src.format == kFmtBGR) {
    if (src.pitch == packed->pitch && src.frame_stride == packed->frame_stride) {
      CU(h, cudaMemcpyAsync(d, frames, (size_t)packed->frame_stride * n_frames, cudaMemcpyHostToDevice, h->copy_stream));
      return VNECT_OK;
    }
  } else {
    const vnect_yuv_layout l = packed_yuv_layout(src.format, H, W);
    if (src.pitch == l.y_pitch && src.uv_pitch == l.uv_pitch && src.u_offset == l.u_offset && src.v_offset == l.v_offset &&
        (n_frames == 1 || src.frame_stride == l.frame_stride)) {
      CU(h, cudaMemcpyAsync(d, frames, (size_t)l.frame_stride * n_frames, cudaMemcpyHostToDevice, h->copy_stream));
      return VNECT_OK;
    }
  }
  for (int i = 0; i < n_frames; ++i)
    if (int rc = stage_frame(h, d + (size_t)i * packed->frame_stride, frames + (size_t)i * src.frame_stride, H, W, src))
      return rc;
  return VNECT_OK;
}

// Whether a call's frames need the oriented path: some frame's stream has a non-identity orientation.  Ids that
// stage_frame_meta refuses are skipped here, and so is a frame count it refuses.
static bool any_oriented(vnect_t* h, int n_frames, const int32_t* stream_ids) {
  if (n_frames < 1 || n_frames > h->cfg.max_frames) return false;
  for (int i = 0; i < n_frames; ++i) {
    const int sid = stream_ids ? stream_ids[i] : i;
    if (sid >= 0 && sid < h->cfg.max_streams && h->orient[sid] != VNECT_ORIENT_IDENTITY) return true;
  }
  return false;
}

// Whether a tracked call recovers lost people: some frame's stream has a recovery threshold (vnect_set_track_recovery).
// Ids that stage_frame_meta refuses are skipped here, and so is a frame count it refuses.
static bool any_recovering(vnect_t* h, int n_frames, const int32_t* stream_ids) {
  if (n_frames < 1 || n_frames > h->cfg.max_frames) return false;
  for (int i = 0; i < n_frames; ++i) {
    const int sid = stream_ids ? stream_ids[i] : i;
    if (sid >= 0 && sid < h->cfg.max_streams && h->recover[sid] > 0.0) return true;
  }
  return false;
}

// The pending vnect_request_scores buffer, consumed by the result-producing call that takes it, accepted or refused.
static double* take_scores(vnect_t* h) {
  if (!h) return nullptr;
  double* s = h->score_req;
  h->score_req = nullptr;
  return s;
}

// The scores of the call's n_frames frames -> the caller's buffer, on the handle's stream after the call's kernels
// (outside any graph, so the pointer is not part of a graph key)
static int copy_scores(vnect_t* h, double* scores, int n_frames, cudaMemcpyKind kind) {
  if (scores) CU(h, cudaMemcpyAsync(scores, h->d_scores, (size_t)n_frames * kJoints * sizeof(double), kind, h->stream));
  return VNECT_OK;
}

// The current lane's frame table for n_frames uniform frames at `frames` (device), laid out as `src` describes:
// a uniform call with oriented frames runs the table pipeline on it.
static void uniform_table(vnect_t* h, const uint8_t* frames, int n_frames, int H, int W, const FrameSource& src) {
  for (int i = 0; i < n_frames; ++i) {
    FrameDesc& t = h->cur->h_table[i];
    t.data = frames + (size_t)i * src.frame_stride;
    t.height = H;
    t.width = W;
    t.pitch = src.pitch;
    t.uv_pitch = src.uv_pitch;
    t.u_offset = src.u_offset;
    t.v_offset = src.v_offset;
  }
}

// vnect_estimate_device / vnect_estimate_device_yuv once the frame description is validated
static int estimate_device(vnect_t* h, const uint8_t* dev_frames, int32_t n_frames, int32_t H, int32_t W,
                           const FrameSource& src, const int32_t* stream_ids, const double* t2d, const double* t3d,
                           double* dev_joints2d, float* dev_joints3d, double* dev_scores) {
  // alternate lanes for the per-call meta so the host can run one call ahead of the GPU
  int rc = lane_acquire(h, (int)(h->device_calls++ & 1));
  if (rc) return rc;
  const bool oriented = any_oriented(h, n_frames, stream_ids);
  if (oriented) uniform_table(h, dev_frames, n_frames, H, W, src);
  // the per-call meta travels on the copy stream, under the previous call's kernels
  if ((rc = stage_frame_meta(h, n_frames, stream_ids, t2d, t3d, h->copy_stream, 0, oriented))) return rc;
  CU(h, cudaEventRecord(h->cur->copy_done, h->copy_stream));
  CU(h, cudaStreamWaitEvent(h->stream, h->cur->copy_done, 0));
  const int lane = (int)(h->cur - h->lanes);
  if ((rc = run_pipeline(h, lane, dev_frames, n_frames, H, W, oriented ? table_source(src.format) : src, dev_joints2d,
                         dev_joints3d, false, false, oriented, dev_scores != nullptr)))
    return rc;
  if ((rc = copy_scores(h, dev_scores, n_frames, cudaMemcpyDeviceToDevice))) return rc;
  if ((rc = snapshot_nonfinite(h))) return rc;
  CU(h, cudaEventRecord(h->cur->done, h->stream));
  h->cur->pending = true;
  return VNECT_OK;
}

// vnect_submit / vnect_submit_yuv once the arguments are validated
static int submit(vnect_t* h, int32_t lane, const uint8_t* frames, int32_t n_frames, int32_t H, int32_t W,
                  const FrameSource& src, const int32_t* stream_ids, const double* t2d, const double* t3d,
                  double* joints2d, float* joints3d, double* scores) {
  int rc = lane_acquire(h, lane);
  if (rc) return rc;
  const bool oriented = any_oriented(h, n_frames, stream_ids);
  if (oriented) uniform_table(h, h->cur->d_frames, n_frames, H, W, packed_source(src.format, H, W));
  // host -> device on the copy stream (tightly packed on the device), overlapping the previous lane's kernels
  if ((rc = stage_frame_meta(h, n_frames, stream_ids, t2d, t3d, h->copy_stream, 0, oriented))) return rc;
  FrameSource packed;
  if ((rc = stage_frames(h, frames, n_frames, H, W, src, &packed))) return rc;
  CU(h, cudaEventRecord(h->cur->copy_done, h->copy_stream));
  CU(h, cudaStreamWaitEvent(h->stream, h->cur->copy_done, 0));
  if ((rc = run_pipeline(h, lane, h->cur->d_frames, n_frames, H, W, oriented ? table_source(src.format) : packed,
                         h->cur->d_out2d, h->cur->d_out3d, false, false, oriented, scores != nullptr)))
    return rc;
  CU(h, cudaMemcpyAsync(joints2d, h->cur->d_out2d, (size_t)n_frames * kJoints * 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaMemcpyAsync(joints3d, h->cur->d_out3d, (size_t)n_frames * kJoints * 3 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  if ((rc = copy_scores(h, scores, n_frames, cudaMemcpyDeviceToHost))) return rc;
  if ((rc = snapshot_nonfinite(h))) return rc;
  CU(h, cudaEventRecord(h->cur->done, h->stream));
  h->cur->pending = true;
  return VNECT_OK;
}

// vnect_track / vnect_track_yuv once the arguments are validated
static int track(vnect_t* h, const uint8_t* frames, int32_t n_frames, int32_t FH, int32_t FW, const FrameSource& src,
                 const int32_t* stream_ids, const double* t2d, const double* t3d, double* joints2d, float* joints3d,
                 int32_t* boxes_used, double* scores) {
  int rc = lane_acquire(h, 0);
  if (rc) return rc;
  // oriented frames or a recovering stream: the table pipeline, on a table of the staged frames
  const bool oriented = any_oriented(h, n_frames, stream_ids), recover = any_recovering(h, n_frames, stream_ids);
  if (oriented || recover) uniform_table(h, h->cur->d_frames, n_frames, FH, FW, packed_source(src.format, FH, FW));
  if ((rc = stage_frame_meta(h, n_frames, stream_ids, t2d, t3d, h->copy_stream, 0, oriented, recover))) return rc;
  FrameSource packed;
  if ((rc = stage_frames(h, frames, n_frames, FH, FW, src, &packed))) return rc;
  CU(h, cudaEventRecord(h->cur->copy_done, h->copy_stream));
  CU(h, cudaStreamWaitEvent(h->stream, h->cur->copy_done, 0));
  if ((rc = run_pipeline(h, 0, h->cur->d_frames, n_frames, FH, FW,
                         oriented || recover ? table_source(src.format) : packed, h->cur->d_out2d, h->cur->d_out3d,
                         true, false, oriented, scores != nullptr, recover)))
    return rc;
  CU(h, cudaMemcpyAsync(joints2d, h->cur->d_out2d, (size_t)n_frames * kJoints * 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaMemcpyAsync(joints3d, h->cur->d_out3d, (size_t)n_frames * kJoints * 3 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  if (boxes_used)
    CU(h, cudaMemcpyAsync(boxes_used, h->d_boxes_used, (size_t)n_frames * 4 * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  if ((rc = copy_scores(h, scores, n_frames, cudaMemcpyDeviceToHost))) return rc;
  if ((rc = snapshot_nonfinite(h))) return rc;
  CU(h, cudaEventRecord(h->cur->done, h->stream));
  h->cur->pending = true;
  return lane_acquire(h, 0);  // synchronises and reports non-finite maps
}

// ------------------------------------------------------------------------------------------------ mixed-size batches
static_assert(sizeof(vnect_frame) == sizeof(FrameDesc) && sizeof(FrameDesc) == 48 &&
                  offsetof(vnect_frame, data) == offsetof(FrameDesc, data) &&
                  offsetof(vnect_frame, height) == offsetof(FrameDesc, height) &&
                  offsetof(vnect_frame, width) == offsetof(FrameDesc, width) &&
                  offsetof(vnect_frame, pitch) == offsetof(FrameDesc, pitch) &&
                  offsetof(vnect_frame, uv_pitch) == offsetof(FrameDesc, uv_pitch) &&
                  offsetof(vnect_frame, u_offset) == offsetof(FrameDesc, u_offset) &&
                  offsetof(vnect_frame, v_offset) == offsetof(FrameDesc, v_offset),
              "the device frame table is a copy of the caller's vnect_frame array");

static FrameSource frame_source(const vnect_frame& f, int format) {
  FrameSource s = bgr_source(f.pitch, 0);
  s.format = format;
  s.uv_pitch = f.uv_pitch;
  s.u_offset = f.u_offset;
  s.v_offset = f.v_offset;
  return s;
}

// Checks every entry of a mixed-size call's frame table before anything is staged or launched and before any filter
// state or timestamp mirror is touched; `host`: the frames are staged into the lane's buffer, so each must fit max_input.
static int check_frames(vnect_t* h, const vnect_frame* frames, int n_frames, int format, bool host) {
  if (n_frames < 1 || n_frames > h->cfg.max_frames) return fail(h, VNECT_E_INVALID, "n_frames %d not in [1, %d]", n_frames, h->cfg.max_frames);
  if (!frames) return fail(h, VNECT_E_INVALID, "null frame table");
  if (format != kFmtBGR && format != VNECT_FMT_NV12 && format != VNECT_FMT_I420)
    return fail(h, VNECT_E_INVALID, "unknown pixel format %d", format);
  for (int i = 0; i < n_frames; ++i) {
    const vnect_frame& f = frames[i];
    int rc = VNECT_OK;
    if (!f.data) {
      rc = fail(h, VNECT_E_INVALID, "null data");
    } else if (f.height < 2 || f.width < 2) {
      rc = fail(h, VNECT_E_INVALID, "frame %dx%d smaller than 2x2", f.height, f.width);
    } else if (host && (rc = check_host_frame_size(h, f.height, f.width))) {
    } else if (format == kFmtBGR) {
      if (f.pitch < (int64_t)f.width * 3) rc = fail(h, VNECT_E_INVALID, "pitch %lld smaller than a row", (long long)f.pitch);
    } else {
      vnect_yuv_layout l{};
      l.format = format;
      l.y_pitch = f.pitch;
      l.uv_pitch = f.uv_pitch;
      l.u_offset = f.u_offset;
      l.v_offset = f.v_offset;
      rc = check_yuv_layout(h, &l, f.height, f.width);
    }
    if (rc) {
      h->err = "frame " + std::to_string(i) + ": " + h->err;
      return rc;
    }
  }
  return VNECT_OK;
}

// vnect_submit_frames / vnect_track_frames / vnect_submit_track_frames once the table is validated: the frames are
// staged into the lane's buffer one after another (BGR packed tight, YUV in cv2's layout) and the table points at the
// staged copies.  `synchronous`: wait for the lane before returning (vnect_track_frames).  `sequence`: a stream id
// may repeat (vnect_submit_sequence).
static int submit_frames(vnect_t* h, int32_t lane, const vnect_frame* frames, int32_t n_frames, int32_t format,
                         const int32_t* stream_ids, const double* t2d, const double* t3d, double* joints2d,
                         float* joints3d, bool tracked, int32_t* boxes_used, bool synchronous, double* scores,
                         bool sequence = false) {
  int rc = lane_acquire(h, lane);
  if (rc) return rc;
  uint8_t* d = h->cur->d_frames;
  for (int i = 0; i < n_frames; ++i) {  // each frame is within max_input, so the sum fits d_frames_bytes
    const int H = frames[i].height, W = frames[i].width;
    FrameDesc& t = h->cur->h_table[i];
    t.data = d;
    t.height = H;
    t.width = W;
    if (format == kFmtBGR) {
      t.pitch = (int64_t)W * 3;
      t.uv_pitch = t.u_offset = t.v_offset = 0;
      d += (size_t)H * W * 3;
    } else {
      const vnect_yuv_layout l = packed_yuv_layout(format, H, W);
      t.pitch = l.y_pitch;
      t.uv_pitch = l.uv_pitch;
      t.u_offset = l.u_offset;
      t.v_offset = l.v_offset;
      d += (size_t)l.frame_stride;
    }
  }
  // ids, timestamps, the table and any orientation codes in one copy; a refused id or timestamp returns before any
  // frame copy is queued
  const bool oriented = any_oriented(h, n_frames, stream_ids);
  const bool recover = tracked && any_recovering(h, n_frames, stream_ids);
  rc = sequence ? stage_sequence_meta(h, n_frames, stream_ids, t2d, t3d, h->copy_stream, oriented)
                : stage_frame_meta(h, n_frames, stream_ids, t2d, t3d, h->copy_stream, n_frames, oriented, recover);
  if (rc) return rc;
  for (int i = 0; i < n_frames; ++i)
    if ((rc = stage_frame(h, const_cast<uint8_t*>(h->cur->h_table[i].data), frames[i].data, frames[i].height,
                          frames[i].width, frame_source(frames[i], format))))
      return rc;
  CU(h, cudaEventRecord(h->cur->copy_done, h->copy_stream));
  CU(h, cudaStreamWaitEvent(h->stream, h->cur->copy_done, 0));
  if ((rc = run_pipeline(h, lane, nullptr, n_frames, 0, 0, table_source(format), h->cur->d_out2d, h->cur->d_out3d, tracked,
                         sequence, oriented, scores != nullptr, recover)))
    return rc;
  CU(h, cudaMemcpyAsync(joints2d, h->cur->d_out2d, (size_t)n_frames * kJoints * 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaMemcpyAsync(joints3d, h->cur->d_out3d, (size_t)n_frames * kJoints * 3 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  if (boxes_used)
    CU(h, cudaMemcpyAsync(boxes_used, h->d_boxes_used, (size_t)n_frames * 4 * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  if ((rc = copy_scores(h, scores, n_frames, cudaMemcpyDeviceToHost))) return rc;
  CU(h, cudaEventRecord(h->cur->done, h->stream));
  h->cur->pending = true;
  return synchronous ? lane_acquire(h, lane) : VNECT_OK;  // synchronises and reports non-finite maps
}

// vnect_estimate_device_frames / vnect_track_device_frames once the table is validated: the caller's device pointers
// are used as they are; the lanes alternate for the per-call meta so the host can run one call ahead of the GPU
static int device_frames(vnect_t* h, const vnect_frame* frames, int32_t n_frames, int32_t format,
                         const int32_t* stream_ids, const double* t2d, const double* t3d, double* dev_joints2d,
                         float* dev_joints3d, bool tracked, int32_t* dev_boxes_used, double* dev_scores,
                         bool sequence = false) {
  int rc = lane_acquire(h, (int)(h->device_calls++ & 1));
  if (rc) return rc;
  memcpy(h->cur->h_table, frames, (size_t)n_frames * sizeof(FrameDesc));
  const bool oriented = any_oriented(h, n_frames, stream_ids);
  const bool recover = tracked && any_recovering(h, n_frames, stream_ids);
  rc = sequence ? stage_sequence_meta(h, n_frames, stream_ids, t2d, t3d, h->copy_stream, oriented)
                : stage_frame_meta(h, n_frames, stream_ids, t2d, t3d, h->copy_stream, n_frames, oriented, recover);
  if (rc) return rc;
  CU(h, cudaEventRecord(h->cur->copy_done, h->copy_stream));
  CU(h, cudaStreamWaitEvent(h->stream, h->cur->copy_done, 0));
  const int lane = (int)(h->cur - h->lanes);
  if ((rc = run_pipeline(h, lane, nullptr, n_frames, 0, 0, table_source(format), dev_joints2d, dev_joints3d, tracked,
                         sequence, oriented, dev_scores != nullptr, recover)))
    return rc;
  if (dev_boxes_used)  // outside the graph, so the caller's pointer stays out of its key
    CU(h, cudaMemcpyAsync(dev_boxes_used, h->d_boxes_used, (size_t)n_frames * 4 * sizeof(int), cudaMemcpyDeviceToDevice,
                          h->stream));
  if ((rc = copy_scores(h, dev_scores, n_frames, cudaMemcpyDeviceToDevice))) return rc;
  CU(h, cudaEventRecord(h->cur->done, h->stream));
  h->cur->pending = true;
  return VNECT_OK;
}

int vnect_submit_frames(vnect_t* h, int32_t lane, const vnect_frame* frames, int32_t n_frames, int32_t format,
                        const int32_t* stream_ids, const double* t2d, const double* t3d, double* joints2d,
                        float* joints3d) {
  double* const scores = take_scores(h);  // consumed, accepted or refused
  if (!h || !h->finalized) return fail(h, VNECT_E_INVALID, "handle not finalized");
  ON_DEVICE(h);
  if (lane < 0 || lane > 1) return fail(h, VNECT_E_INVALID, "lane must be 0 or 1");
  if (!joints2d || !joints3d) return fail(h, VNECT_E_INVALID, "null buffer");
  if (int rc = check_frames(h, frames, n_frames, format, true)) return rc;
  return submit_frames(h, lane, frames, n_frames, format, stream_ids, t2d, t3d, joints2d, joints3d, false, nullptr,
                       false, scores);
}

int vnect_track_frames(vnect_t* h, const vnect_frame* frames, int32_t n_frames, int32_t format,
                       const int32_t* stream_ids, const double* t2d, const double* t3d, double* joints2d,
                       float* joints3d, int32_t* boxes_used) {
  double* const scores = take_scores(h);  // consumed, accepted or refused
  if (!h || !h->finalized) return fail(h, VNECT_E_INVALID, "handle not finalized");
  ON_DEVICE(h);
  if (!joints2d || !joints3d) return fail(h, VNECT_E_INVALID, "null buffer");
  if (int rc = check_frames(h, frames, n_frames, format, true)) return rc;
  return submit_frames(h, 0, frames, n_frames, format, stream_ids, t2d, t3d, joints2d, joints3d, true, boxes_used,
                       true, scores);
}

// Pipelined and device-resident tracking.  A tracked call no longer has to wait for its results: every kernel that
// reads or writes tracking state runs on the handle's stream in submission order, whichever lane carried the call.
//   d_boxes         frame_geometry_kernel of call k+1 reads the box track_update_frames_kernel of call k wrote.
//   d_boxes_used    written by call k's geometry kernel, read by call k's copy-out; both on the handle's stream, and
//                   call k+1's geometry kernel is enqueued after that copy.
//   d_raw_argmax    written by every call's post-process; vnect_get_raw_argmax waits for all lanes, so it reads the
//                   most recent call's.
//   d_geoms         the uniform tracked path's geometry; the table path uses the lane's own L.d_geoms.
// What a lane stages (meta, table, frames) is only rewritten after lane_acquire has waited for that lane's previous
// call, as for vnect_submit.
int vnect_submit_track_frames(vnect_t* h, int32_t lane, const vnect_frame* frames, int32_t n_frames, int32_t format,
                              const int32_t* stream_ids, const double* t2d, const double* t3d, double* joints2d,
                              float* joints3d, int32_t* boxes_used) {
  double* const scores = take_scores(h);  // consumed, accepted or refused
  if (!h || !h->finalized) return fail(h, VNECT_E_INVALID, "handle not finalized");
  ON_DEVICE(h);
  if (lane < 0 || lane > 1) return fail(h, VNECT_E_INVALID, "lane must be 0 or 1");
  if (!joints2d || !joints3d) return fail(h, VNECT_E_INVALID, "null buffer");
  if (int rc = check_frames(h, frames, n_frames, format, true)) return rc;
  return submit_frames(h, lane, frames, n_frames, format, stream_ids, t2d, t3d, joints2d, joints3d, true, boxes_used,
                       false, scores);
}

int vnect_estimate_device_frames(vnect_t* h, const vnect_frame* frames, int32_t n_frames, int32_t format,
                                 const int32_t* stream_ids, const double* t2d, const double* t3d,
                                 double* dev_joints2d, float* dev_joints3d) {
  double* const scores = take_scores(h);  // consumed, accepted or refused
  if (!h || !h->finalized) return fail(h, VNECT_E_INVALID, "handle not finalized");
  ON_DEVICE(h);
  if (!dev_joints2d || !dev_joints3d) return fail(h, VNECT_E_INVALID, "null buffer");
  if (int rc = check_frames(h, frames, n_frames, format, false)) return rc;
  return device_frames(h, frames, n_frames, format, stream_ids, t2d, t3d, dev_joints2d, dev_joints3d, false, nullptr,
                       scores);
}

int vnect_track_device_frames(vnect_t* h, const vnect_frame* frames, int32_t n_frames, int32_t format,
                              const int32_t* stream_ids, const double* t2d, const double* t3d, double* dev_joints2d,
                              float* dev_joints3d, int32_t* dev_boxes_used) {
  double* const scores = take_scores(h);  // consumed, accepted or refused
  if (!h || !h->finalized) return fail(h, VNECT_E_INVALID, "handle not finalized");
  ON_DEVICE(h);
  if (!dev_joints2d || !dev_joints3d) return fail(h, VNECT_E_INVALID, "null buffer");
  if (int rc = check_frames(h, frames, n_frames, format, false)) return rc;
  return device_frames(h, frames, n_frames, format, stream_ids, t2d, t3d, dev_joints2d, dev_joints3d, true,
                       dev_boxes_used, scores);
}

// Sequence calls (include/vnect_b200.h): the table paths above with a stream id allowed to repeat.  Filter state is
// read and written only by sequence_filter_kernel on the handle's stream, so a stream continues across sequence calls
// on either lane and across ordinary calls in submission order.
int vnect_submit_sequence(vnect_t* h, int32_t lane, const vnect_frame* frames, int32_t n_frames, int32_t format,
                          const int32_t* stream_ids, const double* t2d, const double* t3d, double* joints2d,
                          float* joints3d) {
  double* const scores = take_scores(h);  // consumed, accepted or refused
  if (!h || !h->finalized) return fail(h, VNECT_E_INVALID, "handle not finalized");
  ON_DEVICE(h);
  if (lane < 0 || lane > 1) return fail(h, VNECT_E_INVALID, "lane must be 0 or 1");
  if (!joints2d || !joints3d) return fail(h, VNECT_E_INVALID, "null buffer");
  if (int rc = check_frames(h, frames, n_frames, format, true)) return rc;
  return submit_frames(h, lane, frames, n_frames, format, stream_ids, t2d, t3d, joints2d, joints3d, false, nullptr,
                       false, scores, true);
}

int vnect_estimate_device_sequence(vnect_t* h, const vnect_frame* frames, int32_t n_frames, int32_t format,
                                   const int32_t* stream_ids, const double* t2d, const double* t3d,
                                   double* dev_joints2d, float* dev_joints3d) {
  double* const scores = take_scores(h);  // consumed, accepted or refused
  if (!h || !h->finalized) return fail(h, VNECT_E_INVALID, "handle not finalized");
  ON_DEVICE(h);
  if (!dev_joints2d || !dev_joints3d) return fail(h, VNECT_E_INVALID, "null buffer");
  if (int rc = check_frames(h, frames, n_frames, format, false)) return rc;
  return device_frames(h, frames, n_frames, format, stream_ids, t2d, t3d, dev_joints2d, dev_joints3d, false, nullptr,
                       scores, true);
}

int vnect_estimate_device(vnect_t* h, const uint8_t* dev_bgr, int32_t n_frames, int32_t H, int32_t W, int64_t pitch,
                          int64_t frame_stride, const int32_t* stream_ids, const double* t2d, const double* t3d,
                          double* dev_joints2d, float* dev_joints3d) {
  double* const scores = take_scores(h);  // consumed, accepted or refused
  if (!h || !h->finalized) return fail(h, VNECT_E_INVALID, "handle not finalized");
  ON_DEVICE(h);
  if (!dev_bgr || !dev_joints2d || !dev_joints3d) return fail(h, VNECT_E_INVALID, "null buffer");
  if (H < 2 || W < 2 || pitch < (int64_t)W * 3) return fail(h, VNECT_E_INVALID, "bad frame geometry %dx%d pitch %lld", H, W, (long long)pitch);
  return estimate_device(h, dev_bgr, n_frames, H, W, bgr_source(pitch, frame_stride), stream_ids, t2d, t3d,
                         dev_joints2d, dev_joints3d, scores);
}

int vnect_estimate_device_yuv(vnect_t* h, const uint8_t* dev_frames, int32_t n_frames, int32_t H, int32_t W,
                              const vnect_yuv_layout* layout, const int32_t* stream_ids, const double* t2d,
                              const double* t3d, double* dev_joints2d, float* dev_joints3d) {
  double* const scores = take_scores(h);  // consumed, accepted or refused
  if (!h || !h->finalized) return fail(h, VNECT_E_INVALID, "handle not finalized");
  ON_DEVICE(h);
  if (!dev_frames || !dev_joints2d || !dev_joints3d) return fail(h, VNECT_E_INVALID, "null buffer");
  if (int rc = check_yuv_layout(h, layout, H, W)) return rc;
  return estimate_device(h, dev_frames, n_frames, H, W, yuv_source(*layout), stream_ids, t2d, t3d, dev_joints2d,
                         dev_joints3d, scores);
}

int vnect_submit(vnect_t* h, int32_t lane, const uint8_t* bgr, int32_t n_frames, int32_t H, int32_t W, int64_t pitch,
                 int64_t frame_stride, const int32_t* stream_ids, const double* t2d, const double* t3d, double* joints2d,
                 float* joints3d) {
  double* const scores = take_scores(h);  // consumed, accepted or refused
  if (!h || !h->finalized) return fail(h, VNECT_E_INVALID, "handle not finalized");
  ON_DEVICE(h);
  if (lane < 0 || lane > 1) return fail(h, VNECT_E_INVALID, "lane must be 0 or 1");
  if (!bgr || !joints2d || !joints3d) return fail(h, VNECT_E_INVALID, "null buffer");
  if (n_frames < 1 || n_frames > h->cfg.max_frames) return fail(h, VNECT_E_INVALID, "n_frames %d not in [1, %d]", n_frames, h->cfg.max_frames);
  if (int rc = check_host_frame_size(h, H, W)) return rc;
  if (pitch < (int64_t)W * 3) return fail(h, VNECT_E_INVALID, "pitch smaller than a row");
  return submit(h, lane, bgr, n_frames, H, W, bgr_source(pitch, frame_stride), stream_ids, t2d, t3d, joints2d, joints3d,
                scores);
}

int vnect_submit_yuv(vnect_t* h, int32_t lane, const uint8_t* frames, int32_t n_frames, int32_t H, int32_t W,
                     const vnect_yuv_layout* layout, const int32_t* stream_ids, const double* t2d, const double* t3d,
                     double* joints2d, float* joints3d) {
  double* const scores = take_scores(h);  // consumed, accepted or refused
  if (!h || !h->finalized) return fail(h, VNECT_E_INVALID, "handle not finalized");
  ON_DEVICE(h);
  if (lane < 0 || lane > 1) return fail(h, VNECT_E_INVALID, "lane must be 0 or 1");
  if (!frames || !joints2d || !joints3d) return fail(h, VNECT_E_INVALID, "null buffer");
  if (n_frames < 1 || n_frames > h->cfg.max_frames) return fail(h, VNECT_E_INVALID, "n_frames %d not in [1, %d]", n_frames, h->cfg.max_frames);
  if (int rc = check_host_frame_size(h, H, W)) return rc;
  if (int rc = check_yuv_layout(h, layout, H, W)) return rc;
  return submit(h, lane, frames, n_frames, H, W, yuv_source(*layout), stream_ids, t2d, t3d, joints2d, joints3d,
                scores);
}

int vnect_track_set_box(vnect_t* h, int32_t stream_id, int32_t x, int32_t y, int32_t w, int32_t hh) {
  if (!h || !h->d_boxes) return fail(h, VNECT_E_INVALID, "handle not created");
  ON_DEVICE(h);
  if (stream_id < 0 || stream_id >= h->cfg.max_streams) return fail(h, VNECT_E_INVALID, "stream id out of range");
  if (x < 0 || y < 0 || w < 2 || hh < 2) return fail(h, VNECT_E_INVALID, "box must have x, y >= 0 and w, h >= 2");
  const int4 b = make_int4(x, y, w, hh);
  CU(h, cudaStreamSynchronize(h->stream));
  CU(h, cudaMemcpy(h->d_boxes + stream_id, &b, sizeof b, cudaMemcpyHostToDevice));
  return VNECT_OK;
}

int vnect_track_set_boxes(vnect_t* h, int32_t n, const int32_t* stream_ids, const int32_t* xywh) {
  if (!h || !h->d_boxes) return fail(h, VNECT_E_INVALID, "handle not created");
  ON_DEVICE(h);
  if (n < 0) return fail(h, VNECT_E_INVALID, "n %d below 0", n);
  if (n == 0) return VNECT_OK;
  if (!stream_ids || !xywh) return fail(h, VNECT_E_INVALID, "null buffer");
  h->seen_stamp.resize(h->cfg.max_streams, 0);
  const unsigned int stamp = ++h->seen_epoch;
  for (int i = 0; i < n; ++i) {  // everything is checked before the first launch
    const int sid = stream_ids[i];
    const int32_t* b = xywh + 4 * i;
    if (sid < 0 || sid >= h->cfg.max_streams) return fail(h, VNECT_E_INVALID, "stream id %d not in [0, %d)", sid, h->cfg.max_streams);
    if (h->seen_stamp[sid] == stamp) return fail(h, VNECT_E_INVALID, "stream id %d appears twice", sid);
    h->seen_stamp[sid] = stamp;
    if (b[0] < 0 || b[1] < 0 || b[2] < 2 || b[3] < 2)
      return fail(h, VNECT_E_INVALID, "box %d of stream %d must have x, y >= 0 and w, h >= 2", i, sid);
  }
  for (int i0 = 0; i0 < n; i0 += kSeedBoxes) {
    BoxSeeds s;
    s.n = std::min(kSeedBoxes, n - i0);
    for (int i = 0; i < s.n; ++i) {
      const int32_t* b = xywh + 4 * (i0 + i);
      s.box[i] = make_int4(b[0], b[1], b[2], b[3]);
      s.stream_id[i] = stream_ids[i0 + i];
    }
    track_seed_boxes_kernel<<<1, kSeedBoxes, 0, h->stream>>>(s, h->d_boxes);
    CU(h, cudaGetLastError());
    ++h->launches;
  }
  return VNECT_OK;
}

int vnect_track_get_box(vnect_t* h, int32_t stream_id, int32_t* xywh) {
  if (!h || !h->d_boxes || !xywh) return fail(h, VNECT_E_INVALID, "handle not created / null buffer");
  ON_DEVICE(h);
  if (stream_id < 0 || stream_id >= h->cfg.max_streams) return fail(h, VNECT_E_INVALID, "stream id out of range");
  CU(h, cudaStreamSynchronize(h->stream));
  int4 b;
  CU(h, cudaMemcpy(&b, h->d_boxes + stream_id, sizeof b, cudaMemcpyDeviceToHost));
  xywh[0] = b.x; xywh[1] = b.y; xywh[2] = b.z; xywh[3] = b.w;
  return VNECT_OK;
}

int vnect_set_orientations(vnect_t* h, int32_t n, const int32_t* stream_ids, const int32_t* codes) {
  if (!h || h->orient.empty()) return fail(h, VNECT_E_INVALID, "handle not created");
  if (n < 0) return fail(h, VNECT_E_INVALID, "n %d below 0", n);
  if (n == 0) return VNECT_OK;
  if (!stream_ids || !codes) return fail(h, VNECT_E_INVALID, "null buffer");
  h->seen_stamp.resize(h->cfg.max_streams, 0);
  const unsigned int stamp = ++h->seen_epoch;
  for (int i = 0; i < n; ++i) {  // everything is checked before the first change
    const int sid = stream_ids[i];
    if (sid < 0 || sid >= h->cfg.max_streams) return fail(h, VNECT_E_INVALID, "stream id %d not in [0, %d)", sid, h->cfg.max_streams);
    if (h->seen_stamp[sid] == stamp) return fail(h, VNECT_E_INVALID, "stream id %d appears twice", sid);
    h->seen_stamp[sid] = stamp;
    if (codes[i] < VNECT_ORIENT_IDENTITY || codes[i] > VNECT_ORIENT_TRANSVERSE)
      return fail(h, VNECT_E_INVALID, "orientation %d of stream %d not in [0, 8)", codes[i], sid);
  }
  for (int i = 0; i < n; ++i) h->orient[stream_ids[i]] = codes[i];
  return VNECT_OK;
}

int vnect_get_orientation(vnect_t* h, int32_t stream_id, int32_t* code) {
  if (!h || h->orient.empty() || !code) return fail(h, VNECT_E_INVALID, "handle not created / null buffer");
  if (stream_id < 0 || stream_id >= h->cfg.max_streams) return fail(h, VNECT_E_INVALID, "stream id out of range");
  *code = h->orient[stream_id];
  return VNECT_OK;
}

int vnect_request_scores(vnect_t* h, double* scores) {
  if (!h) return fail(h, VNECT_E_INVALID, "null handle");
  h->score_req = scores;
  return VNECT_OK;
}

int vnect_set_track_recovery(vnect_t* h, int32_t n, const int32_t* stream_ids, const double* min_mean_score) {
  if (!h || h->recover.empty()) return fail(h, VNECT_E_INVALID, "handle not created");
  if (n < 0) return fail(h, VNECT_E_INVALID, "n %d below 0", n);
  if (n == 0) return VNECT_OK;
  if (!stream_ids || !min_mean_score) return fail(h, VNECT_E_INVALID, "null buffer");
  h->seen_stamp.resize(h->cfg.max_streams, 0);
  const unsigned int stamp = ++h->seen_epoch;
  for (int i = 0; i < n; ++i) {  // everything is checked before the first change
    const int sid = stream_ids[i];
    if (sid < 0 || sid >= h->cfg.max_streams) return fail(h, VNECT_E_INVALID, "stream id %d not in [0, %d)", sid, h->cfg.max_streams);
    if (h->seen_stamp[sid] == stamp) return fail(h, VNECT_E_INVALID, "stream id %d appears twice", sid);
    h->seen_stamp[sid] = stamp;
    if (!(min_mean_score[i] >= 0.0 && min_mean_score[i] < INFINITY))
      return fail(h, VNECT_E_INVALID, "recovery threshold %g of stream %d is not a finite value >= 0", min_mean_score[i], sid);
  }
  for (int i = 0; i < n; ++i) h->recover[stream_ids[i]] = min_mean_score[i];
  return VNECT_OK;
}

int vnect_get_track_recovery(vnect_t* h, int32_t stream_id, double* min_mean_score) {
  if (!h || h->recover.empty() || !min_mean_score) return fail(h, VNECT_E_INVALID, "handle not created / null buffer");
  if (stream_id < 0 || stream_id >= h->cfg.max_streams) return fail(h, VNECT_E_INVALID, "stream id out of range");
  *min_mean_score = h->recover[stream_id];
  return VNECT_OK;
}

int vnect_track(vnect_t* h, const uint8_t* frames, int32_t n_frames, int32_t FH, int32_t FW, int64_t pitch,
                int64_t frame_stride, const int32_t* stream_ids, const double* t2d, const double* t3d, double* joints2d,
                float* joints3d, int32_t* boxes_used) {
  double* const scores = take_scores(h);  // consumed, accepted or refused
  if (!h || !h->finalized) return fail(h, VNECT_E_INVALID, "handle not finalized");
  ON_DEVICE(h);
  if (!frames || !joints2d || !joints3d) return fail(h, VNECT_E_INVALID, "null buffer");
  if (n_frames < 1 || n_frames > h->cfg.max_frames) return fail(h, VNECT_E_INVALID, "n_frames %d not in [1, %d]", n_frames, h->cfg.max_frames);
  if (int rc = check_host_frame_size(h, FH, FW)) return rc;
  if (pitch < (int64_t)FW * 3) return fail(h, VNECT_E_INVALID, "pitch smaller than a row");
  return track(h, frames, n_frames, FH, FW, bgr_source(pitch, frame_stride), stream_ids, t2d, t3d, joints2d, joints3d,
               boxes_used, scores);
}

int vnect_track_yuv(vnect_t* h, const uint8_t* frames, int32_t n_frames, int32_t FH, int32_t FW,
                    const vnect_yuv_layout* layout, const int32_t* stream_ids, const double* t2d, const double* t3d,
                    double* joints2d, float* joints3d, int32_t* boxes_used) {
  double* const scores = take_scores(h);  // consumed, accepted or refused
  if (!h || !h->finalized) return fail(h, VNECT_E_INVALID, "handle not finalized");
  ON_DEVICE(h);
  if (!frames || !joints2d || !joints3d) return fail(h, VNECT_E_INVALID, "null buffer");
  if (n_frames < 1 || n_frames > h->cfg.max_frames) return fail(h, VNECT_E_INVALID, "n_frames %d not in [1, %d]", n_frames, h->cfg.max_frames);
  if (int rc = check_host_frame_size(h, FH, FW)) return rc;
  if (int rc = check_yuv_layout(h, layout, FH, FW)) return rc;
  return track(h, frames, n_frames, FH, FW, yuv_source(*layout), stream_ids, t2d, t3d, joints2d, joints3d, boxes_used,
               scores);
}

int vnect_wait(vnect_t* h, int32_t lane) {
  if (!h || lane < 0 || lane > 1) return fail(h, VNECT_E_INVALID, "bad handle or lane");
  ON_DEVICE(h);
  return lane_acquire(h, lane);
}

int vnect_estimate(vnect_t* h, const uint8_t* bgr, int32_t n_frames, int32_t H, int32_t W, int64_t pitch,
                   int64_t frame_stride, const int32_t* stream_ids, const double* t2d, const double* t3d,
                   double* joints2d, float* joints3d) {
  int rc = vnect_submit(h, 0, bgr, n_frames, H, W, pitch, frame_stride, stream_ids, t2d, t3d, joints2d, joints3d);
  if (rc) return rc;
  return vnect_wait(h, 0);
}

int vnect_preprocess(vnect_t* h, const uint8_t* bgr, int32_t n_frames, int32_t H, int32_t W, int64_t pitch,
                     int64_t frame_stride, float* out_nhwc, double* scaler_offsets) {
  if (!h || !h->x1) return fail(h, VNECT_E_INVALID, "handle not created");
  ON_DEVICE(h);
  if (!bgr || !out_nhwc) return fail(h, VNECT_E_INVALID, "null buffer");
  if (n_frames < 1 || n_frames > h->cfg.max_frames) return fail(h, VNECT_E_INVALID, "n_frames out of range");
  if (H < 2 || W < 2 || H > h->cfg.max_input_h || W > h->cfg.max_input_w) return fail(h, VNECT_E_INVALID, "frame size outside max_input");
  const int64_t dpitch = (int64_t)W * 3, dstride = dpitch * H;
  if (lane_acquire(h, 0)) return VNECT_E_CUDA;
  for (int i = 0; i < n_frames; ++i)
    CU(h, cudaMemcpy2DAsync(h->cur->d_frames + (size_t)i * dstride, dpitch, bgr + (size_t)i * frame_stride, pitch, dpitch, H, cudaMemcpyHostToDevice, h->stream));
  const Geometry g = squarify_geometry(h->S, H, W);
  int rc = run_preprocess(h, h->cur->d_frames, n_frames, H, W, bgr_source(dpitch, dstride), g);
  if (rc) return rc;
  const int n = n_frames * h->n_scales, S = h->S;
  stem_to_f32_kernel<<<grid_for((int64_t)n * S * S, 256, h->num_sms), 256, 0, h->stream>>>(h->x1, h->d_f32_in, n, S, h->stem_rpp, h->stem_pitch);
  CU(h, cudaGetLastError());
  ++h->launches;
  CU(h, cudaMemcpyAsync(out_nhwc, h->d_f32_in, (size_t)n * S * S * 3 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaStreamSynchronize(h->stream));
  if (scaler_offsets) {
    scaler_offsets[0] = g.scaler;
    scaler_offsets[1] = g.off_x;
    scaler_offsets[2] = g.off_y;
  }
  return VNECT_OK;
}

// caller-supplied NHWC maps [n_frames*n_scales][hs][hs][21] -> the planar fp32 maps the CNN writes, then to h->maps on
// the handle's stream.  A copy from pageable memory has read its source when it returns, so the vector may go.
static int stage_maps(vnect_t* h, const float* hm, const float* xm, const float* ym, const float* zm, int n_frames) {
  const int n = n_frames * h->n_scales, hs = h->hs;
  const size_t plane = (size_t)hs * hs;
  std::vector<float> planar((size_t)n * 84 * plane);
  const float* ins[4] = {hm, xm, ym, zm};
  for (int i = 0; i < n; ++i)
    for (int m = 0; m < 4; ++m)
      for (int j = 0; j < kJoints; ++j) {
        float* dst = planar.data() + ((size_t)i * 84 + m * kJoints + j) * plane;
        const float* src = ins[m] + (size_t)i * plane * kJoints + j;
        for (size_t px = 0; px < plane; ++px) dst[px] = src[px * kJoints];
      }
  CU(h, cudaMemcpyAsync(h->maps, planar.data(), planar.size() * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  return VNECT_OK;
}

int vnect_postprocess(vnect_t* h, const float* hm, const float* xm, const float* ym, const float* zm, int32_t n_frames,
                      const int32_t* stream_ids, const double* t2d, const double* t3d, double scaler, int32_t offset_x,
                      int32_t offset_y, double* joints2d, float* joints3d, int32_t* raw_argmax) {
  double* const scores = take_scores(h);  // consumed, accepted or refused
  if (!h || !h->x1) return fail(h, VNECT_E_INVALID, "handle not created");
  ON_DEVICE(h);
  if (!hm || !xm || !ym || !zm || !joints2d || !joints3d) return fail(h, VNECT_E_INVALID, "null buffer");
  int rc = lane_acquire(h, 0);
  if (rc) return rc;
  if ((rc = stage_frame_meta(h, n_frames, stream_ids, t2d, t3d, h->stream))) return rc;
  if ((rc = stage_maps(h, hm, xm, ym, zm, n_frames))) return rc;
  if ((rc = run_postprocess(h, n_frames, scaler, offset_x, offset_y, h->cur->d_out2d, h->cur->d_out3d, nullptr, false,
                            nullptr, scores != nullptr)))
    return rc;
  CU(h, cudaMemcpyAsync(joints2d, h->cur->d_out2d, (size_t)n_frames * kJoints * 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaMemcpyAsync(joints3d, h->cur->d_out3d, (size_t)n_frames * kJoints * 3 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  if (raw_argmax)
    CU(h, cudaMemcpyAsync(raw_argmax, h->d_raw_argmax, (size_t)n_frames * kJoints * 2 * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  if ((rc = copy_scores(h, scores, n_frames, cudaMemcpyDeviceToHost))) return rc;
  CU(h, cudaStreamSynchronize(h->stream));
  return VNECT_OK;
}

// vnect_postprocess for a sequence call: the argmax launch and sequence_filter_kernel on the given maps, lane 0.
int vnect_postprocess_sequence(vnect_t* h, const float* hm, const float* xm, const float* ym, const float* zm,
                               int32_t n_frames, const int32_t* stream_ids, const double* t2d, const double* t3d,
                               double scaler, int32_t offset_x, int32_t offset_y, double* joints2d, float* joints3d,
                               int32_t* raw_argmax) {
  double* const scores = take_scores(h);  // consumed, accepted or refused
  if (!h || !h->x1) return fail(h, VNECT_E_INVALID, "handle not created");
  ON_DEVICE(h);
  if (!hm || !xm || !ym || !zm || !joints2d || !joints3d) return fail(h, VNECT_E_INVALID, "null buffer");
  int rc = lane_acquire(h, 0);
  if (rc) return rc;
  vnect_handle::Lane* L = h->cur;
  if ((rc = stage_sequence_meta(h, n_frames, stream_ids, t2d, t3d, h->stream))) return rc;
  if ((rc = stage_maps(h, hm, xm, ym, zm, n_frames))) return rc;
  if ((rc = run_postprocess(h, n_frames, scaler, offset_x, offset_y, L->d_out2d, L->d_out3d, nullptr, false, L->d_seg,
                            scores != nullptr)))
    return rc;
  CU(h, cudaMemcpyAsync(joints2d, L->d_out2d, (size_t)n_frames * kJoints * 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaMemcpyAsync(joints3d, L->d_out3d, (size_t)n_frames * kJoints * 3 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  if (raw_argmax)
    CU(h, cudaMemcpyAsync(raw_argmax, h->d_raw_argmax, (size_t)n_frames * kJoints * 2 * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  if ((rc = copy_scores(h, scores, n_frames, cudaMemcpyDeviceToHost))) return rc;
  CU(h, cudaStreamSynchronize(h->stream));
  return VNECT_OK;
}

// The tracked tail of vnect_track_frames on caller-supplied maps: the three launches of run_pipeline's table path after
// the CNN (frame geometry from the stream boxes, post-process with per-frame geometry, box update), on lane 0's table.
// Only the frame sizes of the table are read, so its entries carry no data pointer.
int vnect_track_postprocess(vnect_t* h, const float* hm, const float* xm, const float* ym, const float* zm,
                            int32_t n_frames, const int32_t* frame_hw, const int32_t* stream_ids, const double* t2d,
                            const double* t3d, double* joints2d, float* joints3d, int32_t* boxes_used) {
  double* const scores = take_scores(h);  // consumed, accepted or refused
  if (!h || !h->x1) return fail(h, VNECT_E_INVALID, "handle not created");
  ON_DEVICE(h);
  if (!hm || !xm || !ym || !zm || !frame_hw || !joints2d || !joints3d) return fail(h, VNECT_E_INVALID, "null buffer");
  if (n_frames < 1 || n_frames > h->cfg.max_frames) return fail(h, VNECT_E_INVALID, "n_frames %d not in [1, %d]", n_frames, h->cfg.max_frames);
  for (int i = 0; i < n_frames; ++i)  // before the ids and timestamps are checked and recorded, as check_frames does
    if (frame_hw[2 * i] < 2 || frame_hw[2 * i + 1] < 2)
      return fail(h, VNECT_E_INVALID, "frame %d: frame %dx%d smaller than 2x2", i, frame_hw[2 * i], frame_hw[2 * i + 1]);
  int rc = lane_acquire(h, 0);
  if (rc) return rc;
  vnect_handle::Lane* L = h->cur;
  for (int i = 0; i < n_frames; ++i) {
    FrameDesc& t = L->h_table[i];
    memset(&t, 0, sizeof t);
    t.height = frame_hw[2 * i];
    t.width = frame_hw[2 * i + 1];
  }
  const bool recover = any_recovering(h, n_frames, stream_ids);
  if ((rc = stage_frame_meta(h, n_frames, stream_ids, t2d, t3d, h->stream, n_frames, false, recover))) return rc;
  if ((rc = stage_maps(h, hm, xm, ym, zm, n_frames))) return rc;
  frame_geometry_kernel<<<(n_frames + 63) / 64, 64, 0, h->stream>>>(L->d_table, h->d_boxes, L->d_stream_ids, n_frames,
                                                                    h->S, L->d_geoms, h->d_boxes_used);
  CU(h, cudaGetLastError());
  ++h->launches;
  if ((rc = run_postprocess(h, n_frames, 1.0, 0, 0, L->d_out2d, L->d_out3d, L->d_geoms, false, nullptr,
                            scores != nullptr || recover)))
    return rc;
  if (recover)
    track_update_frames_recover_kernel<<<n_frames, 32, 0, h->stream>>>(L->d_out2d, L->d_stream_ids, L->d_table, nullptr,
                                                                       h->d_scores, L->d_recover, h->d_boxes);
  else
    track_update_frames_kernel<<<n_frames, 32, 0, h->stream>>>(L->d_out2d, L->d_stream_ids, L->d_table, h->d_boxes);
  CU(h, cudaGetLastError());
  ++h->launches;
  CU(h, cudaMemcpyAsync(joints2d, L->d_out2d, (size_t)n_frames * kJoints * 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaMemcpyAsync(joints3d, L->d_out3d, (size_t)n_frames * kJoints * 3 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  if (boxes_used)
    CU(h, cudaMemcpyAsync(boxes_used, h->d_boxes_used, (size_t)n_frames * 4 * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  if ((rc = copy_scores(h, scores, n_frames, cudaMemcpyDeviceToHost))) return rc;
  CU(h, cudaStreamSynchronize(h->stream));
  return VNECT_OK;
}

int vnect_reset_stream(vnect_t* h, int32_t stream_id) {
  if (!h || !h->d_st2d) return fail(h, VNECT_E_INVALID, "handle not finalized");
  ON_DEVICE(h);
  const int ms = h->cfg.max_streams;
  if (stream_id < -1 || stream_id >= ms) return fail(h, VNECT_E_INVALID, "stream id out of range");
  const int lo = stream_id < 0 ? 0 : stream_id, hi = stream_id < 0 ? ms : stream_id + 1;
  std::vector<FilterState> s2((size_t)(hi - lo) * kJoints * 2), s3((size_t)(hi - lo) * kJoints * 3);
  FilterState z;
  memset(&z, 0, sizeof z);
  z.freq = 30.0;  // estimator.py:35,41
  for (auto& s : s2) s = z;
  for (auto& s : s3) s = z;
  CU(h, cudaStreamSynchronize(h->stream));
  CU(h, cudaMemcpy(h->d_st2d + (size_t)lo * kJoints * 2, s2.data(), s2.size() * sizeof(FilterState), cudaMemcpyHostToDevice));
  CU(h, cudaMemcpy(h->d_st3d + (size_t)lo * kJoints * 3, s3.data(), s3.size() * sizeof(FilterState), cudaMemcpyHostToDevice));
  {
    FilterState za = z;
    za.freq = 120.0;  // joints2angles.py:36
    std::vector<FilterState> sa((size_t)(hi - lo) * 8, za);
    CU(h, cudaMemcpy(h->d_st_ang + (size_t)lo * 8, sa.data(), sa.size() * sizeof(FilterState), cudaMemcpyHostToDevice));
    for (int i = lo; i < hi; ++i) h->last_t_ang[i] = NAN;
  }
  for (int i = lo; i < hi; ++i) h->last_t2d[i] = h->last_t3d[i] = NAN;
  // the tracked crop box restarts as the whole frame (run_estimator.py:68: rect = 0, 0, W_img, H_img); the geometry
  // kernel clips it to the actual frame size
  std::vector<int4> full((size_t)(hi - lo), make_int4(0, 0, 1 << 30, 1 << 30));
  CU(h, cudaMemcpy(h->d_boxes + lo, full.data(), full.size() * sizeof(int4), cudaMemcpyHostToDevice));
  return VNECT_OK;
}

int vnect_filter(vnect_t* h, int32_t stream_id, int32_t dim, int32_t values_are_f32, double t, double* values) {
  if (!h || !h->x1 || !values) return fail(h, VNECT_E_INVALID, "handle not created / null buffer");
  ON_DEVICE(h);
  if (stream_id < 0 || stream_id >= h->cfg.max_streams || (dim != 2 && dim != 3)) return fail(h, VNECT_E_INVALID, "bad stream id or dim");
  std::vector<double>& last = dim == 2 ? h->last_t2d : h->last_t3d;
  if (last[stream_id] == last[stream_id] && last[stream_id] != 0.0 && t != 0.0) {
    if (t == last[stream_id])
      return fail(h, VNECT_E_ZERO_DT, "float division by zero (stream %d: repeated timestamp %.17g)", stream_id, t);
    if (t < last[stream_id])
      return fail(h, VNECT_E_INVALID, "alpha should be in (0.0, 1.0] (stream %d: timestamp %.17g earlier than the previous %.17g)", stream_id, t, last[stream_id]);
  }
  last[stream_id] = t;
  const int n = kJoints * dim;
  CU(h, cudaMemcpyAsync(h->d_filter_scratch, values, n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  FilterState* st = dim == 2 ? h->d_st2d + (size_t)stream_id * kJoints * 2 : h->d_st3d + (size_t)stream_id * kJoints * 3;
  const FilterCfg cfg = dim == 2 ? FilterCfg{30.0, 1.7, 0.3, 0.4} : FilterCfg{30.0, 0.8, 0.4, 0.4};
  joint_filter_kernel<<<1, 64, 0, h->stream>>>(st, cfg, h->d_filter_scratch, t, dim, values_are_f32 ? 1 : 0);
  CU(h, cudaGetLastError());
  ++h->launches;
  CU(h, cudaMemcpyAsync(values, h->d_filter_scratch, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaStreamSynchronize(h->stream));
  return VNECT_OK;
}

// waits for every submitted batch: the per-call scratch (raw argmax) and the per-stream state are then at rest.  A lane
// stays pending, so that its vnect_wait (or its next use) still reports NaN / Inf maps of the batch it carried.
static int quiesce(vnect_t* h) {
  for (auto& L : h->lanes)
    if (L.pending) CU(h, cudaEventSynchronize(L.done));
  CU(h, cudaStreamSynchronize(h->stream));
  return VNECT_OK;
}

int vnect_joints2angles(vnect_t* h, const float* joints3d, int32_t n, const int32_t* stream_ids, const double* t,
                        double* angles) {
  if (!h || !h->d_st_ang || !joints3d || !angles) return fail(h, VNECT_E_INVALID, "handle not created / null buffer");
  ON_DEVICE(h);
  if (n < 1 || n > h->cfg.max_frames) return fail(h, VNECT_E_INVALID, "n %d not in [1, %d]", n, h->cfg.max_frames);
  std::vector<int> ids(n);
  for (int i = 0; i < n; ++i) {
    ids[i] = stream_ids ? stream_ids[i] : i;
    if (ids[i] < 0 || ids[i] >= h->cfg.max_streams) return fail(h, VNECT_E_INVALID, "stream id out of range");
    if (t) {  // same clock rules as the joint filters (OneEuroFilter.py:21-22, 66)
      const double last = h->last_t_ang[ids[i]];
      if (last == last && last != 0.0 && t[i] != 0.0) {
        if (t[i] == last) return fail(h, VNECT_E_ZERO_DT, "float division by zero (stream %d: repeated timestamp %.17g)", ids[i], t[i]);
        if (t[i] < last) return fail(h, VNECT_E_INVALID, "alpha should be in (0.0, 1.0] (stream %d: timestamp %.17g earlier than the previous %.17g)", ids[i], t[i], last);
      }
    }
  }
  if (t) for (int i = 0; i < n; ++i) h->last_t_ang[ids[i]] = t[i];
  CU(h, cudaMemcpyAsync(h->d_ang_in, joints3d, (size_t)n * kJoints * 3 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  CU(h, cudaMemcpyAsync(h->d_ang_ids, ids.data(), n * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  if (t) CU(h, cudaMemcpyAsync(h->d_ang_t, t, n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  AnglesParams ap;
  ap.joints3d = h->d_ang_in; ap.stream_ids = h->d_ang_ids; ap.t = t ? h->d_ang_t : nullptr;
  ap.st = h->d_st_ang; ap.angles = h->d_ang_out; ap.n = n;
  joints2angles_kernel<<<(n + 63) / 64, 64, 0, h->stream>>>(ap);
  CU(h, cudaGetLastError());
  ++h->launches;
  CU(h, cudaMemcpyAsync(angles, h->d_ang_out, (size_t)n * 8 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(h, cudaStreamSynchronize(h->stream));  // ids is a host temporary
  return VNECT_OK;
}

int vnect_get_raw_argmax(vnect_t* h, int32_t n_frames, int32_t* raw_argmax) {
  if (!h || !h->d_raw_argmax || !raw_argmax) return fail(h, VNECT_E_INVALID, "handle not created / null buffer");
  ON_DEVICE(h);
  if (n_frames < 1 || n_frames > h->cfg.max_frames) return fail(h, VNECT_E_INVALID, "n_frames out of range");
  if (int rc = quiesce(h)) return rc;
  CU(h, cudaMemcpy(raw_argmax, h->d_raw_argmax, (size_t)n_frames * kJoints * 2 * sizeof(int), cudaMemcpyDeviceToHost));
  return VNECT_OK;
}

// Per-stream temporal state as plain doubles (VNECT_STREAM_STATE_DOUBLES of them): 105 filters x {prev, s_x, s_dx,
// lasttime, freq, has_prev, has_time} (2D filters first, [21][2], then 3D, [21][3]), then the host-side last timestamps
// (2D, 3D; NaN = none) and the tracked box (x, y, w, h).
int vnect_export_stream_state(vnect_t* h, int32_t stream_id, double* state) {
  if (!h || !h->d_st2d || !state) return fail(h, VNECT_E_INVALID, "handle not created / null buffer");
  ON_DEVICE(h);
  if (stream_id < 0 || stream_id >= h->cfg.max_streams) return fail(h, VNECT_E_INVALID, "stream id out of range");
  if (int rc = quiesce(h)) return rc;
  std::vector<FilterState> st(kJoints * 5);
  CU(h, cudaMemcpy(st.data(), h->d_st2d + (size_t)stream_id * kJoints * 2, kJoints * 2 * sizeof(FilterState), cudaMemcpyDeviceToHost));
  CU(h, cudaMemcpy(st.data() + kJoints * 2, h->d_st3d + (size_t)stream_id * kJoints * 3, kJoints * 3 * sizeof(FilterState), cudaMemcpyDeviceToHost));
  for (int i = 0; i < kJoints * 5; ++i) {
    double* o = state + 7 * i;
    o[0] = st[i].prev; o[1] = st[i].s_x; o[2] = st[i].s_dx; o[3] = st[i].lasttime; o[4] = st[i].freq;
    o[5] = st[i].has_prev; o[6] = st[i].has_time;
  }
  int4 b;
  CU(h, cudaMemcpy(&b, h->d_boxes + stream_id, sizeof b, cudaMemcpyDeviceToHost));
  double* tail = state + 7 * kJoints * 5;
  tail[0] = h->last_t2d[stream_id]; tail[1] = h->last_t3d[stream_id];
  tail[2] = b.x; tail[3] = b.y; tail[4] = b.z; tail[5] = b.w;
  return VNECT_OK;
}

int vnect_import_stream_state(vnect_t* h, int32_t stream_id, const double* state) {
  if (!h || !h->d_st2d || !state) return fail(h, VNECT_E_INVALID, "handle not created / null buffer");
  ON_DEVICE(h);
  if (stream_id < 0 || stream_id >= h->cfg.max_streams) return fail(h, VNECT_E_INVALID, "stream id out of range");
  std::vector<FilterState> st(kJoints * 5);
  for (int i = 0; i < kJoints * 5; ++i) {
    const double* o = state + 7 * i;
    memset(&st[i], 0, sizeof(FilterState));
    st[i].prev = o[0]; st[i].s_x = o[1]; st[i].s_dx = o[2]; st[i].lasttime = o[3]; st[i].freq = o[4];
    st[i].has_prev = o[5] != 0.0; st[i].has_time = o[6] != 0.0;
  }
  if (int rc = quiesce(h)) return rc;
  CU(h, cudaMemcpy(h->d_st2d + (size_t)stream_id * kJoints * 2, st.data(), kJoints * 2 * sizeof(FilterState), cudaMemcpyHostToDevice));
  CU(h, cudaMemcpy(h->d_st3d + (size_t)stream_id * kJoints * 3, st.data() + kJoints * 2, kJoints * 3 * sizeof(FilterState), cudaMemcpyHostToDevice));
  const double* tail = state + 7 * kJoints * 5;
  h->last_t2d[stream_id] = tail[0];
  h->last_t3d[stream_id] = tail[1];
  const int4 b = make_int4((int)tail[2], (int)tail[3], (int)tail[4], (int)tail[5]);
  CU(h, cudaMemcpy(h->d_boxes + stream_id, &b, sizeof b, cudaMemcpyHostToDevice));
  return VNECT_OK;
}

int vnect_set_stream(vnect_t* h, void* cuda_stream) {
  if (!h) return VNECT_E_INVALID;
  ON_DEVICE(h);
  if (h->own_stream && h->stream) {
    cudaStreamSynchronize(h->stream);
    cudaStreamDestroy(h->stream);
  }
  h->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
  h->own_stream = false;
  return VNECT_OK;
}

int vnect_set_packed_results(vnect_t* h, void* dev_packed) {
  if (!h) return VNECT_E_INVALID;
  ON_DEVICE(h);
  CU(h, cudaStreamSynchronize(h->stream));
  for (auto& kv : h->graphs)  // the pointer is baked into the captured post-process launch
    if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  h->graphs.clear();
  h->d_packed = reinterpret_cast<double*>(dev_packed);
  return VNECT_OK;
}

int vnect_synchronize(vnect_t* h) {
  if (!h) return VNECT_E_INVALID;
  ON_DEVICE(h);
  CU(h, cudaStreamSynchronize(h->stream));
  return VNECT_OK;
}

int vnect_get_tap(vnect_t* h, const char* name, int32_t n, float* out_nhwc, int64_t capacity_elems, int32_t* dims4) {
  if (!h || !h->finalized || !name) return fail(h, VNECT_E_INVALID, "handle not finalized");
  ON_DEVICE(h);
  auto it = h->acts.find(name);
  if (it == h->acts.end()) return fail(h, VNECT_E_INVALID, "no activation named '%s'", name);
  const Act& a = it->second;
  if (n < 1 || n > h->cap_fw) return fail(h, VNECT_E_INVALID, "n out of range");
  if (dims4) { dims4[0] = n; dims4[1] = a.H; dims4[2] = a.W; dims4[3] = a.C; }
  const size_t elems = (size_t)n * a.H * a.W * a.C;
  if (!out_nhwc) return VNECT_OK;
  if ((int64_t)elems > capacity_elems) return fail(h, VNECT_E_INVALID, "buffer too small for tap '%s'", name);
  std::vector<__half> tmp((size_t)n * a.img_px * a.C);
  CU(h, cudaStreamSynchronize(h->stream));
  CU(h, cudaMemcpy(tmp.data(), a.p, tmp.size() * sizeof(__half), cudaMemcpyDeviceToHost));
  size_t o = 0;
  for (int i = 0; i < n; ++i)
    for (int y = 0; y < a.H; ++y)
      for (int x = 0; x < a.W; ++x) {
        const __half* src = tmp.data() + ((size_t)i * a.img_px + (size_t)y * a.row_px + x) * a.C;
        for (int c = 0; c < a.C; ++c) out_nhwc[o++] = __half2float(src[c]);
      }
  return VNECT_OK;
}

int vnect_get_input(vnect_t* h, int32_t n, uint16_t* out, int64_t capacity, int32_t* dims4) {
  if (!h || !h->x1) return fail(h, VNECT_E_INVALID, "handle not created");
  ON_DEVICE(h);
  if (n < 1 || n > h->cap_fw) return fail(h, VNECT_E_INVALID, "n out of range");
  if (dims4) { dims4[0] = n; dims4[1] = 2; dims4[2] = h->stem_rpp; dims4[3] = h->stem_pitch; }
  const size_t elems = (size_t)n * 2 * h->stem_rpp * h->stem_pitch;
  if (!out) return VNECT_OK;
  if ((int64_t)elems > capacity) return fail(h, VNECT_E_INVALID, "buffer too small for the network input");
  CU(h, cudaStreamSynchronize(h->stream));
  CU(h, cudaMemcpy(out, h->x1, elems * sizeof(__half), cudaMemcpyDeviceToHost));
  return VNECT_OK;
}

int vnect_get_maps(vnect_t* h, int32_t n_frames, float* out, int64_t capacity, int32_t* dims4) {
  if (!h || !h->maps) return fail(h, VNECT_E_INVALID, "handle not created");
  ON_DEVICE(h);
  if (n_frames < 1 || n_frames > h->cfg.max_frames) return fail(h, VNECT_E_INVALID, "n_frames out of range");
  const int n = n_frames * h->n_scales;
  if (dims4) { dims4[0] = n; dims4[1] = 4 * kJoints; dims4[2] = h->hs; dims4[3] = h->hs; }
  const size_t elems = (size_t)n * 4 * kJoints * h->hs * h->hs;
  if (!out) return VNECT_OK;
  if ((int64_t)elems > capacity) return fail(h, VNECT_E_INVALID, "buffer too small for the maps");
  CU(h, cudaStreamSynchronize(h->stream));
  CU(h, cudaMemcpy(out, h->maps, elems * sizeof(float), cudaMemcpyDeviceToHost));
  return VNECT_OK;
}

// CRC32C (Castagnoli) of a host buffer, slicing-by-4: the checksum TensorFlow checkpoints carry per tensor and per
// index block (vnect_b200/tf_checkpoint.py verifies the 58 MB of weights with it).
uint32_t vnect_crc32c(const void* data, uint64_t n) {
  static uint32_t tab[4][256];
  static bool init = false;
  if (!init) {
    for (uint32_t i = 0; i < 256; ++i) {
      uint32_t c = i;
      for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ 0x82F63B78u : c >> 1;
      tab[0][i] = c;
    }
    for (uint32_t i = 0; i < 256; ++i)
      for (int t = 1; t < 4; ++t) tab[t][i] = (tab[t - 1][i] >> 8) ^ tab[0][tab[t - 1][i] & 0xFF];
    init = true;
  }
  const uint8_t* p = static_cast<const uint8_t*>(data);
  uint32_t c = 0xFFFFFFFFu;
  while (n >= 4) {
    c ^= (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
    c = tab[3][c & 0xFF] ^ tab[2][(c >> 8) & 0xFF] ^ tab[1][(c >> 16) & 0xFF] ^ tab[0][c >> 24];
    p += 4;
    n -= 4;
  }
  while (n--) c = tab[0][(c ^ *p++) & 0xFF] ^ (c >> 8);
  return c ^ 0xFFFFFFFFu;
}

int vnect_check_finite(vnect_t* h, int32_t n, int64_t* counts) {
  if (!h || !h->finalized || !counts) return fail(h, VNECT_E_INVALID, "handle not finalized / null buffer");
  ON_DEVICE(h);
  if (n < 1 || n > h->cap_fw) return fail(h, VNECT_E_INVALID, "n out of range");
  CU(h, cudaStreamSynchronize(h->stream));
  int i = 0;
  for (const Step& st : h->steps) {
    // the activation a step writes carries the step's (first) scope name, fused steps are "a+b" / "a>b"
    std::string name = st.name.substr(0, st.name.find_first_of("+>"));
    if (name == "conv1") name = "pool1";
    auto it = h->acts.find(name);
    if (it == h->acts.end()) {  // block tails write the block's activation (scope without the branch suffix)
      it = h->acts.find(name.substr(0, name.find("_branch")));
    }
    unsigned long long c = 0;
    if (it != h->acts.end()) {
      const Act& a = it->second;
      CU(h, cudaMemsetAsync(h->d_scan, 0, sizeof(unsigned long long), h->stream));
      count_nonfinite_kernel<<<h->num_sms * 4, 256, 0, h->stream>>>(a.p, (size_t)n * a.img_px * a.C, h->d_scan);
      CU(h, cudaGetLastError());
      CU(h, cudaMemcpyAsync(&c, h->d_scan, sizeof c, cudaMemcpyDeviceToHost, h->stream));
      CU(h, cudaStreamSynchronize(h->stream));
    }
    counts[i++] = (int64_t)c;
  }
  return VNECT_OK;
}

int64_t vnect_launch_count(vnect_t* h) { return h ? h->launches : 0; }

const char* vnect_step_name(vnect_t* h, int32_t i) {
  if (!h || i < 0 || i >= (int)h->steps.size()) return nullptr;
  return h->steps[i].name.c_str();
}

int vnect_step_path(vnect_t* h, int32_t i, int32_t* out) {
  if (!h || !h->finalized || !out) return fail(h, VNECT_E_INVALID, "handle not finalized / null buffer");
  if (i < 0 || i >= (int)h->steps.size()) return fail(h, VNECT_E_INVALID, "step %d not in [0, %zu)", i, h->steps.size());
  const Step& st = h->steps[i];
  for (int k = 0; k < 12; ++k) out[k] = 0;
  if (st.kind != 0) {
    out[0] = st.stem_pool.cg;
    out[1] = st.stem_pool.r.n_xt;
    return VNECT_OK;
  }
  const ConvLaunch& L = st.launch;
  const int32_t v[12] = {L.block_n, L.epi, L.cg, L.b_resident, L.halo, L.p.im2col, L.p.mode, L.n2, L.p.tw, L.p.th, L.p.H, L.p.W};
  for (int k = 0; k < 12; ++k) out[k] = v[k];
  return VNECT_OK;
}

double vnect_info(vnect_t* h, const char* key) {
  if (!h || !key) return NAN;
  const std::string k = key;
  if (k == "num_sms") return h->num_sms;
  if (k == "conv_launches_per_forward") return h->conv_steps;
  if (k == "launches_per_forward") return (double)h->steps.size();
  if (k == "gemm_flops_per_forward") {  // executed GEMM work incl. channel / tile padding, per image
    double f = 0;
    for (const Step& st : h->steps)
      if (st.kind == 0) f += st.launch.flops / h->cap_fw;
      else f += 2.0 * (h->S / 2) * (h->S / 2) * 64 * 224;  // conv1 with its K padded to 7 rows x 8 px x 4 ch
    return f;
  }
  if (k == "hm_size") return h->hs;
  if (k == "max_forwards") return h->cap_fw;
  if (k == "cached_graphs") return (double)h->graphs.size();
  return NAN;
}

int vnect_time_forward(vnect_t* h, int32_t n, int32_t reps, float* total_ms, float* per_layer_ms) {
  if (!h || !h->finalized) return fail(h, VNECT_E_INVALID, "handle not finalized");
  ON_DEVICE(h);
  if (n < 1 || n > h->cap_fw || reps < 1) return fail(h, VNECT_E_INVALID, "bad n/reps");
  const int ns = (int)h->steps.size();
  std::vector<cudaEvent_t> ev(ns + 1);
  for (auto& e : ev) CU(h, cudaEventCreate(&e));
  cudaEvent_t e0, e1;
  CU(h, cudaEventCreate(&e0));
  CU(h, cudaEventCreate(&e1));
  int rc = run_forward(h, n);  // warm-up
  if (rc) return rc;
  CU(h, cudaEventRecord(e0, h->stream));
  for (int r = 0; r < reps; ++r)
    if ((rc = run_forward(h, n))) return rc;
  CU(h, cudaEventRecord(e1, h->stream));
  CU(h, cudaEventSynchronize(e1));
  float ms = 0;
  CU(h, cudaEventElapsedTime(&ms, e0, e1));
  if (total_ms) *total_ms = ms / reps;
  if (per_layer_ms) {
    std::vector<double> acc(ns, 0.0);
    for (int r = 0; r < reps; ++r) {
      if ((rc = run_forward(h, n, ev.data()))) return rc;
      CU(h, cudaStreamSynchronize(h->stream));
      for (int i = 0; i < ns; ++i) {
        float t = 0;
        CU(h, cudaEventElapsedTime(&t, ev[i], ev[i + 1]));
        acc[i] += t;
      }
    }
    for (int i = 0; i < ns; ++i) per_layer_ms[i] = (float)(acc[i] / reps);
  }
  for (auto& e : ev) cudaEventDestroy(e);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  return VNECT_OK;
}

int vnect_time_prepost(vnect_t* h, int32_t n_frames, int32_t reps, float* pre_ms, float* post_ms) {
  if (!h || !h->finalized) return fail(h, VNECT_E_INVALID, "handle not finalized");
  ON_DEVICE(h);
  if (n_frames < 1 || n_frames > h->cfg.max_frames || reps < 1) return fail(h, VNECT_E_INVALID, "bad n_frames/reps");
  int rc = lane_acquire(h, 0);
  if (rc) return rc;
  cudaEvent_t e0, e1;
  CU(h, cudaEventCreate(&e0));
  CU(h, cudaEventCreate(&e1));
  const int S = h->S;
  const Geometry g = squarify_geometry(S, S, S);
  double pre = 0, post = 0;
  std::vector<int32_t> ids(n_frames);
  std::vector<double> t2(n_frames), t3(n_frames);
  for (int i = 0; i < n_frames; ++i) ids[i] = i % h->cfg.max_streams;
  for (int r = -1; r < reps; ++r) {  // r = -1: warm-up
    // fresh, strictly increasing timestamps every repetition (the filters divide by the time step)
    double base = 0;
    for (int i = 0; i < n_frames; ++i) {
      const double last = h->last_t2d[ids[i]] == h->last_t2d[ids[i]] ? h->last_t2d[ids[i]] : 1000.0;
      base = std::max(base, last);
    }
    for (int i = 0; i < n_frames; ++i) { t2[i] = base + 0.033; t3[i] = base + 0.037; }
    for (int i = 0; i < n_frames; ++i) h->last_t3d[ids[i]] = NAN;  // 3D clock readings may trail the 2D ones
    if ((rc = stage_frame_meta(h, n_frames, ids.data(), t2.data(), t3.data(), h->stream))) return rc;
    float ms = 0;
    CU(h, cudaEventRecord(e0, h->stream));
    if ((rc = run_preprocess(h, h->cur->d_frames, n_frames, S, S, bgr_source((int64_t)S * 3, (int64_t)S * S * 3), g))) return rc;
    CU(h, cudaEventRecord(e1, h->stream));
    CU(h, cudaEventSynchronize(e1));
    CU(h, cudaEventElapsedTime(&ms, e0, e1));
    if (r >= 0) pre += ms;
    CU(h, cudaEventRecord(e0, h->stream));
    if ((rc = run_postprocess(h, n_frames, g.scaler, g.off_x, g.off_y, h->cur->d_out2d, h->cur->d_out3d, nullptr, false))) return rc;
    CU(h, cudaEventRecord(e1, h->stream));
    CU(h, cudaEventSynchronize(e1));
    CU(h, cudaEventElapsedTime(&ms, e0, e1));
    if (r >= 0) post += ms;
  }
  if (h->d_post_trace) {  // developer diagnostics: where a (frame, joint) block of the last launch spent its time
    const int nb = n_frames * kJoints;
    std::vector<unsigned long long> tr((size_t)nb * 16);
    CU(h, cudaMemcpy(tr.data(), h->d_post_trace, tr.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    unsigned long long t0 = ~0ull, t1 = 0;
    for (int b = 0; b < nb; ++b) { t0 = std::min(t0, tr[(size_t)b * 16]); for (int k = 0; k <= 10; ++k) t1 = std::max(t1, tr[(size_t)b * 16 + k]); }
    static const char* names[] = {"start", "pdl_wait", "staged", "sum pass", "reduced", "marked", "exact+reduce", "2D filter", "gather", "fence+atomic", "tail"};
    fprintf(stderr, "post-process trace (%d blocks, kernel span %.2f us): phase end relative to the block's start, mean / max us; block start spread %.2f us\n",
            nb, (t1 - t0) * 1e-3, 0.0);
    double start_max = 0;
    for (int b = 0; b < nb; ++b) start_max = std::max(start_max, (tr[(size_t)b * 16] - t0) * 1e-3);
    fprintf(stderr, "  last block started %.2f us after the first\n", start_max);
    for (int b = 0; b < nb; ++b)
      if (tr[(size_t)b * 16 + 10] > tr[(size_t)b * 16]) {  // a block that ran the tail: SM cycles per ns over its lifetime
        fprintf(stderr, "  SM clock during the kernel: %.0f MHz\n",
                1e3 * (double)(tr[(size_t)b * 16 + 12] - tr[(size_t)b * 16 + 11]) / (double)(tr[(size_t)b * 16 + 10] - tr[(size_t)b * 16]));
        break;
      }
    {  // survivors per block and the spread of the blocks' own durations (start -> fence + counter)
      std::vector<double> dur;
      std::vector<unsigned long long> nqs;
      for (int b = 0; b < nb; ++b) {
        dur.push_back((tr[(size_t)b * 16 + 9] - tr[(size_t)b * 16]) * 1e-3);
        nqs.push_back(tr[(size_t)b * 16 + 13]);
      }
      std::sort(dur.begin(), dur.end());
      std::sort(nqs.begin(), nqs.end());
      fprintf(stderr, "  block duration p50 %.2f p90 %.2f p99 %.2f max %.2f us; surviving quads per block p50 %llu p90 %llu p99 %llu max %llu\n",
              dur[nb / 2], dur[nb * 9 / 10], dur[nb * 99 / 100], dur[nb - 1], nqs[nb / 2], nqs[nb * 9 / 10], nqs[nb * 99 / 100], nqs[nb - 1]);
    }
    {  // inside "exact+reduce": the exact cells are in shared memory (blocks on the few-quads path only)
      double sum = 0; int cnt = 0;
      for (int b = 0; b < nb; ++b) {
        const unsigned long long v = tr[(size_t)b * 16 + 14], s0 = tr[(size_t)b * 16 + 5];
        if (v >= s0 && v <= t1) { sum += (v - s0) * 1e-3; ++cnt; }
      }
      fprintf(stderr, "  exact cells ready %.2f us after the marking barrier (%d blocks)\n", cnt ? sum / cnt : 0.0, cnt);
    }
    for (int k = 1; k <= 10; ++k) {
      double sum = 0, mx = 0; int cnt = 0;
      for (int b = 0; b < nb; ++b) {
        const unsigned long long v = tr[(size_t)b * 16 + k], s0 = tr[(size_t)b * 16];
        if (v < s0 || v > t1) continue;  // stale slot (tail runs in one block per frame)
        if (k == 10 && v < tr[(size_t)b * 16 + 9]) continue;
        sum += (v - s0) * 1e-3; mx = std::max(mx, (v - s0) * 1e-3); ++cnt;
      }
      fprintf(stderr, "  %-14s %7.2f / %7.2f us  (%d blocks)\n", names[k], cnt ? sum / cnt : 0.0, mx, cnt);
    }
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (pre_ms) *pre_ms = (float)(pre / reps);
  if (post_ms) *post_ms = (float)(post / reps);
  return VNECT_OK;
}

void vnect_destroy(vnect_t* h) {
  if (!h) return;
  ON_DEVICE(h);
  if (h->copy_stream) cudaStreamSynchronize(h->copy_stream);
  if (h->stream) cudaStreamSynchronize(h->stream);
  for (auto& kv : h->graphs)
    if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  for (void* p : h->allocs) cudaFree(p);
  for (auto& L : h->lanes) {
    if (L.h_meta) cudaFreeHost(L.h_meta);
    if (L.h_nonfinite) cudaFreeHost(L.h_nonfinite);
    if (L.copy_done) cudaEventDestroy(L.copy_done);
    if (L.done) cudaEventDestroy(L.done);
  }
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

}  // extern "C"
