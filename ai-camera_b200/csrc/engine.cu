// Engine: loads a flat ".aicw" weight blob and runs YOLOv8 detect or the DeepSORT ReID net as
// a static list of kernel launches over preallocated NHWC bf16 buffers.
//
// Replaces the TensorRT engine object of the reference
// (/root/reference/src/trt_utils/trt_engine.py: _init_engine :45-60 -> engine_create,
//  infer :151-203 -> yolo_forward / reid_forward).  Architectures are the named public ones
// (SURVEY.md Appendix D); the reference itself holds no network definition.
//
// Data layout in HBM: every activation is NHWC bf16, [max_batch][H][W][C].  Concatenations
// (C2f, SPPF, the FPN/PAN joins) are never materialised by a copy: producers write straight
// into channel slices of the wider buffer (conv out_coff/out_cstride), and consumers read a
// slice (in_coff/in_cstride).
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <vector>

#include "conv_chain.cuh"
#include "conv_tc.cuh"
#include "frame_table.cuh"
#include "layers.cuh"
#include "stem_pool.cuh"

namespace aicam {

bool profile_enabled();
int nms_impl(const float* boxes, const float* scores, const int32_t* labels, int batch, int anchors, const aicam_nms_params* p,
             int32_t* num_dets, float* boxes_lb, float* boxes_orig, float* out_scores, int32_t* out_labels, int32_t* keep_index,
             void* workspace, size_t workspace_bytes, void* stream, const FrameRec* recs);
int decode_nms_impl(const float* head, int batch, int anchors, int nc, const aicam_nms_params* p, int32_t* num_dets,
                    float* boxes_lb, float* boxes_orig, float* scores, int32_t* labels, void* workspace,
                    size_t workspace_bytes, void* stream, const FrameRec* recs);

namespace {

struct BlobTensor {
  std::vector<int> dims;
  const float* data;
  size_t count;
};

struct Buffer {
  __nv_bfloat16* ptr;
  int h, w, c;
  int pad = 0;  // border kind (conv_tc.cuh): 1: stored [batch][h + 2][w + 2][c], 2: [batch][h + 1][w + 1][c] (shared border);
                // the border is zero and no kernel ever writes anything but zeros there
};

struct View {
  int buf = -1;        // index into buffers; -1 = external input, -2 = external output
  int coff = 0;        // first channel
  long long eoff = 0;  // extra element offset (Detect levels inside the head tensor)
};

// A run of consecutive CONV ops that conv_chain.cu can execute as ONE launch (the op list keeps the single layers
// right behind the CHAIN op: they run when the chain kernel declines the geometry or is switched off)
struct ChainOp {
  int nstages = 0;
  int conv[CHAIN_MAX_STAGES];  // indices into the engine's convs
  int act[CHAIN_MAX_STAGES];
  int nsrc[CHAIN_MAX_STAGES];
  int src_buf[CHAIN_MAX_STAGES][2], src_coff[CHAIN_MAX_STAGES][2], src_c[CHAIN_MAX_STAGES][2];
  int res_buf[CHAIN_MAX_STAGES], res_coff[CHAIN_MAX_STAGES], res_mode[CHAIN_MAX_STAGES];
  int in_c = 0;   // channels of the input view loaded as buffer 0
  int covers = 0; // CONV ops that follow and are skipped when the chain has been launched
};

struct Op {
  enum Type { CONV, MAXPOOL, UPSAMPLE, AVGL2, STEMPOOL, SPPF3, CHAIN } type;
  int chain = -1;
  int conv = -1;
  View in, out, res;
  int h = 0, w = 0, c = 0;  // input spatial size / channels moved (pool, upsample)
  int k = 0, stride = 1;
  int act = 0, res_mode = 0, out_f32 = 0;
  int s2d_c0 = 0;   // conv reads its input space-to-depth (h, w are the space-to-depth sizes), c0 channels per pixel
  int out_s2d = 0;  // conv stores its output space-to-depth (for the next stride-2 layer)
  int only_fmt = 0; // 0: always; 2: only when the input is NOT format 3; 3: only when the input is format 3 (the two stems of yolov8n)
  int lane = 0;     // 0: the caller's stream; 1, 2: the engine's side streams (independent tail chains, joined at the end)
};

}  // namespace

}  // namespace aicam

struct aicam_engine {
  int kind = 0, device = 0, max_batch = 0;
  uint32_t params[8] = {0};
  std::vector<aicam::PackedConv> convs;
  aicam::StemPool stem;            // reid: fused conv.0 + ReLU + maxpool
  int stem_in8 = -1;               // reid: NHWC8 copy of the input crops
  int s2d_in = -1;                 // yolov8: space-to-depth copy of an NHWC4 input (callers may pass it directly)
  int stem4 = -1;                  // yolov8n: index (in convs) of the stem re-expressed over 4x4 pixel blocks (input format 3), or -1
  std::map<std::string, int> conv_by_name;
  std::vector<aicam::Buffer> buffers;
  std::vector<aicam::Op> ops;
  std::vector<aicam::ChainOp> chains;
  double macs_per_item = 0.0;
  // external tensor geometry
  int in_h = 0, in_w = 0;
  int out_cstride = 0;         // yolov8: 64 + nc
  long long out_img_stride = 0;
  int num_anchors = 0;
  int feat_buf = -1;           // reid: buffer feeding the average pool
  // The six chains of the Detect head (3 levels x {box, class}) are independent of each other: they run on the
  // caller's stream and two side streams, forked after the neck and joined before run_ops returns, so that the
  // small late layers fill each other's launch gaps and idle SMs (also inside a CUDA-graph capture).
  cudaStream_t side[2] = {nullptr, nullptr};
  cudaEvent_t ev_fork = nullptr, ev_join[2] = {nullptr, nullptr};
};

namespace aicam {

namespace {

// channels per pixel of the dense input when a layer qualifies for the space-to-depth window path, else 0
int s2d_channels(int k, int s, int cin, int in_cstride) {
  static const bool off = getenv("AICAM_NO_S2D") != nullptr;
  if (off || k != 3 || s != 2) return 0;
  if (cin <= 4 && in_cstride == 4) return 4;
  if (cin == 16 && in_cstride == 16) return 16;
  return 0;
}

struct Builder {
  aicam_engine* e;
  std::map<std::string, BlobTensor>* tensors;
  int err = AICAM_OK;

  int buf(int h, int w, int c, int pad = 0) {
    Buffer b{nullptr, h, w, c, pad};
    const size_t bytes = static_cast<size_t>(e->max_batch) * (h + pad_ext(pad)) * (w + pad_ext(pad)) * c * sizeof(__nv_bfloat16);
    if (cudaMalloc(&b.ptr, bytes) != cudaSuccess) {
      err = fail(AICAM_ERR_CUDA, "engine: cudaMalloc of an activation buffer failed");
      b.ptr = nullptr;
    } else {
      cudaMemset(b.ptr, 0, bytes);
    }
    e->buffers.push_back(b);
    return static_cast<int>(e->buffers.size()) - 1;
  }

  int conv(const std::string& name, View in, int h, int w, View out, int cin, int cout, int k, int s, int act,
           View res = View(), int res_mode = 0, int out_f32 = 0) {
    if (err) return err;
    auto wi = tensors->find(name + ".weight");
    auto bi = tensors->find(name + ".bias");
    if (wi == tensors->end() || bi == tensors->end())
      return err = fail(AICAM_ERR_IO, "engine: blob has no tensor " + name + ".weight/.bias");
    const BlobTensor& wt = wi->second;
    if (wt.dims.size() != 4 || wt.dims[0] != cout || wt.dims[1] != cin || wt.dims[2] != k || wt.dims[3] != k ||
        static_cast<int>(bi->second.count) != cout)
      return err = fail(AICAM_ERR_IO, "engine: tensor " + name + " has an unexpected shape");
    PackedConv pc;
    if (int rc = pack_conv_weights(wt.data, bi->second.data, cout, cin, k, s, &pc)) return err = rc;
    e->convs.push_back(pc);
    e->conv_by_name[name] = static_cast<int>(e->convs.size()) - 1;
    Op op;
    op.type = Op::CONV;
    op.conv = static_cast<int>(e->convs.size()) - 1;
    op.in = in; op.out = out; op.res = res;
    op.h = h; op.w = w; op.k = k; op.stride = s;
    op.act = act; op.res_mode = res_mode; op.out_f32 = out_f32;
    e->ops.push_back(op);
    const int ho = (h + 2 * (k / 2) - k) / s + 1, wo = (w + 2 * (k / 2) - k) / s + 1;
    e->macs_per_item += static_cast<double>(ho) * wo * cout * cin * k * k;
    return AICAM_OK;
  }

  // 3x3 stride-2 layer over a space-to-depth input of (h2 x w2) 2x2 blocks with c0 channels per pixel
  // The yolov8n stem once more space-to-depth: the 3x3 stride-2 layer over the 640 grid is a 2x2 window over the 320 grid of
  // 2x2 blocks (format 2, 16 channels); computing the 2x2 OUTPUT pixels of an output block together makes it a 3x3
  // stride-2 layer over that 320 grid with 16 input and 4 x 16 output channels [(oy, ox)][co] - exactly the layer type
  // pack_conv_weights_s2d packs (model.1), now reading 4x4 pixel blocks of 64 channels (format 3) and storing plain 64-channel
  // pixels = the space-to-depth tensor model.1 reads.  Why: a 16-channel pixel is a 32-byte TMA request and the window kernel
  // is bound by the request rate there (6.5 M loads + 3.3 M stores per 64 frames); 64-channel blocks need a quarter of them.
  int stem_4x4(const std::string& name, View in, int h4, int w4, View out, int c1) {
    if (err) return err;
    auto wi = tensors->find(name + ".weight");
    auto bi = tensors->find(name + ".bias");
    if (wi == tensors->end() || bi == tensors->end()) return err = fail(AICAM_ERR_IO, "engine: blob has no tensor " + name);
    const float* w = wi->second.data;  // [c1][3][3][3]
    const int cout = 4 * c1;
    std::vector<float> w2(static_cast<size_t>(cout) * 16 * 9, 0.0f), b2(cout);
    // image row 4Y + 2 oy + dy - 1 = 2 u + py with u = 2Y + e - 1 (e: tap of the 320-grid layer), py: row parity inside the block
    for (int oy = 0; oy < 2; ++oy)
      for (int ox = 0; ox < 2; ++ox)
        for (int co = 0; co < c1; ++co) {
          const int o = (oy * 2 + ox) * c1 + co;
          b2[o] = bi->second.data[co];
          for (int dy = 0; dy < 3; ++dy)
            for (int dx = 0; dx < 3; ++dx) {
              const int ry = 2 * oy + dy - 1, rx = 2 * ox + dx - 1;  // -1 .. 3
              const int e = (ry + 2) / 2, f = (rx + 2) / 2;           // floor(r / 2) + 1
              const int py = (ry + 2) & 1, px = (rx + 2) & 1;
              for (int c = 0; c < 3; ++c)
                w2[(static_cast<size_t>(o) * 16 + (py * 2 + px) * 4 + c) * 9 + e * 3 + f] = w[(static_cast<size_t>(co) * 3 + c) * 9 + dy * 3 + dx];
            }
        }
    PackedConv pc;
    if (int rc = pack_conv_weights_s2d(w2.data(), b2.data(), cout, 16, 16, &pc)) return err = rc;
    e->convs.push_back(pc);
    e->stem4 = static_cast<int>(e->convs.size()) - 1;
    Op op;
    op.type = Op::CONV;
    op.conv = e->stem4;
    op.in = in; op.out = out;
    op.h = h4; op.w = w4; op.k = 2; op.stride = 1;
    op.act = 1; op.s2d_c0 = 16; op.out_s2d = 0; op.only_fmt = 3;
    e->ops.push_back(op);
    return AICAM_OK;
  }

  int conv_s2d(const std::string& name, View in, int h2, int w2, View out, int cin, int cout, int c0, int act, int out_s2d) {
    if (err) return err;
    auto wi = tensors->find(name + ".weight");
    auto bi = tensors->find(name + ".bias");
    if (wi == tensors->end() || bi == tensors->end())
      return err = fail(AICAM_ERR_IO, "engine: blob has no tensor " + name + ".weight/.bias");
    const BlobTensor& wt = wi->second;
    if (wt.dims.size() != 4 || wt.dims[0] != cout || wt.dims[1] != cin || wt.dims[2] != 3 || wt.dims[3] != 3 ||
        static_cast<int>(bi->second.count) != cout)
      return err = fail(AICAM_ERR_IO, "engine: tensor " + name + " has an unexpected shape");
    PackedConv pc;
    if (int rc = pack_conv_weights_s2d(wt.data, bi->second.data, cout, cin, c0, &pc)) return err = rc;
    e->convs.push_back(pc);
    e->conv_by_name[name] = static_cast<int>(e->convs.size()) - 1;
    Op op;
    op.type = Op::CONV;
    op.conv = static_cast<int>(e->convs.size()) - 1;
    op.in = in; op.out = out;
    op.h = h2; op.w = w2; op.k = 2; op.stride = 1;
    op.act = act; op.s2d_c0 = c0; op.out_s2d = out_s2d;
    e->ops.push_back(op);
    e->macs_per_item += static_cast<double>(h2) * w2 * cout * cin * 9;
    return AICAM_OK;
  }

  void pool(View in, View out, int h, int w, int c, int k, int s) {
    Op op; op.type = Op::MAXPOOL; op.in = in; op.out = out; op.h = h; op.w = w; op.c = c; op.k = k; op.stride = s;
    e->ops.push_back(op);
  }
  void upsample(View in, View out, int h, int w, int c) {
    Op op; op.type = Op::UPSAMPLE; op.in = in; op.out = out; op.h = h; op.w = w; op.c = c;
    e->ops.push_back(op);
  }

  static View V(int b, int coff = 0, long long eoff = 0) { View v; v.buf = b; v.coff = coff; v.eoff = eoff; return v; }

  // ---- fused chains (conv_chain.cu).  begin_chain() goes BEFORE the conv() calls of the layers it covers; stage() names
  // each of them in order with its sources (buffer 0 = the chain's input view, i = the output of stage i - 1)
  // Measured on B200 (profiles/r2_chain_bench.txt): the fused kernel is bit-for-bit as good as the single layers but NOT
  // faster - halo recomputation in shared-memory-limited tiles costs more tensor-pipe time than the launches it saves -
  // so the engines keep the single layers unless AICAM_CHAIN=1 asks for the chains (AICAM_CHAIN=pair,head,tail,full
  // picks kinds).
  static bool chains_enabled(const char* what) {
    const char* on = getenv("AICAM_CHAIN");
    if (on == nullptr || on[0] == '0') return false;
    return on[0] == '1' || strstr(on, what) != nullptr;
  }
  int begin_chain(View in, int in_c, View out, int h, int w, int out_f32) {
    Op op; op.type = Op::CHAIN; op.in = in; op.out = out; op.h = h; op.w = w; op.out_f32 = out_f32;
    ChainOp c; c.in_c = in_c;
    e->chains.push_back(c);
    op.chain = static_cast<int>(e->chains.size()) - 1;
    e->ops.push_back(op);
    return op.chain;
  }
  void chain_stage(int chain, const std::string& conv_name, int act, int b0, int coff0, int c0, int b1 = -1, int coff1 = 0, int c1 = 0,
                   int res_buf = -1, int res_coff = 0, int res_mode = 0) {
    if (err) return;
    ChainOp& c = e->chains[chain];
    const int s = c.nstages++;
    c.conv[s] = e->conv_by_name[conv_name];
    c.act[s] = act;
    c.nsrc[s] = b1 >= 0 ? 2 : 1;
    c.src_buf[s][0] = b0; c.src_coff[s][0] = coff0; c.src_c[s][0] = c0;
    c.src_buf[s][1] = std::max(b1, 0); c.src_coff[s][1] = coff1; c.src_c[s][1] = c1;
    c.res_buf[s] = res_buf; c.res_coff[s] = res_coff; c.res_mode[s] = res_mode;
    c.covers = c.nstages;
  }

  // Ultralytics C2f: cv1 -> split -> n chained Bottlenecks (3x3, 3x3, optional shortcut) -> cv2 on the concat
  void c2f(const std::string& name, View in, int cin, View out, int cout, int n, bool shortcut, int h, int w) {
    const int c = cout / 2;
    const int cat = buf(h, w, (2 + n) * c);
    const int tmp = buf(h, w, c);
    const std::string m0 = name + ".m.0", ml = name + ".m." + std::to_string(n - 1);
    // Fusion plan (conv_chain.cu): narrow blocks (c <= 32) keep everything after cv1 - or, with few input channels, the
    // whole block - in shared memory; wide blocks fuse each Bottleneck pair only (their operands fill shared memory)
    const bool full = n == 1 && c <= 16 && cin <= 32 && c % 16 == 0 && chains_enabled("full");
    const bool tail = !full && c <= 32 && c % 16 == 0 && chains_enabled("tail");
    const bool pairs = c % 16 == 0 && chains_enabled("pair");
    int ch_full = -1;
    if (full) ch_full = begin_chain(in, cin, out, h, w, 0);
    conv(name + ".cv1.conv", in, h, w, V(cat, 0), cin, 2 * c, 1, 1, 1);
    int ch_tail = -1;
    for (int j = 0; j < n; ++j) {
      const std::string m = name + ".m." + std::to_string(j);
      int ch_pair = -1;
      if (!full) {
        if (tail && j == n - 1) ch_tail = begin_chain(V(cat, 0), (2 + j) * c, out, h, w, 0);
        else if (pairs) ch_pair = begin_chain(V(cat, (1 + j) * c), c, V(cat, (2 + j) * c), h, w, 0);
      }
      conv(m + ".cv1.conv", V(cat, (1 + j) * c), h, w, V(tmp, 0), c, c, 3, 1, 1);
      conv(m + ".cv2.conv", V(tmp, 0), h, w, V(cat, (2 + j) * c), c, c, 3, 1, 1,
           shortcut ? V(cat, (1 + j) * c) : View(), shortcut ? 1 : 0);
      if (ch_pair >= 0) {
        chain_stage(ch_pair, m + ".cv1.conv", 1, 0, 0, c);
        chain_stage(ch_pair, m + ".cv2.conv", 1, 1, 0, c, -1, 0, 0, shortcut ? 0 : -1, 0, shortcut ? 1 : 0);
      }
    }
    conv(name + ".cv2.conv", V(cat, 0), h, w, out, (2 + n) * c, cout, 1, 1, 1);
    if (ch_full >= 0) {
      chain_stage(ch_full, name + ".cv1.conv", 1, 0, 0, cin);
      chain_stage(ch_full, m0 + ".cv1.conv", 1, 1, c, c);
      chain_stage(ch_full, m0 + ".cv2.conv", 1, 2, 0, c, -1, 0, 0, shortcut ? 1 : -1, c, shortcut ? 1 : 0);
      chain_stage(ch_full, name + ".cv2.conv", 1, 1, 0, 2 * c, 3, 0, c);
    }
    if (ch_tail >= 0) {  // buffer 0 = the concatenation so far: [cv1 out (2c) | m.0 .. m.(n-2) outputs]
      chain_stage(ch_tail, ml + ".cv1.conv", 1, 0, n * c, c);
      chain_stage(ch_tail, ml + ".cv2.conv", 1, 1, 0, c, -1, 0, 0, shortcut ? 0 : -1, n * c, shortcut ? 1 : 0);
      chain_stage(ch_tail, name + ".cv2.conv", 1, 0, 0, (1 + n) * c, 2, 0, c);
    }
  }

  void build_yolov8() {
    const int c1 = e->params[0], c2 = e->params[1], c3 = e->params[2], c4 = e->params[3], c5 = e->params[4];
    const int ns = e->params[5], nl = e->params[6], nc = e->params[7];
    const int cb = std::max(16, std::max(c3 / 4, 64));
    const int cc = std::max(c3, std::min(nc, 100));
    const int S = AICAM_YOLO_INPUT;
    e->in_h = e->in_w = S;
    const int h2 = S / 2, h4 = S / 4, h8 = S / 8, h16 = S / 16, h32 = S / 32;
    e->num_anchors = h8 * h8 + h16 * h16 + h32 * h32;
    e->out_cstride = AICAM_HEAD_DFL + nc;
    e->out_img_stride = static_cast<long long>(e->num_anchors) * e->out_cstride;

    const int a0 = buf(h2, h2, c1), a1 = buf(h4, h4, c2), a2 = buf(h4, h4, c2), a3 = buf(h8, h8, c3);
    const int cat14 = buf(h8, h8, c4 + c3);    // [up(n12) | P3]
    const int a5 = buf(h16, h16, c4);
    const int cat11 = buf(h16, h16, c5 + c4);  // [up(P5) | P4]
    const int a7 = buf(h32, h32, c5), a8 = buf(h32, h32, c5);
    const int cats = buf(h32, h32, 2 * c5);    // SPPF concat: 4 x c5/2
    const int cat20 = buf(h32, h32, c4 + c5);  // [conv19(o4) | P5]
    const int cat17 = buf(h16, h16, c3 + c4);  // [conv16(o3) | n12]
    const int o3 = buf(h8, h8, c3), o4 = buf(h16, h16, c4), o5 = buf(h32, h32, c5);

    // The two stride-2 layers at full resolution run as 2x2 windows over space-to-depth tensors: the input
    // arrives (or is repacked) as [S/2][S/2][2x2][RGB0], the stem stores its output as [S/4][S/4][2x2][c1].
    const bool s2d0 = s2d_channels(3, 2, 3, 4) != 0;
    const bool s2d1 = s2d0 && c1 == 16 && s2d_channels(3, 2, c1, c1) != 0;
    if (s2d0) {
      e->s2d_in = buf(h2, h2, 16);
      conv_s2d("model.0.conv", V(-1), h2, h2, V(a0), 3, c1, 4, 1, s2d1 ? 1 : 0);
      static const bool no_stem4 = getenv("AICAM_NO_STEM4") != nullptr;
      if (s2d1 && !no_stem4) {  // the same layer over format-3 input; run_ops picks one of the two by the input's format
        e->ops.back().only_fmt = 2;
        stem_4x4("model.0.conv", V(-1), h4, h4, V(a0), c1);
      }
    } else {
      conv("model.0.conv", V(-1), S, S, V(a0), 3, c1, 3, 2, 1);
    }
    if (s2d1) conv_s2d("model.1.conv", V(a0), h4, h4, V(a1), c1, c2, 16, 1, 0);
    else conv("model.1.conv", V(a0), h2, h2, V(a1), c1, c2, 3, 2, 1);
    c2f("model.2", V(a1), c2, V(a2), c2, ns, true, h4, h4);
    conv("model.3.conv", V(a2), h4, h4, V(a3), c2, c3, 3, 2, 1);
    c2f("model.4", V(a3), c3, V(cat14, c4), c3, nl, true, h8, h8);
    conv("model.5.conv", V(cat14, c4), h8, h8, V(a5), c3, c4, 3, 2, 1);
    c2f("model.6", V(a5), c4, V(cat11, c5), c4, nl, true, h16, h16);
    conv("model.7.conv", V(cat11, c5), h16, h16, V(a7), c4, c5, 3, 2, 1);
    c2f("model.8", V(a7), c5, V(a8), c5, ns, true, h32, h32);
    // SPPF
    const int hc = c5 / 2;
    conv("model.9.cv1.conv", V(a8), h32, h32, V(cats, 0), c5, hc, 1, 1, 1);
    {  // three chained 5x5 pools: one fused launch when eligible (layers.cu), else three max-pool launches
      Op op; op.type = Op::SPPF3; op.in = V(cats, 0); op.out = V(cats, hc); op.h = h32; op.w = h32; op.c = hc; op.k = 5; op.stride = 1;
      e->ops.push_back(op);
    }
    conv("model.9.cv2.conv", V(cats, 0), h32, h32, V(cat20, c4), 4 * hc, c5, 1, 1, 1);
    // FPN top-down
    upsample(V(cat20, c4), V(cat11, 0), h32, h32, c5);
    c2f("model.12", V(cat11, 0), c5 + c4, V(cat17, c3), c4, ns, false, h16, h16);
    upsample(V(cat17, c3), V(cat14, 0), h16, h16, c4);
    c2f("model.15", V(cat14, 0), c4 + c3, V(o3), c3, ns, false, h8, h8);
    // PAN bottom-up
    conv("model.16.conv", V(o3), h8, h8, V(cat17, 0), c3, c3, 3, 2, 1);
    c2f("model.18", V(cat17, 0), c3 + c4, V(o4), c4, ns, false, h16, h16);
    conv("model.19.conv", V(o4), h16, h16, V(cat20, 0), c4, c4, 3, 2, 1);
    c2f("model.21", V(cat20, 0), c4 + c5, V(o5), c5, ns, false, h32, h32);
    // Detect
    const int lvl_in[3] = {o3, o4, o5};
    const int lvl_c[3] = {c3, c4, c5};
    const int lvl_h[3] = {h8, h16, h32};
    long long anchor_base = 0;
    // opt-in: measured on B200 the persistent one-CTA-per-SM kernels of different chains only delay each other
    // (5.68 ms per step on one stream, 5.74 with three)
    static const bool no_lanes = getenv("AICAM_HEAD_STREAMS") == nullptr;
    int chain = 0;
    auto set_lane = [&](size_t first_op, int lane) {
      for (size_t i = first_op; i < e->ops.size(); ++i) e->ops[i].lane = no_lanes ? 0 : lane;
    };
    for (int l = 0; l < 3; ++l) {
      const int hh = lvl_h[l];
      const int b1 = buf(hh, hh, cb), b2 = buf(hh, hh, cb), k1 = buf(hh, hh, cc), k2 = buf(hh, hh, cc);
      const std::string p2 = "model.22.cv2." + std::to_string(l), p3 = "model.22.cv3." + std::to_string(l);
      const long long eoff = anchor_base * e->out_cstride;
      // each branch (3x3 -> 3x3 -> 1x1 into the fp32 head tensor) is one fused launch when conv_chain.cu takes it
      const bool fuse = no_lanes && chains_enabled("head");
      size_t first = e->ops.size();
      const int ch2 = fuse && cb % 16 == 0 ? begin_chain(V(lvl_in[l]), lvl_c[l], V(-2, 0, eoff), hh, hh, 1) : -1;
      conv(p2 + ".0.conv", V(lvl_in[l]), hh, hh, V(b1), lvl_c[l], cb, 3, 1, 1);
      conv(p2 + ".1.conv", V(b1), hh, hh, V(b2), cb, cb, 3, 1, 1);
      conv(p2 + ".2", V(b2), hh, hh, V(-2, 0, eoff), cb, AICAM_HEAD_DFL, 1, 1, 0, View(), 0, 1);
      if (ch2 >= 0) {
        chain_stage(ch2, p2 + ".0.conv", 1, 0, 0, lvl_c[l]);
        chain_stage(ch2, p2 + ".1.conv", 1, 1, 0, cb);
        chain_stage(ch2, p2 + ".2", 0, 2, 0, cb);
      }
      set_lane(first, chain++ % 3);
      first = e->ops.size();
      const int ch3 = fuse && cc % 16 == 0 && nc % 16 == 0 ? begin_chain(V(lvl_in[l]), lvl_c[l], V(-2, AICAM_HEAD_DFL, eoff), hh, hh, 1) : -1;
      conv(p3 + ".0.conv", V(lvl_in[l]), hh, hh, V(k1), lvl_c[l], cc, 3, 1, 1);
      conv(p3 + ".1.conv", V(k1), hh, hh, V(k2), cc, cc, 3, 1, 1);
      conv(p3 + ".2", V(k2), hh, hh, V(-2, AICAM_HEAD_DFL, eoff), cc, nc, 1, 1, 0, View(), 0, 1);
      if (ch3 >= 0) {
        chain_stage(ch3, p3 + ".0.conv", 1, 0, 0, lvl_c[l]);
        chain_stage(ch3, p3 + ".1.conv", 1, 1, 0, cc);
        chain_stage(ch3, p3 + ".2", 0, 2, 0, cc);
      }
      set_lane(first, chain++ % 3);
      anchor_base += static_cast<long long>(hh) * hh;
    }
  }

  void build_reid() {
    const int H = AICAM_REID_H, W = AICAM_REID_W;
    e->in_h = H; e->in_w = W;
    int h = H / 2, w = W / 2, c = 64;
    int cur = -1, pad1 = 0;
    static const bool unfused = getenv("AICAM_NO_STEM_FUSION") != nullptr;
    static const bool no_pad = getenv("AICAM_NO_PADDED_REID") != nullptr;
    static const bool no_pad1 = getenv("AICAM_NO_PADDED_L1") != nullptr;
    // border kind of the trunk's activations: 2 = shared border (default), 1 = symmetric border (AICAM_REID_PAD=1)
    static const int pad_kind = getenv("AICAM_REID_PAD") ? std::max(1, std::min(2, atoi(getenv("AICAM_REID_PAD")))) : 2;
    auto wi = tensors->find("conv.0.weight");
    auto bi = tensors->find("conv.0.bias");
    if (!unfused && wi != tensors->end() && bi != tensors->end() && wi->second.dims.size() == 4 && wi->second.dims[0] == 64 &&
        wi->second.dims[1] == 3 && wi->second.dims[2] == 3 && static_cast<int>(bi->second.count) == 64) {
      pad1 = (no_pad || no_pad1) ? 0 : pad_kind;  // the fused stem writes the zero-bordered layout directly
      cur = buf(h, w, c, pad1);
      // fused stem: crops NHWC4 -> NHWC8 -> conv3x3 + ReLU + maxpool 3x3 s2 in one kernel (stem_pool.cu)
      if (int rc = pack_stem_pool(wi->second.data, bi->second.data, 64, 3, &e->stem)) { err = rc; return; }
      e->stem_in8 = buf(H, W, 8);
      Op op; op.type = Op::STEMPOOL; op.in = V(-1); op.out = V(cur); op.h = H; op.w = W;
      e->ops.push_back(op);
      e->macs_per_item += static_cast<double>(H) * W * 64 * 3 * 9;
    } else {
      cur = buf(h, w, c);
      const int s0 = buf(H, W, 64);
      conv("conv.0", V(-1), H, W, V(s0), 3, 64, 3, 1, 2);
      pool(V(s0), V(cur), H, W, 64, 3, 2);
    }
    const int widths[4] = {64, 128, 256, 512};
    for (int li = 0; li < 4; ++li) {
      const int cout = widths[li];
      for (int b = 0; b < 2; ++b) {
        const std::string name = "layer" + std::to_string(li + 1) + "." + std::to_string(b);
        const int s = (li > 0 && b == 0) ? 2 : 1;
        const int ho = h / s, wo = w / s;
        // layers 2-4 live in zero-bordered buffers: their 3x3 stride-1 convolutions run over the flat padded
        // raster (conv_win.cu, operand mode 4) instead of nine im2col loads per tile on these small maps
        const int pd = li > 0 ? (no_pad ? 0 : pad_kind) : pad1;
        const int t = buf(ho, wo, cout, pd), o = buf(ho, wo, cout, pd);
        conv(name + ".conv1", V(cur), h, w, V(t), c, cout, 3, s, 2);
        int resbuf = cur;
        if (tensors->count(name + ".downsample.0.weight")) {
          resbuf = buf(ho, wo, cout, pd);
          conv(name + ".downsample.0", V(cur), h, w, V(resbuf), c, cout, 1, s, 0);
        }
        conv(name + ".conv2", V(t), ho, wo, V(o), cout, cout, 3, 1, 2, V(resbuf), 2);
        if (pd && !err) {  // zero-bordered 3x3 stride-1 layers with 64 / 128 channels run on CTA pairs (conv_pair.cu)
          if (s == 1) pack_pair_weights(&e->convs[e->conv_by_name[name + ".conv1"]]);
          pack_pair_weights(&e->convs[e->conv_by_name[name + ".conv2"]]);
        }
        cur = o; h = ho; w = wo; c = cout;
      }
    }
    e->feat_buf = cur;
    e->out_cstride = c;
    Op op; op.type = Op::AVGL2; op.in = V(cur); op.h = h; op.w = w; op.c = c;
    e->ops.push_back(op);
  }
};

// Dense per-anchor arrays of the fused Detect decode (aicam_yolo_detect): when given, the six 1x1 head layers decode their
// rows in the epilogue and the fp32 head tensor is never written
struct DecodeTarget {
  float* boxes;
  float* scores;
  int* labels;
};

int run_ops(aicam_engine* e, const void* input, int batch, void* output, cudaStream_t stream,
            const int* n_dev = nullptr, int input_is_s2d = 0, const DecodeTarget* dec = nullptr) {
  // input_is_s2d: 0: NHWC4 (yolov8) / NHWC4 crops (reid); 1: the engine's space-to-depth / NHWC8 input format; 2: yolov8n,
  // 4x4 pixel blocks (aicam_preprocess format 3)
  if (input_is_s2d == 2 && e->stem4 < 0) return fail(AICAM_ERR_UNSUPPORTED, "engine: this engine has no 4x4-block stem (input format 3)");
  const void* input_s2d = input;
  if (e->s2d_in >= 0 && !input_is_s2d) {
    __nv_bfloat16* dst = e->buffers[e->s2d_in].ptr;
    if (int rc = launch_space_to_depth(static_cast<const __nv_bfloat16*>(input), batch, e->in_h, e->in_w, 4, dst, stream, n_dev)) return rc;
    input_s2d = dst;
  } else if (e->s2d_in < 0 && input_is_s2d && e->kind == AICAM_KIND_YOLOV8) {
    return fail(AICAM_ERR_UNSUPPORTED, "engine: this engine was built without the space-to-depth stem");
  } else if (e->kind == AICAM_KIND_REID && input_is_s2d && e->stem_in8 < 0) {
    return fail(AICAM_ERR_UNSUPPORTED, "engine: this engine was built without the fused NHWC8 stem");
  }
  cudaStream_t main_stream = stream;
  bool forked = false, used[2] = {false, false};
  auto join = [&]() -> int {
    for (int i = 0; i < 2; ++i)
      if (used[i]) {
        AICAM_CUDA_OK(cudaEventRecord(e->ev_join[i], e->side[i]));
        AICAM_CUDA_OK(cudaStreamWaitEvent(main_stream, e->ev_join[i], 0));
      }
    return AICAM_OK;
  };
  int skip = 0;  // single-layer ops covered by a chain that has just been launched
  for (const Op& op : e->ops) {
    if (skip > 0) { --skip; continue; }
    if (op.only_fmt == 3 && input_is_s2d != 2) continue;
    if (op.only_fmt == 2 && input_is_s2d == 2) continue;
    stream = main_stream;
    if (op.lane > 0 && e->side[op.lane - 1] && !profile_enabled()) {  // (per-launch timing: one kernel at a time)
      if (!forked) {
        AICAM_CUDA_OK(cudaEventRecord(e->ev_fork, main_stream));
        forked = true;
      }
      if (!used[op.lane - 1]) {
        AICAM_CUDA_OK(cudaStreamWaitEvent(e->side[op.lane - 1], e->ev_fork, 0));
        used[op.lane - 1] = true;
      }
      stream = e->side[op.lane - 1];
    }
    auto geom = [&](const View& v, int fallback_c, const __nv_bfloat16** ptr, long long* img_stride, int* cstride) {
      if (v.buf >= 0) {
        const Buffer& b = e->buffers[v.buf];
        *ptr = b.ptr; *cstride = b.c; *img_stride = static_cast<long long>(b.h + pad_ext(b.pad)) * (b.w + pad_ext(b.pad)) * b.c;
      } else if (v.buf == -1) {
        *ptr = static_cast<const __nv_bfloat16*>(input); *cstride = 4;
        *img_stride = static_cast<long long>(e->in_h) * e->in_w * 4;
      } else {
        *ptr = nullptr; *cstride = e->out_cstride; *img_stride = e->out_img_stride;
      }
      (void)fallback_c;
    };
    const __nv_bfloat16 *ip = nullptr, *op_ = nullptr, *rp = nullptr;
    long long is = 0, os = 0, rs = 0;
    int ic = 0, oc = 0, rc_ = 0;
    geom(op.in, 0, &ip, &is, &ic);
    int rc = AICAM_OK;
    switch (op.type) {
      case Op::CONV: {
        geom(op.out, 0, &op_, &os, &oc);
        ConvLaunch L;
        const PackedConv& pc = e->convs[op.conv];
        L.in = ip; L.in_img_stride = is; L.in_cstride = ic; L.in_coff = op.in.coff;
        if (op.s2d_c0) {  // the same bytes viewed as (h x w) blocks of 4 c0 channels
          if (op.in.buf == -1) L.in = static_cast<const __nv_bfloat16*>(input_s2d);
          L.in_cstride = 4 * op.s2d_c0;
          L.in_img_stride = static_cast<long long>(op.h) * op.w * L.in_cstride;
        }
        L.out_s2d = op.out_s2d;
        L.batch = batch; L.h = op.h; L.w = op.w;
        L.ho = (op.h + 2 * (op.k / 2) - op.k) / op.stride + 1;
        L.wo = (op.w + 2 * (op.k / 2) - op.k) / op.stride + 1;
        if (op.s2d_c0) { L.ho = op.h; L.wo = op.w; }
        if (op.out.buf == -2) {
          L.out = static_cast<float*>(output) + op.out.eoff;
        } else {
          L.out = const_cast<__nv_bfloat16*>(op_) + op.out.eoff;
        }
        L.out_img_stride = os; L.out_cstride = oc; L.out_coff = op.out.coff; L.out_f32 = op.out_f32;
        if (op.only_fmt == 3) L.out_cstride = pc.cout;  // 4x4-block stem: (h x w) pixels of 4 c1 channels = the same bytes as the buffer's 2x2 blocks
        L.res = nullptr; L.res_img_stride = 0; L.res_cstride = 0; L.res_coff = 0; L.res_mode = 0;
        if (op.res_mode) {
          geom(op.res, 0, &rp, &rs, &rc_);
          L.res = rp; L.res_img_stride = rs; L.res_cstride = rc_; L.res_coff = op.res.coff; L.res_mode = op.res_mode;
        }
        L.act = op.act;
        L.batch_dev = n_dev;
        L.in_pad = op.in.buf >= 0 ? e->buffers[op.in.buf].pad : 0;
        L.out_pad = op.out.buf >= 0 ? e->buffers[op.out.buf].pad : 0;
        if (op.res_mode && op.res.buf >= 0 && e->buffers[op.res.buf].pad != L.out_pad)
          return fail(AICAM_ERR_INVALID_ARG, "engine: residual and output layouts differ");
        if (dec && op.out.buf == -2) {  // a Detect-head 1x1 layer: decode in the epilogue, nothing is stored through L.out
          L.decode = op.out.coff == 0 ? 1 : 2;
          L.dec_anchor_base = static_cast<int>(op.out.eoff / e->out_cstride);
          L.dec_anchors = e->num_anchors;
          L.dec_boxes = dec->boxes; L.dec_scores = dec->scores; L.dec_labels = dec->labels;
          L.out = dec->boxes;  // (any aligned address: the planner checks it, the kernel does not use it)
        }
        rc = launch_conv(pc, L, stream);
        break;
      }
      case Op::CHAIN: {
        const ChainOp& c = e->chains[op.chain];
        if (n_dev) break;  // (device-side batch counts: single layers)
        if (dec && op.out.buf == -2) break;  // (fused decode: the single layers carry it)
        geom(op.out, 0, &op_, &os, &oc);
        ChainSpec sp;
        sp.nstages = c.nstages;
        for (int s = 0; s < c.nstages; ++s) {
          ChainStageSpec& T = sp.st[s];
          T.pc = &e->convs[c.conv[s]];
          T.act = c.act[s]; T.nsrc = c.nsrc[s];
          for (int j = 0; j < 2; ++j) { T.src_buf[j] = c.src_buf[s][j]; T.src_coff[j] = c.src_coff[s][j]; T.src_c[j] = c.src_c[s][j]; }
          T.res_buf = c.res_buf[s]; T.res_coff = c.res_coff[s]; T.res_mode = c.res_mode[s];
        }
        if (op.in.buf < 0 || (op.in.buf >= 0 && e->buffers[op.in.buf].pad) || (op.out.buf >= 0 && e->buffers[op.out.buf].pad)) break;
        sp.in = ip; sp.in_img_stride = is; sp.in_cstride = ic; sp.in_coff = op.in.coff; sp.in_c = c.in_c;
        sp.batch = batch; sp.h = op.h; sp.w = op.w;
        if (op.out.buf == -2) sp.out = static_cast<float*>(output) + op.out.eoff;
        else sp.out = const_cast<__nv_bfloat16*>(op_) + op.out.eoff;
        sp.out_img_stride = os; sp.out_cstride = oc; sp.out_coff = op.out.coff; sp.out_f32 = op.out_f32;
        const int crc = try_launch_conv_chain(sp, stream);
        if (crc < 0) rc = crc;
        else if (crc == 1) skip = c.covers;
        break;
      }
      case Op::MAXPOOL:
        geom(op.out, 0, &op_, &os, &oc);
        rc = launch_maxpool(ip, is, ic, op.in.coff, batch, op.h, op.w, op.c, op.k, op.stride,
                            const_cast<__nv_bfloat16*>(op_), os, oc, op.out.coff, stream, n_dev);
        break;
      case Op::SPPF3: {
        static const bool unfused = getenv("AICAM_NO_SPPF_FUSION") != nullptr;
        rc = unfused ? 0 : try_launch_sppf_pool3(const_cast<__nv_bfloat16*>(ip), is, ic, op.in.coff, batch, op.h, op.w, op.c, stream, n_dev);
        if (rc == 1) { rc = AICAM_OK; break; }
        if (rc < 0) break;
        for (int r = 0; r < 3 && !rc; ++r)
          rc = launch_maxpool(ip, is, ic, op.in.coff + r * op.c, batch, op.h, op.w, op.c, op.k, op.stride, const_cast<__nv_bfloat16*>(ip), is, ic,
                              op.in.coff + (r + 1) * op.c, stream, n_dev);
        break;
      }
      case Op::UPSAMPLE:
        geom(op.out, 0, &op_, &os, &oc);
        rc = launch_upsample2x(ip, is, ic, op.in.coff, batch, op.h, op.w, op.c, const_cast<__nv_bfloat16*>(op_), os,
                               oc, op.out.coff, stream, n_dev);
        break;
      case Op::STEMPOOL: {
        geom(op.out, 0, &op_, &os, &oc);
        const __nv_bfloat16* in8 = ip;  // caller-provided NHWC8 crops ...
        if (!input_is_s2d) {             // ... or an NHWC4 tensor repacked here
          __nv_bfloat16* tmp = e->buffers[e->stem_in8].ptr;
          rc = launch_nhwc4_to_nhwc8(ip, batch, op.h, op.w, tmp, n_dev, stream);
          in8 = tmp;
        }
        if (!rc) rc = launch_stem_pool(e->stem, in8, batch, op.h, op.w, n_dev, const_cast<__nv_bfloat16*>(op_), stream,
                                       op.out.buf >= 0 ? e->buffers[op.out.buf].pad : 0);
        break;
      }
      case Op::AVGL2: {
        // a padded buffer is summed border and all (the border is zero) and divided by the interior count
        const int pd = op.in.buf >= 0 ? e->buffers[op.in.buf].pad : 0;
        rc = launch_avgpool_l2norm(ip, batch, (op.h + pad_ext(pd)) * (op.w + pad_ext(pd)), op.h * op.w, op.c, static_cast<float*>(output),
                                   stream, n_dev);
        break;
      }
    }
    if (rc) {
      join();  // never leave a side stream un-joined (an open graph capture would be invalidated)
      return rc;
    }
  }
  return join();
}

}  // namespace

}  // namespace aicam

using namespace aicam;

extern "C" {

int aicam_engine_create(const char* blob_path, int device, int max_batch, aicam_engine** out) {
  if (!blob_path || !out || max_batch <= 0) return fail(AICAM_ERR_INVALID_ARG, "engine_create: bad arguments");
  *out = nullptr;
  std::ifstream f(blob_path, std::ios::binary | std::ios::ate);
  if (!f) return fail(AICAM_ERR_IO, std::string("engine_create: weight blob not found: ") + blob_path);
  const size_t size = static_cast<size_t>(f.tellg());
  std::vector<char> raw(size);
  f.seekg(0);
  f.read(raw.data(), size);
  if (size < 48 || std::memcmp(raw.data(), "AICW0001", 8) != 0)
    return fail(AICAM_ERR_IO, std::string("engine_create: not an AICW0001 weight blob: ") + blob_path);
  uint32_t head[10];
  std::memcpy(head, raw.data() + 8, sizeof(head));
  const uint32_t kind = head[0], n_tensors = head[9];
  const size_t entry = 64 + 4 + 16 + 8 + 8;
  if (n_tensors > (size - 48) / entry) return fail(AICAM_ERR_IO, "engine_create: truncated blob header");
  std::map<std::string, BlobTensor> tensors;
  for (uint32_t i = 0; i < n_tensors; ++i) {
    const char* p = raw.data() + 48 + i * entry;
    char name[65] = {0};
    std::memcpy(name, p, 64);
    uint32_t nd, dims[4];
    uint64_t off, nbytes;
    std::memcpy(&nd, p + 64, 4);
    std::memcpy(dims, p + 68, 16);
    std::memcpy(&off, p + 84, 8);
    std::memcpy(&nbytes, p + 92, 8);
    // (written so that nothing can wrap: off and nbytes are untrusted 64-bit values)
    if (nd > 4 || off > size || nbytes > size - off || off % 4 != 0 || nbytes % 4 != 0)
      return fail(AICAM_ERR_IO, "engine_create: corrupt tensor entry");
    BlobTensor t;
    uint64_t prod = 1;
    for (uint32_t d = 0; d < nd; ++d) {
      if (dims[d] == 0 || dims[d] > (1u << 24)) return fail(AICAM_ERR_IO, "engine_create: corrupt tensor dimensions");
      t.dims.push_back(static_cast<int>(dims[d]));
      prod *= dims[d];
      if (prod > (1ull << 32)) return fail(AICAM_ERR_IO, "engine_create: corrupt tensor dimensions");
    }
    t.data = reinterpret_cast<const float*>(raw.data() + off);
    t.count = nbytes / 4;
    // every tensor must hold exactly prod(dims) floats: the packers index it by its dims
    if (t.count != prod) return fail(AICAM_ERR_IO, "engine_create: tensor byte count differs from its dimensions");
    tensors[name] = t;
  }
  AICAM_CUDA_OK(cudaSetDevice(device));
  cudaDeviceProp prop;
  AICAM_CUDA_OK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(AICAM_ERR_UNSUPPORTED, "engine_create: this library contains sm_100a code only (tcgen05/TMEM)");
  aicam_engine* e = new aicam_engine();
  e->kind = static_cast<int>(kind);
  e->device = device;
  e->max_batch = max_batch;
  std::memcpy(e->params, head + 1, 32);
  Builder b{e, &tensors};
  if (kind == AICAM_KIND_YOLOV8) {
    b.build_yolov8();
  } else if (kind == AICAM_KIND_REID) {
    b.build_reid();
  } else {
    delete e;
    return fail(AICAM_ERR_IO, "engine_create: unknown model kind in blob");
  }
  if (b.err) {
    aicam_engine_destroy(e);
    return b.err;
  }
  bool lanes = false;
  for (const auto& op : e->ops) lanes = lanes || op.lane > 0;
  if (lanes) {
    for (int i = 0; i < 2; ++i) {
      AICAM_CUDA_OK(cudaStreamCreateWithFlags(&e->side[i], cudaStreamNonBlocking));
      AICAM_CUDA_OK(cudaEventCreateWithFlags(&e->ev_join[i], cudaEventDisableTiming));
    }
    AICAM_CUDA_OK(cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming));
  }
  AICAM_CUDA_OK(cudaDeviceSynchronize());
  *out = e;
  return AICAM_OK;
}

void aicam_engine_destroy(aicam_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  for (auto& c : e->convs) free_packed_conv(&c);
  free_stem_pool(&e->stem);
  for (auto& b : e->buffers)
    if (b.ptr) cudaFree(b.ptr);
  for (int i = 0; i < 2; ++i) {
    if (e->side[i]) cudaStreamDestroy(e->side[i]);
    if (e->ev_join[i]) cudaEventDestroy(e->ev_join[i]);
  }
  if (e->ev_fork) cudaEventDestroy(e->ev_fork);
  delete e;
}

int aicam_engine_kind(const aicam_engine* e) { return e ? e->kind : 0; }
int aicam_engine_max_batch(const aicam_engine* e) { return e ? e->max_batch : 0; }
int aicam_engine_num_classes(const aicam_engine* e) {
  if (!e) return 0;
  return e->kind == AICAM_KIND_YOLOV8 ? static_cast<int>(e->params[7]) : e->out_cstride;
}
int aicam_engine_num_anchors(const aicam_engine* e) { return e ? e->num_anchors : 0; }
double aicam_engine_flops_per_item(const aicam_engine* e) { return e ? 2.0 * e->macs_per_item : 0.0; }
int aicam_engine_num_launches(const aicam_engine* e) {
  if (!e) return 0;
  int n = 0;
  for (const auto& op : e->ops) {
    if (op.only_fmt == 2) continue;  // (the stem exists twice, one of the two runs)
    n += op.type == aicam::Op::STEMPOOL ? 2 : (op.type == aicam::Op::CHAIN ? 0 : 1);
  }  // upper bound: NHWC8 repack + fused stem; chains replace layers
  return n;
}

int aicam_engine_io_count(const aicam_engine* e, int is_output) {
  if (!e) return 0;
  if (e->kind == AICAM_KIND_YOLOV8) return is_output ? 4 : 1;
  return 1;
}

int aicam_engine_io_info(const aicam_engine* e, int is_output, int index, int topk, aicam_tensor_info* info) {
  if (!e || !info || index < 0 || index >= aicam_engine_io_count(e, is_output))
    return fail(AICAM_ERR_INVALID_ARG, "engine_io_info: bad arguments");
  std::memset(info, 0, sizeof(*info));
  auto set = [&](const char* name, int dtype, int ndim, int d0, int d1, int d2, int d3, int dyn) {
    std::strncpy(info->name, name, sizeof(info->name) - 1);
    info->dtype = dtype; info->ndim = ndim; info->is_dynamic = dyn;
    info->shape[0] = d0; info->shape[1] = d1; info->shape[2] = d2; info->shape[3] = d3;
  };
  if (e->kind == AICAM_KIND_YOLOV8) {
    // the reference engine: `images` 1x3x640x640 (scripts/export_trt_engines.sh:25-28) and the four outputs of its
    // embedded NMS (src/detector/yolo_detector.py:49-54)
    if (!is_output) set("images", AICAM_DTYPE_F32, 4, 1, 3, e->in_h, e->in_w, 0);
    else if (index == 0) set("num_dets", AICAM_DTYPE_I32, 2, 1, 1, 0, 0, 0);
    else if (index == 1) set("bboxes", AICAM_DTYPE_F32, 3, 1, topk, 4, 0, 0);
    else if (index == 2) set("scores", AICAM_DTYPE_F32, 2, 1, topk, 0, 0, 0);
    else set("labels", AICAM_DTYPE_I32, 2, 1, topk, 0, 0, 0);
  } else {
    // `input` Nx3x128x64, dynamic batch (export_trt_engines.sh:31-34); one (N, feature_dim) output (reid_model.py:46)
    if (!is_output) set("input", AICAM_DTYPE_F32, 4, -1, 3, e->in_h, e->in_w, 1);
    else set("output", AICAM_DTYPE_F32, 2, -1, e->out_cstride, 0, 0, 1);
  }
  return AICAM_OK;
}

int aicam_engine_set_bias(aicam_engine* e, const char* name, const float* host, int n) {
  if (!e || !name || !host) return fail(AICAM_ERR_INVALID_ARG, "engine_set_bias: bad arguments");
  auto it = e->conv_by_name.find(name);
  if (it == e->conv_by_name.end()) return fail(AICAM_ERR_INVALID_ARG, std::string("engine_set_bias: no layer ") + name);
  PackedConv& pc = e->convs[it->second];
  if (n != pc.cout) return fail(AICAM_ERR_INVALID_ARG, "engine_set_bias: length differs from the layer's cout");
  AICAM_CUDA_OK(cudaSetDevice(e->device));
  AICAM_CUDA_OK(cudaMemcpy(pc.bias, host, sizeof(float) * n, cudaMemcpyHostToDevice));
  if (pc.bias_host) std::memcpy(pc.bias_host, host, sizeof(float) * n);  // (kernel-argument copy: takes effect at the next launch / capture)
  if (e->stem4 >= 0 && std::string(name) == "model.0.conv") {  // the 4x4-block form of the stem repeats the bias per output sub-pixel
    PackedConv& p4 = e->convs[e->stem4];
    std::vector<float> b4(p4.cout);
    for (int i = 0; i < p4.cout; ++i) b4[i] = host[i % n];
    AICAM_CUDA_OK(cudaMemcpy(p4.bias, b4.data(), sizeof(float) * p4.cout, cudaMemcpyHostToDevice));
    if (p4.bias_host) std::memcpy(p4.bias_host, b4.data(), sizeof(float) * p4.cout);
  }
  return AICAM_OK;
}

int aicam_engine_get_bias(aicam_engine* e, const char* name, float* host, int n) {
  if (!e || !name || !host) return fail(AICAM_ERR_INVALID_ARG, "engine_get_bias: bad arguments");
  auto it = e->conv_by_name.find(name);
  if (it == e->conv_by_name.end()) return fail(AICAM_ERR_INVALID_ARG, std::string("engine_get_bias: no layer ") + name);
  PackedConv& pc = e->convs[it->second];
  if (n != pc.cout) return fail(AICAM_ERR_INVALID_ARG, "engine_get_bias: length differs from the layer's cout");
  AICAM_CUDA_OK(cudaSetDevice(e->device));
  AICAM_CUDA_OK(cudaMemcpy(host, pc.bias, sizeof(float) * n, cudaMemcpyDeviceToHost));
  return AICAM_OK;
}

int aicam_yolo_forward(aicam_engine* e, const void* in_nhwc4, int batch, float* head, void* stream) {
  if (!e || e->kind != AICAM_KIND_YOLOV8) return fail(AICAM_ERR_INVALID_ARG, "yolo_forward: not a yolov8 engine");
  if (!in_nhwc4 || !head) return fail(AICAM_ERR_INVALID_ARG, "yolo_forward: null tensor");
  if (batch < 0 || batch > e->max_batch) return fail(AICAM_ERR_CAPACITY, "yolo_forward: batch exceeds max_batch");
  return run_ops(e, in_nhwc4, batch, head, static_cast<cudaStream_t>(stream));
}

int aicam_engine_fused_decode(const aicam_engine* e) {
  static const bool off = getenv("AICAM_NO_DECODE_FUSION") != nullptr;
  if (!e || e->kind != AICAM_KIND_YOLOV8 || off) return 0;
  const int nc = static_cast<int>(e->params[7]);
  return (nc % 16 == 0 && nc <= 80 && e->num_anchors == 8400) ? 1 : 0;  // one n-tile of whole 16-column groups per branch
}

// aicam_yolo_detect[_table]; recs: the frame table's records (per-frame un-letterboxing and packed slot), or null;
// n_dev: the table's device count of present frames, which the network runs over (packed to the front of `in`), or null
static int yolo_detect_impl(aicam_engine* e, const void* in, int in_is_s2d, int batch, const aicam_nms_params* p, float* head,
                            int32_t* num_dets, float* boxes_lb, float* boxes_orig, float* scores, int32_t* labels, void* workspace,
                            size_t workspace_bytes, void* stream, const FrameRec* recs, const int* n_dev) {
  if (!e || e->kind != AICAM_KIND_YOLOV8) return fail(AICAM_ERR_INVALID_ARG, "yolo_detect: not a yolov8 engine");
  if (batch < 0 || batch > e->max_batch) return fail(AICAM_ERR_CAPACITY, "yolo_detect: batch exceeds max_batch");
  if (in_is_s2d < 0 || in_is_s2d > 2) return fail(AICAM_ERR_INVALID_ARG, "yolo_detect: in_is_s2d must be 0, 1 or 2");
  if (in_is_s2d && e->s2d_in < 0) return fail(AICAM_ERR_UNSUPPORTED, "yolo_detect: this engine was built without the space-to-depth stem");
  if (!in || !p || !num_dets || !boxes_lb || !scores || !labels) return fail(AICAM_ERR_INVALID_ARG, "yolo_detect: null argument");
  const int anchors = e->num_anchors, nc = static_cast<int>(e->params[7]);
  if (batch == 0) return AICAM_OK;
  if (!aicam_engine_fused_decode(e)) {
    if (!head) return fail(AICAM_ERR_INVALID_ARG, "yolo_detect: this engine needs the fp32 head tensor (no fused decode)");
    if (int rc = run_ops(e, in, batch, head, static_cast<cudaStream_t>(stream), n_dev, in_is_s2d)) return rc;
    return decode_nms_impl(head, batch, anchors, nc, p, num_dets, boxes_lb, boxes_orig, scores, labels, workspace, workspace_bytes,
                           stream, recs);
  }
  const size_t need = aicam_decode_nms_workspace(batch, anchors, p);
  if (need == 0 || !workspace || workspace_bytes < need) return fail(AICAM_ERR_CAPACITY, "yolo_detect: workspace too small");
  // the workspace layout of aicam_decode_nms: dense boxes, scores, labels, then (256-aligned) the suppression masks
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  const size_t dense = static_cast<size_t>(batch) * anchors * 24;
  DecodeTarget dec;
  dec.boxes = reinterpret_cast<float*>(ws);
  dec.scores = reinterpret_cast<float*>(ws + static_cast<size_t>(batch) * anchors * 16);
  dec.labels = reinterpret_cast<int*>(ws + static_cast<size_t>(batch) * anchors * 20);
  uint8_t* mask = ws + (dense + 255) / 256 * 256;
  if (int rc = run_ops(e, in, batch, nullptr, static_cast<cudaStream_t>(stream), n_dev, in_is_s2d, &dec)) return rc;
  return nms_impl(dec.boxes, dec.scores, dec.labels, batch, anchors, p, num_dets, boxes_lb, boxes_orig, scores, labels, nullptr,
                  mask, workspace_bytes - static_cast<size_t>(mask - ws), stream, recs);
}

int aicam_yolo_detect(aicam_engine* e, const void* in, int in_is_s2d, int batch, const aicam_nms_params* p, float* head,
                      int32_t* num_dets, float* boxes_lb, float* boxes_orig, float* scores, int32_t* labels, void* workspace,
                      size_t workspace_bytes, void* stream) {
  return yolo_detect_impl(e, in, in_is_s2d, batch, p, head, num_dets, boxes_lb, boxes_orig, scores, labels, workspace, workspace_bytes,
                          stream, nullptr, nullptr);
}

int aicam_yolo_detect_table(aicam_engine* e, const void* in, int in_is_s2d, const aicam_frame_table* t, const aicam_nms_params* p,
                            float* head, int32_t* num_dets, float* boxes_lb, float* boxes_orig, float* scores, int32_t* labels,
                            void* workspace, size_t workspace_bytes, void* stream) {
  if (!t) return fail(AICAM_ERR_INVALID_ARG, "yolo_detect_table: null frame table");
  return yolo_detect_impl(e, in, in_is_s2d, t->n, p, head, num_dets, boxes_lb, boxes_orig, scores, labels, workspace, workspace_bytes,
                          stream, t->recs(), t->counts() + 3);
}

int aicam_yolo_forward_s2d(aicam_engine* e, const void* in_s2d16, int batch, float* head, void* stream) {
  if (!e || e->kind != AICAM_KIND_YOLOV8) return fail(AICAM_ERR_INVALID_ARG, "yolo_forward_s2d: not a yolov8 engine");
  if (!in_s2d16 || !head) return fail(AICAM_ERR_INVALID_ARG, "yolo_forward_s2d: null tensor");
  if (batch < 0 || batch > e->max_batch) return fail(AICAM_ERR_CAPACITY, "yolo_forward_s2d: batch exceeds max_batch");
  return run_ops(e, in_s2d16, batch, head, static_cast<cudaStream_t>(stream), nullptr, true);
}

int aicam_engine_accepts_s2d(const aicam_engine* e) { return e && e->s2d_in >= 0 ? (e->stem4 >= 0 ? 2 : 1) : 0; }

int aicam_engine_accepts_nhwc8(const aicam_engine* e) { return e && e->kind == AICAM_KIND_REID && e->stem_in8 >= 0 ? 1 : 0; }

int aicam_reid_forward_nhwc8(aicam_engine* e, const void* crops_nhwc8, int n, const int32_t* n_dev, float* feats, void* stream) {
  if (!e || e->kind != AICAM_KIND_REID) return fail(AICAM_ERR_INVALID_ARG, "reid_forward_nhwc8: not a reid engine");
  if (!crops_nhwc8 || !feats || !n_dev) return fail(AICAM_ERR_INVALID_ARG, "reid_forward_nhwc8: null tensor (a device-side count is required)");
  if (n < 0 || n > e->max_batch) return fail(AICAM_ERR_CAPACITY, "reid_forward_nhwc8: capacity exceeds max_batch");
  return run_ops(e, crops_nhwc8, n, feats, static_cast<cudaStream_t>(stream), n_dev, true);
}

int aicam_reid_forward(aicam_engine* e, const void* crops_nhwc4, int n, const int32_t* n_dev, float* feats,
                       void* stream) {
  if (!e || e->kind != AICAM_KIND_REID) return fail(AICAM_ERR_INVALID_ARG, "reid_forward: not a reid engine");
  if (!crops_nhwc4 || !feats) return fail(AICAM_ERR_INVALID_ARG, "reid_forward: null tensor");
  if (n < 0) return fail(AICAM_ERR_INVALID_ARG, "reid_forward: negative batch");
  if (n_dev) {
    if (n > e->max_batch) return fail(AICAM_ERR_CAPACITY, "reid_forward: capacity exceeds max_batch");
    return run_ops(e, crops_nhwc4, n, feats, static_cast<cudaStream_t>(stream), n_dev);
  }
  // crops beyond the engine's workspace are processed in slices of max_batch
  const long long in_stride = static_cast<long long>(AICAM_REID_H) * AICAM_REID_W * 4;
  for (int s = 0; s < n; s += e->max_batch) {
    const int nb = std::min(e->max_batch, n - s);
    int rc = run_ops(e, static_cast<const __nv_bfloat16*>(crops_nhwc4) + s * in_stride, nb,
                     feats + static_cast<long long>(s) * e->out_cstride, static_cast<cudaStream_t>(stream));
    if (rc) return rc;
  }
  return AICAM_OK;
}

int aicam_nchw_to_nhwc4(const float* in, int n, int h, int w, void* out, void* stream) {
  if (!in || !out || n < 0) return fail(AICAM_ERR_INVALID_ARG, "nchw_to_nhwc4: bad arguments");
  return launch_nchw_to_nhwc4(in, n, h, w, static_cast<__nv_bfloat16*>(out), static_cast<cudaStream_t>(stream));
}

int aicam_conv2d(const aicam_conv_desc* d, const void* in, const float* w, const float* bias, const void* res,
                 void* out, void* stream) {
  if (!d || !in || !w || !out) return fail(AICAM_ERR_INVALID_ARG, "conv2d: null argument");
  PackedConv pc;
  const int c0 = (d->h % 2 == 0 && d->w % 2 == 0) ? s2d_channels(d->ksize, d->stride, d->cin, d->cin <= 4 ? 4 : d->cin) : 0;
  if (c0) {  // 3x3 stride 2 over 3/4 or 16 dense channels: repack space-to-depth, 2x2 window kernel
    if (int rc = pack_conv_weights_s2d(w, bias, d->cout, d->cin, c0, &pc)) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    __nv_bfloat16* s2 = nullptr;
    if (cudaMalloc(&s2, static_cast<size_t>(d->batch) * d->h * d->w * c0 * 2) != cudaSuccess) {
      free_packed_conv(&pc);
      return fail(AICAM_ERR_CUDA, "conv2d: cudaMalloc failed");
    }
    int rc = launch_space_to_depth(static_cast<const __nv_bfloat16*>(in), d->batch, d->h, d->w, c0, s2, st);
    ConvLaunch L;
    L.in = s2; L.in_cstride = 4 * c0; L.in_coff = 0;
    L.batch = d->batch; L.h = d->h / 2; L.w = d->w / 2; L.ho = L.h; L.wo = L.w;
    L.in_img_stride = static_cast<long long>(L.h) * L.w * L.in_cstride;
    L.out = out; L.out_img_stride = static_cast<long long>(L.ho) * L.wo * d->cout; L.out_cstride = d->cout;
    L.out_coff = 0; L.out_f32 = d->out_f32;
    L.res = static_cast<const __nv_bfloat16*>(res); L.res_img_stride = L.out_img_stride; L.res_cstride = d->cout;
    L.res_coff = 0; L.res_mode = res ? d->res_mode : 0;
    L.act = d->act;
    if (!rc) rc = launch_conv(pc, L, st);
    cudaError_t se = cudaStreamSynchronize(st);
    cudaFree(s2);
    free_packed_conv(&pc);
    if (rc) return rc;
    if (se != cudaSuccess) return fail(AICAM_ERR_CUDA, std::string("conv2d: ") + cudaGetErrorString(se));
    return AICAM_OK;
  }
  return aicam_conv2d_padded(d, in, w, bias, res, out, 0, 0, stream);
}

int aicam_conv2d_padded(const aicam_conv_desc* d, const void* in, const float* w, const float* bias, const void* res,
                        void* out, int in_pad, int out_pad, void* stream) {
  if (!d || !in || !w || !out) return fail(AICAM_ERR_INVALID_ARG, "conv2d: null argument");
  PackedConv pc;
  if (int rc = pack_conv_weights(w, bias, d->cout, d->cin, d->ksize, d->stride, &pc)) return rc;
  ConvLaunch L;
  const int cs = pc.cin_pad;
  if (in_pad < 0 || in_pad > 2 || out_pad < 0 || out_pad > 2) return fail(AICAM_ERR_INVALID_ARG, "conv2d_padded: border kinds are 0, 1, 2");
  const int ip = in_pad, opd = out_pad;
  L.in = static_cast<const __nv_bfloat16*>(in);
  L.in_img_stride = static_cast<long long>(d->h + pad_ext(ip)) * (d->w + pad_ext(ip)) * cs; L.in_cstride = cs; L.in_coff = 0;
  L.batch = d->batch; L.h = d->h; L.w = d->w;
  L.ho = (d->h + 2 * (d->ksize / 2) - d->ksize) / d->stride + 1;
  L.wo = (d->w + 2 * (d->ksize / 2) - d->ksize) / d->stride + 1;
  L.out = out; L.out_img_stride = static_cast<long long>(L.ho + pad_ext(opd)) * (L.wo + pad_ext(opd)) * d->cout; L.out_cstride = d->cout;
  L.out_coff = 0; L.out_f32 = d->out_f32;
  L.res = static_cast<const __nv_bfloat16*>(res); L.res_img_stride = L.out_img_stride; L.res_cstride = d->cout;
  L.res_coff = 0; L.res_mode = res ? d->res_mode : 0;
  L.act = d->act;
  L.in_pad = ip; L.out_pad = opd;
  if (ip && opd) pack_pair_weights(&pc);
  int rc = launch_conv(pc, L, static_cast<cudaStream_t>(stream));
  cudaError_t se = cudaStreamSynchronize(static_cast<cudaStream_t>(stream));
  free_packed_conv(&pc);
  if (rc) return rc;
  if (se != cudaSuccess) return fail(AICAM_ERR_CUDA, std::string("conv2d: ") + cudaGetErrorString(se));
  return AICAM_OK;
}

int aicam_reid_stem_pool(const void* in_nhwc4, int n, int h, int w, const float* weights_oihw, const float* bias, void* out,
                         void* stream) {
  if (!in_nhwc4 || !weights_oihw || !out || n <= 0 || h <= 0 || w <= 0)
    return fail(AICAM_ERR_INVALID_ARG, "reid_stem_pool: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  StemPool sp;
  if (int rc = pack_stem_pool(weights_oihw, bias, 64, 3, &sp)) return rc;
  __nv_bfloat16* in8 = nullptr;
  cudaError_t ce = cudaMalloc(&in8, static_cast<size_t>(n) * h * w * 16);
  if (ce != cudaSuccess) {
    free_stem_pool(&sp);
    return fail(AICAM_ERR_CUDA, std::string("reid_stem_pool: ") + cudaGetErrorString(ce));
  }
  int rc = launch_nhwc4_to_nhwc8(static_cast<const __nv_bfloat16*>(in_nhwc4), n, h, w, in8, nullptr, st);
  if (!rc) rc = launch_stem_pool(sp, in8, n, h, w, nullptr, static_cast<__nv_bfloat16*>(out), st);
  cudaError_t se = cudaStreamSynchronize(st);
  cudaFree(in8);
  free_stem_pool(&sp);
  if (rc) return rc;
  if (se != cudaSuccess) return fail(AICAM_ERR_CUDA, std::string("reid_stem_pool: ") + cudaGetErrorString(se));
  return AICAM_OK;
}

int aicam_conv2d_bench(const aicam_conv_desc* d, int iters, double* mean_ms, void* stream) {
  if (!d || !mean_ms || iters <= 0) return fail(AICAM_ERR_INVALID_ARG, "conv2d_bench: bad arguments");
  std::vector<float> w(static_cast<size_t>(d->cout) * d->cin * d->ksize * d->ksize), b(d->cout, 0.1f);
  uint32_t seed = 12345u;
  for (auto& v : w) { seed = seed * 1664525u + 1013904223u; v = (static_cast<int>(seed >> 16) % 2001 - 1000) * 1e-4f; }
  PackedConv pc;
  const int c0 = (d->h % 2 == 0 && d->w % 2 == 0) ? s2d_channels(d->ksize, d->stride, d->cin, d->cin <= 4 ? 4 : d->cin) : 0;
  if (int rc = c0 ? pack_conv_weights_s2d(w.data(), b.data(), d->cout, d->cin, c0, &pc)
                  : pack_conv_weights(w.data(), b.data(), d->cout, d->cin, d->ksize, d->stride, &pc))
    return rc;
  ConvLaunch L;
  const int cs = c0 ? c0 : pc.cin_pad;
  const int ho = (d->h + 2 * (d->ksize / 2) - d->ksize) / d->stride + 1;
  const int wo = (d->w + 2 * (d->ksize / 2) - d->ksize) / d->stride + 1;
  // AICAM_BENCH_PAD=1: 3x3 stride-1 layers are timed over zero-bordered tensors (operand mode 4)
  const int bp = (getenv("AICAM_BENCH_PAD") && d->ksize == 3 && d->stride == 1 && !c0) ? std::max(1, std::min(2, atoi(getenv("AICAM_BENCH_PAD")))) : 0;
  const int be = pad_ext(bp);
  const size_t in_elems = static_cast<size_t>(d->batch) * (d->h + be) * (d->w + be) * cs;
  const size_t out_elems = static_cast<size_t>(d->batch) * (ho + be) * (wo + be) * d->cout;
  __nv_bfloat16 *in = nullptr, *res = nullptr;
  void* out = nullptr;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  AICAM_CUDA_OK(cudaMalloc(&in, in_elems * 2));
  AICAM_CUDA_OK(cudaMalloc(&out, out_elems * (d->out_f32 ? 4 : 2)));
  AICAM_CUDA_OK(cudaMemset(in, 0x3c, in_elems * 2));  // bf16 0x3c3c ~ 0.0115
  if (d->res_mode) {
    AICAM_CUDA_OK(cudaMalloc(&res, out_elems * 2));
    AICAM_CUDA_OK(cudaMemset(res, 0x3c, out_elems * 2));
  }
  L.in = in; L.in_img_stride = static_cast<long long>(d->h + be) * (d->w + be) * cs; L.in_cstride = cs; L.in_coff = 0;
  L.batch = d->batch; L.h = d->h; L.w = d->w; L.ho = ho; L.wo = wo;
  L.in_pad = bp; L.out_pad = bp;
  if (bp) pack_pair_weights(&pc);
  if (c0) {  // the timed launches read the same bytes as an already space-to-depth tensor
    L.in_cstride = 4 * c0; L.h = d->h / 2; L.w = d->w / 2; L.ho = L.h; L.wo = L.w;
  }
  L.out = out; L.out_img_stride = static_cast<long long>(ho + be) * (wo + be) * d->cout; L.out_cstride = d->cout; L.out_coff = 0;
  L.out_f32 = d->out_f32;
  L.res = res; L.res_img_stride = L.out_img_stride; L.res_cstride = d->cout; L.res_coff = 0; L.res_mode = d->res_mode;
  L.act = d->act;
  int rc = AICAM_OK;
  for (int i = 0; i < 3 && !rc; ++i) rc = launch_conv(pc, L, st);
  if (getenv("AICAM_CONV_TRACE")) {  // per-phase clock64 stamps of CTA 0 (debug aid)
    long long* tr = nullptr;
    cudaMalloc(&tr, 512 * 8);
    cudaMemset(tr, 0, 512 * 8);
    L.trace = tr;
    launch_conv(pc, L, st);
    cudaStreamSynchronize(st);
    L.trace = nullptr;
    std::vector<long long> h(512);
    cudaMemcpy(h.data(), tr, 512 * 8, cudaMemcpyDeviceToHost);
    cudaFree(tr);
    long long t0 = 0;
    for (int k = 0; k < 512 && !t0; ++k) t0 = h[k];
    for (int k = 0; k < 512; ++k) if (h[k] && h[k] < t0) t0 = h[k];
    printf("trace of CTA 0, cycles since its first stamp; per tile: MMA[wait_acc_empty acc_empty_ok a_full_ok issued] "
           "PROD[wait_a_empty a_empty_ok] EPI[wait_acc_full acc_full_ok barA res_ok finished barB]\n");
    for (int t = 0; t < 24; ++t) {
      const long long* r = h.data() + t * 16;
      if (!r[8] && !r[0]) break;
      auto rel = [&](long long v) { return v ? v - t0 : -1ll; };
      printf("  tile %2d  MMA %7lld %7lld %7lld %7lld  PROD %7lld %7lld  EPI %7lld %7lld %7lld %7lld %7lld %7lld\n", t, rel(r[0]),
             rel(r[1]), rel(r[2]), rel(r[3]), rel(r[4]), rel(r[5]), rel(r[8]), rel(r[9]), rel(r[10]), rel(r[11]), rel(r[12]), rel(r[13]));
    }
    fflush(stdout);
  }
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  cudaEventRecord(e0, st);
  for (int i = 0; i < iters && !rc; ++i) rc = launch_conv(pc, L, st);
  cudaEventRecord(e1, st);
  cudaError_t se = cudaStreamSynchronize(st);
  float ms = 0.0f;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(in); cudaFree(out); if (res) cudaFree(res);
  free_packed_conv(&pc);
  if (rc) return rc;
  if (se != cudaSuccess) return fail(AICAM_ERR_CUDA, std::string("conv2d_bench: ") + cudaGetErrorString(se));
  *mean_ms = ms / iters;
  return AICAM_OK;
}

}  // extern "C"
