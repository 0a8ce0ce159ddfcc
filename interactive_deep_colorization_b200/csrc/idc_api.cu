// C ABI of libidc_b200.so (include/idc_b200.h): context, layer plan, weight packing, forward.
// The plan restates the wiring of SIGGRAPHGenerator.forward
// (/root/reference/models/pytorch/model.py:134-175) as a list of gather-GEMM ops; both engines
// (idc_simt.cu FP32 CUDA cores, idc_umma.cu tcgen05) execute the same list.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>

#include "idc_internal.h"

using namespace idc;

struct idc_ctx : public idc::Ctx {};

namespace {

int fail(Ctx* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (c) c->err = buf;
  return code;
}

#define CUDA_TRY(c, expr)                                                                         \
  do {                                                                                            \
    cudaError_t e__ = (expr);                                                                     \
    if (e__ != cudaSuccess)                                                                       \
      return fail(c, IDC_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

constexpr float kBnEps = 1e-5f;  // nn.BatchNorm2d default (SURVEY q7)

int add_buf(Ctx* c, const char* name, int H, int W, int C) {
  ActBuf b;
  b.name = name; b.H = H; b.W = W; b.C = C;
  c->bufs.push_back(b);
  c->buf_index[name] = (int)c->bufs.size() - 1;
  return (int)c->bufs.size() - 1;
}

// 3x3 conv (optionally dilated, optionally reading the ::2 decimation of its source)
void add_conv(Ctx* c, const char* name, const char* wkey, const char* in, int s, int dil, const char* out, int act,
              const char* bnkey, bool gadd = false) {
  ConvOp op;
  op.name = name; op.kind = OP_CONV; op.wkey[0] = wkey; op.bnkey = bnkey ? bnkey : "";
  const ActBuf& ib = c->bufs[c->buf_index.at(in)];
  const ActBuf& ob = c->bufs[c->buf_index.at(out)];
  op.nsrc = 1;
  op.src[0].buf = c->buf_index.at(in); op.src[0].s = s; op.src[0].cin = ib.C;
  op.ncls = 1; op.ntaps = 9;
  for (int ky = 0; ky < 3; ++ky)
    for (int kx = 0; kx < 3; ++kx) {
      Tap& t = op.taps[0][ky * 3 + kx];
      t.src = 0; t.ky = ky; t.kx = kx; t.ty = s * (ky - 1) * dil; t.tx = s * (kx - 1) * dil;
    }
  op.Hl = ob.H; op.Wl = ob.W; op.out_buf = c->buf_index.at(out); op.os = 1;
  op.cout = ob.C; op.cout_pad = ob.C; op.K = 9 * ib.C;
  op.epi.act = act; op.epi.has_bn = bnkey != nullptr; op.epi.gadd = gadd;
  op.flops_per_image = 2.0 * op.Hl * op.Wl * (double)op.cout * op.K;
  c->ops.push_back(op);
}

// ConvTranspose2d(4x4, s2, p1) of `lo` + Conv2d(3x3) of the skip tensor, summed, then ReLU
// (model.py:156-157,162-165: modelNup(x) + modelKshortN(skip), followed by modelN[0] = ReLU).
void add_up(Ctx* c, const char* name, const char* dkey, const char* lo, const char* skey, const char* skip,
            const char* out) {
  ConvOp op;
  op.name = name; op.kind = OP_UP; op.wkey[0] = dkey; op.wkey[1] = skey;
  op.src_deconv[0] = true; op.src_k[0] = 4;
  const ActBuf& lb = c->bufs[c->buf_index.at(lo)];
  const ActBuf& sb = c->bufs[c->buf_index.at(skip)];
  const ActBuf& ob = c->bufs[c->buf_index.at(out)];
  op.nsrc = 2;
  op.src[0].buf = c->buf_index.at(lo); op.src[0].s = 1; op.src[0].cin = lb.C;
  op.src[1].buf = c->buf_index.at(skip); op.src[1].s = 2; op.src[1].cin = sb.C;
  op.ncls = 4; op.ntaps = 13;
  for (int cls = 0; cls < 4; ++cls) {
    const int py = cls >> 1, px = cls & 1;
    // oy = 2*iy - 1 + ky  =>  parity 0: (ky=1, iy=y), (ky=3, iy=y-1); parity 1: (ky=0, iy=y+1), (ky=2, iy=y)
    const int kys[2][2] = {{1, 3}, {0, 2}};
    const int tys[2][2] = {{0, -1}, {1, 0}};
    int t = 0;
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < 2; ++b) {
        Tap& tp = op.taps[cls][t++];
        tp.src = 0; tp.ky = kys[py][a]; tp.kx = kys[px][b]; tp.ty = tys[py][a]; tp.tx = tys[px][b];
      }
    for (int ky = 0; ky < 3; ++ky)
      for (int kx = 0; kx < 3; ++kx) {
        Tap& tp = op.taps[cls][t++];
        tp.src = 1; tp.ky = ky; tp.kx = kx; tp.ty = py + ky - 1; tp.tx = px + kx - 1;
      }
  }
  op.Hl = lb.H; op.Wl = lb.W; op.out_buf = c->buf_index.at(out); op.os = 2;
  op.cout = ob.C; op.cout_pad = ob.C; op.K = 4 * lb.C + 9 * sb.C;
  op.epi.act = ACT_RELU;
  op.flops_per_image = 2.0 * 4 * op.Hl * op.Wl * (double)op.cout * op.K;
  c->ops.push_back(op);
}

void build_plan(Ctx* c) {
  const int H = c->H, W = c->W;
  add_buf(c, "a1_1", H, W, 64); add_buf(c, "conv1_2", H, W, 64);
  add_buf(c, "a2_1", H / 2, W / 2, 128); add_buf(c, "conv2_2", H / 2, W / 2, 128);
  add_buf(c, "a3_1", H / 4, W / 4, 256); add_buf(c, "a3_2", H / 4, W / 4, 256); add_buf(c, "conv3_3", H / 4, W / 4, 256);
  const char* n8[] = {"a4_1", "a4_2", "conv4_3", "a5_1", "a5_2", "conv5_3", "a6_1", "a6_2", "conv6_3",
                      "a7_1", "a7_2", "conv7_3"};
  for (const char* nm : n8) add_buf(c, nm, H / 8, W / 8, 512);
  add_buf(c, "a8_1", H / 4, W / 4, 256); add_buf(c, "a8_2", H / 4, W / 4, 256); add_buf(c, "conv8_3", H / 4, W / 4, 256);
  add_buf(c, "a9_1", H / 2, W / 2, 128); add_buf(c, "conv9_3", H / 2, W / 2, 128);
  add_buf(c, "a10_1", H, W, 128);
  const bool keep10 = c->simt || (c->flags & IDC_FLAG_KEEP_CONV10);
  if (keep10) add_buf(c, "conv10_2", H, W, 128);

  // model1 (conv1_1 is the fused pack+conv kernel in idc_heads.cu)            model.py:13-17
  add_conv(c, "c1_2", "model1.2", "a1_1", 1, 1, "conv1_2", ACT_RELU, "model1.4");
  // model2 on conv1_2[:, :, ::2, ::2]                                        model.py:149, 21-25
  add_conv(c, "c2_1", "model2.0", "conv1_2", 2, 1, "a2_1", ACT_RELU, nullptr);
  add_conv(c, "c2_2", "model2.2", "a2_1", 1, 1, "conv2_2", ACT_RELU, "model2.4");
  // model3                                                                   model.py:150, 29-35
  add_conv(c, "c3_1", "model3.0", "conv2_2", 2, 1, "a3_1", ACT_RELU, nullptr);
  add_conv(c, "c3_2", "model3.2", "a3_1", 1, 1, "a3_2", ACT_RELU, nullptr);
  add_conv(c, "c3_3", "model3.4", "a3_2", 1, 1, "conv3_3", ACT_RELU, "model3.6");
  // model4 (+ global-hints vector added to conv4_3norm, deploy_nodist.prototxt:501-527)  model.py:151, 39-45
  add_conv(c, "c4_1", "model4.0", "conv3_3", 2, 1, "a4_1", ACT_RELU, nullptr);
  add_conv(c, "c4_2", "model4.2", "a4_1", 1, 1, "a4_2", ACT_RELU, nullptr);
  add_conv(c, "c4_3", "model4.4", "a4_2", 1, 1, "conv4_3", ACT_RELU, "model4.6", c->glob);
  // model5, model6 (dilation 2), model7                                       model.py:48-72
  add_conv(c, "c5_1", "model5.0", "conv4_3", 1, 2, "a5_1", ACT_RELU, nullptr);
  add_conv(c, "c5_2", "model5.2", "a5_1", 1, 2, "a5_2", ACT_RELU, nullptr);
  add_conv(c, "c5_3", "model5.4", "a5_2", 1, 2, "conv5_3", ACT_RELU, "model5.6");
  add_conv(c, "c6_1", "model6.0", "conv5_3", 1, 2, "a6_1", ACT_RELU, nullptr);
  add_conv(c, "c6_2", "model6.2", "a6_1", 1, 2, "a6_2", ACT_RELU, nullptr);
  add_conv(c, "c6_3", "model6.4", "a6_2", 1, 2, "conv6_3", ACT_RELU, "model6.6");
  add_conv(c, "c7_1", "model7.0", "conv6_3", 1, 1, "a7_1", ACT_RELU, nullptr);
  add_conv(c, "c7_2", "model7.2", "a7_1", 1, 1, "a7_2", ACT_RELU, nullptr);
  add_conv(c, "c7_3", "model7.4", "a7_2", 1, 1, "conv7_3", ACT_RELU, "model7.6");
  // decoder level 8                                                          model.py:156-157, 75-83
  add_up(c, "up8", "model8up.0", "conv7_3", "model3short8.0", "conv3_3", "a8_1");
  add_conv(c, "c8_2", "model8.1", "a8_1", 1, 1, "a8_2", ACT_RELU, nullptr);
  add_conv(c, "c8_3", "model8.3", "a8_2", 1, 1, "conv8_3", ACT_RELU, "model8.5");
  // class head on conv8_3 (dist only)                                        model.py:105, 160
  if (c->dist) {
    ConvOp op;
    op.name = "class"; op.kind = OP_CLASS; op.wkey[0] = "model_class.0";
    const ActBuf& ib = c->bufs[c->buf_index.at("conv8_3")];
    op.nsrc = 1; op.src[0].buf = c->buf_index.at("conv8_3"); op.src[0].s = 1; op.src[0].cin = ib.C;
    op.ncls = 1; op.ntaps = 1;
    op.taps[0][0] = Tap{0, 0, 0, 0, 0};
    op.Hl = ib.H; op.Wl = ib.W; op.out_buf = -1; op.os = 1;
    op.cout = 529; op.cout_pad = 576; op.K = ib.C; op.out_f32 = true; op.src_k[0] = 1;
    op.flops_per_image = 2.0 * op.Hl * op.Wl * 529.0 * op.K;
    c->ops.push_back(op);
  }
  // Caffe-spec 313-bin head (row a14): hyper-column = conv3x3(conv3_3) + sum_l deconv4x4s2(conv{4..7}_3) +
  // conv3x3(conv8_3) -> ReLU (deploy_nopred.prototxt:651-763), then pred_313 = conv1x1 384->313 (:765-775)
  if (c->caffe313) {
    add_buf(c, "hyper", H / 4, W / 4, 384);
    ConvOp op;
    op.name = "hyper"; op.kind = OP_HYPER;
    const char* dsrc[4] = {"conv4_3", "conv5_3", "conv6_3", "conv7_3"};
    const char* dkey[4] = {"caffe.conv4_pred", "caffe.conv5_pred", "caffe.conv6_pred", "caffe.conv7_pred"};
    op.nsrc = 6;
    for (int s = 0; s < 4; ++s) {
      op.src[s].buf = c->buf_index.at(dsrc[s]); op.src[s].s = 1; op.src[s].cin = 512;
      op.wkey[s] = dkey[s]; op.src_deconv[s] = true; op.src_k[s] = 4;
    }
    op.src[4].buf = c->buf_index.at("conv3_3"); op.src[4].s = 2; op.src[4].cin = 256; op.wkey[4] = "caffe.conv3_pred";
    op.src[5].buf = c->buf_index.at("conv8_3"); op.src[5].s = 2; op.src[5].cin = 256; op.wkey[5] = "caffe.conv8_pred";
    op.ncls = 4; op.ntaps = 34;
    for (int cls = 0; cls < 4; ++cls) {
      const int py = cls >> 1, px = cls & 1;
      const int kys[2][2] = {{1, 3}, {0, 2}};
      const int tys[2][2] = {{0, -1}, {1, 0}};
      int t = 0;
      for (int s = 0; s < 4; ++s)
        for (int a = 0; a < 2; ++a)
          for (int b = 0; b < 2; ++b)
            op.taps[cls][t++] = Tap{s, kys[py][a], kys[px][b], tys[py][a], tys[px][b]};
      for (int s = 4; s < 6; ++s)
        for (int ky = 0; ky < 3; ++ky)
          for (int kx = 0; kx < 3; ++kx) op.taps[cls][t++] = Tap{s, ky, kx, py + ky - 1, px + kx - 1};
    }
    op.Hl = H / 8; op.Wl = W / 8; op.out_buf = c->buf_index.at("hyper"); op.os = 2;
    op.cout = 384; op.cout_pad = 384; op.K = 4 * 4 * 512 + 2 * 9 * 256;
    op.epi.act = ACT_RELU;
    op.flops_per_image = 2.0 * 4 * op.Hl * op.Wl * 384.0 * op.K;
    c->ops.push_back(op);

    ConvOp pr;
    pr.name = "pred313"; pr.kind = OP_CLASS; pr.wkey[0] = "caffe.pred_313"; pr.src_k[0] = 1;
    pr.nsrc = 1; pr.src[0].buf = c->buf_index.at("hyper"); pr.src[0].s = 1; pr.src[0].cin = 384;
    pr.ncls = 1; pr.ntaps = 1; pr.taps[0][0] = Tap{0, 0, 0, 0, 0};
    pr.Hl = H / 4; pr.Wl = W / 4; pr.out_buf = -1; pr.os = 1;
    pr.cout = 313; pr.cout_pad = 320; pr.K = 384; pr.out_f32 = true;
    pr.flops_per_image = 2.0 * pr.Hl * pr.Wl * 313.0 * pr.K;
    c->ops.push_back(pr);
  }
  // level 9                                                                  model.py:162-163, 86-93
  add_up(c, "up9", "model9up.0", "conv8_3", "model2short9.0", "conv2_2", "a9_1");
  add_conv(c, "c9_2", "model9.1", "a9_1", 1, 1, "conv9_3", ACT_RELU, "model9.3");
  // level 10                                                                 model.py:164-165, 96-102
  add_up(c, "up10", "model10up.0", "conv9_3", "model1short10.0", "conv1_2", "a10_1");
  if (keep10) {
    add_conv(c, "c10_2", "model10.1", "a10_1", 1, 1, "conv10_2", ACT_LEAKY02, nullptr);
  } else {
    // conv10_2 never leaves the SM: model_out (1x1 128->2, tanh, x110) runs in the epilogue
    add_buf(c, "conv10_2_virtual", 0, 0, 128);
    ConvOp op;
    op.name = "c10_2"; op.kind = OP_CONV; op.wkey[0] = "model10.1";
    const ActBuf& ib = c->bufs[c->buf_index.at("a10_1")];
    op.nsrc = 1; op.src[0].buf = c->buf_index.at("a10_1"); op.src[0].s = 1; op.src[0].cin = ib.C;
    op.ncls = 1; op.ntaps = 9;
    for (int ky = 0; ky < 3; ++ky)
      for (int kx = 0; kx < 3; ++kx) op.taps[0][ky * 3 + kx] = Tap{0, ky, kx, ky - 1, kx - 1};
    op.Hl = ib.H; op.Wl = ib.W; op.out_buf = -1; op.os = 1;
    op.cout = 128; op.cout_pad = 128; op.K = 9 * ib.C;
    op.epi.act = ACT_LEAKY02; op.fuse_out_head = true;
    op.flops_per_image = 2.0 * op.Hl * op.Wl * 128.0 * op.K;
    c->ops.push_back(op);
  }
}

// ---------------------------------------------------------------------------------------------
// weight arena
// ---------------------------------------------------------------------------------------------
struct ArenaLayout {
  size_t off = 0;
  template <typename T>
  size_t take(size_t count) {
    off = (off + 255) & ~size_t(255);
    size_t o = off;
    off += count * sizeof(T);
    return o;
  }
};

const char* kGlobKeys[4] = {"glob.0", "glob.1", "glob.2", "glob.3"};

// Assigns arena offsets to every packed tensor (deterministic: same on every rank).
size_t layout_arena(Ctx* c, char* base) {
  ArenaLayout L;
  auto P = [&](size_t o) { return base ? base + o : nullptr; };
  c->w11 = (float*)P(L.take<float>(36 * 64));
  c->b11 = (float*)P(L.take<float>(64));
  c->wout = (float*)P(L.take<float>(256));
  c->bout = (float*)P(L.take<float>(4));
  for (auto& op : c->ops) {
    op.epi.bias = (float*)P(L.take<float>(op.cout_pad));
    op.epi.scale = (float*)P(L.take<float>(op.cout_pad));
    op.epi.shift = (float*)P(L.take<float>(op.cout_pad));
    const size_t nw = (size_t)op.ncls * op.K * op.cout_pad;
    if (c->simt) {
      op.w_simt = (float*)P(L.take<float>(nw));
    } else {
      op.w_hi = (__half*)P(L.take<__half>(nw));
      op.w_lo = (__half*)P(L.take<__half>(nw));
    }
  }
  if (c->glob) {
    for (int l = 0; l < 4; ++l) {
      const int cin = l == 0 ? 316 : 512;
      c->gw[l] = (float*)P(L.take<float>((size_t)512 * cin));
      c->gb[l] = (float*)P(L.take<float>(512));
      c->gscale[l] = (float*)P(L.take<float>(512));
      c->gshift[l] = (float*)P(L.take<float>(512));
    }
  }
  return (L.off + 255) & ~size_t(255);
}

const HostTensor* find(Ctx* c, const std::string& key) {
  auto it = c->raw.find(key);
  return it == c->raw.end() ? nullptr : &it->second;
}

bool check_dims(const HostTensor* t, std::initializer_list<int64_t> d) {
  if (!t || t->dims.size() != d.size()) return false;
  size_t i = 0;
  for (int64_t v : d)
    if (t->dims[i++] != v) return false;
  return true;
}

void split_f16(float v, __half& hi, __half& lo) {
  hi = __float2half_rn(v);
  lo = __float2half_rn(v - __half2float(hi));
}

// BN(eval) -> y = x*scale + shift   (model.py:17.. ; F.batch_norm with running stats)
void fold_bn(const HostTensor& g, const HostTensor& b, const HostTensor& m, const HostTensor& v, int C, float* scale,
             float* shift) {
  for (int i = 0; i < C; ++i) {
    const double s = (double)g.data[i] / sqrt((double)v.data[i] + (double)kBnEps);
    scale[i] = (float)s;
    shift[i] = (float)((double)b.data[i] - (double)m.data[i] * s);
  }
}

int pack_weights(Ctx* c, char* host) {
  // translate device pointers (already laid out relative to c->arena) to host staging pointers
  auto H = [&](void* dev) { return host + ((char*)dev - c->arena); };
  // conv1_1: [36][64], k = (ky*3+kx)*4 + cin                                       model.py:13
  {
    const HostTensor* w = find(c, "model1.0.weight");
    const HostTensor* b = find(c, "model1.0.bias");
    if (!check_dims(w, {64, 4, 3, 3}) || !check_dims(b, {64})) return fail(c, IDC_ERR_KEY, "missing/bad model1.0.*");
    float* dst = (float*)H(c->w11);
    for (int co = 0; co < 64; ++co)
      for (int ci = 0; ci < 4; ++ci)
        for (int t = 0; t < 9; ++t) dst[(t * 4 + ci) * 64 + co] = w->data[((size_t)co * 4 + ci) * 9 + t];
    memcpy(H(c->b11), b->data.data(), 64 * sizeof(float));
  }
  {
    const HostTensor* w = find(c, "model_out.0.weight");
    const HostTensor* b = find(c, "model_out.0.bias");
    if (!check_dims(w, {2, 128, 1, 1}) || !check_dims(b, {2})) return fail(c, IDC_ERR_KEY, "missing/bad model_out.0.*");
    memcpy(H(c->wout), w->data.data(), 256 * sizeof(float));
    float* bo = (float*)H(c->bout);
    bo[0] = b->data[0]; bo[1] = b->data[1]; bo[2] = bo[3] = 0.f;
  }
  for (auto& op : c->ops) {
    float* bias = (float*)H(op.epi.bias);
    float* scale = (float*)H(op.epi.scale);
    float* shift = (float*)H(op.epi.shift);
    for (int i = 0; i < op.cout_pad; ++i) { bias[i] = 0.f; scale[i] = 1.f; shift[i] = 0.f; }
    const HostTensor* w[kMaxSrc] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    for (int s = 0; s < op.nsrc; ++s) {
      w[s] = find(c, op.wkey[s] + ".weight");
      const HostTensor* b = find(c, op.wkey[s] + ".bias");
      const int cin = op.src[s].cin, k = op.src_k[s];
      const bool ok = op.src_deconv[s] ? check_dims(w[s], {cin, op.cout, k, k}) : check_dims(w[s], {op.cout, cin, k, k});
      if (!ok || !check_dims(b, {op.cout})) return fail(c, IDC_ERR_KEY, "missing/bad %s.*", op.wkey[s].c_str());
      for (int i = 0; i < op.cout; ++i) bias[i] += b->data[i];
    }
    if (op.epi.has_bn) {
      const HostTensor* g = find(c, op.bnkey + ".weight");
      const HostTensor* b = find(c, op.bnkey + ".bias");
      const HostTensor* m = find(c, op.bnkey + ".running_mean");
      const HostTensor* v = find(c, op.bnkey + ".running_var");
      if (!check_dims(g, {op.cout}) || !check_dims(b, {op.cout}) || !check_dims(m, {op.cout}) ||
          !check_dims(v, {op.cout}))
        return fail(c, IDC_ERR_KEY, "missing/bad %s.*", op.bnkey.c_str());
      fold_bn(*g, *b, *m, *v, op.cout, scale, shift);
    }
    // weight value of (class, tap, ci, co)
    auto wval = [&](int cls, int t, int ci, int co) -> float {
      const Tap& tp = op.taps[cls][t];
      const HostTensor* ww = w[tp.src];
      const int cin = op.src[tp.src].cin, k = op.src_k[tp.src];
      if (op.src_deconv[tp.src])  // ConvTranspose2d / Caffe Deconvolution weight is [Cin][Cout][k][k]
        return ww->data[(((size_t)ci * op.cout + co) * k + tp.ky) * k + tp.kx];
      return ww->data[(((size_t)co * cin + ci) * k + tp.ky) * k + tp.kx];
    };
    if (c->simt) {
      float* dst = (float*)H(op.w_simt);
      memset(dst, 0, sizeof(float) * (size_t)op.ncls * op.K * op.cout_pad);
      for (int cls = 0; cls < op.ncls; ++cls) {
        int k0 = 0;
        for (int t = 0; t < op.ntaps; ++t) {
          const int cin = op.src[op.taps[cls][t].src].cin;
          for (int ci = 0; ci < cin; ++ci)
            for (int co = 0; co < op.cout; ++co)
              dst[((size_t)cls * op.K + k0 + ci) * op.cout_pad + co] = wval(cls, t, ci, co);
          k0 += cin;
        }
      }
    } else {
      // K-major FP16 hi/lo rows, one row per (class, cout); per-output-channel power-of-two scale so
      // the lo term stays in FP16's normal range; the epilogue multiplies by 1/scale (exact).
      __half* hi = (__half*)H(op.w_hi);
      __half* lo = (__half*)H(op.w_lo);
      memset(hi, 0, sizeof(__half) * (size_t)op.ncls * op.K * op.cout_pad);
      memset(lo, 0, sizeof(__half) * (size_t)op.ncls * op.K * op.cout_pad);
      for (int co = 0; co < op.cout; ++co) {
        float mx = 0.f;
        for (int cls = 0; cls < op.ncls; ++cls)
          for (int t = 0; t < op.ntaps; ++t) {
            const int cin = op.src[op.taps[cls][t].src].cin;
            for (int ci = 0; ci < cin; ++ci) mx = fmaxf(mx, fabsf(wval(cls, t, ci, co)));
          }
        int e = 0;
        if (mx > 0.f) {
          frexpf(mx, &e);       // mx = f * 2^e, f in [0.5, 1)
          e = 9 - e;            // scaled max in [256, 512)
          e = std::max(-24, std::min(24, e));
        }
        const float sc = ldexpf(1.f, e);
        // acc = sum (a * 2^S)(w * 2^e); stored output = v * 2^Sout  (all exact powers of two)
        const int sout = (op.out_f32 || op.fuse_out_head) ? 0 : kActScaleLog2;
        bias[co] = ldexpf(bias[co], e + kActScaleLog2);
        scale[co] = ldexpf(scale[co], -(e + kActScaleLog2) + sout);
        shift[co] = ldexpf(shift[co], sout);
        for (int cls = 0; cls < op.ncls; ++cls) {
          int k0 = 0;
          for (int t = 0; t < op.ntaps; ++t) {
            const int cin = op.src[op.taps[cls][t].src].cin;
            for (int ci = 0; ci < cin; ++ci) {
              const size_t idx = ((size_t)cls * op.cout_pad + co) * op.K + k0 + ci;
              split_f16(wval(cls, t, ci, co) * sc, hi[idx], lo[idx]);
            }
            k0 += cin;
          }
        }
      }
    }
  }
  if (c->glob) {
    for (int l = 0; l < 4; ++l) {
      const int cin = l == 0 ? 316 : 512;
      const std::string k = kGlobKeys[l];
      const HostTensor* w = find(c, k + ".weight");
      const HostTensor* b = find(c, k + ".bias");
      const HostTensor* g = find(c, k + ".bn.weight");
      const HostTensor* bb = find(c, k + ".bn.bias");
      const HostTensor* m = find(c, k + ".bn.running_mean");
      const HostTensor* v = find(c, k + ".bn.running_var");
      if (!check_dims(w, {512, cin}) || !check_dims(b, {512}) || !check_dims(g, {512}) || !check_dims(bb, {512}) ||
          !check_dims(m, {512}) || !check_dims(v, {512}))
        return fail(c, IDC_ERR_KEY, "missing/bad %s.* (global hints)", k.c_str());
      memcpy(H(c->gw[l]), w->data.data(), sizeof(float) * 512 * cin);
      memcpy(H(c->gb[l]), b->data.data(), sizeof(float) * 512);
      fold_bn(*g, *bb, *m, *v, 512, (float*)H(c->gscale[l]), (float*)H(c->gshift[l]));
    }
  }
  return IDC_OK;
}

int alloc_workspace(Ctx* c) {
  for (auto& b : c->bufs) {
    if (b.H == 0) continue;
    const size_t elems = (size_t)c->max_n * b.H * b.W * b.C;
    if (c->simt) {
      CUDA_TRY(c, cudaMalloc(&b.p0, elems * sizeof(float)));
    } else {
      CUDA_TRY(c, cudaMalloc(&b.p0, elems * sizeof(__half)));
      if (!c->fast) CUDA_TRY(c, cudaMalloc(&b.p1, elems * sizeof(__half)));
    }
  }
  if (c->dist) CUDA_TRY(c, cudaMalloc(&c->logits, sizeof(float) * (size_t)c->max_n * (c->H / 4) * (c->W / 4) * 576));
  if (c->caffe313) {
    CUDA_TRY(c, cudaMalloc(&c->logits313, sizeof(float) * (size_t)c->max_n * (c->H / 4) * (c->W / 4) * 320));
    CUDA_TRY(c, cudaMalloc(&c->pts313, sizeof(float) * 313 * 2));
  }
  for (auto& op : c->ops)
    if (op.out_f32) op.out_f32_ptr = (op.name == "pred313") ? c->logits313 : c->logits;
  if (c->glob) {
    CUDA_TRY(c, cudaMalloc(&c->gvec, sizeof(float) * (size_t)c->max_n * 512));
    CUDA_TRY(c, cudaMalloc(&c->gtmp, sizeof(float) * (size_t)2 * c->max_n * 512));
  }
  CUDA_TRY(c, cudaHostAlloc(&c->h_err, 64, cudaHostAllocMapped));
  memset(c->h_err, 0, 64);
  CUDA_TRY(c, cudaHostGetDevicePointer(&c->d_err, c->h_err, 0));
  return IDC_OK;
}

int plan_engines(Ctx* c) {
  if (c->simt) return IDC_OK;
  c->splitk_ws_floats = 0; c->splitk_max_tiles = 0;
  for (auto& op : c->ops) {
    int rc = umma_plan_op(c, op);
    if (rc != IDC_OK) return rc;
  }
  if (c->splitk_ws) { cudaFree(c->splitk_ws); c->splitk_ws = nullptr; }
  if (c->splitk_counters) { cudaFree(c->splitk_counters); c->splitk_counters = nullptr; }
  if (c->splitk_ws_floats) {
    CUDA_TRY(c, cudaMalloc(&c->splitk_ws, c->splitk_ws_floats * sizeof(float)));
    CUDA_TRY(c, cudaMalloc(&c->splitk_counters, sizeof(int) * 2 * (size_t)c->splitk_max_tiles));
    CUDA_TRY(c, cudaMemset(c->splitk_counters, 0, sizeof(int) * 2 * (size_t)c->splitk_max_tiles));
  }
  return IDC_OK;
}

// idc_forward_host's copy/compute overlap: the batch is cut into image chunks; conv1_1 of chunk k waits for the
// H2D of chunk k only (issued on Ctx::s_in), and the last op (c10_2 + fused model_out) runs per chunk so that the
// D2H of ab chunk k (on Ctx::s_out) overlaps the compute of chunk k+1.  Everything in between runs on the whole batch.
struct HostPipe {
  static constexpr int kMaxChunks = 8;   // == the size of Ctx::ev_in / ev_out
  int nchunks = 0;
  int start[kMaxChunks + 1] = {};        // image ranges [start[k], start[k+1])
  float* ab_dst = nullptr;    // pinned host destination of out_ab (caller's buffer or the staging block)
};

// idc_set_click: layout of the click answer block (device d_clickout, pinned host h_clickout)
constexpr int kClickInit = 8, kClickMaxIter = 100;                       // the defaults of LhnContext.ab_reccs
constexpr size_t kClickHdr = 32, kClickPmf = 544 * sizeof(float);
constexpr size_t kClickRes = (size_t)kClickInit * (3 * 32 + 2) * sizeof(double);
constexpr size_t kClickCopy = kClickHdr + kClickPmf + kClickRes;         // what travels back per click
constexpr size_t kClickBytes = kClickCopy + 529 * 2 * sizeof(float);     // + the default gamut grid (device only)

// After the class conv of a small-batch forward: the clicked pixel's pmf straight from its 529 logits (same per-row
// softmax routine as the full map, so the same bits), K-means on it (K from the click header), the block to pinned host
// memory.  Runs next to the full-map softmax on a branch of the dist head's side branch.
bool click_tail_on(Ctx* c, int n) { return c->click_mode && c->d_clickout && n <= 4; }

cudaError_t click_tail(Ctx* c, int n, cudaStream_t st) {
  if (!click_tail_on(c, n)) return cudaSuccess;
  int* hdr = reinterpret_cast<int*>(c->d_clickout);
  float* pmf = reinterpret_cast<float*>(c->d_clickout + kClickHdr);
  double* res = reinterpret_cast<double*>(c->d_clickout + kClickHdr + kClickPmf);
  const float* pts = reinterpret_cast<const float*>(c->d_clickout + kClickCopy);
  cudaError_t e = launch_click_pmf(c, c->d_click, n, hdr, pmf, st);
  if (e != cudaSuccess) return e;
  if ((e = launch_ab_reccs(pmf, 1, pts, 0, kClickMaxIter, kClickInit, res, st, hdr)) != cudaSuccess) return e;
  c->launch_count += 2;
  return cudaMemcpyAsync(c->h_clickout, c->d_clickout, kClickCopy, cudaMemcpyDeviceToHost, st);
}

// persistent-grid cap (CTAs, even) that leaves kClickInit SMs to the side branch
int side_branch_cap(Ctx* c) {
  cudaDeviceProp prop;
  static int sms[64] = {};
  int& n = sms[c->dev < 64 ? c->dev : 0];
  if (!n) { cudaGetDeviceProperties(&prop, c->dev); n = prop.multiProcessorCount; }
  return ((n - kClickInit) / 2) * 2;
}

int run_forward(Ctx* c, int n, const float* L, const float* ab, const float* mask, float maskcent, const float* glob,
                float* out_ab, float* out_dist, uint8_t* out_rgb, cudaStream_t st, const HostPipe* hp = nullptr,
                double* out_abq = nullptr) {
  c->launch_count = 0;
  c->gadd_active = false;
  c->click_served = false;
  pdl_break(c);                        // whatever precedes this forward on `st` is not one of its kernels
  std::vector<cudaEvent_t>* ev = nullptr;
  auto mark = [&]() {
    if (!ev) return;
    cudaEvent_t e;
    if (!c->prof_pool.empty()) { e = c->prof_pool.back(); c->prof_pool.pop_back(); }
    else cudaEventCreate(&e);
    cudaEventRecord(e, st);
    ev->push_back(e);
    pdl_break(c);                      // per-op timing: kernels must not overlap their predecessors
  };
  if (c->profiling) { c->prof_runs.emplace_back(); ev = &c->prof_runs.back(); }
  mark();
  if (hp) CUDA_TRY(c, cudaStreamWaitEvent(st, c->ev_in[0], 0));     // covers the glob vector too
  if (glob && c->glob) {
    CUDA_TRY(c, launch_global_mlp(c, n, glob, st));
    c->gadd_active = true;
  }
  const size_t HW = (size_t)c->H * c->W;
  const bool c11_umma = c->opt.conv1_1_umma && !c->simt && c->w11_umma;
  if (hp) {
    for (int k = 0; k < hp->nchunks; ++k) {
      CUDA_TRY(c, cudaStreamWaitEvent(st, c->ev_in[k], 0));
      pdl_break(c);
      if (c11_umma) CUDA_TRY(c, launch_conv1_1_umma(c, hp->start[k + 1] - hp->start[k], L, ab, mask, maskcent, st, hp->start[k]));
      else CUDA_TRY(c, launch_conv1_1(c, hp->start[k + 1] - hp->start[k], L, ab, mask, maskcent, st, hp->start[k]));
    }
  } else {
    if (c11_umma) CUDA_TRY(c, launch_conv1_1_umma(c, n, L, ab, mask, maskcent, st));
    else CUDA_TRY(c, launch_conv1_1(c, n, L, ab, mask, maskcent, st));
  }
  mark();
  // Interactive batches: the dist head (class 1x1 conv + 529-way softmax) only depends on conv8_3, and decoder levels
  // 9-10 do not depend on it -> it runs on a side stream (a parallel branch of the click graph) on the ~20 SMs the
  // 128-CTA launches of the main chain leave idle, instead of sitting between c8_3 and up9 on the critical path.
  const bool side_dist = c->opt.side_dist && !c->simt && out_dist && n <= 4 && !hp && !ev;
  bool forked = false;
  for (size_t oi = 0; oi < c->ops.size(); ++oi) {
    ConvOp& op = c->ops[oi];
    if (side_dist && op.kind == OP_CLASS && op.name == "class") {
      if (!c->s_side) {
        CUDA_TRY(c, cudaStreamCreateWithFlags(&c->s_side, cudaStreamNonBlocking));
        CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
        CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
      }
      cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
      CUDA_TRY(c, cudaStreamIsCapturing(st, &cap));
      const bool main_chain = c->chain;
      CUDA_TRY(c, cudaEventRecord(c->ev_fork, st));
      CUDA_TRY(c, cudaStreamWaitEvent(c->s_side, c->ev_fork, 0));
      pdl_break(c);                                        // first kernel of the branch follows an event wait
      CUDA_TRY(c, umma_run_op(c, op, n, nullptr, (float)c->opt.tanh_scale, c->s_side, 0, 16));
      const bool click = click_tail_on(c, n);
      if (click) {   // idc_set_click: clicked pixel's pmf + suggestions only need the logits -> a branch of the branch
        if (!c->s_click) {
          CUDA_TRY(c, cudaStreamCreateWithFlags(&c->s_click, cudaStreamNonBlocking));
          CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_click[0], cudaEventDisableTiming));
          CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_click[1], cudaEventDisableTiming));
        }
        CUDA_TRY(c, cudaEventRecord(c->ev_click[0], c->s_side));
        CUDA_TRY(c, cudaStreamWaitEvent(c->s_click, c->ev_click[0], 0));
        CUDA_TRY(c, click_tail(c, n, c->s_click));
        CUDA_TRY(c, cudaEventRecord(c->ev_click[1], c->s_click));
        if (cap != cudaStreamCaptureStatusActive) pdl_break(c);      // live stream: the record sits between class and softmax
      }
      CUDA_TRY(c, launch_softmax529(c, n, out_dist, c->s_side));     // PDL-chained behind `class` on the side stream
      if (click) CUDA_TRY(c, cudaStreamWaitEvent(c->s_side, c->ev_click[1], 0));
      CUDA_TRY(c, cudaEventRecord(c->ev_join, c->s_side));
      // in a capture the event record is not a node: up9 keeps its programmatic edge to c8_3; on a live stream the
      // record sits between the two kernels, so the next launch is serialised normally
      c->chain = (cap == cudaStreamCaptureStatusActive) ? main_chain : false;
      forked = true;
      continue;
    }
    if (c->simt) {
      CUDA_TRY(c, simt_run_op(c, op, n, st));
    } else if (hp && op.fuse_out_head) {
      for (int k = 0; k < hp->nchunks; ++k) {
        const int i0 = hp->start[k], nk = hp->start[k + 1] - i0;
        CUDA_TRY(c, umma_run_op(c, op, nk, out_ab, (float)c->opt.tanh_scale, st, i0));
        CUDA_TRY(c, cudaEventRecord(c->ev_out[k], st));
        pdl_break(c);
        CUDA_TRY(c, cudaStreamWaitEvent(c->s_out, c->ev_out[k], 0));
        CUDA_TRY(c, cudaMemcpyAsync(hp->ab_dst + (size_t)i0 * 2 * HW, out_ab + (size_t)i0 * 2 * HW,
                                    (size_t)nk * 2 * HW * sizeof(float), cudaMemcpyDeviceToHost, c->s_out));
      }
    } else {
      // announced click: the suggestion kernel (8 CTAs of 1024 threads, a whole SM each) runs on the side branch next
      // to decoder levels 9-10; a 148-CTA launch would queue behind it on 8 SMs and finish that much later.  Leaving 8
      // SMs free costs nothing: 512 tiles are 4 rounds on 148 and on 140 CTAs alike.
      const int cap = (forked && c->click_mode && c->d_clickout) ? side_branch_cap(c) : 0;
      CUDA_TRY(c, umma_run_op(c, op, n, op.fuse_out_head ? out_ab : nullptr, (float)c->opt.tanh_scale, st, 0, cap));
    }
    mark();
  }
  const bool fused = !c->simt && !(c->flags & IDC_FLAG_KEEP_CONV10);
  if (!fused) CUDA_TRY(c, launch_out_head(c, n, out_ab, st));
  if (out_dist && !forked) {
    CUDA_TRY(c, launch_softmax529(c, n, out_dist, st));
    CUDA_TRY(c, click_tail(c, n, st));
    pdl_break(c);
  }
  if (out_rgb) {
    CUDA_TRY(c, launch_lab2rgb(c, n, c->H, c->W, L, 50.0f, out_ab, out_rgb, st, out_abq));
    c->launch_count++;
  }
  if (forked) {
    CUDA_TRY(c, cudaStreamWaitEvent(st, c->ev_join, 0));   // join: whatever follows on `st` sees the distribution
    pdl_break(c);
  }
  mark();
  pdl_break(c);
  c->last_n = n;
  return IDC_OK;
}

int check_forward_args(Ctx* c, int n, int h, int w, const void* L, const void* ab, const void* mask, const void* glob,
                       const void* out_ab, const void* out_dist, bool resident_l_ok = false) {
  if (!c->weights_ready) return fail(c, IDC_ERR_STATE, "idc_forward before idc_finalize_weights");
  if (n < 1 || n > c->max_n) return fail(c, IDC_ERR_ARG, "n=%d outside [1,%d]", n, c->max_n);
  if (h != c->H || w != c->W) return fail(c, IDC_ERR_ARG, "geometry %dx%d != ctx geometry %dx%d", h, w, c->H, c->W);
  if ((!L && !resident_l_ok) || !ab || !mask || !out_ab) return fail(c, IDC_ERR_ARG, "null L/ab/mask/out_ab");
  if (out_dist && !c->dist) return fail(c, IDC_ERR_ARG, "out_dist requires IDC_FLAG_DIST");
  if (glob && !c->glob) return fail(c, IDC_ERR_ARG, "glob requires IDC_FLAG_GLOBAL_HINTS");
  return IDC_OK;
}

}  // namespace

// =============================================================================================
extern "C" {

const char* idc_version(void) { return "idc_b200 0.1 sm_100a (tcgen05 split-fp16 + fp32 simt engines)"; }

int idc_create(int device, int max_n, int h, int w, unsigned flags, idc_ctx** out) {
  if (!out) return IDC_ERR_ARG;
  *out = nullptr;
  if (max_n < 1 || h < 8 || w < 8 || (h % 8) || (w % 8)) return IDC_ERR_ARG;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return IDC_ERR_CUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return IDC_ERR_CUDA;
  if (prop.major != 10) return IDC_ERR_UNSUPPORTED;  // sm_100a cubins only; no fallback
  if (cudaSetDevice(device) != cudaSuccess) return IDC_ERR_CUDA;
  idc_ctx* c = new idc_ctx();
  c->dev = device; c->max_n = max_n; c->H = h; c->W = w; c->flags = flags;
  c->simt = flags & IDC_FLAG_ENGINE_SIMT;
  c->fast = (flags & IDC_FLAG_FAST_FP16) && !c->simt;
  c->dist = flags & IDC_FLAG_DIST;
  c->glob = flags & IDC_FLAG_GLOBAL_HINTS;
  c->caffe313 = flags & IDC_FLAG_CAFFE313;
  build_plan(c);
  int rc = alloc_workspace(c);
  if (rc != IDC_OK) {
    fprintf(stderr, "idc_create: %s\n", c->err.c_str());
    idc_destroy(c);
    return rc;
  }
  cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking);
  *out = c;
  return IDC_OK;
}

int idc_set_option(idc_ctx* c, const char* name, int value) {
  if (!c || !name) return IDC_ERR_ARG;
  struct { const char* n; int* v; } tab[] = {
      {"halo", &c->opt.halo}, {"pairs", &c->opt.pairs}, {"mt", &c->opt.mt}, {"chunk_kb", &c->opt.chunk_kb},
      {"split_k", &c->opt.split_k}, {"host_pipe", &c->opt.host_pipe},
      {"pdl", &c->opt.pdl}, {"split_pairs", &c->opt.split_pairs}, {"tanh_scale", &c->opt.tanh_scale},
      {"side_dist", &c->opt.side_dist}, {"split_bn128", &c->opt.split_bn128}, {"conv1_1_umma", &c->opt.conv1_1_umma}};
  for (auto& t : tab)
    if (!strcmp(t.n, name)) {
      *t.v = value;
      if (c->weights_ready && strcmp(name, "host_pipe") && strcmp(name, "tanh_scale") && strcmp(name, "side_dist") && strcmp(name, "conv1_1_umma")) {      // plan-time option changed after planning: re-plan
        CUDA_TRY(c, cudaSetDevice(c->dev));
        CUDA_TRY(c, cudaDeviceSynchronize());
        int rc = plan_engines(c);
        if (rc != IDC_OK) return rc;
      }
      if (c->graph_exec) { cudaGraphExecDestroy(c->graph_exec); c->graph_exec = nullptr; }
      return IDC_OK;
    }
  return fail(c, IDC_ERR_KEY, "unknown option '%s'", name);
}

int idc_load_tensor(idc_ctx* c, const char* key, const void* data, int dtype, int ndim, const int64_t* dims) {
  if (!c || !key || !data || ndim < 0 || ndim > 8 || (ndim && !dims)) return fail(c, IDC_ERR_ARG, "bad load_tensor args");
  HostTensor t;
  size_t count = 1;
  for (int i = 0; i < ndim; ++i) {
    if (dims[i] < 0) return fail(c, IDC_ERR_ARG, "negative dim");
    t.dims.push_back(dims[i]);
    count *= (size_t)dims[i];
  }
  t.data.resize(count);
  switch (dtype) {
    case IDC_F32: memcpy(t.data.data(), data, count * sizeof(float)); break;
    case IDC_F64: for (size_t i = 0; i < count; ++i) t.data[i] = (float)((const double*)data)[i]; break;
    case IDC_I64: for (size_t i = 0; i < count; ++i) t.data[i] = (float)((const int64_t*)data)[i]; break;
    default: return fail(c, IDC_ERR_ARG, "unknown dtype %d", dtype);
  }
  c->raw[key] = std::move(t);
  c->weights_ready = false;
  return IDC_OK;
}

int idc_reserve_weights(idc_ctx* c) {
  if (!c) return IDC_ERR_ARG;
  CUDA_TRY(c, cudaSetDevice(c->dev));
  if (!c->arena) {
    c->arena_bytes = layout_arena(c, nullptr);
    CUDA_TRY(c, cudaMalloc(&c->arena, c->arena_bytes));
    layout_arena(c, c->arena);
  }
  return IDC_OK;
}

int idc_finalize_weights(idc_ctx* c) {
  if (!c) return IDC_ERR_ARG;
  int rc = idc_reserve_weights(c);
  if (rc != IDC_OK) return rc;
  std::vector<char> host(c->arena_bytes, 0);
  rc = pack_weights(c, host.data());
  if (rc != IDC_OK) return rc;
  if (c->caffe313) {
    const HostTensor* pts = find(c, "caffe.pts_in_hull");
    if (!check_dims(pts, {313, 2})) return fail(c, IDC_ERR_KEY, "missing/bad caffe.pts_in_hull [313,2]");
    CUDA_TRY(c, cudaMemcpy(c->pts313, pts->data.data(), sizeof(float) * 626, cudaMemcpyHostToDevice));
  }
  CUDA_TRY(c, cudaMemcpy(c->arena, host.data(), c->arena_bytes, cudaMemcpyHostToDevice));
  return idc_adopt_weights(c);
}

int idc_adopt_weights(idc_ctx* c) {
  if (!c || !c->arena) return fail(c, IDC_ERR_STATE, "no arena");
  CUDA_TRY(c, cudaSetDevice(c->dev));
  int rc = plan_engines(c);
  if (rc != IDC_OK) return rc;
  // conv1_1 takes its weights as a kernel parameter: read them back from the (possibly received) arena
  CUDA_TRY(c, cudaMemcpy(c->h_w11.w, c->w11, sizeof(c->h_w11.w), cudaMemcpyDeviceToHost));
  CUDA_TRY(c, cudaMemcpy(c->h_w11.b, c->b11, sizeof(c->h_w11.b), cudaMemcpyDeviceToHost));
  if (!c->simt) CUDA_TRY(c, conv1_1_umma_pack(c));      // tensor-core conv1_1: derived on the device, so ranks != 0 need nothing extra
  c->raw.clear();
  c->weights_ready = true;
  if (c->graph_exec) { cudaGraphExecDestroy(c->graph_exec); c->graph_exec = nullptr; }
  return IDC_OK;
}

int idc_weights_arena(idc_ctx* c, void** dev_ptr, size_t* bytes) {
  if (!c || !dev_ptr || !bytes) return IDC_ERR_ARG;
  if (!c->arena) return fail(c, IDC_ERR_STATE, "arena not allocated");
  *dev_ptr = c->arena; *bytes = c->arena_bytes;
  return IDC_OK;
}

int idc_forward(idc_ctx* c, int n, int h, int w, const float* L, const float* ab, const float* mask, float maskcent,
                const float* glob, float* out_ab, float* out_dist, uint8_t* out_rgb, void* stream) {
  if (!c) return IDC_ERR_ARG;
  int rc = check_forward_args(c, n, h, w, L, ab, mask, glob, out_ab, out_dist);
  if (rc != IDC_OK) return rc;
  CUDA_TRY(c, cudaSetDevice(c->dev));
  if (int werr = *(volatile int*)c->h_err) {           // left by an earlier (asynchronous) forward
    *(volatile int*)c->h_err = 0;
    return fail(c, IDC_ERR_WATCHDOG, "device pipeline watchdog fired earlier (code %d)", werr);
  }
  return run_forward(c, n, L, ab, mask, maskcent, glob, out_ab, out_dist, out_rgb, (cudaStream_t)stream);
}

static bool is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}

int idc_forward_host(idc_ctx* c, int n, int h, int w, const float* L, const float* ab, const float* mask,
                     float maskcent, const float* glob, float* out_ab, float* out_dist, uint8_t* out_rgb) {
  return idc_forward_host_q(c, n, h, w, L, ab, mask, maskcent, glob, out_ab, out_dist, out_rgb, nullptr);
}

// Small batches (the interactive click): ONE graph launch does everything -- the H2D of the inputs, the kernels
// (chained by programmatic dependent launch), the D2H of the results.
//   * pinned caller buffers (idc_host_alloc; see LhnContext.click_buffers): the copy nodes read / write the caller's
//     memory directly -- no CPU copy at all.  Buffers laid out back to back ([L | ab | mask | glob], [ab | rgb | abq])
//     travel as ONE copy each way.  The graph is keyed on the pointers and re-captured when they change.
//   * pageable caller buffers: staged through the context's pinned blocks by the CPU (one copy node each way).
static int forward_host_small(idc_ctx* c, int n, const float* L, const float* ab, const float* mask, float maskcent,
                              const float* glob, float* out_ab, float* out_dist, uint8_t* out_rgb, double* out_abq) {
  const size_t HW = (size_t)c->H * c->W, HW4 = (size_t)(c->H / 4) * (c->W / 4);
  cudaStream_t st = c->own_stream;
  const bool copy_dist = out_dist != nullptr;
  const bool want_dist = copy_dist || (c->dist_resident && c->dist);
  const bool want_rgb = out_rgb != nullptr, want_glob = glob != nullptr, want_q = out_abq != nullptr;
  // compact device layouts for this n
  float* dL = c->d_in; float* dab = dL + (size_t)n * HW; float* dmask = dab + (size_t)n * 2 * HW;
  float* dglob = dmask + (size_t)n * HW;
  const size_t b_ab = (size_t)n * 2 * HW * sizeof(float), b_rgb = (size_t)n * 3 * HW, b_q = (size_t)n * 2 * HW * sizeof(double);
  char* dsm = c->d_small; char* hsm = c->h_small;
  float* dout = reinterpret_cast<float*>(dsm);
  uint8_t* drgb = reinterpret_cast<uint8_t*>(dsm + b_ab);
  double* dq = reinterpret_cast<double*>(dsm + b_ab + b_rgb);
  float* ddist = c->d_out + (size_t)c->max_n * 2 * HW;
  const size_t out_bytes = b_ab + (want_rgb ? b_rgb : 0) + (want_q ? b_q : 0);
  const uintptr_t flags = (uintptr_t)n | ((uintptr_t)want_dist << 8) | ((uintptr_t)want_rgb << 9) | ((uintptr_t)want_glob << 10) |
                          ((uintptr_t)want_q << 11) | ((uintptr_t)copy_dist << 12) | ((uintptr_t)c->click_mode << 13);
  c->click_served = false;
  const bool have_L = L != nullptr;          // false: the image set by idc_set_image stays where it is
  const size_t in_floats = (size_t)n * (have_L ? 4 : 3) * HW + (want_glob ? (size_t)n * 316 : 0);
  const void* direct_key[8] = {(void*)(flags | (1u << 16)), L, ab, mask, glob, out_ab, out_rgb, out_abq};
  // fast path: same pinned buffers as the captured graph -> replay without touching the driver's pointer tables
  bool direct = c->graph_exec && !copy_dist && memcmp(direct_key, c->graph_ptrs, sizeof(direct_key)) == 0 &&
                c->graph_maskcent == maskcent;
  bool replay = direct;
  if (!direct) {
    direct = !copy_dist && (!have_L || is_pinned(L)) && is_pinned(ab) && is_pinned(mask) && (!glob || is_pinned(glob)) &&
             is_pinned(out_ab) && (!out_rgb || is_pinned(out_rgb)) && (!out_abq || is_pinned(out_abq));
  }
  const void* staged_key[8] = {(void*)(flags | ((uintptr_t)have_L << 17)), nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  const void** key = direct ? direct_key : staged_key;
  if (!direct) {   // stage the inputs
    if (have_L) memcpy(c->h_in, L, (size_t)n * HW * sizeof(float));
    memcpy(c->h_in + (size_t)n * HW, ab, (size_t)n * 2 * HW * sizeof(float));
    memcpy(c->h_in + (size_t)n * 3 * HW, mask, (size_t)n * HW * sizeof(float));
    if (want_glob) memcpy(c->h_in + (size_t)n * 4 * HW, glob, (size_t)n * 316 * sizeof(float));
  }
  if (!replay && (!c->graph_exec || memcmp(key, c->graph_ptrs, sizeof(staged_key)) != 0 || c->graph_maskcent != maskcent)) {
    if (c->graph_exec) { cudaGraphExecDestroy(c->graph_exec); c->graph_exec = nullptr; }
    cudaGraph_t g = nullptr;
    CUDA_TRY(c, cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    const bool prof = c->profiling;
    c->profiling = false;            // event timing is meaningless inside a capture
    cudaError_t ce = cudaSuccess;
    auto cp = [&](void* dst, const void* src, size_t bytes, cudaMemcpyKind kind) {
      if (ce == cudaSuccess && bytes) ce = cudaMemcpyAsync(dst, src, bytes, kind, st);
    };
    if (direct) {
      const bool contig = (!have_L || ab == L + (size_t)n * HW) && mask == ab + (size_t)n * 2 * HW &&
                          (!want_glob || glob == mask + (size_t)n * HW);
      if (contig) {
        cp(have_L ? dL : dab, have_L ? L : ab, in_floats * sizeof(float), cudaMemcpyHostToDevice);
      } else {
        if (have_L) cp(dL, L, (size_t)n * HW * sizeof(float), cudaMemcpyHostToDevice);
        cp(dab, ab, (size_t)n * 2 * HW * sizeof(float), cudaMemcpyHostToDevice);
        cp(dmask, mask, (size_t)n * HW * sizeof(float), cudaMemcpyHostToDevice);
        if (want_glob) cp(dglob, glob, (size_t)n * 316 * sizeof(float), cudaMemcpyHostToDevice);
      }
    } else {
      const size_t off = have_L ? 0 : (size_t)n * HW;
      cp(c->d_in + off, c->h_in + off, in_floats * sizeof(float), cudaMemcpyHostToDevice);
    }
    int rc = IDC_OK;
    if (ce == cudaSuccess)
      rc = run_forward(c, n, dL, dab, dmask, maskcent, want_glob ? dglob : nullptr, dout, want_dist ? ddist : nullptr,
                       want_rgb ? drgb : nullptr, st, nullptr, want_q ? dq : nullptr);
    if (rc == IDC_OK) {
      if (direct) {
        const char* o0 = reinterpret_cast<const char*>(out_ab);
        const bool contig = (!want_rgb || reinterpret_cast<const char*>(out_rgb) == o0 + b_ab) &&
                            (!want_q || reinterpret_cast<const char*>(out_abq) == o0 + b_ab + b_rgb);
        if (contig) {
          cp(out_ab, dsm, out_bytes, cudaMemcpyDeviceToHost);
        } else {
          cp(out_ab, dout, b_ab, cudaMemcpyDeviceToHost);
          if (want_rgb) cp(out_rgb, drgb, b_rgb, cudaMemcpyDeviceToHost);
          if (want_q) cp(out_abq, dq, b_q, cudaMemcpyDeviceToHost);
        }
      } else {
        cp(hsm, dsm, out_bytes, cudaMemcpyDeviceToHost);
        if (copy_dist)
          cp(c->h_out + (size_t)c->max_n * 2 * HW, ddist, (size_t)n * 529 * HW4 * sizeof(float), cudaMemcpyDeviceToHost);
      }
    }
    c->profiling = prof;
    cudaError_t ce2 = cudaStreamEndCapture(st, &g);
    if (rc != IDC_OK) { if (g) cudaGraphDestroy(g); return rc; }
    if (ce != cudaSuccess) { if (g) cudaGraphDestroy(g); CUDA_TRY(c, ce); }
    CUDA_TRY(c, ce2);
    ce = cudaGraphInstantiate(&c->graph_exec, g, 0);
    cudaGraphDestroy(g);
    CUDA_TRY(c, ce);
    memcpy(c->graph_ptrs, key, sizeof(staged_key));
    c->graph_maskcent = maskcent;
    c->graph_launches = c->launch_count;
  }
  if (c->dbg_graph_timing) CUDA_TRY(c, cudaEventRecord(c->dbg_ev[0], st));
  CUDA_TRY(c, cudaGraphLaunch(c->graph_exec, st));
  if (c->dbg_graph_timing) CUDA_TRY(c, cudaEventRecord(c->dbg_ev[1], st));
  c->launch_count = c->graph_launches;
  c->last_n = n;
  CUDA_TRY(c, cudaStreamSynchronize(st));
  if (c->dbg_graph_timing) cudaEventElapsedTime(&c->dbg_graph_ms, c->dbg_ev[0], c->dbg_ev[1]);
  if (!direct) {
    memcpy(out_ab, hsm, b_ab);
    if (want_rgb) memcpy(out_rgb, hsm + b_ab, b_rgb);
    if (want_q) memcpy(out_abq, hsm + b_ab + b_rgb, b_q);
    if (copy_dist) memcpy(out_dist, c->h_out + (size_t)c->max_n * 2 * HW, (size_t)n * 529 * HW4 * sizeof(float));
  }
  c->dist_valid_n = want_dist ? n : 0;
  c->click_served = want_dist && c->click_mode && c->h_clickout;     // the side branch delivered the click's answer
  if (have_L) c->image_n = n;          // the planes just uploaded are the resident image now
  return IDC_OK;
}

static int ensure_host_staging(idc_ctx* c) {
  if (c->d_in) return IDC_OK;
  const size_t HW = (size_t)c->H * c->W, HW4 = (size_t)(c->H / 4) * (c->W / 4);
  const int small_n = c->max_n < 4 ? c->max_n : 4;
  c->in_floats = (size_t)c->max_n * (4 * HW + 316);
  c->out_floats = (size_t)c->max_n * (2 * HW + (c->dist ? 529 * HW4 : 0));
  const size_t small_bytes = (size_t)small_n * (2 * HW * 4 + 3 * HW + 2 * HW * 8);
  CUDA_TRY(c, cudaMalloc(&c->d_in, c->in_floats * sizeof(float)));
  CUDA_TRY(c, cudaMalloc(&c->d_out, c->out_floats * sizeof(float)));
  CUDA_TRY(c, cudaMalloc(&c->d_rgb, (size_t)c->max_n * HW * 3));
  CUDA_TRY(c, cudaMalloc(&c->d_small, small_bytes));
  CUDA_TRY(c, cudaMallocHost(&c->h_in, c->in_floats * sizeof(float)));
  CUDA_TRY(c, cudaMallocHost(&c->h_out, c->out_floats * sizeof(float)));
  CUDA_TRY(c, cudaMallocHost(&c->h_rgb, (size_t)c->max_n * HW * 3));
  CUDA_TRY(c, cudaMallocHost(&c->h_small, small_bytes));
  return IDC_OK;
}

int idc_set_image(idc_ctx* c, int n, int h, int w, const float* L) {
  if (!c) return IDC_ERR_ARG;
  if (n < 0 || n > c->max_n) return fail(c, IDC_ERR_ARG, "n=%d outside [0,%d]", n, c->max_n);
  if (n == 0 || !L) { c->image_n = 0; return IDC_OK; }
  if (h != c->H || w != c->W) return fail(c, IDC_ERR_ARG, "geometry %dx%d != ctx geometry %dx%d", h, w, c->H, c->W);
  CUDA_TRY(c, cudaSetDevice(c->dev));
  int rc = ensure_host_staging(c);
  if (rc != IDC_OK) return rc;
  c->image_n = 0;
  CUDA_TRY(c, cudaStreamSynchronize(c->own_stream));
  // the L planes sit at the head of the input block for every batch size (small and large path alike)
  CUDA_TRY(c, cudaMemcpy(c->d_in, L, (size_t)n * c->H * c->W * sizeof(float), cudaMemcpyHostToDevice));
  c->image_n = n;
  return IDC_OK;
}

int idc_forward_host_q(idc_ctx* c, int n, int h, int w, const float* L, const float* ab, const float* mask,
                       float maskcent, const float* glob, float* out_ab, float* out_dist, uint8_t* out_rgb,
                       double* out_abq) {
  if (!c) return IDC_ERR_ARG;
  int rc = check_forward_args(c, n, h, w, L, ab, mask, glob, out_ab, out_dist, /*resident_l_ok=*/true);   // NULL L: idc_set_image
  if (rc != IDC_OK) return rc;
  if (out_abq && !out_rgb) return fail(c, IDC_ERR_ARG, "out_abq (quantised ab) is derived from out_rgb: pass both");
  CUDA_TRY(c, cudaSetDevice(c->dev));
  if (int werr = *(volatile int*)c->h_err) {           // a watchdog left over from an asynchronous idc_forward
    *(volatile int*)c->h_err = 0;
    return fail(c, IDC_ERR_WATCHDOG, "device pipeline watchdog fired earlier (code %d)", werr);
  }
  const size_t HW = (size_t)c->H * c->W, HW4 = (size_t)(c->H / 4) * (c->W / 4);
  rc = ensure_host_staging(c);
  if (rc != IDC_OK) return rc;
  if (!L && c->image_n != n)
    return fail(c, IDC_ERR_STATE, "L_mc is NULL but no %d-image set is resident (idc_set_image)", n);
  const bool use_graph = !(c->flags & IDC_FLAG_NO_GRAPH) && n <= 4;
  if (use_graph) {
    rc = forward_host_small(c, n, L, ab, mask, maskcent, glob, out_ab, out_dist, out_rgb, out_abq);
    if (rc != IDC_OK) return rc;
    if (int werr = *(volatile int*)c->h_err) {
      *(volatile int*)c->h_err = 0;
      return fail(c, IDC_ERR_WATCHDOG, "device pipeline watchdog fired (code %d)", werr);
    }
    return IDC_OK;
  }
  if (out_abq && !c->d_abq) {
    CUDA_TRY(c, cudaMalloc(&c->d_abq, (size_t)c->max_n * 2 * HW * sizeof(double)));
    CUDA_TRY(c, cudaMallocHost(&c->h_abq, (size_t)c->max_n * 2 * HW * sizeof(double)));
  }
  cudaStream_t st = c->own_stream;
  // device-side layout of the staging block: [L | ab | mask | glob], [out_ab | out_dist]
  float* dL = c->d_in; float* dab = dL + (size_t)c->max_n * HW; float* dmask = dab + (size_t)c->max_n * 2 * HW;
  float* dglob = dmask + (size_t)c->max_n * HW;
  float* dout = c->d_out; float* ddist = dout + (size_t)c->max_n * 2 * HW;
  auto h2d = [&](float* d, const float* src, size_t count, size_t stage_off) -> cudaError_t {
    const float* s = src;
    if (!is_pinned(src)) {   // pageable caller memory: stage through our pinned block
      memcpy(c->h_in + stage_off, src, count * sizeof(float));
      s = c->h_in + stage_off;
    }
    return cudaMemcpyAsync(d, s, count * sizeof(float), cudaMemcpyHostToDevice, st);
  };
  // large batches: chunked copy/compute overlap (see HostPipe); option host_pipe=0 turns it off for A/B runs
  const bool pipe_on = c->opt.host_pipe != 0;
  const bool fused_head = !c->simt && !(c->flags & IDC_FLAG_KEEP_CONV10);
  HostPipe hp;
  bool last_splits = false;
  for (auto& op : c->ops) if (op.fuse_out_head) last_splits = umma_op_uses_split_k(op);
  if (pipe_on && n >= 8 && fused_head && !last_splits && !c->profiling) {
    hp.nchunks = n >= 32 ? 4 : 2;   // measured: 8 chunks at n = 64 is 1.3 % slower end to end than 4
    for (int k = 0; k <= hp.nchunks; ++k) hp.start[k] = (int)((long long)n * k / hp.nchunks);
    hp.ab_dst = is_pinned(out_ab) ? out_ab : c->h_out;
    if (!c->s_in) {
      CUDA_TRY(c, cudaStreamCreateWithFlags(&c->s_in, cudaStreamNonBlocking));
      CUDA_TRY(c, cudaStreamCreateWithFlags(&c->s_out, cudaStreamNonBlocking));
      for (int k = 0; k < HostPipe::kMaxChunks; ++k) {
        CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_in[k], cudaEventDisableTiming));
        CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_out[k], cudaEventDisableTiming));
      }
    }
  }
  if (hp.nchunks) {
    cudaStream_t compute = st;
    st = c->s_in;                                   // the h2d lambda copies on `st`
    if (glob) CUDA_TRY(c, h2d(dglob, glob, (size_t)n * 316, (size_t)c->max_n * 4 * HW));
    for (int k = 0; k < hp.nchunks; ++k) {
      const size_t i0 = hp.start[k], nk = hp.start[k + 1] - hp.start[k];
      if (L) CUDA_TRY(c, h2d(dL + i0 * HW, L + i0 * HW, nk * HW, i0 * HW));
      CUDA_TRY(c, h2d(dab + i0 * 2 * HW, ab + i0 * 2 * HW, nk * 2 * HW, (size_t)c->max_n * HW + i0 * 2 * HW));
      CUDA_TRY(c, h2d(dmask + i0 * HW, mask + i0 * HW, nk * HW, (size_t)c->max_n * 3 * HW + i0 * HW));
      CUDA_TRY(c, cudaEventRecord(c->ev_in[k], c->s_in));
    }
    st = compute;
  } else {
    if (L) CUDA_TRY(c, h2d(dL, L, n * HW, 0));
    CUDA_TRY(c, h2d(dab, ab, n * 2 * HW, (size_t)c->max_n * HW));
    CUDA_TRY(c, h2d(dmask, mask, n * HW, (size_t)c->max_n * 3 * HW));
    if (glob) CUDA_TRY(c, h2d(dglob, glob, (size_t)n * 316, (size_t)c->max_n * 4 * HW));
  }

  const bool copy_dist = out_dist != nullptr;
  const bool want_dist = copy_dist || (c->dist_resident && c->dist);
  const bool want_rgb = out_rgb != nullptr, want_glob = glob != nullptr;
  rc = run_forward(c, n, dL, dab, dmask, maskcent, want_glob ? dglob : nullptr, dout, want_dist ? ddist : nullptr,
                   want_rgb ? c->d_rgb : nullptr, st, hp.nchunks ? &hp : nullptr, out_abq ? c->d_abq : nullptr);
  if (rc != IDC_OK) return rc;
  auto d2h = [&](void* dst, const void* d, size_t bytes, void* stage) -> cudaError_t {
    if (is_pinned(dst)) return cudaMemcpyAsync(dst, d, bytes, cudaMemcpyDeviceToHost, st);
    return cudaMemcpyAsync(stage, d, bytes, cudaMemcpyDeviceToHost, st);
  };
  if (!hp.nchunks) CUDA_TRY(c, d2h(out_ab, dout, n * 2 * HW * sizeof(float), c->h_out));
  if (copy_dist) CUDA_TRY(c, d2h(out_dist, ddist, n * 529 * HW4 * sizeof(float), c->h_out + (size_t)c->max_n * 2 * HW));
  if (want_rgb) CUDA_TRY(c, d2h(out_rgb, c->d_rgb, n * HW * 3, c->h_rgb));
  if (out_abq) CUDA_TRY(c, d2h(out_abq, c->d_abq, n * 2 * HW * sizeof(double), c->h_abq));
  CUDA_TRY(c, cudaStreamSynchronize(st));
  if (hp.nchunks) CUDA_TRY(c, cudaStreamSynchronize(c->s_out));
  if (L) c->image_n = n;
  if (!is_pinned(out_ab)) memcpy(out_ab, c->h_out, n * 2 * HW * sizeof(float));
  if (copy_dist && !is_pinned(out_dist)) memcpy(out_dist, c->h_out + (size_t)c->max_n * 2 * HW, n * 529 * HW4 * sizeof(float));
  c->dist_valid_n = want_dist ? n : 0;
  if (want_rgb && !is_pinned(out_rgb)) memcpy(out_rgb, c->h_rgb, n * HW * 3);
  if (out_abq && !is_pinned(out_abq)) memcpy(out_abq, c->h_abq, n * 2 * HW * sizeof(double));
  if (int werr = *(volatile int*)c->h_err) {
    *(volatile int*)c->h_err = 0;
    return fail(c, IDC_ERR_WATCHDOG, "device pipeline watchdog fired (code %d)", werr);
  }
  return IDC_OK;
}

void* idc_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (bytes == 0 || cudaHostAlloc(&p, bytes, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return p;
}

int idc_host_free(void* p) {
  if (!p) return IDC_ERR_ARG;
  return cudaFreeHost(p) == cudaSuccess ? IDC_OK : IDC_ERR_CUDA;
}

int idc_set_dist_resident(idc_ctx* c, int on) {
  if (!c) return IDC_ERR_ARG;
  if (on && !c->dist) return fail(c, IDC_ERR_ARG, "resident dist requires IDC_FLAG_DIST");
  c->dist_resident = on != 0;
  return IDC_OK;
}

// does the pinned click block hold the answer for this pixel?
static bool click_answers(idc_ctx* c, int img, int y4, int x4) {
  if (!c->click_served || !c->h_clickout) return false;
  const int* hdr = reinterpret_cast<const int*>(c->h_clickout);
  return hdr[7] == 1 && hdr[0] == img && hdr[1] == y4 && hdr[2] == x4;
}

int idc_set_click(idc_ctx* c, int img, int y4, int x4, int K) {
  if (!c) return IDC_ERR_ARG;
  if (!c->dist) return fail(c, IDC_ERR_ARG, "idc_set_click requires IDC_FLAG_DIST");
  if (K < 0 || K > 32) return fail(c, IDC_ERR_ARG, "idc_set_click: need 0 <= K <= 32");
  CUDA_TRY(c, cudaSetDevice(c->dev));
  if (!c->h_click) {
    CUDA_TRY(c, cudaHostAlloc(&c->h_click, 64, cudaHostAllocMapped));
    memset(c->h_click, 0, 64);
    c->h_click[1] = -1;
    CUDA_TRY(c, cudaHostGetDevicePointer(&c->d_click, c->h_click, 0));
    CUDA_TRY(c, cudaMalloc(&c->d_clickout, kClickBytes));
    CUDA_TRY(c, cudaMemset(c->d_clickout, 0, kClickBytes));
    CUDA_TRY(c, cudaMallocHost(&c->h_clickout, kClickCopy));
    memset(c->h_clickout, 0, kClickCopy);
    float pts[529 * 2];   // the PyTorch wrapper's gamut grid (data/colorize_image.py:283): bin i = (g[i % 23], g[i / 23])
    for (int i = 0; i < 529; ++i) { pts[2 * i] = -110.f + 10.f * (i % 23); pts[2 * i + 1] = -110.f + 10.f * (i / 23); }
    CUDA_TRY(c, cudaMemcpy(c->d_clickout + kClickCopy, pts, sizeof(pts), cudaMemcpyHostToDevice));
  }
  volatile int* h = c->h_click;
  h[0] = img; h[1] = y4; h[2] = x4; h[3] = K; h[4] = h[4] + 1;
  c->click_mode = y4 >= 0;           // part of the graph key: switching the mode re-captures the click graph once
  c->click_served = false;
  return IDC_OK;
}

int idc_fetch_dist(idc_ctx* c, int img, int y4, int x4, float* out) {
  if (!c || !out) return IDC_ERR_ARG;
  if (img < 0 || img >= c->dist_valid_n || !c->d_out)
    return fail(c, IDC_ERR_STATE, "no resident distribution for image %d (run idc_forward_host with resident mode on)", img);
  const int H4 = c->H / 4, W4 = c->W / 4;
  const size_t HW = (size_t)c->H * c->W, HW4 = (size_t)H4 * W4;
  const float* d = c->d_out + (size_t)c->max_n * 2 * HW + (size_t)img * 529 * HW4;
  CUDA_TRY(c, cudaSetDevice(c->dev));
  if (y4 < 0) {
    CUDA_TRY(c, cudaMemcpy(out, d, 529 * HW4 * sizeof(float), cudaMemcpyDeviceToHost));
    return IDC_OK;
  }
  if (y4 >= H4 || x4 < 0 || x4 >= W4) return fail(c, IDC_ERR_ARG, "pixel (%d,%d) outside the %dx%d grid", y4, x4, H4, W4);
  if (click_answers(c, img, y4, x4)) {       // idc_set_click: the forward already brought this pixel back
    memcpy(out, c->h_clickout + kClickHdr, 529 * sizeof(float));
    return IDC_OK;
  }
  // one float per bin, bins are HW4 floats apart (NCHW)
  CUDA_TRY(c, cudaMemcpy2D(out, sizeof(float), d + (size_t)y4 * W4 + x4, HW4 * sizeof(float), sizeof(float), 529,
                           cudaMemcpyDeviceToHost));
  return IDC_OK;
}

// shared by idc_ab_reccs / idc_ab_reccs_pmf.  scratch (doubles): [kReccsMaxInit][3*32+2] results, then the 529x2
// gamut points as floats.
constexpr int kReccsMaxInit = 16, kReccsRes = 3 * 32 + 2;
constexpr size_t kReccsScratchBytes = (size_t)kReccsMaxInit * kReccsRes * sizeof(double) + 529 * 2 * sizeof(float);

static bool reccs_args_ok(int K, int max_iter, int n_init) {
  return K >= 1 && K <= 32 && max_iter >= 1 && n_init >= 1 && n_init <= kReccsMaxInit;
}

// best restart = lowest inertia; restarts within 1e-9 (relative) of it count as ties -> lowest index
static void reccs_pick(const double* res, int K, int n_init, float* centers_host, float* conf_host, int* iters_out) {
  const int stride = 3 * K + 2;
  double best = res[stride - 1];
  for (int v = 1; v < n_init; ++v) best = std::min(best, res[v * stride + stride - 1]);
  int pick = 0;
  while (res[pick * stride + stride - 1] > best * (1.0 + 1e-9) + 1e-300) ++pick;
  const double* r = res + (size_t)pick * stride;
  for (int i = 0; i < 2 * K; ++i) centers_host[i] = (float)r[i];
  if (conf_host) for (int k = 0; k < K; ++k) conf_host[k] = (float)r[2 * K + k];
  if (iters_out) *iters_out = (int)r[3 * K];
}

static cudaError_t reccs_run(const float* pmf_dev, size_t bin_stride, double* scratch, int K, int max_iter, int n_init,
                             const float* pts_host, float* centers_host, float* conf_host, int* iters_out) {
  float pts[529 * 2];
  if (pts_host) {
    memcpy(pts, pts_host, sizeof(pts));
  } else {   // the PyTorch wrapper's gamut grid (data/colorize_image.py:283, quirk q3): bin i = (g[i % 23], g[i / 23])
    for (int i = 0; i < 529; ++i) { pts[2 * i] = -110.f + 10.f * (i % 23); pts[2 * i + 1] = -110.f + 10.f * (i / 23); }
  }
  float* pts_dev = reinterpret_cast<float*>(scratch + (size_t)kReccsMaxInit * kReccsRes);
  cudaError_t e = cudaMemcpy(pts_dev, pts, sizeof(pts), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return e;
  if ((e = launch_ab_reccs(pmf_dev, bin_stride, pts_dev, K, max_iter, n_init, scratch, 0)) != cudaSuccess) return e;
  const int stride = 3 * K + 2;
  double res[kReccsMaxInit * kReccsRes];
  if ((e = cudaMemcpy(res, scratch, (size_t)n_init * stride * sizeof(double), cudaMemcpyDeviceToHost)) != cudaSuccess) return e;
  reccs_pick(res, K, n_init, centers_host, conf_host, iters_out);
  return cudaSuccess;
}

int idc_ab_reccs(idc_ctx* c, int img, int y4, int x4, int K, int max_iter, int n_init, const float* pts_host,
                 float* centers_host, float* conf_host, int* iters_out) {
  if (!c || !centers_host) return IDC_ERR_ARG;
  if (!reccs_args_ok(K, max_iter, n_init))
    return fail(c, IDC_ERR_ARG, "idc_ab_reccs: need 1 <= K <= 32, max_iter >= 1, 1 <= n_init <= %d", kReccsMaxInit);
  if (img < 0 || img >= c->dist_valid_n || !c->d_out)
    return fail(c, IDC_ERR_STATE, "no resident distribution for image %d (run idc_forward_host with resident mode on)", img);
  const int H4 = c->H / 4, W4 = c->W / 4;
  if (y4 < 0 || y4 >= H4 || x4 < 0 || x4 >= W4) return fail(c, IDC_ERR_ARG, "pixel (%d,%d) outside the %dx%d grid", y4, x4, H4, W4);
  const size_t HW = (size_t)c->H * c->W, HW4 = (size_t)H4 * W4;
  // idc_set_click with the same pixel and K, default restarts / iterations / gamut grid: the click graph already
  // clustered this pmf on its side branch and the results are in pinned host memory
  if (click_answers(c, img, y4, x4) && reinterpret_cast<const int*>(c->h_clickout)[3] == K && max_iter == kClickMaxIter &&
      n_init == kClickInit) {
    bool default_pts = pts_host == nullptr;
    if (!default_pts) {
      default_pts = true;
      for (int i = 0; i < 529 && default_pts; ++i)
        default_pts = pts_host[2 * i] == -110.f + 10.f * (i % 23) && pts_host[2 * i + 1] == -110.f + 10.f * (i / 23);
    }
    if (default_pts) {
      reccs_pick(reinterpret_cast<const double*>(c->h_clickout + kClickHdr + kClickPmf), K, n_init, centers_host, conf_host,
                 iters_out);
      return IDC_OK;
    }
  }
  const float* d = c->d_out + (size_t)c->max_n * 2 * HW + (size_t)img * 529 * HW4 + (size_t)y4 * W4 + x4;
  CUDA_TRY(c, cudaSetDevice(c->dev));
  if (!c->d_reccs) CUDA_TRY(c, cudaMalloc(&c->d_reccs, kReccsScratchBytes));
  CUDA_TRY(c, reccs_run(d, HW4, c->d_reccs, K, max_iter, n_init, pts_host, centers_host, conf_host, iters_out));
  return IDC_OK;
}

int idc_ab_reccs_pmf(int device, const float* pmf_host, int K, int max_iter, int n_init, const float* pts_host,
                     float* centers_host, float* conf_host, int* iters_out) {
  if (!pmf_host || !centers_host || !reccs_args_ok(K, max_iter, n_init)) return IDC_ERR_ARG;
  if (cudaSetDevice(device) != cudaSuccess) return IDC_ERR_CUDA;
  char* buf = nullptr;
  if (cudaMalloc(&buf, kReccsScratchBytes + 529 * sizeof(float)) != cudaSuccess) return IDC_ERR_CUDA;
  float* pmf_dev = reinterpret_cast<float*>(buf + kReccsScratchBytes);
  cudaError_t e = cudaMemcpy(pmf_dev, pmf_host, 529 * sizeof(float), cudaMemcpyHostToDevice);
  if (e == cudaSuccess)
    e = reccs_run(pmf_dev, 1, reinterpret_cast<double*>(buf), K, max_iter, n_init, pts_host, centers_host, conf_host, iters_out);
  cudaFree(buf);
  return e == cudaSuccess ? IDC_OK : IDC_ERR_CUDA;
}

int idc_caffe313_pred_ab(idc_ctx* c, int n, float T, float* out_ab, void* stream) {
  if (!c || !out_ab || n < 1 || n > c->max_n) return IDC_ERR_ARG;
  if (!c->caffe313) return fail(c, IDC_ERR_STATE, "ctx was not created with IDC_FLAG_CAFFE313");
  CUDA_TRY(c, cudaSetDevice(c->dev));
  CUDA_TRY(c, launch_decode313(c, n, T, out_ab, (cudaStream_t)stream));
  return IDC_OK;
}

int idc_caffe313_dist_pixel(idc_ctx* c, int img, int y, int x, float S, float* out313_host) {
  if (!c || !out313_host || img < 0 || img >= c->max_n || y < 0 || y >= c->H || x < 0 || x >= c->W) return IDC_ERR_ARG;
  if (!c->caffe313) return fail(c, IDC_ERR_STATE, "ctx was not created with IDC_FLAG_CAFFE313");
  CUDA_TRY(c, cudaSetDevice(c->dev));
  float* d = nullptr;
  CUDA_TRY(c, cudaMalloc(&d, 320 * sizeof(float)));
  cudaError_t e = launch_dist313_pixel(c, img, y, x, S, d, 0);
  if (e == cudaSuccess) e = cudaMemcpy(out313_host, d, 313 * sizeof(float), cudaMemcpyDeviceToHost);
  cudaFree(d);
  CUDA_TRY(c, e);
  return IDC_OK;
}

int idc_lab2rgb_u8(int device, int n, int h, int w, const float* L, const float* ab, uint8_t* rgb, void* stream) {
  if (n < 1 || h < 1 || w < 1 || !L || !ab || !rgb) return IDC_ERR_ARG;
  if (cudaSetDevice(device) != cudaSuccess) return IDC_ERR_CUDA;
  return launch_lab2rgb(nullptr, n, h, w, L, 0.0f, ab, rgb, (cudaStream_t)stream) == cudaSuccess ? IDC_OK : IDC_ERR_CUDA;
}

int idc_global_stats(int device, int h, int w, const uint8_t* rgb, const float* pts313, float* out316, void* stream) {
  if (h < 4 || w < 4 || (h % 4) || (w % 4) || !rgb || !pts313 || !out316) return IDC_ERR_ARG;
  if (cudaSetDevice(device) != cudaSuccess) return IDC_ERR_CUDA;
  return launch_global_stats(h, w, rgb, pts313, out316, (cudaStream_t)stream) == cudaSuccess ? IDC_OK : IDC_ERR_CUDA;
}

int idc_rgb2lab_f64(int device, int n, int h, int w, const uint8_t* rgb, double* lab, void* stream) {
  if (n < 1 || h < 1 || w < 1 || !rgb || !lab) return IDC_ERR_ARG;
  if (cudaSetDevice(device) != cudaSuccess) return IDC_ERR_CUDA;
  return launch_rgb2lab(n, h, w, rgb, lab, (cudaStream_t)stream) == cudaSuccess ? IDC_OK : IDC_ERR_CUDA;
}

int idc_zoom_lab2rgb_u8(int device, int h_in, int w_in, const double* ab, int h, int w, const double* L_full,
                        uint8_t* rgb, void* stream) {
  if (h_in < 1 || w_in < 1 || h < 1 || w < 1 || !ab || !L_full || !rgb) return IDC_ERR_ARG;
  if (cudaSetDevice(device) != cudaSuccess) return IDC_ERR_CUDA;
  return launch_zoom_lab2rgb(ab, h_in, w_in, L_full, h, w, rgb, (cudaStream_t)stream) == cudaSuccess ? IDC_OK : IDC_ERR_CUDA;
}

int idc_resize_u8_linear(int device, int h_src, int w_src, const uint8_t* src, int h_dst, int w_dst, uint8_t* dst, void* stream) {
  if (h_src < 1 || w_src < 1 || h_dst < 1 || w_dst < 1 || !src || !dst) return IDC_ERR_ARG;
  if (cudaSetDevice(device) != cudaSuccess) return IDC_ERR_CUDA;
  return launch_resize_linear_u8(src, h_src, w_src, dst, h_dst, w_dst, (cudaStream_t)stream) == cudaSuccess ? IDC_OK : IDC_ERR_CUDA;
}

int idc_cubic_lab2rgb_u8(int device, int h_in, int w_in, const double* ab, int h, int w, const double* L, uint8_t* rgb,
                         void* stream) {
  if (h_in < 1 || w_in < 1 || h < 1 || w < 1 || !ab || !L || !rgb) return IDC_ERR_ARG;
  if (cudaSetDevice(device) != cudaSuccess) return IDC_ERR_CUDA;
  return launch_cubic_lab2rgb(ab, h_in, w_in, L, h, w, rgb, (cudaStream_t)stream) == cudaSuccess ? IDC_OK : IDC_ERR_CUDA;
}

int idc_get_activation(idc_ctx* c, const char* name, float* out, size_t out_floats, int* ch, int* h, int* w) {
  if (!c || !name) return IDC_ERR_ARG;
  auto it = c->buf_index.find(name);
  if (it == c->buf_index.end() || c->bufs[it->second].H == 0) return fail(c, IDC_ERR_KEY, "no activation '%s'", name);
  const ActBuf& b = c->bufs[it->second];
  if (ch) *ch = b.C;
  if (h) *h = b.H;
  if (w) *w = b.W;
  if (!out) return IDC_OK;
  const int n = c->last_n > 0 ? c->last_n : 1;
  if (out_floats < (size_t)n * b.C * b.H * b.W) return fail(c, IDC_ERR_ARG, "output too small");
  CUDA_TRY(c, cudaSetDevice(c->dev));
  CUDA_TRY(c, launch_act_to_nchw(c, b, n, out, 0));
  CUDA_TRY(c, cudaDeviceSynchronize());
  return IDC_OK;
}

int idc_set_activation(idc_ctx* c, const char* name, int n, const float* in) {
  if (!c || !name || !in || n < 1 || n > c->max_n) return IDC_ERR_ARG;
  auto it = c->buf_index.find(name);
  if (it == c->buf_index.end() || c->bufs[it->second].H == 0) return fail(c, IDC_ERR_KEY, "no activation '%s'", name);
  CUDA_TRY(c, cudaSetDevice(c->dev));
  CUDA_TRY(c, launch_nchw_to_act(c, c->bufs[it->second], n, in, 0));
  CUDA_TRY(c, cudaDeviceSynchronize());
  c->last_n = n;
  return IDC_OK;
}

int idc_run_op(idc_ctx* c, const char* op_name, int n, void* stream) {
  if (!c || !op_name || n < 1 || n > c->max_n) return IDC_ERR_ARG;
  if (!c->weights_ready) return fail(c, IDC_ERR_STATE, "weights not finalized");
  CUDA_TRY(c, cudaSetDevice(c->dev));
  for (auto& op : c->ops)
    if (op.name == op_name) {
      if (op.fuse_out_head) return fail(c, IDC_ERR_ARG, "op %s has a fused head; use IDC_FLAG_KEEP_CONV10", op_name);
      c->gadd_active = false;
      if (c->simt) CUDA_TRY(c, simt_run_op(c, op, n, (cudaStream_t)stream));
      else CUDA_TRY(c, umma_run_op(c, op, n, nullptr, (float)c->opt.tanh_scale, (cudaStream_t)stream));
      c->last_n = n;
      return IDC_OK;
    }
  return fail(c, IDC_ERR_KEY, "no op '%s'", op_name);
}

int idc_set_profiling(idc_ctx* c, int enable) {
  if (!c) return IDC_ERR_ARG;
  c->profiling = enable != 0;
  return IDC_OK;
}

int idc_get_profile(idc_ctx* c, float* ms, int max_slots) {
  if (!c || !ms) return IDC_ERR_ARG;
  const int slots = (int)c->ops.size() + 2;
  if (max_slots < slots) return fail(c, IDC_ERR_ARG, "need %d slots", slots);
  CUDA_TRY(c, cudaSetDevice(c->dev));
  CUDA_TRY(c, cudaDeviceSynchronize());
  if (int werr = *(volatile int*)c->h_err) {
    *(volatile int*)c->h_err = 0;
    return fail(c, IDC_ERR_WATCHDOG, "device pipeline watchdog fired (code %d)", werr);
  }
  for (int i = 0; i < slots; ++i) ms[i] = 0.f;
  int runs = 0;
  for (auto& ev : c->prof_runs) {
    if ((int)ev.size() == slots + 1) {
      for (int i = 0; i < slots; ++i) {
        float t = 0.f;
        cudaEventElapsedTime(&t, ev[i], ev[i + 1]);
        ms[i] += t;
      }
      runs++;
    }
    for (cudaEvent_t e : ev) c->prof_pool.push_back(e);
  }
  c->prof_runs.clear();
  if (runs) for (int i = 0; i < slots; ++i) ms[i] /= runs;
  return slots;
}

double idc_op_flops(idc_ctx* c, int i) {
  return (c && i >= 0 && i < (int)c->ops.size()) ? c->ops[i].flops_per_image : 0.0;
}

// experiments (tools/): per-CTA cycle counters of the LAST tcgen05 launch; out[148*16] long long (read + clear)
extern "C" int idc_debug_counters(idc_ctx* c, int enable, long long* out_host) {
  if (!c) return IDC_ERR_ARG;
  CUDA_TRY(c, cudaSetDevice(c->dev));
  if (enable && !c->dbgbuf) {
    CUDA_TRY(c, cudaMalloc(&c->dbgbuf, 256 * 16 * sizeof(long long)));
    CUDA_TRY(c, cudaMemset(c->dbgbuf, 0, 256 * 16 * sizeof(long long)));
  }
  if (out_host && c->dbgbuf) {
    CUDA_TRY(c, cudaDeviceSynchronize());
    CUDA_TRY(c, cudaMemcpy(out_host, c->dbgbuf, 148 * 16 * sizeof(long long), cudaMemcpyDeviceToHost));
    CUDA_TRY(c, cudaMemset(c->dbgbuf, 0, 256 * 16 * sizeof(long long)));
  }
  if (!enable && c->dbgbuf) { cudaFree(c->dbgbuf); c->dbgbuf = nullptr; }
  return IDC_OK;
}

// experiments (tools/click_breakdown.py): device time of the click graph (copy nodes included), measured with two
// events around the graph launch.  enable = 1 / 0; returns the last span in *ms when non-null.
extern "C" int idc_debug_graph_timing(idc_ctx* c, int enable, float* ms) {
  if (!c) return IDC_ERR_ARG;
  CUDA_TRY(c, cudaSetDevice(c->dev));
  if (enable && !c->dbg_ev[0]) {
    CUDA_TRY(c, cudaEventCreate(&c->dbg_ev[0]));
    CUDA_TRY(c, cudaEventCreate(&c->dbg_ev[1]));
  }
  c->dbg_graph_timing = enable != 0 && c->dbg_ev[0];
  if (ms) *ms = c->dbg_graph_ms;
  return IDC_OK;
}

int idc_num_ops(idc_ctx* c) { return c ? (int)c->ops.size() : 0; }
const char* idc_op_name(idc_ctx* c, int i) {
  return (c && i >= 0 && i < (int)c->ops.size()) ? c->ops[i].name.c_str() : nullptr;
}
int idc_last_launch_count(idc_ctx* c) { return c ? c->launch_count : 0; }

double idc_flops_per_image(idc_ctx* c) {
  if (!c) return 0;
  double f = 2.0 * c->H * c->W * 64.0 * 36.0 + 2.0 * c->H * c->W * 2.0 * 128.0;  // model1.0 + model_out
  for (auto& op : c->ops) f += op.flops_per_image;
  return f;
}

const char* idc_last_error(idc_ctx* c) { return c ? c->err.c_str() : "null ctx"; }

int idc_destroy(idc_ctx* c) {
  if (!c) return IDC_ERR_ARG;
  cudaSetDevice(c->dev);
  cudaDeviceSynchronize();
  if (c->graph_exec) cudaGraphExecDestroy(c->graph_exec);
  for (auto& op : c->ops) umma_free_op(op);
  for (auto& ev : c->prof_runs) for (cudaEvent_t e : ev) cudaEventDestroy(e);
  for (cudaEvent_t e : c->prof_pool) cudaEventDestroy(e);
  for (auto& b : c->bufs) { if (b.p0) cudaFree(b.p0); if (b.p1) cudaFree(b.p1); }
  if (c->arena) cudaFree(c->arena);
  if (c->logits) cudaFree(c->logits);
  if (c->logits313) cudaFree(c->logits313);
  if (c->pts313) cudaFree(c->pts313);
  if (c->splitk_ws) cudaFree(c->splitk_ws);
  if (c->splitk_counters) cudaFree(c->splitk_counters);
  if (c->w11_umma) cudaFree(c->w11_umma);
  if (c->d_reccs) cudaFree(c->d_reccs);
  if (c->gvec) cudaFree(c->gvec);
  if (c->gtmp) cudaFree(c->gtmp);
  if (c->h_err) cudaFreeHost(c->h_err);
  if (c->d_in) cudaFree(c->d_in);
  if (c->d_out) cudaFree(c->d_out);
  if (c->d_rgb) cudaFree(c->d_rgb);
  if (c->d_small) cudaFree(c->d_small);
  if (c->h_small) cudaFreeHost(c->h_small);
  if (c->d_abq) cudaFree(c->d_abq);
  if (c->h_abq) cudaFreeHost(c->h_abq);
  if (c->h_in) cudaFreeHost(c->h_in);
  if (c->h_out) cudaFreeHost(c->h_out);
  if (c->h_rgb) cudaFreeHost(c->h_rgb);
  if (c->h_click) cudaFreeHost(c->h_click);
  if (c->d_clickout) cudaFree(c->d_clickout);
  if (c->h_clickout) cudaFreeHost(c->h_clickout);
  if (c->dbg_ev[0]) { cudaEventDestroy(c->dbg_ev[0]); cudaEventDestroy(c->dbg_ev[1]); }
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  if (c->s_click) { cudaStreamDestroy(c->s_click); cudaEventDestroy(c->ev_click[0]); cudaEventDestroy(c->ev_click[1]); }
  if (c->s_side) { cudaStreamDestroy(c->s_side); cudaEventDestroy(c->ev_fork); cudaEventDestroy(c->ev_join); }
  if (c->s_in) {
    cudaStreamDestroy(c->s_in); cudaStreamDestroy(c->s_out);
    for (int k = 0; k < HostPipe::kMaxChunks; ++k) { cudaEventDestroy(c->ev_in[k]); cudaEventDestroy(c->ev_out[k]); }
  }
  delete c;
  return IDC_OK;
}

}  // extern "C"
