// tflite_reader.hpp — reads the colour classifier out of a TensorFlow-Lite flatbuffer (host code, no TFLite, no
// flatbuffers library).  The reference loads models/dam_net/dam_net.tflite with tf.lite.Interpreter
// (scripts/color_classifier_server.py:66-71, path from the launch parameter ~model_path); the drop-in shell hands
// the same file to cp_color_net_load_tflite.
//
// Two readers over one walker:
//   read_color_net    exactly the architecture cone_color_kernel evaluates (color_net.cuh): the operator list must
//                     be CONV_2D, MAX_POOL_2D, CONV_2D, MAX_POOL_2D, MUL, ADD, RESHAPE, FULLY_CONNECTED, SOFTMAX with
//                     float32 tensors, 3x3 VALID stride-1 convolutions with fused ReLU, 2x2 stride-2 VALID pools,
//                     softmax beta 1 and a 1x15x12x1 input.
//   read_color_graph  any sequential float32 CNN of the subset below, lowered to the layer program
//                     color_graph_kernel runs (a retrained or reconverted classifier).
// Anything else is refused with a message — never evaluated approximately.
// The file is untrusted input: every offset is bounds-checked before it is followed.
//
// The subset read_color_graph accepts (and cones_perception_b200/tflite_model.py checks the same way):
//   one subgraph, one float32 input [1,15,12,1], one output [1,n] with 1 <= n <= 3; at most kGraphMaxOps operators
//   that form a chain (each one's first input, or either input of MUL / ADD, is the previous output; every other
//   input is a constant); activations [1,...] of rank 2 to 4; no quantisation parameters.
//   CONV_2D            SAME / VALID, any stride, dilation 1; filter [Co][kh][kw][Ci], bias [Co]
//   DEPTHWISE_CONV_2D  the same, filter [1][kh][kw][Ci*m], bias [Ci*m], depth_multiplier m (0 = derived)
//   MAX_POOL_2D, AVERAGE_POOL_2D  SAME / VALID, any filter and stride
//   MEAN               axes {1,2} (int32 constant), keep_dims either way
//   MUL, ADD           a float32 constant that is a scalar (every dimension 1), [C] or [1,1,1,C]
//   RELU, RELU6        standalone
//   RESHAPE            to the output tensor's shape, the element count unchanged (an int32 shape input is allowed)
//   FULLY_CONNECTED    default weights format, keep_num_dims false; weights [N][K], K = elements in, bias optional
//   SOFTMAX            the last operator, any finite beta
//   fused activations NONE, RELU, RELU6, RELU_N1_TO_1.  TANH, dilation != 1, other types, branches, custom ops and
//   other operators are refused.  The largest input + output pair of a layer must fit kGraphSmemBytes.
//
// Schema slots used (tensorflow/lite/schema/schema.fbs v3): Model{1 operator_codes, 2 subgraphs, 4 buffers},
// OperatorCode{0 deprecated_builtin_code:int8, 1 custom_code, 3 builtin_code:int32}, SubGraph{0 tensors, 1 inputs,
// 2 outputs, 3 operators}, Tensor{0 shape, 1 type, 2 buffer, 4 quantization}, QuantizationParameters{2 scale},
// Operator{0 opcode_index, 1 inputs, 2 outputs, 4 builtin_options}, Buffer{0 data},
// Conv2DOptions{0 padding, 1 stride_w, 2 stride_h, 3 activation, 4/5 dilation},
// DepthwiseConv2DOptions{0 padding, 1 stride_w, 2 stride_h, 3 depth_multiplier, 4 activation, 5/6 dilation},
// Pool2DOptions{0 padding, 1 stride_w, 2 stride_h, 3 filter_w, 4 filter_h, 5 activation},
// FullyConnectedOptions{0 activation, 1 weights_format, 2 keep_num_dims}, SoftmaxOptions{0 beta},
// Mul/AddOptions{0 activation}, ReducerOptions{0 keep_dims}.
#pragma once
#include <stdint.h>
#include <string.h>

#include <cmath>
#include <string>
#include <vector>

namespace cp_tflite {

struct Error {
  std::string what;
};

class Buf {
 public:
  Buf(const uint8_t* p, size_t n) : p_(p), n_(n) {}
  template <typename T>
  T rd(size_t pos) const {
    if (pos > n_ || n_ - pos < sizeof(T)) throw Error{"offset outside the file"};
    T v;
    memcpy(&v, p_ + pos, sizeof(T));
    return v;
  }
  const uint8_t* at(size_t pos, size_t len) const {
    if (pos > n_ || n_ - pos < len) throw Error{"vector outside the file"};
    return p_ + pos;
  }
  size_t size() const { return n_; }

 private:
  const uint8_t* p_;
  size_t n_;
};

struct Table {
  const Buf* b = nullptr;
  size_t pos = 0, vt = 0;
  uint16_t vt_len = 0;
  Table() {}
  Table(const Buf& buf, size_t p) : b(&buf), pos(p) {
    const int32_t so = buf.rd<int32_t>(p);
    const int64_t v = (int64_t)p - so;
    if (v < 0) throw Error{"vtable before the file"};
    vt = (size_t)v;
    vt_len = buf.rd<uint16_t>(vt);
    if (vt_len < 4) throw Error{"short vtable"};
  }
  size_t field(int slot) const {   // absolute position, 0 = absent
    const size_t e = 4 + 2 * (size_t)slot;
    if (e + 2 > vt_len) return 0;
    const uint16_t o = b->rd<uint16_t>(vt + e);
    return o ? pos + o : 0;
  }
  template <typename T>
  T scalar(int slot, T dflt) const {
    const size_t f = field(slot);
    return f ? b->rd<T>(f) : dflt;
  }
  size_t indirect(int slot) const {
    const size_t f = field(slot);
    return f ? f + b->rd<uint32_t>(f) : 0;
  }
  bool has(int slot) const { return field(slot) != 0; }
  Table table(int slot) const {
    const size_t p = indirect(slot);
    if (!p) throw Error{"missing table"};
    return Table(*b, p);
  }
  uint32_t vec_len(int slot) const {
    const size_t p = indirect(slot);
    return p ? b->rd<uint32_t>(p) : 0;
  }
  const uint8_t* vec_data(int slot, size_t elem) const {
    const size_t p = indirect(slot);
    if (!p) return nullptr;
    return b->at(p + 4, (size_t)b->rd<uint32_t>(p) * elem);
  }
  Table vec_table(int slot, uint32_t i) const {
    const size_t p = indirect(slot);
    if (!p || i >= b->rd<uint32_t>(p)) throw Error{"table index out of range"};
    const size_t e = p + 4 + 4 * (size_t)i;
    return Table(*b, e + b->rd<uint32_t>(e));
  }
  int32_t vec_i32(int slot, uint32_t i) const {
    const size_t p = indirect(slot);
    if (!p || i >= b->rd<uint32_t>(p)) throw Error{"index out of range"};
    return b->rd<int32_t>(p + 4 + 4 * (size_t)i);
  }
};

struct ColorNetWeights {
  uint32_t c1 = 0, c2 = 0, classes = 0;
  std::vector<float> conv1_w, conv1_b, conv2_w, conv2_b, bn_scale, bn_shift, dense_w, dense_b;
};

enum { OP_ADD = 0, OP_CONV_2D = 3, OP_FULLY_CONNECTED = 9, OP_MAX_POOL_2D = 17, OP_MUL = 18, OP_RESHAPE = 22, OP_SOFTMAX = 25 };

inline ColorNetWeights read_color_net(const uint8_t* data, size_t bytes) {
  Buf buf(data, bytes);
  if (bytes < 8 || memcmp(data + 4, "TFL3", 4) != 0) throw Error{"not a TFL3 flatbuffer"};
  Table model(buf, buf.rd<uint32_t>(0));
  std::vector<int32_t> codes;
  for (uint32_t i = 0; i < model.vec_len(1); ++i) {
    Table oc = model.vec_table(1, i);
    if (oc.has(1)) throw Error{"custom operators are not supported"};
    int32_t code = oc.scalar<int32_t>(3, 0);
    if (code == 0) code = oc.scalar<int8_t>(0, 0);
    codes.push_back(code);
  }
  if (model.vec_len(2) != 1) throw Error{"expected one subgraph"};
  Table sg = model.vec_table(2, 0);
  const uint32_t n_tensors = sg.vec_len(0), n_buffers = model.vec_len(4);

  auto shape_of = [&](int32_t t) {
    if (t < 0 || (uint32_t)t >= n_tensors) throw Error{"tensor index out of range"};
    Table tt = sg.vec_table(0, (uint32_t)t);
    if (tt.scalar<int8_t>(1, 0) != 0) throw Error{"only float32 tensors are supported"};
    std::vector<int32_t> s(tt.vec_len(0));
    for (uint32_t i = 0; i < s.size(); ++i) s[i] = tt.vec_i32(0, i);
    return s;
  };
  auto constant = [&](int32_t t, size_t expect) {
    if (t < 0 || (uint32_t)t >= n_tensors) throw Error{"tensor index out of range"};
    Table tt = sg.vec_table(0, (uint32_t)t);
    if (tt.scalar<int8_t>(1, 0) != 0) throw Error{"only float32 constants are supported"};
    const uint32_t bi = tt.scalar<uint32_t>(2, 0);
    if (bi >= n_buffers) throw Error{"buffer index out of range"};
    Table bt = model.vec_table(4, bi);
    if (bt.vec_len(0) != expect * 4) throw Error{"constant tensor has an unexpected size"};
    std::vector<float> v(expect);
    if (expect) memcpy(v.data(), bt.vec_data(0, 1), expect * 4);
    return v;
  };
  struct OpView {
    int32_t code;
    std::vector<int32_t> in, out;
    Table opt;
    bool has_opt;
  };
  const int32_t want[9] = {OP_CONV_2D, OP_MAX_POOL_2D, OP_CONV_2D, OP_MAX_POOL_2D, OP_MUL, OP_ADD, OP_RESHAPE, OP_FULLY_CONNECTED, OP_SOFTMAX};
  if (sg.vec_len(3) != 9) throw Error{"unexpected operator count (dam_net has 9)"};
  std::vector<OpView> ops;
  for (uint32_t i = 0; i < 9; ++i) {
    Table o = sg.vec_table(3, i);
    const uint32_t ci = o.scalar<uint32_t>(0, 0);
    if (ci >= codes.size()) throw Error{"opcode index out of range"};
    OpView v;
    v.code = codes[ci];
    if (v.code != want[i]) throw Error{"unexpected operator sequence: not the dam_net architecture"};
    for (uint32_t k = 0; k < o.vec_len(1); ++k) v.in.push_back(o.vec_i32(1, k));
    for (uint32_t k = 0; k < o.vec_len(2); ++k) v.out.push_back(o.vec_i32(2, k));
    v.has_opt = o.has(4);
    if (v.has_opt) v.opt = o.table(4);
    ops.push_back(v);
  }
  // the operators must form a chain: each consumes the previous output
  if (sg.vec_len(1) != 1 || sg.vec_len(2) != 1 || ops[0].in.empty() || ops[0].in[0] != sg.vec_i32(1, 0))
    throw Error{"unexpected graph inputs"};
  for (int i = 1; i < 9; ++i)
    if (ops[i].in.empty() || ops[i - 1].out.size() != 1 || ops[i].in[0] != ops[i - 1].out[0]) throw Error{"operators do not form a chain"};
  if (ops[8].out.size() != 1 || ops[8].out[0] != sg.vec_i32(2, 0)) throw Error{"unexpected graph output"};

  const std::vector<int32_t> in_shape = shape_of(ops[0].in[0]);
  if (in_shape != std::vector<int32_t>{1, 15, 12, 1}) throw Error{"input must be 1x15x12x1"};
  auto check_conv = [&](const OpView& o) {
    if (o.in.size() != 3 || !o.has_opt) throw Error{"CONV_2D needs filter, bias and options"};
    if (o.opt.scalar<int8_t>(0, 0) != 1 /*VALID*/ || o.opt.scalar<int32_t>(1, 0) != 1 || o.opt.scalar<int32_t>(2, 0) != 1 ||
        o.opt.scalar<int8_t>(3, 0) != 1 /*RELU*/ || o.opt.scalar<int32_t>(4, 1) != 1 || o.opt.scalar<int32_t>(5, 1) != 1)
      throw Error{"CONV_2D must be VALID, stride 1, dilation 1, fused ReLU"};
  };
  auto check_pool = [&](const OpView& o) {
    if (!o.has_opt || o.opt.scalar<int8_t>(0, 0) != 1 || o.opt.scalar<int32_t>(1, 0) != 2 || o.opt.scalar<int32_t>(2, 0) != 2 ||
        o.opt.scalar<int32_t>(3, 0) != 2 || o.opt.scalar<int32_t>(4, 0) != 2 || o.opt.scalar<int8_t>(5, 0) != 0)
      throw Error{"MAX_POOL_2D must be 2x2, stride 2, VALID, no activation"};
  };
  ColorNetWeights w;
  check_conv(ops[0]);
  const std::vector<int32_t> f1 = shape_of(ops[0].in[1]);
  if (f1.size() != 4 || f1[1] != 3 || f1[2] != 3 || f1[3] != 1 || f1[0] < 1 || f1[0] > 16) throw Error{"first convolution must be [c1<=16][3][3][1]"};
  w.c1 = (uint32_t)f1[0];
  w.conv1_w = constant(ops[0].in[1], (size_t)w.c1 * 9);
  w.conv1_b = constant(ops[0].in[2], w.c1);
  check_pool(ops[1]);
  check_conv(ops[2]);
  const std::vector<int32_t> f2 = shape_of(ops[2].in[1]);
  if (f2.size() != 4 || f2[1] != 3 || f2[2] != 3 || (uint32_t)f2[3] != w.c1 || f2[0] < 1 || f2[0] > 32) throw Error{"second convolution must be [c2<=32][3][3][c1]"};
  w.c2 = (uint32_t)f2[0];
  w.conv2_w = constant(ops[2].in[1], (size_t)w.c2 * 9 * w.c1);
  w.conv2_b = constant(ops[2].in[2], w.c2);
  check_pool(ops[3]);
  for (int i = 4; i <= 5; ++i) {
    if (ops[i].in.size() != 2) throw Error{"MUL / ADD need one constant operand"};
    if (ops[i].has_opt && ops[i].opt.scalar<int8_t>(0, 0) != 0) throw Error{"MUL / ADD must have no fused activation"};
  }
  w.bn_scale = constant(ops[4].in[1], w.c2);
  w.bn_shift = constant(ops[5].in[1], w.c2);
  if (ops[7].in.size() != 3) throw Error{"FULLY_CONNECTED needs weights and bias"};
  if (ops[7].has_opt && ops[7].opt.scalar<int8_t>(0, 0) != 0) throw Error{"FULLY_CONNECTED must have no fused activation"};
  const std::vector<int32_t> fd = shape_of(ops[7].in[1]);
  if (fd.size() != 2 || (uint32_t)fd[1] != 2 * w.c2 || fd[0] < 1 || fd[0] > 4) throw Error{"dense layer must be [classes<=4][2*c2]"};
  w.classes = (uint32_t)fd[0];
  w.dense_w = constant(ops[7].in[1], (size_t)w.classes * 2 * w.c2);
  w.dense_b = constant(ops[7].in[2], w.classes);
  if (ops[8].has_opt && ops[8].opt.scalar<float>(0, 1.0f) != 1.0f) throw Error{"SOFTMAX beta must be 1"};
  return w;
}

// ---- any sequential float32 CNN of the subset above: the layer program of color_graph_kernel -----------------
constexpr uint32_t kGraphMaxOps = 64;
constexpr size_t kGraphSmemBytes = 227 * 1024;   // dynamic shared memory one block may hold on sm_100a
enum { OP_AVERAGE_POOL_2D = 1, OP_DEPTHWISE_CONV_2D = 4, OP_RELU = 19, OP_RELU6 = 21, OP_MEAN = 40 };

enum GraphOp : int32_t { G_CONV, G_DWCONV, G_MAXPOOL, G_AVGPOOL, G_MEAN, G_MUL, G_ADD, G_CLAMP, G_FC, G_SOFTMAX };

// One layer.  Activations are row-major [h][w][c] (NHWC without the batch of 1; a tensor of rank < 4 is
// [1][elements / last dim][last dim]).  Offsets count floats: w / b into the weight buffer, src / dst into the
// kernel's shared memory.
struct GraphLayer {
  int32_t op;
  int32_t ih, iw, ic, oh, ow, oc;
  int32_t kh, kw, sh, sw, pt, pl;   // filter, stride, padding before (top, left)
  int32_t m;                        // depthwise multiplier; MUL / ADD: constant length (1 or ic)
  uint32_t w, b, src, dst;
  float lo, hi;                     // activation clamp; SOFTMAX: lo = beta
};

struct ColorGraph {
  std::vector<GraphLayer> layers;
  std::vector<float> weights;   // conv [kh][kw][ci][co], depthwise [kh][kw][c], FC [K][N], then biases
  uint32_t classes = 0;
  uint32_t smem_floats = 0;     // the largest input + output pair of a layer
  uint32_t out = 0, logits = 0; // shared-memory offsets of the output and of the final SOFTMAX's input
};

inline const char* builtin_name(int32_t code) {
  switch (code) {
    case OP_ADD: return "ADD";
    case OP_AVERAGE_POOL_2D: return "AVERAGE_POOL_2D";
    case OP_CONV_2D: return "CONV_2D";
    case OP_DEPTHWISE_CONV_2D: return "DEPTHWISE_CONV_2D";
    case OP_FULLY_CONNECTED: return "FULLY_CONNECTED";
    case OP_MAX_POOL_2D: return "MAX_POOL_2D";
    case OP_MUL: return "MUL";
    case OP_RELU: return "RELU";
    case OP_RELU6: return "RELU6";
    case OP_RESHAPE: return "RESHAPE";
    case OP_SOFTMAX: return "SOFTMAX";
    case OP_MEAN: return "MEAN";
    case 14: return "LOGISTIC";
    case 20: return "RELU_N1_TO_1";
    case 28: return "TANH";
    default: return nullptr;
  }
}

inline ColorGraph read_color_graph(const uint8_t* data, size_t bytes) {
  Buf buf(data, bytes);
  if (bytes < 8 || memcmp(data + 4, "TFL3", 4) != 0) throw Error{"not a TFL3 flatbuffer"};
  Table model(buf, buf.rd<uint32_t>(0));
  std::vector<int32_t> codes;
  for (uint32_t i = 0; i < model.vec_len(1); ++i) {
    Table oc = model.vec_table(1, i);
    if (oc.has(1)) throw Error{"custom operators are not supported"};
    int32_t code = oc.scalar<int32_t>(3, 0);
    if (code == 0) code = oc.scalar<int8_t>(0, 0);
    codes.push_back(code);
  }
  if (model.vec_len(2) != 1) throw Error{"expected one subgraph"};
  Table sg = model.vec_table(2, 0);
  const uint32_t n_tensors = sg.vec_len(0), n_buffers = model.vec_len(4);
  const uint32_t n_ops = sg.vec_len(3);
  if (n_ops < 1 || n_ops > kGraphMaxOps) throw Error{"operator count " + std::to_string(n_ops) + " outside 1.." + std::to_string(kGraphMaxOps)};
  if (sg.vec_len(1) != 1 || sg.vec_len(2) != 1) throw Error{"expected one graph input and one graph output"};

  struct TensorView {
    std::vector<int32_t> shape;
    int8_t type;
    const uint8_t* data;
    size_t bytes;
  };
  auto tensor = [&](int32_t t, const char* what) {
    if (t < 0 || (uint32_t)t >= n_tensors) throw Error{std::string(what) + ": tensor index out of range"};
    Table tt = sg.vec_table(0, (uint32_t)t);
    TensorView v;
    v.type = tt.scalar<int8_t>(1, 0);
    const uint32_t rank = tt.vec_len(0);
    if (rank > 4) throw Error{std::string(what) + ": tensor rank above 4"};
    for (uint32_t i = 0; i < rank; ++i) {
      const int32_t d = tt.vec_i32(0, i);
      if (d < 1 || d > (1 << 20)) throw Error{std::string(what) + ": tensor dimension outside 1..2^20"};
      v.shape.push_back(d);
    }
    if (tt.has(4)) {
      Table q = tt.table(4);
      if (q.vec_len(2) != 0) throw Error{std::string(what) + ": quantised tensors are not supported"};
    }
    const uint32_t bi = tt.scalar<uint32_t>(2, 0);
    v.data = nullptr;
    v.bytes = 0;
    if (bi >= n_buffers) throw Error{std::string(what) + ": buffer index out of range"};
    Table bt = model.vec_table(4, bi);
    v.bytes = bt.vec_len(0);
    if (v.bytes) v.data = bt.vec_data(0, 1);
    return v;
  };
  auto numel = [](const std::vector<int32_t>& s) {
    uint64_t n = 1;
    for (int32_t d : s) n *= (uint64_t)d;
    return n;
  };
  ColorGraph g;
  // a float32 constant of the given shape, appended to the weight buffer in file order
  auto constant = [&](int32_t t, const char* what, const std::vector<int32_t>& want) {
    const TensorView v = tensor(t, what);
    if (v.type != 0) throw Error{std::string(what) + ": only float32 constants are supported"};
    if (v.shape != want) throw Error{std::string(what) + ": constant has an unexpected shape"};
    const uint64_t n = numel(want);
    if (n > (1u << 26) || v.bytes != n * 4) throw Error{std::string(what) + ": constant tensor has an unexpected size"};
    std::vector<float> f(n);
    memcpy(f.data(), v.data, n * 4);
    return f;
  };
  auto put = [&](const std::vector<float>& f) {
    if (g.weights.size() + f.size() > (1u << 28)) throw Error{"weights above 2^28 floats"};
    const uint32_t o = (uint32_t)g.weights.size();
    g.weights.insert(g.weights.end(), f.begin(), f.end());
    return o;
  };
  auto act_range = [&](int8_t a, const char* what, GraphLayer& L) {
    switch (a) {
      case 0: L.lo = -INFINITY; L.hi = INFINITY; return;
      case 1: L.lo = 0.f; L.hi = INFINITY; return;
      case 2: L.lo = -1.f; L.hi = 1.f; return;
      case 3: L.lo = 0.f; L.hi = 6.f; return;
      default: throw Error{std::string(what) + ": fused activation " + std::to_string(a) + " is not supported (NONE, RELU, RELU6, RELU_N1_TO_1)"};
    }
  };
  // output extent and padding before, TFLite's ComputePaddingHeightWidth with dilation 1
  auto window = [](int8_t padding, int32_t in, int32_t k, int32_t s, int32_t& out, int32_t& pad) {
    if (padding == 0) {
      out = (in + s - 1) / s;
      const int32_t total = (out - 1) * s + k - in;
      pad = total > 0 ? total / 2 : 0;
    } else {
      out = in >= k ? (in - k) / s + 1 : 0;
      pad = 0;
    }
  };

  int32_t cur = sg.vec_i32(1, 0);
  std::vector<int32_t> shape;
  {
    const TensorView in = tensor(cur, "graph input");
    if (in.type != 0 || in.shape != std::vector<int32_t>{1, 15, 12, 1} || in.bytes) throw Error{"input must be a float32 1x15x12x1 tensor"};
    shape = in.shape;
  }
  for (uint32_t i = 0; i < n_ops; ++i) {
    Table o = sg.vec_table(3, i);
    const uint32_t ci = o.scalar<uint32_t>(0, 0);
    if (ci >= codes.size()) throw Error{"opcode index out of range"};
    const int32_t code = codes[ci];
    const char* name = builtin_name(code);
    const std::string where = "operator " + std::to_string(i) + " (" + (name ? name : "builtin " + std::to_string(code)) + ")";
    const char* wh = where.c_str();
    std::vector<int32_t> in, out;
    for (uint32_t k = 0; k < o.vec_len(1); ++k) in.push_back(o.vec_i32(1, k));
    for (uint32_t k = 0; k < o.vec_len(2); ++k) out.push_back(o.vec_i32(2, k));
    const bool has_opt = o.has(4);
    Table opt = has_opt ? o.table(4) : Table();
    if (out.size() != 1) throw Error{where + ": expected one output"};
    if (in.empty()) throw Error{where + ": no input"};
    int chain = in[0] == cur ? 0 : -1;
    if (chain < 0 && (code == OP_MUL || code == OP_ADD) && in.size() == 2 && in[1] == cur) chain = 1;
    if (chain < 0) throw Error{where + ": the operators do not form a chain"};
    if (i + 1 < n_ops && code == OP_SOFTMAX) throw Error{where + ": SOFTMAX must be the last operator"};
    const bool spatial = code == OP_CONV_2D || code == OP_DEPTHWISE_CONV_2D || code == OP_MAX_POOL_2D ||
                         code == OP_AVERAGE_POOL_2D || code == OP_MEAN;
    if (spatial && shape.size() != 4) throw Error{where + ": input must be [1,H,W,C]"};
    const int32_t C = shape.back();
    const int32_t H = shape.size() == 4 ? shape[1] : 1;
    const int32_t W = (int32_t)(numel(shape) / (uint64_t)C / (uint64_t)H);
    GraphLayer L{};
    L.ih = H; L.iw = W; L.ic = C;
    L.kh = L.kw = L.sh = L.sw = 1;
    L.lo = -INFINITY; L.hi = INFINITY;
    std::vector<int32_t> next;
    bool emit = true;
    if (code == OP_CONV_2D || code == OP_DEPTHWISE_CONV_2D) {
      const bool dw = code == OP_DEPTHWISE_CONV_2D;
      if (in.size() != 3 || in[2] < 0 || !has_opt) throw Error{where + ": needs filter, bias and options"};
      const int8_t pad = opt.scalar<int8_t>(0, 0);
      L.sw = opt.scalar<int32_t>(1, 0);
      L.sh = opt.scalar<int32_t>(2, 0);
      if (pad != 0 && pad != 1) throw Error{where + ": padding must be SAME or VALID"};
      if (L.sw < 1 || L.sh < 1 || L.sw > 64 || L.sh > 64) throw Error{where + ": stride outside 1..64"};
      if (opt.scalar<int32_t>(dw ? 5 : 4, 1) != 1 || opt.scalar<int32_t>(dw ? 6 : 5, 1) != 1) throw Error{where + ": dilation must be 1"};
      act_range(opt.scalar<int8_t>(dw ? 4 : 3, 0), wh, L);
      const TensorView f = tensor(in[1], wh);
      if (f.shape.size() != 4) throw Error{where + ": filter must be rank 4"};
      L.kh = f.shape[1];
      L.kw = f.shape[2];
      if (dw) {
        if (f.shape[0] != 1 || f.shape[3] % C) throw Error{where + ": filter must be [1][kh][kw][C*m]"};
        L.m = f.shape[3] / C;
        const int32_t m = opt.scalar<int32_t>(3, 0);
        if (m != 0 && m != L.m) throw Error{where + ": depth_multiplier disagrees with the filter"};
        L.oc = f.shape[3];
        L.w = put(constant(in[1], wh, f.shape));   // [1][kh][kw][oc] is already [kh][kw][oc]
      } else {
        if (f.shape[3] != C) throw Error{where + ": filter must be [Co][kh][kw][C]"};
        L.oc = f.shape[0];
        const std::vector<float> w = constant(in[1], wh, f.shape);
        std::vector<float> t(w.size());   // [co][ky][kx][ci] -> [ky][kx][ci][co]
        const size_t K = (size_t)L.kh * L.kw * C;
        for (size_t co = 0; co < (size_t)L.oc; ++co)
          for (size_t k = 0; k < K; ++k) t[k * L.oc + co] = w[co * K + k];
        L.w = put(t);
      }
      L.b = put(constant(in[2], wh, {L.oc}));
      window(pad, H, L.kh, L.sh, L.oh, L.pt);
      window(pad, W, L.kw, L.sw, L.ow, L.pl);
      L.op = dw ? G_DWCONV : G_CONV;
    } else if (code == OP_MAX_POOL_2D || code == OP_AVERAGE_POOL_2D) {
      if (in.size() != 1 || !has_opt) throw Error{where + ": needs one input and options"};
      const int8_t pad = opt.scalar<int8_t>(0, 0);
      L.sw = opt.scalar<int32_t>(1, 0);
      L.sh = opt.scalar<int32_t>(2, 0);
      L.kw = opt.scalar<int32_t>(3, 0);
      L.kh = opt.scalar<int32_t>(4, 0);
      if (pad != 0 && pad != 1) throw Error{where + ": padding must be SAME or VALID"};
      if (L.sw < 1 || L.sh < 1 || L.sw > 64 || L.sh > 64) throw Error{where + ": stride outside 1..64"};
      if (L.kw < 1 || L.kh < 1 || L.kw > 64 || L.kh > 64) throw Error{where + ": filter outside 1..64"};
      act_range(opt.scalar<int8_t>(5, 0), wh, L);
      window(pad, H, L.kh, L.sh, L.oh, L.pt);
      window(pad, W, L.kw, L.sw, L.ow, L.pl);
      L.oc = C;
      L.op = code == OP_MAX_POOL_2D ? G_MAXPOOL : G_AVGPOOL;
    } else if (code == OP_MEAN) {
      if (in.size() != 2) throw Error{where + ": needs the axes input"};
      const TensorView ax = tensor(in[1], wh);
      if (ax.type != 2 || ax.bytes != 8 || numel(ax.shape) != 2) throw Error{where + ": axes must be an int32 constant {1, 2}"};
      int32_t a[2];
      memcpy(a, ax.data, 8);
      if (!((a[0] == 1 && a[1] == 2) || (a[0] == 2 && a[1] == 1))) throw Error{where + ": only axes {1, 2} are supported"};
      L.oh = L.ow = 1;
      L.oc = C;
      L.op = G_MEAN;
      const bool keep = has_opt && opt.scalar<uint8_t>(0, 0) != 0;
      next = keep ? std::vector<int32_t>{1, 1, 1, C} : std::vector<int32_t>{1, C};
    } else if (code == OP_MUL || code == OP_ADD) {
      if (in.size() != 2) throw Error{where + ": needs two inputs"};
      const int32_t k = in[1 - chain];
      const TensorView c = tensor(k, wh);
      const uint64_t n = numel(c.shape);
      const bool per_channel = c.shape == std::vector<int32_t>{C} || c.shape == std::vector<int32_t>{1, 1, 1, C};
      if (n != 1 && !per_channel) throw Error{where + ": the constant must be a scalar, [C] or [1,1,1,C]"};
      L.m = (int32_t)n;
      L.w = put(constant(k, wh, c.shape));
      act_range(has_opt ? opt.scalar<int8_t>(0, 0) : (int8_t)0, wh, L);
      L.oh = L.ih; L.ow = L.iw; L.oc = C;
      L.op = code == OP_MUL ? G_MUL : G_ADD;
    } else if (code == OP_RELU || code == OP_RELU6) {
      if (in.size() != 1) throw Error{where + ": needs one input"};
      act_range(code == OP_RELU ? 1 : 3, wh, L);
      L.oh = L.ih; L.ow = L.iw; L.oc = C;
      L.op = G_CLAMP;
    } else if (code == OP_RESHAPE) {
      if (in.size() > 2) throw Error{where + ": too many inputs"};
      if (in.size() == 2 && in[1] >= 0 && tensor(in[1], wh).bytes == 0) throw Error{where + ": the shape input must be a constant"};
      next = tensor(out[0], wh).shape;
      if (numel(next) != numel(shape)) throw Error{where + ": the element count changes"};
      emit = false;
    } else if (code == OP_FULLY_CONNECTED) {
      if (in.size() < 2 || in.size() > 3) throw Error{where + ": needs weights and an optional bias"};
      if (has_opt && opt.scalar<int8_t>(1, 0) != 0) throw Error{where + ": only the default weights format is supported"};
      if (has_opt && opt.scalar<uint8_t>(2, 0) != 0) throw Error{where + ": keep_num_dims is not supported"};
      act_range(has_opt ? opt.scalar<int8_t>(0, 0) : (int8_t)0, wh, L);
      const TensorView f = tensor(in[1], wh);
      const uint64_t K = numel(shape);
      if (f.shape.size() != 2 || (uint64_t)f.shape[1] != K) throw Error{where + ": weights must be [N][elements of the input]"};
      const int32_t N = f.shape[0];
      const std::vector<float> w = constant(in[1], wh, f.shape);
      std::vector<float> t(w.size());   // [n][k] -> [k][n]
      for (size_t n = 0; n < (size_t)N; ++n)
        for (size_t k = 0; k < K; ++k) t[k * N + n] = w[n * K + k];
      L.w = put(t);
      L.b = put(in.size() == 3 && in[2] >= 0 ? constant(in[2], wh, {N}) : std::vector<float>(N, 0.f));
      L.ih = L.iw = 1; L.ic = (int32_t)K;
      L.oh = L.ow = 1; L.oc = N;
      L.op = G_FC;
      next = {1, N};
    } else if (code == OP_SOFTMAX) {
      if (in.size() != 1) throw Error{where + ": needs one input"};
      if ((uint64_t)C != numel(shape)) throw Error{where + ": input must hold its elements in the last dimension"};
      L.lo = has_opt ? opt.scalar<float>(0, 1.0f) : 1.0f;
      if (!std::isfinite(L.lo)) throw Error{where + ": beta must be finite"};
      L.oh = L.ih; L.ow = L.iw; L.oc = C;
      L.op = G_SOFTMAX;
    } else {
      throw Error{where + ": operator not supported"};
    }
    for (size_t k = 1; k < in.size(); ++k)
      if ((int)k != chain && in[k] >= 0 && tensor(in[k], wh).bytes == 0) throw Error{where + ": an input other than the chain is not a constant"};
    if (emit) {
      if (L.oh < 1 || L.ow < 1 || L.oc < 1) throw Error{where + ": empty output"};
      if (next.empty()) next = shape.size() == 4 ? std::vector<int32_t>{1, L.oh, L.ow, L.oc} : shape;
      g.layers.push_back(L);
    }
    const TensorView ot = tensor(out[0], wh);
    if (ot.type != 0 || ot.bytes) throw Error{where + ": output must be a float32 activation"};
    if (ot.shape != next) throw Error{where + ": the output tensor's shape disagrees with the operator"};
    if (next.size() < 2 || next[0] != 1) throw Error{where + ": activations must be [1,...] of rank 2 to 4"};
    shape = next;
    cur = out[0];
  }
  if (cur != sg.vec_i32(2, 0)) throw Error{"the last operator's output is not the graph output"};
  if (shape.size() != 2 || shape[1] < 1 || shape[1] > 3) throw Error{"output must be [1,n] with 1 <= n <= 3"};
  if (g.layers.empty()) throw Error{"no operator computes anything"};
  g.classes = (uint32_t)shape[1];
  // ping-pong from both ends of one buffer: layer i reads one end and writes the other
  uint64_t pair = 0;
  for (const GraphLayer& L : g.layers)
    pair = std::max<uint64_t>(pair, (uint64_t)L.ih * L.iw * L.ic + (uint64_t)L.oh * L.ow * L.oc);
  if (pair * 4 > kGraphSmemBytes)
    throw Error{"activations need " + std::to_string(pair * 4) + " bytes of shared memory for one layer's input and output, above the " +
                std::to_string(kGraphSmemBytes) + "-byte budget"};
  g.smem_floats = (uint32_t)pair;
  bool right = false;
  for (GraphLayer& L : g.layers) {
    const uint32_t n_in = (uint32_t)(L.ih * L.iw * L.ic), n_out = (uint32_t)(L.oh * L.ow * L.oc);
    L.src = right ? g.smem_floats - n_in : 0;
    L.dst = right ? 0 : g.smem_floats - n_out;
    right = !right;
  }
  const GraphLayer& last = g.layers.back();
  g.out = last.dst;
  g.logits = last.op == G_SOFTMAX ? last.src : last.dst;
  return g;
}

}  // namespace cp_tflite
