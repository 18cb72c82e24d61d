// color_net.cuh — the reference's cone-colour classifier on the device (SURVEY §8 f3).
//
// The reference evaluates models/dam_net/dam_net.tflite with the TFLite interpreter inside a Python ROS
// service (scripts/color_classifier_server.py:66-71 loads it, :108-120 runs it per cone): the 15x12x1 uint8
// range image is cast to float32 without scaling (:108), and the answer is argmax + 1 when the largest softmax
// output is >= 0.8, else 0 = unknown (:116-120).  The graph in that file is
//     CONV_2D 3x3 (1 -> 16, VALID, ReLU) -> MAX_POOL 2x2/2 -> CONV_2D 3x3 (16 -> 32, VALID, ReLU) -> MAX_POOL 2x2/2
//     -> MUL, ADD (folded batch normalisation, per channel) -> RESHAPE (flatten, NHWC) -> FULLY_CONNECTED (64 -> 3)
//     -> SOFTMAX
// cone_color_kernel evaluates exactly this architecture (channel counts are parameters up to the shared-memory
// budget below), one CTA per cone, chained behind cone_raster_kernel so that only one byte per cone travels back.
// color_graph_kernel (below) evaluates any other graph cp_tflite::read_color_graph accepts (a retrained classifier);
// on dam_net it gives the same bits but takes 1.7x as long, so dam_net keeps its own kernel (DESIGN §4.5).
//
// Arithmetic: fp32, every accumulation in the order of TFLite's reference kernels (filter_y, filter_x,
// in_channel; then the bias), multiply and add rounded separately (no FMA contraction), which is also the order
// of the numpy checker (oracle/dam_net_ref.py) — logits are bit-identical to it; the softmax differs from numpy
// only by expf's last ulp.  75 k multiply-adds per cone: latency-bound, no tensor-core shape (K = 9 and 144).
#pragma once
#include "color_kernels.cuh"
#include "tflite_reader.hpp"

namespace cp {

constexpr int kNetThreads = 128;
constexpr int kNetMaxC1 = 16, kNetMaxC2 = 32, kNetMaxClasses = 4;
constexpr int kConv1H = kImgRows - 2, kConv1W = kImgCols - 2;   // 13 x 10
constexpr int kPool1H = kConv1H / 2, kPool1W = kConv1W / 2;     // 6 x 5
constexpr int kConv2H = kPool1H - 2, kConv2W = kPool1W - 2;     // 4 x 3
constexpr int kPool2H = kConv2H / 2, kPool2W = kConv2W / 2;     // 2 x 1
constexpr u32 kConeLowConfidence = 16u;  // flag: the decision sits within 2e-6 of the 0.8 threshold

// Weights as laid out by cp_color_net_load (transposed so that consecutive threads read consecutive words):
//   w1t[9][c1]  b1[c1]  w2t[9 * c1][c2]  b2[c2]  scale[c2]  shift[c2]  wd[classes][kPool2H * kPool2W * c2]  bd[classes]
struct ColorNetDev {
  const float* w1t;
  const float* b1;
  const float* w2t;
  const float* b2;
  const float* scale;
  const float* shift;
  const float* wd;
  const float* bd;
  u32 c1, c2, classes;
  float threshold;
};

// A cone without an image (raster_flags beyond CP_CONE_AMBIGUOUS: an empty crop, or one numpy would raise on) gets
// colour 255 and zero outputs; returns true for it.  The whole CTA calls this.
__device__ __forceinline__ bool color_no_image(u32 cone, u32 rf, u32 NC, uint8_t* __restrict__ colors,
                                               float* __restrict__ probs, float* __restrict__ logits_out,
                                               u32* __restrict__ flags_out) {
  if (!(rf & ~kConeAmbiguous)) return false;   // the service skips (empty) or raises (bad index / intensity)
  if (threadIdx.x == 0) {
    colors[cone] = 255;
    if (flags_out) flags_out[cone] = rf;
  }
  if (probs && threadIdx.x < NC) probs[(size_t)cone * NC + threadIdx.x] = 0.f;
  if (logits_out && threadIdx.x < NC) logits_out[(size_t)cone * NC + threadIdx.x] = 0.f;
  return true;
}

// The service's answer from the network's outputs p[NC] (and the logits l[NC] reported beside them): argmax + 1 when
// the largest output is >= threshold, else 0 (:116-120); CP_CONE_LOW_CONFIDENCE when it lies within 2e-6 of it.
// One thread calls this.
__device__ __forceinline__ void color_decide(u32 cone, u32 rf, const float* p, const float* l, u32 NC, float threshold,
                                             uint8_t* __restrict__ colors, float* __restrict__ probs,
                                             float* __restrict__ logits_out, u32* __restrict__ flags_out) {
  float best = -INFINITY;
  u32 arg = 0;
  for (u32 j = 0; j < NC; ++j) {
    if (probs) probs[(size_t)cone * NC + j] = p[j];
    if (logits_out) logits_out[(size_t)cone * NC + j] = l[j];
    if (p[j] > best) {   // np.argmax: first maximum
      best = p[j];
      arg = j;
    }
  }
  colors[cone] = best >= threshold ? (uint8_t)(arg + 1) : (uint8_t)0;
  if (flags_out) flags_out[cone] = rf | (fabsf(best - threshold) < 2e-6f ? kConeLowConfidence : 0u);
}

// grid = cones.  images [n][15][12] uint8; raster_flags (optional) = cone_raster_kernel's flags: a cone whose image
// could not be drawn (empty crop, numpy would raise) gets colour 255 and zero probabilities.
__global__ void __launch_bounds__(kNetThreads) cone_color_kernel(const uint8_t* __restrict__ images,
                                                                 const u32* __restrict__ raster_flags,
                                                                 const __grid_constant__ ColorNetDev net,
                                                                 uint8_t* __restrict__ colors,
                                                                 float* __restrict__ probs, float* __restrict__ logits_out,
                                                                 u32* __restrict__ flags_out) {
  __shared__ float s_in[kImgPix];
  __shared__ float s_a[kConv1H * kConv1W * kNetMaxC1];   // conv1 output, later conv2 output
  __shared__ float s_b[kPool1H * kPool1W * kNetMaxC1];   // pool1 output, later the flattened features
  __shared__ float s_logit[kNetMaxClasses];
  const u32 cone = blockIdx.x, tid = threadIdx.x;
  const u32 C1 = net.c1, C2 = net.c2, NC = net.classes;
  const u32 rf = raster_flags ? raster_flags[cone] : 0u;
  if (color_no_image(cone, rf, NC, colors, probs, logits_out, flags_out)) return;
  for (u32 i = tid; i < kImgPix; i += kNetThreads) s_in[i] = (float)images[(size_t)cone * kImgPix + i];
  __syncthreads();
  // conv1 + ReLU: out[y][x][c], c fastest
  for (u32 o = tid; o < kConv1H * kConv1W * C1; o += kNetThreads) {
    const u32 c = o % C1, x = (o / C1) % kConv1W, y = o / (C1 * kConv1W);
    float acc = 0.f;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
      for (int kx = 0; kx < 3; ++kx)
        acc = __fadd_rn(acc, __fmul_rn(s_in[(y + ky) * kImgCols + x + kx], __ldg(net.w1t + (ky * 3 + kx) * C1 + c)));
    acc = __fadd_rn(acc, __ldg(net.b1 + c));
    s_a[o] = fmaxf(acc, 0.f);
  }
  __syncthreads();
  // pool1 2x2 stride 2 (VALID: the odd last row of 13 is dropped)
  for (u32 o = tid; o < kPool1H * kPool1W * C1; o += kNetThreads) {
    const u32 c = o % C1, x = (o / C1) % kPool1W, y = o / (C1 * kPool1W);
    const float* p = s_a + ((2 * y) * kConv1W + 2 * x) * C1 + c;
    s_b[o] = fmaxf(fmaxf(p[0], p[C1]), fmaxf(p[kConv1W * C1], p[kConv1W * C1 + C1]));
  }
  __syncthreads();
  // conv2 + ReLU into s_a
  for (u32 o = tid; o < kConv2H * kConv2W * C2; o += kNetThreads) {
    const u32 c = o % C2, x = (o / C2) % kConv2W, y = o / (C2 * kConv2W);
    float acc = 0.f;
    for (int ky = 0; ky < 3; ++ky)
      for (int kx = 0; kx < 3; ++kx) {
        const float* in = s_b + ((y + ky) * kPool1W + x + kx) * C1;
        const float* w = net.w2t + (size_t)((ky * 3 + kx) * C1) * C2 + c;
        for (u32 ci = 0; ci < C1; ++ci) acc = __fadd_rn(acc, __fmul_rn(in[ci], __ldg(w + (size_t)ci * C2)));
      }
    acc = __fadd_rn(acc, __ldg(net.b2 + c));
    s_a[o] = fmaxf(acc, 0.f);
  }
  __syncthreads();
  // pool2 (4x3 -> 2x1: the third column is dropped) + per-channel scale, shift; flatten in NHWC order
  for (u32 o = tid; o < kPool2H * kPool2W * C2; o += kNetThreads) {
    const u32 c = o % C2, y = o / C2;
    const float* p = s_a + ((2 * y) * kConv2W) * C2 + c;
    const float m = fmaxf(fmaxf(p[0], p[C2]), fmaxf(p[kConv2W * C2], p[kConv2W * C2 + C2]));
    s_b[o] = __fadd_rn(__fmul_rn(m, __ldg(net.scale + c)), __ldg(net.shift + c));
  }
  __syncthreads();
  if (tid < NC) {
    const u32 K = kPool2H * kPool2W * C2;
    float acc = 0.f;
    for (u32 k = 0; k < K; ++k) acc = __fadd_rn(acc, __fmul_rn(s_b[k], __ldg(net.wd + (size_t)tid * K + k)));
    s_logit[tid] = __fadd_rn(acc, __ldg(net.bd + tid));
  }
  __syncthreads();
  if (tid == 0) {
    float m = s_logit[0];
    for (u32 j = 1; j < NC; ++j) m = fmaxf(m, s_logit[j]);
    float e[kNetMaxClasses], s = 0.f;
    for (u32 j = 0; j < NC; ++j) {
      e[j] = expf(__fsub_rn(s_logit[j], m));
      s = __fadd_rn(s, e[j]);
    }
    for (u32 j = 0; j < NC; ++j) e[j] = __fdiv_rn(e[j], s);
    color_decide(cone, rf, e, s_logit, NC, net.threshold, colors, probs, logits_out, flags_out);
  }
}

// ---- color_graph_kernel: any graph cp_tflite::read_color_graph accepts -----------------------------------------
// The loader lowers the graph to a layer program (GraphLayer, tflite_reader.hpp) passed by value; all weights sit in
// one device buffer.  One CTA per cone; the activations ping-pong between the two ends of one dynamic shared-memory
// buffer of smem_floats floats (layer i reads one end and writes the other, so the largest input + output pair of
// a layer is what must fit), each layer spreads its outputs over the threads, and a barrier separates layers.
// Arithmetic in the order of TFLite's reference kernels, as cone_color_kernel: multiplies and adds rounded
// separately; convolution sums over (filter_y, filter_x, in_channel) and depthwise over (filter_y, filter_x),
// skipping taps outside the input, then adds the bias and clamps; AVERAGE_POOL divides by the in-bounds taps; MEAN
// sums over h, then w, and divides by H*W; FULLY_CONNECTED sums its inputs in order; SOFTMAX is
// expf((x - max) * beta) / sum.  The numpy checker (oracle/color_graph_ref.py) evaluates the same order, so outputs
// before the softmax are bit-identical to it.
constexpr int kGraphThreads = 128;
constexpr int kGraphMaxOps = (int)cp_tflite::kGraphMaxOps;
constexpr int kGraphMaxClasses = 3;

struct ColorGraphDev {
  const float* w;
  u32 n_layers, classes, out, logits;
  float threshold;
  cp_tflite::GraphLayer layer[kGraphMaxOps];
};

__device__ __forceinline__ float clampf(float v, float lo, float hi) { return fminf(fmaxf(v, lo), hi); }

__global__ void __maxnreg__(64) color_graph_kernel(const uint8_t* __restrict__ images,
                                                                    const u32* __restrict__ raster_flags,
                                                                    const __grid_constant__ ColorGraphDev net,
                                                                    uint8_t* __restrict__ colors,
                                                                    float* __restrict__ probs,
                                                                    float* __restrict__ logits_out,
                                                                    u32* __restrict__ flags_out) {
  extern __shared__ float s_act[];
  const u32 cone = blockIdx.x, tid = threadIdx.x, NC = net.classes;
  const u32 rf = raster_flags ? raster_flags[cone] : 0u;
  if (color_no_image(cone, rf, NC, colors, probs, logits_out, flags_out)) return;
  for (u32 i = tid; i < kImgPix; i += kGraphThreads) s_act[i] = (float)images[(size_t)cone * kImgPix + i];
  __syncthreads();
  const float* __restrict__ W = net.w;
  for (u32 l = 0; l < net.n_layers; ++l) {
    const cp_tflite::GraphLayer& L = net.layer[l];
    const float* in = s_act + L.src;
    float* out = s_act + L.dst;
    const int IH = L.ih, IW = L.iw, IC = L.ic, OW = L.ow, OC = L.oc;
    const u32 n_out = (u32)(L.oh * OW * OC);
    switch (L.op) {
      case cp_tflite::G_CONV:
        for (u32 o = tid; o < n_out; o += kGraphThreads) {
          const int c = (int)(o % OC), x = (int)((o / OC) % OW), y = (int)(o / (OC * OW));
          const int y0 = y * L.sh - L.pt, x0 = x * L.sw - L.pl;
          float acc = 0.f;
          for (int ky = 0; ky < L.kh; ++ky) {
            const int iy = y0 + ky;
            if (iy < 0 || iy >= IH) continue;
            for (int kx = 0; kx < L.kw; ++kx) {
              const int ix = x0 + kx;
              if (ix < 0 || ix >= IW) continue;
              const float* a = in + (iy * IW + ix) * IC;
              const float* w = W + L.w + (size_t)((ky * L.kw + kx) * IC) * OC + c;
              for (int ci = 0; ci < IC; ++ci) acc = __fadd_rn(acc, __fmul_rn(a[ci], __ldg(w + (size_t)ci * OC)));
            }
          }
          out[o] = clampf(__fadd_rn(acc, __ldg(W + L.b + c)), L.lo, L.hi);
        }
        break;
      case cp_tflite::G_DWCONV:
        for (u32 o = tid; o < n_out; o += kGraphThreads) {
          const int c = (int)(o % OC), x = (int)((o / OC) % OW), y = (int)(o / (OC * OW)), ci = c / L.m;
          const int y0 = y * L.sh - L.pt, x0 = x * L.sw - L.pl;
          float acc = 0.f;
          for (int ky = 0; ky < L.kh; ++ky) {
            const int iy = y0 + ky;
            if (iy < 0 || iy >= IH) continue;
            for (int kx = 0; kx < L.kw; ++kx) {
              const int ix = x0 + kx;
              if (ix < 0 || ix >= IW) continue;
              acc = __fadd_rn(acc, __fmul_rn(in[(iy * IW + ix) * IC + ci], __ldg(W + L.w + (size_t)(ky * L.kw + kx) * OC + c)));
            }
          }
          out[o] = clampf(__fadd_rn(acc, __ldg(W + L.b + c)), L.lo, L.hi);
        }
        break;
      case cp_tflite::G_MAXPOOL:
      case cp_tflite::G_AVGPOOL:
        for (u32 o = tid; o < n_out; o += kGraphThreads) {
          const int c = (int)(o % OC), x = (int)((o / OC) % OW), y = (int)(o / (OC * OW));
          const int y0 = y * L.sh - L.pt, x0 = x * L.sw - L.pl;
          float m = -INFINITY, sum = 0.f;
          int count = 0;
          for (int ky = 0; ky < L.kh; ++ky) {
            const int iy = y0 + ky;
            if (iy < 0 || iy >= IH) continue;
            for (int kx = 0; kx < L.kw; ++kx) {
              const int ix = x0 + kx;
              if (ix < 0 || ix >= IW) continue;
              const float v = in[(iy * IW + ix) * IC + c];
              m = fmaxf(m, v);
              sum = __fadd_rn(sum, v);
              ++count;
            }
          }
          out[o] = clampf(L.op == cp_tflite::G_MAXPOOL ? m : __fdiv_rn(sum, (float)count), L.lo, L.hi);
        }
        break;
      case cp_tflite::G_MEAN:
        for (u32 c = tid; c < (u32)OC; c += kGraphThreads) {
          float sum = 0.f;
          for (int y = 0; y < IH; ++y)
            for (int x = 0; x < IW; ++x) sum = __fadd_rn(sum, in[(y * IW + x) * IC + c]);
          out[c] = __fdiv_rn(sum, (float)(IH * IW));
        }
        break;
      case cp_tflite::G_MUL:
      case cp_tflite::G_ADD:
        for (u32 o = tid; o < n_out; o += kGraphThreads) {
          const float k = __ldg(W + L.w + (L.m == 1 ? 0u : o % (u32)OC));
          out[o] = clampf(L.op == cp_tflite::G_MUL ? __fmul_rn(in[o], k) : __fadd_rn(in[o], k), L.lo, L.hi);
        }
        break;
      case cp_tflite::G_CLAMP:
        for (u32 o = tid; o < n_out; o += kGraphThreads) out[o] = clampf(in[o], L.lo, L.hi);
        break;
      case cp_tflite::G_FC:
        for (u32 n = tid; n < (u32)OC; n += kGraphThreads) {
          float acc = 0.f;
          for (int k = 0; k < IC; ++k) acc = __fadd_rn(acc, __fmul_rn(in[k], __ldg(W + L.w + (size_t)k * OC + n)));
          out[n] = clampf(__fadd_rn(acc, __ldg(W + L.b + n)), L.lo, L.hi);
        }
        break;
      case cp_tflite::G_SOFTMAX:
        if (tid == 0) {
          float m = in[0];
          for (int j = 1; j < OC; ++j) m = fmaxf(m, in[j]);
          float s = 0.f;
          for (int j = 0; j < OC; ++j) {
            out[j] = expf(__fmul_rn(__fsub_rn(in[j], m), L.lo));
            s = __fadd_rn(s, out[j]);
          }
          for (int j = 0; j < OC; ++j) out[j] = __fdiv_rn(out[j], s);
        }
        break;
    }
    __syncthreads();
  }
  if (tid == 0) color_decide(cone, rf, s_act + net.out, s_act + net.logits, NC, net.threshold, colors, probs, logits_out, flags_out);
}

}  // namespace cp
