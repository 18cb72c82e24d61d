"""TEST INFRASTRUCTURE — numpy forward pass of every colour classifier `cones_perception_b200.tflite_model.load`
accepts: dam_net and the retrained sequential CNNs the device evaluates with color_graph_kernel.  The checker for
`cp_color_net_load_tflite` with such a model.  Only tests/ and tools/ may import this.

Same contract as `oracle/dam_net_ref.py` (which restates dam_net alone): the 15x12 uint8 image is cast to float32
without scaling, the graph is evaluated in fp32, and the answer is `argmax + 1` when the largest output is >= 0.8,
else 0 (`decide`).  The operators are restated from TFLite's published reference kernels (`tensorflow/lite/kernels/
internal/reference/{conv,depthwiseconv_float,pooling,reduce,fully_connected,softmax}.h`): NHWC, OHWI filters, SAME /
VALID padding with taps outside the input skipped, accumulation in the order filter_y, filter_x, in_channel
(depthwise: filter_y, filter_x), multiply and add rounded separately, bias added after the accumulation, then the
fused activation; the average pool divides by the in-bounds taps, MEAN sums over h then w and divides by H*W,
softmax is exp((x - max) * beta) / sum.  On dam_net it gives dam_net_ref.forward's outputs bit for bit
(tests/test_color_graphs.py).

**Parity unpinned**, as for dam_net: no TFLite interpreter is available to compare with.
"""
from __future__ import annotations

import numpy as np

from oracle.dam_net_ref import THRESHOLD, decide  # noqa: F401  (the service's decision, shared)

_CLAMP = {"NONE": (None, None), "RELU": (0.0, None), "RELU6": (0.0, 6.0), "RELU_N1_TO_1": (-1.0, 1.0)}


def _act(x, act):
    lo, hi = _CLAMP[act]
    if lo is not None:
        x = np.maximum(x, np.float32(lo))
    if hi is not None:
        x = np.minimum(x, np.float32(hi))
    return x


def _taps(n_in, n_out, k, s, pad):
    """For each filter offset: (output indices, input indices) of the taps inside the input."""
    out = []
    for d in range(k):
        src = np.arange(n_out) * s - pad + d
        ok = (src >= 0) & (src < n_in)
        out.append((np.nonzero(ok)[0], src[ok]))
    return out


def _window(o, H, W, kh, kw):
    Ho, pt = _window1(o["padding"], H, kh, o["stride_h"])
    Wo, pl = _window1(o["padding"], W, kw, o["stride_w"])
    return Ho, Wo, _taps(H, Ho, kh, o["stride_h"], pt), _taps(W, Wo, kw, o["stride_w"], pl)


def _window1(padding, n, k, s):
    if padding == "SAME":
        out = (n + s - 1) // s
        return out, max((out - 1) * s + k - n, 0) // 2
    return (n - k) // s + 1, 0


def conv2d(x, w, b, o):
    """x [B,H,W,Ci], w [Co,kh,kw,Ci]: sequential fp32 accumulation over (ky, kx, ci) like the reference kernel,
    taps outside the input skipped, then the bias, then the activation."""
    B, H, W, Ci = x.shape
    Co, kh, kw, _ = w.shape
    Ho, Wo, ty, tx = _window(o, H, W, kh, kw)
    acc = np.zeros((B, Ho, Wo, Co), np.float32)
    for ky in range(kh):
        oy, iy = ty[ky]
        for kx in range(kw):
            ox, ix = tx[kx]
            if not len(oy) or not len(ox):
                continue
            for ci in range(Ci):
                acc[:, oy[:, None], ox[None, :], :] += x[:, iy[:, None], ix[None, :], ci, None] * w[None, None, None, :, ky, kx, ci]
    return _act(acc + b, o["act"])


def depthwise_conv2d(x, w, b, o):
    """x [B,H,W,C], w [1,kh,kw,C*m]: output channel c reads input channel c // m; accumulation over (ky, kx)."""
    B, H, W, C = x.shape
    _, kh, kw, Co = w.shape
    xr = np.repeat(x, Co // C, axis=3)
    Ho, Wo, ty, tx = _window(o, H, W, kh, kw)
    acc = np.zeros((B, Ho, Wo, Co), np.float32)
    for ky in range(kh):
        oy, iy = ty[ky]
        for kx in range(kw):
            ox, ix = tx[kx]
            if len(oy) and len(ox):
                acc[:, oy[:, None], ox[None, :], :] += xr[:, iy[:, None], ix[None, :], :] * w[0, ky, kx]
    return _act(acc + b, o["act"])


def pool(x, o, average):
    """MAX_POOL_2D / AVERAGE_POOL_2D over the taps inside the input; the average divides by their count."""
    B, H, W, C = x.shape
    Ho, Wo, ty, tx = _window(o, H, W, o["filter_h"], o["filter_w"])
    acc = np.full((B, Ho, Wo, C), 0.0 if average else -np.inf, np.float32)
    cnt = np.zeros((Ho, Wo), np.float32)
    for ky in range(o["filter_h"]):
        oy, iy = ty[ky]
        for kx in range(o["filter_w"]):
            ox, ix = tx[kx]
            v = x[:, iy[:, None], ix[None, :], :]
            if average:
                acc[:, oy[:, None], ox[None, :], :] += v
                cnt[oy[:, None], ox[None, :]] += 1
            else:
                acc[:, oy[:, None], ox[None, :], :] = np.maximum(acc[:, oy[:, None], ox[None, :], :], v)
    if average:
        acc = acc / cnt[None, :, :, None]
    return _act(acc, o["act"])


def mean(x, o):
    """MEAN over axes {1,2} of x [B,H,W,C]: summed over h, then w, divided by H*W."""
    B, H, W, C = x.shape
    s = np.zeros((B, C), np.float32)
    for h in range(H):
        for w in range(W):
            s += x[:, h, w, :]
    y = s / np.float32(H * W)
    return y.reshape(B, 1, 1, C) if o.get("keep_dims") else y


def forward_batch(graph, images_u8: np.ndarray):
    """[B,15,12] uint8 images -> (outputs [B,n], logits [B,n]), all arithmetic fp32.  logits: the input of the final
    SOFTMAX, or the output when there is none."""
    imgs = np.asarray(images_u8)
    B = len(imgs)
    x = imgs.astype(np.float32).reshape((B,) + tuple(graph.tensors[graph.inputs[0]].shape[1:]))
    const = lambda i: graph.tensors[i].data
    logits = None
    for op in graph.ops:
        o = op.options
        if op.kind in ("MUL", "ADD"):
            k = const(next(i for i in op.inputs if graph.tensors[i].data is not None))   # either operand
            k = k.reshape(-1) if k.size > 1 else k.reshape(())
        if op.kind == "CONV_2D":
            y = conv2d(x, const(op.inputs[1]), const(op.inputs[2]), o)
        elif op.kind == "DEPTHWISE_CONV_2D":
            y = depthwise_conv2d(x, const(op.inputs[1]), const(op.inputs[2]), o)
        elif op.kind in ("MAX_POOL_2D", "AVERAGE_POOL_2D"):
            y = pool(x, o, op.kind == "AVERAGE_POOL_2D")
        elif op.kind == "MEAN":
            y = mean(x, o)
        elif op.kind == "MUL":
            y = _act(x * k, o["act"])
        elif op.kind == "ADD":
            y = _act(x + k, o["act"])
        elif op.kind == "RELU":
            y = _act(x, "RELU")
        elif op.kind == "RELU6":
            y = _act(x, "RELU6")
        elif op.kind == "RESHAPE":
            shape = tuple(graph.tensors[op.outputs[0]].shape[1:])
            y = x.reshape((B,) + shape) if shape else x.reshape(B, -1)   # NHWC row-major
        elif op.kind == "FULLY_CONNECTED":
            w = const(op.inputs[1])
            b = const(op.inputs[2]) if len(op.inputs) > 2 and op.inputs[2] >= 0 else np.zeros(w.shape[0], np.float32)
            xf = x.reshape(B, -1)
            acc = np.zeros((B, w.shape[0]), np.float32)
            for k_ in range(w.shape[1]):            # sequential over the input features
                acc += xf[:, k_, None] * w[None, :, k_]
            y = _act(acc + b, o["act"])
        elif op.kind == "SOFTMAX":
            xf = x.reshape(B, -1)
            logits = xf
            z = (xf - xf.max(axis=1, keepdims=True)) * np.float32(o["beta"])
            e = np.exp(z.astype(np.float32)).astype(np.float32)
            s = np.zeros((B, 1), np.float32)
            for j in range(e.shape[1]):
                s = (s + e[:, j:j + 1]).astype(np.float32)
            y = (e / s).astype(np.float32).reshape(x.shape)
        else:
            raise ValueError(op.kind)
        x = y.astype(np.float32)
    out = x.reshape(B, -1)
    return out, (logits if logits is not None else out)


def forward(graph, image_u8: np.ndarray):
    """One 15x12 uint8 image -> (outputs [n], logits [n]): softmax probabilities and their input for dam_net."""
    p, l = forward_batch(graph, np.asarray(image_u8)[None])
    return p[0], l[0]
