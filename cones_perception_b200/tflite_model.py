"""A minimal reader for TensorFlow-Lite flatbuffers — just enough to load the colour classifier the reference
ships (`models/dam_net/dam_net.tflite`, loaded by `scripts/color_classifier_server.py:66-71` through
`tf.lite.Interpreter`).  No TensorFlow, no `flatbuffers` package: the flatbuffer wire format is walked by hand.

`load` accepts exactly the sequential float32 CNNs the library evaluates on the device (the contract of
`cp_color_net_load_tflite`, checked the same way by `csrc/tflite_reader.hpp::read_color_graph`): one input
[1,15,12,1], one output [1,n] with 1 <= n <= 3, at most 64 operators in a chain (each one's first input, or either
input of MUL / ADD, is the previous output; every other input is a constant), activations [1,...] of rank 2 to 4,
no quantisation, and only these operators: CONV_2D and DEPTHWISE_CONV_2D (SAME / VALID, any stride, dilation 1),
MAX_POOL_2D and AVERAGE_POOL_2D, MEAN over axes {1,2}, MUL / ADD with a scalar, [C] or [1,1,1,C] constant, RELU,
RELU6, RESHAPE, FULLY_CONNECTED (default weights format, bias optional, keep_num_dims false) and a final SOFTMAX
(finite beta); fused activations NONE, RELU, RELU6, RELU_N1_TO_1.  The largest input + output pair of a layer must
fit 227 KB.  Anything else raises `UnsupportedModel`, so that a different model is refused instead of being
evaluated wrongly.

Schema facts used (tensorflow/lite/schema/schema.fbs, v3):
  Model        : 0 version, 1 operator_codes, 2 subgraphs, 3 description, 4 buffers
  OperatorCode : 0 deprecated_builtin_code (int8), 1 custom_code, 2 version, 3 builtin_code (int32)
  SubGraph     : 0 tensors, 1 inputs, 2 outputs, 3 operators, 4 name
  Tensor       : 0 shape, 1 type, 2 buffer, 3 name, 4 quantization     QuantizationParameters: 2 scale
  Operator     : 0 opcode_index, 1 inputs, 2 outputs, 3 builtin_options_type, 4 builtin_options
  Buffer       : 0 data
  Conv2DOptions        : 0 padding, 1 stride_w, 2 stride_h, 3 fused_activation, 4 dilation_w, 5 dilation_h
  Pool2DOptions        : 0 padding, 1 stride_w, 2 stride_h, 3 filter_width, 4 filter_height, 5 fused_activation
  DepthwiseConv2DOptions: 0 padding, 1 stride_w, 2 stride_h, 3 depth_multiplier, 4 fused_activation, 5 dilation_w,
                         6 dilation_h
  FullyConnectedOptions: 0 fused_activation, 1 weights_format, 2 keep_num_dims
  SoftmaxOptions       : 0 beta          Mul/AddOptions: 0 fused_activation          ReducerOptions: 0 keep_dims
"""
from __future__ import annotations

import struct
from dataclasses import dataclass, field

import numpy as np


class UnsupportedModel(ValueError):
    pass


BUILTIN = {0: "ADD", 1: "AVERAGE_POOL_2D", 3: "CONV_2D", 4: "DEPTHWISE_CONV_2D", 9: "FULLY_CONNECTED",
           17: "MAX_POOL_2D", 18: "MUL", 19: "RELU", 21: "RELU6", 22: "RESHAPE", 25: "SOFTMAX", 40: "MEAN"}
ACT = {0: "NONE", 1: "RELU", 2: "RELU_N1_TO_1", 3: "RELU6", 4: "TANH", 5: "SIGN_BIT"}
MAX_OPS = 64
SMEM_BYTES = 227 * 1024      # dynamic shared memory one block may hold on sm_100a
PADDING = {0: "SAME", 1: "VALID"}
TENSOR_TYPE = {0: np.float32, 1: np.float16, 2: np.int32, 3: np.uint8, 4: np.int64, 9: np.int8}


class _Table:
    """One flatbuffer table: field slot -> absolute position (0 when the field is absent)."""

    def __init__(self, buf: bytes, pos: int):
        self.buf, self.pos = buf, pos
        vt = pos - struct.unpack_from("<i", buf, pos)[0]
        vt_len = struct.unpack_from("<H", buf, vt)[0]
        self.slots = [struct.unpack_from("<H", buf, vt + 4 + 2 * i)[0] for i in range((vt_len - 4) // 2)]

    def _at(self, slot: int) -> int:
        return self.pos + self.slots[slot] if slot < len(self.slots) and self.slots[slot] else 0

    def scalar(self, slot: int, fmt: str, default=0):
        p = self._at(slot)
        return struct.unpack_from("<" + fmt, self.buf, p)[0] if p else default

    def _indirect(self, slot: int) -> int:
        p = self._at(slot)
        return p + struct.unpack_from("<I", self.buf, p)[0] if p else 0

    def table(self, slot: int):
        p = self._indirect(slot)
        return _Table(self.buf, p) if p else None

    def string(self, slot: int) -> str:
        p = self._indirect(slot)
        if not p:
            return ""
        n = struct.unpack_from("<I", self.buf, p)[0]
        return self.buf[p + 4:p + 4 + n].decode("utf-8", "replace")

    def vector(self, slot: int, dtype) -> np.ndarray:
        p = self._indirect(slot)
        if not p:
            return np.zeros(0, dtype)
        n = struct.unpack_from("<I", self.buf, p)[0]
        return np.frombuffer(self.buf, dtype=dtype, count=n, offset=p + 4).copy()

    def tables(self, slot: int) -> list["_Table"]:
        p = self._indirect(slot)
        if not p:
            return []
        n = struct.unpack_from("<I", self.buf, p)[0]
        out = []
        for i in range(n):
            e = p + 4 + 4 * i
            out.append(_Table(self.buf, e + struct.unpack_from("<I", self.buf, e)[0]))
        return out


@dataclass
class Tensor:
    name: str
    shape: tuple
    dtype: type
    data: np.ndarray | None      # constant tensors only
    quant_scale: tuple = ()      # QuantizationParameters.scale (refused when not empty)


@dataclass
class Op:
    kind: str
    inputs: list
    outputs: list
    options: dict = field(default_factory=dict)


@dataclass
class Graph:
    tensors: list
    ops: list
    inputs: list
    outputs: list
    description: str = ""


def load(path_or_bytes) -> Graph:
    buf = path_or_bytes if isinstance(path_or_bytes, (bytes, bytearray)) else open(path_or_bytes, "rb").read()
    buf = bytes(buf)
    if len(buf) < 8 or buf[4:8] != b"TFL3":
        raise UnsupportedModel("not a TFL3 flatbuffer")
    model = _Table(buf, struct.unpack_from("<I", buf, 0)[0])
    codes = []
    for oc in model.tables(1):
        code = oc.scalar(3, "i", 0) or oc.scalar(0, "b", 0)
        if oc.string(1):
            raise UnsupportedModel(f"custom operator {oc.string(1)!r}")
        codes.append(code)
    buffers = [b.vector(0, np.uint8) for b in model.tables(4)]
    sgs = model.tables(2)
    if len(sgs) != 1:
        raise UnsupportedModel(f"{len(sgs)} subgraphs")
    sg = sgs[0]
    tensors = []
    for t in sg.tables(0):
        ttype = t.scalar(1, "b", 0)
        if ttype not in TENSOR_TYPE:
            raise UnsupportedModel(f"tensor type {ttype}")
        dt = TENSOR_TYPE[ttype]
        shape = tuple(int(v) for v in t.vector(0, np.int32))
        bi = t.scalar(2, "I", 0)
        if bi >= len(buffers):
            raise UnsupportedModel("buffer index out of range")
        raw = buffers[bi]
        data = None
        if raw.size:
            if raw.size != int(np.prod(shape, dtype=np.int64)) * np.dtype(dt).itemsize:
                raise UnsupportedModel(f"tensor {len(tensors)}: constant tensor has an unexpected size")
            data = raw.view(dt).reshape(shape) if shape else raw.view(dt)
        q = t.table(4)
        scale = tuple(float(v) for v in q.vector(2, np.float32)) if q is not None else ()
        tensors.append(Tensor(t.string(3), shape, dt, data, scale))
    ops = []
    for o in sg.tables(3):
        ci = o.scalar(0, "I", 0)
        if ci >= len(codes):
            raise UnsupportedModel("opcode index out of range")
        code = codes[ci]
        kind = BUILTIN.get(code)
        if kind is None:
            raise UnsupportedModel(f"operator {len(ops)}: builtin operator code {code} is not supported")
        opt = o.table(4)
        options = {}
        act = lambda slot: ACT.get(opt.scalar(slot, "b"), "UNKNOWN") if opt is not None else "NONE"
        if kind in ("CONV_2D", "DEPTHWISE_CONV_2D") and opt is not None:
            dw = kind == "DEPTHWISE_CONV_2D"
            options = {"padding": PADDING.get(opt.scalar(0, "b"), "UNKNOWN"), "stride_w": opt.scalar(1, "i"),
                       "stride_h": opt.scalar(2, "i"), "act": act(4 if dw else 3),
                       "dilation_w": opt.scalar(5 if dw else 4, "i", 1), "dilation_h": opt.scalar(6 if dw else 5, "i", 1)}
            if dw:
                options["depth_multiplier"] = opt.scalar(3, "i")
        elif kind in ("MAX_POOL_2D", "AVERAGE_POOL_2D") and opt is not None:
            options = {"padding": PADDING.get(opt.scalar(0, "b"), "UNKNOWN"), "stride_w": opt.scalar(1, "i"),
                       "stride_h": opt.scalar(2, "i"), "filter_w": opt.scalar(3, "i"),
                       "filter_h": opt.scalar(4, "i"), "act": act(5)}
        elif kind == "FULLY_CONNECTED":
            options = {"act": act(0), "weights_format": opt.scalar(1, "b") if opt is not None else 0,
                       "keep_num_dims": bool(opt.scalar(2, "B")) if opt is not None else False}
        elif kind == "SOFTMAX":
            options = {"beta": opt.scalar(0, "f", 1.0) if opt is not None else 1.0}
        elif kind in ("MUL", "ADD"):
            options = {"act": act(0)}
        elif kind == "MEAN":
            options = {"keep_dims": bool(opt.scalar(0, "B")) if opt is not None else False}
        ops.append(Op(kind, [int(v) for v in o.vector(1, np.int32)], [int(v) for v in o.vector(2, np.int32)], options))
    g = Graph(tensors, ops, [int(v) for v in sg.vector(1, np.int32)], [int(v) for v in sg.vector(2, np.int32)],
              model.string(3))
    check(g)
    return g


_ACT_OK = ("NONE", "RELU", "RELU6", "RELU_N1_TO_1")


def _window(padding, n, k, s):
    """Output extent and padding before (TFLite's ComputePaddingHeightWidth, dilation 1)."""
    if padding == "SAME":
        out = (n + s - 1) // s
        return out, max((out - 1) * s + k - n, 0) // 2
    return ((n - k) // s + 1 if n >= k else 0), 0


def check(g: Graph) -> list:
    """Raises UnsupportedModel unless `g` is in the accepted subset (module docstring).  Returns the activation
    shape after each operator."""
    def where(i, op):
        return f"operator {i} ({op.kind})"

    def is_const(t):
        return t >= 0 and g.tensors[t].data is not None

    def tensor_ok(t, w):
        if t >= len(g.tensors):
            raise UnsupportedModel(f"{w}: tensor index out of range")
        if g.tensors[t].quant_scale:
            raise UnsupportedModel(f"{w}: quantised tensors are not supported")
        if len(g.tensors[t].shape) > 4 or any(d < 1 or d > 1 << 20 for d in g.tensors[t].shape):
            raise UnsupportedModel(f"{w}: tensor shape outside rank 4 / dimensions 1..2^20")

    if not 1 <= len(g.ops) <= MAX_OPS:
        raise UnsupportedModel(f"operator count {len(g.ops)} outside 1..{MAX_OPS}")
    if len(g.inputs) != 1 or len(g.outputs) != 1:
        raise UnsupportedModel("expected one graph input and one graph output")
    cur = g.inputs[0]
    tensor_ok(cur, "graph input")
    t0 = g.tensors[cur]
    if t0.dtype != np.float32 or t0.shape != (1, 15, 12, 1) or t0.data is not None:
        raise UnsupportedModel("input must be a float32 1x15x12x1 tensor")
    shape, shapes, pair, layers = (1, 15, 12, 1), [], 0, 0
    for i, op in enumerate(g.ops):
        w, o = where(i, op), op.options
        if len(op.outputs) != 1:
            raise UnsupportedModel(f"{w}: expected one output")
        ins = op.inputs
        for t in ins + op.outputs:
            if t >= 0:
                tensor_ok(t, w)
        if not ins:
            raise UnsupportedModel(f"{w}: no input")
        chain = 0 if ins[0] == cur else (1 if op.kind in ("MUL", "ADD") and len(ins) == 2 and ins[1] == cur else -1)
        if chain < 0:
            raise UnsupportedModel(f"{w}: the operators do not form a chain")
        if op.kind == "SOFTMAX" and i + 1 < len(g.ops):
            raise UnsupportedModel(f"{w}: SOFTMAX must be the last operator")
        if op.kind in ("CONV_2D", "DEPTHWISE_CONV_2D", "MAX_POOL_2D", "AVERAGE_POOL_2D", "MEAN") and len(shape) != 4:
            raise UnsupportedModel(f"{w}: input must be [1,H,W,C]")
        C = shape[-1]
        H = shape[1] if len(shape) == 4 else 1
        n_in = int(np.prod(shape))
        for k in range(1, len(ins)):
            if k != chain and ins[k] >= 0 and not is_const(ins[k]):
                raise UnsupportedModel(f"{w}: an input other than the chain is not a constant")

        def fconst(t, want=None):
            ten = g.tensors[t]
            if ten.dtype != np.float32:
                raise UnsupportedModel(f"{w}: only float32 constants are supported")
            if ten.data is None or (want is not None and ten.shape != tuple(want)):
                raise UnsupportedModel(f"{w}: constant has an unexpected shape")
            return ten

        def fused(a):
            if a not in _ACT_OK:
                raise UnsupportedModel(f"{w}: fused activation {a} is not supported (NONE, RELU, RELU6, RELU_N1_TO_1)")

        def spatial(kh, kw):
            if o.get("padding") not in ("SAME", "VALID"):
                raise UnsupportedModel(f"{w}: padding must be SAME or VALID")
            if not (1 <= o["stride_w"] <= 64 and 1 <= o["stride_h"] <= 64):
                raise UnsupportedModel(f"{w}: stride outside 1..64")
            oh, _ = _window(o["padding"], H, kh, o["stride_h"])
            ow, _ = _window(o["padding"], shape[2], kw, o["stride_w"])
            return oh, ow

        emit, nxt = True, None
        if op.kind in ("CONV_2D", "DEPTHWISE_CONV_2D"):
            dw = op.kind == "DEPTHWISE_CONV_2D"
            if len(ins) != 3 or ins[2] < 0 or not o:
                raise UnsupportedModel(f"{w}: needs filter, bias and options")
            if o["padding"] not in ("SAME", "VALID"):
                raise UnsupportedModel(f"{w}: padding must be SAME or VALID")
            if not (1 <= o["stride_w"] <= 64 and 1 <= o["stride_h"] <= 64):
                raise UnsupportedModel(f"{w}: stride outside 1..64")
            if o["dilation_w"] != 1 or o["dilation_h"] != 1:
                raise UnsupportedModel(f"{w}: dilation must be 1")
            fused(o["act"])
            f = g.tensors[ins[1]].shape
            if len(f) != 4:
                raise UnsupportedModel(f"{w}: filter must be rank 4")
            if dw:
                if f[0] != 1 or f[3] % C:
                    raise UnsupportedModel(f"{w}: filter must be [1][kh][kw][C*m]")
                if o["depth_multiplier"] not in (0, f[3] // C):
                    raise UnsupportedModel(f"{w}: depth_multiplier disagrees with the filter")
            elif f[3] != C:
                raise UnsupportedModel(f"{w}: filter must be [Co][kh][kw][C]")
            fconst(ins[1], f)
            co = f[3] if dw else f[0]
            fconst(ins[2], (co,))
            oh, ow = spatial(f[1], f[2])
            nxt = (1, oh, ow, co)
        elif op.kind in ("MAX_POOL_2D", "AVERAGE_POOL_2D"):
            if len(ins) != 1 or not o:
                raise UnsupportedModel(f"{w}: needs one input and options")
            if o["padding"] not in ("SAME", "VALID"):
                raise UnsupportedModel(f"{w}: padding must be SAME or VALID")
            if not (1 <= o["stride_w"] <= 64 and 1 <= o["stride_h"] <= 64):
                raise UnsupportedModel(f"{w}: stride outside 1..64")
            if not (1 <= o["filter_w"] <= 64 and 1 <= o["filter_h"] <= 64):
                raise UnsupportedModel(f"{w}: filter outside 1..64")
            fused(o["act"])
            oh, ow = spatial(o["filter_h"], o["filter_w"])
            nxt = (1, oh, ow, C)
        elif op.kind == "MEAN":
            if len(ins) != 2:
                raise UnsupportedModel(f"{w}: needs the axes input")
            ax = g.tensors[ins[1]]
            if ax.dtype != np.int32 or ax.data is None or ax.data.size != 2:
                raise UnsupportedModel(f"{w}: axes must be an int32 constant {{1, 2}}")
            if sorted(int(v) for v in ax.data.reshape(-1)) != [1, 2]:
                raise UnsupportedModel(f"{w}: only axes {{1, 2}} are supported")
            nxt = (1, 1, 1, C) if o.get("keep_dims") else (1, C)
        elif op.kind in ("MUL", "ADD"):
            if len(ins) != 2:
                raise UnsupportedModel(f"{w}: needs two inputs")
            c = g.tensors[ins[1 - chain]]
            if int(np.prod(c.shape)) != 1 and c.shape not in ((C,), (1, 1, 1, C)):
                raise UnsupportedModel(f"{w}: the constant must be a scalar, [C] or [1,1,1,C]")
            fconst(ins[1 - chain])
            fused(o["act"])
        elif op.kind in ("RELU", "RELU6"):
            if len(ins) != 1:
                raise UnsupportedModel(f"{w}: needs one input")
        elif op.kind == "RESHAPE":
            if len(ins) > 2:
                raise UnsupportedModel(f"{w}: too many inputs")
            if len(ins) == 2 and ins[1] >= 0 and not is_const(ins[1]):
                raise UnsupportedModel(f"{w}: the shape input must be a constant")
            nxt = g.tensors[op.outputs[0]].shape
            if int(np.prod(nxt)) != n_in:
                raise UnsupportedModel(f"{w}: the element count changes")
            emit = False
        elif op.kind == "FULLY_CONNECTED":
            if not 2 <= len(ins) <= 3:
                raise UnsupportedModel(f"{w}: needs weights and an optional bias")
            if o["weights_format"] != 0:
                raise UnsupportedModel(f"{w}: only the default weights format is supported")
            if o["keep_num_dims"]:
                raise UnsupportedModel(f"{w}: keep_num_dims is not supported")
            fused(o["act"])
            f = g.tensors[ins[1]].shape
            if len(f) != 2 or f[1] != n_in:
                raise UnsupportedModel(f"{w}: weights must be [N][elements of the input]")
            fconst(ins[1], f)
            if len(ins) == 3 and ins[2] >= 0:
                fconst(ins[2], (f[0],))
            nxt = (1, f[0])
        elif op.kind == "SOFTMAX":
            if len(ins) != 1:
                raise UnsupportedModel(f"{w}: needs one input")
            if C != n_in:
                raise UnsupportedModel(f"{w}: input must hold its elements in the last dimension")
            if not np.isfinite(o["beta"]):
                raise UnsupportedModel(f"{w}: beta must be finite")
        else:
            raise UnsupportedModel(f"{w}: operator not supported")
        if nxt is None:
            nxt = shape
        if emit:
            if min(nxt) < 1:
                raise UnsupportedModel(f"{w}: empty output")
            pair = max(pair, n_in + int(np.prod(nxt)))
            layers += 1
        out = g.tensors[op.outputs[0]]
        if out.dtype != np.float32 or out.data is not None:
            raise UnsupportedModel(f"{w}: output must be a float32 activation")
        if out.shape != tuple(nxt):
            raise UnsupportedModel(f"{w}: the output tensor's shape disagrees with the operator")
        if len(nxt) < 2 or nxt[0] != 1:
            raise UnsupportedModel(f"{w}: activations must be [1,...] of rank 2 to 4")
        shape, cur = tuple(nxt), op.outputs[0]
        shapes.append(shape)
    if cur != g.outputs[0]:
        raise UnsupportedModel("the last operator's output is not the graph output")
    if len(shape) != 2 or not 1 <= shape[1] <= 3:
        raise UnsupportedModel("output must be [1,n] with 1 <= n <= 3")
    if not layers:
        raise UnsupportedModel("no operator computes anything")
    if pair * 4 > SMEM_BYTES:
        raise UnsupportedModel(f"activations need {pair * 4} bytes of shared memory for one layer's input and output, "
                               f"above the {SMEM_BYTES}-byte budget")
    return shapes
