"""TEST INFRASTRUCTURE — writes a `cones_perception_b200.tflite_model.Graph` as a TFL3 flatbuffer, by hand (no
`flatbuffers` package).  The tests use it to build classifiers of other architectures than dam_net with seeded
weights, and damaged or unsupported files for the readers to refuse.  It writes what the Graph holds without
checking it.

Layout: the buffer is written front to back.  Every table's vtable sits just before it (soffset > 0) and every
object a table or vector points at is written after the pointer, so all uoffsets are positive as the format
requires.  Schema slots as in tflite_model.py's docstring.
"""
from __future__ import annotations

import struct

import numpy as np

from cones_perception_b200 import tflite_model as T

_CODE = {v: k for k, v in T.BUILTIN.items()}
_CODE.update({"TANH": 28, "LOGISTIC": 14, "RELU_N1_TO_1": 20})
_ACT = {v: k for k, v in T.ACT.items()}
_PAD = {"SAME": 0, "VALID": 1}
_TYPE = {np.dtype(np.float32): 0, np.dtype(np.float16): 1, np.dtype(np.int32): 2, np.dtype(np.uint8): 3,
         np.dtype(np.int64): 4, np.dtype(np.int8): 9}
# BuiltinOptions union members
_OPT_TYPE = {"CONV_2D": 1, "DEPTHWISE_CONV_2D": 2, "MAX_POOL_2D": 5, "AVERAGE_POOL_2D": 5, "FULLY_CONNECTED": 8,
             "SOFTMAX": 9, "ADD": 11, "RESHAPE": 17, "MUL": 21, "MEAN": 27}


class _Table:
    """fields: list of (slot, fmt, value) for scalars or (slot, None, child) for offsets to a child object."""

    def __init__(self, fields):
        self.fields = fields


class _Vec:
    def __init__(self, fmt=None, items=(), raw=None, tables=None, align=4):
        self.fmt, self.items, self.raw, self.tables, self.align = fmt, list(items), raw, tables, align


class _Str:
    def __init__(self, s):
        self.s = s.encode()


class _Builder:
    def __init__(self):
        self.b = bytearray()

    def pad_to(self, align, extra=0):
        while (len(self.b) + extra) % align:
            self.b.append(0)

    def emit(self, obj) -> int:
        if isinstance(obj, _Table):
            return self._table(obj)
        if isinstance(obj, _Str):
            self.pad_to(4)
            pos = len(self.b)
            self.b += struct.pack("<I", len(obj.s)) + obj.s + b"\0"
            return pos
        return self._vec(obj)

    def _vec(self, v: _Vec) -> int:
        if v.tables is not None:
            self.pad_to(4)
            pos = len(self.b)
            self.b += struct.pack("<I", len(v.tables)) + bytes(4 * len(v.tables))
            for i, t in enumerate(v.tables):
                child = self.emit(t)
                slot = pos + 4 + 4 * i
                struct.pack_into("<I", self.b, slot, child - slot)
            return pos
        data = v.raw if v.raw is not None else b"".join(struct.pack("<" + v.fmt, x) for x in v.items)
        n = len(v.raw) if v.raw is not None else len(v.items)
        self.pad_to(v.align, 4)
        pos = len(self.b)
        self.b += struct.pack("<I", n) + data
        return pos

    def _table(self, t: _Table) -> int:
        fields = sorted(t.fields, key=lambda f: f[0])
        n_slots = max((f[0] for f in fields), default=-1) + 1
        # inline layout after the 4-byte soffset
        layout, off = [], 4
        for slot, fmt, val in fields:
            size = 4 if fmt is None else struct.calcsize("<" + fmt)
            while off % size:
                off += 1
            layout.append((slot, fmt, val, off))
            off += size
        table_len = off
        vt = [0] * n_slots
        for slot, _, _, o in layout:
            vt[slot] = o
        vtable = struct.pack("<HH", 4 + 2 * n_slots, table_len) + struct.pack(f"<{n_slots}H", *vt)
        self.pad_to(2)
        # the table must start 4-aligned right after its vtable
        while (len(self.b) + len(vtable)) % 4:
            self.b += b"\0\0"
        vt_pos = len(self.b)
        self.b += vtable
        pos = len(self.b)
        self.b += bytes(table_len)
        struct.pack_into("<i", self.b, pos, pos - vt_pos)
        for slot, fmt, val, o in layout:
            if fmt is not None:
                struct.pack_into("<" + fmt, self.b, pos + o, val)
        for slot, fmt, val, o in layout:
            if fmt is None:
                child = self.emit(val)
                struct.pack_into("<I", self.b, pos + o, child - (pos + o))
        return pos


def _options(op: T.Op):
    o = op.options
    act = lambda: _ACT[o.get("act", "NONE")]
    if op.kind == "CONV_2D":
        return _Table([(0, "b", _PAD[o["padding"]]), (1, "i", o["stride_w"]), (2, "i", o["stride_h"]),
                       (3, "b", act()), (4, "i", o.get("dilation_w", 1)), (5, "i", o.get("dilation_h", 1))])
    if op.kind == "DEPTHWISE_CONV_2D":
        return _Table([(0, "b", _PAD[o["padding"]]), (1, "i", o["stride_w"]), (2, "i", o["stride_h"]),
                       (3, "i", o.get("depth_multiplier", 0)), (4, "b", act()),
                       (5, "i", o.get("dilation_w", 1)), (6, "i", o.get("dilation_h", 1))])
    if op.kind in ("MAX_POOL_2D", "AVERAGE_POOL_2D"):
        return _Table([(0, "b", _PAD[o["padding"]]), (1, "i", o["stride_w"]), (2, "i", o["stride_h"]),
                       (3, "i", o["filter_w"]), (4, "i", o["filter_h"]), (5, "b", act())])
    if op.kind == "FULLY_CONNECTED":
        return _Table([(0, "b", act()), (1, "b", o.get("weights_format", 0)),
                       (2, "B", int(o.get("keep_num_dims", False)))])
    if op.kind == "SOFTMAX":
        return _Table([(0, "f", o.get("beta", 1.0))])
    if op.kind in ("MUL", "ADD"):
        return _Table([(0, "b", act())])
    if op.kind == "MEAN":
        return _Table([(0, "B", int(o.get("keep_dims", False)))])
    return None


def write(g: T.Graph) -> bytes:
    kinds = []
    for op in g.ops:
        if op.kind not in kinds:
            kinds.append(op.kind)
    codes = []
    for k in kinds:
        if k.startswith("custom:"):      # a custom operator: builtin code CUSTOM (32) and its name
            codes.append(_Table([(0, "b", 32), (1, None, _Str(k[7:])), (2, "i", 1), (3, "i", 32)]))
            continue
        c = _CODE[k]
        codes.append(_Table([(0, "b", min(c, 127)), (2, "i", 1), (3, "i", c)]))
    buffers = [_Table([])]
    tensors = []
    for t in g.tensors:
        bi = 0
        if t.data is not None:
            buffers.append(_Table([(0, None, _Vec(raw=np.ascontiguousarray(t.data).tobytes(), align=16))]))
            bi = len(buffers) - 1
        f = [(0, None, _Vec("i", t.shape)), (1, "b", _TYPE[np.dtype(t.dtype)]), (2, "I", bi), (3, None, _Str(t.name))]
        if t.quant_scale:
            f.append((4, None, _Table([(2, None, _Vec("f", t.quant_scale))])))
        tensors.append(_Table(f))
    ops = []
    for op in g.ops:
        f = [(0, "I", kinds.index(op.kind)), (1, None, _Vec("i", op.inputs)), (2, None, _Vec("i", op.outputs))]
        opt = _options(op)
        if opt is not None:
            f += [(3, "B", _OPT_TYPE[op.kind]), (4, None, opt)]
        ops.append(_Table(f))
    sg = _Table([(0, None, _Vec(tables=tensors)), (1, None, _Vec("i", g.inputs)), (2, None, _Vec("i", g.outputs)),
                 (3, None, _Vec(tables=ops)), (4, None, _Str("main"))])
    model = _Table([(0, "I", 3), (1, None, _Vec(tables=codes)), (2, None, _Vec(tables=[sg])),
                    (3, None, _Str(g.description)), (4, None, _Vec(tables=buffers))])
    bld = _Builder()
    bld.b += bytes(4) + b"TFL3"
    root = bld.emit(model)
    struct.pack_into("<I", bld.b, 0, root)
    return bytes(bld.b)
