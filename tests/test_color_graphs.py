"""Retrained colour classifiers: any sequential float32 CNN of the subset cp_color_net_load_tflite accepts
(csrc/tflite_reader.hpp::read_color_graph, cones_perception_b200/tflite_model.check) runs on the device through
color_graph_kernel, dam_net's own architecture through cone_color_kernel.

Models of other architectures are written with oracle/tflite_writer.py and seeded weights.  CPU: the writer round
trip, the numpy checker's new operators against a float64 loop formulation, and the Python reader's refusals.
GPU: logits bit for bit against the numpy checker, dam_net through both kernels, every colour entry point and the
C++ node with a retrained model loaded, and the loader's refusals."""
import ctypes as C
import os

import numpy as np
import pytest

from cones_perception_b200 import api, scans
from cones_perception_b200 import tflite_model as T
from cones_perception_b200.pointcloud2 import PointCloud2
from oracle import color_graph_ref as D
from oracle import dam_net_ref
from oracle import oracle as O
from oracle import tflite_writer as TW

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
EXT = 0.05
UNSURE = api.CONE_AMBIGUOUS | api.CONE_LOW_CONFIDENCE


def dam_net_bytes() -> bytes:
    return np.load(os.path.join(GOLD, "dam_net_model.npz"))["tflite"].tobytes()


class Net:
    """A sequential Graph under construction; every layer appends its constants and one activation."""

    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.t = [T.Tensor("input", (1, 15, 12, 1), np.float32, None)]
        self.ops, self.shape = [], (1, 15, 12, 1)

    def const(self, a, dtype=np.float32):
        a = np.ascontiguousarray(a, dtype)
        self.t.append(T.Tensor(f"c{len(self.t)}", a.shape, dtype, a))
        return len(self.t) - 1

    def op(self, kind, consts, options, shape, first=True):
        self.t.append(T.Tensor(f"a{len(self.t)}", tuple(shape), np.float32, None))
        cur = self.cur()
        ins = [cur] + consts if first else consts + [cur]
        self.ops.append(T.Op(kind, ins, [len(self.t) - 1], options))
        self.shape = tuple(shape)
        return self

    def cur(self):
        return self.ops[-1].outputs[0] if self.ops else 0

    def _w(self, *shape, scale=None):
        fan = int(np.prod(shape[1:])) if len(shape) > 1 else 1
        return self.rng.normal(0, scale or 1.0 / np.sqrt(fan), shape)

    def conv(self, co, k, stride=1, padding="VALID", act="RELU", in_scale=1.0):
        _, H, W, ci = self.shape
        w = self._w(co, k, k, ci) * in_scale
        b = self.rng.normal(0, 0.1, co)
        ho, _ = T._window(padding, H, k, stride)
        wo, _ = T._window(padding, W, k, stride)
        cw, cb = self.const(w), self.const(b)
        return self.op("CONV_2D", [cw, cb], {"padding": padding, "stride_w": stride, "stride_h": stride, "act": act,
                                             "dilation_w": 1, "dilation_h": 1}, (1, ho, wo, co))

    def depthwise(self, m, k, stride=1, padding="SAME", act="RELU"):
        _, H, W, c = self.shape
        cw, cb = self.const(self._w(1, k, k, c * m, scale=0.4)), self.const(self.rng.normal(0, 0.1, c * m))
        ho, _ = T._window(padding, H, k, stride)
        wo, _ = T._window(padding, W, k, stride)
        return self.op("DEPTHWISE_CONV_2D", [cw, cb], {"padding": padding, "stride_w": stride, "stride_h": stride,
                                                       "act": act, "dilation_w": 1, "dilation_h": 1,
                                                       "depth_multiplier": m}, (1, ho, wo, c * m))

    def pool(self, kind, k, stride, padding="VALID", act="NONE"):
        _, H, W, c = self.shape
        ho, _ = T._window(padding, H, k, stride)
        wo, _ = T._window(padding, W, k, stride)
        return self.op(kind, [], {"padding": padding, "stride_w": stride, "stride_h": stride, "filter_w": k,
                                  "filter_h": k, "act": act}, (1, ho, wo, c))

    def mean(self, keep=False):
        c = self.shape[-1]
        return self.op("MEAN", [self.const(np.array([1, 2]), np.int32)], {"keep_dims": keep},
                       (1, 1, 1, c) if keep else (1, c))

    def eltwise(self, kind, shape_of_const, act="NONE", first=True):
        k = self.const(self.rng.uniform(0.5, 1.5, shape_of_const) if kind == "MUL"
                       else self.rng.normal(0, 0.2, shape_of_const))
        return self.op(kind, [k], {"act": act}, self.shape, first)

    def reshape(self, shape):
        return self.op("RESHAPE", [self.const(np.array(shape), np.int32)], {}, shape)

    def fc(self, n, act="NONE", bias=True, scale=1.0):
        k = int(np.prod(self.shape))
        consts = [self.const(self._w(n, k) * scale)] + ([self.const(self.rng.normal(0, 0.1, n))] if bias else [])
        return self.op("FULLY_CONNECTED", consts, {"act": act, "weights_format": 0, "keep_num_dims": False}, (1, n))

    def softmax(self, beta=1.0):
        return self.op("SOFTMAX", [], {"beta": beta}, self.shape)

    def graph(self):
        return T.Graph(self.t, self.ops, [0], [self.cur()], "test model")

    def bytes(self):
        return TW.write(self.graph())


def arch_same_stride2():
    """SAME convolution with stride 2 and RELU6."""
    return (Net(11).conv(8, 3, 2, "SAME", "RELU6", in_scale=0.02).conv(16, 3, 1, "SAME", "RELU")
            .pool("MAX_POOL_2D", 2, 2, "SAME").reshape((1, 4 * 3 * 16)).fc(3, scale=10).softmax())


def arch_separable():
    """Separable (depthwise + 1x1) -> SAME average pool -> MEAN -> FC RELU -> FC -> SOFTMAX beta 0.5."""
    return (Net(12).conv(8, 3, 1, "VALID", "RELU", in_scale=0.02).depthwise(2, 3, 1, "SAME", "RELU")
            .conv(16, 1, 1, "VALID", "RELU").pool("AVERAGE_POOL_2D", 3, 2, "SAME").mean()
            .fc(32, "RELU").fc(3, scale=30).softmax(0.5))


def arch_no_softmax():
    """A head without SOFTMAX: scalar MUL, per-channel ADD with the activation second, MEAN keep_dims, FC no bias."""
    return (Net(13).conv(12, 3, 1, "SAME", "RELU", in_scale=0.02).eltwise("MUL", ())
            .eltwise("ADD", (1, 1, 1, 12), first=False).depthwise(1, 3, 2, "VALID", "RELU_N1_TO_1").mean(keep=True)
            .reshape((1, 12)).fc(3, bias=False, scale=10))


def arch_two_classes():
    """Two classes: 5x5 SAME RELU_N1_TO_1, VALID average pool, standalone RELU6 and RELU, per-channel MUL."""
    return (Net(14).conv(6, 5, 1, "SAME", "RELU_N1_TO_1", in_scale=0.02).pool("AVERAGE_POOL_2D", 2, 2, "VALID")
            .op("RELU6", [], {}, (1, 7, 6, 6)).eltwise("MUL", (6,)).op("RELU", [], {}, (1, 7, 6, 6))
            .reshape((1, 7 * 6 * 6)).fc(2).softmax())


def arch_at_limit(channels=321):
    """The largest activation pair fits the 227 KB budget with 11 floats to spare (321 channels of 15x12)."""
    return Net(15).conv(channels, 3, 1, "SAME", "RELU", in_scale=0.02).mean().fc(3, scale=10).softmax()


ARCHS = {"same_stride2": arch_same_stride2, "separable": arch_separable, "no_softmax": arch_no_softmax,
         "two_classes": arch_two_classes, "at_limit": arch_at_limit}


def dam_net_plus_reshape():
    """dam_net with one identity RESHAPE [1,64] -> [1,64] before the dense layer: not dam_net's operator list."""
    g = T.load(dam_net_bytes())
    t = list(g.tensors)
    ops = list(g.ops)
    r = next(i for i, o in enumerate(ops) if o.kind == "RESHAPE")
    t.append(T.Tensor("identity", (1, 64), np.float32, None))
    ops.insert(r + 1, T.Op("RESHAPE", [ops[r].outputs[0]], [len(t) - 1], {}))
    fc = ops[r + 2]
    ops[r + 2] = T.Op(fc.kind, [len(t) - 1] + fc.inputs[1:], fc.outputs, fc.options)
    return TW.write(T.Graph(t, ops, g.inputs, g.outputs, g.description))


def sample_images(n=96, seed=0):
    z = np.load(os.path.join(GOLD, "cone_images.npz"))
    rng = np.random.default_rng(seed)
    return np.concatenate([z["real_images"][:n // 2], rng.integers(0, 256, (n - n // 2, 15, 12), dtype=np.uint8)])


# ---- refused constructs --------------------------------------------------------------------------------------
def _mutated(fn):
    n = arch_same_stride2()
    fn(n)
    return n.bytes()


def _opt(i, **kw):
    def f(n):
        n.ops[i].options.update(kw)
    return f


def _tensor(i, **kw):
    def f(n):
        t = n.t[n.ops[i].inputs[1]] if i >= 0 else n.t[0]
        for k, v in kw.items():
            setattr(t, k, v)
        if "dtype" in kw and t.data is not None:
            t.data = t.data.astype(kw["dtype"])
    return f


def _append(kind, options=None):
    def f(n):
        n.ops.pop()          # drop the SOFTMAX, put the operator there, then SOFTMAX again
        n.t.pop()
        n.op(kind, [], options or {}, n.shape).softmax()
    return f


def _branch(n):
    n.ops[1].inputs[2] = n.ops[0].outputs[0]     # the second conv's bias is an activation


def _softmax_not_last(n):
    n.ops.pop()
    n.t.pop()
    n.softmax().fc(3)


REFUSED = {
    "tanh_operator": lambda: _mutated(_append("TANH")),
    "logistic_operator": lambda: _mutated(_append("LOGISTIC")),
    "fused_tanh": lambda: _mutated(_opt(0, act="TANH")),
    "dilation_2": lambda: _mutated(_opt(0, dilation_w=2)),
    "int8_constant": lambda: _mutated(_tensor(0, dtype=np.int8)),
    "quantised_constant": lambda: _mutated(_tensor(0, quant_scale=(0.5,))),
    "quantised_input": lambda: _mutated(_tensor(-1, quant_scale=(0.5,))),
    "branch": lambda: _mutated(_branch),
    "custom_op": lambda: _mutated(_append("custom:MyOp")),
    "softmax_not_last": lambda: _mutated(_softmax_not_last),
    "four_classes": lambda: Net(1).conv(4, 3).mean().fc(4).softmax().bytes(),
    "nonfinite_beta": lambda: Net(1).conv(4, 3).mean().fc(3).softmax(float("inf")).bytes(),
    "mean_axis_1": lambda: (lambda n: (setattr(n.t[n.ops[1].inputs[1]], "data", np.array([1, 1], np.int32)), n)[1])(
        Net(1).conv(4, 3).mean().fc(3)).bytes(),
    "mul_2d_constant": lambda: Net(1).conv(4, 3).eltwise("MUL", (2, 4)).mean().fc(3).bytes(),
    "reshape_changes_count": lambda: Net(1).conv(4, 3).mean().reshape((1, 3)).bytes(),
    "fc_keep_num_dims": lambda: (lambda n: (n.ops[-1].options.update(keep_num_dims=True), n)[1])(
        Net(1).conv(4, 3).mean().fc(3)).bytes(),
    "over_budget": lambda: arch_at_limit(322).bytes(),
    "wrong_input_shape": lambda: (lambda n: (setattr(n.t[0], "shape", (1, 15, 12, 2)), n)[1])(
        Net(1).conv(4, 3).mean().fc(3)).bytes(),
}


# ---- CPU ----------------------------------------------------------------------------------------------------------
def test_writer_round_trips_dam_net():
    raw = dam_net_bytes()
    g = T.load(raw)
    g2 = T.load(TW.write(g))
    assert [(o.kind, o.inputs, o.outputs, o.options) for o in g.ops] == \
        [(o.kind, o.inputs, o.outputs, o.options) for o in g2.ops]
    assert (g.inputs, g.outputs, g.description) == (g2.inputs, g2.outputs, g2.description)
    assert len(g.tensors) == len(g2.tensors)
    for a, b in zip(g.tensors, g2.tensors):
        assert (a.name, a.shape, a.dtype, a.quant_scale) == (b.name, b.shape, b.dtype, b.quant_scale)
        assert (a.data is None) == (b.data is None)
        if a.data is not None:
            assert a.data.tobytes() == b.data.tobytes()
    # still dam_net's operator list: the device runs it on cone_color_kernel
    assert [o.kind for o in g2.ops] == ["CONV_2D", "MAX_POOL_2D", "CONV_2D", "MAX_POOL_2D", "MUL", "ADD", "RESHAPE",
                                        "FULLY_CONNECTED", "SOFTMAX"]
    img = sample_images(8)
    p1, l1 = D.forward_batch(g, img)
    p2, l2 = D.forward_batch(g2, img)
    assert np.array_equal(l1.view(np.uint32), l2.view(np.uint32))


def test_graph_checker_equals_the_dam_net_checker_on_dam_net():
    """On dam_net (and on random networks of its architecture) the general checker gives dam_net_ref.forward's
    probabilities and logits bit for bit, and the values pinned in dam_net_model.npz."""
    from tests.test_dam_net import _graph_of, _random_net
    g = T.load(dam_net_bytes())
    z = np.load(os.path.join(GOLD, "dam_net_model.npz"))
    imgs = np.load(os.path.join(GOLD, "cone_images.npz"))
    real = imgs["real_images"]
    for batch in (real, imgs["synth_images"]):
        p, l = D.forward_batch(g, batch)
        for i in range(0, len(batch), 5):
            rp, rl = dam_net_ref.forward(g, batch[i])
            assert np.array_equal(l[i].view(np.uint32), rl.view(np.uint32)), i
            assert np.array_equal(p[i].view(np.uint32), rp.view(np.uint32)), i
    p, l = D.forward_batch(g, real)
    for i in range(0, len(real), 7):
        assert np.array_equal(l[i].view(np.uint32), z["real_logits"][i].view(np.uint32))
        assert np.array_equal(p[i].view(np.uint32), z["real_probs"][i].view(np.uint32))
    rng = np.random.default_rng(3)
    for c1, c2, nc in ((5, 7, 2), (16, 32, 3)):
        rg = _graph_of(_random_net(rng, c1, c2, nc))
        x = rng.integers(0, 256, (6, 15, 12), dtype=np.uint8)
        for i in range(len(x)):
            rp, rl = dam_net_ref.forward(rg, x[i])
            p, l = D.forward(rg, x[i])
            assert np.array_equal(l.view(np.uint32), rl.view(np.uint32))
            assert np.array_equal(p.view(np.uint32), rp.view(np.uint32))


@pytest.mark.parametrize("arch", sorted(ARCHS))
def test_written_architectures_are_accepted(arch):
    g = T.load(ARCHS[arch]().bytes())
    p, l = D.forward_batch(g, sample_images(8))
    assert p.shape == l.shape == (8, g.tensors[g.outputs[0]].shape[1]) and np.isfinite(p).all()


def _loops(x, op, g):
    """float64 loop formulation of one operator on one image x [H,W,C]."""
    o = op.options
    const = lambda i: g.tensors[i].data.astype(np.float64)
    H, W, Ci = x.shape
    if op.kind in ("CONV_2D", "DEPTHWISE_CONV_2D", "MAX_POOL_2D", "AVERAGE_POOL_2D"):
        if op.kind == "CONV_2D":
            w = const(op.inputs[1])
            kh, kw, Co = w.shape[1], w.shape[2], w.shape[0]
        elif op.kind == "DEPTHWISE_CONV_2D":
            w = const(op.inputs[1])
            kh, kw, Co = w.shape[1], w.shape[2], w.shape[3]
        else:
            kh, kw, Co = o["filter_h"], o["filter_w"], Ci
        Ho, pt = T._window(o["padding"], H, kh, o["stride_h"])
        Wo, pl = T._window(o["padding"], W, kw, o["stride_w"])
        y = np.zeros((Ho, Wo, Co))
        for oy in range(Ho):
            for ox in range(Wo):
                for c in range(Co):
                    vals = []
                    for ky in range(kh):
                        for kx in range(kw):
                            iy, ix = oy * o["stride_h"] - pt + ky, ox * o["stride_w"] - pl + kx
                            if 0 <= iy < H and 0 <= ix < W:
                                if op.kind == "CONV_2D":
                                    vals.append(np.dot(x[iy, ix, :], w[c, ky, kx, :]))
                                elif op.kind == "DEPTHWISE_CONV_2D":
                                    vals.append(x[iy, ix, c // (Co // Ci)] * w[0, ky, kx, c])
                                else:
                                    vals.append(x[iy, ix, c])
                    if op.kind == "MAX_POOL_2D":
                        y[oy, ox, c] = max(vals)
                    elif op.kind == "AVERAGE_POOL_2D":
                        y[oy, ox, c] = sum(vals) / len(vals)
                    else:
                        y[oy, ox, c] = sum(vals) + const(op.inputs[2])[c]
        lo, hi = D._CLAMP[o["act"]]
        return np.clip(y, -np.inf if lo is None else lo, np.inf if hi is None else hi)
    if op.kind == "MEAN":
        return x.sum(axis=(0, 1)) / (H * W)
    raise ValueError(op.kind)


@pytest.mark.parametrize("case", ["same_stride2", "separable", "at_limit_small", "dw_stride2_valid", "mean"])
def test_checker_agrees_with_float64_loops(case):
    """The checker's new operators (SAME padding, strides, depthwise, the average pool's in-bounds count at the
    borders, MEAN) against a direct loop formulation in float64."""
    nets = {"same_stride2": Net(1).conv(5, 3, 2, "SAME", "RELU6", in_scale=0.02),
            "separable": Net(2).conv(3, 3, 1, "VALID", "NONE", in_scale=0.02).depthwise(2, 3, 1, "SAME", "NONE"),
            "at_limit_small": Net(3).conv(4, 1, 1, "VALID", "NONE", in_scale=0.02).pool("AVERAGE_POOL_2D", 3, 2, "SAME"),
            "dw_stride2_valid": Net(4).conv(2, 2, 1, "SAME", "RELU", in_scale=0.02).depthwise(3, 3, 2, "VALID", "RELU_N1_TO_1"),
            "mean": Net(5).conv(3, 3, 1, "SAME", "NONE", in_scale=0.02).pool("MAX_POOL_2D", 3, 2, "SAME").mean()}
    n = nets[case]
    g = T.Graph(n.t, n.ops, [0], [n.cur()])
    img = sample_images(4, seed=7)
    x = img.astype(np.float32).reshape(4, 15, 12, 1)
    for op in n.ops:
        sub = T.Graph(n.t, [op], [op.inputs[0]], [op.outputs[0]])
        got = _run_one(sub, x)
        for b in range(len(x)):
            ref = _loops(x[b].astype(np.float64), op, g)
            scale = max(1.0, float(np.max(np.abs(ref))))
            assert np.max(np.abs(got[b].reshape(ref.shape) - ref)) <= 2e-5 * scale, (case, op.kind)
        x = got


def _run_one(g, x):
    """The checker's implementation of one operator on a batch of activations."""
    op = g.ops[0]
    o = op.options
    const = lambda i: g.tensors[i].data
    if op.kind == "CONV_2D":
        return D.conv2d(x, const(op.inputs[1]), const(op.inputs[2]), o)
    if op.kind == "DEPTHWISE_CONV_2D":
        return D.depthwise_conv2d(x, const(op.inputs[1]), const(op.inputs[2]), o)
    if op.kind in ("MAX_POOL_2D", "AVERAGE_POOL_2D"):
        return D.pool(x, o, op.kind == "AVERAGE_POOL_2D")
    if op.kind == "MEAN":
        return D.mean(x, o)
    raise ValueError(op.kind)


def test_average_pool_counts_only_inside_taps():
    """SAME 3x3 average pool of an all-ones image is 1 everywhere, the corners included."""
    n = Net(0)
    n.pool("AVERAGE_POOL_2D", 3, 1, "SAME")
    y = D.pool(np.ones((1, 15, 12, 1), np.float32), n.ops[0].options, True)
    assert np.array_equal(y, np.ones_like(y))


@pytest.mark.parametrize("case", sorted(REFUSED))
def test_python_reader_refuses(case):
    with pytest.raises(T.UnsupportedModel):
        T.load(REFUSED[case]())


# ---- GPU ----------------------------------------------------------------------------------------------------------
def _assert_logits_exact(h, g, imgs):
    nc = g.tensors[g.outputs[0]].shape[1]
    colors, probs, logits = h.classify_images(imgs, nc)
    p, l = D.forward_batch(g, imgs)
    assert np.array_equal(logits.view(np.uint32), l.view(np.uint32))
    softmax = g.ops[-1].kind == "SOFTMAX"
    if softmax:
        assert np.max(np.abs(probs - p)) <= 1e-6
    else:
        assert np.array_equal(probs.view(np.uint32), p.view(np.uint32))
    for i in range(len(imgs)):
        if abs(float(p[i].max()) - 0.8) > 2e-6:
            assert int(colors[i]) == D.decide(p[i]), i
    return colors


@pytest.mark.gpu
def test_dam_net_through_the_graph_kernel_equals_cone_color_kernel():
    z = np.load(os.path.join(GOLD, "cone_images.npz"))
    imgs = np.concatenate([z["real_images"], z["synth_images"]])
    assert len(imgs) == 577 + 256
    cfg = scans.config(2)
    with api.ConesGpu(max_points=cfg.points_per_frame) as a, api.ConesGpu(max_points=cfg.points_per_frame) as b:
        a.color_net_load_tflite(dam_net_bytes())
        b.color_net_load_tflite(dam_net_plus_reshape())
        ca, pa, la = a.classify_images(imgs)
        cb, pb, lb = b.classify_images(imgs)
        assert np.array_equal(la.view(np.uint32), lb.view(np.uint32))
        assert np.array_equal(ca, cb)
        assert np.array_equal(pa.view(np.uint32), pb.view(np.uint32))
        assert a.last_launch_count() == b.last_launch_count() == 1
        # the per-cone flags through the crop path: both kernels share the decision tail
        frame = scans.generate(cfg, 1, base_seed=3)[0].copy()
        frame[:, 3] = np.clip(frame[:, 3] * 2.5, 0, 255)
        msg = PointCloud2.from_xyzi(frame)
        outs = []
        for hh in (a, b):
            cl, _ = hh.detect(msg, cfg.detect, cfg.ground)
            outs.append(hh.cone_colors([(float(c["x"]), float(c["y"])) for c in cl] + [(55.0, 55.0)]))
        for x, y in zip(*outs):
            assert np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8))


@pytest.mark.gpu
@pytest.mark.parametrize("arch", sorted(ARCHS))
def test_graph_logits_bit_for_bit(arch):
    n = ARCHS[arch]()
    g = T.load(n.bytes())
    imgs = sample_images(160, seed=sorted(ARCHS).index(arch))
    with api.ConesGpu(max_points=1024) as h:
        h.color_net_load_tflite(n.bytes())
        colors = _assert_logits_exact(h, g, imgs)
        assert len(set(colors.tolist())) >= 1


def _cpu_chain(g, got, cloud_pts, clusters, ext=EXT):
    """crops -> to_image -> numpy forward -> decide, per cluster of one frame."""
    colors, probs, flags, counts = got
    for k, r in enumerate(clusters):
        cx, cy = O.extend(float(r["x"]), float(r["y"]), ext)
        crop = O.reconstruct_cone(cloud_pts, cx, cy)
        assert int(counts[k]) == len(crop), k
        if len(crop) == 0:
            assert flags[k] & api.CONE_EMPTY and colors[k] == api.COLOR_NO_ANSWER, k
            continue
        img, fl = O.to_image(np.stack([crop["x"], crop["y"], crop["z"], crop["intensity"]], 1))
        if flags[k] & UNSURE:
            assert int(flags[k]) & ~UNSURE == fl, k
            continue
        assert int(flags[k]) == fl, k
        if fl:
            assert colors[k] == api.COLOR_NO_ANSWER, k
            continue
        p, _ = D.forward(g, img)
        assert np.max(np.abs(p - probs[k])) <= 1e-6, k
        assert int(colors[k]) == D.decide(p), k


def _bright(frames):
    out = np.array(frames, np.float32, copy=True)
    out[..., 3] = np.clip(out[..., 3] * 2.5, 0, 255)
    return out


@pytest.mark.gpu
def test_every_colour_entry_point_with_a_retrained_model():
    from tests.test_gpu_batch_track import Answers, assert_same, reference
    model = arch_separable().bytes()
    g = T.load(model)
    cfg = scans.config(2)
    frames = _bright(scans.generate(cfg, 8, base_seed=2040))
    with api.ConesGpu(max_points=8 * cfg.points_per_frame, max_frames=8, max_point_step=32) as h:
        h.color_net_load_tflite(model)
        _, off, cl = h.detect_batch([PointCloud2.from_xyzi(f) for f in frames], cfg.detect, cfg.ground)
        staged = h.batch_cone_colors()
        assert len(cl) > 50
        for f in (0, 7):
            a, b = int(off[f]), int(off[f + 1])
            _cpu_chain(g, tuple(x[a:b] for x in staged), O.points32(frames[f]), cl[a:b])
            c = np.array([O.extend(float(r["x"]), float(r["y"]), EXT) for r in cl[a:b]], np.float32)
            col, pr, fl = h.cone_colors(c, frame=f)                      # cp_cone_colors, the per-frame call
            assert np.array_equal(col, staged[0][a:b]) and np.array_equal(fl, staged[2][a:b])
            assert np.array_equal(pr.view(np.uint32), staged[1][a:b].view(np.uint32))
        h.set_color_cloud(True)
        ground = h.batch_cone_colors()
        for f in (0, 7):
            a, b = int(off[f]), int(off[f + 1])
            msg = O.ground_node(O.view_of_xyzi(np.ascontiguousarray(frames[f]), True), cfg.ground)[0]
            _cpu_chain(g, tuple(x[a:b] for x in ground), msg, cl[a:b])
        h.set_color_cloud(False)
        assert ((staged[0] >= 1) & (staged[0] <= 3)).any()
        p = api.track_params(True, True)
        got = h.batch_track(p)
        exp = reference(cl, off, [0, 8], p, Answers(staged[0], staged[2], p.cone_position_extension_length))
        assert_same(got, exp)


@pytest.mark.gpu
def test_cpp_node_with_a_retrained_model():
    """ConeDetector::load_color_model on a retrained file: cloud_handler publishes what the tracker driven by the
    CPU chain publishes, and replay publishes what cloud_handler publishes."""
    from cones_perception_b200.params import to_c_detect
    from tests.test_gpu_batch_track import _host_lib, _publish
    from tests.test_host_shell import CAP, as_arrays
    from tests.util import TrackerReference
    model = arch_same_stride2().bytes()
    g = T.load(model)
    lib = _host_lib()
    lib.ch_detector_handle.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_uint32,
                                       C.c_void_p, C.c_void_p, C.c_void_p]
    cfg = scans.config(1)
    frames = _bright(scans.generate(cfg, 4, base_seed=40))
    d = cfg.detect
    cd = to_c_detect(d)
    buf = (C.c_uint8 * len(model)).from_buffer_copy(model)
    raw = {}

    def service(need):
        out = []
        for p in need:
            c = O.reconstruct_cone(raw["pts"], float(p[0]), float(p[1]), 0.228)
            if len(c) == 0:
                continue
            img, fl = O.to_image(np.stack([c["x"], c["y"], c["z"], c["intensity"]], 1).astype(np.float32))
            if fl:
                return []
            out.append(D.decide(D.forward(g, img)[0]))
        return out

    det = lib.ch_detector_create(cfg.points_per_frame, 0, C.byref(cd), 1, 1, 0)
    assert det, lib.ch_last_error()
    try:
        assert lib.ch_detector_load_color_model(det, buf, len(model)) == 0, lib.ch_last_error()
        ref = TrackerReference(True, True, d.cones_matching_dist_theshold, d.cone_position_extension_length,
                               color_fn=service)
        coloured = 0
        for f in frames:
            out = np.zeros((4, CAP, 2), np.float32)
            counts = np.zeros(4, np.uint32)
            step, nf, nsec = C.c_uint32(), C.c_uint32(), C.c_uint32()
            rc = lib.ch_detector_handle(det, f.ctypes.data, len(f), 1, out.ctypes.data, counts.ctypes.data, CAP,
                                        C.byref(step), C.byref(nf), C.byref(nsec))
            assert rc == 0, lib.ch_last_error()
            raw["pts"] = O.from_msg(O.view_of_xyzi(f))
            cl, _, _ = O.detect(O.view_of_xyzi(f), d, None, O.CANONICAL)
            exp = as_arrays(ref.update([(c["x"], c["y"]) for c in cl]))
            for k in range(4):
                assert counts[k] == len(exp[k]), k
                assert np.array_equal(out[k, :counts[k]].view(np.uint32), exp[k].view(np.uint32))
            coloured += int(counts[1:].sum())
        assert coloured > 0
    finally:
        lib.ch_detector_destroy(det)
    cfg2 = scans.config(2)
    frames2 = list(_bright(scans.generate(cfg2, 10, base_seed=300)))
    cd2 = to_c_detect(cfg2.detect)
    per_msg = lib.ch_detector_create(cfg2.points_per_frame, 0, C.byref(cd2), 1, 1, 1)
    rep = lib.ch_detector_create_replay(4 * cfg2.points_per_frame, 4, 0, C.byref(cd2), 1, 1, 1)
    try:
        assert per_msg and rep, lib.ch_last_error()
        for det in (per_msg, rep):
            assert lib.ch_detector_load_color_model(det, buf, len(model)) == 0, lib.ch_last_error()
        assert _publish(lib, rep, frames2, True) == _publish(lib, per_msg, frames2, False)
    finally:
        lib.ch_detector_destroy(per_msg)
        lib.ch_detector_destroy(rep)


@pytest.mark.gpu
def test_loader_refusals_agree_with_the_python_reader():
    good = {k: f().bytes() for k, f in ARCHS.items()}
    good["dam_net"] = dam_net_bytes()
    good["dam_net_plus_reshape"] = dam_net_plus_reshape()
    with api.ConesGpu(max_points=1024) as h:
        for name, b in good.items():
            T.load(b)
            h.color_net_load_tflite(b)
        for name, make in REFUSED.items():
            b = make()
            with pytest.raises(T.UnsupportedModel):
                T.load(b)
            with pytest.raises(api.ConesGpuError) as e:
                h.color_net_load_tflite(b)
            assert e.value.status == api.CP_E_PARAM, name
        with pytest.raises(api.ConesGpuError) as e:
            h.color_net_load_tflite(REFUSED["over_budget"]())
        assert "bytes of shared memory" in str(e.value)


@pytest.mark.gpu
def test_random_damage_is_refused_or_classifies():
    raw = bytearray(arch_separable().bytes())
    imgs = sample_images(16)
    rng = np.random.default_rng(5)
    refused = loaded = 0
    with api.ConesGpu(max_points=1024) as h:
        for _ in range(300):
            b = bytearray(raw)
            for pos in rng.integers(0, min(len(b), 6000), 4):
                b[int(pos)] = int(rng.integers(0, 256))
            try:
                h.color_net_load_tflite(bytes(b))
            except api.ConesGpuError as e:
                assert e.status == api.CP_E_PARAM
                refused += 1
                continue
            colors, _, _ = h.classify_images(imgs)
            assert len(colors) == len(imgs)
            loaded += 1
        assert refused > 0 and loaded > 0
        g = T.load(bytes(raw))
        h.color_net_load_tflite(bytes(raw))
        _assert_logits_exact(h, g, imgs)


@pytest.mark.gpu
def test_outputs_follow_the_loaded_model():
    dam = T.load(dam_net_bytes())
    other = arch_two_classes()
    imgs = sample_images(64)
    with api.ConesGpu(max_points=1024) as h:
        for model, g in ((dam_net_bytes(), dam), (other.bytes(), other.graph()), (dam_net_bytes(), dam)):
            h.color_net_load_tflite(model)
            _assert_logits_exact(h, g, imgs)
