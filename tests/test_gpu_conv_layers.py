"""Every conv layer of the shipped networks, under every tile the autotuner may pick for it, against float64 references.

The engine times up to ten (BN, MT) tile candidates per GEMM and keeps the fastest (engine.cu build_program), so on a shared GPU any
candidate can end up running.  It relies on every candidate accumulating in the same K order.  This file builds the networks on the
CPU, records each distinct conv the plan builder emits, and runs that layer alone, once per candidate, in one plan:
  * every candidate's output buffer is bit-identical to every other's, and frame i's output is the same at batch 1, 8 and 32;
  * frames 0 and B-1 pass gpu_util.check_conv against a float64 conv of the fp16 operands;
  * halos stay zero, the output buffer's other channels keep their contents bit for bit, and no output element is left unwritten
    (the output slice starts as NaN);
  * the input and residual buffers hold +-3e4 outside the channels the op reads, so a kernel that reads past its slice fails.
The same layers run at batch 1 through the SIMT validation kernel (conv_impl 1).  A last test checks that the single-layer
replicas are faithful: inside the whole YOLOv8l and UFLDv2-res34 engines every GEMM step has the replica's candidate list and,
at the chosen tile, the replica's kernel configuration."""
import zlib
from collections import defaultdict

import numpy as np
import pytest
from scipy.special import expit

import adas_b200  # noqa: F401
from adas_b200 import _capi, plan
from gpu_util import check_conv, conv_reference, from_padded

SILU, RELU, NONE = plan.ACT_SILU, plan.ACT_RELU, plan.ACT_NONE
JUNK = 3.0e4                            # contents of channels an op must not read (finite: a NaN would hide in a max)

# (id, builder kind, builder kwargs, batches).  Batch 32 only for the two networks the benchmark runs, to keep the file's wall time down.
NETWORKS = [
    ("yolov8l", "yolov8", dict(scale="l"), (1, 8, 32)),
    ("ufldv2-res34-culane", "ufldv2", dict(backbone="34"), (1, 8, 32)),
    ("yolov5n", "yolov5", dict(scale="n"), (1, 8)),
    ("ufldv2-res18-culane", "ufldv2", dict(backbone="18"), (1, 8)),
    ("ufldv2-res18-tusimple", "ufldv2", dict(backbone="18", cfg="tusimple"), (1, 8)),
    ("ufldv1-res18-tusimple", "ufldv1", dict(backbone="18", cfg="tusimple"), (1, 8)),
    ("ufldv1-res18-culane", "ufldv1", dict(backbone="18", cfg="culane"), (1, 8)),
]


# ---------------------------------------------------------------------------------------------------------------------------------
# the layers the builders emit
# ---------------------------------------------------------------------------------------------------------------------------------
class Layer:
    """One conv as a network plan holds it: geometry of its input / residual / output buffers and its folded weights."""

    def __init__(self, pb, x, w, b, k, s, pad, act, out, res, res_pre, ops, net_step, stem4=False):
        bi = lambda v: pb.buffers[v.buf]            # rows_per_img, C, dtype, H, W, flags
        self.net_step = net_step                    # index of this layer's last op (its GEMM) in the network plan
        self.image = x.buf == pb.image.buf
        self.in_H, self.in_W, self.in_C, self.in_coff, self.cin = x.H, x.W, bi(x)[1], x.coff, x.C
        self.w, self.b = w, (np.zeros(w.shape[0], np.float32) if b is None else b)
        self.cout, self.cin_real = int(w.shape[0]), int(w.shape[1])
        self.n_store = (self.cout + 7) // 8 * 8
        self.k, self.s, self.pad, self.act, self.stem4 = k, s, pad, act, stem4
        self.Ho, self.Wo = out.H, out.W
        self.out_C, self.out_coff, self.out_f32 = bi(out)[1], out.coff, bi(out)[2] == 1
        self.res = None
        if res is not None:
            self.res = dict(C=bi(res)[1], coff=res.coff, pre=bool(res_pre), shared=res.buf == out.buf)
        self.route = tuple(op[0] for op in ops)
        g = ops[-1][1]
        self.ntaps, self.s2 = (g[3], g[16]) if ops[-1][0] == plan.OP_GEMM else (0, 0)
        assert x.buf != out.buf and (res is None or res.buf != x.buf)
        self.K = k * k * self.cin_real

    def key(self):
        r = tuple(sorted(self.res.items())) if self.res else None
        return (self.in_H, self.in_W, self.in_C, self.in_coff, self.cin, self.image, self.cin_real, self.cout, self.k, self.s, self.pad,
                self.act, self.route, self.ntaps, self.s2, self.stem4, r, self.out_C, self.out_coff, self.out_f32)

    @property
    def tuned(self):
        return self.route[-1] == plan.OP_GEMM

    def __repr__(self):
        r = "" if not self.res else f" res({'pre' if self.res['pre'] else 'post'} C{self.res['C']}@{self.res['coff']}" \
                                    f"{' shared' if self.res['shared'] else ''})"
        route = "stem4" if self.stem4 else {plan.OP_STEMCONV: "stemconv", plan.OP_IM2COL: "im2col"}.get(self.route[0], "taps")
        return (f"{self.in_H}x{self.in_W} C{self.in_C}@{self.in_coff} {self.cin_real}->{self.cout} k{self.k}s{self.s}p{self.pad} "
                f"act{self.act} {route}{' s2' if self.s2 else ''}{r} -> C{self.out_C}@{self.out_coff}{' f32' if self.out_f32 else ''}")


def _record(kind, kw):
    """Builds the network plan on the CPU and returns every conv the builder emitted, in order."""
    layers = []
    conv0, stem0 = plan.PlanBuilder.conv, plan.PlanBuilder.stem7x7s2

    def conv(pb, x, w, b, k, s, act, out=None, res=None, res_pre_act=False, out_f32=False, pad=None, tile=None):
        n0 = len(pb.ops)
        v = conv0(pb, x, w, b, k, s, act, out=out, res=res, res_pre_act=res_pre_act, out_f32=out_f32, pad=pad, tile=tile)
        layers.append(Layer(pb, x, w, b, k, s, k // 2 if pad is None else pad, act, v, res, res_pre_act, pb.ops[n0:], len(pb.ops) - 1))
        return v

    def stem(pb, x, w, b, act, tile=None):
        n0 = len(pb.ops)
        v = stem0(pb, x, w, b, act, tile=tile)
        layers.append(Layer(pb, x, w, b, 7, 2, 3, act, v, None, False, pb.ops[n0:], len(pb.ops) - 1, stem4=True))
        return v

    plan.PlanBuilder.conv, plan.PlanBuilder.stem7x7s2 = conv, stem
    try:
        W = plan.synth_weights("ufldv2" if kind == "ufldv1" else kind, 0)
        pb = {"yolov8": plan.build_yolov8, "yolov5": plan.build_yolov5, "ufldv1": plan.build_ufldv1, "ufldv2": plan.build_ufldv2}[kind](W, **kw)
    finally:
        plan.PlanBuilder.conv, plan.PlanBuilder.stem7x7s2 = conv0, stem0
    return pb, layers


_NETS = {}


def network_layers(net_id):
    """(plan builder, every conv layer in emission order, the distinct ones) of one network, cached per process."""
    if net_id not in _NETS:
        _, kind, kw, _ = next(n for n in NETWORKS if n[0] == net_id)
        pb, layers = _record(kind, kw)
        distinct = {}
        for L in layers:
            distinct.setdefault(L.key(), L)
        _NETS[net_id] = (pb, layers, list(distinct.values()))
    return _NETS[net_id]


# ---------------------------------------------------------------------------------------------------------------------------------
# single-layer plans
# ---------------------------------------------------------------------------------------------------------------------------------
def _layer_plan(L, path, tiles=(None,)):
    """One plan holding the layer once per entry of `tiles` (None = the engine's own tile choice).  Every copy reads the same input
    (and residual, unless the residual shares the output buffer); each writes its own output buffer.  Returns the input view's buffer,
    the shared residual buffer (or None) and [(output buffer, GEMM step)] per copy."""
    pb = plan.PlanBuilder(plan.MODEL_YOLOV8, 3, L.in_H, L.in_W)
    x = pb.image if L.image else plan.PlanBuilder.sub(pb.new_padded(L.in_H, L.in_W, L.in_C), L.in_coff, L.cin)
    shared_res = None
    if L.res and not L.res["shared"]:
        shared_res = pb.new_padded(L.Ho, L.Wo, L.res["C"])
    copies = []
    for t in tiles:
        ob = pb.new_padded(L.Ho, L.Wo, L.out_C, f32=L.out_f32)
        out = pb.sub(ob, L.out_coff, L.n_store)
        res = None
        if L.res:
            res = pb.sub(ob if L.res["shared"] else shared_res, L.res["coff"], L.cout)
        if L.stem4:
            pb.stem7x7s2(x, L.w, L.b, L.act, tile=t)
        else:
            pb.conv(x, L.w, L.b, L.k, L.s, L.act, out=out, res=res, res_pre_act=L.res is not None and L.res["pre"], out_f32=L.out_f32,
                    pad=L.pad, tile=t)
        copies.append((ob.buf, len(pb.ops) - 1))
    if L.stem4:      # stem7x7s2 allocates its own output buffer (the next one after its re-layout buffer)
        copies = [(pb.ops[step][1][11], step) for _, step in copies]
    pb.write(path)
    return x.buf, (shared_res.buf if shared_res else None), copies


def _junk(rows, C):
    """+-JUNK in a fixed pattern: what the channels an op must not read (or must not write) hold."""
    period = np.where((np.arange(3)[:, None] + 2 * np.arange(C)[None, :]) % 3 == 0, -JUNK, JUNK).astype(np.float16)
    return np.tile(period, ((rows + 2) // 3, 1))[:rows]


def _frames(L, seed, B, C, H, W):
    """Frames 0..B-1 of seeded N(0, 1) content, [B, C, H, W] fp16: frame i is the same at every batch size."""
    return np.stack([np.random.default_rng([seed, i]).standard_normal((C, H, W), dtype=np.float32).astype(np.float16) for i in range(B)])


def _padded(frames_nchw, C_buf, coff, rows_junk=True):
    """Padded NHWC buffer [B*(H+2)*(W+2), C_buf] holding `frames` in channels coff.., JUNK in the others, zero halo."""
    B, c, H, W = frames_nchw.shape
    buf = _junk(B * (H + 2) * (W + 2), C_buf).reshape(B, H + 2, W + 2, C_buf) if rows_junk else np.zeros((B, H + 2, W + 2, C_buf), np.float16)
    buf[:, 1:-1, 1:-1, coff:coff + c] = frames_nchw.transpose(0, 2, 3, 1)
    buf[:, 0] = 0; buf[:, -1] = 0; buf[:, :, 0] = 0; buf[:, :, -1] = 0
    return buf.reshape(-1, C_buf)


class LayerData:
    """Seeded inputs of one layer at batch B: the input buffer, the residual (separate buffer, or slice of the output buffer) and
    the initial output buffer (NaN in the output slice's interior, JUNK elsewhere, zero halo)."""

    def __init__(self, L, B):
        self.seed = zlib.crc32(repr(L.key()).encode())
        if L.image:
            x = _frames(L, self.seed, B, 3, L.in_H, L.in_W)
            self.x_frames = x
            self.x_buf = _padded(np.concatenate([x, np.zeros_like(x[:, :1])], 1), 4, 0, rows_junk=False)   # (R, G, B, 0) as preprocessing writes it
        else:
            x = _frames(L, self.seed, B, L.cin, L.in_H, L.in_W)
            self.x_frames = x[:, :L.cin_real]
            self.x_buf = _padded(x, L.in_C, L.in_coff)
        self.r_frames = self.r_buf = None
        dt = np.float32 if L.out_f32 else np.float16
        out0 = _junk(B * (L.Ho + 2) * (L.Wo + 2), L.out_C).astype(dt).reshape(B, L.Ho + 2, L.Wo + 2, L.out_C)
        if L.res:
            self.r_frames = _frames(L, self.seed + 1, B, L.cout, L.Ho, L.Wo)
            if L.res["shared"]:
                out0[:, 1:-1, 1:-1, L.res["coff"]:L.res["coff"] + L.cout] = self.r_frames.transpose(0, 2, 3, 1)
            else:
                self.r_buf = _padded(self.r_frames, L.res["C"], L.res["coff"])
        out0[:, 1:-1, 1:-1, L.out_coff:L.out_coff + L.n_store] = np.nan
        out0[:, 0] = 0; out0[:, -1] = 0; out0[:, :, 0] = 0; out0[:, :, -1] = 0
        self.out0 = out0.reshape(-1, L.out_C)
        self.keep = np.ones(L.out_C, bool)                # channels the op must leave as they were
        self.keep[L.out_coff:L.out_coff + L.n_store] = False


_REFS = {}


def _reference(L, data, frame):
    """(ref, mag) of one frame, cached per layer: every candidate and every batch size must produce the same bits."""
    key = (L.key(), frame)
    if key not in _REFS:
        import torch
        w16 = np.zeros((L.n_store, L.cin_real, L.k, L.k), np.float16)
        w16[:L.cout] = L.w.astype(np.float16)
        b = np.zeros(L.n_store, np.float32)
        b[:L.cout] = L.b
        r16 = None
        if L.res is not None:
            r16 = np.zeros((1, L.n_store, L.Ho, L.Wo), np.float16)
            r16[:, :L.cout] = data.r_frames[frame:frame + 1]
        dev = "cuda" if torch.cuda.is_available() else "cpu"
        _REFS[key] = conv_reference(data.x_frames[frame:frame + 1], w16, b, L.s, L.pad, L.act, r16, bool(L.res and L.res["pre"]), device=dev)
    return _REFS[key]


def _interior(buf, L, B):
    return buf.reshape(B, L.Ho + 2, L.Wo + 2, -1)[:, 1:-1, 1:-1]


def _check_copy(L, data, got, B, what):
    """Halo zero, untouched channels as they were, and frames 0 and B-1 within check_conv of the float64 reference."""
    v = got.reshape(B, L.Ho + 2, L.Wo + 2, L.out_C)
    halo = np.concatenate([v[:, 0].ravel(), v[:, -1].ravel(), v[:, :, 0].ravel(), v[:, :, -1].ravel()])
    assert not np.any(halo != 0), f"{what}: {int((halo != 0).sum())} halo entries are not zero"
    assert got[:, data.keep].tobytes() == data.out0[:, data.keep].tobytes(), f"{what}: the op changed channels outside its output slice"
    worst = 0.0
    for f in sorted({0, B - 1}):
        ref, mag = _reference(L, data, f)
        g = from_padded(got[f * (L.Ho + 2) * (L.Wo + 2):(f + 1) * (L.Ho + 2) * (L.Wo + 2)], 1, L.Ho, L.Wo, L.out_coff, L.n_store)
        worst = max(worst, check_conv(g, ref, mag, L.K, L.act, not L.out_f32, f"{what} frame {f}"))
    return worst


def _mode(desc):
    """Epilogue mode of a v3 GEMM from its description string."""
    f = dict(kv.split("=") for kv in desc.replace("|", " ").split() if "=" in kv)
    if f.get("res") not in (None, "0"):
        return "residual via TMA" if f.get("res_tma") == "1" else "residual direct"
    if f.get("f32") == "1":
        return "fp32"
    return "staged" if f.get("tma_st") == "1" else "direct"


def _write_inputs(eng, data, xb, rb, copies):
    eng.write_buffer(xb, data.x_buf)
    if rb is not None:
        eng.write_buffer(rb, data.r_buf)
    for ob, _ in copies:
        eng.write_buffer(ob, data.out0)


# ---------------------------------------------------------------------------------------------------------------------------------
# the sweep
# ---------------------------------------------------------------------------------------------------------------------------------
_SEEN = set()                           # layers already swept for an earlier network of this session


@pytest.mark.gpu
@pytest.mark.parametrize("net_id,batches", [(n[0], n[3]) for n in NETWORKS], ids=[n[0] for n in NETWORKS])
def test_conv_layers_every_candidate(tmp_path, net_id, batches):
    _, layers, distinct = network_layers(net_id)
    worst = defaultdict(float)
    runs = new = 0
    for li, L in enumerate(distinct):
        first_of_session = L.key() not in _SEEN
        _SEEN.add(L.key())
        new += first_of_session
        what = f"{net_id} layer {li} [{L!r}]"
        bits = None                                     # output buffer of the largest batch (frames compared at the smaller ones)
        for B in sorted(batches, reverse=True):
            data = LayerData(L, B)
            path0 = str(tmp_path / f"l{li}_b{B}_auto.b200w")
            xb, rb, copies = _layer_plan(L, path0)
            tiles, chosen = [None], 0
            if L.tuned:
                eng = _capi.Engine(path0, 0, max_batch=B)
                tiles, chosen = eng.step_tiles(B, copies[0][1])
                eng.close()
                assert tiles and 0 <= chosen < len(tiles), f"{what}: no tile candidates at batch {B}"
            path = str(tmp_path / f"l{li}_b{B}.b200w")
            xb, rb, copies = _layer_plan(L, path, tiles)
            eng = _capi.Engine(path, 0, max_batch=B)
            _write_inputs(eng, data, xb, rb, copies)
            eng.run(B)
            got = eng.read_buffer(copies[0][0], B)
            for t, (ob, _) in zip(tiles[1:], copies[1:]):
                assert eng.read_buffer(ob, B).tobytes() == got.tobytes(), \
                    f"{what} batch {B}: tile {t} differs from tile {tiles[0]} (candidates {tiles})"
            modes = {_mode(eng.time_step(B, step, 1)[2]) if L.tuned else "stem conv" for _, step in copies}
            eng.close()
            runs += len(copies)
            ratio = _check_copy(L, data, got, B, f"{what} batch {B} tile {tiles[0]}")
            for m in modes:
                worst[m] = max(worst[m], ratio)
            if bits is None:
                bits = got
            else:
                assert got.tobytes() == bits[:got.shape[0]].tobytes(), f"{what}: frames 0..{B - 1} at batch {B} differ from batch {max(batches)}"
    print(f"\n[conv-layers] {net_id}: {len(layers)} convs, {len(distinct)} distinct ({new} not in an earlier network), {runs} (layer, batch, "
          f"candidate) runs")
    for m, r in sorted(worst.items()):
        print(f"[conv-layers] {net_id} {m}: worst |got - ref| / bound = {r:.3f}")


@pytest.mark.gpu
@pytest.mark.parametrize("net_id", [n[0] for n in NETWORKS])
def test_conv_layers_simt(tmp_path, net_id):
    """The same layers at batch 1 through the SIMT validation kernel (conv_impl 1)."""
    _, _, distinct = network_layers(net_id)
    worst = 0.0
    for li, L in enumerate(distinct):
        data = LayerData(L, 1)
        path = str(tmp_path / f"l{li}.b200w")
        xb, rb, copies = _layer_plan(L, path)
        eng = _capi.Engine(path, 0, max_batch=1, conv_impl=1)
        _write_inputs(eng, data, xb, rb, copies)
        eng.run(1)
        got = eng.read_buffer(copies[0][0], 1)
        eng.close()
        worst = max(worst, _check_copy(L, data, got, 1, f"{net_id} layer {li} [{L!r}] conv_impl 1"))
    print(f"\n[conv-layers] {net_id} SIMT kernel: worst |got - ref| / bound = {worst:.3f}")


@pytest.mark.gpu
@pytest.mark.parametrize("net_id", ["yolov8l", "ufldv2-res34-culane"])
def test_layer_replicas_match_the_network(tmp_path, net_id):
    """Inside the whole engine at batch 8, every GEMM step has the candidate list of its single-layer replica, and the replica forced
    to the step's chosen tile describes the same kernel configuration (M, N, K, tile, slab, stages, TMA store, residual TMA): a
    replica that differed, e.g. in pointer alignment, would send the sweep above through another code path."""
    pb, layers, _ = network_layers(net_id)
    path = str(tmp_path / "net.b200w")
    pb.write(path)
    B = 8
    net = _capi.Engine(path, 0, max_batch=B)
    n_gemm = 0
    for li, L in enumerate(layers):
        tiles, chosen = net.step_tiles(B, L.net_step)
        if not L.tuned:
            assert tiles == [], f"layer {li} [{L!r}]: a stem conv reports GEMM tiles"
            continue
        n_gemm += 1
        desc = net.time_step(B, L.net_step, 1)[2]
        p0 = str(tmp_path / f"r{li}.b200w")
        _, _, copies = _layer_plan(L, p0)
        rep = _capi.Engine(p0, 0, max_batch=B)
        rtiles, _ = rep.step_tiles(B, copies[0][1])
        rep.close()
        assert rtiles == tiles, f"layer {li} [{L!r}]: replica candidates {rtiles}, network {tiles}"
        p1 = str(tmp_path / f"r{li}_t.b200w")
        _, _, copies = _layer_plan(L, p1, [tiles[chosen]])
        rep = _capi.Engine(p1, 0, max_batch=B)
        rdesc = rep.time_step(B, copies[0][1], 1)[2]
        rep.close()
        assert rdesc == desc, f"layer {li} [{L!r}]:\n  replica {rdesc}\n  network {desc}"
    net.close()
    print(f"\n[conv-layers] {net_id}: {n_gemm} GEMM steps match their replicas")


# ---------------------------------------------------------------------------------------------------------------------------------
# the network layers (CPU)
# ---------------------------------------------------------------------------------------------------------------------------------
def test_recorded_layers_cover_the_risky_paths():
    """The sweep reaches the paths whole-network tests used to be the only cover for."""
    _, v5, d5 = network_layers("yolov5n")
    _, v8, d8 = network_layers("yolov8l")
    _, u34, d34 = network_layers("ufldv2-res34-culane")
    for net, layers in (("yolov5n", v5), ("yolov8l", v8), ("ufldv2-res34-culane", u34)):
        steps = [L.net_step for L in layers]
        assert steps == sorted(set(steps)), net
    assert any(L.res and L.n_store % 64 for L in d5), "residual with a direct-store epilogue"
    assert any(L.out_coff % 64 for L in d5), "output slice at an offset that is not a multiple of 64"
    assert any(L.k == 1 and L.route == (plan.OP_GEMM,) and L.cin_real % 64 for L in d5), "1x1 conv with a K tail"
    assert sum(1 for L in v8 if L.res and L.res["shared"]) == 18, "C2f bottlenecks whose residual shares the output buffer"
    assert any(L.in_C > L.cin for L in d8), "input buffer wider than the slice the op reads"
    assert any(L.stem4 for L in d34) and any(L.route[0] == plan.OP_STEMCONV for L in d8)
    print(f"\n[conv-layers] distinct conv layers: yolov8l {len(d8)}, yolov5n {len(d5)}, ufldv2-res34-culane {len(d34)}")


# ---------------------------------------------------------------------------------------------------------------------------------
# checker self-tests (CPU)
# ---------------------------------------------------------------------------------------------------------------------------------
def _operands(rng, cin, cout, k, H, W, res=False):
    x = rng.standard_normal((1, cin, H, W), dtype=np.float32).astype(np.float16)
    w = (rng.standard_normal((cout, cin, k, k), dtype=np.float32) * np.float32(np.sqrt(2.0 / (cin * k * k)))).astype(np.float16)
    b = (0.3 * rng.standard_normal(cout)).astype(np.float32)
    r = rng.standard_normal((1, cout, H, W), dtype=np.float32).astype(np.float16) if res else None
    return x, w, b, r


# real K: 3x3 256->128 (C2f bottleneck of YOLOv8l), 1x1 1280 (YOLOv8l C2f cv2), 1x1 144 (YOLOv5n C3, tail of 16)
SELF_CASES = [(256, 128, 3, SILU, "post", True), (1280, 96, 1, SILU, None, True), (144, 40, 1, SILU, "post", True),
              (256, 64, 3, RELU, "pre", True), (144, 80, 1, NONE, None, False)]


def _conv32(x, w, b, act, r, pre, pad):
    """float32 conv of the fp16 operands (torch's CPU kernel: another summation order) with the fp32 epilogue."""
    import torch
    import torch.nn.functional as F
    t = lambda a: torch.from_numpy(a.astype(np.float32))
    z = F.conv2d(t(x), t(w), t(b), padding=pad)
    if r is not None and pre:
        z = z + t(r)
    z = F.silu(z) if act == SILU else F.relu(z) if act == RELU else z
    if r is not None and not pre:
        z = z + t(r)
    return z.numpy()


def _out(a, f16):
    return a.astype(np.float16) if f16 else a.astype(np.float32)


@pytest.mark.parametrize("cin,cout,k,act,res,f16", SELF_CASES)
def test_check_conv_rejects_kernel_defects(cin, cout, k, act, res, f16):
    """Wrong answers of the kind a conv GEMM defect produces, built from the float64 reference: each must fail check_conv."""
    rng = np.random.default_rng(cin + cout)
    H = W = 6
    pad = k // 2
    x, w, b, r = _operands(rng, cin, cout, k, H, W, res is not None)
    pre = res == "pre"
    K = k * k * cin
    ref, mag = conv_reference(x, w, b, 1, pad, act, r, pre)
    check_conv(_out(ref, f16), ref, mag, K, act, f16)
    wrong = {}
    # the last K block (64 channels, or the tail) of one tap dropped
    w2 = w.copy()
    kb = cin - (cin % 64 or 64)
    w2[:, kb:, k - 1, k - 1] = 0
    wrong["last K block of one tap dropped"] = conv_reference(x, w2, b, 1, pad, act, r, pre)[0]
    if r is not None:
        wrong["residual read from the neighbouring 8 channels"] = conv_reference(x, w, b, 1, pad, act, np.roll(r, -8, axis=1), pre)[0]
    n0 = 32 if cout > 32 else 16
    b2 = b.copy()
    b2[:cout - n0] = b[n0:]                                   # tile n reads the bias of tile n + 1
    wrong["next N tile's bias"] = conv_reference(x, w, b2, 1, pad, act, r, pre)[0]
    if act != NONE:
        skipped = ref.copy()
        last = (cout - 1) // 32 * 32
        skipped[:, last:] = conv_reference(x, w[last:], b[last:], 1, pad, NONE, None if r is None else r[:, last:], pre)[0]
        wrong["activation skipped on the last partial N tile"] = skipped
    shifted = ref.copy()
    shifted[:, :, 2, 1:] = ref[:, :, 2, :-1]
    wrong["output row taken from the neighbouring pixel"] = shifted
    # accumulation in fp16: products summed in K order with an fp16 running sum
    xs = np.pad(x.astype(np.float32), ((0, 0), (0, 0), (pad, pad), (pad, pad)))
    acc = np.zeros((cout, H, W), np.float16)
    for dy in range(k):
        for dx in range(k):
            patch = xs[0, :, dy:dy + H, dx:dx + W]
            for c in range(cin):
                acc = (acc + (w[:, c, dy, dx].astype(np.float32)[:, None, None] * patch[c][None]).astype(np.float16)).astype(np.float16)
    z = acc.astype(np.float64)[None] + b[None, :, None, None]
    if r is not None and pre:
        z = z + r
    z = z * expit(z) if act == SILU else np.maximum(z, 0) if act == RELU else z
    if r is not None and not pre:
        z = z + r
    wrong["accumulation in fp16"] = z
    for name, g in wrong.items():
        with pytest.raises(AssertionError):
            check_conv(_out(g, f16), ref, mag, K, act, f16, name)


def _silu2_emulated(z, rng):
    """numpy float32 emulation of tc_common.cuh silu2 on pairs of values, with ex2.approx and rcp.approx perturbed by their documented
    worst relative errors (2^-22 and 2^-23; sign chosen at random per element)."""
    z = z.astype(np.float32).reshape(-1, 2)
    L = np.float32(-1.4426950408889634)
    e = lambda a: a * (np.float32(1) + np.where(rng.random(a.shape) < 0.5, -1, 1).astype(np.float32) * np.float32(2.0 ** -22))
    t = np.maximum(z, np.float32(-40)) * L
    a = np.float32(1) + e(np.exp2(t.astype(np.float64)).astype(np.float32))
    p = a[:, 0] * a[:, 1]
    rcp = (np.float32(1) / p) * (np.float32(1) + np.where(rng.random(p.shape) < 0.5, -1, 1).astype(np.float32) * np.float32(2.0 ** -23))
    out = np.stack([z[:, 0] * (rcp * a[:, 1]), z[:, 1] * (rcp * a[:, 0])], 1)
    return out.astype(np.float32)


@pytest.mark.parametrize("cin,cout,k,act,res,f16", SELF_CASES)
def test_check_conv_accepts_fp32_conv_and_silu2(cin, cout, k, act, res, f16):
    """A float32 conv of the same fp16 operands passes, and so does its pre-activation sum sent through an emulation of silu2 with
    ex2 / rcp at their documented error bounds."""
    rng = np.random.default_rng(10 + cin + cout)
    x, w, b, r = _operands(rng, cin, cout, k, 6, 6, res is not None)
    pre = res == "pre"
    K = k * k * cin
    ref, mag = conv_reference(x, w, b, 1, k // 2, act, r, pre)
    check_conv(_out(_conv32(x, w, b, act, r, pre, k // 2), f16), ref, mag, K, act, f16, "fp32 conv")
    if act == SILU:
        z = _conv32(x, w, b, NONE, r if pre else None, pre, k // 2)
        got = _silu2_emulated(z, rng).reshape(z.shape)
        if r is not None and not pre:
            got = got + r.astype(np.float32)
        check_conv(_out(got, f16), ref, mag, K, act, f16, "silu2 emulation")
        # the SiLU bound alone, without the accumulation term, on a range of arguments where the approximations show
        zz = np.linspace(-45, 45, 20000).astype(np.float32)
        ref2 = zz.astype(np.float64) * expit(zz.astype(np.float64))
        check_conv(_silu2_emulated(zz, rng).ravel(), ref2, np.zeros_like(ref2), 0, SILU, False, "silu2 alone")


def test_silu_bound_is_not_vacuous():
    """The SiLU term rejects a sigmoid computed in fp16 (relative error ~2^-11)."""
    zz = np.linspace(-10, 10, 2001)
    ref = zz * expit(zz)
    got = zz * expit(zz).astype(np.float16).astype(np.float64)
    with pytest.raises(AssertionError):
        check_conv(got.astype(np.float32), ref, np.zeros_like(ref), 0, SILU, False, "fp16 sigmoid")
