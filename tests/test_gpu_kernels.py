"""GPU: single-kernel parity through the C ABI (test hooks write/read plan buffers).
conv_impl 0 = tcgen05 implicit GEMM (product), 1 = SIMT validation kernel.  Convs are checked element by element against a float64
conv of the fp16 operands (gpu_util.check_conv); tests/test_gpu_conv_layers.py sweeps every conv layer of the shipped networks."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import adas_b200  # noqa: F401
from adas_b200 import _capi, plan
from gpu_util import check_conv, conv_reference, from_padded, halo_is_zero, to_padded

pytestmark = pytest.mark.gpu


def _run_conv(tmp_path, impl, B, cin, cout, H, W, k, s, act, residual=None, out_f32=False, pad=None, seed=0, im_c=None, tile=None,
              out_slice=None):
    """tile = (BN, MT) forces the tile shape of the tcgen05 kernel; out_slice = (C_total, coff) writes the result into a channel
    slice of a wider (concat) buffer whose other channels must stay untouched."""
    if pad is None and k == 1:
        pad = 0
    rng = np.random.default_rng(seed)
    pb = plan.PlanBuilder(plan.MODEL_YOLOV5, 3, H, W)
    xin = pb.new_padded(H, W, im_c or cin)
    w = (rng.standard_normal((cout, cin, k, k)) * np.sqrt(2.0 / (cin * k * k))).astype(np.float32)
    b = (rng.standard_normal(cout) * 0.1).astype(np.float32)
    res_view = None
    pd = k // 2 if pad is None else pad
    Ho, Wo = (H + 2 * pd - k) // s + 1, (W + 2 * pd - k) // s + 1
    if residual:
        res_view = pb.new_padded(Ho, Wo, cout)
    out_view = None
    if out_slice:
        cat = pb.new_padded(Ho, Wo, out_slice[0])
        out_view = pb.sub(cat, out_slice[1], cout)
    out = pb.conv(xin, w, b, k, s, act, res=res_view, res_pre_act=(residual == "pre"), out_f32=out_f32, pad=pad, out=out_view, tile=tile)
    path = str(tmp_path / f"conv_{impl}_{seed}.b200w")
    pb.write(path)
    eng = _capi.Engine(path, device=0, max_batch=B, conv_impl=impl)
    x = rng.standard_normal((B, cin, H, W)).astype(np.float32)
    eng.write_buffer(xin.buf, to_padded(x, im_c or cin))
    r = None
    if residual:
        r = rng.standard_normal((B, cout, Ho, Wo)).astype(np.float32)
        eng.write_buffer(res_view.buf, to_padded(r, cout))
    sentinel = None
    if out_slice:               # the rest of the concat buffer holds a sentinel pattern (interior only: halos stay zero)
        sentinel = rng.standard_normal((B, out_slice[0], Ho, Wo)).astype(np.float32)
        eng.write_buffer(out.buf, to_padded(sentinel, out_slice[0]))
    for _ in range(3):          # eager, graph capture, graph replay
        eng.run(B)
    got_buf = eng.read_buffer(out.buf, B)
    got = from_padded(got_buf, B, Ho, Wo, out.coff, cout)
    if out_slice:
        full = from_padded(got_buf, B, Ho, Wo, 0, out_slice[0])
        keep = np.ones(out_slice[0], bool); keep[out.coff:out.coff + cout] = False
        assert np.array_equal(full[:, keep], sentinel.astype(np.float16).astype(np.float32)[:, keep]), "conv wrote outside its channel slice"
    r16 = r.astype(np.float16) if residual else None
    ref, mag = conv_reference(x.astype(np.float16), w.astype(np.float16), b, s, pd, act, r16, residual == "pre")
    ratio = check_conv(got, ref, mag, k * k * cin, act, not out_f32, f"impl {impl} {B}x{cin}->{cout} {H}x{W} k{k} s{s} tile {tile}")
    assert halo_is_zero(got_buf, B, Ho, Wo), "conv wrote into the zero halo"
    eng.close()
    return ratio


CASES = [
    # B cin cout H  W  k s act residual out_f32
    (2, 64, 64, 20, 24, 3, 1, 1, None, False),        # tap mode, single k-block per tap
    (1, 128, 256, 40, 40, 3, 1, 1, "post", False),     # tap mode, 2 k-blocks, BN=256, YOLO shortcut
    (2, 256, 128, 12, 52, 3, 1, 2, "pre", False),      # ResNet block: residual before ReLU, ragged M tail
    (1, 200, 64, 17, 23, 1, 1, 1, None, False),        # 1x1, K = 200 = 3*64 + 8 (TMA zero-fills the tail)
    (2, 64, 80, 20, 20, 1, 1, 0, None, True),          # fp32 head output, N = 80
    (1, 320, 320, 16, 16, 1, 1, 1, None, False),       # N = 320 -> two 160-wide tiles
    (2, 64, 128, 32, 48, 3, 2, 1, None, False),        # stride 2 -> im2col + GEMM
    (1, 16, 32, 24, 24, 3, 1, 1, None, False),         # thin channels -> im2col path
    (1, 512, 8, 10, 50, 1, 1, 0, None, False),         # UFLD pool conv, N = 8
    (1, 64, 512, 8, 8, 3, 1, 1, None, False),          # M = 100 rows (one partial tile), N = 512
    (1, 128, 256, 20, 28, 1, 2, 0, None, False),       # ResNet downsample: 1x1 stride 2 through the strided TMA map
    (2, 256, 512, 40, 40, 3, 2, 1, None, False),       # stride-2 3x3, output 20x20 -> 20x6 patches, N = 512
    (1, 64, 64, 160, 96, 3, 2, 2, "pre", False),       # stride-2 3x3 with residual, 48-wide output rows
]


@pytest.mark.parametrize("impl", [1, 0])
@pytest.mark.parametrize("case", CASES)
def test_conv_parity(tmp_path, impl, case):
    B, cin, cout, H, W, k, s, act, residual, f32 = case
    _run_conv(tmp_path, impl, B, cin, cout, H, W, k, s, act, residual, f32, seed=cin + cout + k)


TILE_CASES = [
    # (B cin cout H W k s act residual) , (BN, MT)   -- tcgen05 kernel only: every epilogue / accumulator / operand-fetch mode
    ((2, 256, 256, 40, 40, 3, 1, 1, "post"), (256, 1)),     # plain 9 taps, staged stores, 4 chunks
    ((2, 256, 256, 40, 40, 3, 1, 1, None), (256, 2)),       # one 512-column accumulator set
    ((2, 256, 256, 40, 40, 3, 1, 1, "post"), (128, 2)),     # slab, two sub-tiles, two accumulator stages
    ((2, 128, 128, 80, 80, 3, 1, 1, None), (128, 1)),       # slab, many tiles per CTA (accumulator / staging ping-pong)
    ((2, 128, 128, 48, 80, 3, 1, 2, "pre"), (128, 4)),      # four sub-tiles, one accumulator stage, residual before ReLU
    ((2, 256, 256, 20, 20, 3, 1, 1, None), (64, 3)),        # 64-wide tiles, three sub-tiles
    ((1, 256, 320, 40, 40, 3, 1, 1, None), (128, 1)),       # N = 320: last N tile half outside the tensor (TMA clips it)
    ((1, 256, 320, 40, 40, 3, 1, 1, None), (192, 1)),       # 192-wide tiles
    ((1, 256, 320, 40, 40, 3, 1, 1, None), (160, 1)),       # direct-store epilogue (BN not a multiple of 64)
    ((2, 256, 512, 40, 40, 3, 2, 1, None), (256, 1)),       # stride 2, 4-D TMA store of output patches
    ((2, 256, 512, 40, 40, 3, 2, 1, None), (128, 2)),       # stride 2 with two patches per CTA tile
    ((3, 128, 256, 80, 80, 3, 2, 1, None), (128, 3)),       # stride 2, three patches, patch count not a multiple of MT
    ((1, 64, 64, 160, 96, 3, 2, 2, "pre"), (64, 2)),        # stride 2 with residual, 48-wide output rows (clipped patches)
    ((2, 1024, 512, 40, 40, 1, 1, 1, None), (256, 2)),      # 1x1, long K, 256x256 tiles
    ((2, 320, 128, 80, 80, 1, 1, 1, None), (128, 3)),       # 1x1, K = 320 (five k-blocks)
    ((1, 200, 64, 17, 23, 1, 1, 1, None), (64, 1)),         # K tail (200 = 3*64 + 8), ragged M
    ((2, 64, 80, 20, 20, 1, 1, 0, None), (80, 1)),          # fp16 N = 80 through the direct path
]


@pytest.mark.parametrize("case,tile", TILE_CASES)
def test_conv_tile_shapes(tmp_path, case, tile):
    B, cin, cout, H, W, k, s, act, residual = case
    _run_conv(tmp_path, 0, B, cin, cout, H, W, k, s, act, residual, False, seed=cin + cout + k + tile[0] + tile[1], tile=tile)


def test_conv_tile_shapes_agree_bitwise(tmp_path):
    """Every tile shape accumulates in the same K order: outputs are bit-identical whatever (BN, MT) is chosen."""
    B, cin, cout, H, W = 2, 128, 256, 40, 40
    outs = []
    for i, tile in enumerate(((256, 1), (256, 2), (128, 1), (128, 2), (64, 4), (192, 1), (160, 1))):
        rng = np.random.default_rng(5)
        pb = plan.PlanBuilder(plan.MODEL_YOLOV5, 3, H, W)
        xin = pb.new_padded(H, W, cin)
        w = (rng.standard_normal((cout, cin, 3, 3)) * np.sqrt(2.0 / (cin * 9))).astype(np.float32)
        b = (rng.standard_normal(cout) * 0.1).astype(np.float32)
        out = pb.conv(xin, w, b, 3, 1, 1, tile=tile)
        path = str(tmp_path / f"bit_{i}.b200w")
        pb.write(path)
        eng = _capi.Engine(path, device=0, max_batch=B)
        eng.write_buffer(xin.buf, to_padded(rng.standard_normal((B, cin, H, W)).astype(np.float32), cin))
        eng.run(B)
        outs.append(eng.read_buffer(out.buf, B).copy())
        eng.close()
    for o in outs[1:]:
        assert np.array_equal(o.view(np.uint16), outs[0].view(np.uint16))


def test_conv_into_concat_slice(tmp_path):
    """Producers write their channel slice of a concat buffer; the neighbours' channels and the halo must stay untouched."""
    for (case, tile, sl) in (((2, 128, 128, 40, 40, 3, 1, 1, "post"), (128, 2), (384, 128)),
                             ((2, 256, 64, 20, 24, 1, 1, 1, None), (64, 1), (192, 64)),
                             ((2, 128, 256, 40, 40, 3, 2, 1, None), (128, 2), (512, 256)),
                             ((1, 64, 40, 24, 24, 1, 1, 1, None), None, (96, 56))):
        B, cin, cout, H, W, k, s, act, residual = case
        _run_conv(tmp_path, 0, B, cin, cout, H, W, k, s, act, residual, False, seed=cout + sl[0], tile=tile, out_slice=sl)


@pytest.mark.parametrize("impl", [1, 0])
def test_stem_convs(tmp_path, impl):
    # image convs: C=3 stored as 4 channels; 7x7 s2 p3 (UFLD stem), 6x6 s2 p2 (YOLOv5), 3x3 s2 (YOLOv8)
    for (k, s, pad) in ((7, 2, 3), (6, 2, 2), (3, 2, 1)):
        _run_conv(tmp_path, impl, 1, 3, 64, 64, 96, k, s, 2, pad=pad, seed=k, im_c=4)


@pytest.mark.parametrize("k,pad,cout,act", [(3, 1, 64, 1), (3, 1, 16, 1), (3, 1, 48, 0), (6, 2, 16, 1), (6, 2, 32, 2), (7, 3, 64, 2)])
def test_stem_conv_direct(tmp_path, k, pad, cout, act):
    """stem_conv.cu: k x k stride-2 conv straight from the C=4 image (YOLOv8 3x3, YOLOv5 6x6 p2, ResNet 7x7 p3) -- borders that reach
    beyond the one-pixel halo, widths that are not a multiple of the 16-pixel warp tile, batch > 1, every supported Cout."""
    rng = np.random.default_rng(100 + k + cout)
    for (B, H, W) in ((2, 64, 96), (3, 36, 50), (1, 20, 34)):
        pb = plan.PlanBuilder(plan.MODEL_YOLOV8, 3, H, W)
        w = (rng.standard_normal((cout, 3, k, k)) * np.sqrt(2.0 / (3 * k * k))).astype(np.float32)
        b = (rng.standard_normal(cout) * 0.1).astype(np.float32)
        out = pb.conv(pb.image, w, b, k, 2, act, pad=pad)
        assert [op[0] for op in pb.ops] == [plan.OP_STEMCONV]
        path = str(tmp_path / f"stemd_{k}_{cout}_{H}.b200w")
        pb.write(path)
        eng = _capi.Engine(path, 0, max_batch=B)
        x = rng.standard_normal((B, 3, H, W)).astype(np.float32)
        eng.write_buffer(pb.image.buf, to_padded(x, 4))
        for _ in range(3):
            eng.run(B)
        Ho, Wo = (H + 2 * pad - k) // 2 + 1, (W + 2 * pad - k) // 2 + 1
        got_buf = eng.read_buffer(out.buf, B)
        got = from_padded(got_buf, B, Ho, Wo, 0, cout)
        ref = F.conv2d(torch.from_numpy(x).half().float(), torch.from_numpy(w).half().float(), torch.from_numpy(b), stride=2, padding=pad)
        ref = {0: lambda t: t, 1: F.silu, 2: F.relu}[act](ref).numpy()
        err = float(np.abs(got - ref).max()) / max(1.0, float(np.abs(ref).max()))
        assert err < 2e-3, (k, cout, H, err)
        assert halo_is_zero(got_buf, B, Ho, Wo)
        # frame 0 alone gives the same bits (batch invariance)
        eng1 = _capi.Engine(path, 0, max_batch=1)
        eng1.write_buffer(pb.image.buf, to_padded(x[:1], 4))
        eng1.run(1)
        assert np.array_equal(eng1.read_buffer(out.buf, 1), got_buf[:got_buf.shape[0] // B])
        eng1.close(); eng.close()


@pytest.mark.parametrize("impl", [1, 0])
def test_stem_repack_7x7s2(tmp_path, impl):
    """UFLD/ResNet stem without a patch matrix: stempack re-layout + 4 vertical GEMM taps == conv2d(7, stride 2, pad 3)."""
    rng = np.random.default_rng(11)
    for (B, H, W) in ((2, 32, 64), (1, 64, 160)):
        pb = plan.PlanBuilder(plan.MODEL_UFLDV2, 3, H, W)
        w = (rng.standard_normal((64, 3, 7, 7)) * 0.1).astype(np.float32)
        b = (rng.standard_normal(64) * 0.1).astype(np.float32)
        out = pb.stem7x7s2(pb.image, w, b, plan.ACT_RELU)
        path = str(tmp_path / f"stem_{impl}_{H}.b200w")
        pb.write(path)
        eng = _capi.Engine(path, 0, max_batch=B, conv_impl=impl)
        x = rng.standard_normal((B, 3, H, W)).astype(np.float32)
        eng.write_buffer(pb.image.buf, to_padded(x, 4))
        for _ in range(3):
            eng.run(B)
        got_buf = eng.read_buffer(out.buf, B)
        got = from_padded(got_buf, B, H // 2, W // 2, 0, 64)
        ref = F.relu(F.conv2d(torch.from_numpy(x).half().float(), torch.from_numpy(w).half().float(), torch.from_numpy(b), stride=2, padding=3)).numpy()
        err = float(np.abs(got - ref).max()) / max(1.0, float(np.abs(ref).max()))
        assert err < 4e-3, (impl, H, err)
        assert halo_is_zero(got_buf, B, H // 2, W // 2)
        eng.close()


@pytest.mark.parametrize("impl", [1, 0])
def test_fc_swap_ab(tmp_path, impl):
    """FC layers (swap-AB plan ops) with at most 48 MiB of fp16 weights: impl 0 runs them as fc_stream_kernel, impl 1 through the
    SIMT validation kernel.  The tcgen05 swap-AB GEMM, which takes the larger FCs, is checked in test_gpu_lane_head.py."""
    rng = np.random.default_rng(3)
    for (B, K, N, act) in ((3, 4992, 2048, 2), (8, 2048, 9128, 0), (1, 256, 136, 0)):
        pb = plan.PlanBuilder(plan.MODEL_UFLDV2, 3, 8, 8)
        xin = pb.new_dense(1, K)
        out = pb.new_dense(1, N, f32=(act == 0))
        w = (rng.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32)
        b = rng.standard_normal(N).astype(np.float32) * 0.1
        pb.fc(xin, K, w, b, act, out)
        path = str(tmp_path / f"fc_{impl}_{N}.b200w")
        pb.write(path)
        eng = _capi.Engine(path, 0, max_batch=B, conv_impl=impl)
        x = rng.standard_normal((B, K)).astype(np.float16)
        eng.write_buffer(xin, x)
        for _ in range(3):
            eng.run(B)
        got = eng.read_buffer(out, B).astype(np.float32)
        if impl == 0:
            assert "fc_stream" in eng.time_step(B, 0, 1)[2]
        ref = x.astype(np.float32) @ w.astype(np.float16).astype(np.float32).T + b
        if act == 2:
            ref = np.maximum(ref, 0)
        err = float(np.abs(got - ref).max()) / max(1.0, float(np.abs(ref).max()))
        assert err < 3e-3, (impl, B, K, N, err)
        eng.close()


def test_glue_ops(tmp_path):
    rng = np.random.default_rng(5)
    B, C, H, W = 2, 32, 10, 14
    pb = plan.PlanBuilder(plan.MODEL_YOLOV5, 3, H, W)
    xin = pb.new_padded(H, W, C)
    mp5 = pb.maxpool(xin, 5, 1, 2)
    mp3 = pb.maxpool(xin, 3, 2, 1)
    up = pb.new_padded(2 * H, 2 * W, 2 * C)
    pb.upsample2x(xin, pb.sub(up, C, C))
    path = str(tmp_path / "glue.b200w")
    pb.write(path)
    eng = _capi.Engine(path, 0, max_batch=B)
    x = rng.standard_normal((B, C, H, W)).astype(np.float32)
    eng.write_buffer(xin.buf, to_padded(x, C))
    eng.run(B)
    xt = torch.from_numpy(x).half().float()
    g5 = from_padded(eng.read_buffer(mp5.buf, B), B, H, W, 0, C)
    assert np.array_equal(g5, F.max_pool2d(xt, 5, 1, 2).numpy())
    g3 = from_padded(eng.read_buffer(mp3.buf, B), B, mp3.H, mp3.W, 0, C)
    assert np.array_equal(g3, F.max_pool2d(xt, 3, 2, 1).numpy())
    gu = from_padded(eng.read_buffer(up.buf, B), B, 2 * H, 2 * W, C, C)
    assert np.array_equal(gu, F.interpolate(xt, scale_factor=2, mode="nearest").numpy())
    eng.close()


def test_association_kernels(golden_dir):
    g = np.load(os.path.join(golden_dir, "track.npz"))
    from oracle import post
    for k in range(7):
        a, b, sc = g[f"assoc{k}_a"], g[f"assoc{k}_b"], g[f"assoc{k}_sc"]
        cost = _capi.iou_cost([a], [b])[0]
        fused = _capi.iou_cost([a], [b], [sc])[0]
        assert np.array_equal(cost, g[f"assoc{k}_cost"])
        assert np.array_equal(fused, post.iou_cost(a, b, sc))
        for nm, c, th in (("iou", cost, 0.5), ("fuse", fused, 0.8), ("fuse7", fused, 0.7)):
            x, y = _capi.lap([c], [th])[0]
            assert np.array_equal(x, g[f"assoc{k}_{nm}_x"]), (k, nm)
        x, y, c2 = _capi.associate(a, b, sc, 0.8, want_cost=True)
        assert np.array_equal(x, g[f"assoc{k}_fuse_x"]) and np.array_equal(c2, fused)
    # optimality on random dense problems vs the scipy restatement
    rng = np.random.default_rng(9)
    costs = [rng.uniform(0, 1, (int(t), int(d))) for t, d in rng.integers(1, 60, (24, 2))]
    th = [0.8] * len(costs)
    for (x, y), c in zip(_capi.lap(costs, th), costs):
        xo, yo, tot = post.lapjv_extended(c, 0.8)
        mine = c[np.nonzero(x >= 0)[0], x[x >= 0]].sum() + 0.4 * ((x < 0).sum() + (y < 0).sum())
        assert abs(mine - tot) < 1e-9
        assert np.array_equal(x, xo)


def test_comm_single_rank_gather():
    """adas_comm_*: the C-driven NCCL gather (own communicator, private stream) with world size 1 -- every call is asynchronous, the
    staging ring is reused, the last block wins.  The 2 / 8 rank path is exercised by `bench.py --gpus N` (SCALE runs)."""
    rec = np.arange(8 * 300 * 7, dtype=np.float32).reshape(8, 300, 7)
    c = _capi.Comm(0, 0, 1, _capi.Comm.unique_id(), rec.nbytes)
    for i in range(11):                      # more calls than ring slots
        rec[0, 0, 0] = float(i)
        c.all_gather(rec)
    c.sync()
    out = c.read()
    assert out.shape == (1, rec.size)
    assert out[0, 0] == 10.0 and np.array_equal(out[0, 1:], rec.ravel()[1:])
    assert c.info() == (1, 11)
    c.close()
