"""The UFLD lane head, kernel by kernel, against float64 references, and batch invariance of the whole lane network.

The head is pool conv -> LayerNorm -> FC1 -> ReLU -> FC2 (plan.build_ufldv2).  Three kernels run it:
  * the swap-AB tcgen05 GEMM (gemm_v3.cu, transposed = 1): every FC with more than 48 MiB of fp16 weights, i.e. every UFLD FC2;
  * fc_stream_kernel (elementwise.cu): the smaller FCs (FC1); conv_impl 1 runs the same shapes through the SIMT validation kernel;
  * layernorm_kernel (elementwise.cu): the CULane LayerNorm over the padded pool-conv slab.
Each output element is held to its own error bound (check_fc / check_ln), not to a fraction of the output's range, so a wrong
small element cannot hide behind a large one.  The checkers' self-tests need no GPU: they show that the bounds reject the answers
plausible kernel defects produce and accept legitimate fp32 rounding."""
import re

import numpy as np
import pytest
from scipy.special import expit

import synth
import adas_b200  # noqa: F401
from adas_b200 import _capi, plan
from gpu_util import U16, U32, cached_plan, to_padded
from gpu_util import check as _check

FC_STREAM_MAX_BYTES = 48 << 20          # engine.cu: an FC with at most this many bytes of fp16 weights runs as fc_stream_kernel
RELU, SILU, NONE = plan.ACT_RELU, plan.ACT_SILU, plan.ACT_NONE


# ---------------------------------------------------------------------------------------------------------------------------------
# float64 references and per-element checkers
# ---------------------------------------------------------------------------------------------------------------------------------
def _act64(z, act):
    if act == RELU:
        return np.maximum(z, 0.0)
    if act == SILU:
        return z * expit(z)
    return z


def fc_reference(x16, w16, b, act, chunk=8192):
    """float64 act(x w^T + b) on the fp16 operands, and mag = sum_k |x_k w_k| of every output (the scale of its fp32 accumulation
    error).  Computed in chunks of output features: the CULane FC2 weights (91224 x 2048) take 1.5 GB in float64."""
    x = x16.astype(np.float64)
    ax = np.abs(x)
    N = w16.shape[0]
    ref = np.empty((x.shape[0], N))
    mag = np.empty((x.shape[0], N))
    for n0 in range(0, N, chunk):
        w = w16[n0:n0 + chunk].astype(np.float64)
        ref[:, n0:n0 + chunk] = x @ w.T + b[n0:n0 + chunk]
        mag[:, n0:n0 + chunk] = ax @ np.abs(w).T
    return _act64(ref, act), mag


def check_fc(got, ref, mag, K, f16_out, what="fc"):
    """Per element: |got - ref| <= K 2^-24 sum_k |x_k w_k| (fp32 accumulation of K products) + 2^-11 |ref| (fp16 output rounding)
    + 1e-6.  Returns the worst |got - ref| / bound."""
    tol = K * U32 * mag + (U16 * np.abs(ref) if f16_out else 0.0) + 1e-6
    return _check(got, ref, tol, what)


def layernorm_reference(x16, real, gamma, beta, eps):
    """float64 LayerNorm of every row of x16 [rows, D] with the mean and variance of its real entries (Dn = real.sum() of them).
    Returns (out, gamma * xhat, gamma * mean / sqrt(var + eps)), all zero on the structural (halo) entries."""
    x = x16.astype(np.float64)
    xr = x[:, real]
    mean = xr.mean(1, keepdims=True)
    sd = np.sqrt(((xr - mean) ** 2).mean(1, keepdims=True) + eps)
    gx = np.where(real, gamma * (x - mean) / sd, 0.0)
    return np.where(real, gx + beta, 0.0), gx, np.where(real, gamma * mean / sd, 0.0)


def check_ln(got, lnref, real, what="layernorm"):
    """Per real entry: |got - ref| <= 2^-11 |ref| (fp16 output rounding) + 2e-4 |gamma xhat| (fp32 variance and scaling)
    + 2^-22 |gamma mean / sd| (the mean is an fp32 number: a few of its roundings shift every xhat by that much) + 1e-6.  Halo entries
    must be exactly zero.  `lnref` is what layernorm_reference returned for these rows.  Returns the worst |got - ref| / bound."""
    ref, gx, gm = lnref
    halo = got[:, ~real].astype(np.float32)
    assert not halo.any(), f"{what}: {int((halo != 0).sum())} halo entries are not zero"
    tol = U16 * np.abs(ref) + 2e-4 * np.abs(gx) + 2.0 ** -22 * np.abs(gm) + 1e-6
    return _check(got[:, real], ref[:, real], tol[:, real], what)


def _report(kernel, case, ratio):
    print(f"[lane-head] {kernel} {case}: worst |got - ref| / bound = {ratio:.3f}")


# ---------------------------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------------------------
def _fc_operands(rng, B, K, N, x_cols=None):
    """fp16 activations [B, x_cols] (columns past K are large garbage no FC may read), fp16 weights [N, K] ~ N(0, 1/K), fp32 bias."""
    x16 = rng.standard_normal((B, x_cols or K)).astype(np.float16)
    x16[:, K:] = (1e3 * rng.standard_normal((B, (x_cols or K) - K))).astype(np.float16)
    w16 = np.empty((N, K), np.float16)
    for n0 in range(0, N, 8192):
        w16[n0:n0 + 8192] = rng.standard_normal((min(8192, N - n0), K), dtype=np.float32) / np.float32(np.sqrt(K))
    return x16, w16, (0.1 * rng.standard_normal(N)).astype(np.float32)


def _slab_mask(H, W, C):
    """Real (interior) entries of one image's padded NHWC slab, flattened."""
    m = np.zeros((H + 2, W + 2, C), bool)
    m[1:-1, 1:-1] = True
    return m.ravel()


# LayerNorm row contents: (name, scale, offset) -> scale * (offset + N(0, 1)) on the real entries
LN_ROWS = [("N(0,1)", 1.0, 0.0), ("mean/std 5", 1.0, 5.0), ("mean/std 20", 1.0, 20.0), ("mean/std 100", 1.0, 100.0),
           ("zeros", 0.0, 0.0), ("fp16 outliers", 1.0, 0.0), ("mean/std -100", 1.0, -100.0), ("mean/std 100 at std 0.01", 0.01, 100.0)]


def _ln_inputs(rng, real, rows):
    """fp16 slab rows cycling through LN_ROWS (zero halo), and gamma / beta random on the real entries, zero on the halo."""
    D, Dn = real.size, int(real.sum())
    x16 = np.zeros((rows, D), np.float16)
    for r in range(rows):
        name, scale, off = LN_ROWS[r % len(LN_ROWS)]
        v = scale * (off + rng.standard_normal(Dn))
        if name == "fp16 outliers":
            v[rng.choice(Dn, 4, replace=False)] = (60000.0, -60000.0, 59008.0, -61024.0)
        x16[r, real] = v.astype(np.float16)
    gamma = np.where(real, 1.0 + 0.25 * rng.standard_normal(D), 0.0).astype(np.float32)
    beta = np.where(real, 0.5 * rng.standard_normal(D), 0.0).astype(np.float32)
    return x16, gamma, beta


# ---------------------------------------------------------------------------------------------------------------------------------
# checker self-tests (CPU)
# ---------------------------------------------------------------------------------------------------------------------------------
def _as_out(r, f16):
    return r.astype(np.float16 if f16 else np.float32)


@pytest.mark.parametrize("act,f16", [(NONE, False), (RELU, True), (SILU, False)])
def test_check_fc_rejects_kernel_defects(act, f16):
    """Wrong answers of the kind a swap-AB or weight-stream defect produces, built from the float64 reference: each must fail."""
    rng = np.random.default_rng(1)
    B, K, N = 6, 2048, 300                   # the last 128-row M tile holds features 256..299
    x16, w16, b = _fc_operands(rng, B, K, N)
    ref, mag = fc_reference(x16, w16, b, act)
    check_fc(_as_out(ref, f16), ref, mag, K, f16)
    wrong = {"last 64-term K block dropped": fc_reference(x16[:, :K - 64], w16[:, :K - 64], b, act)[0]}
    n = int(np.argmax((ref[:, :-1] > 0.5).any(0) & (np.abs(np.diff(b)) > 0.05)))     # a visible output, a bias unlike the next
    b2 = b.copy()
    b2[n] = b[n + 1]
    wrong["feature %d uses its neighbour's bias" % n] = fc_reference(x16, w16, b2, act)[0]
    shifted = ref.copy()
    shifted[3] = ref[2]
    wrong["batch column 2 shifted into column 3"] = shifted
    if act != NONE:
        skipped = ref.copy()
        skipped[:, 256:] = fc_reference(x16, w16[256:], b[256:], NONE)[0]
        wrong["activation skipped in the last M tile"] = skipped
    for name, g in wrong.items():
        with pytest.raises(AssertionError):
            check_fc(_as_out(g, f16), ref, mag, K, f16, name)


@pytest.mark.parametrize("act,f16", [(NONE, False), (RELU, True), (SILU, False)])
def test_check_fc_accepts_fp32_matmul(act, f16):
    """A float32 matmul of the same fp16 operands (BLAS sgemm: blocked, another summation order) is within the bound."""
    rng = np.random.default_rng(2)
    for B, K, N in ((6, 2048, 300), (5, 8, 13), (3, 4992, 64)):
        x16, w16, b = _fc_operands(rng, B, K, N)
        ref, mag = fc_reference(x16, w16, b, act)
        z = x16.astype(np.float32) @ w16.astype(np.float32).T + b
        got = np.maximum(z, 0) if act == RELU else z * expit(z) if act == SILU else z
        check_fc(_as_out(got.astype(np.float32), f16), ref, mag, K, f16)


def _butterfly(a):
    """Lane 0 of a 32-lane xor-shuffle sum over the last axis (fp32)."""
    lanes = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        a = a + a[..., lanes ^ o]
    return a[..., 0]


def _kernel_order_sum(x, square=False):
    """fp32 row sums of x [rows, D] (or of x*x, fused multiply-add) in layernorm_kernel's order: 256 threads stride over the row,
    then a butterfly over each warp's lanes and one over the 8 warp totals."""
    R, D = x.shape
    acc = np.zeros((R, 256), np.float32)
    for i0 in range(0, D, 256):
        seg = x[:, i0:i0 + 256]
        n = seg.shape[1]
        if square:
            acc[:, :n] = (acc[:, :n].astype(np.float64) + seg.astype(np.float64) ** 2).astype(np.float32)
        else:
            acc[:, :n] += seg
    warps = _butterfly(acc.reshape(R, 8, 32))
    return _butterfly(np.concatenate([warps, np.zeros((R, 24), np.float32)], 1))


def _one_pass_fp32(x16, Dn, gamma, beta, eps):
    """fp32 emulation of the one-pass statistics var = E[x^2] - mean^2, sums in the kernel's order."""
    x = x16.astype(np.float32)
    mean = _kernel_order_sum(x) / np.float32(Dn)
    ex2 = _kernel_order_sum(x, square=True) / np.float32(Dn)
    var = np.maximum(ex2.astype(np.float64) - mean.astype(np.float64) ** 2, 0).astype(np.float32)
    rstd = (1.0 / np.sqrt(var + np.float32(eps))).astype(np.float32)
    return ((x - mean[:, None]) * rstd[:, None] * gamma + beta).astype(np.float16)


def _two_pass_fp32(x16, real, gamma, beta, eps, dn=None):
    """fp32 two-pass statistics over the real entries: the mean, then the mean squared deviation from it (divided by dn)."""
    x = x16.astype(np.float32)
    dn = np.float32(dn or real.sum())
    xr = x[:, real]
    mean = xr.sum(1, dtype=np.float32) / dn
    var = ((xr - mean[:, None]) ** 2).sum(1, dtype=np.float32) / dn
    rstd = np.float32(1) / np.sqrt(var + np.float32(eps))
    return np.where(real, (x - mean[:, None]) * rstd[:, None] * gamma + beta, 0).astype(np.float16)


def test_check_ln_rejects_one_pass_variance_and_wrong_count():
    """At |mean|/std = 100 the one-pass variance E[x^2] - mean^2 cancels about 13 of fp32's 24 bits; normalising by the slab length
    instead of the real feature count is wrong at any offset.  The bound must reject both."""
    rng = np.random.default_rng(3)
    real = _slab_mask(10, 50, 8)                                     # CULane res34 pool conv: slab 4992, 4000 real features
    Dn = int(real.sum())
    x16, gamma, beta = _ln_inputs(rng, real, 16)
    big = [r for r in range(16) if abs(LN_ROWS[r % len(LN_ROWS)][2]) == 100.0]
    for eps in (1e-5, 1e-6):
        with pytest.raises(AssertionError):
            check_ln(_one_pass_fp32(x16[big], Dn, gamma, beta, eps), layernorm_reference(x16[big], real, gamma, beta, eps), real, "one-pass")
        with pytest.raises(AssertionError):
            check_ln(_two_pass_fp32(x16[:2], real, gamma, beta, eps, dn=real.size), layernorm_reference(x16[:2], real, gamma, beta, eps), real,
                     "statistics over the slab length")


def test_check_ln_accepts_two_pass_fp32():
    """Two-pass fp32 statistics pass on every row kind; the one-pass formula passes too while |mean|/std stays at or below 20, so
    the bound is aimed at the cancellation, not at fp32 rounding in general."""
    rng = np.random.default_rng(4)
    for geom in ((10, 50, 8), (5, 7, 8)):
        real = _slab_mask(*geom)
        x16, gamma, beta = _ln_inputs(rng, real, 16)
        small = [r for r in range(16) if LN_ROWS[r % len(LN_ROWS)][2] in (0.0, 5.0, 20.0)]
        for eps in (1e-5, 1e-6):
            lnref = layernorm_reference(x16, real, gamma, beta, eps)
            check_ln(_two_pass_fp32(x16, real, gamma, beta, eps), lnref, real, f"two-pass {geom}")
            check_ln(_one_pass_fp32(x16[small], int(real.sum()), gamma, beta, eps), [a[small] for a in lnref], real, f"one-pass {geom}")


# ---------------------------------------------------------------------------------------------------------------------------------
# FC kernels on the GPU
# ---------------------------------------------------------------------------------------------------------------------------------
def _fc_plan(tmp_path, name, K, w16, b, act, f16_out, x_cols=None, slab=None):
    """One FC op: input = a dense [1, x_cols] row per image, or the padded feature map `slab` = (H, W, C) read flat."""
    pb = plan.PlanBuilder(plan.MODEL_UFLDV2, 3, 8, 8)
    xin = pb.new_padded(*slab).buf if slab else pb.new_dense(1, x_cols or K)
    out = pb.new_dense(1, w16.shape[0], f32=not f16_out)
    pb.fc(xin, K, w16, b, act, out)
    path = str(tmp_path / f"{name}.b200w")
    pb.write(path)
    return path, xin, out


def _run_op(eng, xin, out, x16):
    """Runs the plan on the rows of x16 and returns its output rows.  The output rows are set to NaN first, so an element the
    kernel leaves unwritten cannot pass for the result of an earlier run."""
    B = x16.shape[0]
    info = eng.buffer_info(out)
    eng.write_buffer(out, np.full((B * info["rows_per_img"], info["C"]), np.nan, info["dtype"]))
    eng.write_buffer(xin, x16)
    eng.run(B)
    return eng.read_buffer(out, B)


def _same_bits(a, b):
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def _check_smaller_batches(eng, xin, out, x16, got, batches, kernel_tag):
    """Rows of x16 run again at each smaller batch size (batch 1: every row) come out bit for bit as in the full batch, through
    the same kernel."""
    B = x16.shape[0]
    for bs in batches:
        r0 = bs if 2 * bs <= B else 0
        assert _same_bits(_run_op(eng, xin, out, x16[r0:r0 + bs]), got[r0:r0 + bs]), f"batch {bs} (rows {r0}..) differs from batch {B}"
        if kernel_tag:
            assert kernel_tag in eng.time_step(bs, 0, 1)[2]
    for r in range(B):
        assert _same_bits(_run_op(eng, xin, out, x16[r:r + 1]), got[r:r + 1]), f"row {r}: batch 1 differs from batch {B}"
    if kernel_tag:
        assert kernel_tag in eng.time_step(1, 0, 1)[2]


SWAP_AB_CASES = [
    # batches (the first checked against float64, the others row by row against it), K, N, activation, fp16 output
    ((32, 8), 2048, 91224, NONE, False),    # UFLDv2 CULane FC2 (373 MB): BN 32 and 16, ragged last M tile, many tiles per CTA
    ((17,), 1000, 25177, RELU, True),       # K tail 1000 = 15*64 + 40, last M tile of 89 rows, batch tail inside a 32-wide tile
    ((3,), 1024, 24577, NONE, False),       # one weight row over the fc_stream limit: the last M tile has a single row
    ((144,), 1024, 25000, SILU, True),      # batch > 128: BN 144, MT = 1, 256-column sub-tiles
    ((8,), 2048, 14472, NONE, False),       # UFLD v1 CULane FC2
]


@pytest.mark.gpu
@pytest.mark.parametrize("batches,K,N,act,f16", SWAP_AB_CASES, ids=[f"B{c[0][0]}-K{c[1]}-N{c[2]}" for c in SWAP_AB_CASES])
def test_fc_swap_ab_tcgen05_vs_float64(tmp_path, batches, K, N, act, f16):
    """The tcgen05 swap-AB GEMM (rows = output features, columns = images) on FCs too large for the weight stream.  Catches a
    dropped or doubled K tail, a misplaced bias, stores into the wrong batch column or past the last feature, an activation
    skipped in a partial tile, and per-image results that change with the batch (BN = ceil16(batch) changes the tile)."""
    assert N * K * 2 > FC_STREAM_MAX_BYTES
    rng = np.random.default_rng(N)
    x16, w16, b = _fc_operands(rng, batches[0], K, N)
    path, xin, out = _fc_plan(tmp_path, f"fc_{N}", K, w16, b, act, f16)
    eng = _capi.Engine(path, 0, max_batch=batches[0])
    for _ in range(2):                        # eager, then graph capture; _run_op's launch is a graph replay
        eng.write_buffer(xin, x16)
        eng.run(batches[0])
    got = _run_op(eng, xin, out, x16)
    desc = eng.time_step(batches[0], 0, 1)[2]
    assert "tr=1 | v3" in desc, desc
    ref, mag = fc_reference(x16, w16, b, act)
    tile = re.search(r"BN=\d+ MT=\d+", desc).group()
    _report("swap-AB", f"B={batches[0]} K={K} N={N} ({tile})", check_fc(got, ref, mag, K, f16, f"swap-AB {N}"))
    _check_smaller_batches(eng, xin, out, x16, got, batches[1:], "tr=1 | v3")
    eng.close()


FC_STREAM_CASES = [
    # batches, K, N, activation, fp16 output, input layout
    ((32, 16, 9, 8, 7), 4992, 2048, RELU, True, "slab"),    # CULane FC1 reading the padded 10x50x8 slab: up to 4 y-groups, nb tails
    ((9,), 2048, 1000, NONE, False, "wide"),                # input rows of K + 64 columns: x_ld != K
    ((5,), 8, 13, RELU, True, "dense"),                     # one 16-byte chunk (warps 1-7 get no K), N % 8 != 0 (clamp, guard)
    ((12,), 1000, 2047, SILU, False, "dense"),              # SiLU, fp32 out, ragged last feature group, second y-group of 4
    ((3,), 1024, 24576, NONE, False, "dense"),              # exactly 48 MiB of weights: the largest FC that still streams
]


@pytest.mark.gpu
@pytest.mark.parametrize("impl", [0, 1])
@pytest.mark.parametrize("batches,K,N,act,f16,layout", FC_STREAM_CASES, ids=[f"B{c[0][0]}-K{c[1]}-N{c[2]}-{c[5]}" for c in FC_STREAM_CASES])
def test_fc_stream_vs_float64(tmp_path, impl, batches, K, N, act, f16, layout):
    """fc_stream_kernel (impl 0) and the SIMT validation kernel (impl 1).  Catches a second y-group or an nb tail that reads or
    writes the wrong rows, a feature clamp / guard that lets the last group spill, a warp with an empty K slice that adds garbage,
    a wrong SiLU, K used as the row stride, a slab whose halo or feature order is read wrongly, and results that change with the
    batch."""
    rng = np.random.default_rng(K + N)
    B = batches[0]
    if layout == "slab":
        # the plan packer's layout (plan.build_ufldv2): NCHW feature f = c*H*W + h*W + w sits at slab entry ((h+1)*(W+2) + w+1)*8 + c
        H, W, C = 10, 50, 8
        xd, wd, b = _fc_operands(rng, B, H * W * C, N)
        ci, hi, wi = np.meshgrid(np.arange(C), np.arange(H), np.arange(W), indexing="ij")
        w16 = np.zeros((N, K), np.float16)
        w16[:, (((hi + 1) * (W + 2) + wi + 1) * C + ci).ravel()] = wd
        x16 = to_padded(xd.reshape(B, C, H, W).astype(np.float32), C).reshape(B, K)
        ref, mag = fc_reference(xd, wd, b, act)
    else:
        x16, w16, b = _fc_operands(rng, B, K, N, x_cols=K + 64 if layout == "wide" else None)
        ref, mag = fc_reference(x16[:, :K], w16, b, act)
    assert N * K * 2 <= FC_STREAM_MAX_BYTES
    path, xin, out = _fc_plan(tmp_path, f"fcs_{N}", K, w16, b, act, f16, x_cols=x16.shape[1], slab=(H, W, C) if layout == "slab" else None)
    eng = _capi.Engine(path, 0, max_batch=B, conv_impl=impl)
    for _ in range(2):
        eng.write_buffer(xin, x16)
        eng.run(B)
    got = _run_op(eng, xin, out, x16)
    tag = "fc_stream" if impl == 0 else None
    if tag:
        assert tag in eng.time_step(B, 0, 1)[2]
    _report("fc_stream" if impl == 0 else "simt-fc", f"B={B} K={K} N={N} {layout}", check_fc(got, ref, mag, K, f16, f"impl {impl} N={N}"))
    _check_smaller_batches(eng, xin, out, x16, got, batches[1:], tag)
    eng.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# LayerNorm on the GPU
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("eps", [1e-5, 1e-6])
@pytest.mark.parametrize("geom", [(10, 50, 8), (5, 7, 8)], ids=["culane-slab4992", "slab504"])
def test_layernorm_vs_float64(tmp_path, geom, eps):
    """layernorm_kernel over padded slabs: CULane res34 (4992 entries, 4000 real) and one with fewer than two entries per thread.
    Rows with |mean|/std up to 100, all zeros (variance 0: the output is fp16(beta) exactly) and fp16 outliers near 6e4, at batch
    32, 8, 2 and 1.  Catches variance lost to cancellation, statistics over the slab length instead of the real count, a halo
    written non-zero, a reduction that drops a warp or a thread's tail, and rows that depend on the batch."""
    rng = np.random.default_rng(geom[0] + int(1e6 * eps))
    real = _slab_mask(*geom)
    D, Dn = real.size, int(real.sum())
    x16, gamma, beta = _ln_inputs(rng, real, 32)
    pb = plan.PlanBuilder(plan.MODEL_UFLDV2, 3, 8, 8)
    xin = pb.new_padded(*geom)
    out = pb.new_dense(1, D)
    pb.layernorm(xin.buf, D, Dn, gamma, beta, eps, out)
    path = str(tmp_path / "ln.b200w")
    pb.write(path)
    eng = _capi.Engine(path, 0, max_batch=32)
    lnref = layernorm_reference(x16, real, gamma, beta, eps)
    got32 = _run_op(eng, xin.buf, out, x16)
    kinds = [LN_ROWS[r % len(LN_ROWS)][0] for r in range(32)]
    worst = {}
    for r in range(32):
        worst[kinds[r]] = max(worst.get(kinds[r], 0.0), check_ln(got32[r:r + 1], [a[r:r + 1] for a in lnref], real, f"row {r} ({kinds[r]})"))
        if kinds[r] == "zeros":
            assert _same_bits(got32[r, real], beta[real].astype(np.float16)), "zero-variance row is not fp16(beta)"
    for k, v in worst.items():
        _report("layernorm", f"{geom} eps={eps:g} {k}", v)
    for bs, r0 in ((8, 8), (2, 2)):
        assert _same_bits(_run_op(eng, xin.buf, out, x16[r0:r0 + bs]), got32[r0:r0 + bs]), f"batch {bs} differs from batch 32"
    for r in range(32):
        assert _same_bits(_run_op(eng, xin.buf, out, x16[r:r + 1]), got32[r:r + 1]), f"row {r}: batch 1 differs from batch 32"
    eng.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# whole lane networks: per-frame results do not depend on the batch
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind,kw,B", [("ufldv2", dict(backbone="34"), 32), ("ufldv2", dict(backbone="18", cfg="tusimple"), 8),
                                        ("ufldv1", dict(backbone="18", cfg="culane"), 8)],
                         ids=["v2-res34-culane-b32", "v2-res18-tusimple-b8", "v1-res18-culane-b8"])
def test_ufld_batch_invariance(kind, kw, B):
    """Frame k of a batch-B run equals the same frame run alone (and, at B = 32, frames 8..15 run as a batch of 8), bit for bit:
    the head tensors of `infer` and the lane points, counts, status and coordinates of `ufld_detect`.  The three head kernels take
    other tile and grid shapes at every one of these batch sizes."""
    path, _, _ = cached_plan(kind, **kw)
    cfg = (plan.UFLD_V1_DATASETS if kind == "ufldv1" else plan.UFLD_DATASETS)[kw.get("cfg", "culane")]
    eng = _capi.Engine(path, 0, max_batch=B)
    frames = np.stack([synth.frame(500 + s) for s in range(B)])
    x = _capi.ufld_preprocess(frames, (cfg["in_h"], cfg["in_w"]), cfg["crop_ratio"])
    heads = eng.infer(x)
    # batch-1 runs in descending frame order: the device rows a run leaves unwritten then hold another frame's result
    subsets = [(8, 16)] if B == 32 else []
    for k0, k1 in subsets + [(k, k + 1) for k in reversed(range(B))]:
        part = eng.infer(x[k0:k1])
        for i, (p, h) in enumerate(zip(part, heads)):
            assert _same_bits(p, h[k0:k1]), f"head {i}: frames {k0}..{k1 - 1} run as a batch of {k1 - k0} differ from the batch of {B}"
    pts, npts, status, coords = eng.ufld_detect(frames, want_coords=True)
    assert npts.any(), "no lane points at this operating point: the comparison below would be empty"
    for k in reversed(range(B)):
        p1, n1, s1, c1 = eng.ufld_detect(frames[k:k + 1], want_coords=True)
        assert np.array_equal(n1[0], npts[k]) and np.array_equal(s1[0], status[k]), f"frame {k}: lane counts / status differ"
        for lane in range(4):
            n = int(npts[k, lane])
            assert np.array_equal(p1[0, lane, :n], pts[k, lane, :n]) and _same_bits(c1[0, lane, :n], coords[k, lane, :n]), (k, lane)
    eng.close()
