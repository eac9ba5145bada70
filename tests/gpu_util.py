"""Helpers for the GPU parity tests: padded-NHWC packing, cached plan files, and float64 references with per-element checkers."""
import os

import numpy as np

import adas_b200  # noqa: F401
from adas_b200 import plan

U32, U16 = 2.0 ** -24, 2.0 ** -11      # unit roundoff of fp32 and of fp16
SILU_SLOPE = 1.1                        # max |SiLU'(z)| = 1.0998: how far an accumulation error can grow through the activation
SILU_REL = 2.0 ** -20                   # tc_common.cuh silu2: ex2.approx + rcp.approx (PTX: 2^-22 / 2^-23 relative) and four fp32 roundings


def check(got, ref, tol, what):
    """Asserts |got - ref| <= tol element by element (a NaN fails) and returns the worst |got - ref| / tol."""
    err = np.abs(got.astype(np.float64) - ref)
    bad = ~(err <= tol)
    if bad.any():
        i = np.unravel_index(np.argmax(bad), bad.shape)
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} elements outside the bound; first at {i}: got {got[i]}, "
                             f"reference {ref[i]:.7g}, bound {tol[i]:.3g}")
    return float((err / tol).max())


def conv_reference(x16, w16, b, s, pad, act, r16=None, res_pre=False, device="cpu"):
    """float64 act(conv(x, w) + b (+ r)) (+ r) on the fp16 operands, and mag = conv(|x|, |w|) + |b| + |r|, the scale of every
    output's fp32 accumulation error.  x16 [n, cin, H, W] and w16 [cout, cin, k, k] fp16, b [cout] fp32, r16 [n, cout, Ho, Wo]
    fp16 added before (res_pre) or after the activation.  Returns float64 numpy arrays [n, cout, Ho, Wo]."""
    import torch
    import torch.nn.functional as F
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(device=device, dtype=torch.float64)
    x, w, bb = t(x16), t(w16), t(b)
    z = F.conv2d(x, w, bb, stride=s, padding=pad)
    mag = F.conv2d(x.abs(), w.abs(), bb.abs(), stride=s, padding=pad)
    if r16 is not None:
        r = t(r16)
        mag = mag + r.abs()
        if res_pre:
            z = z + r
    if act == plan.ACT_SILU:
        z = z * torch.sigmoid(z)
    elif act == plan.ACT_RELU:
        z = torch.clamp(z, min=0.0)
    if r16 is not None and not res_pre:
        z = z + r
    return z.cpu().numpy(), mag.cpu().numpy()


def check_conv(got, ref, mag, K, act, f16_out, what="conv"):
    """Per element: |got - ref| <= 1.1 (K + 2) 2^-24 mag (fp32 accumulation of K products, the bias and the residual, through the
    activation's slope) + 2^-20 |ref| (SiLU only) + 2^-11 |ref| (fp16 output only) + 1e-6.  K = k * k * cin_real.  Returns the
    worst |got - ref| / bound."""
    tol = SILU_SLOPE * (K + 2) * U32 * mag + (SILU_REL * np.abs(ref) if act == plan.ACT_SILU else 0.0) \
        + (U16 * np.abs(ref) if f16_out else 0.0) + 1e-6
    return check(got, ref, tol, what)



def to_padded(x_nchw: np.ndarray, C: int) -> np.ndarray:
    """[B,c,H,W] float -> [B*(H+2)*(W+2), C] fp16 with zero halo / zero extra channels."""
    B, c, H, W = x_nchw.shape
    out = np.zeros((B, H + 2, W + 2, C), np.float16)
    out[:, 1:-1, 1:-1, :c] = x_nchw.transpose(0, 2, 3, 1).astype(np.float16)
    return out.reshape(-1, C)


def from_padded(buf: np.ndarray, B: int, H: int, W: int, coff: int, c: int) -> np.ndarray:
    """[B*(H+2)*(W+2), ld] -> [B,c,H,W] float32 interior."""
    v = buf.reshape(B, H + 2, W + 2, -1)[:, 1:-1, 1:-1, coff:coff + c]
    return v.astype(np.float32).transpose(0, 3, 1, 2)


def halo_is_zero(buf: np.ndarray, B: int, H: int, W: int) -> bool:
    v = buf.reshape(B, H + 2, W + 2, -1).astype(np.float32)
    return not (v[:, 0].any() or v[:, -1].any() or v[:, :, 0].any() or v[:, :, -1].any())


def cached_plan(kind: str, seed: int = 0, **kw):
    """Build (once per process tree) the synthetic plan + return (path, Weights-like state_dict)."""
    CACHE = plan.cache_dir()
    import zlib
    prof = zlib.crc32(repr((plan.SYNTH_PROFILES.get("ufldv2" if kind == "ufldv1" else kind), plan.PLAN_VERSION)).encode()) & 0xffff      # a changed operating point is a new plan
    tag = kind + "_" + "_".join(f"{k}{v}" for k, v in sorted(kw.items())) + f"_s{seed}_{prof:04x}"
    path = os.path.join(CACHE, tag + ".b200w")
    variant = kw.get("scale", kw.get("backbone"))             # calibrated BatchNorm statistics exist for the tested variants
    W = plan.synth_weights("ufldv2" if kind == "ufldv1" else kind, seed, variant=variant)
    if kind == "yolov8":
        pb = plan.build_yolov8(W, **kw)
    elif kind == "yolov5":
        pb = plan.build_yolov5(W, **kw)
    elif kind == "ufldv1":
        pb = plan.build_ufldv1(W, **kw)
    else:
        pb = plan.build_ufldv2(W, **kw)
    if not os.path.isfile(path):
        pb.write(path + ".tmp")
        os.replace(path + ".tmp", path)
    return path, W.state_dict, pb
