"""Float64 reference and element-wise comparator for the convolution epilogues (csrc/conv_gemm.cuh).

Torch only, so that the CPU tests can import it. The reference runs the kernel's own sequence of steps in float64 on
the bf16-rounded operands:  pre = acc * scale + shift + residual * res_scale + res_shift;  y = relu(pre);
bit = (pre > 0).  Every stored element must satisfy

    |got - ref| <= 2^-8 |ref| + E,   E = C_ACC * |scale| * conv(|x|, |w|) + 2^-22 (|shift| + |res * res_scale| + |res_shift|)

where conv(|x|, |w|) is the float64 convolution of the absolute values (the scale of the fp32 accumulation). 2^-8 |ref|
is the final bf16 rounding (half an ulp at the bottom of a binade); E covers the fp32 accumulation and the fp32
epilogue arithmetic.
"""
from __future__ import annotations

import torch

# Accumulation constant of E, calibrated on a B200 (PR description: largest observed error / bound). The worst-case fp32
# bound K * 2^-24 at K = 4608 is 2^-11.8; a bf16 ulp is 2^-7 relative.
C_ACC = 2.0 ** -16
REL = 2.0 ** -8
C_ADD = 2.0 ** -22


def bits_to_bool(bits: torch.Tensor, channels: int) -> torch.Tensor:
    """[rows][channels/8] uint8 ReLU mask -> [rows][channels] bool (channel c = byte c // 8, bit c % 8)."""
    b = bits.reshape(-1, channels // 8).to(torch.int32)
    shifts = torch.arange(8, device=b.device, dtype=torch.int32)
    return ((b.unsqueeze(-1) >> shifts) & 1).reshape(-1, channels).bool()


def bool_to_bits(mask: torch.Tensor) -> torch.Tensor:
    """Inverse of bits_to_bool."""
    rows, channels = mask.shape
    m = mask.reshape(rows, channels // 8, 8).to(torch.int32)
    weights = (1 << torch.arange(8, device=m.device, dtype=torch.int32))
    return (m * weights).sum(-1).to(torch.uint8)


def epilogue_ref(acc, absacc, scale=None, shift=None, res=None, res_scale=None, res_shift=None, relu=False):
    """acc, absacc: float64 [rows][C] conv(x, w) and conv(|x|, |w|); res: [rows][C] (any float dtype, used as given);
    the per-channel vectors are [C]. Returns (pre, ref, E), all float64 [rows][C]."""
    acc = acc.double()
    pre = acc.clone()
    e_acc = absacc.double().clone()
    e_add = torch.zeros_like(pre)
    if scale is not None:
        pre = pre * scale.double()
        e_acc = e_acc * scale.double().abs()
    if shift is not None:
        pre = pre + shift.double()
        e_add = e_add + shift.double().abs()
    if res is not None:
        r = res.double()
        if res_scale is not None:
            r = r * res_scale.double()
            e_add = e_add + r.abs() + res_shift.double().abs()
            r = r + res_shift.double()
        else:
            e_add = e_add + r.abs()
        pre = pre + r
    ref = pre.clamp_min(0.0) if relu else pre
    return pre, ref, C_ACC * e_acc + C_ADD * e_add


def describe(idx, C, got, ref, bound, limit=8):
    rows = []
    for flat in idx[:limit].tolist():
        r, c = divmod(flat, C)
        rows.append(f"row {r} (M tile {r // 128}, row {r % 128}) ch {c} (64-chunk {c // 64}): got {got[r, c]:.6g} "
                    f"ref {ref[r, c]:.6g} bound {bound[r, c]:.3g}")
    return "\n  ".join(rows)


def check_values(got, ref, E, what="output"):
    """Every element within 2^-8 |ref| + E, no exception. Returns the largest |got - ref| / bound."""
    g = got.double().reshape(ref.shape)
    bound = REL * ref.abs() + E
    err = (g - ref).abs()
    bad = ~(err <= bound)   # NaN (unwritten) fails too
    if bad.any():
        idx = bad.flatten().nonzero().flatten()
        raise AssertionError(f"{what}: {idx.numel()} of {ref.numel()} elements out of bound\n  "
                             + describe(idx, ref.shape[1], g, ref, bound))
    zero_ok = bound > 0
    return float((err[zero_ok] / bound[zero_ok]).max()) if zero_ok.any() else 0.0


def check_bits(bits, y, pre, E, what="ReLU bits"):
    """bits == (y > 0) exactly (the backward pass relies on it), and bits == (pre > 0) wherever |pre| > E."""
    C = pre.shape[1]
    b = bits_to_bool(bits, C)
    yp = y.double().reshape(pre.shape) > 0
    bad = b != yp
    if bad.any():
        idx = bad.flatten().nonzero().flatten()
        r, c = divmod(int(idx[0]), C)
        raise AssertionError(f"{what}: {idx.numel()} bits differ from (y > 0); first at row {r} (M tile {r // 128}) "
                             f"ch {c}: bit {int(b[r, c])} y {float(y.reshape(pre.shape)[r, c])}")
    decided = pre.abs() > E
    bad = decided & (b != (pre > 0))
    if bad.any():
        idx = bad.flatten().nonzero().flatten()
        r, c = divmod(int(idx[0]), C)
        raise AssertionError(f"{what}: {idx.numel()} bits differ from the float64 sign; first at row {r} "
                             f"(M tile {r // 128}) ch {c}: bit {int(b[r, c])} pre {float(pre[r, c]):.6g}")


def check_stat_slots(partial, y, C, rtol=1e-5, second=None, what="statistics"):
    """partial [slots][2][C]: the fp64 sum over slots of sum / second moment equals the fp64 sum over the stored bf16 y
    (second = the factor of the second row: y itself for sum y^2, or the raw tensor for sum y * raw), within rtol of the
    sum of absolute values."""
    yd = y.double().reshape(-1, C)
    sd = yd if second is None else second.double().reshape(-1, C)
    got = partial.double().sum(0)
    for i, (want, scale) in enumerate(((yd.sum(0), yd.abs().sum(0)), ((yd * sd).sum(0), (yd * sd).abs().sum(0)))):
        err = (got[i] - want).abs()
        bad = err > rtol * scale + 1e-30
        if bad.any():
            c = int(bad.nonzero()[0])
            raise AssertionError(f"{what}: row {i} of the slots differs in {int(bad.sum())} channels; first ch {c}: "
                                 f"got {float(got[i, c]):.9g} want {float(want[c]):.9g}")


def conv_nhwc_f64(x, w, k, stride):
    """x (N,H,W,Cin), w (Cout,k,k,Cin), any dtype -> float64 (N*Ho*Wo, Cout) conv and conv of absolute values."""
    xd = x.double().permute(0, 3, 1, 2)
    wd = w.double().permute(0, 3, 1, 2)
    pad = k // 2
    acc = torch.nn.functional.conv2d(xd, wd, stride=stride, padding=pad)
    absacc = torch.nn.functional.conv2d(xd.abs(), wd.abs(), stride=stride, padding=pad)
    C = acc.shape[1]
    return acc.permute(0, 2, 3, 1).reshape(-1, C), absacc.permute(0, 2, 3, 1).reshape(-1, C)


def dgrad_nhwc_f64(dy, w, k, stride):
    """dy (N,Ho,Wo,Cout), w (Cout,k,k,Cin) -> float64 (N*H*W, Cin) conv_transpose and its absolute-value counterpart."""
    dd = dy.double().permute(0, 3, 1, 2)
    wd = w.double().permute(0, 3, 1, 2)
    kw = dict(stride=stride, padding=k // 2, output_padding=stride - 1)
    acc = torch.nn.functional.conv_transpose2d(dd, wd, **kw)
    absacc = torch.nn.functional.conv_transpose2d(dd.abs(), wd.abs(), **kw)
    C = acc.shape[1]
    return acc.permute(0, 2, 3, 1).reshape(-1, C), absacc.permute(0, 2, 3, 1).reshape(-1, C)
