"""Float64 reference, planning mirror and element-wise comparators for the weight-gradient GEMMs (wgrad_kernel,
wgrad_xpose_kernel and wgrad_reduce_kernel in csrc/conv_gemm.cuh / csrc/conv_ops.cu).

Torch only, so that the CPU tests can import it. The kernels compute, for every row co and packed column
j = tap * width + ci of dW,
    dW[co][j] += sum over output pixels p of M[p][co] * A_tap[p][ci]
where M is dy (rows < co_split or every row of a plain launch) or x itself (the stacked rows of [dy | x]^T x and of
the Gram matrix x^T x), and A_tap is the input x seen through filter tap `tap` (zero outside the image). The stem reads
its space-to-depth input through four overlapping 128-byte windows: tap p = s2d row offset p - 2, column block q of
16 channels = s2d column offset q, so dW is [64][256] = [64][p 4][q 4][16].

The reference builds A_tap from padded, shifted views of x tap by tap (no im2col) and sums in chunks of pixels on
whatever device the tensors live on. It also returns A = sum_p |M| |A_tap|, the scale of the rounding bound.

Two comparators:
  exact  small-integer operands whose every partial sum stays below 2^20: fp32 accumulation is then exact in any order
         and the result must equal float64 bit for bit. A mismatch is explained from the planned split decomposition:
         which k-block or split is missing or doubled, which tap's block landed in these columns, which row this is.
  bound  real bf16 operands: |got - ref| <= 2^-23 (L + S + 2) A + 2^-24 |ref|, L = 4 MMA accumulate steps per k-block
         of one split, S = number of splits. It holds whatever rounding the tensor core applies inside one step.
Accumulation: every path adds its sum to dW with one rounding, so a run from a start D must give fl(D + run from 0)
bit for bit (check_accumulated).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

EXACT_LIMIT = 2.0 ** 20     # every partial sum below this is exact in fp32 (24-bit significand, integer operands)
SENTINEL = 1024             # floats (4 KB) on each side of dW
SENTINEL_VALUE = -1.2345678e-3
INFO_KEYS = ("xpose", "n", "stacked", "co_split", "num_taps", "co_tiles", "ci_tiles", "splits", "kblocks", "grid",
             "scratch")
MODES = {"conv": 0, "stacked": 1, "gram": 2}


# ------------------------------------------------------------------------------------------------------------------
# planning mirror (plan_conv_wgrad / plan_conv_wgrad_gram / plan_gram)
# ------------------------------------------------------------------------------------------------------------------
def _shrink(splits: int, kblocks: int) -> int:
    """The planner's "no empty split" loop: lower the count until the last split owns at least one k-block."""
    while splits > 1:
        per = -(-kblocks // splits)
        if per * (splits - 1) < kblocks:
            break
        splits -= 1
    return splits


def plan(mode: str, shape, sms: int) -> dict:
    """What launch_wgrad runs for `shape` = (N, H, W, Cin, Cout, k, stride, kind) on `sms` SMs. The first eleven keys are
    the fields of argus_conv2d_wgrad_launch_info; the rest describe the decomposition (rows of dW, packed width, width
    of one tap's columns, pixels, k-blocks per split, the split count before the k-block cap and before the shrink)."""
    N, H, W, Cin, Cout, k, stride, kind = shape
    if mode == "stacked":
        rows, co_split, stacked, k, kind = Cout + Cin, Cout, 1, 1, 0
    elif mode == "gram":
        rows, co_split, stacked, k, kind = Cin, 0, 1, 1, 0
    else:
        rows, co_split, stacked = Cout, 0, 0
    pixels = N * (H // stride) * (W // stride)
    ext = 64 if kind == 1 else Cin
    bn = next((b for b in (256, 128, 64) if ext >= b and ext % b == 0), 64)
    taps = 4 if kind == 1 else k * k
    ktot = 256 if kind == 1 else k * k * Cin
    co_tiles, ci_tiles, kblocks = -(-rows // 128), -(-ext // bn), -(-pixels // 64)
    base = co_tiles * ci_tiles * taps
    uncapped = max(1, sms // base)
    capped = min(uncapped, max(1, kblocks // 4))
    splits = _shrink(capped, kblocks)
    xpose = mode == "conv" and rows == 64 and (kind == 1 or (k == 3 and Cin == 64))
    if xpose:
        n = 4 if taps * (ext // 64) <= 4 else 10
        uncapped = sms
        capped = max(1, min(sms, kblocks // 4))
        splits = _shrink(capped, kblocks)
        grid, scratch = splits, splits * 64 * ktot
    else:
        n = bn
        grid = min(base * splits, sms)
        scratch = 0 if splits <= 1 else splits * rows * ktot
    per = -(-kblocks // splits)
    return dict(xpose=int(xpose), n=n, stacked=stacked, co_split=co_split, num_taps=taps, co_tiles=co_tiles,
                ci_tiles=ci_tiles, splits=splits, kblocks=kblocks, grid=grid, scratch=scratch,
                rows=rows, ktot=ktot, width=64 if kind == 1 else Cin, pixels=pixels, per=per,
                uncapped=uncapped, capped=capped, kind=kind, k=k, stride=stride)


def info_tuple(p: dict) -> tuple:
    return tuple(p[key] for key in INFO_KEYS)


def split_of(kb: int, p: dict) -> int:
    return kb // p["per"]


def where(co: int, col: int, p: dict) -> str:
    """(co, tap, ci) of a packed element, with its co tile and ci tile (or box) as the kernel tiles the work."""
    if p["kind"] == 1:
        tap, ci = divmod(col, 64)
        s = f"co {co}, tap {tap} (s2d row offset {tap - 2}), slot {ci} (column block {ci // 16}, channel {ci % 16})"
    else:
        tap, ci = divmod(col, p["width"])
        s = f"co {co}, tap {tap}, ci {ci}"
    if p["xpose"]:
        return s + f" [transposed kernel: box {col // 64}]"
    return s + f" [co tile {co // 128}, ci tile {ci // p['n']}]"


# ------------------------------------------------------------------------------------------------------------------
# operands and float64 reference
# ------------------------------------------------------------------------------------------------------------------
class Problem:
    """One weight-gradient launch: dy (N, Ho, Wo, Cout) or (P, Cout) bf16, x (N, H, W, Cin) bf16 (the stem: the s2d
    input (N, H/2, W/2 + 4, 16)), mode conv / stacked / gram."""

    def __init__(self, mode: str, shape, dy, x):
        self.mode, self.shape = mode, tuple(shape)
        N, H, W, Cin, Cout, k, stride, kind = shape
        if mode != "conv":
            k, kind = 1, 0
        self.k, self.stride, self.kind = k, stride, kind
        self.N, self.Ho, self.Wo = N, H // stride, W // stride
        self.dy = None if dy is None else dy.reshape(N, self.Ho, self.Wo, -1)
        self.x = x
        self.taps = self._tap_views()
        self.ktot = 256 if kind == 1 else k * k * Cin

    def _tap_views(self):
        """[(column offset, (N, Ho, Wo, width) view of x)] in the kernel's tap order."""
        x, Ho, Wo = self.x, self.Ho, self.Wo
        if self.kind == 1:
            xp = F.pad(x, (0, 0, 0, 0, 2, 1))           # s2d rows i + p - 2 for p = 0..3, zero outside
            return [(p * 64 + q * 16, xp[:, p:p + Ho, q:q + Wo, :]) for p in range(4) for q in range(4)]
        k, s, pad = self.k, self.stride, self.k // 2
        xp = F.pad(x, (0, 0, pad, pad, pad, pad)) if pad else x
        C = x.shape[-1]
        return [((kh * k + kw) * C, xp[:, kh:kh + s * Ho:s, kw:kw + s * Wo:s, :]) for kh in range(k) for kw in range(k)]

    def m_parts(self):
        """(N, Ho, Wo, .) pieces of the M operand, concatenated along channels: dy, [dy | x_s], or x_s."""
        xs = self.x[:, ::self.stride, ::self.stride, :] if self.mode != "conv" else None
        return {"conv": [self.dy], "stacked": [self.dy, xs], "gram": [xs]}[self.mode]

    def chunks(self, pixels: int = 1 << 16):
        """(first pixel, M chunk [pc, rows], [(column offset, A_tap chunk [pc, width])]) in float64."""
        per = max(1, pixels // (self.Ho * self.Wo))
        for n0 in range(0, self.N, per):
            n1 = min(self.N, n0 + per)
            m = torch.cat([t[n0:n1].reshape(-1, t.shape[-1]).double() for t in self.m_parts()], 1)
            yield n0 * self.Ho * self.Wo, m, [(off, v[n0:n1].reshape(-1, v.shape[-1]).double()) for off, v in self.taps]

    def reference(self, kb0: int = 0, kb1: int | None = None):
        """(ref, A): float64 [rows][ktot] of sum_p M^T A_tap in the packed layout, and of |M|^T |A_tap|, over the pixels
        of k-blocks kb0 .. kb1 - 1 (default: all)."""
        lo, hi = kb0 * 64, (1 << 62) if kb1 is None else kb1 * 64
        ref = A = None
        for first, m, taps in self.chunks():
            if ref is None:
                ref = torch.zeros(m.shape[1], self.ktot, dtype=torch.float64, device=m.device)
                A = torch.zeros_like(ref)
            r0, r1 = max(lo - first, 0), min(hi - first, m.shape[0])
            if r0 >= r1:
                continue
            m = m[r0:r1]
            ma = m.abs()
            for off, a in taps:
                a = a[r0:r1]
                ref[:, off:off + a.shape[1]] += m.t() @ a
                A[:, off:off + a.shape[1]] += ma.t() @ a.abs()
        return ref, A

    def split_sums(self, p: dict):
        """The planned split-K decomposition in float64: the sum of every split (k-blocks ks * per .. (ks + 1) * per - 1)."""
        return [self.reference(ks * p["per"], min((ks + 1) * p["per"], p["kblocks"]))[0] for ks in range(p["splits"])]

    def kblock_terms(self, co: int, col: int) -> torch.Tensor:
        """float64 contribution of every 64-pixel k-block to element (co, col)."""
        tap_off, a_col = None, None
        for off, v in self.taps:
            if off <= col < off + v.shape[-1]:
                tap_off, a_col = off, col - off
        assert tap_off is not None, "column outside every tap"
        terms = []
        for _, m, taps in self.chunks():
            a = dict(taps)[tap_off]
            terms.append(m[:, co] * a[:, a_col])
        t = torch.cat(terms)
        t = F.pad(t, (0, (-t.numel()) % 64))
        return t.view(-1, 64).sum(1)


def stem_mask(device=None) -> torch.Tensor:
    """[64][256] bool: the packed stem slots that alias a real filter tap (kh = 2p + a - 1, kw = 2q + b - 1 inside the
    7x7 filter, channel (2a + b) * 3 + c of the three image channels). The others hold sums the forward never uses."""
    m = torch.zeros(4, 4, 16, dtype=torch.bool, device=device)
    for p in range(4):
        for q in range(4):
            for a in range(2):
                for b in range(2):
                    if 0 <= 2 * p + a - 1 < 7 and 0 <= 2 * q + b - 1 < 7:
                        m[p, q, (a * 2 + b) * 3:(a * 2 + b) * 3 + 3] = True
    return m.reshape(1, 256).expand(64, 256)


# ------------------------------------------------------------------------------------------------------------------
# comparators
# ------------------------------------------------------------------------------------------------------------------
class WgradMismatch(AssertionError):
    pass


def bound(ref: torch.Tensor, A: torch.Tensor, p: dict) -> torch.Tensor:
    L = 4 * p["per"]
    return 2.0 ** -23 * (L + p["splits"] + 2) * A + 2.0 ** -24 * ref.abs()


def _explain(prob: Problem, got: torch.Tensor, ref: torch.Tensor, co: int, col: int, p: dict) -> str:
    g, r = float(got[co, col]), float(ref[co, col])
    if g != g:
        return "NaN (stale split-K scratch or an unwritten element)"
    d = g - r
    notes = []
    width = 64 if p["kind"] == 1 else p["width"]
    terms = prob.kblock_terms(co, col)
    last = p["kblocks"] - 1
    ragged = " (the ragged last k-block)" if p["pixels"] % 64 else ""
    for sign, what in ((-1, "missing"), (1, "counted twice")):
        hits = torch.nonzero(terms == sign * d).flatten().tolist()
        if hits and d != 0:
            names = ", ".join(f"k-block {kb} (split {split_of(kb, p)}){ragged if kb == last else ''}" for kb in hits[:4])
            notes.append(f"{names} {what}" + (f" ({len(hits)} k-blocks match)" if len(hits) > 1 else ""))
        per = p["per"]
        sums = F.pad(terms, (0, (-terms.numel()) % per)).view(-1, per).sum(1)
        hits = torch.nonzero(sums == sign * d).flatten().tolist()
        if hits and d != 0:
            notes.append(f"split {hits[0]} (k-blocks {hits[0] * per}..{min((hits[0] + 1) * per, p['kblocks']) - 1}) "
                         + ("missing" if sign < 0 else "added twice"))
    if col >= width:
        prev = float(ref[co, col - width])
        if g == prev:
            notes.append("holds the previous tap's value: a tap's block was written into the next tap's columns")
        elif g == r + prev:
            notes.append("the previous tap's block was added into this tap's columns")
    rows = [i for i in torch.nonzero(ref[:, col] == g).flatten().tolist() if i != co]
    same_row = [i for i in rows[:8] if torch.equal(got[co].double(), ref[i])]
    if same_row:
        notes.append(f"the whole row equals the reference of row {same_row[0]}: rows swapped")
    if g == 0 and r != 0:
        notes.append("zero: never written")
    return "; ".join(notes) if notes else "no single k-block, split, tap or row explains the difference"


def _fail(prob, got, ref, bad, p, what, extra):
    idx = torch.nonzero(bad)
    lines = []
    for co, col in idx[:3].tolist():
        lines.append(f"  {where(co, col, p)}: got {float(got[co, col])!r}, want {float(ref[co, col])!r}{extra(co, col)}"
                     f" -- {_explain(prob, got, ref, co, col, p)}")
    raise WgradMismatch(f"{what}: {idx.shape[0]} of {bad.numel()} elements wrong\n" + "\n".join(lines))


def check_exact(prob: Problem, got: torch.Tensor, ref: torch.Tensor, A: torch.Tensor, p: dict, what: str = "") -> None:
    """got [rows][ktot] fp32 from dW = 0 must equal the float64 reference bit for bit."""
    if float(A.max()) >= EXACT_LIMIT:
        raise ValueError(f"{what}: operands not exact (sum |M||A| reaches {float(A.max())})")
    bad = ~(got.double() == ref)
    if bool(bad.any()):
        _fail(prob, got, ref, bad, p, what + " (exact)", lambda co, col: "")


def check_bound(prob: Problem, got: torch.Tensor, ref: torch.Tensor, A: torch.Tensor, p: dict, what: str = "") -> float:
    """got [rows][ktot] fp32 from dW = 0 against the rounding bound; returns the largest err / bound."""
    b = bound(ref, A, p)
    err = (got.double() - ref).abs()
    bad = ~(err <= b)
    if bool(bad.any()):
        _fail(prob, got, ref, bad, p, what + " (rounding bound)",
              lambda co, col: f", err/bound {float(err[co, col] / b[co, col]):.3g}")
    return float((err / b.clamp_min(1e-300)).max())


def check_sentinels(buf: torch.Tensor, n: int, p: dict, what: str = "") -> None:
    """buf = [SENTINEL | dW (n floats) | SENTINEL]: both guards must still hold SENTINEL_VALUE bit for bit. A write
    past dW is named as the (row >= rows, column) it would be."""
    want = torch.tensor(SENTINEL_VALUE, dtype=torch.float32).view(torch.int32).item()
    b = buf.view(torch.int32)
    pre = torch.nonzero(b[:SENTINEL] != want).flatten().tolist()
    post = torch.nonzero(b[SENTINEL + n:] != want).flatten().tolist()
    msgs = []
    if pre:
        msgs.append(f"{len(pre)} words before dW written (first at -{SENTINEL - pre[0]})")
    if post:
        co, col = divmod(n + post[0], p["ktot"])
        msgs.append(f"{len(post)} words past dW written: first is row {co} (>= {p['rows']} rows), column {col}, "
                    f"value {float(buf[SENTINEL + n + post[0]])!r}")
    if msgs:
        raise WgradMismatch(f"{what}: " + "; ".join(msgs))


def check_accumulated(got: torch.Tensor, start: torch.Tensor, from_zero: torch.Tensor, p: dict, what: str = "") -> None:
    """A run from dW = start must equal fl(start + run from 0) bit for bit (one fp32 rounding per element)."""
    want = start + from_zero
    bad = got.view(torch.int32) != want.view(torch.int32)
    if bool(bad.any()):
        idx = torch.nonzero(bad)
        co, col = idx[0].tolist()
        raise WgradMismatch(f"{what}: {idx.shape[0]} elements differ from fl(D + result from 0), first "
                            f"{where(co, col, p)}: got {float(got[co, col])!r}, D {float(start[co, col])!r}, "
                            f"from 0 {float(from_zero[co, col])!r}, want {float(want[co, col])!r}")


# ------------------------------------------------------------------------------------------------------------------
# operands
# ------------------------------------------------------------------------------------------------------------------
def _ints(shape, lo, hi, density, gen, device):
    v = torch.randint(lo, hi + 1, shape, generator=gen, device=device, dtype=torch.int8)
    keep = torch.rand(shape, generator=gen, device=device) < density
    return (v * keep).to(torch.bfloat16)


def input_shape(shape):
    N, H, W, Cin, Cout, k, stride, kind = shape
    return (N, H // 2, W // 2 + 4, 16) if kind == 1 else (N, H, W, Cin)


def make_operands(mode: str, shape, exact: bool, gen, device):
    """(dy, x) bf16. exact: dy in {-1, 0, 1} and x in {-2..2}, sparse enough on long K that every sum stays far below
    2^20; otherwise real values with post-ReLU (nonnegative) x and dy offset from zero, so that the sums do not cancel.
    The stem input has zero s2d padding columns as the packing kernel writes it; its four spare channels are filled too."""
    N, H, W, Cin, Cout, k, stride, kind = shape
    Ho, Wo = H // stride, W // stride
    xshape, dyshape = input_shape(shape), (N, Ho, Wo, Cout)
    dens = min(0.5, 2.0 ** 15 / (N * Ho * Wo))
    if exact:
        x = _ints(xshape, -2, 2, dens, gen, device)
        dy = _ints(dyshape, -1, 1, dens, gen, device) if mode != "gram" else None
    else:
        x = torch.randn(xshape, generator=gen, device=device).relu().to(torch.bfloat16)
        dy = (torch.randn(dyshape, generator=gen, device=device) * 0.5 + 0.25).to(torch.bfloat16) \
            if mode != "gram" else None
    if kind == 1:
        x[:, :, :2] = 0
        x[:, :, 2 + W // 2:] = 0
    return dy, x
