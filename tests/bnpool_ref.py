"""Float64 references and element-wise comparators for the batch-norm and pooling passes (csrc/elementwise.cu).

Torch only, so that the CPU tests can import it. Each reference runs the kernel's own sequence of steps in float64 on
the same bf16 / fp32 operands, and each check asserts every element: there is no allowed fraction of mismatches, and a
NaN (an unwritten sentinel) fails. Rows are the (rows, C) view of an NHWC tensor; the batch-norm passes stream it as
16-byte vectors of eight channels, vector i = row * C / 8 + channel / 8, in ring stages of 512 vectors (stage i // 512;
the vectors past the last full stage are the ragged tail that block 0 runs from global memory). Failures name the row,
the channel, the stage and the tail position.

Bounds (u = 2^-24, one fp32 rounding):
  apply      |y - ref| <= 2^-8 |ref| + 2^-22 (|x sc| + |sh| + |residual term|)
  sums       |got - ref| <= K_SUM u sum|term|   (per-thread fp32 sums, then a fixed-order block reduction)
  bn dx      2^-8 |ref| + 2^-22 (|sc| g_abs + |k1 x| + |c2 mean| + |sc sum g / M|) + the sums' bounds carried through
             k0 / k1 (c2 = -k1; k0 = c2 mean - sc sum g / M is formed from those two terms)
  finalize   two fp32 ulps, plus the float64 reordering bound of the variance where the mean is far from zero
             (scale and shift also carry the one-ulp rounding of invstd and of scale they are formed from)
2^-8 |ref| is one bf16 rounding (half an ulp at the bottom of a binade, twice over). K_SUM is calibrated on a B200
(largest observed error / bound in the PR description).
"""
from __future__ import annotations

import torch

REL = 2.0 ** -8
C_ADD = 2.0 ** -22
U32 = 2.0 ** -24
U64 = 2.0 ** -53
K_SUM = 32.0       # backward dgamma / dbeta and apply column sums, in units of u * sum|term|
RING_VEC = 512     # vectors per ring stage


def bits_to_bool(bits: torch.Tensor, channels: int) -> torch.Tensor:
    """[rows][channels/8] uint8 mask -> [rows][channels] bool (channel c = byte c // 8, bit c % 8)."""
    b = bits.reshape(-1, channels // 8).to(torch.int32)
    shifts = torch.arange(8, device=b.device, dtype=torch.int32)
    return ((b.unsqueeze(-1) >> shifts) & 1).reshape(-1, channels).bool()


def bool_to_bits(mask: torch.Tensor) -> torch.Tensor:
    rows, channels = mask.shape
    m = mask.reshape(rows, channels // 8, 8).to(torch.int32)
    return (m * (1 << torch.arange(8, device=m.device, dtype=torch.int32))).sum(-1).to(torch.uint8)


def ring_geometry(rows: int, C: int, sms: int) -> dict:
    """Launch geometry of the ring passes: grid = min(nvec / 512, 2 x SMs) (at least 1), full stages, tail."""
    nvec = rows * (C // 8)
    nfull = nvec // RING_VEC
    grid = max(1, min(nfull, 2 * sms))
    return dict(nvec=nvec, grid=grid, nfull=nfull, stages_per_cta=nfull / grid, tail=nvec - nfull * RING_VEC)


def where(flat: int, C: int, nvec: int | None = None) -> str:
    r, c = divmod(flat, C)
    v = r * (C // 8) + c // 8
    s = f"row {r} ch {c} (vector {v}, ring stage {v // RING_VEC}"
    if nvec is not None and v >= nvec // RING_VEC * RING_VEC:
        s += f", tail position {v - nvec // RING_VEC * RING_VEC}"
    return s + ")"


def _fail(what, bad, C, nvec, lines, limit=6):
    idx = bad.flatten().nonzero().flatten()
    out = [f"{what}: {idx.numel()} of {bad.numel()} elements wrong"]
    for flat in idx[:limit].tolist():
        out.append("  " + where(flat, C, nvec) + ": " + lines(flat))
    raise AssertionError("\n".join(out))


def check_close(got, ref, bound, what, nvec=None):
    """Every element of got within bound of ref (float64 [rows][C] each). NaN fails. Returns max |err| / bound."""
    C = ref.shape[-1]
    ref = ref.reshape(-1, C)
    bound = bound.reshape(-1, C)
    g = got.double().reshape(-1, C)
    err = (g - ref).abs()
    bad = ~(err <= bound)
    if bad.any():
        gf, rf, bf = g.flatten(), ref.flatten(), bound.flatten()
        _fail(what, bad, C, nvec, lambda i: f"got {gf[i]:.8g} ref {rf[i]:.8g} bound {bf[i]:.3g}")
    pos = bound > 0
    return float((err[pos] / bound[pos]).max()) if pos.any() else 0.0


def check_equal(got, want, what, nvec=None):
    """Exact equality (value for value, NaN fails)."""
    C = want.shape[-1]
    g, w = got.reshape(-1, C), want.reshape(-1, C)
    bad = ~(g == w)
    if bad.any():
        gf, wf = g.flatten(), w.flatten()
        _fail(what, bad, C, nvec, lambda i: f"got {gf[i].item()} want {wf[i].item()}")


# ---------------------------------------------------------------------------------------------------- apply
def apply_ref(x, scale, shift, res=None, rscale=None, rshift=None, relu=True):
    """pre = x sc + sh [+ res | + res rs + rb]; ref = [relu](pre). Returns (pre, ref, E) in float64."""
    xs = x.double() * scale.double()
    pre = xs + shift.double()
    e = xs.abs() + shift.double().abs()
    if res is not None:
        r = res.double()
        if rscale is not None:
            r = r * rscale.double()
            e = e + r.abs() + rshift.double().abs()
            r = r + rshift.double()
        else:
            e = e + r.abs()
        pre = pre + r
    return pre, (pre.clamp_min(0.0) if relu else pre), C_ADD * e


def check_apply(y, pre, ref, E, what="bn_apply y"):
    """y within 2^-8 |ref| + E. Returns the largest error / bound."""
    nvec = ref.numel() // 8
    return check_close(y, ref, REL * ref.abs() + E, what, nvec)


def check_bits(bits, y, pre, E, what="ReLU bits"):
    """bits == (stored y > 0) exactly, and == (pre > 0) wherever |pre| exceeds the apply bound."""
    C = pre.shape[-1]
    nvec = pre.numel() // 8
    b = bits_to_bool(bits, C)
    yp = y.double().reshape(-1, C) > 0
    bad = b != yp
    if bad.any():
        bf, yf = b.flatten(), y.reshape(-1).double()
        _fail(what + " vs y > 0", bad, C, nvec, lambda i: f"bit {int(bf[i])} y {float(yf[i]):.6g}")
    decided = pre.abs() > E + REL * pre.abs()
    bad = decided & (b != (pre > 0))
    if bad.any():
        bf, pf = b.flatten(), pre.flatten()
        _fail(what + " vs sign(pre)", bad, C, nvec, lambda i: f"bit {int(bf[i])} pre {float(pf[i]):.6g}")


def check_colsum(partial, y, k=K_SUM, what="column sums"):
    """partial [blocks][C]: the float64 sum over the blocks equals the float64 column sum of the STORED y within
    k u sum|y|. Returns the largest error / bound."""
    C = partial.shape[-1]
    yd = y.double().reshape(-1, C)
    got = partial.double().reshape(-1, C).sum(0)
    want, scale = yd.sum(0), yd.abs().sum(0)
    bound = k * U32 * scale
    err = (got - want).abs()
    bad = ~(err <= bound)
    if bad.any():
        c = int(bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} channels wrong; first ch {c}: got {float(got[c]):.9g} "
                             f"want {float(want[c]):.9g} bound {float(bound[c]):.3g}")
    pos = bound > 0
    return float((err[pos] / bound[pos]).max()) if pos.any() else 0.0


# ---------------------------------------------------------------------------------------------------- finalize
def ulp32(v: torch.Tensor) -> torch.Tensor:
    """fp32 ulp of |v| (float64 in, float64 out); the smallest normal's ulp below it."""
    a = v.double().abs().clamp_min(2.0 ** -126)
    return torch.exp2(torch.floor(torch.log2(a)) - 23)


def finalize_ref(partial, count, gamma, beta, eps, momentum=None, running_mean=None, running_var=None):
    """partial [slots][2][C] fp32 (sum x, sum x^2). Returns a dict of float64 references and bounds: the reference
    mean / invstd / scale / shift / running statistics, the summation-order bound `var_err` of the float64 variance
    (what cancellation between E[x^2] and mean^2 makes of two reorderings of the same sums), and `cond`, how much
    larger E[x^2] is than the variance."""
    p = partial.double()
    slots = p.shape[0]
    eps = float(torch.tensor(eps, dtype=torch.float32))      # the kernel takes eps as an fp32 argument
    s0, s1 = p[:, 0].sum(0), p[:, 1].sum(0)
    a0, a1 = p[:, 0].abs().sum(0), p[:, 1].abs().sum(0)
    mean = s0 / count
    var_raw = s1 / count - mean * mean
    var = var_raw.clamp_min(0.0)
    # both sums are float64 over the same fp32 numbers in another order: each is off by at most 2 (slots + 32) u64 sum|p|
    g = 2 * (slots + 32) * U64
    var_err = g * a1 / count + 2 * mean.abs() * g * a0 / count + 4 * U64 * (s1.abs() / count + mean * mean)
    invstd = 1.0 / torch.sqrt(var + eps)
    r = dict(mean=mean, var=var, var_err=var_err, invstd=invstd, cond=(s1 / count) / var.clamp_min(1e-300),
             mean_err=g * a0 / count)
    inv32 = invstd.float().double()
    r["gamma_abs"] = gamma.double().abs()
    r["scale"] = gamma.double() * inv32
    r["shift"] = beta.double() - mean.float().double() * r["scale"]
    r["shift_mag"] = beta.double().abs() + (mean * r["scale"]).abs()
    if running_mean is not None:
        unbiased = var * count / (count - 1) if count > 1 else var
        r["running_mean"] = (1 - momentum) * running_mean.double() + momentum * mean
        r["running_var"] = (1 - momentum) * running_var.double() + momentum * unbiased
        r["rm_mag"] = ((1 - momentum) * running_mean.double()).abs() + (momentum * mean).abs()
        r["rv_mag"] = ((1 - momentum) * running_var.double()).abs() + (momentum * unbiased).abs()
        r["unbiased_err"] = var_err * (count / (count - 1) if count > 1 else 1.0)
    return r


def check_finalize(out: dict, ref: dict, eps, ulps=2.0) -> dict:
    """out: the kernel's mean, invstd, scale, shift (+ running_mean, running_var). Each within `ulps` fp32 ulps of its
    magnitude, plus what the float64 reordering of the sums can move it (ref['var_err'] carried through). Returns the
    largest error / bound per quantity."""
    d_invstd = 0.5 * ref["invstd"] ** 3 * ref["var_err"]          # |d invstd / d var| * var_err
    # scale = fp32(gamma * invstd32): its own rounding, plus one ulp of invstd carried (an ulp of invstd can be 1.9
    # ulps of scale when the two lie in different binades); shift = beta - mean32 * scale carries the scale's bound
    scale_bound = (ulps * ulp32(ref["scale"]) + ref["gamma_abs"] * ulp32(ref["invstd"])
                   + ref["scale"].abs() / ref["invstd"] * d_invstd)
    checks = {
        "mean": (ref["mean"], ulps * ulp32(ref["mean"]) + ref["mean_err"]),
        "invstd": (ref["invstd"], ulps * ulp32(ref["invstd"]) + d_invstd),
        "scale": (ref["scale"], scale_bound),
        "shift": (ref["shift"], ulps * ulp32(ref["shift_mag"]) + ref["mean"].abs() * scale_bound
                  + ref["scale"].abs() * ref["mean_err"]),
    }
    if "running_mean" in out:
        checks["running_mean"] = (ref["running_mean"], ulps * ulp32(ref["rm_mag"]) + ref["mean_err"])
        checks["running_var"] = (ref["running_var"], ulps * ulp32(ref["rv_mag"]) + ref["unbiased_err"])
    ratios = {}
    for name, (want, bound) in checks.items():
        got = out[name].double()
        err = (got - want).abs()
        bad = ~(err <= bound)
        if bad.any():
            c = int(bad.nonzero()[0])
            raise AssertionError(f"finalize {name}: {int(bad.sum())} channels wrong; first ch {c}: got {float(got[c]):.9g} "
                                 f"want {float(want[c]):.9g} bound {float(bound[c]):.3g} (E[x^2]/var "
                                 f"{float(ref['cond'][c]):.3g})")
        ratios[name] = float((err / bound).max())
    return ratios


# ---------------------------------------------------------------------------------------------------- backward
def bn_mask(mode, dy, x, out, scale, shift):
    """The kernel's g: mode 0 dy; 1 dy where fmaf(x, sc, sh) > 0; 2 dy where out > 0; 3 dy where the bit is set.
    Mode 1 is decided in float64: a bf16 x times an fp32 sc is exact there (8 + 24 bits), and rounding x sc + sh never
    changes its sign, so this is the sign fmaf sees: no element can lie within rounding of the decision."""
    C = x.shape[-1]
    d = dy.double().reshape(-1, C)
    if mode == 0:
        return d
    if mode == 1:
        keep = x.double().reshape(-1, C) * scale.double() + shift.double() > 0
    elif mode == 2:
        keep = out.double().reshape(-1, C) > 0
    else:
        keep = bits_to_bool(out, C)
    return torch.where(keep, d, torch.zeros_like(d))


def bn_backward_ref(g, x, scale, mean, invstd, g_abs=None, k=K_SUM):
    """g float64 [rows][C] (the masked gradient), x the bf16 layer output, per-channel fp32 vectors.
    Returns dict(dbeta, dgamma, db_bound, dg_bound, dx, dx_bound). g_abs: per-element sum of |contributions| to g when
    the kernel forms g from several terms (the stem's un-pooling); |g| otherwise."""
    C = g.shape[-1]
    xd = x.double().reshape(-1, C)
    M = xd.shape[0]
    mu, is_, sc = mean.double(), invstd.double(), scale.double()
    ga = g.abs() if g_abs is None else g_abs
    dbeta = g.sum(0)
    dgamma = (g * (xd - mu)).sum(0) * is_
    # the kernel sums g and g x in fp32 and centres once per thread: (sum g x - mu sum g) is
    db_bound = k * U32 * ga.sum(0)
    dg_bound = k * U32 * ((ga * xd.abs()).sum(0) + mu.abs() * ga.sum(0)) * is_
    c2 = sc * dgamma * is_ / M
    k1 = -c2
    kb = sc * dbeta / M
    dx = sc * g + k1 * xd + (c2 * mu - kb)
    e = (sc.abs() * ga + (k1 * xd).abs() + (c2 * mu).abs() + kb.abs())
    carried = (sc * is_).abs() / M * (xd - mu).abs() * is_ * dg_bound + sc.abs() / M * db_bound
    dx_bound = REL * dx.abs() + C_ADD * e + carried
    return dict(dbeta=dbeta, dgamma=dgamma, db_bound=db_bound, dg_bound=dg_bound, dx=dx, dx_bound=dx_bound)


def check_sums(got, want, bound, what):
    err = (got.double() - want).abs()
    bad = ~(err <= bound)
    if bad.any():
        c = int(bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} channels wrong; first ch {c}: got {float(got[c]):.9g} "
                             f"want {float(want[c]):.9g} bound {float(bound[c]):.3g}")
    pos = bound > 0
    return float((err[pos] / bound[pos]).max()) if pos.any() else 0.0


def check_bn_backward(dgamma, dbeta, dx, ref, what="bn backward"):
    """dgamma / dbeta (this call's sums) and dx against bn_backward_ref. Returns the largest error / bound of each."""
    return dict(dbeta=check_sums(dbeta, ref["dbeta"], ref["db_bound"], what + " dbeta"),
                dgamma=check_sums(dgamma, ref["dgamma"], ref["dg_bound"], what + " dgamma"),
                dx=check_close(dx, ref["dx"], ref["dx_bound"], what + " dx", ref["dx"].numel() // 8))


# ---------------------------------------------------------------------------------------------------- pooling
def pool_windows(t, fill):
    """t (N, H, W, C) -> (N, H/2, W/2, C, 9) taps of the 3x3 / stride 2 / pad 1 windows (tap kh * 3 + kw), with
    `fill` at the padded (out-of-bounds) taps, and the matching in-bounds mask."""
    N, H, W, C = t.shape
    tp = torch.full((N, H + 1, W + 1, C), fill, dtype=t.dtype, device=t.device)
    tp[:, 1:, 1:] = t
    ok = torch.zeros(H + 1, W + 1, dtype=torch.bool, device=t.device)
    ok[1:, 1:] = True
    taps, oks = [], []
    for kh in range(3):
        for kw in range(3):
            taps.append(tp[:, kh:kh + H - 1:2, kw:kw + W - 1:2])
            oks.append(ok[kh:kh + H - 1:2, kw:kw + W - 1:2])
    okt = torch.stack(oks, -1)[None, :, :, None, :].expand(N, H // 2, W // 2, C, 9)
    return torch.stack(taps, -1), okt


def check_maxpool_forward(x, scale, shift, y, idx, what="maxpool"):
    """x (N, H, W, C) bf16; scale / shift fp32 [C] or None; y, idx the kernel's outputs (idx may be None).
    idx: every byte in 0..8, naming an in-bounds tap whose raw value is the window extremum of sign(sc) x (exactly);
    where that extremum is unique, the first maximum. y: relu(fma(x_tap, sc, sh)) within the apply bound, or with
    scale None the window maximum exactly. Returns the largest error / bound of y."""
    N, H, W, C = x.shape
    sgn = torch.ones(C, dtype=torch.float64, device=x.device)
    if scale is not None:
        sgn = torch.where(scale < 0, -1.0, 1.0).double()
    taps, ok = pool_windows(x.double(), 0.0)
    key = torch.where(ok, taps * sgn[:, None], torch.tensor(float("-inf"), dtype=torch.float64, device=x.device))
    best, first = key.max(-1)               # torch returns the first maximal index
    n_best = (key == best[..., None]).sum(-1)
    flat = lambda t: t.reshape(-1, C)
    if idx is not None:
        ii = idx.long()
        bad = (ii < 0) | (ii > 8)
        if bad.any():
            _fail(what + " idx out of 0..8", flat(bad), C, None, lambda i: f"idx {int(ii.flatten()[i])}")
        tap_ok = ok.gather(-1, ii[..., None])[..., 0]
        if (~tap_ok).any():
            _fail(what + " idx names an out-of-bounds tap", flat(~tap_ok), C, None,
                  lambda i: f"idx {int(ii.flatten()[i])}")
        picked = key.gather(-1, ii[..., None])[..., 0]
        bad = ~(picked == best)
        if bad.any():
            pf, bf = picked.flatten(), best.flatten()
            _fail(what + " idx names a non-maximal tap", flat(bad), C, None,
                  lambda i: f"idx {int(ii.flatten()[i])} value {float(pf[i])} max {float(bf[i])}")
        bad = (n_best == 1) & (ii != first)
        if bad.any():
            _fail(what + " idx is not the unique maximum", flat(bad), C, None,
                  lambda i: f"idx {int(ii.flatten()[i])} first max {int(first.flatten()[i])}")
    xmax = best * sgn                          # the raw value of the extremal tap
    if scale is None:
        check_equal(y.double().reshape(-1, C), flat(xmax), what + " y (no scale)")
        return 0.0
    pre, ref, E = apply_ref(xmax, scale, shift)
    return check_close(y, flat(ref), flat(REL * ref.abs() + E), what + " y")


def unpool_ref(dy, idx, H, W):
    """Float64 scatter of dy (N, H/2, W/2, C) through the arg-max bytes: (dx, sum|contributions|), (N, H, W, C)."""
    N, Ho, Wo, C = dy.shape
    dev = dy.device
    ii = idx.long()
    hh = (2 * torch.arange(Ho, device=dev) - 1)[None, :, None, None] + ii // 3
    ww = (2 * torch.arange(Wo, device=dev) - 1)[None, None, :, None] + ii % 3
    nn_ = torch.arange(N, device=dev)[:, None, None, None].expand_as(ii)
    cc = torch.arange(C, device=dev)[None, None, None, :].expand_as(ii)
    hh, ww = hh.clamp(0, H - 1), ww.clamp(0, W - 1)   # the checked forward never names a padded tap
    d = dy.double()
    dx = torch.zeros(N, H, W, C, dtype=torch.float64, device=dev)
    dabs = torch.zeros_like(dx)
    dx.index_put_((nn_, hh, ww, cc), d, accumulate=True)
    dabs.index_put_((nn_, hh, ww, cc), d.abs(), accumulate=True)
    return dx, dabs


def check_maxpool_backward(dx, dy, idx, what="maxpool backward"):
    N, Ho, Wo, C = dy.shape
    ref, dabs = unpool_ref(dy, idx, 2 * Ho, 2 * Wo)
    return check_close(dx, ref.reshape(-1, C), (REL * ref.abs() + C_ADD * dabs).reshape(-1, C), what)


def check_avgpool_forward(y, x, what="avgpool"):
    """x (N, HW, C) bf16: y within 2^-8 |mean| + HW u mean|x|."""
    xd = x.double()
    HW = x.shape[1]
    ref = xd.mean(1)
    bound = REL * ref.abs() + HW * U32 * xd.abs().mean(1)
    return check_close(y, ref, bound, what)


def avgpool_backward_ref(dy, N, HW, C, bits=None):
    """The kernel's exact arithmetic: bf16(fp32(dy) * fp32(1 / HW)), masked by the bits. (N * HW, C) bf16."""
    inv = torch.tensor(1.0, dtype=torch.float32) / HW
    v = (dy.float().reshape(N, 1, C) * inv.to(dy.device)).expand(N, HW, C).reshape(N * HW, C)
    if bits is not None:
        v = torch.where(bits_to_bool(bits, C), v, torch.zeros_like(v))
    return v.bfloat16()
