"""Float64 reference and element-wise comparators for the algebraic batch-norm backward (csrc/bn_algebra.cu:
bn_alg_coeffs_kernel, bn_alg_matrix_kernel + bn_alg_matrix_reduce_kernel, bn_alg_dw_kernel) and for the way the model
assembles it with the H / Gram GEMMs and the K-concatenated dgrad.

Torch only, so that the CPU tests can import it. With P = rows, inv = fl32(1 / P) (the kernel takes it as a float):
    H = g^T act,  G = act^T act,  s = colsum(act),  db = sum of the statistics slots (column sums of g)
    t = rowdot(W, H),  dgamma = invstd (t - mean db),  c2 = scale dgamma invstd inv
    k1 = -c2,  k0 = c2 mean - scale db inv
    B0 = bf16(fl32(scale W)),  M = W^T diag(k1) W  (stored as bf16),  bias = W^T k0
    dW = diag(scale) H + diag(k1) W G + k0 (x) s,   dAct = g B0 + act M + bias

Stage comparators start from the GPU's own inputs to the stage, so that a failure points at one kernel:
  coeffs   dbeta, dgamma, k1, k0 within 1 fp32 ulp of the float64 value (the kernel works in fp64 on the fp32 H)
  bstack   rows 0..O-1 bit for bit
  matrix   |got - M| <= 2^-8 (|M| + E) + E,  E = 2^-24 (O/8 + 8 + 2) sum_o |W_oj k1_o W_oi|  (o-sum of O/8 terms in one
           of kSplitO = 8 fixed chunks, then the 8 partials in order); the bias likewise, without the bf16 rounding
  dW       |got - ref| <= 2^-24 (C + 4) (|scale H| + |k0 s| + |k1| sum_j |W_oj G_ji|); a run from a start D must give
           fl32(D + run from 0) bit for bit
  dAct     a float64 product of [g | act] with the GPU's B-stack plus the GPU's bias, bounded as tests/epilogue_ref.py
The end-to-end comparator takes only g, act, W, the batch-norm constants and the slots, and composes the stage bounds
with the weight-gradient bound of tests/wgrad_ref.py for H and G.
"""
from __future__ import annotations

import torch

import epilogue_ref as er
import wgrad_ref as wr

U = 2.0 ** -24          # fp32 unit roundoff
K_SPLIT_O = 8           # bn_alg_matrix_kernel's fixed o-chunks
EPS = 1e-5
SENTINEL = 1024         # 4 KB of fp32 on each side of an fp32 output
SENTINEL_F32 = -1.2345678e-3
SENTINEL_BF16 = 0x7FA5  # a NaN pattern no kernel writes; 2048 of them (4 KB) around bf16 outputs


class BnAlgMismatch(AssertionError):
    pass


# ------------------------------------------------------------------------------------------------------------------
# reference
# ------------------------------------------------------------------------------------------------------------------
def ulp32(x: torch.Tensor) -> torch.Tensor:
    """fp32 ulp of fl32(x) (the smallest subnormal for 0)."""
    a = x.double().abs().float().double()
    _, e = torch.frexp(a)
    return torch.ldexp(torch.ones_like(a), e - 24).clamp_min(2.0 ** -149)


def inv_rows32(rows: int) -> float:
    return torch.tensor(1.0 / rows, dtype=torch.float32).item()


def sample(act: torch.Tensor, stride: int) -> torch.Tensor:
    """(N, H, W, C) -> (rows, C): the pixels a stride-`stride` 1x1 convolution reads."""
    return act[:, ::stride, ::stride, :].reshape(-1, act.shape[-1])


def slot_parts(stat: torch.Tensor, slots: int, stride: int, O: int) -> torch.Tensor:
    """[slots][O] float64: slot k's column sums at stat + k * stride."""
    flat = stat.reshape(-1)
    idx = torch.arange(slots, device=stat.device).view(-1, 1) * stride + torch.arange(O, device=stat.device).view(1, -1)
    return flat[idx].double()


def coefficients(W, H, db, scale, mean, invstd, rows, mirror=True):
    """dgamma, k1, k0 in float64 from H and db (mirror: inv = fl32(1 / rows) as the kernel has it)."""
    t = (W.double() * H.double()).sum(1)
    is_, mu, sc = invstd.double(), mean.double(), scale.double()
    inv = inv_rows32(rows) if mirror else 1.0 / rows
    dg = is_ * (t - mu * db)
    c2 = sc * dg * is_ * inv
    return dict(t=t, dgamma=dg, dbeta=db, k1=-c2, k0=c2 * mu - sc * db * inv)


def algebra(g, act, W, scale, mean, invstd, stride, db=None, mirror=True):
    """The whole algebra in float64 from bf16 g (N, Ho, Wo, O) and act (N, H, W, C). db defaults to colsum(g).
    mirror=True applies the roundings the kernels make on purpose (fl32(1/rows), B0 = bf16(fl32(scale W)), M in bf16);
    mirror=False is the exact backward of BatchNorm2d(train) o conv1x1 given mean / invstd / scale."""
    O, C = W.shape
    N, Hh, Ww, _ = act.shape
    gs = g.reshape(-1, O).double()
    a = sample(act, stride).double()
    rows = gs.shape[0]
    Wd = W.double()
    H, G, s = gs.t() @ a, a.t() @ a, a.sum(0)
    if db is None:
        db = gs.sum(0)
    c = coefficients(W, H, db, scale, mean, invstd, rows, mirror)
    sc = scale.double()
    if mirror:
        B0 = (scale.float().view(-1, 1) * W.float()).bfloat16().double()
    else:
        B0 = sc.view(-1, 1) * Wd
    M = Wd.t() @ (c["k1"].view(-1, 1) * Wd)
    Mb = M.float().bfloat16().double() if mirror else M
    bias = Wd.t() @ c["k0"]
    dW = sc.view(-1, 1) * H + c["k1"].view(-1, 1) * (Wd @ G) + c["k0"].view(-1, 1) * s.view(1, -1)
    dact_s = gs @ B0 + a @ Mb + bias
    dact = torch.zeros(N, Hh, Ww, C, dtype=torch.float64, device=g.device)
    dact[:, ::stride, ::stride, :] = dact_s.view(N, Hh // stride, Ww // stride, C)
    return dict(c, H=H, G=G, s=s, B0=B0, M=M, Mb=Mb, bias=bias, dW=dW, dact=dact, dact_s=dact_s, rows=rows)


# ------------------------------------------------------------------------------------------------------------------
# helpers of the comparators
# ------------------------------------------------------------------------------------------------------------------
def _ratio(err, b):
    ok = b > 0
    return float((err[ok] / b[ok]).max()) if bool(ok.any()) else 0.0


def _check(what, got, ref, b, explain, name_of, limit=3):
    got = got.double().reshape(ref.shape)
    err = (got - ref).abs()
    bad = ~(err <= b)      # NaN fails too
    if bool(bad.any()):
        idx = torch.nonzero(bad.reshape(ref.shape) if ref.dim() else bad.view(1))
        lines = []
        for ix in idx[:limit].tolist():
            ix = tuple(ix)
            gv, rv, bv = float(got[ix]), float(ref[ix]), float(b[ix])
            lines.append(f"  {name_of(ix)}: got {gv!r}, want {rv!r}, bound {bv:.3g}"
                         f"{'' if gv != gv else f', err/bound {abs(gv - rv) / max(bv, 1e-300):.3g}'} -- {explain(ix, gv, rv, bv)}")
        raise BnAlgMismatch(f"{what}: {idx.shape[0]} of {ref.numel()} elements out of bound\n" + "\n".join(lines))
    return _ratio(err, b)


def _chunks(O):
    n = O // K_SPLIT_O
    return [(z, z * n, (z + 1) * n) for z in range(K_SPLIT_O)]


def _chunk_note(d, contribs, b, O):
    """The o-chunk whose contribution (float64, per chunk) equals the difference d within b."""
    notes = []
    for sign, what in ((-1.0, "missing"), (1.0, "added twice")):
        diffs = [abs(d - sign * float(v)) for v in contribs]
        z = min(range(len(diffs)), key=diffs.__getitem__)
        if diffs[z] <= b and float(contribs[z]) != 0.0:
            _, lo, hi = _chunks(O)[z]
            notes.append(f"o-chunk {z} (o = {lo}..{hi - 1}) {what}")
    return notes


def _pixel(r, N, Ho, Wo, stride):
    n, rem = divmod(r, Ho * Wo)
    h, w = divmod(rem, Wo)
    return n, h * stride, w * stride


# ------------------------------------------------------------------------------------------------------------------
# stage comparators
# ------------------------------------------------------------------------------------------------------------------
def check_coeffs(W, H, stat, slots, stat_stride, scale, mean, invstd, rows, dgamma, dbeta, k1k0, what=""):
    """bn_alg_coeffs_kernel from dgamma = dbeta = 0: every value within 1 fp32 ulp of float64 on the GPU's H and slots.
    Returns the largest err / bound per quantity."""
    O = W.shape[0]
    parts = slot_parts(stat, slots, stat_stride, O)
    db = parts.sum(0)
    c = coefficients(W, H, db, scale, mean, invstd, rows)
    worst = {}
    for name, got, ref in (("dbeta", dbeta, db), ("dgamma", dgamma, c["dgamma"]), ("k1", k1k0[:O], c["k1"]),
                           ("k0", k1k0[O:2 * O], c["k0"])):
        b = ulp32(ref)

        def explain(ix, gv, rv, bv, name=name):
            o = ix[0]
            notes = []
            if gv != gv:
                return "NaN: never written"
            if rv != 0 and gv == -float(torch.tensor(rv).float()):
                notes.append("wrong sign")
            notes.append(f"{(gv - float(torch.tensor(rv).float())) / bv:+.3g} ulps from fl32(want)")
            if name == "dbeta":
                p = parts[:, o]
                for sign, how in ((-1.0, "missing"), (1.0, "counted twice")):
                    cand = (db[o] + sign * p - gv).abs() <= bv
                    if bool(cand.any()):
                        k = int(torch.nonzero(cand)[-1])
                        notes.append(f"equals the slot sum with slot {k} of {slots} {how}")
                        break
            if name == "dgamma" and gv == 0 and rv != 0:
                notes.append("zero: never written")
            return "; ".join(notes)

        worst[name] = _check(f"{what} coeffs {name}", got, ref, b, explain, lambda ix: f"channel o = {ix[0]}")
    return worst


def check_accumulated(got, start, from_zero, what=""):
    """An output that is ADDED to: a run from `start` must equal fl32(start + run from 0) bit for bit."""
    want = start.float() + from_zero.float()
    bad = got.view(torch.int32) != want.view(torch.int32)
    if bool(bad.any()):
        ix = tuple(torch.nonzero(bad)[0].tolist())
        gv = float(got[ix])
        note = ""
        if gv == float(from_zero[ix]) and float(start[ix]) != 0:
            note = " -- equals the result from 0: the start value was overwritten, not added to"
        elif gv == float(start[ix]):
            note = " -- equals the start value: nothing was added"
        raise BnAlgMismatch(f"{what}: {int(bad.sum())} elements differ from fl32(start + result from 0); first at "
                            f"{ix}: got {gv!r}, start {float(start[ix])!r}, from 0 {float(from_zero[ix])!r}{note}")


def check_bstack_rows(W, scale, bstack, what=""):
    """Rows 0..O-1 of the B-stack: bf16(fl32(scale_o * W_oi)) bit for bit."""
    O = W.shape[0]
    want = (scale.float().view(-1, 1) * W.float()).bfloat16()
    got = bstack[:O].reshape(want.shape)
    bad = got.view(torch.int16) != want.view(torch.int16)
    if bool(bad.any()):
        o, i = torch.nonzero(bad)[0].tolist()
        note = "no other row matches"
        for r in (o - 1, o + 1, o - 2, o + 2):
            if 0 <= r < O and torch.equal(got[o].view(torch.int16), want[r].view(torch.int16)):
                note = f"row {o} holds row {r}'s values: the B-stack rows are shifted by {o - r}"
                break
        raise BnAlgMismatch(f"{what} B-stack row o = {o} (of {O}), column i = {i}: got {float(got[o, i])!r}, want "
                            f"{float(want[o, i])!r}; {int(bad.sum())} elements differ -- {note}")


def matrix_bounds(W, k1k0):
    O, C = W.shape
    Wd, Wa = W.double(), W.double().abs()
    k1, k0 = k1k0[:O].double(), k1k0[O:2 * O].double()
    gam = (O // K_SPLIT_O + K_SPLIT_O + 2) * U
    M = Wd.t() @ (k1.view(-1, 1) * Wd)
    EM = gam * (Wa.t() @ (k1.abs().view(-1, 1) * Wa))
    bias = Wd.t() @ k0
    Eb = gam * (Wa.t() @ k0.abs())
    return M, EM, bias, Eb


def check_matrix(W, k1k0, bstack, bias, what=""):
    """bn_alg_matrix_kernel + reduce from the GPU's k1k0: M (B-stack rows O..O+C-1, bf16) and the bias (fp32)."""
    O, C = W.shape
    Wd = W.double()
    k1, k0 = k1k0[:O].double(), k1k0[O:2 * O].double()
    M, EM, bref, Eb = matrix_bounds(W, k1k0)
    gotM = bstack[O:O + C].double()
    bM = 2.0 ** -8 * (M.abs() + EM) + EM

    def explain_m(ix, gv, rv, bv):
        j, i = ix
        if gv != gv:
            return "NaN: never written"
        contribs = [(Wd[lo:hi, j] * k1[lo:hi] * Wd[lo:hi, i]).sum() for _, lo, hi in _chunks(O)]
        notes = _chunk_note(gv - rv, contribs, bv + 2.0 ** -8 * abs(gv), O)   # got is the bf16 of a different sum
        return "; ".join(notes) if notes else "no single o-chunk explains the difference"

    def explain_b(ix, gv, rv, bv):
        i = ix[0]
        if gv != gv:
            return "NaN: never written"
        if gv == 0 and bool((bias.double() == 0).all()):
            return "the whole bias is zero: never written"
        contribs = [(k0[lo:hi] * Wd[lo:hi, i]).sum() for _, lo, hi in _chunks(O)]
        notes = _chunk_note(gv - rv, contribs, bv, O)
        if rv != 0 and abs(gv + rv) <= bv:
            notes.append("wrong sign")
        return "; ".join(notes) if notes else "no single o-chunk explains the difference"

    wm = _check(f"{what} M = W^T diag(k1) W", gotM, M, bM, explain_m,
                lambda ix: f"M[j = {ix[0]}][i = {ix[1]}] (B-stack row {O + ix[0]})")
    wb = _check(f"{what} bias = k0^T W", bias, bref, Eb + 2.0 ** -149, explain_b, lambda ix: f"bias[i = {ix[0]}]")
    return dict(M=wm, bias=wb)


def check_dw(W, H, G, s, scale, k1k0, dW, what=""):
    """bn_alg_dw_kernel from dW = 0 on the GPU's H, G, s and k1k0."""
    O, C = W.shape
    Wd = W.double()
    k1, k0, sc = k1k0[:O].double().view(-1, 1), k1k0[O:2 * O].double().view(-1, 1), scale.double().view(-1, 1)
    Hd, Gd, sd = H.double(), G.double(), s.double().view(1, -1)
    terms = {"diag(scale) H": sc * Hd, "k0 (x) s": k0 * sd, "diag(k1) W G": k1 * (Wd @ Gd)}
    ref = sum(terms.values())
    b = (C + 4) * U * ((sc * Hd).abs() + (k0 * sd).abs() + k1.abs() * (Wd.abs() @ Gd.abs())) + 2.0 ** -149

    def explain(ix, gv, rv, bv):
        o, i = ix
        if gv != gv:
            return "NaN: never written"
        notes = [f"{name} {how} in row o = {o}" for name, t in terms.items() for sign, how in ((-1, "missing"), (1, "added twice"))
                 if float(t[o, i]) != 0 and abs(gv - rv - sign * float(t[o, i])) <= bv]
        return "; ".join(notes) if notes else "no single term explains the difference"

    return _check(f"{what} dW", dW, ref, b, explain, lambda ix: f"dW[o = {ix[0]}][i = {ix[1]}]")


def _dact_check(what, dact, ref_s, bound_s, stride, bias, sentinel=True, chunk_explain=None):
    """dact (N, H, W, C) bf16 against ref_s / bound_s on the pixels the dgrad writes; at stride 2 the other pixels must
    still hold SENTINEL_BF16 (sentinel=True) or zero. Failures name (pixel (n, h, w), channel)."""
    N, Hh, Ww, C = dact.shape
    Ho, Wo = Hh // stride, Ww // stride
    got_s = sample(dact, stride).double()
    refd = ref_s.view(N, Ho, Wo, C)
    if stride > 1:
        keep = torch.ones(N, Hh, Ww, dtype=torch.bool, device=dact.device)
        keep[:, ::stride, ::stride] = False
        want_bits = SENTINEL_BF16 if sentinel else 0
        wrote = keep.unsqueeze(-1) & (dact.view(torch.int16) != torch.tensor(want_bits, dtype=torch.int16))
        if bool(wrote.any()):
            n, h, w, c = torch.nonzero(wrote)[0].tolist()
            gv = float(dact[n, h, w, c])
            note = ""
            for dh, dw in ((0, -1), (-1, 0), (-1, -1), (0, 1), (1, 0)):
                hh, ww = h + dh, w + dw
                if 0 <= hh < Hh and 0 <= ww < Ww and hh % stride == 0 and ww % stride == 0:
                    rv, bv = float(refd[n, hh // stride, ww // stride, c]), float(bound_s.view(N, Ho, Wo, C)[n, hh // stride, ww // stride, c])
                    if abs(gv - rv) <= bv:
                        note = f" -- holds the value for pixel ({n}, {hh}, {ww}): the output was written one pixel off"
                        break
            raise BnAlgMismatch(f"{what} dAct: {int(wrote.sum())} elements of pixels a stride-{stride} dgrad does not "
                                f"write were changed; first pixel ({n}, {h}, {w}) channel {c}: {gv!r}{note}")

    def explain(ix, gv, rv, bv):
        r, i = ix
        if gv != gv:
            return "NaN: never written"
        notes = []
        bi = float(bias[i])
        if bi != 0 and abs(gv - rv + bi) <= bv:
            notes.append("the difference is -bias[i]: bias missing")
        if chunk_explain is not None:
            notes += chunk_explain(r, i, gv - rv, bv)
        return "; ".join(notes) if notes else "no single term explains the difference"

    def name_of(ix):
        n, h, w = _pixel(ix[0], N, Ho, Wo, stride)
        return f"pixel ({n}, {h}, {w}) channel {ix[1]}"

    return _check(f"{what} dAct", got_s, ref_s, bound_s, explain, name_of)


def check_dact(g, act, bstack, bias, dact, stride, what="", sentinel=True):
    """The K-concatenated dgrad: [g | act_s] (float64) times the GPU's B-stack plus the GPU's bias."""
    O = g.shape[-1]
    gs = g.reshape(-1, O).double()
    a = sample(act, stride).double()
    B = bstack.double()
    acc = gs @ B[:O] + a @ B[O:]
    absacc = gs.abs() @ B[:O].abs() + a.abs() @ B[O:].abs()
    _, ref, E = er.epilogue_ref(acc, absacc, shift=bias)
    return _dact_check(what, dact, ref, er.REL * ref.abs() + E, stride, bias, sentinel)


# ------------------------------------------------------------------------------------------------------------------
# end to end
# ------------------------------------------------------------------------------------------------------------------
def colsum_bound(a: torch.Tensor, sms: int) -> torch.Tensor:
    """fp32 bound of colsum_pixels_bf16: a thread's sequential row sum, the row lanes of a block, then the blocks."""
    rows, C = a.shape
    lanes = min(C // 8, 256)
    row_lanes = 256 // lanes
    blocks = max(1, min(-(-rows // row_lanes), 4 * sms))
    seq = -(-rows // (blocks * row_lanes))
    return (seq + row_lanes + blocks + 4) * U * a.abs().sum(0)


def check_end_to_end(g, act, W, scale, mean, invstd, stat, slots, stat_stride, stride, got, sms, what="",
                     sentinel=True):
    """The whole chain (H / Gram GEMM, colsum, small kernels, concat dgrad) against the float64 algebra of g, act, W, the
    batch-norm constants and the statistics slots. got: dgamma, dbeta, dW (from 0) and dact. The bound composes the
    weight-gradient bound of H and G (the stacked launch's plan on `sms` SMs), the colsum bound and the stage bounds."""
    O, C = W.shape
    N, Hh, Ww, _ = act.shape
    db = slot_parts(stat, slots, stat_stride, O).sum(0)
    ref = algebra(g, act, W, scale, mean, invstd, stride, db=db)
    rows = ref["rows"]
    gs, a = g.reshape(-1, O).double(), sample(act, stride).double()
    Wd, Wa = W.double(), W.double().abs()
    p = wr.plan("stacked", (N, Hh, Ww, C, O, 1, stride, 0), sms)
    gamH = 2.0 ** -23 * (4 * p["per"] + p["splits"] + 2)
    eH = gamH * (gs.abs().t() @ a.abs()) + U * ref["H"].abs()
    eG = gamH * (a.abs().t() @ a.abs()) + U * ref["G"].abs()
    es = colsum_bound(a, sms)
    sc, is_, mu = scale.double(), invstd.double(), mean.double()
    inv = inv_rows32(rows)
    k1, k0 = ref["k1"], ref["k0"]
    e_dg = is_ * (Wa * eH).sum(1)
    e_k1 = (sc * is_ * inv).abs() * e_dg + 2 * U * k1.abs()
    e_k0 = mu.abs() * e_k1 + 2 * U * k0.abs()
    gam = (O // K_SPLIT_O + K_SPLIT_O + 2) * U
    e_M = Wa.t() @ (e_k1.view(-1, 1) * Wa) + gam * (Wa.t() @ (k1.abs().view(-1, 1) * Wa))
    e_bias = Wa.t() @ e_k0 + gam * (Wa.t() @ k0.abs())
    worst = {}
    worst["dbeta"] = _check(f"{what} end-to-end dbeta", got["dbeta"], db, ulp32(db), lambda *x: "", lambda ix: f"channel o = {ix[0]}")
    worst["dgamma"] = _check(f"{what} end-to-end dgamma", got["dgamma"], ref["dgamma"], e_dg + ulp32(ref["dgamma"]),
                             lambda *x: "", lambda ix: f"channel o = {ix[0]}")
    WG = Wd @ ref["G"]
    b_dw = (sc.abs().view(-1, 1) * eH + e_k1.view(-1, 1) * WG.abs() + k1.abs().view(-1, 1) * (Wa @ eG)
            + e_k0.view(-1, 1) * ref["s"].abs().view(1, -1) + k0.abs().view(-1, 1) * es.view(1, -1)
            + (C + 4) * U * ((sc.view(-1, 1) * ref["H"]).abs() + (k0.view(-1, 1) * ref["s"].view(1, -1)).abs()
                             + k1.abs().view(-1, 1) * (Wa @ ref["G"].abs())) + 2.0 ** -149)
    worst["dW"] = _check(f"{what} end-to-end dW", got["dW"], ref["dW"], b_dw, lambda *x: "",
                         lambda ix: f"dW[o = {ix[0]}][i = {ix[1]}]")
    absacc = gs.abs() @ ref["B0"].abs() + a.abs() @ ref["Mb"].abs()
    E = (er.C_ACC * absacc + er.C_ADD * ref["bias"].abs() + a.abs() @ (2.0 ** -7 * ref["M"].abs() + 2 * e_M)
         + e_bias)
    bound = er.REL * ref["dact_s"].abs() + E
    try:
        worst["dact"] = _dact_check(f"{what} end-to-end", got["dact"], ref["dact_s"], bound, stride, ref["bias"], sentinel)
    except BnAlgMismatch as e:
        # o-chunk z adds act M_z + bias_z to dAct (the parts of M and of the bias from o in chunk z, one split of the same
        # launch); name the chunk whose contribution, once removed or added, brings every written element within its bound
        got_s = sample(got["dact"], stride).double()
        for z, lo, hi in _chunks(O):
            Mz = Wd[lo:hi].t() @ (k1[lo:hi].view(-1, 1) * Wd[lo:hi])
            cz, slack = a @ Mz + Wd[lo:hi].t() @ k0[lo:hi], bound + 2.0 ** -7 * (a.abs() @ Mz.abs())
            for sign, how in ((-1.0, "missing"), (1.0, "added twice")):
                if bool(((got_s - ref["dact_s"] - sign * cz).abs() <= slack).all()):
                    raise BnAlgMismatch(f"{e}\n  every difference is o-chunk {z} (o = {lo}..{hi - 1}) {how} (its part of M and of the bias)") from None
        raise
    return worst
