"""CPU: the float64 reference of tests/bnalg_ref.py is the backward of BatchNorm2d(train) o conv1x1, and each comparator
rejects the faults the GPU table is there to catch, with a message that names the fault.

The "GPU outputs" here come from an fp32 model of the kernels (emulate) that follows their arithmetic: coefficients in
fp64 rounded once, M as fp32 sums over the 8 o-chunks added in order, fp32 dW, and the concat dgrad in fp32 rounded to
bf16 into a sentinel-filled output."""
import pytest
import torch
import torch.nn.functional as F

import bnalg_ref as br

SMS = 148


def emulate(W, H, G, s, stat, slots, stat_stride, scale, mean, invstd, rows, chunk_weight=None):
    O, C = W.shape
    parts = br.slot_parts(stat, slots, stat_stride, O)
    c = br.coefficients(W, H, parts.sum(0), scale, mean, invstd, rows)
    k1, k0 = c["k1"].float(), c["k0"].float()
    bstack = torch.empty(O + C, C, dtype=torch.bfloat16)
    bstack[:O] = (scale.float().view(-1, 1) * W.float()).bfloat16()
    Wf = W.float()
    M = torch.zeros(C, C)
    bias = torch.zeros(C)
    for z, lo, hi in br._chunks(O):
        wz = 1.0 if chunk_weight is None else chunk_weight[z]
        for _ in range(int(wz)):
            M = M + (Wf[lo:hi] * k1[lo:hi].view(-1, 1)).t() @ Wf[lo:hi]
            bias = bias + Wf[lo:hi].t() @ k0[lo:hi]
    bstack[O:] = M.bfloat16()
    dW = scale.float().view(-1, 1) * H.float() + k0.view(-1, 1) * s.float().view(1, -1) + k1.view(-1, 1) * (Wf @ G.float())
    return dict(dgamma=c["dgamma"].float(), dbeta=c["dbeta"].float(), k1k0=torch.cat([k1, k0]), bstack=bstack,
                bias=bias, dW=dW)


def emulate_dact(g, act, bstack, bias, stride, offset=(0, 0)):
    N, Hh, Ww, C = act.shape
    O = g.shape[-1]
    out = torch.full((N, Hh, Ww, C), 0, dtype=torch.int16).fill_(br.SENTINEL_BF16).view(torch.bfloat16)
    v = (g.reshape(-1, O).float() @ bstack[:O].float() + br.sample(act, stride).float() @ bstack[O:].float() + bias)
    out[:, offset[0]::stride, offset[1]::stride, :] = v.bfloat16().view(N, Hh // stride, Ww // stride, C)
    return out


def problem(O=256, C=64, N=2, Hh=8, stride=1, slots=5, seed=0, offset=0.0):
    gen = torch.Generator().manual_seed(seed)
    act = (torch.randn(N, Hh, Hh, C, generator=gen).relu() + offset).bfloat16()
    W = (torch.randn(O, C, generator=gen) / C ** 0.5).bfloat16()
    Ho = Hh // stride
    g = (torch.randn(N, Ho, Ho, O, generator=gen) * (torch.rand(N, Ho, Ho, O, generator=gen) > 0.5)).bfloat16()
    a = br.sample(act, stride).double()
    raw = a @ W.double().t()
    mean, var = raw.mean(0), raw.var(0, unbiased=False)
    invstd = (1.0 / torch.sqrt(var + br.EPS)).float()
    gamma = torch.rand(O, generator=gen) + 0.5
    scale = gamma * invstd
    rows = a.shape[0]
    # slots: random split of the column sums of g (layout [slots][2][O], the second row NaN: it must not be read)
    gs = g.reshape(rows, O).float()
    cut = torch.randint(0, slots, (rows,), generator=gen)
    stat = torch.full((slots, 2, O), float("nan"))
    for k in range(slots):
        stat[k, 0] = gs[cut == k].sum(0)
    H, G, s = (gs.t() @ a.float()), a.float().t() @ a.float(), a.float().sum(0)
    return dict(act=act, W=W, g=g, mean=mean.float(), invstd=invstd, scale=scale, rows=rows, stat=stat, slots=slots,
                stride=stride, H=H, G=G, s=s, O=O, C=C)


def run(p, **kw):
    return emulate(p["W"], p["H"], p["G"], p["s"], p["stat"], p["slots"], 2 * p["O"], p["scale"], p["mean"], p["invstd"],
                   p["rows"], **kw)


def coeffs(p, out):
    return br.check_coeffs(p["W"], p["H"], p["stat"], p["slots"], 2 * p["O"], p["scale"], p["mean"], p["invstd"],
                           p["rows"], out["dgamma"], out["dbeta"], out["k1k0"])


# ------------------------------------------------------------------------------------------------------------------
# the reference is the backward of BatchNorm2d(train) o conv1x1
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("stride", [1, 2])
@pytest.mark.parametrize("N,Hh,C,O", [(2, 4, 8, 16), (3, 6, 16, 24)])
def test_reference_matches_autograd(N, Hh, C, O, stride):
    gen = torch.Generator().manual_seed(N + Hh + C + stride)
    x = (torch.randn(N, C, Hh, Hh, generator=gen, dtype=torch.float64) + 0.5).requires_grad_()
    w = torch.randn(O, C, generator=gen, dtype=torch.float64).requires_grad_()
    gamma = (torch.randn(O, generator=gen, dtype=torch.float64)).requires_grad_()
    beta = torch.randn(O, generator=gen, dtype=torch.float64).requires_grad_()
    y = F.conv2d(x, w.view(O, C, 1, 1), stride=stride)
    out = F.batch_norm(y, None, None, gamma, beta, training=True, eps=br.EPS)
    up = torch.randn(out.shape, generator=gen, dtype=torch.float64)
    out.backward(up)
    yd = y.detach()
    mean = yd.mean((0, 2, 3))
    invstd = 1.0 / torch.sqrt(yd.var((0, 2, 3), unbiased=False) + br.EPS)
    scale = gamma.detach() * invstd
    ref = br.algebra(up.permute(0, 2, 3, 1), x.detach().permute(0, 2, 3, 1), w.detach(), scale, mean, invstd, stride,
                     mirror=False)
    for got, want in ((ref["dgamma"], gamma.grad), (ref["dbeta"], beta.grad), (ref["dW"], w.grad),
                      (ref["dact"], x.grad.permute(0, 2, 3, 1))):
        assert ((got - want).norm() / want.norm()).item() < 1e-10


def test_emulation_passes_every_comparator():
    for stride in (1, 2):
        p = problem(stride=stride, offset=4.0 if stride == 2 else 0.0)
        out = run(p)
        coeffs(p, out)
        br.check_bstack_rows(p["W"], p["scale"], out["bstack"])
        br.check_matrix(p["W"], out["k1k0"], out["bstack"], out["bias"])
        br.check_dw(p["W"], p["H"], p["G"], p["s"], p["scale"], out["k1k0"], out["dW"])
        dact = emulate_dact(p["g"], p["act"], out["bstack"], out["bias"], stride)
        br.check_dact(p["g"], p["act"], out["bstack"], out["bias"], dact, stride)
        got = dict(dgamma=out["dgamma"], dbeta=out["dbeta"], dW=out["dW"], dact=dact)
        worst = br.check_end_to_end(p["g"], p["act"], p["W"], p["scale"], p["mean"], p["invstd"], p["stat"], p["slots"],
                                    2 * p["O"], stride, got, SMS)
        assert all(v <= 1 for v in worst.values()), worst


# ------------------------------------------------------------------------------------------------------------------
# each fault is rejected, and the message names it
# ------------------------------------------------------------------------------------------------------------------
def next_up(x, n):
    for _ in range(n):
        x = torch.nextafter(x, torch.tensor(float("inf")))
    return x


def test_dgamma_two_ulps_off_in_one_channel():
    p = problem()
    out = run(p)
    out["dgamma"][37] = next_up(out["dgamma"][37], 2)
    with pytest.raises(br.BnAlgMismatch, match=r"(?s)coeffs dgamma.*channel o = 37.*\+2 ulps from fl32\(want\)"):
        coeffs(p, out)


def test_k0_wrong_sign_in_one_channel():
    p = problem()
    out = run(p)
    out["k1k0"][p["O"] + 5] *= -1
    with pytest.raises(br.BnAlgMismatch, match=r"(?s)coeffs k0.*channel o = 5.*wrong sign"):
        coeffs(p, out)


def test_dbeta_summed_over_one_slot_too_few():
    p = problem(slots=7)
    out = run(dict(p, slots=6))
    out = dict(run(p), dbeta=out["dbeta"])
    with pytest.raises(br.BnAlgMismatch, match=r"(?s)coeffs dbeta.*slot 6 of 7 missing"):
        coeffs(p, out)


@pytest.mark.parametrize("weight,how", [(0, "missing"), (2, "added twice")])
def test_one_o_chunk_of_M(weight, how):
    p = problem(O=512)
    cw = [1] * 8
    cw[3] = weight
    out = run(p, chunk_weight=cw)
    with pytest.raises(br.BnAlgMismatch, match=rf"(?s)M = W\^T diag\(k1\) W.*o-chunk 3 \(o = 192..255\) {how}"):
        br.check_matrix(p["W"], out["k1k0"], out["bstack"], out["bias"])
    # the end-to-end comparator names the chunk too, from dAct alone
    dact = emulate_dact(p["g"], p["act"], out["bstack"], out["bias"], 1)
    got = dict(dgamma=out["dgamma"], dbeta=out["dbeta"], dW=out["dW"], dact=dact)
    with pytest.raises(br.BnAlgMismatch, match=rf"(?s)end-to-end dAct.*o-chunk 3 \(o = 192..255\) {how}"):
        br.check_end_to_end(p["g"], p["act"], p["W"], p["scale"], p["mean"], p["invstd"], p["stat"], p["slots"],
                            2 * p["O"], 1, got, SMS)


def test_missing_bias():
    p = problem()
    out = run(p)
    zero = torch.zeros_like(out["bias"])
    with pytest.raises(br.BnAlgMismatch, match=r"(?s)bias = k0\^T W.*the whole bias is zero"):
        br.check_matrix(p["W"], out["k1k0"], out["bstack"], zero)
    dact = emulate_dact(p["g"], p["act"], out["bstack"], zero, 1)
    with pytest.raises(br.BnAlgMismatch, match=r"(?s)dAct.*pixel \(\d+, \d+, \d+\) channel \d+.*bias missing"):
        br.check_dact(p["g"], p["act"], out["bstack"], out["bias"], dact, 1)


def test_b0_rows_shifted_by_one():
    p = problem()
    out = run(p)
    O = p["O"]
    out["bstack"][1:O] = out["bstack"][0:O - 1].clone()
    with pytest.raises(br.BnAlgMismatch, match=r"(?s)B-stack row o = 1 .*shifted by 1"):
        br.check_bstack_rows(p["W"], p["scale"], out["bstack"])


def test_dw_missing_k0_s_in_one_row():
    p = problem()
    out = run(p)
    O = p["O"]
    out["dW"][9] -= out["k1k0"][O + 9] * p["s"]
    with pytest.raises(br.BnAlgMismatch, match=r"(?s)dW\[o = 9\].*k0 \(x\) s missing in row o = 9"):
        br.check_dw(p["W"], p["H"], p["G"], p["s"], p["scale"], out["k1k0"], out["dW"])


def test_dw_overwritten_instead_of_added():
    p = problem()
    out = run(p)
    D = torch.randn(out["dW"].shape, generator=torch.Generator().manual_seed(1))
    with pytest.raises(br.BnAlgMismatch, match=r"(?s)start value was overwritten, not added to"):
        br.check_accumulated(out["dW"].clone(), D, out["dW"], "dW from D")
    br.check_accumulated(D + out["dW"], D, out["dW"], "dW from D")


def test_stride2_dact_written_one_pixel_off():
    p = problem(stride=2)
    out = run(p)
    dact = emulate_dact(p["g"], p["act"], out["bstack"], out["bias"], 2, offset=(0, 1))
    with pytest.raises(br.BnAlgMismatch, match=r"(?s)pixel \(0, 0, 1\).*written one pixel off"):
        br.check_dact(p["g"], p["act"], out["bstack"], out["bias"], dact, 2)
