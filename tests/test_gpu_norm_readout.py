"""The GraphNorm, readout, column-sum and LayerNorm kernels (csrc/norm.cu, pair_ops.cu, nodefeat.cu) one entry point at a time
against a plain torch float64 evaluation of the same formulas, autograd for the gradients.

Inputs are fp32 numbers (helpers.r32), so the kernel and the reference start from the same values. Dropout masks are read back
from the device (a GraphNorm with weight 0 and bias 1 returns its mask; see _keep) and used by the reference of every kernel of
the family at the same seeds and shape: a kernel that indexes its mask differently from the others fails its comparison.

Every bound is a-priori and per element, through helpers.assert_close, with no floor relative to a tensor's largest element:
  - an output that is a sum passes `absum` (the same sum over absolute values) and `nterms` (the roundings one term can meet,
    derived next to the call); the column sums fold their fp32 partials into double every kFoldRows = 8 rows (norm.cu), so
    their nterms does not grow with the row count;
  - an elementwise output is bounded by a fixed number of roundings on the absolute values of its terms, |x| + |a*mean| standing
    for |x - a*mean| so that the rounding of the fp32 statistics is covered, plus (as `atol`) what the fp32 statistics and
    column sums it reads may be off by, propagated to first order from their own bounds.
Every comparison also asserts that its bound rejects at least one plausible wrong reference (_check)."""
import math
import zlib

import numpy as np
import pytest
import torch

from helpers import U32 as U, assert_close, r32

pytestmark = pytest.mark.gpu

F64 = torch.float64
EPS = float(np.float32(1e-5))              # the kernels take eps as an fp32 number
CS = (4, 8, 12, 20, 32, 36, 64, 68, 128, 132, 260, 1020, 1024)
MODES = ((False, 0.0), (True, 0.0), (False, 0.3), (True, 0.5))   # (relu, dropout p)
SEED, SEED_F, SEED_R = 0x5EED, 1234, 77


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from twowl_b200 import ops as ops_mod
    return ops_mod


def _cap_rows(C):
    """A row count past the norm kernels' grid cap (4 CTAs x 148 SMs, each given 4 iterations of 256 / (C/4) row slots before
    another CTA is added): the grid-stride loops then take more than 4 iterations."""
    return 4 * 148 * 4 * (256 // (C // 4)) + 37


def _check(got, ref, what, wrongs, rtol=0.0, atol=0.0, absum=None, nterms=0):
    """assert_close(got, ref) with the given bound, and the same bound rejecting at least one of the plausible wrong references
    `wrongs` = [(name, tensor)]: a bound that accepts every one of them could not notice such a mistake."""
    ref = torch.as_tensor(ref).detach().double().cpu()
    cpu = lambda t: t.detach().double().cpu() if isinstance(t, torch.Tensor) else t  # noqa: E731
    tol = dict(rtol=rtol, atol=cpu(atol), absum=cpu(absum), nterms=nterms)
    assert_close(got.reshape(ref.shape), ref, what=what, **tol)
    assert wrongs, what
    for name, wrong in wrongs:
        try:
            assert_close(wrong.reshape(ref.shape), ref, what=what, **tol)
        except AssertionError:
            return
    raise AssertionError(f"{what}: the bound also accepts every wrong reference: {[n for n, _ in wrongs]}")


def _gen(*key):
    return torch.Generator().manual_seed(zlib.crc32(repr(key).encode()))


def _randn(g, *shape):
    return torch.randn(*shape, generator=g, dtype=F64)


def _gn_input(g, M, C):
    """[M, C] fp32-exact values on the device; columns by c % 4: |mean|/std ~ 1e3, constant (variance 0), an outlier in row 0
    (the shift row of the device statistics), plain."""
    x = _randn(g, M, C)
    kind = torch.arange(C) % 4
    x[:, kind == 0] += 1e3
    x[:, kind == 1] = 0.5 + torch.arange(C)[kind == 1].to(F64) / 8
    x[0, kind == 2] += 64.0
    return r32(x).cuda()


def _gn_params(g, C):
    """(weight, bias, mean_scale); mean_scale cycles through 0.75, 0, 1 and a random value so that every column kind of
    _gn_input meets each of them (C >= 16); the large-mean column 0 gets 0.75."""
    w = r32(torch.rand(C, generator=g, dtype=F64) + 0.5)
    b = r32(_randn(g, C) * 0.5)
    c = torch.arange(C)
    choice = torch.stack((torch.full((C,), 0.75, dtype=F64), torch.zeros(C, dtype=F64), torch.ones(C, dtype=F64),
                          torch.rand(C, generator=g, dtype=F64)))
    a = r32(choice[(c + c // 4) % 4, c])
    return w.cuda(), b.cuda(), a.cuda()


def _f(t):
    return t.float().contiguous()


class _Stats:
    """GraphNorm (mean, inv_std) of x in fp64, and a-priori bounds (absolute) of the device's fp32 ones: the device sums x - x[0]
    and (x - x[0])^2 per column (row 0 is its shift), in fp32 chains of 8 rows folded into double."""

    def __init__(self, x, a):
        M = x.shape[0]
        self.mean = x.mean(0)
        xc = x - a * self.mean
        self.inv = ((xc * xc).mean(0) + EPS).rsqrt()
        d = (x - x[0]).abs()
        self.s1, s2 = d.sum(0) / M, (d * d).sum(0) / M
        ms = (self.mean - x[0]).abs()
        # the variance's sensitivity to the two sums: var = s2 - ms^2 (+ (1-a)^2 mean^2), inv = (var + eps)^-1/2
        self.var_terms = 0.5 * self.inv ** 3 * (s2 + 2 * (ms + (1 - a) ** 2 * self.mean.abs()) * self.s1)
        # nterms 12: a term rounds twice (x - x0, then its square's fma) + 7 adds of an 8-row fp32 chain + 3 for the fp64 adds
        self.e_mean = 12 * U * self.s1 + U * self.mean.abs()
        self.e_inv = 12 * U * self.var_terms + U * self.inv


class _Branch:
    """One GraphNorm(+Dropout+ReLU) branch of the device, in fp64: the statistics, the device's mask `keep` (0 or 1/(1-p) as
    the fp32 number the device multiplies by), and the error bound `err` of the device's value drop(GN(x)) per element."""

    def __init__(self, x, w, b, a, keep, relu):
        self.x, self.w, self.b, self.a, self.keep, self.relu = x, w, b, a, keep, relu
        self.st = st = _Stats(x, a)
        self.t = x.abs() + (a * st.mean).abs()           # |x| + |a mean| in place of |x - a mean|
        self.yd = (w * st.inv * (x - a * st.mean) + b) * keep
        # 6 roundings: w*inv, a*mean, sc*nm, b - sc*nm, the fma, the mask product
        self.terms = keep * ((w * st.inv).abs() * self.t + b.abs())
        self.stat = keep * (w.abs() * self.t * st.e_inv + (w * st.inv * a).abs() * st.e_mean)
        self.err = 6 * U * self.terms + self.stat
        self.rmask = torch.ones_like(x)
        self.ties = 0

    def resolve(self, dev_act):
        """The ReLU mask. Where |drop(GN(x))| is within its own error bound either decision is right: take the device's (its
        act(drop(GN(x))) of this branch alone, dev_act > 0)."""
        if self.relu:
            m = self.yd > 0
            tie = self.yd.abs() <= self.err
            m[tie] = dev_act.double()[tie] > 0
            self.rmask = m.to(F64)
            self.ties = int((tie & (self.keep > 0)).sum())
            assert self.ties <= 4 + self.x.numel() // 10, self.ties      # a mask bug would not hide among so few
        return self

    def h(self):
        return self.yd * self.rmask

    def e_h(self):
        return self.err * self.rmask


def _act(x, w, b, a, keep, relu, rmask=None):
    """act(drop(GN(x))) in fp64, differentiable in every argument -> (value, x - a*mean). rmask None: the ReLU decides from the
    fp64 value itself (the wrong references)."""
    mean = x.mean(0)
    xc = x - a * mean
    inv = ((xc * xc).mean(0) + EPS).rsqrt()
    y = (w * inv * xc + b) * keep
    if relu:
        y = y * (rmask if rmask is not None else (y.detach() > 0).to(F64))
    return y, xc


def _keep(ops, M, C, p, seed, seed_r=None, branch="f"):
    """The device's dropout mask at (seed, shape), read back: weight 0 and bias 1 make every pre-dropout value 1.
    seed_r=None: graphnorm_apply's; else the mask of `branch` of graphnorm_apply2 at (seed_f = seed, seed_r), the other branch
    given weight 0 and bias 0 (it adds 0)."""
    z, o = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
    x = torch.zeros(M, C, device="cuda")
    stats = torch.cat((z, o))
    if seed_r is None:
        return ops.graphnorm_apply(x, stats, z, o, z, p, seed, False).double()
    one, off = (z, o, z), (z, z, z)
    pf, pr = (one, off) if branch == "f" else (off, one)
    return ops.graphnorm_apply2(x, x, stats, stats, pf, pr, p, seed, seed_r, False).double()


def _mask_sanity(keeps, p, seed_pairs):
    """Keep rate within 5 sigma of 1-p; different seeds give different masks."""
    for k in keeps:
        n = k.numel()
        rate = float((k > 0).double().mean())
        assert abs(rate - (1 - p)) <= 5 * math.sqrt(p * (1 - p) / n), (rate, p, n)
        assert bool(((k == 0) | (k == float(np.float32(1) / (np.float32(1) - np.float32(p))))).all())
    for k1, k2 in seed_pairs:
        if k1.numel() >= 256:
            assert not torch.equal(k1, k2)


def _sum_bounds(br, gy, e_gy, rows=None):
    """Bounds of the device's column sums A = sum g_y, B = sum g_y*n over the given rows (positions) of a branch, and of
    sum g_o = inv*w*(A - B*inv*mean*(1-a)) made from them. e_gy: the error of the device's g_y per element."""
    st, a, w = br.st, br.a, br.w
    t = br.t if rows is None else br.t[rows]
    n_abs = t * st.inv
    e_n = st.inv * a.abs() * st.e_mean + t * st.e_inv          # the device's n from its fp32 statistics
    s = dict(absA=gy.abs().sum(0), absB=(gy.abs() * n_abs).sum(0), eA=e_gy.sum(0),
             eB=(e_gy * n_abs + gy.abs() * e_n).sum(0))
    # nterms: A 10 = 1 (the mask product) + 7 (an 8-row fp32 chain) + 2 (fp64 adds); B 13 = 3 more for n = (x - nm)*ni and the fma
    s["E_A"] = 10 * U * s["absA"] + s["eA"]
    s["E_B"] = 13 * U * s["absB"] + s["eB"]
    return s


def _dparams_check(dp, br, s, A, B, sgo, g_in, what, wrongs):
    """dparams [4C] = [dweight = B, dbias = A, dmean_scale = -mean * sum g_o, colsum(dx) = (1-a) * sum g_o] (norm.cu:224).
    g_in: the column sum of the op's incoming gradient (what a colsum(dx) of the wrong tensor would give)."""
    C = br.w.numel()
    st, a, w = br.st, br.a, br.w
    om = 1 - a
    e_sgo = (w.abs() * st.inv * (s["E_A"] + st.inv * (st.mean * om).abs() * s["E_B"])
             + w.abs() * (A.abs() + 2 * st.inv * (B * st.mean * om).abs()) * st.e_inv
             + w.abs() * st.inv ** 2 * (B * om).abs() * st.e_mean)
    wr = lambda i: [(n, t[i * C:(i + 1) * C]) for n, t in wrongs]  # noqa: E731
    _check(dp[:C], B, what + " dweight", wr(0), rtol=U, atol=s["eB"], absum=s["absB"], nterms=13)   # nterms: _sum_bounds
    _check(dp[C:2 * C], A, what + " dbias", wr(1), rtol=U, atol=s["eA"], absum=s["absA"], nterms=10)  # nterms: _sum_bounds
    # derived from A and B in fp64, one fp32 store: their bounds propagated
    _check(dp[2 * C:3 * C], -st.mean * sgo, what + " dmean_scale", wr(2), rtol=2 * U,
           atol=st.mean.abs() * e_sgo + sgo.abs() * st.e_mean)
    _check(dp[3 * C:], om * sgo, what + " colsum(dx)",
           wr(3) + [("colsum(dx) replaced by sum g_o", sgo), ("the incoming gradient's column sum", g_in)], rtol=2 * U,
           atol=om.abs() * e_sgo)
    return e_sgo


def _dx_bounds(br, s, B, sgo, e_sgo, gy, e_gy, M):
    """dx = sc*(g_y - n*B/M) - a*sum g_o/M per element -> (terms for 8 roundings, atol from the sums and the statistics)."""
    st, a, w = br.st, br.a, br.w
    sc = (w * st.inv).abs()
    n_abs = br.t * st.inv
    e_n = st.inv * a.abs() * st.e_mean + br.t * st.e_inv
    terms = sc * (gy.abs() + n_abs * B.abs() / M) + (a * sgo).abs() / M
    atol = (sc * (e_gy + n_abs * s["E_B"] / M) + a.abs() * e_sgo / M
            + w.abs() * st.e_inv * (gy.abs() + n_abs * B.abs() / M) + sc * e_n * B.abs() / M)
    return terms, atol


def _row0_wrong(br, gy, rows=None):
    """dparams with the first row's (position's) terms left out of the column sums A and B."""
    x = br.x if rows is None else br.x[rows]
    n = (x - br.a * br.st.mean) * br.st.inv
    z = torch.zeros_like(br.a)
    return torch.cat(((gy * n)[1:].sum(0), gy[1:].sum(0), z, z))


def _dparams_ref(leaves, xc):
    """(A, B, sum g_o) of one branch from its autograd leaves: dbias, dweight, and the gradient of x - a*mean summed."""
    x, w, b, a = leaves
    return b.grad, w.grad, xc.grad.sum(0)


def _leaves(x, w, b, a):
    return [t.detach().clone().requires_grad_(True) for t in (x, w, b, a)]


# ------------------------------------------------------------------------------------------------ one GraphNorm

@pytest.mark.parametrize("relu,p", MODES)
@pytest.mark.parametrize("M", [1, 2, 7, 1009, "cap"])
@pytest.mark.parametrize("C", CS)
def test_graphnorm_single_branch(ops, C, M, relu, p):
    """graphnorm_stats, graphnorm_stats_from_moments, graphnorm_apply (with an addend) and graphnorm_bwd."""
    M = _cap_rows(C) if M == "cap" else M
    g = _gen("single", C, M, relu, p)
    x = _gn_input(g, M, C)
    w, b, a = _gn_params(g, C)
    dout = r32(_randn(g, M, C)).cuda()
    add = r32(_randn(g, M, C)).cuda()
    ones = torch.ones_like(a)

    st = _Stats(x, a)
    wrong_st = _Stats(x, ones)
    ref = torch.cat((st.mean, st.inv))
    # nterms 12: _Stats (2 roundings in a term + 7 in an 8-row chain + 3 in fp64)
    tol = dict(rtol=U, absum=torch.cat((st.s1, st.var_terms)), nterms=12)
    wrongs = [("mean_scale ignored", torch.cat((wrong_st.mean, wrong_st.inv))),
              ("mean_scale applied to the stored mean", torch.cat((a * st.mean, st.inv)))]
    stats = ops.graphnorm_stats(_f(x), _f(a), EPS)
    _check(stats, ref, "graphnorm_stats", wrongs, **tol)
    # from exact fp64 moments: no fp32 sum, only fp64 arithmetic and the fp32 store (the fp64 cancellation of sum x^2/M - mean^2
    # is 2^-52 * 1e6 at most here, far below one fp32 rounding of inv)
    mom = torch.cat((x.sum(0), (x * x).sum(0)))
    _check(ops.graphnorm_stats_from_moments(mom, M, _f(a), EPS), ref, "graphnorm_stats_from_moments", wrongs, rtol=2 * U)

    keep = _keep(ops, M, C, p, SEED) if p > 0 else torch.ones_like(x)
    if p > 0:
        _mask_sanity([keep], p, [(keep, _keep(ops, M, C, p, SEED + 1))])
        assert torch.equal(keep, _keep(ops, M, C, p, SEED))
    br = _Branch(x, w, b, a, keep, relu)
    out = ops.graphnorm_apply(_f(x), stats, _f(w), _f(b), _f(a), p, SEED, relu, addend=_f(add))
    act = ops.graphnorm_apply(_f(x), stats, _f(w), _f(b), _f(a), p, SEED, relu)
    br.resolve(act)
    wrongs = [("mean_scale ignored", _act(x, w, b, ones, keep, relu)[0] + add)]
    if relu:
        wrongs.append(("ReLU mask omitted", br.yd + add))
    if p > 0:
        wrongs.append(("dropout mask ignored", _act(x, w, b, a, torch.ones_like(x), relu)[0] + add))
    # 6 roundings of _Branch + 1 for the addend
    _check(out, br.h() + add, "graphnorm_apply", wrongs, atol=br.stat, absum=br.terms + (br.h() + add).abs(), nterms=7)

    lv = _leaves(x, w, b, a)
    h, xc = _act(*lv, keep, relu, br.rmask)
    xc.retain_grad()
    (h * dout).sum().backward()
    A, B, sgo = _dparams_ref(lv, xc)
    wl = _leaves(x, w, b, ones)
    hw, _ = _act(*wl, keep, relu)
    (hw * dout).sum().backward()
    wrong_dp = [("mean_scale ignored", torch.cat((wl[1].grad, wl[2].grad, wl[3].grad, torch.zeros_like(a))))]
    dx_wrongs = [("mean_scale ignored", wl[0].grad)]
    if relu:
        l2 = _leaves(x, w, b, a)
        h2, _ = _act(*l2, keep, False)
        (h2 * dout).sum().backward()
        wrong_dp.append(("ReLU mask omitted", torch.cat((l2[1].grad, l2[2].grad, l2[3].grad, torch.zeros_like(a)))))
        dx_wrongs.append(("ReLU mask omitted", l2[0].grad))
    if p > 0:
        l3 = _leaves(x, w, b, a)
        h3, _ = _act(*l3, torch.ones_like(x), relu)
        (h3 * dout).sum().backward()
        wrong_dp.append(("dropout mask ignored", torch.cat((l3[1].grad, l3[2].grad, l3[3].grad, torch.zeros_like(a)))))
        dx_wrongs.append(("dropout mask ignored", l3[0].grad))
    dx, dp = ops.graphnorm_bwd(_f(x), _f(dout), stats, _f(w), _f(b), _f(a), p, SEED, relu)
    gy = dout * keep * br.rmask
    wrong_dp.append(("row 0 left out", _row0_wrong(br, gy)))
    e_gy = torch.zeros_like(gy)
    s = _sum_bounds(br, gy, e_gy)
    e_sgo = _dparams_check(dp, br, s, A, B, sgo, dout.sum(0), "graphnorm_bwd", wrong_dp)
    terms, atol = _dx_bounds(br, s, B, sgo, e_sgo, gy, e_gy, M)
    # 8 roundings: sc, x - nm, * ni, the stored B/M, n * bm, g_y - ., sc * (.), - corr (corr itself: its fp32 store)
    _check(dx, lv[0].grad, "graphnorm_bwd dx", dx_wrongs, atol=atol, absum=terms, nterms=8)


# ------------------------------------------------------------------------------------------------ two branches

def _two_branches(ops, g, M, C, relu, p):
    xf, xr = _gn_input(g, M, C), _gn_input(g, M, C)
    pf, pr = _gn_params(g, C), _gn_params(g, C)
    sf, sr = ops.graphnorm_stats(_f(xf), _f(pf[2]), EPS), ops.graphnorm_stats(_f(xr), _f(pr[2]), EPS)
    if p > 0:
        kf, kr = _keep(ops, M, C, p, SEED_F, SEED_R), _keep(ops, M, C, p, SEED_F, SEED_R, "r")
        _mask_sanity([kf, kr], p, [(kf, kr), (kf, _keep(ops, M, C, p, SEED_F + 1, SEED_R))])
        assert torch.equal(kf, _keep(ops, M, C, p, SEED_F, SEED_R))
    else:
        kf = kr = torch.ones_like(xf)
    bf, brr = _Branch(xf, *pf, kf, relu), _Branch(xr, *pr, kr, relu)
    z = torch.zeros_like(pf[0])
    f32 = lambda t: tuple(_f(v) for v in t)  # noqa: E731
    P = dict(pf=f32(pf), pr=f32(pr))
    bf.resolve(ops.graphnorm_apply2(_f(xf), _f(xr), sf, sr, P["pf"], (z, z, z), p, SEED_F, SEED_R, relu))
    brr.resolve(ops.graphnorm_apply2(_f(xf), _f(xr), sf, sr, (z, z, z), P["pr"], p, SEED_F, SEED_R, relu))
    return bf, brr, sf, sr, P


def _wrong_h(bf, brr, which):
    """act(drop(GN_f(xf))) + act(drop(GN_r(xr))) with one plausible mistake."""
    ones = torch.ones_like(bf.a)
    if which == "mean_scale ignored":
        return _act(bf.x, bf.w, bf.b, ones, bf.keep, bf.relu)[0] + _act(brr.x, brr.w, brr.b, ones, brr.keep, brr.relu)[0]
    if which == "keep_f and keep_r swapped":
        return _act(bf.x, bf.w, bf.b, bf.a, brr.keep, bf.relu)[0] + _act(brr.x, brr.w, brr.b, brr.a, bf.keep, brr.relu)[0]
    assert which == "ReLU mask omitted"
    return bf.yd + brr.yd


def _wrong_names(relu, p):
    return ["mean_scale ignored"] + (["ReLU mask omitted"] if relu else []) + (["keep_f and keep_r swapped"] if p > 0 else [])


def _two_branch_grads(bf, brr, loss_of_h, which=None):
    """Autograd of loss_of_h(act_f + act_r) -> (leaves_f, leaves_r, xc_f, xc_r); `which` = a mistake of _wrong_h."""
    lf, lr = _leaves(bf.x, bf.w, bf.b, bf.a), _leaves(brr.x, brr.w, brr.b, brr.a)
    kf, kr, mf, mr = bf.keep, brr.keep, bf.rmask, brr.rmask
    if which == "mean_scale ignored":
        lf[3], lr[3] = torch.ones_like(bf.a), torch.ones_like(bf.a)
        mf = mr = None
    elif which == "keep_f and keep_r swapped":
        kf, kr, mf, mr = kr, kf, None, None
    hf, xcf = _act(*lf, kf, bf.relu and which != "ReLU mask omitted", mf)
    hr, xcr = _act(*lr, kr, brr.relu and which != "ReLU mask omitted", mr)
    xcf.retain_grad()
    xcr.retain_grad()
    loss_of_h(hf + hr).backward()
    return lf, lr, xcf, xcr


def _wrong_dp(l):
    z = torch.zeros_like(l[1].grad)
    return torch.cat((l[1].grad, l[2].grad, z if l[3].grad is None else l[3].grad, z))


@pytest.mark.parametrize("relu,p", MODES)
@pytest.mark.parametrize("M", [1, 2, 7, 1009, "cap"])
@pytest.mark.parametrize("C", CS)
def test_graphnorm_two_branches(ops, C, M, relu, p):
    """graphnorm_apply2 and graphnorm_bwd2 (its sums and apply halves, M_total == M)."""
    M = _cap_rows(C) if M == "cap" else M
    g = _gen("two", C, M, relu, p)
    bf, brr, sf, sr, P = _two_branches(ops, g, M, C, relu, p)
    dout = r32(_randn(g, M, C)).cuda()
    names = _wrong_names(relu, p)

    out = ops.graphnorm_apply2(_f(bf.x), _f(brr.x), sf, sr, P["pf"], P["pr"], p, SEED_F, SEED_R, relu)
    h = bf.h() + brr.h()
    # each branch: 6 roundings of _Branch; + 1 for the sum of the two
    _check(out, h, "graphnorm_apply2", [(n, _wrong_h(bf, brr, n)) for n in names], atol=bf.stat + brr.stat,
           absum=bf.terms + brr.terms + h.abs(), nterms=6)

    lf, lr, xcf, xcr = _two_branch_grads(bf, brr, lambda hh: (hh * dout).sum())
    wrong = {n: _two_branch_grads(bf, brr, lambda hh: (hh * dout).sum(), n) for n in names}
    dxf, dxr, dpf, dpr = ops.graphnorm_bwd2(_f(bf.x), _f(brr.x), _f(dout), sf, sr, P["pf"], P["pr"], p, SEED_F, SEED_R, relu)
    for br, l, xc, dx, dp, k, tag in ((bf, lf, xcf, dxf, dpf, 0, "f"), (brr, lr, xcr, dxr, dpr, 1, "r")):
        A, B, sgo = _dparams_ref(l, xc)
        gy = dout * br.keep * br.rmask
        e_gy = torch.zeros_like(gy)
        s = _sum_bounds(br, gy, e_gy)
        e_sgo = _dparams_check(dp, br, s, A, B, sgo, dout.sum(0), "graphnorm_bwd2 " + tag,
                               [(n, _wrong_dp(wrong[n][k])) for n in names] + [("row 0 left out", _row0_wrong(br, gy))])
        terms, atol = _dx_bounds(br, s, B, sgo, e_sgo, gy, e_gy, M)
        _check(dx, l[0].grad, "graphnorm_bwd2 dx" + tag, [(n, wrong[n][k][0].grad) for n in names],   # 8 roundings: _dx_bounds
               atol=atol, absum=terms, nterms=8)


# ------------------------------------------------------------------------------------------------ readout

LINK_CASES = ("L0", "L1", "L2", "L3", "hot", "strided", "masked", "long")
HOT_ROW, HOT_N = 5, 300


def _links(g, case, M, C):
    """Readout row ids int64 [2L] on the device (a 1-D view, strided for "strided") and whether masks may occur.
      L0..L3: that many links; hot: L = 1001 (odd: the two-links-per-iteration loop of the grouped forward runs both ways), row
      HOT_ROW selected by HOT_N positions, some self pairs; strided: every second element of a longer list (sidx = 2);
      masked: a negative id in slot 0, slot 1 or both, and a packed tail of -2; long: 2L past the grid cap of the row-sparse
      backward."""
    rnd = lambda n: torch.randint(0, M, (n,), generator=g, dtype=torch.int64)  # noqa: E731
    if case[0] == "L":
        return rnd(2 * int(case[1])).cuda()
    if case == "hot":
        idx = rnd(2002)
        idx[torch.randperm(2002, generator=g)[:HOT_N]] = HOT_ROW
        self_pairs = torch.randperm(1001, generator=g)[:50]
        idx[2 * self_pairs + 1] = idx[2 * self_pairs]
        return idx.cuda()
    if case == "strided":
        return rnd(4 * 257).cuda()[::2]
    if case == "masked":
        L = 301
        idx = rnd(2 * L).view(L, 2)
        sel = torch.randperm(L - 40, generator=g)[:90]
        idx[sel[:30], 0] = -1
        idx[sel[30:60], 1] = -1
        idx[sel[60:], :] = -1
        idx[L - 40:] = -2
        return idx.reshape(-1).cuda()
    assert case == "long"
    L = max(1001, _cap_rows(C) // 2 + 1) | 1
    return rnd(2 * L).cuda()


def _readout_nterms(C):
    # a lane's fma chain over its ceil(C/128) float4 (4 each), 1 for h0*h1, a 5-level xor tree, the bias add
    return 4 * (-(-C // 128)) + 7


@pytest.mark.parametrize("relu,p", MODES)
@pytest.mark.parametrize("case", LINK_CASES)
@pytest.mark.parametrize("C", CS)
def test_gn2_readout(ops, C, case, relu, p):
    """gn2_readout_fwd, gn2_readout_bwd and gn2_readout_bwd_prepare (G, dparams_f/r, dw, db, consts, and dx rebuilt from consts)."""
    M = 3001
    g = _gen("readout", C, case, relu, p)
    bf, brr, sf, sr, P = _two_branches(ops, g, M, C, relu, p)
    idx = _links(g, case, M, C)
    L = idx.numel() // 2
    w = r32(_randn(g, 1, C)).cuda()
    bias = r32(_randn(g, 1)).cuda()
    dpred = r32(_randn(g, L)).cuda()
    names = _wrong_names(relu, p)
    args = (_f(bf.x), _f(brr.x), sf, sr, P["pf"], P["pr"], p, SEED_F, SEED_R, relu, idx)

    pred = ops.gn2_readout_fwd(*args, _f(w), _f(bias)).reshape(-1)
    dxf, dxr, dpf, dpr, dw, db = ops.gn2_readout_bwd(*args, _f(w), _f(dpred))
    G, head, nxt, consts, dpf2, dpr2, dw2, db2 = ops.gn2_readout_bwd_prepare(*args, _f(w), _f(dpred))
    torch.cuda.synchronize()
    for a_, b_ in ((dpf, dpf2), (dpr, dpr2), (dw, dw2), (db, db2)):
        assert torch.equal(a_, b_)          # the same row-sparse half

    i = idx.reshape(L, 2) if L else idx.reshape(0, 2)
    tail = (i[:, 0] == -2).nonzero()
    valid = (i >= 0).all(1)
    if tail.numel():
        valid[int(tail[0]):] = False
    if not bool(valid.any()):
        assert bool((pred == 0).all()) and bool((dpf == 0).all()) and bool((dpr == 0).all())
        assert bool((dw == 0).all()) and bool((db == 0).all()) and bool((dxf == 0).all()) and bool((dxr == 0).all())
        return
    assert bool((pred[~valid] == 0).all()), "a masked link's logit is exactly 0"
    i0, i1 = i[valid, 0], i[valid, 1]
    gl = dpred[valid]

    h = bf.h() + brr.h()
    e_h = bf.e_h() + brr.e_h() + U * h.abs()
    wv = w.reshape(-1)

    def pred_of(hh, ww=wv, bb=bias):
        out = torch.zeros(L, dtype=F64, device="cuda")
        out[valid] = (hh[i0] * hh[i1] * ww).sum(1) + bb
        return out

    ref = pred_of(h)
    absum = torch.zeros(L, dtype=F64, device="cuda")
    absum[valid] = (h[i0] * h[i1] * wv).abs().sum(1) + bias.abs()
    atol = torch.zeros(L, dtype=F64, device="cuda")
    atol[valid] = (wv.abs() * (h[i0].abs() * e_h[i1] + h[i1].abs() * e_h[i0])).sum(1)
    wrongs = [(n, pred_of(_wrong_h(bf, brr, n))) for n in names] + [("bias left out", pred_of(h, bb=0.0)),
                                                                     ("w ignored", pred_of(h, ww=1.0))]
    _check(pred, ref, "gn2_readout_fwd", wrongs, atol=atol, absum=absum,
           nterms=_readout_nterms(C))

    def loss(hh):
        return (pred_of(hh, wl, bl) * dpred).sum()

    wl, bl = wv.clone().requires_grad_(True), bias.clone().requires_grad_(True)
    lf, lr, xcf, xcr = _two_branch_grads(bf, brr, loss)
    ref_dw, ref_db = wl.grad, bl.grad
    wrong = {}
    for n in names:
        wl, bl = wv.clone().requires_grad_(True), bias.clone().requires_grad_(True)
        wrong[n] = _two_branch_grads(bf, brr, loss, n)

    # G at every valid position j: dpred[l] * w * h[partner]; the rows of masked positions are never read
    pos = torch.arange(2 * L, device="cuda").reshape(L, 2)[valid].reshape(-1)
    ra, rb = idx[pos], idx[pos ^ 1]
    gpos = dpred[pos // 2].unsqueeze(1)
    refG = gpos * wv * h[rb]
    shifted = dpred[(pos // 2 + 1) % L].unsqueeze(1) * wv * h[rb]
    # 2 roundings: g*w, then * h
    own = gpos * wv * h[ra]
    _check(G[pos], refG, "gn2_readout G", [("dpred of link l sent to link l+1", shifted),
                                          ("a position's own row in place of its partner's", own)], atol=(gpos * wv).abs() * e_h[rb],
           absum=refG.abs(), nterms=2)
    e_G = (gpos * wv).abs() * e_h[rb] + 2 * U * refG.abs()

    hp = h[i0] * h[i1]
    # dw: 1 for h0*h1, 1 for the fma, 7 in an 8-row chain, 2 in fp64
    _check(dw, ref_dw, "gn2_readout dw", [("dpred of link l sent to link l+1", (torch.roll(gl, -1).unsqueeze(1) * hp).sum(0)),
                                          ("link 0 left out", (gl.unsqueeze(1) * hp)[1:].sum(0))],
           atol=(gl.abs().unsqueeze(1) * (h[i0].abs() * e_h[i1] + h[i1].abs() * e_h[i0])).sum(0),
           absum=(gl.unsqueeze(1) * hp).abs().sum(0), nterms=11)
    # db: 7 in an 8-row chain + 3 in fp64
    _check(db, ref_db, "gn2_readout db", [("both positions of a link counted", 2 * gl.sum().reshape(1))],
           absum=gl.abs().sum().reshape(1), nterms=10)

    cnt = torch.zeros(M, dtype=F64, device="cuda").index_add_(0, ra, torch.ones_like(ra, dtype=F64))
    Gsum = torch.zeros(M, C, dtype=F64, device="cuda").index_add_(0, ra, G[pos].double())
    Gabs = torch.zeros(M, C, dtype=F64, device="cuda").index_add_(0, ra, refG.abs())
    eGs = torch.zeros(M, C, dtype=F64, device="cuda").index_add_(0, ra, e_G)
    dup = int(torch.nonzero(cnt > 1)[0]) if bool((cnt > 1).any()) else None
    for br, l, xc, dx, dp, k, tag in ((bf, lf, xcf, dxf, dpf, 0, "f"), (brr, lr, xcr, dxr, dpr, 1, "r")):
        A, B, sgo = _dparams_ref(l, xc)
        m = br.keep[ra] * br.rmask[ra]
        gy = refG * m
        s = _sum_bounds(br, gy, e_G * m + U * gy.abs(), rows=ra)
        e_sgo = _dparams_check(dp, br, s, A, B, sgo, refG.sum(0), "gn2_readout dparams_" + tag,
                               [(n, _wrong_dp(wrong[n][k])) for n in names] + [("position 0 left out", _row0_wrong(br, gy, ra))])
        # the dense pass: g_y of a row = its positions' G added in ascending order (cnt - 1 roundings) times the mask
        gyr = br.keep * br.rmask * Gsum
        e_gyr = br.keep * br.rmask * ((cnt.unsqueeze(1) + 1) * U * Gabs + eGs)
        terms, atol = _dx_bounds(br, s, B, sgo, e_sgo, gyr.abs(), e_gyr, M)
        wrongs = [(n, wrong[n][k][0].grad) for n in names]
        if dup is not None:      # the last position of a row selected several times left out of its chain
            last = int((ra == dup).nonzero()[-1])
            sc = br.w * br.st.inv
            drop = l[0].grad.clone()
            drop[dup] -= sc * br.keep[dup] * br.rmask[dup] * refG[last]
            wrongs.append(("one duplicate position's gradient dropped", drop))
        _check(dx, l[0].grad, "gn2_readout dx" + tag, wrongs, atol=atol, absum=terms, nterms=8)   # 8 roundings: _dx_bounds

        # consts [4][C] = (P, Q, sc, of): dx = P*x + Q + sc*g_y
        st, a, wb, bb = br.st, br.a, br.w, br.b
        nm = a * st.mean
        Pr = -wb * st.inv ** 2 * B / M
        corr = a * sgo / M
        e_P = 4 * U * Pr.abs() + 2 * Pr.abs() * st.e_inv / st.inv + wb.abs() * st.inv ** 2 * s["E_B"] / M
        e_corr = a.abs() * e_sgo / M + U * corr.abs()
        e_Q = 4 * U * ((Pr * nm).abs() + corr.abs()) + e_P * nm.abs() + Pr.abs() * a.abs() * st.e_mean + e_corr
        e_sc = U * (wb * st.inv).abs() + wb.abs() * st.e_inv
        e_of = 3 * U * ((wb * st.inv * nm).abs() + bb.abs()) + nm.abs() * e_sc + (wb * st.inv * a).abs() * st.e_mean
        cref = torch.cat((Pr, -Pr * nm - corr, wb * st.inv, bb - wb * st.inv * nm))
        # mean_scale ignored: nm = mean
        cw = torch.cat((Pr, -Pr * st.mean - sgo / M, wb * st.inv, bb - wb * st.inv * st.mean))
        cs = consts[4 * C * k:4 * C * (k + 1)]
        _check(cs, cref, "gn2_readout consts_" + tag, [("mean_scale ignored", cw)], atol=torch.cat((e_P, e_Q, e_sc, e_of)))
        # dx rebuilt in fp64 from the device's consts and G
        Pd, Qd, scd = (cs[j * C:(j + 1) * C].double() for j in range(3))
        rebuilt = Pd * br.x + Qd + scd * br.keep * br.rmask * Gsum
        _check(rebuilt, l[0].grad, "gn2_readout dx from consts " + tag, wrongs,
               atol=br.x.abs() * e_P + e_Q + gyr.abs() * e_sc + scd.abs() * br.keep * br.rmask * eGs)


@pytest.mark.parametrize("case", ("L1", "L3", "hot", "strided", "long"))
@pytest.mark.parametrize("C", CS)
def test_readout_unfused(ops, C, case):
    """readout_fwd and readout_bwd (pair_ops.cu): pred = sum_c H[i0,c] H[i1,c] w[c] + b and its gradients."""
    M = 3001
    g = _gen("unfused", C, case)
    H = r32(_randn(g, M, C)).cuda()
    idx = _links(g, case, M, C)
    L = idx.numel() // 2
    w = r32(_randn(g, 1, C)).cuda()
    bias = r32(_randn(g, 1)).cuda()
    dpred = r32(_randn(g, L)).cuda()
    pred = ops.readout_fwd(_f(H), idx, _f(w), _f(bias)).reshape(-1)
    dH, dw, db = ops.readout_bwd(_f(H), idx, _f(w), _f(dpred).reshape(L, 1))

    i = idx.reshape(L, 2)
    i0, i1 = i[:, 0], i[:, 1]
    Hl, wl, bl = (t.clone().requires_grad_(True) for t in (H, w.reshape(-1), bias))
    ref = (Hl[i0] * Hl[i1] * wl).sum(1) + bl
    (ref * dpred).sum().backward()
    _check(pred, ref, "readout_fwd", [("w ignored", (H[i0] * H[i1]).sum(1) + bias),
                                      ("link l's partner row taken from link l+1", (H[i0] * H[torch.roll(i1, -1)] * w).sum(1) + bias)],
           absum=(H[i0] * H[i1] * w).abs().sum(1) + bias.abs(), nterms=_readout_nterms(C))

    pos = torch.arange(2 * L, device="cuda")
    Gabs = (dpred[pos // 2].unsqueeze(1) * w * H[idx[pos ^ 1]]).abs()
    cnt = torch.zeros(M, dtype=F64, device="cuda").index_add_(0, idx, torch.ones(2 * L, dtype=F64, device="cuda"))
    absG = torch.zeros(M, C, dtype=F64, device="cuda").index_add_(0, idx, Gabs)
    wrongs = [("dpred of link l sent to link l+1", _readout_dH(H, idx, w, torch.roll(dpred, 1))),
              ("a position's own row in place of its partner's", _readout_dH(H, idx, w, dpred, own=True))]
    if bool((cnt > 1).any()):
        r = int(torch.nonzero(cnt > 1)[0])
        last = int((idx == r).nonzero()[-1])
        drop = Hl.grad.clone()
        drop[r] -= dpred[last // 2] * w.reshape(-1) * H[idx[last ^ 1]]
        wrongs.append(("one duplicate position's gradient dropped", drop))
    # a row's positions added in sorted order: cnt - 1 roundings, + 2 inside a term (g*w, * H)
    _check(dH, Hl.grad, "readout_bwd dH", wrongs, absum=(cnt.unsqueeze(1) + 1) * absG, nterms=1)
    P = dpred.unsqueeze(1) * H[i0] * H[i1]
    # dw = colsum of g*(H0*H1): 2 roundings in a term, 7 in an 8-row chain, 2 in fp64
    _check(dw, wl.grad, "readout_bwd dw", [("dpred of link l sent to link l+1", (torch.roll(dpred, -1).unsqueeze(1) * H[i0] * H[i1]).sum(0))]
           + [("row 0 left out", P[1:].sum(0))], absum=P.abs().sum(0), nterms=11)
    # db: fp64 partials of fp32 values, one fp32 store
    _check(db, bl.grad, "readout_bwd db", [("row 0 left out", dpred[1:].sum().reshape(1)),
                                           ("both positions of a link counted", 2 * dpred.sum().reshape(1))],
           absum=dpred.abs().sum().reshape(1), nterms=2)


def _readout_dH(H, idx, w, dpred, own=False):
    L = idx.numel() // 2
    pos = torch.arange(2 * L, device="cuda")
    G = dpred[pos // 2].unsqueeze(1) * w * H[idx[pos if own else pos ^ 1]]
    return torch.zeros_like(H).index_add_(0, idx, G)


# ------------------------------------------------------------------------------------------------ column sums

@pytest.mark.parametrize("M", [1, 2, 7, 1009, "cap"])
@pytest.mark.parametrize("C", CS)
def test_colsum(ops, C, M):
    M = _cap_rows(C) if M == "cap" else M
    g = _gen("colsum", C, M)
    x = _gn_input(g, M, C)
    ref = x.sum(0)
    # nterms 10: 7 adds of an 8-row fp32 chain + 3 for the fp64 adds; independent of M
    _check(ops.colsum(_f(x)), ref, "colsum", [("row 0 left out", x[1:].sum(0)), ("last row twice", ref + x[-1])],
           absum=x.abs().sum(0), nterms=10)


def test_colsum_of_a_million_rows_keeps_its_m_independent_bound(ops):
    """10^6 rows: the 8-row fold keeps the error within nterms = 10 roundings of sum |x|, while one sequential fp32 sum of the
    same columns breaks that bound - what the fold into double is for."""
    M, C = 1_000_003, 32
    g = _gen("colsum-1e6")
    x = r32(1.0 + 0.5 * torch.rand(M, C, generator=g, dtype=F64))
    x[:, 1] *= -3e2
    xd = x.cuda()
    ref = xd.sum(0)
    absum = xd.abs().sum(0)
    got = ops.colsum(_f(xd))
    seq = torch.from_numpy(np.cumsum(x.float().numpy(), axis=0, dtype=np.float32)[-1].astype(np.float64)).cuda()
    # nterms 10: 7 adds of an 8-row fp32 chain + 3 for the fp64 adds
    _check(got, ref, "colsum 1e6 rows", [("one sequential fp32 sum", seq), ("row 0 left out", ref - xd[0])], absum=absum, nterms=10)
    broken = int(((seq - ref).abs() > 10 * U * absum).sum())
    assert broken >= C // 2, f"a sequential fp32 sum breaks the bound in only {broken} of {C} columns"


# ------------------------------------------------------------------------------------------------ LayerNorm

def _ln_input(g, M, C):
    """Rows by m % 3: plain, constant, offset 1e3."""
    z = _randn(g, M, C)
    k = torch.arange(M) % 3
    z[k == 1] = 0.375 * (1 + torch.arange(M)[k == 1].to(F64) % 5).unsqueeze(1)
    z[k == 2] += 1e3
    return r32(z).cuda()


def _ln_keep(ops, M, C, p, seed):
    """The device's LayerNorm dropout mask at (seed, shape): kept where the output at p is nonzero, read on a probe input whose
    normalised values are never 0 (row = 0..C-1: the mean (C-1)/2 is no integer), the kept value the fp32 1/(1-p)."""
    probe = torch.arange(C, dtype=torch.float32, device="cuda").repeat(M, 1)
    y0, _ = ops.bias_layernorm_fwd(probe, None, EPS, 0.0, seed)
    yp, _ = ops.bias_layernorm_fwd(probe, None, EPS, p, seed)
    assert bool((y0 != 0).all())
    inv_keep = float(np.float32(1) / (np.float32(1) - np.float32(p)))
    return (yp != 0).double() * inv_keep


@pytest.mark.parametrize("p", [0.0, 0.3, 0.5])
@pytest.mark.parametrize("M,with_bias", [(1, True), (7, False), (10007, True)])
@pytest.mark.parametrize("C", CS)
def test_bias_layernorm(ops, C, M, with_bias, p):
    """bias_layernorm_fwd / _bwd: y = dropout(LayerNorm(z + bias)) without affine parameters, stats = (mean, inv_std) per row."""
    g = _gen("ln", C, M, with_bias, p)
    z = _ln_input(g, M, C)
    bias = r32(_randn(g, C)).cuda() if with_bias else torch.zeros(C, dtype=F64, device="cuda")
    gout = r32(_randn(g, M, C)).cuda()
    keep = _ln_keep(ops, M, C, p, SEED) if p > 0 else torch.ones_like(z)
    if p > 0:
        _mask_sanity([keep], p, [(keep, _ln_keep(ops, M, C, p, SEED + 1))])
        assert torch.equal(keep, _ln_keep(ops, M, C, p, SEED))
    bptr = _f(bias) if with_bias else None
    y, stats = ops.bias_layernorm_fwd(_f(z), bptr, EPS, p, SEED)
    dz = ops.bias_layernorm_bwd(_f(gout), _f(z), bptr, stats, p, SEED)
    if p > 0:
        y0, _ = ops.bias_layernorm_fwd(_f(z), bptr, EPS, 0.0, SEED)
        assert bool((y[keep == 0] == 0).all()) and bool((y[(keep > 0) & (y0 != 0)] != 0).all())

    def ln(zz, bb, kk, unbiased=False):
        u = zz + bb
        mean = u.mean(1, keepdim=True)
        d = u - mean
        var = (d * d).sum(1, keepdim=True) / (C - 1 if unbiased else C)
        inv = (var + EPS).rsqrt()
        return d * inv * kk, mean, inv

    zl = z.clone().requires_grad_(True)
    ref, mean, inv = ln(zl, bias, keep)
    (ref * gout).sum().backward()
    u = z + bias
    ua = z.abs() + bias.abs()
    d = (u - mean.detach()).abs()
    mean, inv, ref = mean.detach(), inv.detach(), ref.detach()
    lanes = -(-C // 128)
    # mean: 1 rounding in z + bias, 2 in a float4's pairwise sum, a lane's chain over its `lanes` float4, a 5-level xor tree, / C
    nt_m = 9 + lanes
    e_m = nt_m * U * ua.sum(1, keepdim=True) / C
    # sum (u - mean)^2: each difference is off by the rounding of z + bias and its own (U (|u| + d)), the square's rounding, then
    # the sum's roundings as for the mean; a mean that is off by e_m adds C e_m^2 (second order: sum (u - mean) = 0)
    e_q = 2 * U * (d * (ua + d)).sum(1, keepdim=True) + nt_m * U * (d * d).sum(1, keepdim=True) + 3 * C * e_m ** 2
    var = (d * d).sum(1, keepdim=True) / C
    e_inv = 0.5 * inv ** 3 * (e_q / C + 2 * U * (var + EPS)) + 2 * U * inv
    no_bias = ln(z, torch.zeros_like(bias), keep)
    _check(stats, torch.cat((mean, inv), 1), "bias_layernorm stats",
           [("variance with C - 1", torch.cat((mean, ln(z, bias, keep, True)[2]), 1))]
           + ([("bias left out", torch.cat((no_bias[1], no_bias[2]), 1))] if with_bias else []),
           atol=torch.cat((e_m, e_inv), 1))
    e_n = inv * (U * (ua + d) + e_m) + d * e_inv        # the device's n = (u - mean) * inv from its fp32 statistics
    wrongs = [("variance with C - 1", ln(z, bias, keep, True)[0])]
    if p > 0:
        wrongs.append(("dropout mask ignored", ln(z, bias, torch.ones_like(z))[0]))
    # 2 roundings: n's product, the mask's
    _check(y, ref, "bias_layernorm_fwd", wrongs, atol=keep * e_n, absum=keep * d * inv, nterms=2)

    gp = gout * keep
    n = (u - mean) * inv
    s1, s2 = gp.sum(1, keepdim=True) / C, (gp * n).sum(1, keepdim=True) / C
    # the row sums of g' and g'*n: 1 (mask product) + 1 (g'*n) + the mean's order (nt_m - 1); then / C
    E_s1 = (nt_m + 1) * U * gp.abs().sum(1, keepdim=True) / C
    E_s2 = (nt_m + 2) * U * (gp * n).abs().sum(1, keepdim=True) / C + (gp.abs() * e_n).sum(1, keepdim=True) / C
    terms = inv * (gp.abs() + s1.abs() + n.abs() * s2.abs())
    atol = inv * (E_s1 + n.abs() * E_s2 + e_n * s2.abs()) + e_inv * (gp.abs() + s1.abs() + n.abs() * s2.abs())
    zw = z.clone().requires_grad_(True)
    (ln(zw, bias, keep, True)[0] * gout).sum().backward()
    wrongs = [("variance with C - 1", zw.grad)]
    if p > 0:
        zk = z.clone().requires_grad_(True)
        (ln(zk, bias, torch.ones_like(z))[0] * gout).sum().backward()
        wrongs.append(("dropout mask ignored", zk.grad))
    # 4 roundings: g' - m1, n * m2, the difference, * inv
    _check(dz, zl.grad, "bias_layernorm_bwd", wrongs, atol=atol, absum=terms, nterms=4)
