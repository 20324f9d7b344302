"""The row-tile MLP engine (csrc/rb200_tile.cuh) and the weight-gradient kernels after it vs fp64
torch, in every compiled tile configuration, called through the C ABI with no trainer between.

Entry points: rb200_mlp_forward, rb200_mlp_backward, the row paths of rb200_linear_forward and
rb200_linear_backward_dx, rb200_mlp_wgrad (mma.sync, and tcgen05 with RB200_WGRAD_TC=1) with
rb200_grad_reduce, and the fused trainer kernels through their golden cases.

pick_rows_cfg (csrc/rb200_rows.cuh) compiles four tiles: {512, 256} threads x {32, 16} k-chunk.
The KC=16 ones are picked automatically only for hidden widths of several hundred and more;
RB200_FORCE_CFG="nt,kc" (read on every call) forces one, and the `tile_cfg` fixture runs each
case under every one.  A forced tile that does not fit is refused with RB200_E_SMEM.

Comparison rules
  * random operands: per tensor G.rel_err < 1e-5, and per row: the max error over a row relative
    to that row's scale < 1e-5.  The scale of an element is max(|ref|, sum of |terms|) -- what a
    3xTF32 dot product is accurate to even when it cancels to ~0 -- so one wrong row tile of
    small magnitude fails even when the tensor maximum hides it.
  * dyadic operands (weights k/16 with |k| <= 7, inputs k/8): every activation has at most 22
    significant bits and every sum stays below 2^22 quanta (test_dyadic_operands_are_exact checks
    this on the CPU), so the 3xTF32 products and fp32 sums are exact and the kernel must equal
    fp64 bit for bit: a dropped chunk, a wrong column or contaminated padding is a hard failure.
References are computed on the CPU in fp64.
"""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from reagent_b200 import _lib
from tests import golden_util as G

TOL = 1e-5
E_SMEM = -3
ACTS = list(_lib.ACT)  # linear, relu, tanh, leaky_relu, sigmoid, softplus
TILE_CFGS = ["auto", "512,32", "512,16", "256,32", "256,16"]
NAN = float("nan")


@pytest.fixture(params=TILE_CFGS)
def tile_cfg(request, monkeypatch):
    if request.param == "auto":
        monkeypatch.delenv("RB200_FORCE_CFG", raising=False)
    else:
        monkeypatch.setenv("RB200_FORCE_CFG", request.param)
    return request.param


def _tile_rows(cfg):
    """Row-tile height R at batches <= 16 * 148 (where auto prefers the 16-row tiles)."""
    return 32 if cfg.startswith("512") else 16


# ------------------------------------------------------------------------------------------
# fp64 references (torch semantics)
# ------------------------------------------------------------------------------------------
def act64(z, act):
    if act == "relu":
        return torch.relu(z)
    if act == "tanh":
        return torch.tanh(z)
    if act == "leaky_relu":
        return F.leaky_relu(z, 0.01)
    if act == "sigmoid":
        return torch.sigmoid(z)
    if act == "softplus":
        return F.softplus(z)  # beta 1, threshold 20
    assert act == "linear", act
    return z


def act_grad64(z, y, act):
    """d act(z) / dz as torch's backward evaluates it: relu, tanh and sigmoid through the output
    y, leaky_relu and softplus through the pre-activation z (softplus: 1 above the threshold)."""
    if act == "relu":
        return (y > 0).to(z.dtype)
    if act == "tanh":
        return 1.0 - y * y
    if act == "leaky_relu":
        return torch.where(z > 0, torch.ones_like(z), torch.full_like(z, 0.01))
    if act == "sigmoid":
        return y * (1.0 - y)
    if act == "softplus":
        return torch.where(z > 20, torch.ones_like(z), torch.sigmoid(z))
    return torch.ones_like(z)


def forward64(net, x):
    """Pre-activations, outputs and term magnitudes (|h| . |W|^T + |b|) of every layer."""
    zs, hs, mags, h = [], [], [], x
    for W, b, a in zip(net["W"], net["b"], net["acts"]):
        mags.append(h.abs() @ W.abs().t() + b.abs())
        z = h @ W.t() + b
        h = act64(z, a)
        zs.append(z)
        hs.append(h)
    return zs, hs, mags


def dz_chain64(net, zs, hs, dz_last):
    """dZ_{l-1} = (dZ_l . W_l) * act'_{l-1} for every layer, with term magnitudes.  `hs` are the
    outputs the backward reads (the fp32 values a kernel sees), `zs` the pre-activations."""
    L = len(net["W"])
    dz, mag = [None] * L, [None] * L
    dz[L - 1], mag[L - 1] = dz_last, dz_last.abs()
    for l in range(L - 1, 0, -1):
        d = act_grad64(zs[l - 1], hs[l - 1], net["acts"][l - 1])
        dz[l - 1] = (dz[l] @ net["W"][l]) * d
        mag[l - 1] = (dz[l].abs() @ net["W"][l].abs()) * d.abs()
    return dz, mag


def wgrad64(inputs, dz):
    """[(dW, db, |dZ|^T.|A|, sum |dZ|)] per layer: dW_l = dZ_l^T . A_l, db_l = column sums."""
    return [(d.t() @ a, d.sum(0), d.abs().t() @ a.abs(), d.abs().sum(0)) for a, d in zip(inputs, dz)]


# ------------------------------------------------------------------------------------------
# operands
# ------------------------------------------------------------------------------------------
def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _dyadic(shape, g, lo, hi, denom):
    return torch.randint(lo, hi + 1, shape, generator=g).double() / denom


def _randn(shape, g, scale=1.0):
    # fp32 values (then widened): the fp32 copy the kernel gets is the fp64 operand exactly
    return (torch.randn(shape, generator=g) * scale).double()


def make_net(dims, acts, seed, dyadic=False):
    g = _gen(seed)
    W, b = [], []
    for K, N in zip(dims[:-1], dims[1:]):
        if dyadic:
            W.append(_dyadic((N, K), g, -7, 7, 16))
            b.append(_dyadic((N,), g, -7, 7, 16))
        else:
            W.append(_randn((N, K), g, K ** -0.5))
            b.append(_randn((N,), g, 0.1))
    return {"dims": list(dims), "W": W, "b": b, "acts": list(acts)}


def make_input(B, D, seed, dyadic=False):
    g = _gen(seed + 1)
    return _dyadic((B, D), g, -2, 2, 8) if dyadic else _randn((B, D), g)


def _exact_acts(acts):
    return ["linear" if a == "linear" else "relu" for a in acts]


def _cycle(n_layers):
    order = ["relu", "tanh", "leaky_relu", "sigmoid", "softplus"]
    return [order[i % len(order)] for i in range(n_layers - 1)] + ["linear"]


# name: (dims, acts, batch, width of in0 when the input is cat(in0, in1))
MLP_CASES = {
    "7-5": ([7, 5], ["linear"], 1, None),                                   # K < 8, one row
    "33-17-3": ([33, 17, 3], ["relu", "tanh"], 17, None),                     # K = KC + 1
    "31-15-47-6": ([31, 15, 47, 6], ["tanh", "relu", "linear"], 50, None),     # K = KC - 1
    "16-256-257-1": ([16, 256, 257, 1], ["relu", "tanh", "linear"], 33, None),  # 256-column chunks
    # cat input; 5-wide layer written into the ping-pong buffer the 300-wide layer used
    "cat13+3-300-40-5-9": ([16, 300, 40, 5, 9], ["leaky_relu", "sigmoid", "softplus", "linear"],
                           1000, 13),
    "8x32": ([32] * 9, _cycle(8), 100, None),                               # eight layers
}
# exact variants (activations -> relu): eight layers add 32 bits of quantum, too many for fp32
EXACT_MLP_CASES = [c for c in MLP_CASES if c != "8x32"]


def mlp_case(name, exact):
    dims, acts, B, split = MLP_CASES[name]
    s = sum(dims) + len(dims)
    net = make_net(dims, _exact_acts(acts) if exact else acts, s, exact)
    return net, make_input(B, dims[0], s, exact), split


BWD_SEED = 1  # seed of dz_last in the backward cases (the exactness test generates the same)


def make_dz_last(B, N, seed, dyadic=False):
    g = _gen(seed + 2)
    return _dyadic((B, N), g, -2, 2, 8) if dyadic else _randn((B, N), g)


# ------------------------------------------------------------------------------------------
# device side
# ------------------------------------------------------------------------------------------
class DevNet:
    """A network in a CUDA ParamArena plus a NetWorkspace whose buffers start as NaN."""

    def __init__(self, net, batch):
        from reagent_b200.models.arena import ParamArena
        from reagent_b200.training.workspace import NetWorkspace

        self.net = net
        self.arena = ParamArena(net["dims"], [_lib.ACT[a] for a in net["acts"]])
        self.arena.flat = torch.zeros(self.arena.n, device="cuda")
        for l, (W, b) in enumerate(zip(net["W"], net["b"])):
            self.arena.weight_view(self.arena.flat, l).copy_(W.float())
            self.arena.bias_view(self.arena.flat, l).copy_(b.float())
        self.ws = NetWorkspace(self.arena, batch, "cuda")
        for t in self.ws.hidden + self.ws.dz:
            t.fill_(NAN)
        self.desc = self.arena.desc()
        self.batch = batch

    def param_mask(self):
        """Elements of the arena that are parameters (not alignment padding)."""
        m = torch.zeros(self.arena.n, dtype=torch.bool)
        for l in range(len(self.net["W"])):
            N, K = self.net["dims"][l + 1], self.net["dims"][l]
            m[self.arena.w_off[l]: self.arena.w_off[l] + N * K] = True
            m[self.arena.b_off[l]: self.arena.b_off[l] + N] = True
        return m

    def forward(self, x, split=None):
        """rb200_mlp_forward with save_hidden; returns (rc, out)."""
        if split is None:
            x0, x1, d1 = x.float().cuda().contiguous(), None, 0
        else:
            x0 = x[:, :split].float().cuda().contiguous()
            x1 = x[:, split:].float().cuda().contiguous()
            d1 = x1.shape[1]
        out = torch.full((self.batch, self.net["dims"][-1]), NAN, device="cuda")
        rc = _lib.lib().rb200_mlp_forward(self.desc, x0.data_ptr(), x0.shape[1],
                                          None if x1 is None else x1.data_ptr(), d1, self.batch,
                                          out.data_ptr(), C.byref(self.ws.c), _lib.cur_stream())
        torch.cuda.synchronize()
        return rc, out

    def backward(self, dz_last):
        dzl = dz_last.float().cuda().contiguous()
        rc = _lib.lib().rb200_mlp_backward(self.desc, dzl.data_ptr(), self.batch,
                                           C.byref(self.ws.c), _lib.cur_stream())
        torch.cuda.synchronize()
        return rc


def _cmp(out, ref, mag, exact, what, tensor_tol=TOL):
    got = out.detach().double().cpu()
    assert got.shape == ref.shape, (what, tuple(got.shape), tuple(ref.shape))
    assert bool(torch.isfinite(got).all()), (what, "non-finite (unwritten?) elements",
                                             int((~torch.isfinite(got)).sum()))
    if exact:
        bad = got != ref
        if bool(bad.any()):
            i = tuple(int(v) for v in bad.nonzero()[0])
            raise AssertionError(f"{what}: {int(bad.sum())} elements differ from fp64, first at "
                                 f"{i}: {float(got[i])!r} vs {float(ref[i])!r}")
        return
    err = G.rel_err(got, ref)
    assert err < tensor_tol, (what, "rel_err", err)
    scale = torch.maximum(ref.abs(), mag).reshape(ref.shape[0], -1).amax(1).clamp_min(1e-30)
    row = (got - ref).abs().reshape(ref.shape[0], -1).amax(1) / scale
    assert float(row.max()) < TOL, (what, "row", int(row.argmax()), float(row.max()))


def _check_forward(net, x, split, exact, what=""):
    dn = DevNet(net, x.shape[0])
    rc, out = dn.forward(x, split)
    _lib.check(rc, "rb200_mlp_forward")
    _, hs, mags = forward64(net, x)
    for l, h in enumerate(dn.ws.hidden):
        _cmp(h, hs[l], mags[l], exact, f"{what} hidden[{l}]")
    _cmp(out, hs[-1], mags[-1], exact, f"{what} out")


def _check_backward(net, x, exact, seed, what=""):
    """ws.hidden holds the fp64 forward rounded to fp32, so both sides apply the same
    activation masks and only the backward is under test."""
    B, L = x.shape[0], len(net["W"])
    dn = DevNet(net, B)
    zs, hs, _ = forward64(net, x)
    for l in range(L - 1):
        dn.ws.hidden[l].copy_(hs[l].float())
    h32 = [h.float().double() for h in hs]
    dz_last = make_dz_last(B, net["dims"][-1], seed, exact)
    sentinel = -777.25
    dn.ws.dz[L - 1].fill_(sentinel)  # dz_last comes from its own buffer; this one stays put
    _lib.check(dn.backward(dz_last), "rb200_mlp_backward")
    dz, mag = dz_chain64(net, zs, h32, dz_last)
    for l in range(L - 1):
        _cmp(dn.ws.dz[l], dz[l], mag[l], exact, f"{what} dz[{l}]")
    assert bool((dn.ws.dz[L - 1] == sentinel).all()), f"{what} ws.dz[L-1] was written"


# ------------------------------------------------------------------------------------------
# CPU: the oracle itself, and the preconditions of the exact cases
# ------------------------------------------------------------------------------------------
def test_fp64_helpers_match_autograd():
    """forward64 / dz_chain64 / wgrad64 against torch.autograd in float64, all six activations."""
    dims = [6, 9, 8, 7, 6, 5, 4]
    acts = ["relu", "tanh", "leaky_relu", "sigmoid", "softplus", "linear"]
    net = make_net(dims, acts, 3)
    g = _gen(4)
    x = _randn((11, dims[0]), g, 3.0)
    # softplus pre-activations past the threshold and far below 0
    net["b"][4] = torch.tensor([30.0, -16.0, -9.0, 0.5, 25.0], dtype=torch.float64)
    Ws = [W.clone().requires_grad_(True) for W in net["W"]]
    bs = [b.clone().requires_grad_(True) for b in net["b"]]
    h, zt = x, []
    for W, b, a in zip(Ws, bs, acts):
        z = h @ W.t() + b
        z.retain_grad()
        zt.append(z)
        h = act64(z, a)
    dz_last = _randn((11, dims[-1]), g)
    (zt[-1] * dz_last).sum().backward()

    zs, hs, _ = forward64(net, x)
    for a, b in zip(zs, zt):
        assert torch.equal(a, b.detach())
    assert torch.equal(hs[-1], h.detach())
    dz, _ = dz_chain64(net, zs, hs, dz_last)
    for l, z in enumerate(zt):
        assert torch.allclose(dz[l], z.grad, rtol=1e-12, atol=1e-15), l
    for l, (dW, db, _, _) in enumerate(wgrad64([x] + hs[:-1], dz)):
        assert torch.allclose(dW, Ws[l].grad, rtol=1e-12, atol=1e-15), l
        assert torch.allclose(db, bs[l].grad, rtol=1e-12, atol=1e-15), l


def _low_bit(t):
    """Exponent of the lowest set bit of every nonzero element (fp64, exact)."""
    t = t[t != 0].abs()
    m, e = torch.frexp(t)
    M = (m * 2.0 ** 53).long()
    tz = torch.log2((M & -M).double()).round().long()
    return e.long() - 53 + tz


def _sig_bits(t):
    t = t[t != 0]
    if t.numel() == 0:
        return 0
    _, e = torch.frexp(t.abs())
    return int((e.long() - _low_bit(t)).max())


def _assert_exact_dot(a, w, bias, what):
    """a . w^T (+ bias) is exact in 3xTF32 with fp32 sums: one factor fits TF32 (11 significant
    bits, so its low part is 0), the other 22 (so its hi + lo split is exact), bias is on the
    product grid, and |terms| summed stays below 2^22 quanta (every partial sum exact)."""
    ba, bw = _sig_bits(a), _sig_bits(w)
    assert min(ba, bw) <= 11 and max(ba, bw) <= 22, (what, "significant bits", ba, bw)
    if not bool((a != 0).any()) or not bool((w != 0).any()):
        return
    q = 2.0 ** int(_low_bit(a).min() + _low_bit(w).min())
    mag = a.abs() @ w.abs().t()
    if bias is not None:
        assert bool((torch.remainder(bias, q) == 0).all()), (what, "bias off the grid")
        mag = mag + bias.abs()
    assert float(mag.max()) / q <= 2.0 ** 22, (what, "quanta", float(mag.max()) / q)


@pytest.mark.parametrize("case", EXACT_MLP_CASES)
def test_dyadic_operands_are_exact(case):
    net, x, _ = mlp_case(case, True)
    zs, hs, _ = forward64(net, x)
    for l, a in enumerate([x] + hs[:-1]):
        _assert_exact_dot(a, net["W"][l], net["b"][l], f"fwd layer {l}")
    dz, _ = dz_chain64(net, zs, hs, make_dz_last(x.shape[0], net["dims"][-1], BWD_SEED, True))
    for l in range(len(dz) - 1, 0, -1):
        _assert_exact_dot(dz[l], net["W"][l].t(), None, f"bwd layer {l}")


def test_dyadic_operands_are_exact_other_kernels():
    for act in ACTS:
        net, _, _, dz_last = deriv_case(act)
        _assert_exact_dot(dz_last, net["W"][1].t(), None, f"derivative case {act}")
    for B, K, N, _, _ in LIN_FWD_CASES:
        W, b, x = lin_fwd_case(B, K, N, True)
        _assert_exact_dot(x, W, b, f"linear fwd {B, K, N}")
    for K, N in LIN_BWD_SHAPES:
        W, dz, _ = lin_bwd_case(K, N, True)
        _assert_exact_dot(dz, W.t(), None, f"linear bwd {K, N}")
    for B in WGRAD_EXACT_BATCHES:
        _, inputs, dz = wgrad_case(B, True)
        for l, (a, d) in enumerate(zip(inputs, dz)):
            _assert_exact_dot(d.t(), a.t(), None, f"wgrad B={B} layer {l}")
            _assert_exact_dot(d.t(), torch.ones(1, B, dtype=torch.float64), None, f"bias {l}")


# ------------------------------------------------------------------------------------------
# rb200_mlp_forward / rb200_mlp_backward
# ------------------------------------------------------------------------------------------
MLP_PARAMS = [(c, False) for c in MLP_CASES] + [(c, True) for c in EXACT_MLP_CASES]
MLP_IDS = [f"{c}-{'dyadic' if e else 'rand'}" for c, e in MLP_PARAMS]


@pytest.mark.gpu
@pytest.mark.parametrize("case,exact", MLP_PARAMS, ids=MLP_IDS)
def test_mlp_forward(case, exact, tile_cfg):
    net, x, split = mlp_case(case, exact)
    _check_forward(net, x, split, exact, case)


@pytest.mark.gpu
@pytest.mark.parametrize("case,exact", MLP_PARAMS, ids=MLP_IDS)
def test_mlp_backward(case, exact, tile_cfg):
    net, x, _ = mlp_case(case, exact)
    _check_backward(net, x, exact, BWD_SEED, case)


@pytest.mark.gpu
@pytest.mark.parametrize("edge", ["1", "R-1", "R", "R+1"])
def test_mlp_batch_edges(edge, tile_cfg):
    R = _tile_rows(tile_cfg)
    B = {"1": 1, "R-1": R - 1, "R": R, "R+1": R + 1}[edge]
    net = make_net([20, 72, 24, 6], ["relu", "tanh", "linear"], 7)
    x = make_input(B, 20, 7)
    _check_forward(net, x, 11, False, f"B={B}")
    _check_backward(net, x, False, 2, f"B={B}")


@pytest.mark.gpu
@pytest.mark.parametrize("B", [2368, 2369])
def test_mlp_around_row_tile_switch(B):
    """auto takes 16-row tiles up to batch 16 * 148 = 2368 and 32-row tiles above."""
    lib = _lib.lib()
    assert lib.rb200_num_row_tiles(B, 40, 64) == (148 if B == 2368 else 75)
    net = make_net([40, 64, 64, 5], ["relu", "softplus", "linear"], 8)
    x = make_input(B, 40, 8)
    _check_forward(net, x, None, False, f"B={B}")
    _check_backward(net, x, False, 3, f"B={B}")


@pytest.mark.gpu
def test_mlp_config5_critic_widths():
    net = make_net([576, 256, 256, 1], ["relu", "relu", "linear"], 9)
    x = make_input(16384, 576, 9)
    _check_forward(net, x, 570, False, "critic")
    _check_backward(net, x, False, 4, "critic")


@pytest.mark.gpu
def test_mlp_forward_output_width_limit():
    net = make_net([8, 1024], ["linear"], 10)
    _check_forward(net, make_input(20, 8, 10), None, False, "N=1024")
    dn = DevNet(make_net([8, 1025], ["linear"], 10), 20)
    rc, _ = dn.forward(make_input(20, 8, 10))
    assert rc == E_SMEM, rc


# (pass, dims, batch, tiles that fit).  Floats of shared memory: 2 weight stages (9216 each at
# KC=32, 5120 at KC=16) + R x per-row buffers, against 227 KB = 58112 floats:
#   fwd [8,1400,4]: R * (12 + 2*1404 + 8) -> only R=16 with KC=16 (10240 + 45248)
#   bwd [8,980,4]:  R * (3*984 + 8)        -> only R=16 with KC=16 (10240 + 47360)
#   fwd [8,700,4] at B=4096 (auto: R=32):  R=32 needs KC=16 (10240 + 32*1428)
#   bwd [8,700,4] at B=4096: R=32 never fits (32*(3*704+8) = 67840), R=16 fits with either KC
WIDE_CASES = {
    "fwd-1400": ("fwd", [8, 1400, 4], 40, {"auto", "256,16"}),
    "bwd-980": ("bwd", [8, 980, 4], 40, {"auto", "256,16"}),
    "fwd-700-B4096": ("fwd", [8, 700, 4], 4096, {"auto", "512,16", "256,32", "256,16"}),
    "bwd-700-B4096": ("bwd", [8, 700, 4], 4096, {"auto", "256,32", "256,16"}),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(WIDE_CASES))
def test_mlp_wide_hidden_fits_or_refuses(case, tile_cfg):
    """Hidden widths where only the KC=16 tiles fit: auto must pick them and compute the right
    thing; a forced tile that does not fit is refused with RB200_E_SMEM, never replaced."""
    kind, dims, B, fits = WIDE_CASES[case]
    net = make_net(dims, ["tanh", "linear"], 11)
    x = make_input(B, dims[0], 11)
    if tile_cfg in fits:
        if kind == "fwd":
            _check_forward(net, x, None, False, case)
        else:
            _check_backward(net, x, False, 5, case)
        return
    dn = DevNet(net, B)
    rc = dn.forward(x)[0] if kind == "fwd" else dn.backward(make_dz_last(B, dims[-1], 5))
    assert rc == E_SMEM, (tile_cfg, rc)


def deriv_case(act):
    """Two-layer net [4, H, N] with `act` below a linear head; pre-activations of the hidden
    layer are set directly (softplus down to -16).  dz_last and W1 are dyadic, so dz . W1 is
    exact and the kernel's dz[0] / (dz . W1) is its derivative factor times one rounding."""
    B, H, N = 64, 96, 24
    lo, hi = {"softplus": (-16.0, 16.0), "tanh": (-3.0, 3.0), "sigmoid": (-8.0, 8.0)}.get(act, (-8.0, 8.0))
    g = _gen(20 + ACTS.index(act))
    z = (torch.rand(B, H, generator=g) * (hi - lo) + lo).double()
    z[0, :8] = torch.tensor([-16.0, -12.0, -9.0, -5.0, -1.0, 0.25, 5.0, 9.0]).clamp(lo, hi)
    net = make_net([4, H, N], [act, "linear"], 21, dyadic=True)
    return net, z, act64(z, act).float().double(), make_dz_last(B, N, 22, True)


@pytest.mark.gpu
@pytest.mark.parametrize("act", ACTS)
def test_mlp_backward_derivative_factor(act, tile_cfg):
    """Elementwise act' in the backward.  A max-norm check hides an error in small derivatives
    (softplus at x << 0): here every element of dz[0] / (dz . W1) must match act' to 1e-6."""
    net, z, h32, dz_last = deriv_case(act)
    dn = DevNet(net, z.shape[0])
    dn.ws.hidden[0].copy_(h32.float())
    _lib.check(dn.backward(dz_last), "rb200_mlp_backward")
    acc = dz_last @ net["W"][1]
    d = act_grad64(z, h32, act)
    got = dn.ws.dz[0].double().cpu()
    nz = acc != 0
    ratio = got[nz] / acc[nz]
    err = (ratio - d[nz]).abs() / d[nz].abs().clamp_min(1e-300)
    bad = err > 1e-6
    i = int(err.argmax())
    assert not bool(bad.any()), (f"{act}: {int(bad.sum())} of {int(nz.sum())} elements off by "
                                 f"> 1e-6, at x in [{float(z[nz][bad].min())}, "
                                 f"{float(z[nz][bad].max())}]; worst x={float(z[nz][i])}: factor "
                                 f"{float(ratio[i])} vs act' {float(d[nz][i])}")


# ------------------------------------------------------------------------------------------
# rb200_linear_forward / rb200_linear_backward_dx, row-tile paths (batch < 128 or N < 128)
# ------------------------------------------------------------------------------------------
# (B, K, N, act, bias)
LIN_FWD_CASES = [
    (100, 300, 1000, "tanh", True),      # two 512-column blocks, 256-column chunks inside
    (4096, 72, 100, "sigmoid", True),    # N < 128
    (37, 7, 130, "leaky_relu", True),    # K < 8, scalar staging
    (50, 64, 600, "linear", False),      # no bias
]


def lin_fwd_case(B, K, N, exact):
    net = make_net([K, N], ["linear"], 30 + K + N, exact)
    return net["W"][0], net["b"][0], make_input(B, K, 30 + K + N, exact)


@pytest.mark.gpu
@pytest.mark.parametrize("exact", [False, True], ids=["rand", "dyadic"])
@pytest.mark.parametrize("B,K,N,act,bias", LIN_FWD_CASES)
def test_linear_forward_rows(B, K, N, act, bias, exact, tile_cfg):
    W, b, x = lin_fwd_case(B, K, N, exact)
    if exact:
        act = "relu" if act != "linear" else act
    if not bias:
        b = torch.zeros_like(b)
    out = torch.full((B, N), NAN, device="cuda")
    Wd, bd, xd = W.float().cuda(), b.float().cuda(), x.float().cuda()
    rc = _lib.lib().rb200_linear_forward(Wd.data_ptr(), bd.data_ptr() if bias else None, _lib.ACT[act],
                                         K, N, xd.data_ptr(), B, out.data_ptr(), _lib.cur_stream())
    _lib.check(rc, "rb200_linear_forward")
    torch.cuda.synchronize()
    _cmp(out, act64(x @ W.t() + b, act), x.abs() @ W.abs().t() + b.abs(), exact, "linear fwd")


LIN_BWD_SHAPES = [(130, 257), (7, 300), (33, 1100)]  # (K, N); N > 512 takes two dz slabs


def lin_bwd_case(K, N, exact, B=70):
    net = make_net([K, N], ["linear"], 40 + K + N, exact)
    g = _gen(41 + K)
    dz = _dyadic((B, N), g, -2, 2, 8) if exact else _randn((B, N), g)
    pre = (torch.rand(B, K, generator=g) * 8 - 4).double()
    return net["W"][0], dz, pre


@pytest.mark.gpu
@pytest.mark.parametrize("exact", [False, True], ids=["rand", "dyadic"])
@pytest.mark.parametrize("K,N", LIN_BWD_SHAPES)
def test_linear_backward_dx_rows(K, N, exact, tile_cfg):
    """out = (dz . W) * act'(h_prev) for no h_prev and every act_prev (dyadic: relu / linear)."""
    lib = _lib.lib()
    W, dz, pre = lin_bwd_case(K, N, exact)
    B = dz.shape[0]
    Wd, dzd = W.float().cuda(), dz.float().cuda()
    acc, mag = dz @ W, dz.abs() @ W.abs()
    for act in [None] + (["linear", "relu"] if exact else ACTS):
        h = act64(pre, act or "linear").float().double()
        hd = h.float().cuda()
        out = torch.full((B, K), NAN, device="cuda")
        rc = lib.rb200_linear_backward_dx(Wd.data_ptr(), K, N, dzd.data_ptr(),
                                          None if act is None else hd.data_ptr(),
                                          _lib.ACT[act or "linear"], B, out.data_ptr(), _lib.cur_stream())
        _lib.check(rc, "rb200_linear_backward_dx")
        torch.cuda.synchronize()
        d = act_grad64(pre, h, act) if act else torch.ones_like(pre)
        _cmp(out, acc * d, mag * d.abs(), exact, f"linear bwd act_prev={act}")


# ------------------------------------------------------------------------------------------
# rb200_mlp_wgrad + rb200_grad_reduce (not row-tile kernels: RB200_FORCE_CFG does not apply)
# ------------------------------------------------------------------------------------------
WGRAD_DIMS = [261, 130, 7, 3]  # K, N not multiples of 4 or 64; K > 256 (two tcgen05 k-tiles)
WGRAD_EXACT_BATCHES = [31, 300, 4096]


def wgrad_case(B, exact):
    net = make_net(WGRAD_DIMS, ["relu", "relu", "linear"], 50)
    g = _gen(51 + B)
    mk = (lambda s: _dyadic(s, g, -8, 8, 8)) if exact else (lambda s: _randn(s, g))
    inputs = [mk((B, d)) for d in WGRAD_DIMS[:-1]]
    dz = [mk((B, d)) for d in WGRAD_DIMS[1:]]
    return net, inputs, dz


def _wgrad_kernel_env(monkeypatch, kernel):
    if kernel == "tc":
        monkeypatch.setenv("RB200_WGRAD_TC", "1")
    else:
        monkeypatch.delenv("RB200_WGRAD_TC", raising=False)
    monkeypatch.delenv("RB200_DISABLE_TCGEN05", raising=False)


def _ceil_div(a, b):
    return -(-a // b)


def _run_wgrad(dn, a0, splits):
    lib = _lib.lib()
    gpart = torch.full((splits, dn.arena.n), NAN, device="cuda")
    rc = lib.rb200_mlp_wgrad(dn.desc, a0.data_ptr(), dn.batch, C.byref(dn.ws.c), gpart.data_ptr(),
                             splits, _lib.cur_stream())
    _lib.check(rc, "rb200_mlp_wgrad")
    red = torch.full((dn.arena.n,), NAN, device="cuda")
    _lib.check(lib.rb200_grad_reduce(gpart.data_ptr(), splits, dn.arena.n, red.data_ptr(),
                                     _lib.cur_stream()), "rb200_grad_reduce")
    torch.cuda.synchronize()
    return gpart.cpu(), red.cpu()


def _wgrad_checked(dn, a0, splits, ref, exact, what):
    """One wgrad + reduce: slabs all written (empty ones zero), reduce = slab-order fp32 sum,
    result vs fp64, and a second run bit-identical.  Returns the reduced gradient.

    A slab sums its rows into one fp32 accumulator: 4096 zero-mean products in one slab (splits=1)
    measured 2.9e-5 of the tensor's max on the B200 -- 6e-7 of the sum of |terms|, the rounding
    of a correct fp32 sum that cancels, not a kernel error.  Slabs longer than 1024 rows are held
    to 1e-4 per tensor; the per-row bar against the sum of |terms| stays 1e-5 for every slab
    length, and the dyadic cases are exact at B = 4096 in any split."""
    B, mask = dn.batch, dn.param_mask()
    gpart, red = _run_wgrad(dn, a0, splits)
    gp = gpart[:, mask]
    assert not bool(torch.isnan(gp).any()), (what, "unwritten gradient-partial elements")
    rows = _ceil_div(_ceil_div(B, splits), 32) * 32  # rows per slab, as both kernels cut them
    tensor_tol = TOL if rows <= 1024 else 1e-4
    for s in range(splits):
        if s * rows >= B:
            assert bool((gp[s] == 0).all()), (what, "empty slab", s, "not zero")
    acc = gp[0].clone()
    for s in range(1, splits):
        acc = acc + gp[s]
    assert torch.equal(red[mask], acc), (what, "reduce is not the slab-order fp32 sum")
    for l, (dW, db, mW, mb) in enumerate(ref):
        w = red[dn.arena.w_off[l]: dn.arena.w_off[l] + dW.numel()].view_as(dW)
        b = red[dn.arena.b_off[l]: dn.arena.b_off[l] + db.numel()]
        _cmp(w, dW, mW, exact, f"{what} dW[{l}]", tensor_tol)
        _cmp(b.view(-1, 1), db.view(-1, 1), mb.view(-1, 1), exact, f"{what} db[{l}]", tensor_tol)
    gpart2, _ = _run_wgrad(dn, a0, splits)
    assert torch.equal(gpart2[:, mask], gp), (what, "not deterministic")
    return red[mask]


# (batch, splits): "one", rb200_wgrad_splits(B), rb200_wgrad_splits_for(net, B) or a number
WGRAD_CASES = ([(B, k, None) for B in (1, 31, 33, 300, 4096) for k in ("one", "splits", "splits_for")]
               + [(300, "64", None)]  # slabs 10..63 empty
               + [(B, "splits", "32") for B in (33, 300, 4096)])  # RB200_WGRAD_ROWS=32


@pytest.mark.gpu
@pytest.mark.parametrize("B,split_kind,wgrad_rows", WGRAD_CASES)
def test_wgrad_and_reduce(B, split_kind, wgrad_rows, monkeypatch):
    if wgrad_rows:
        monkeypatch.setenv("RB200_WGRAD_ROWS", wgrad_rows)
    else:
        monkeypatch.delenv("RB200_WGRAD_ROWS", raising=False)
    net, inputs, dz = wgrad_case(B, False)
    dn = DevNet(net, B)
    for l in range(len(WGRAD_DIMS) - 2):
        dn.ws.hidden[l].copy_(inputs[l + 1].float())
    for l in range(len(WGRAD_DIMS) - 1):
        dn.ws.dz[l].copy_(dz[l].float())
    a0 = inputs[0].float().cuda()
    ref = wgrad64(inputs, dz)
    lib = _lib.lib()
    got = {}
    for kernel in ("mma", "tc"):
        _wgrad_kernel_env(monkeypatch, kernel)
        splits = {"one": 1, "splits": lib.rb200_wgrad_splits(B),
                  "splits_for": lib.rb200_wgrad_splits_for(dn.desc, B)}.get(split_kind)
        splits = splits if splits is not None else int(split_kind)
        got[kernel] = _wgrad_checked(dn, a0, splits, ref, False, f"{kernel} splits={splits}")
    assert G.rel_err(got["tc"], got["mma"]) < TOL


@pytest.mark.gpu
@pytest.mark.parametrize("B", WGRAD_EXACT_BATCHES)
def test_wgrad_dyadic_is_exact(B, monkeypatch):
    monkeypatch.delenv("RB200_WGRAD_ROWS", raising=False)
    net, inputs, dz = wgrad_case(B, True)
    dn = DevNet(net, B)
    for l in range(len(WGRAD_DIMS) - 2):
        dn.ws.hidden[l].copy_(inputs[l + 1].float())
    for l in range(len(WGRAD_DIMS) - 1):
        dn.ws.dz[l].copy_(dz[l].float())
    a0 = inputs[0].float().cuda()
    ref = wgrad64(inputs, dz)
    for kernel in ("mma", "tc"):
        _wgrad_kernel_env(monkeypatch, kernel)
        splits = _lib.lib().rb200_wgrad_splits_for(dn.desc, B)
        _wgrad_checked(dn, a0, splits, ref, True, f"{kernel} splits={splits}")


# ------------------------------------------------------------------------------------------
# fused trainer kernels under every tile: the golden cases at the bars of their home tests
# ------------------------------------------------------------------------------------------
FUSED_CASES = [("sac", "sac_twin_odd_dims"), ("td3", "td3_twin"),
               ("dqn_rows", "dqn_timediff_odd_dims"), ("dqn_rows", "dqn_dueling_double"),
               ("pdqn", "pdqn_double_mse"), ("c51", "c51_double")]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,name", FUSED_CASES, ids=[n for _, n in FUSED_CASES])
def test_fused_kernels_golden(kind, name, tile_cfg, monkeypatch):
    from tests import test_actor_critic_gpu as AC
    from tests import test_dqn_gpu as D
    from tests import test_pdqn_c51_gpu as P

    if kind == "sac":
        AC.test_sac_fast_path_matches_reference(name)
    elif kind == "td3":
        AC.test_td3_matches_reference(name, True)
    elif kind == "dqn_rows":
        D.test_dqn_fast_path_matches_reference(name, "rows", monkeypatch)
    elif kind == "pdqn":
        P.test_parametric_dqn_matches_reference(name, True)
    else:
        P.test_c51_matches_reference(name, True)
