"""GPU: every LayerNorm implementation against float64 on rows that are hard for the row statistics, not only on
centred ``randn`` rows.

The rows come from the layer in front of the LayerNorm (its weight ``W`` and bias ``b``), one family per
parametrisation:

* ``centred``: the distribution the other tests use (control);
* ``outlier<j>``: the other columns at std ~1, ``b[j] = +-40`` for one ``j`` in {0, 77, 127} - one unit of the previous
  layer with a large bias, an ordinary trained-network state.  ``max|z - mean| / std`` is ~11 there, so LayerNorm is
  well conditioned and an fp32 kernel owes 1e-5; a one-pass ``E[z^2] - E[z]^2`` loses ~7 bits on these rows, shifted by
  the first element or not (column 0 is the case for that shift, the other two keep the test from encoding one
  algorithm);
* ``offset``: ``b += 30`` in every column (the row's centre far from 0);
* ``chunk``: columns 0..31 ``+50`` (aimed at per-32-column partial statistics);
* ``tiny``: the LayerNorm input's std ~3e-3, so the variance is comparable to ``eps`` (pins where ``eps`` enters);
* ``constant``: ``W = 0`` and a dyadic bias equal in every column: ``var = 0``, the output must be finite and equal
  ``beta (+ residual)`` to 1e-6.

Every form that runs a LayerNorm is covered: each specialisation of the chained kernel (csrc/tc_chain.cu), the 3xTF32
linear's LayerNorm epilogue (csrc/tc_linear.cu), ``ops.layer_norm`` forward and backward on its vector and scalar
paths (csrc/dense.cu), the training tails of tc_train.py, and one training step of the whole model.  The bars hold per
row, so one bad row cannot hide in a large tensor: LayerNorm output ``max|y - y64| <= 1e-5 max|y64|`` over the row,
``rstd`` 1e-5 relative, ``mean`` within ``1e-6 max|z|`` of the row, a stashed LayerNorm input 1e-5 per row, ``dz``
1e-5 per row, ``dgamma`` / ``dbeta`` 1e-5 rel-L2.  References are float64 on the device, in row chunks."""
import pytest
import torch

pytestmark = pytest.mark.gpu

EPS = 1e-5
FAMILIES = ["centred", "outlier0", "outlier77", "outlier127", "offset", "chunk", "tiny", "constant"]
M_TILES = 256 * 74 * 2 + 77          # several tiles per CTA pair, ragged last tile
M_TRAIN = 4_194_304                  # node rows of a 256-graph resize-128 micro-batch
CHUNK = 1 << 18                      # rows per float64 reference chunk
CONST = 2.75                         # the constant rows' value (dyadic: every sum of it is exact)
_f64 = torch.float64


# ---- row families ------------------------------------------------------------------------------------------------
def _family(fam, W, b, h64):
    """The last layer before the LayerNorm for family ``fam``: ``(W [D, K], b [D])`` fp32 on the device, given a
    sample of its float64 input rows ``h64``."""
    D = W.shape[0]
    if fam == "centred":
        return W, b
    if fam == "constant":
        return torch.zeros_like(W), torch.full_like(b, CONST)
    s0 = float((h64[:65536] @ W.double().t()).std(1).mean())      # the rows' spread through W
    b = b.clone()
    if fam.startswith("outlier"):
        j = {"outlier0": 0, "outlier77": 77 if D > 77 else D // 2, "outlier127": D - 1}[fam]
        b *= 0.1
        b[j] = -40.0 if fam == "outlier77" else 40.0
        return W / s0, b
    if fam == "offset":
        return W, b + 30.0
    if fam == "chunk":
        b[:32] += 50.0
        return W, b
    assert fam == "tiny"
    return W * (3e-3 / s0), b * 1e-2


def _lin64(x64, W, b):
    return x64 @ W.double().t() + b.double()


def _ln64(z64, gamma, beta):
    return torch.nn.functional.layer_norm(z64, (z64.shape[1],), gamma.double(), beta.double(), EPS)


# ---- per-row bars ------------------------------------------------------------------------------------------------
def _bad_rows(what, err, scale, bar):
    bad = err > bar
    worst = float((err / scale.clamp_min(1e-30)).max())
    assert not bool(bad.any()), (f"{what}: {int(bad.sum())} of {bad.numel()} rows above the bar, worst row error "
                                 f"{worst:.2e} relative to the row")
    return worst


def _check_ln(what, fam, got, ln64, add64=None):
    """``got`` = LayerNorm output (+ ``add64``) per row.  The bar is relative to the row's largest LayerNorm output;
    with an addend it also allows the rounding of the final fp32 add."""
    assert bool(torch.isfinite(got).all()), f"{what}: non-finite output"
    ref = ln64 if add64 is None else ln64 + add64
    err = (got.double() - ref).abs().amax(1)
    scale = ln64.abs().amax(1)
    bar = (1e-6 if fam == "constant" else 1e-5) * scale
    if add64 is not None:
        bar = bar + 2.0 ** -24 * ref.abs().amax(1)
    return _bad_rows(what + " LayerNorm output", err, scale, bar)


def _check_stats(what, z64, mean=None, rstd=None, z=None):
    """Saved / stashed row statistics and LayerNorm input against float64."""
    zmax = z64.abs().amax(1)
    if z is not None:
        _bad_rows(what + " stashed z", (z.double() - z64).abs().amax(1), zmax, 1e-5 * zmax)
    if mean is not None:
        _bad_rows(what + " mean", (mean.double() - z64.mean(1)).abs(), zmax, 1e-6 * zmax)
    if rstd is not None:
        rs = torch.rsqrt(z64.var(1, unbiased=False) + EPS)
        _bad_rows(what + " rstd", (rstd.double() - rs).abs(), rs, 1e-5 * rs)


def _rel_l2(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _affine(gen):
    gamma = torch.rand(128, generator=gen, device="cuda") + 0.5
    beta = torch.randn(128, generator=gen, device="cuda") * 0.2
    return gamma, beta


# ---- chained kernel (csrc/tc_chain.cu), one case per specialisation chain::launch picks ----------------------------
CHAIN_FORMS = [
    "edge",             # 3 layers, indexed gather0 / gather1, residual by row (Spec<1>, two-tile kernel)
    "node_addend",      # 3 layers, plain addend, residual by row (Spec<2>)
    "prestage",         # first operand relu(R[cls] + P[i0] + Q[i1] + b0), 2 layers, residual by table (Spec<7>)
    "edge_slots1", "edge_slots2", "prestage_slots1", "prestage_slots2",     # paired destination slots / pair sums
    "node2", "node2_agg", "node2_paired",      # two-operand node form: plain, aggregating loader, paired slot rows
    "narrow",           # encoder form: narrow first layer folded in, 2 layers
    "two_layer_res", "two_layer",             # 2 layers with / without a residual (class-table encoder)
    "generic",          # 3 layers, residual by table: the generic Spec<0>
    "stash_edge", "stash_node",               # training forward with the stash
]


def _chain_case(form, M, gen):
    """``(h64, (W, b), run, res64, kind, M, pad)``: float64 input rows of the last layer, the layer itself, ``run(W, b,
    gamma, beta)`` -> output (and the stash), the float64 residual rows, how output rows map to slot rows, the slot
    count, and the padding slots."""
    from graphnet_classifier_b200 import ops
    dev = "cuda"

    def rn(*s, scale=1.0):
        return torch.randn(*s, generator=gen, device=dev) * scale

    def layer():
        return rn(128, 128, scale=1 / 11), rn(128, scale=0.3)

    L0, L1, L2 = layer(), layer(), layer()
    R = 3000
    kind = "rows"
    slots = form.startswith(("edge_slots", "prestage_slots"))
    if slots:
        M += M % 2
        kind = "slots" + form[-1]
    if form in ("edge", "generic", "stash_edge", "edge_slots1", "edge_slots2"):
        A = rn(M, 128)
        P = rn(R, 128)
        if slots:                     # slot 2v, 2v + 1 belong to node v; a negative gather0 index marks a padding slot
            Q = rn(M // 2, 128)
            i0 = torch.randint(0, R, (M,), generator=gen, device=dev).int()
            i0[torch.rand(M, generator=gen, device=dev) < 0.15] = -1
            i1 = (torch.arange(M, device=dev) >> 1).int()
            A[i0 < 0] = 0.0
        else:
            Q = rn(R, 128)
            i0 = torch.randint(0, R, (M,), generator=gen, device=dev).int()
            i1 = torch.randint(0, R, (M,), generator=gen, device=dev).int()
        pre = P.double()[i0.long().clamp_min(0)] + Q.double()[i1.long()]
        h64 = torch.relu(_lin64(torch.relu(_lin64(A.double(), *L0) + pre), *L1))
        kw = dict(gather0=(P, i0), gather1=(Q, i1))
        if form == "generic":
            tab, ti = rn(5, 128), torch.randint(0, 5, (M,), generator=gen, device=dev).int()
            kw["residual"], res64 = (tab, ti), tab.double()[ti.long()]
        else:
            kw["residual"], res64 = A, A.double()
        if slots:
            kw["edge_slots"] = int(form[-1])
        first, rest = A, [L0, L1]
    elif form in ("node_addend", "stash_node"):
        A, T, h = rn(M, 128), rn(M, 128), rn(M, 128)
        h64 = torch.relu(_lin64(torch.relu(_lin64(A.double(), *L0) + T.double()), *L1))
        kw, res64, first, rest = dict(gather0=(T, None), residual=h), h.double(), A, [L0, L1]
    elif form.startswith("prestage"):
        Rt, e_tab = rn(4, 128), rn(4, 128)
        cls = torch.randint(0, 4, (M,), generator=gen, device=dev).int()
        P = rn(R, 128)
        i0 = torch.randint(0, R, (M,), generator=gen, device=dev).int()
        if slots:
            Q = rn(M // 2, 128)
            i0[torch.rand(M, generator=gen, device=dev) < 0.15] = -1
            i1 = (torch.arange(M, device=dev) >> 1).int()
        else:
            Q = rn(R, 128)
            i1 = torch.randint(0, R, (M,), generator=gen, device=dev).int()
        b0 = rn(128, scale=0.2)
        a1 = torch.relu(Rt.double()[cls.long()] + P.double()[i0.long().clamp_min(0)] + Q.double()[i1.long()] + b0.double())
        h64 = torch.relu(_lin64(a1, *L1))
        kw = dict(pre=(Rt, cls, b0), gather0=(P, i0), gather1=(Q, i1), residual=(e_tab, cls))
        if slots:
            kw["edge_slots"] = int(form[-1])
        res64, first, rest = e_tab.double()[cls.long()], None, [L1]
    elif form.startswith("node2"):
        h = rn(M, 128)
        V0, c0 = rn(128, 256, scale=1 / 16), rn(128, scale=0.2)
        kw = dict(operand2=(h, V0[:, 0:128]), residual=h)
        if form == "node2":
            first = rn(M, 128, scale=2.0)
            agg64 = first.double()
        elif form == "node2_agg":     # in-degree 0, 1 or 2, edge ids in any order
            deg = torch.randint(0, 3, (M,), generator=gen, device=dev)
            rowptr = torch.zeros(M + 1, dtype=torch.int32, device=dev)
            rowptr[1:] = torch.cumsum(deg, 0).int()
            E = int(deg.sum())
            eid = torch.randperm(E, generator=gen, device=dev).int()
            first = rn(E, 128, scale=2.0)
            agg64 = torch.zeros(M, 128, dtype=_f64, device=dev)
            agg64.index_add_(0, torch.repeat_interleave(torch.arange(M, device=dev), deg), first.double()[eid.long()])
            kw["agg"] = (rowptr, eid)
        else:
            first = rn(2 * M, 128, scale=2.0)
            agg64 = first.double()[0::2] + first.double()[1::2]
            kw["paired"] = True
        a1 = torch.relu(torch.cat([h.double(), agg64], 1) @ V0.double().t() + c0.double())
        h64 = torch.relu(_lin64(a1, *L1))
        res64, rest = h.double(), [(V0[:, 128:256], c0), L1]
    elif form == "narrow":
        k = 3
        first = torch.rand(M, k, generator=gen, device=dev) * 255
        Wn = (torch.rand(128, k, generator=gen, device=dev) - 0.5) / k ** 0.5
        bn = rn(128, scale=0.3)
        h64 = torch.relu(_lin64(torch.relu(_lin64(first.double(), Wn, bn)), *L1))
        kw, res64, rest = dict(narrow=(Wn, bn)), None, [L1]
    else:
        assert form in ("two_layer_res", "two_layer")
        first = rn(M, 128)
        h64 = torch.relu(_lin64(first.double(), *L1))
        kw, rest = {}, [L1]
        res64 = None
        if form == "two_layer_res":
            r = rn(M, 128)
            kw["residual"], res64 = r, r.double()

    def run(W, b, gamma, beta):
        stash = None
        if form.startswith("stash"):
            stash = tuple(torch.full((M, 128), float("nan"), device=dev) for _ in range(3)) + \
                tuple(torch.full((M,), float("nan"), device=dev) for _ in range(2))
        y = ops.tc_mlp_chain(first, rest + [(W, b)], gamma=gamma, beta=beta, eps=EPS, stash=stash, **kw)
        return y, stash

    return h64, L2, run, res64, kind, M, (i0 < 0 if slots else None)


def _check_slots(what, fam, kind, y, ln64, res64, pad):
    """Slot-row forms: padding slots are +0.0; ``edge_slots=2`` returns the per-node sums ``(0 + y[2v]) + y[2v + 1]``."""
    if kind == "slots1":
        assert bool((y[pad].view(torch.int32) == 0).all()), f"{what}: padding slots are not +0.0"
        return _check_ln(what, fam, y[~pad], ln64[~pad], res64[~pad])
    assert bool(torch.isfinite(y).all()), f"{what}: non-finite output"
    keep = (~pad).double()[:, None]
    ref = (ln64 + res64) * keep
    node = ref[0::2] + ref[1::2]
    ln_abs = ln64.abs() * keep
    scale = torch.maximum(ln_abs[0::2], ln_abs[1::2]).amax(1)
    err = (y.double() - node).abs().amax(1)
    bar = (1e-6 if fam == "constant" else 1e-5) * scale + 2.0 ** -23 * torch.maximum(ref[0::2].abs(), ref[1::2].abs()).amax(1)
    return _bad_rows(what + " pair sums", err, scale, bar)


@pytest.mark.parametrize("fam", FAMILIES)
@pytest.mark.parametrize("form", CHAIN_FORMS)
def test_chain_layernorm_rows(libgnc, form, fam):
    gen = torch.Generator(device="cuda").manual_seed(CHAIN_FORMS.index(form) * 100 + FAMILIES.index(fam))
    h64, (W, b), run, res64, kind, M, pad = _chain_case(form, M_TILES, gen)
    gamma, beta = _affine(gen)
    W, b = _family(fam, W, b, h64)
    y, stash = run(W, b, gamma, beta)
    z64 = _lin64(h64, W, b)
    del h64
    ln64 = _ln64(z64, gamma, beta)
    what = f"chain {form} / {fam}"
    if kind == "rows":
        worst = _check_ln(what, fam, y, ln64, res64)
    else:
        worst = _check_slots(what, fam, kind, y, ln64, res64, pad)
    if stash is not None:
        _, _, z, mean, rstd = stash
        _check_stats(what, z64, mean, rstd, z)
    print(f"LN-ROWS chain {form:16s} {fam:9s} worst row error {worst:.2e}")


# ---- the 3xTF32 linear's LayerNorm epilogue (csrc/tc_linear.cu) ---------------------------------------------------
TC_LINEAR_FORMS = ["none", "row", "table", "ln_save"]


@pytest.mark.parametrize("fam", FAMILIES)
@pytest.mark.parametrize("res", TC_LINEAR_FORMS)
def test_tc_linear_layernorm_rows(libgnc, res, fam):
    from graphnet_classifier_b200 import ops
    gen = torch.Generator(device="cuda").manual_seed(1000 + TC_LINEAR_FORMS.index(res) * 100 + FAMILIES.index(fam))
    M = M_TILES
    A = torch.relu(torch.randn(M, 128, generator=gen, device="cuda") * 2)
    W, b = torch.randn(128, 128, generator=gen, device="cuda") / 11, torch.randn(128, generator=gen, device="cuda") * 0.3
    gamma, beta = _affine(gen)
    h64 = A.double()
    W, b = _family(fam, W, b, h64)
    kw, res64, save = {}, None, None
    if res in ("row", "ln_save"):
        r = torch.randn(M, 128, generator=gen, device="cuda")
        kw["residual"], res64 = r, r.double()
    elif res == "table":
        tab, ti = torch.randn(7, 128, generator=gen, device="cuda"), torch.randint(0, 7, (M,), generator=gen, device="cuda").int()
        kw["residual"], res64 = (tab, ti), tab.double()[ti.long()]
    if res == "ln_save":
        save = (torch.full((M, 160), float("nan"), device="cuda")[:, :128], torch.full((M,), float("nan"), device="cuda"),
                torch.full((M,), float("nan"), device="cuda"))
        kw["ln_save"] = save
    y = ops.tc_linear(A, W, bias=b, gamma=gamma, beta=beta, eps=EPS, **kw)
    z64 = _lin64(h64, W, b)
    what = f"tc_linear residual={res} / {fam}"
    worst = _check_ln(what, fam, y, _ln64(z64, gamma, beta), res64)
    if save is not None:
        _check_stats(what, z64, save[1], save[2], save[0])
    print(f"LN-ROWS tc_linear {res:8s} {fam:9s} worst row error {worst:.2e}")


# ---- ops.layer_norm forward and backward (csrc/dense.cu) ----------------------------------------------------------
# (D, row pitch): the vector kernel's three shapes, and the scalar kernel for an odd width and for a pitch that is not a
# multiple of 4
LN_SHAPES = [(128, 128), (64, 64), (512, 512), (30, 33), (128, 131)]


@pytest.mark.parametrize("fam", FAMILIES)
@pytest.mark.parametrize("D,pitch", LN_SHAPES)
def test_layer_norm_op_rows(libgnc, D, pitch, fam):
    from graphnet_classifier_b200 import ops
    gen = torch.Generator(device="cuda").manual_seed(2000 + LN_SHAPES.index((D, pitch)) * 100 + FAMILIES.index(fam))
    M = M_TILES
    h = torch.relu(torch.randn(M, D, generator=gen, device="cuda"))
    W, b = torch.randn(D, D, generator=gen, device="cuda") / D ** 0.5, torch.randn(D, generator=gen, device="cuda") * 0.3
    gamma = torch.rand(D, generator=gen, device="cuda") + 0.5
    beta = torch.randn(D, generator=gen, device="cuda") * 0.2
    W, b = _family(fam, W, b, h.double())
    buf = torch.full((M, pitch), float("nan"), device="cuda")
    buf[:, :D] = _lin64(h.double(), W, b).float()                   # the LayerNorm input, rows of pitch `pitch`
    z = buf[:, :D]
    r = torch.randn(M, D, generator=gen, device="cuda")
    dy = torch.randn(M, D, generator=gen, device="cuda")
    zg, gg, bg = z.detach().requires_grad_(), gamma.clone().requires_grad_(), beta.clone().requires_grad_()
    y = ops.layer_norm(zg, gg, bg, EPS, r)
    y.backward(dy)
    z64 = z.double().requires_grad_()
    g64, b64 = gamma.double().requires_grad_(), beta.double().requires_grad_()
    ln64 = torch.nn.functional.layer_norm(z64, (D,), g64, b64, EPS)
    ln64.backward(dy.double())
    what = f"layer_norm D={D} pitch={pitch} / {fam}"
    worst = _check_ln(what, fam, y.detach(), ln64.detach(), r.double())
    dz64 = z64.grad
    dzmax = dz64.abs().amax(1)
    _bad_rows(what + " dz", (zg.grad.double() - dz64).abs().amax(1), dzmax, 1e-5 * dzmax)
    assert _rel_l2(gg.grad, g64.grad) < 1e-5, (what, "dgamma", _rel_l2(gg.grad, g64.grad))
    assert _rel_l2(bg.grad, b64.grad) < 1e-5, (what, "dbeta", _rel_l2(bg.grad, b64.grad))
    print(f"LN-ROWS layer_norm D={D:3d} pitch={pitch:3d} {fam:9s} worst row error {worst:.2e}")


# ---- the training tails of tc_train.py --------------------------------------------------------------------------
@pytest.mark.parametrize("fam", FAMILIES)
@pytest.mark.parametrize("M", [M_TILES, M_TRAIN])
@pytest.mark.parametrize("fwd", ["tail", "chain"])
def test_training_tail_rows(libgnc, monkeypatch, fwd, M, fam):
    """``_tail_fwd`` (per-layer forward, LayerNorm in the 3xTF32 epilogue) or ``_mlp_fwd_chain`` (one chained launch with
    the stash), then ``_tail_bwd``, against float64 autograd of the same function.  The float64 ReLUs take the sign
    pattern of the kernels' saved activations (a pre-activation within rounding of zero may fall on either side).
    Weight and bias gradients of the Linear layers are compared at the smaller row count only."""
    from graphnet_classifier_b200 import tc_train
    dev = "cuda"
    gen = torch.Generator(device=dev).manual_seed(3000 + (fwd == "chain") * 100 + (M == M_TRAIN) * 10 + FAMILIES.index(fam))

    def rn(*s, scale=1.0):
        return torch.randn(*s, generator=gen, device=dev) * scale

    W0, b0 = rn(128, 128, scale=1 / 11), rn(128, scale=0.3)
    W2, b2 = rn(128, 128, scale=1 / 11), rn(128, scale=0.3)
    W4, b4 = rn(128, 128, scale=1 / 11), rn(128, scale=0.3)
    gamma, beta = _affine(gen)
    x, T, res = rn(M, 128), rn(M, 128), rn(M, 128)
    if fwd == "tail":
        x = torch.relu(x)                                       # a1: the first layer's ReLU output
    n_cal = min(M, 65536)
    a1_cal = x[:n_cal].double() if fwd == "tail" else torch.relu(_lin64(x[:n_cal].double(), W0, b0) + T[:n_cal].double())
    W4, b4 = _family(fam, W4, b4, torch.relu(_lin64(a1_cal, W2, b2)))
    del a1_cal
    tail_params = (W2, b2, W4, b4, gamma, beta)
    if fwd == "tail":
        y, saved = tc_train._tail_fwd(x, tail_params, EPS, res)
    else:
        y, saved = tc_train._mlp_fwd_chain(x, W0, b0, tail_params, EPS, res, (T, None))
    a1, a2, z3, mean, rstd = saved
    dy = rn(M, 128)
    seen = {}
    ln_bwd = tc_train._ln_bwd

    def keep_dz(*args, **kwargs):
        out = ln_bwd(*args, **kwargs)
        seen["dz"] = out[0]
        return out

    monkeypatch.setattr(tc_train, "_ln_bwd", keep_dz)
    da1, grads = tc_train._tail_bwd(dy, saved, tail_params, True)
    dz3 = seen["dz"]

    # float64 autograd of the same function, row chunk by row chunk; parameter gradients accumulate over the chunks
    P64 = [t.double().requires_grad_() for t in tail_params]
    W2d, b2d, W4d, b4d, gd, btd = P64
    what = f"training {fwd} M={M} / {fam}"
    worst, da1_err2, da1_ref2 = 0.0, 0.0, 0.0
    for lo in range(0, M, CHUNK):
        sl = slice(lo, min(M, lo + CHUNK))
        if fwd == "tail":
            a1d = x[sl].double().requires_grad_()
            pre = a1d
        else:
            pre = (_lin64(x[sl].double(), W0, b0) + T[sl].double()).requires_grad_()
            a1d = pre * (a1[sl] > 0)
        a2d = (a1d @ W2d.t() + b2d) * (a2[sl] > 0)
        z64 = a2d @ W4d.t() + b4d
        z64.retain_grad()
        ln64 = torch.nn.functional.layer_norm(z64, (128,), gd, btd, EPS)
        ln64.backward(dy[sl].double())
        zd = z64.detach()
        worst = max(worst, _check_ln(what, fam, y[sl], ln64.detach(), res[sl].double()))
        _check_stats(what, zd, mean[sl], rstd[sl], z3[sl])
        dzmax = z64.grad.abs().amax(1)
        _bad_rows(what + " dz", (dz3[sl].double() - z64.grad).abs().amax(1), dzmax, 1e-5 * dzmax)
        ref = pre.grad * (x[sl] > 0) if fwd == "tail" else pre.grad
        da1_err2 += float((da1[sl].double() - ref).pow(2).sum())
        da1_ref2 += float(ref.pow(2).sum())
        del pre, a1d, a2d, z64, ln64, zd, ref
    names = ["dW2", "db2", "dW4", "db4", "dgamma", "dbeta"]
    check = names[4:] if M == M_TRAIN else names
    for name, g, p in zip(names, grads, P64):
        if name in check:
            assert _rel_l2(g, p.grad) < 1e-5, (what, name, _rel_l2(g, p.grad))
    if M != M_TRAIN:                    # (constant rows: W4 = 0 passes no gradient to a1)
        assert da1_err2 <= 1e-10 * da1_ref2, (what, "da1", (da1_err2 / max(da1_ref2, 1e-300)) ** 0.5)
    print(f"LN-ROWS training {fwd:5s} M={M:7d} {fam:9s} worst row error {worst:.2e}")


# ---- the model: one node-encoder unit with a large bias ----------------------------------------------------------
def _outlier_node_encoder(fill, r, B, diag):
    """``fill_deterministic``, then the node encoder's last Linear (``model[4]``) scaled so that the LayerNorm input rows
    have std ~1 on the test images, with ``bias[0] = 40``."""
    from oracle import graph_build as ogb
    from oracle.weights import synthetic_images

    def fill_outlier(om, seed=0):
        fill(om, seed=seed)
        enc = om.graph_net.node_encoder.model
        seen = []
        hook = enc[4].register_forward_hook(lambda _m, inp, _out: seen.append(inp[0].detach().double()))
        with torch.no_grad():
            for im in synthetic_images(B, r, seed=3 * r):
                om(ogb.to_model_inputs(*ogb.pixel_graph(im, diag)))
        hook.remove()
        a2 = torch.cat(seen)
        with torch.no_grad():
            s = float((a2 @ enc[4].weight.double().t()).std(1).mean())
            enc[4].weight.div_(s)
            enc[4].bias[0] = 40.0
    return fill_outlier


def test_model_logits_outlier_node_encoder(libgnc):
    """Inference logits of a model whose node-encoder LayerNorm rows have an outlier column, against the float64
    oracle."""
    from graphnet_classifier_b200.models.GNN import CombinedModel, GraphNet
    from graphnet_classifier_b200.pipeline import GraphClassifierPipeline
    from oracle import gnn as ognn
    from oracle import graph_build as ogb
    from oracle.weights import fill_deterministic, synthetic_images
    r, B = 16, 3
    cfg = dict(num_local_features=3, space_dim=2, out_channels=1, n_blocks=3)
    om = ognn.OracleCombinedModel(ognn.OracleGraphNet(**cfg), num_nodes=r * r, classes=2)
    _outlier_node_encoder(fill_deterministic, r, B, False)(om, seed=11)
    gm = CombinedModel(GraphNet(**cfg), num_nodes=r * r, classes=2)
    gm.load_state_dict(om.state_dict())
    gm = gm.cuda()
    om64 = ognn.OracleCombinedModel(ognn.OracleGraphNet(**cfg), num_nodes=r * r, classes=2).double()
    om64.load_state_dict(om.state_dict())
    for mlp in [m for m in om64.modules() if isinstance(m, ognn.OracleMLP)]:
        mlp.forward = (lambda x, mlp=mlp: mlp.model(x.reshape(x.shape[0], -1)))
    imgs = synthetic_images(B, r, seed=3 * r)
    logits = GraphClassifierPipeline(gm, resize_value=r).infer(torch.from_numpy(imgs)).cpu().double()
    with torch.no_grad():
        ref = torch.stack([om64(tuple(t.double() if t.is_floating_point() else t for t in
                                      ogb.to_model_inputs(*ogb.pixel_graph(im)))) for im in imgs]).reshape(logits.shape)
    err = float((logits - ref).abs().max() / ref.abs().max())
    assert err < 1e-5, err


@pytest.mark.parametrize("engine", ["tc", "tc-layerfwd"])
def test_training_gradients_outlier_node_encoder(libgnc, monkeypatch, engine):
    """Loss and all 76 gradients of one training step (the protocol of test_gpu_tc_engine: float32 and float64 oracle,
    the relaxed bar only where the oracle itself is unstable), default training forward and ``tc_train.FWD = "layer"``,
    with the node encoder's LayerNorm rows carrying an outlier column."""
    import test_gpu_tc_engine as tce
    r, B, diag = 16, 3, False
    monkeypatch.setattr(tce, "fill_deterministic", _outlier_node_encoder(tce.fill_deterministic, r, B, diag))
    tce._gradient_parity(monkeypatch, engine, r, diag, B)
