"""Every kernel that sums over rows or edges, at the row counts of myria3d's own training batch (batch_size 32 x
MaximumNumNodes 40 000, configs/datamodule/hdf5_datamodule.yaml: 1 280 000 rows at level 0, then 320 000, 80 000,
20 000, 5 000), against an fp64 evaluation on the device.

Each case runs twice: zero-mean operands (randn, the running sums random-walk around zero) and coherent ones
(activations lrelu(randn + 0.5) or |randn| + 0.3, gradients randn + 0.5: positive means, as after a LeakyReLU).  The
tensor core's fp32 adder truncates towards zero, ~6e-8 of the running sum per MMA, so a long TMEM accumulation chain
is biased by ~3e-8 per chained MMA.  Each case also checks, by kernel name, that the kernel it means to cover is the
one that ran.

Weight gradients: norm-relative error < 5e-6 (tests/helpers.rel_err) and, element by element,
|got - ref| <= 2e-5 * (|gy|^T |a|)_ij, a bound that stays meaningful where the sums cancel.

Measured on an NVIDIA B200 (1 000 W power limit), weight-gradient error against fp64 as norm-relative error, with the
worst element's |err| / (|gy|^T |a|) in brackets:
- tc_tn, splits of the one-wave plan (2 176 rows for fp3, 2 016 for fp4, 736 for the summit MLP, 55 556 for the
  1 000 000-row layer): zero-mean 5.2e-6 .. 1.6e-5 (1.6e-7 .. 7.9e-7), coherent 4.6e-6 .. 1.5e-5 (3.0e-6 .. 7.9e-6);
  the 1 000 000-row layer 3.9e-4 / 3.2e-4 (2.7e-6 / 1.6e-4).  Splits of <= 512 rows: zero-mean 2.9e-6 .. 3.7e-6
  (<= 3.2e-7), coherent 2.5e-6 .. 3.4e-6 (1.7e-6 .. 2.2e-6).
- tc_skinny, one TMEM chain per 8 650-row slab (544 chained MMAs): zero-mean 9.9e-6 / 1.0e-5, coherent 8.6e-6
  (4.6e-6); restarted every 8 chunks (64 chained MMAs): 1.0e-6 .. 1.1e-6 (<= 7.5e-7).
- tma_rows_tn and the FMA kernels (fp32 FFMA, round to nearest): <= 2.9e-6 zero-mean, <= 4.0e-7 coherent (<= 8.7e-7).
The estimate that the unbounded chains land around 1.5-2.5e-5 with coherent operands held for tc_tn (1.5e-5) and was
high for tc_skinny (8.6e-6).  It was wrong in assuming zero-mean sums would hide the bias: in norm-relative terms they
failed as badly, because the truncation is relative to the running sum, which random-walks to the result's size.
"""
import pytest
import torch

from tests.helpers import rand_cloud, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _acts(n, c, coherent, g):
    x = torch.randn(n, c, device=DEV, generator=g)
    return torch.nn.functional.leaky_relu(x + 0.5, 0.2) if coherent else x


def _grads(n, c, coherent, g):
    x = torch.randn(n, c, device=DEV, generator=g)
    return x + 0.5 if coherent else x


class _Options:
    """b200_set_option for the duration of a block, restored afterwards."""

    def __init__(self, lib, **kw):
        self.lib, self.kw, self.before = lib, kw, {}

    def __enter__(self):
        for k, v in self.kw.items():
            self.before[k] = int(self.lib.b200_get_option(k.encode()))
            assert self.lib.b200_set_option(k.encode(), v) == 0
        return self

    def __exit__(self, *exc):
        for k, v in self.before.items():
            self.lib.b200_set_option(k.encode(), v)


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, " ".join(e.key for e in prof.key_averages())


def _bwd_weight(lib, gy, a1, a2, bias, ws=None, ws_bytes=None):
    """b200_linear_bwd_weight (ops.linear's weight / bias gradient), workspace sized as ops.linear sizes it."""
    from myria3d_b200.ops import _p, _stream

    n, cout = gy.shape
    c1, c2 = a1.shape[1], (a2.shape[1] if a2 is not None else 0)
    gw = torch.zeros(cout, c1 + c2, device=DEV)
    gb = torch.zeros(cout, device=DEV) if bias else None
    if ws is None and ws_bytes is None:
        ws_bytes = int(lib.b200_linear_bwd_weight_workspace_bytes(n, c1, c2, cout, 1 if bias else 0))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=DEV) if ws_bytes else None
    rc = lib.b200_linear_bwd_weight(_p(gy), _p(a1), c1, c1, _p(a2), c2, c2, _p(gw), _p(gb), _p(ws), ws_bytes or 0, n, cout,
                                    _stream())
    assert rc == 0, lib.b200_last_error()
    return gw, gb


def _check_weight_grad(what, gw, gb, gy, a1, a2):
    a = torch.cat([a1, a2], 1) if a2 is not None else a1
    gyd, ad = gy.double(), a.double()
    ref = gyd.t() @ ad
    cond = gyd.abs().t() @ ad.abs()  # (|gy|^T |a|)_ij: the size of the terms summed into element ij
    e = rel_err(gw, ref)
    worst = float(((gw.double() - ref).abs() / cond).max())
    print(f"[long-reductions] {what}: dW rel {e:.2e}, max |err| / (|gy|^T|a|) {worst:.2e}")
    assert e < 5e-6, f"{what}: dW norm-relative error {e:.2e}"
    assert worst <= 2e-5, f"{what}: dW element error {worst:.2e} of (|gy|^T |a|)"
    if gb is not None:
        rb = gyd.sum(0)
        eb = rel_err(gb, rb)
        worst_b = float(((gb.double() - rb).abs() / gyd.abs().sum(0)).max())
        print(f"[long-reductions] {what}: db rel {eb:.2e}, max |err| / sum|gy| {worst_b:.2e}")
        assert eb < 5e-6 and worst_b <= 2e-5, f"{what}: bias gradient rel {eb:.2e}, element {worst_b:.2e}"


def _weight_grad_case(lib, n, c1, c2, cout, bias, coherent, kernel, options, seed):
    g = _gen(seed)
    a1 = _acts(n, c1, coherent, g)
    a2 = _acts(n, c2, coherent, g) if c2 else None
    gy = _grads(n, cout, coherent, g)
    with _Options(lib, **options):
        (gw, gb), names = _kernel_names(lambda: _bwd_weight(lib, gy, a1, a2, bias))
    assert kernel in names, f"{kernel} did not run: {names}"
    what = f"{kernel} n={n} {c1}|{c2}->{cout} {'coherent' if coherent else 'zero-mean'}"
    _check_weight_grad(what, gw, gb, gy, a1, a2)


# --------------------------------------------------------------------- tc_tn: rows per split
# fp3 (384 -> 128 at level 2), fp4 (768 -> 256 at level 3), the summit MLP (512 -> 512 at level 4), a level-1 layer
# with the TMA kernels off, and a 1 000 000-row layer whose one-wave plan is 55 556 rows per split
TC_TN = [(80000, 256, 128, 128, True), (20000, 512, 256, 256, True), (5000, 512, 0, 512, True),
         (320000, 64, 0, 128, True), (1000000, 128, 0, 512, True)]


@pytest.mark.parametrize("coherent", [False, True])
@pytest.mark.parametrize("n,c1,c2,cout,bias", TC_TN)
def test_tc_tn_long_reduction(lib, n, c1, c2, cout, bias, coherent):
    """tc_gemm.cu's split-K weight gradient: each split sums its rows in one TMEM accumulator (12 chained MMAs per 32
    rows); the plan bounds a split to 512 rows."""
    _weight_grad_case(lib, n, c1, c2, cout, bias, coherent, "tc_tn_kernel", dict(tma_rows=0), seed=n + cout)


# ------------------------------------------------------------------ tc_skinny: rows per CTA
# (32 -> 33 with a bias column is 33 x 33: tn_skinny_kernel's shape, covered below; without one it is tc_skinny's)
TC_SKINNY = [(1280000, 9, 0, 32, True), (1280000, 32, 0, 4, True), (1280000, 32, 0, 33, False)]


@pytest.mark.parametrize("coherent", [False, True])
@pytest.mark.parametrize("n,c1,c2,cout,bias", TC_SKINNY)
def test_tc_skinny_long_reduction(lib, n, c1, c2, cout, bias, coherent):
    """tc_skinny.cu (fc0 9 -> 32, mlp1 32 -> 4, 32 -> 33 at level 0): one persistent CTA per SM sums n / 148 rows; the
    main (hi * hi) TMEM accumulator chains 8 MMAs per 128-row chunk and is flushed to registers every 8 chunks."""
    _weight_grad_case(lib, n, c1, c2, cout, bias, coherent, "tc_skinny_tn_kernel", dict(tma_rows=0), seed=n + cout)


# --------------------------------------------------- tma_rows_tn: fp32 FMA, registers across row tiles
TMA_TN = [(1280000, 32, 0, 32, True), (1280000, 16, 0, 32, True), (320000, 32, 0, 128, True), (320000, 128, 32, 32, True)]


@pytest.mark.parametrize("coherent", [False, True])
@pytest.mark.parametrize("n,c1,c2,cout,bias", TMA_TN)
def test_tma_rows_tn_long_reduction(lib, n, c1, c2, cout, bias, coherent):
    """tma_rows.cu's weight gradient: each thread keeps a 4 x 4 block of gw in registers over every row tile of its
    CTA and row slice."""
    _weight_grad_case(lib, n, c1, c2, cout, bias, coherent, "tma_rows_tn_kernel", dict(tma_rows=7), seed=n + cout + 1)


# ------------------------------------------------------------------ the FMA fallbacks (A/B reference)
@pytest.mark.parametrize("coherent", [False, True])
@pytest.mark.parametrize("n,c1,c2,cout,bias", TC_TN + TC_SKINNY + TMA_TN)
def test_fma_weight_grad_long_reduction(lib, n, c1, c2, cout, bias, coherent):
    """tensor_cores = 0, tma_rows = 0: the same shapes through tn_skinny_kernel (<= 64 x 64) and
    linear_bwd_weight_kernel (fp32 FFMA, rows per CTA / split)."""
    kernel = "tn_skinny_kernel" if cout <= 64 and c1 + c2 <= 64 else "linear_bwd_weight_kernel"
    _weight_grad_case(lib, n, c1, c2, cout, bias, coherent, kernel, dict(tensor_cores=0, tma_rows=0), seed=n + cout + 2)


# ------------------------------------------------------------------------ split-K workspace
@pytest.mark.parametrize("n,c1,c2,cout", [(80000, 256, 128, 128), (1000000, 128, 0, 512)])
def test_tc_tn_workspace_sized_by_the_same_plan(lib, n, c1, c2, cout):
    """b200_linear_bwd_weight_workspace_bytes sizes the partial tiles of exactly the plan the kernel runs: with that
    many bytes the partials path runs (no fall-back to atomics), two calls are bit-identical, nothing is written past
    the end; without a workspace the (atomic) result is still right."""
    g = _gen(7)
    a1 = _acts(n, c1, True, g)
    a2 = _acts(n, c2, True, g) if c2 else None
    gy = _grads(n, cout, True, g)
    need = int(lib.b200_linear_bwd_weight_workspace_bytes(n, c1, c2, cout, 1))
    guard = 1 << 20
    buf = torch.full((need + guard,), 0xA5, dtype=torch.uint8, device=DEV)
    with _Options(lib, tma_rows=0):
        (gw1, gb1), names = _kernel_names(lambda: _bwd_weight(lib, gy, a1, a2, True, ws=buf, ws_bytes=need))
        gw2, gb2 = _bwd_weight(lib, gy, a1, a2, True, ws=buf, ws_bytes=need)
        (gw0, gb0), names0 = _kernel_names(lambda: _bwd_weight(lib, gy, a1, a2, True, ws=None, ws_bytes=0))
    torch.cuda.synchronize()
    assert "tc_tn_kernel" in names and "tc_reduce_partials_kernel" in names, names
    assert "tc_tn_kernel" in names0 and "tc_reduce_partials_kernel" not in names0, names0
    assert torch.equal(gw1, gw2) and torch.equal(gb1, gb2), "the partials path is not deterministic"
    assert bool((buf[need:] == 0xA5).all()), "the weight gradient wrote past its workspace"
    _check_weight_grad(f"tc_tn workspace n={n}", gw1, gb1, gy, a1, a2)
    _check_weight_grad(f"tc_tn atomics n={n}", gw0, gb0, gy, a1, a2)


# ------------------------------------------------------------------------------- LFA dW_att
def _lfa_case(lib, sizes, c, k, coherent, kernel, seed):
    """ops.lfa_attentive_pool forward + backward vs fp64 autograd on the device (as test_gpu_lfa_tc256.py)."""
    from myria3d_b200 import ops
    from myria3d_b200.randla_net import _Level

    _, pos, _, ptr = rand_cloud(sizes, seed=seed, features=1)
    n = sum(sizes)
    g = _gen(seed)
    x = (torch.randn(n, c // 2, device=DEV, generator=g).abs() + 0.3) if coherent else torch.randn(n, c // 2, device=DEV, generator=g)
    enc_w = torch.randn(c // 2, 7, device=DEV, generator=g) * 0.5
    enc_b = torch.randn(c // 2, device=DEV, generator=g) * 0.1 + (0.5 if coherent else 0.0)
    att_w = torch.randn(c, c, device=DEV, generator=g) / c ** 0.5
    go = _grads(n, c, coherent, g)
    lvl = _Level(ptr.tolist(), torch.device(DEV))
    posd = pos.to(DEV)
    kt = ops.table_width(k)
    nbr, _ = ops.knn(posd, lvl.ptr, posd, lvl.ptr, k, lvl.max_n, kt=kt, want_dist=False)

    def run():
        leaves = [t.clone().requires_grad_(True) for t in (x, enc_w, enc_b, att_w)]
        out = ops.lfa_attentive_pool(leaves[0], posd, nbr, leaves[1], leaves[2], leaves[3])
        out.backward(go)
        return [out.detach()] + [t.grad for t in leaves]

    res, names = _kernel_names(run)
    assert kernel in names, f"{kernel} did not run: {names}"
    nb = nbr.long()
    valid = nb >= 0
    xd, wd, bd, ad = [t.double().requires_grad_(True) for t in (x, enc_w, enc_b, att_w)]
    pd = posd.double()
    pi = pd[:, None, :].expand(-1, kt, -1)
    pj = pd[nb.clamp(min=0)]
    d = pj.float() - pi.float()
    dist = torch.sqrt((d * d).sum(-1)).double()  # the kernels compute the distance in fp32
    q = torch.cat([pi, pj, dist[..., None]], -1)
    pre = q @ wd.t() + bd
    pre.retain_grad()
    e = torch.nn.functional.leaky_relu(pre, 0.2)
    f = torch.cat([xd[nb.clamp(min=0)], e], -1) * valid[..., None]
    a = (f @ ad.t()).masked_fill(~valid[..., None], float("-inf"))
    p = torch.exp(a - a.max(1, keepdim=True).values.detach())
    s = p / (p.sum(1, keepdim=True) + 1e-16)
    ref_out = (s * f).sum(1)
    ref_out.backward(go.double())
    ref = [ref_out.detach(), xd.grad, wd.grad, bd.grad, ad.grad]
    # the encoder gradients sum dpre_e q_e over every edge; with zero-mean operands they cancel to a small fraction of
    # the terms' size, so they are held to the condition-aware bound instead of their own scale
    dpre = pre.grad.reshape(-1, c // 2).abs()
    cond = {"grad_enc_w": dpre.t() @ q.detach().reshape(-1, 7).abs(), "grad_enc_b": dpre.sum(0)}
    tag = f"{kernel} c={c} n={n} {'coherent' if coherent else 'zero-mean'}"
    for name, t, r in zip(["out", "grad_x", "grad_enc_w", "grad_enc_b", "grad_att_w"], res, ref):
        err = float((t.double() - r).abs().max()) / float(r.abs().max())
        print(f"[long-reductions] {tag} {name}: {err:.2e} of scale")
        if name in cond:
            worst = float(((t.double() - r).abs() / cond[name]).max())
            print(f"[long-reductions] {tag} {name}: max |err| / sum|terms| {worst:.2e}")
            assert worst <= 2e-5, f"{tag} {name}: element error {worst:.2e} of the summed terms' size"
            if not coherent:
                continue
        assert err < 1e-5, f"{tag} {name}: off by {err:.2e} of scale"


@pytest.mark.parametrize("coherent", [False, True])
@pytest.mark.parametrize("c,npts", [(8, 40000), (16, 40000), (32, 10000)])
def test_lfa_small_c_long_reduction(lib, c, npts, coherent):
    """c <= 32: dW_att in 4 x 4 register blocks over all tiles of a CTA (lfa.cu; c = 32 on tcgen05, lfa_tc.cu), on 32
    clouds of npts points, K = 16 (20 480 000 edge rows at c = 8 and 16)."""
    kernel = "lfa_tc_kernel" if c == 32 else "lfa_bwd_kernel"
    _lfa_case(lib, [npts] * 32, c, 16, coherent, kernel, seed=c)


@pytest.mark.parametrize("coherent", [False, True])
@pytest.mark.parametrize("c,npts,kernel", [(64, 10000, "lfa_tc_kernel"), (128, 2500, "lfa_tc_kernel"),
                                           (256, 625, "lfa_tc256_kernel")])
def test_lfa_tensor_core_long_reduction(lib, c, npts, kernel, coherent):
    """tcgen05 LFA at levels 1-3 of the full batch: c = 64 / 128 flush their TMEM dW every LTC_FLUSH tiles, c = 256
    reduces dW_att with the bounded split-K GEMM (regression guard)."""
    _lfa_case(lib, [npts] * 32, c, 16, coherent, kernel, seed=c + 1)


# ---------------------------------------------------------- fp64 partials: column statistics, loss, edge moments
def test_column_statistics_full_batch(lib):
    """BatchNorm column statistics of a level-0 layer (fp64 partials per CTA) at 1 280 000 rows with |mean| >> std."""
    from myria3d_b200 import ops

    g = _gen(11)
    n = 1280000
    a = torch.randn(n, 32, device=DEV, generator=g) + 0.2
    w = torch.randn(32, 32, device=DEV, generator=g) / 32 ** 0.5
    b = torch.randn(32, device=DEV, generator=g) + 30.0
    y, stats = ops.linear(a, w, b, want_stats=True)
    st = stats.sum(0)
    yd = y.double()
    mean, var = st[:32] / n, st[32:] / n - (st[:32] / n) ** 2
    e_mean = float(((mean - yd.mean(0)).abs() / yd.mean(0).abs()).max())
    e_var = float(((var - yd.var(0, unbiased=False)).abs() / yd.var(0, unbiased=False)).max())
    print(f"[long-reductions] column statistics n={n}: mean {e_mean:.2e}, var {e_var:.2e}")
    assert e_mean <= 1e-9 and e_var <= 1e-6


def test_cross_entropy_full_batch(lib):
    """The fused weighted cross-entropy (fp64 reduction) over 1 280 000 rows, 20 % ignored, vs fp64 torch."""
    import torch.nn.functional as F

    from myria3d_b200 import ops

    g = _gen(12)
    n, c = 1280000, 6
    logits = (torch.randn(n, c, device=DEV, generator=g) * 3 + 1.0).requires_grad_(True)
    target = torch.randint(0, c, (n,), device=DEV, generator=g)
    target[torch.rand(n, device=DEV, generator=g) < 0.2] = 65
    weight = torch.rand(c, device=DEV, generator=g) + 0.5
    ref_in = logits.detach().double().requires_grad_(True)
    ref = F.cross_entropy(ref_in, target, weight=weight.double(), ignore_index=65)
    ref.backward()
    loss = ops.cross_entropy(logits, target, weight, ignore_index=65)
    loss.backward()
    err = abs(float(loss) - float(ref)) / max(1.0, abs(float(ref)))
    gerr = float((logits.grad.double() - ref_in.grad).abs().max()) / float(ref_in.grad.abs().max())
    print(f"[long-reductions] cross entropy n={n}: loss {err:.2e}, grad {gerr:.2e} of scale")
    assert err <= 2e-6 and gerr <= 2e-6
    assert not logits.grad[target == 65].any()


def test_edge_moments_full_batch(lib):
    """The fp64 edge moments of the encoder fold over 20 480 000 edges (32 clouds x 40 000 points, K = 16)."""
    from myria3d_b200 import ops
    from myria3d_b200.randla_net import _Level

    _, pos, _, ptr = rand_cloud([40000] * 32, seed=13, features=1)
    lvl = _Level(ptr.tolist(), torch.device(DEV))
    posd = pos.to(DEV) * 50.0 + 1000.0  # metric coordinates far from the origin: |mean| >> std
    nbr, _ = ops.knn(posd, lvl.ptr, posd, lvl.ptr, 16, lvl.max_n, kt=16, want_dist=False)
    out = ops.edge_moments(posd, nbr)
    nb = nbr.long()
    m = nb >= 0
    pi = posd.double()[:, None, :].expand(-1, 16, -1)[m]
    pj = posd.double()[nb.clamp(min=0)][m]
    d = posd[nb.clamp(min=0)][m] - posd[:, None, :].expand(-1, 16, -1)[m]
    dist = torch.sqrt((d * d).sum(1, keepdim=True)).double()
    q = torch.cat([pi, pj, dist], 1)
    ref = torch.cat([torch.tensor([float(q.shape[0])], dtype=torch.float64, device=DEV), q.sum(0), (q.t() @ q).flatten()])
    assert float(out[0]) == q.shape[0]
    err = float(((out - ref).abs() / (1e-9 + 1e-8 * ref.abs())).max())
    print(f"[long-reductions] edge moments: max |err| / (1e-9 + 1e-8 |ref|) = {err:.2e}")
    assert err <= 1.0
