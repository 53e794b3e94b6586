"""The c = 256 fused LFA kernels on tcgen05 (lfa_tc256.cu: W_att streamed from L2 through a shared-memory ring) against
the fp32 FMA kernels of lfa.cu and an fp64 evaluation, and the size of the backward workspace they need."""
import pytest
import torch

from tests.helpers import rand_cloud

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.mark.parametrize("k,big", [(16, False), (16, True), (32, False), (32, True)])
def test_lfa_tc256_vs_fma_and_fp64(lib, k, big):
    """Pooled features, x-gradient, encoder and attention-weight gradients at c = 256 on ragged clouds (degrees < K,
    partial last tile); big: many more tiles than CTAs x ring slots, so every CTA reuses its ring and TMEM columns
    across tiles; the big clouds also have ~10^5..10^6 edge rows in the split-K attention-weight GEMM.  fp32-grade:
    <= 1e-5 of the tensor's scale against fp64, for both paths."""
    from myria3d_b200 import ops
    from myria3d_b200.randla_net import _Level

    c = 256
    sizes = [530, 9, 1, 77, 2500] + ([9000, 7000] if big else [])
    _, pos, _, ptr = rand_cloud(sizes, seed=c + k)
    n = sum(sizes)
    g = torch.Generator().manual_seed(c + k + 1)
    x = torch.randn(n, c // 2, generator=g)
    enc_w = torch.randn(c // 2, 7, generator=g) * 0.5
    enc_b = torch.randn(c // 2, generator=g) * 0.1
    att_w = torch.randn(c, c, generator=g) / c ** 0.5
    go = torch.randn(n, c, generator=g)
    lvl = _Level(ptr.tolist(), torch.device(DEV))
    posd = pos.to(DEV)
    kt = ops.table_width(k)
    nbr, _ = ops.knn(posd, lvl.ptr, posd, lvl.ptr, k, lvl.max_n, kt=kt, want_dist=False)

    def run():
        leaves = [t.to(DEV).requires_grad_(True) for t in (x, enc_w, enc_b, att_w)]
        out = ops.lfa_attentive_pool(leaves[0], posd, nbr, leaves[1], leaves[2], leaves[3])
        out.backward(go.to(DEV))
        torch.cuda.synchronize()
        return [out.detach()] + [t.grad for t in leaves]

    assert lib.b200_get_option(b"tensor_cores") == 1
    tc_res = run()
    try:
        assert lib.b200_set_option(b"tensor_cores", 0) == 0
        fma_res = run()
    finally:
        lib.b200_set_option(b"tensor_cores", 1)

    # fp64 ground truth (q = (p_i, p_j, |p_j - p_i|), folded encoder, PyG softmax), evaluated on the device
    nb = nbr.long()
    valid = nb >= 0
    xd, wd, bd, ad = [t.to(DEV).double().requires_grad_(True) for t in (x, enc_w, enc_b, att_w)]
    pd = posd.double()
    pi = pd[:, None, :].expand(-1, kt, -1)
    pj = pd[nb.clamp(min=0)]
    d = pj.float() - pi.float()
    dist = torch.sqrt((d * d).sum(-1)).double()  # the kernels compute the distance in fp32
    q = torch.cat([pi, pj, dist[..., None]], -1)
    e = torch.nn.functional.leaky_relu(q @ wd.t() + bd, 0.2)
    f = torch.cat([xd[nb.clamp(min=0)], e], -1) * valid[..., None]
    a = (f @ ad.t()).masked_fill(~valid[..., None], float("-inf"))
    p = torch.exp(a - a.max(1, keepdim=True).values.detach())
    s = p / (p.sum(1, keepdim=True) + 1e-16)
    ref_out = (s * f).sum(1)
    ref_out.backward(go.to(DEV).double())
    ref = [ref_out.detach(), xd.grad, wd.grad, bd.grad, ad.grad]
    names = ["out", "grad_x", "grad_enc_w", "grad_enc_b", "grad_att_w"]
    for name, t, f_, r in zip(names, tc_res, fma_res, ref):
        scale = float(r.abs().max())
        err_tc = float((t.double() - r).abs().max()) / scale
        err_fma = float((f_.double() - r).abs().max()) / scale
        assert err_tc < 1e-5, f"{name}: tcgen05 path off by {err_tc:.2e} of scale (FMA path: {err_fma:.2e})"
        assert err_fma < 1e-5, f"{name}: FMA path off by {err_fma:.2e} of scale"


@pytest.mark.parametrize("kt", [16, 32])
def test_lfa_tc256_bwd_workspace_honoured(lib, kt):
    """b200_lfa_bwd_workspace_bytes covers the scratch word, the [E, 256] dA / F edge rows and the dW GEMM partials of
    the c = 256 backward: a workspace one byte short is rejected with B200_E_INVALID before anything is launched, and
    with exactly that many bytes nothing is written past its end (guard bytes behind it stay intact)."""
    from myria3d_b200.ops import _p, _stream

    c, n, guard = 256, 3000, 1 << 20
    need = int(lib.b200_lfa_bwd_workspace_bytes(n, c, kt))
    assert need >= 16 + 2 * n * kt * c * 4
    g = torch.Generator(device=DEV).manual_seed(kt)
    x = torch.randn(n, c // 2, device=DEV, generator=g)
    pos = torch.rand(n, 3, device=DEV, generator=g)
    # two valid neighbours (the point and the next one) and kt - 2 empty slots: dA rows are non-zero
    i = torch.arange(n, dtype=torch.int32, device=DEV)
    nbr = torch.full((n, kt), -1, dtype=torch.int32, device=DEV)
    nbr[:, 0], nbr[:, 1] = i, (i + 1) % n
    enc_w, enc_b = torch.randn(c // 2, 7, device=DEV, generator=g), torch.randn(c // 2, device=DEV, generator=g)
    att_w = torch.randn(c, c, device=DEV, generator=g) / c ** 0.5
    att_wt = att_w.t().contiguous()
    go = torch.randn(n, c, device=DEV, generator=g)
    gx, gew, geb, gaw = torch.zeros_like(x), torch.zeros_like(enc_w), torch.zeros_like(enc_b), torch.zeros_like(att_w)
    buf = torch.full((need + guard,), 0xA5, dtype=torch.uint8, device=DEV)

    def call(nbytes):
        return lib.b200_lfa_bwd(_p(x), _p(pos), _p(nbr), _p(enc_w), _p(enc_b), _p(att_wt), _p(att_w), _p(go), _p(gx), _p(gew),
                                _p(geb), _p(gaw), _p(buf), nbytes, n, c, kt, _stream())

    assert call(need - 1) == 1  # B200_E_INVALID
    assert call(need) == 0
    torch.cuda.synchronize()
    assert bool((buf[need:] == 0xA5).all()), "the c = 256 backward wrote past its workspace"
    assert float(gaw.abs().max()) > 0.0 and bool(torch.isfinite(gaw).all()) and bool(torch.isfinite(gx).all())
