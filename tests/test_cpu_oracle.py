"""CPU tests of the oracle (the checker) against the committed golden vectors and the reference's
structural pins (shipped checkpoint, shape tests).  No GPU, no CUDA library calls."""
import os

import numpy as np

import pytest
import torch
import torch.nn.functional as F

from oracle import randla_oracle as O
from oracle.gen_golden import build_net, weight_checksum
from tests.helpers import assert_close, ptr_of, rand_cloud

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "randla_small.pt")
CKPT_LAYOUT = os.path.join(os.path.dirname(__file__), "golden", "ref_ckpt_layout.npz")


def test_oracle_matches_golden_vectors():
    g = torch.load(GOLDEN)
    net = build_net(g["seed"])
    assert abs(weight_checksum(net) - g["weight_checksum"]) < 1e-6 * g["weight_checksum"], "seeded init drifted"
    net.eval()
    with torch.no_grad():
        logits = net(g["x"], g["pos"], g["batch"], g["ptr"], decimation_idx=g["decimation_idx"])
    assert_close(logits, g["logits_eval"], atol=1e-5, what="eval logits vs golden")
    knn0 = O.knn_kdtree(g["pos"], g["ptr"].tolist(), g["pos"], g["ptr"].tolist(), 16)[0]
    assert torch.equal(knn0.int(), g["knn_level0"])

    net = build_net(g["seed"])
    net.train()
    net.mlp_classif.injected_masks = [None, g["dropout_mask"]]
    logits = net(g["x"], g["pos"], g["batch"], g["ptr"], decimation_idx=g["decimation_idx"])
    loss = F.cross_entropy(logits, g["y"], ignore_index=65)
    loss.backward()
    assert_close(logits, g["logits_train"], atol=1e-5, what="train logits vs golden")
    assert abs(float(loss) - g["loss"]) < 1e-5
    params = dict(net.named_parameters())
    for k, v in g["grads"].items():
        assert_close(params[k].grad, v, atol=1e-6, rtol=1e-3, what=f"grad {k}")
    bufs = dict(net.named_buffers())
    for k, v in g["buffers_after_step"].items():
        assert_close(bufs[k], v, atol=1e-6, rtol=1e-5, what=k)


def test_oracle_and_product_strict_load_shipped_checkpoint(tmp_path):
    """State-dict contract (SURVEY.md App. C): 257 entries, 1 113 719 trainable parameters.  The shipped Lightning
    checkpoint is rebuilt from its pickle and storage layout (tests/golden/ref_ckpt_layout.npz) and its trained weights
    (tests/golden/randla_trained_ckpt.pt), both taken from the file by oracle/gen_golden_ckpt_layout.py."""
    from myria3d_b200 import B200RandLANet
    from myria3d_b200.ckpt import load_lightning_checkpoint, net_state_dict
    from oracle.gen_golden_ckpt_layout import rebuild_checkpoint

    weights = torch.load(os.path.join(os.path.dirname(__file__), "golden", "randla_trained_ckpt.pt"))["state_dict"]
    rebuild_checkpoint(CKPT_LAYOUT, weights, str(tmp_path / "shipped.ckpt"))
    ck = load_lightning_checkpoint(str(tmp_path / "shipped.ckpt"))
    assert ck["epoch"] == 100 and ck["pytorch-lightning_version"] == "1.5.9"
    sd = net_state_dict(ck)
    assert len(sd) == 257
    assert sd.keys() == weights.keys() and all(torch.equal(sd[k], v) for k, v in weights.items())
    for cls in (O.OracleRandLANet, B200RandLANet):
        net = cls(9, 7, return_logits=True)
        res = net.load_state_dict(sd, strict=True)
        assert not res.missing_keys and not res.unexpected_keys
        assert sum(p.numel() for p in net.parameters()) == 1113719
    # the trained weights give finite, confident predictions on a synthetic tile
    net = O.OracleRandLANet(9, 7, return_logits=True)
    net.load_state_dict(sd)
    net.eval()
    x, pos, y, batch, ptr = O.synthetic_batch([2000], seed=1, num_classes=7)
    with torch.no_grad():
        out = net(x, pos, batch, ptr)
    assert out.shape == (2000, 7) and torch.isfinite(out).all()


@pytest.mark.parametrize("num_nodes", [[1250, 1250], [50, 50], [1250, 1000]])
def test_fake_run_oracle(num_nodes):
    """tests/myria3d/models/modules/test_randla_nets.py:8-40 on the oracle (sizes /10 for CPU time;
    the 12 500-point originals run on the GPU suite)."""
    x, pos, batch, ptr = rand_cloud(num_nodes, seed=3)
    model = O.OracleRandLANet(9, 6, decimation=4, num_neighbors=16)
    out = model(x, pos, batch, ptr)
    assert out.shape == torch.Size([sum(num_nodes), 6])
    assert [t.numel() for t in model.last_decimation_idx][-1] >= len(num_nodes)


def test_knn_kdtree_equals_bruteforce_and_tie_rule():
    sx, sy = [400, 3, 1], [900, 10, 2]
    g = torch.Generator().manual_seed(0)
    px, py = torch.rand(sum(sx), 3, generator=g), torch.rand(sum(sy), 3, generator=g)
    for k in (1, 10, 16):
        a, da = O.knn_bruteforce(px, ptr_of(sx), py, ptr_of(sy), k)
        b, db = O.knn_kdtree(px, ptr_of(sx), py, ptr_of(sy), k)
        assert torch.equal(a, b) and torch.equal(da, db)
        assert (da == torch.tensor([min(k, 400)] * 900 + [min(k, 3)] * 10 + [1] * 2)).all()
    # duplicates: equal distances resolve to the lower index
    p = torch.tensor([[0.0, 0, 0], [1, 0, 0], [1, 0, 0], [1, 0, 0], [5, 5, 5]])
    nb, _ = O.knn_bruteforce(p, [0, 5], p[:1], [0, 1], 3)
    assert nb.tolist() == [[0, 1, 2]]
    nb, _ = O.knn_kdtree(p, [0, 5], p[:1], [0, 1], 3, extra=1)
    assert nb.tolist() == [[0, 1, 2]]


def test_knn_graph_layout():
    _, pos, _, ptr = rand_cloud([30, 5], seed=1)
    ei = O.knn_graph(pos, 16, ptr.tolist(), "brute")
    assert ei.shape == (2, 30 * 16 + 5 * 5)
    assert (ei[1][1:] >= ei[1][:-1]).all()  # grouped by centre
    assert (ei[0][ei[1] < 30] < 30).all() and (ei[0][ei[1] >= 30] >= 30).all()
    first = torch.cat([torch.tensor([True]), ei[1][1:] != ei[1][:-1]])
    assert torch.equal(ei[0][first], ei[1][first])  # nearest neighbour is the point itself (loop=True)


def test_pyg_softmax_and_scatter():
    src = torch.randn(10, 4)
    index = torch.tensor([0, 0, 0, 1, 1, 2, 2, 2, 2, 2])
    out = O.pyg_softmax(src, index, 3)
    for gidx in range(3):
        m = index == gidx
        assert_close(out[m], torch.softmax(src[m], dim=0), atol=1e-6, what="softmax group")
    assert_close(O.scatter_sum(src, index, 3)[2], src[5:].sum(0), atol=1e-6)
    assert_close(O.scatter_max(src, index, 3)[0], src[:3].max(0).values, atol=0)


def test_decimation_indices_contract():
    torch.manual_seed(0)
    idx, new_ptr = O.decimation_indices([0, 100, 103, 104], 4)
    assert new_ptr == [0, 25, 26, 27]  # max(1, n // 4): clouds never vanish
    assert idx[:25].max() < 100 and idx[25] >= 100 and idx[25] < 103 and idx[26] == 103
    assert len(set(idx.tolist())) == 27
    with pytest.raises(ValueError):
        O.decimation_indices([0, 10], 0.5)


def test_knn_interpolate_k1_is_not_a_pure_gather():
    """(x*w)/w of PyG's knn_interpolate rounds twice: a few elements differ by 1 ulp from x[nn]."""
    g = torch.Generator().manual_seed(0)
    px, py = torch.rand(50, 3, generator=g), torch.rand(400, 3, generator=g)
    x = torch.randn(50, 64, generator=g)
    y = O.knn_interpolate(x, px, py, [0, 50], [0, 400], 1, "brute")
    nn, _ = O.knn_bruteforce(px, [0, 50], py, [0, 400], 1)
    gathered = x[nn[:, 0]]
    assert_close(y, gathered, atol=1e-6, what="interp vs gather")
    assert (y != gathered).any()


def test_block1_net_config_a_runs():
    """BASELINE configs[0]: 1 encoder layer, K=16, 4096 pts/tile, 6 classes, batch 2 -- CPU path."""
    x, pos, y, batch, ptr = O.synthetic_batch([4096, 4096])
    net = O.OracleBlock1Net(9, 6)
    out = net(x, pos, batch, ptr)
    loss = F.cross_entropy(out, y)
    loss.backward()
    assert out.shape == (8192, 6) and torch.isfinite(loss)


def test_stitch_oracle_scatter_order_and_entropy():
    """interpolation.py:113-121,142-166: scatter_add_ on CPU sums in input order (== explicit loop, bit for bit) and the
    entropy restatement equals -sum(p log p) for unsaturated probabilities."""
    from oracle import stitch_oracle as SO

    g = torch.Generator().manual_seed(3)
    logits = torch.randn(4000, 7, generator=g) * 4
    idx = torch.randint(0, 900, (4000,), generator=g)
    a = SO.scatter_sum_rows(logits, idx, 1000)
    b = SO.scatter_sum_rows_loop(logits, idx.tolist(), 1000)
    assert torch.equal(a, b)
    assert not a[900:].any()  # points without a prediction keep zero logits
    out, idx_np = SO.reduce_predictions([logits[:2500], logits[2500:]], [idx[:2500].numpy(), idx[2500:].numpy()], 1000,
                                        {1: "a", 2: "b", 6: "c", 9: "d", 17: "e", 64: "f", 65: "g"})
    p = out["probas"].double()
    torch.testing.assert_close(out["entropy"].double(), -(p * p.clamp_min(1e-30).log()).sum(1), rtol=1e-4, atol=1e-5)
    assert set(np.unique(out["preds"])) <= {1, 2, 6, 9, 17, 64, 65}
    assert torch.equal(out["logits"], a[idx_np])


def test_oracle_matches_trained_checkpoint_golden():
    """tests/golden/randla_trained_ckpt.pt (oracle/gen_golden_ckpt.py): the oracle under the reference's shipped, trained
    weights reproduces the committed logits (regression guard; the fixture carries the weights, so this also runs where
    /root/reference does not exist) and its fp32 arithmetic stays within 1e-4 of the fp64 evaluation."""
    g = torch.load(os.path.join(os.path.dirname(__file__), "golden", "randla_trained_ckpt.pt"))
    assert len(g["state_dict"]) == 257  # SURVEY.md App. C: every entry of the Lightning checkpoint's `model.*`
    net = O.OracleRandLANet(g["num_features"], g["num_classes"], num_neighbors=g["k"], return_logits=True, knn_method="brute")
    net.load_state_dict(g["state_dict"], strict=True)
    net.eval()
    x, pos, _, batch, ptr = O.synthetic_batch(g["sizes"], seed=g["seed"], num_features=9, num_classes=7)
    with torch.no_grad():
        logits = net(x, pos, batch, ptr, decimation_idx=g["decimation_idx"])
    assert_close(logits, g["logits_fp32"], atol=2e-5, what="oracle logits vs trained-checkpoint golden")
    # ... and those logits are what the reference's OWN model file (executed on stand-in PyG primitives with these shipped
    # weights, oracle/gen_golden_ckpt.py) produced, bit for bit
    assert g["reference_model_code_equals_oracle"] and torch.equal(g["logits_reference_model_code"], g["logits_fp32"])
    assert_close(logits, g["logits_fp64"], atol=1e-4 + 10 * g["fp32_vs_fp64_max_err"], what="fp32 oracle vs fp64 oracle")
    assert float(g["logits_fp32"].abs().max()) > 10.0  # realistic magnitudes, unlike the random-init fixtures


def test_oracle_tiles_of_a_batch_are_independent_in_eval_mode():
    """pyg_randla_net.py:180,216-229,250: kNN, decimation and interpolation are per cloud, BatchNorm uses running
    statistics in eval mode -> the logits of a tile do not depend on what else is in the batch (same subsets)."""
    torch.manual_seed(5)
    net = build_net(seed=77)
    net.eval()
    sizes = [600, 350, 90]
    x, pos, _, batch, ptr = O.synthetic_batch(sizes, seed=31)
    with torch.no_grad():
        full = net(x, pos, batch, ptr)
        idx = [t.clone() for t in net.last_decimation_idx]
        # tile 1 alone, with its own share of every level's subset (cloud-local indices)
        lo, hi = int(ptr[1]), int(ptr[2])
        sub_idx, lvl_ptr = [], [int(v) for v in ptr]
        for t in idx:
            nxt = [0]
            for b in range(len(lvl_ptr) - 1):
                nxt.append(nxt[-1] + max(1, (lvl_ptr[b + 1] - lvl_ptr[b]) // 4))
            sub_idx.append(t[nxt[1]:nxt[2]] - lvl_ptr[1])
            lvl_ptr = nxt
        alone = net(x[lo:hi], pos[lo:hi], torch.zeros(hi - lo, dtype=torch.int64), torch.tensor([0, hi - lo]),
                    decimation_idx=sub_idx)
    assert_close(alone, full[lo:hi], atol=2e-5, what="tile alone vs tile inside a batch")


def test_oracle_attentive_pooling_identities():
    """LocalFeatureAggregation.message (:126-152): per centre and channel the softmax weights sum to 1 (up to the 1e-16
    of PyG's softmax), so with W_att = 0 the pooled feature is the neighbourhood MEAN of f; and a cloud smaller than K
    only ever sees its own points."""
    n, k = 40, 16
    g = torch.Generator().manual_seed(2)
    pos = torch.rand(n, 3, generator=g)
    ptr = [0, 9, n]  # first cloud has 9 < K points
    ei = O.knn_graph(pos, k, ptr, method="brute")
    src, dst = ei[0], ei[1]
    assert ((src < 9) == (dst < 9)).all()  # edges never cross clouds
    deg = torch.bincount(dst, minlength=n)
    assert deg[:9].eq(9).all() and deg[9:].eq(k).all()
    f = torch.randn(ei.shape[1], 6, generator=g)
    att = torch.zeros_like(f)  # W_att = 0 -> uniform attention
    s = O.pyg_softmax(att, dst, n)
    assert_close(O.scatter_sum(s, dst, n), torch.ones(n, 6), atol=1e-6, what="softmax weights sum to one")
    pooled = O.scatter_sum(s * f, dst, n)
    mean = O.scatter_sum(f, dst, n) / deg[:, None]
    assert_close(pooled, mean, atol=1e-6, what="uniform attention = neighbourhood mean")


def test_sample_prep_oracle_pins():
    """The 8f-4 oracle against the reference's own numbers: 400 receptive fields per km^2 without overlap, 1 521 with a
    25 m overlap (BASELINE.json configs[3]; pctl/dataset/utils.py:29-38), closed Chebyshev balls, PyG voxel order."""
    from oracle import sample_prep_oracle as SO

    assert len(SO.get_mosaic_of_centers(1000, 50, 0)) == 400 and len(SO.get_mosaic_of_centers(1000, 50, 25)) == 1521
    pos = np.array([[0, 0, 0], [25, 25, 1], [50, 50, 2], [75, 25, 3], [100, 100, 0]], dtype=np.float32)
    fields = SO.split_cloud_into_samples(pos, 100, 50, 0)  # centres (25,25) (25,75) (75,25) (75,75)
    assert [f.tolist() for f in fields] == [[0, 1, 2], [2], [2, 3], [2, 4]]  # the border point 2 belongs to all four
    p = torch.tensor([[0.0, 0.0, 0.0], [0.1, 0.1, 0.1], [0.3, 0.0, 0.0], [1.0, 1.0, 1.0]])
    po, xo, yo, uniq = SO.grid_sampling(p, p.clone(), torch.tensor([2, 1, 0, 1]), 0.25)
    assert po.shape[0] == 3 and torch.allclose(po[0], torch.tensor([0.05, 0.05, 0.05])) and yo.tolist() == [1, 0, 1]


def test_sample_prep_oracle_against_reference_run_vectors():
    """PINNED: tests/golden/ref_sample_prep.npz holds outputs of the reference's OWN functions (oracle/gen_golden_ref.py
    loads pctl/dataset/utils.py and pctl/transforms/transforms.py from /root/reference and runs them on seeded inputs).
    The restatement must reproduce them exactly: receptive-field index sets (incl. points on field borders), mosaic
    centres, the node-budget draws under the same torch seed, NormalizePos."""
    import os
    from oracle import sample_prep_oracle as SO

    ref = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_sample_prep.npz"))
    assert ref["mosaic_counts"].tolist() == [400, 1521]
    for tag in "abc":
        tile, sub, ov = ref[f"split_{tag}_args"].tolist()
        fields = SO.split_cloud_into_samples(ref[f"split_{tag}_pos"], tile, sub, ov)
        off = ref[f"split_{tag}_off"]
        assert len(fields) == len(off) - 1
        assert np.array_equal(np.concatenate(fields), ref[f"split_{tag}_idx"])
        assert [len(f) for f in fields] == np.diff(off).tolist()
        assert np.array_equal(np.stack(SO.get_mosaic_of_centers(tile, sub, ov)), ref[f"split_{tag}_centers"])
    torch.manual_seed(2024)  # the generator's sequence: pos, x, then the transform's randperm
    pos, x = torch.rand(500, 3) * 50.0 - 25.0, torch.rand(500, 4)
    assert np.array_equal(pos.numpy(), ref["max_pos_in"]) and np.array_equal(x.numpy(), ref["max_x_in"])
    choice = SO.maximum_num_nodes(500, 200)
    assert np.array_equal(pos[choice].numpy(), ref["max_pos_out"]) and np.array_equal(x[choice].numpy(), ref["max_x_out"])
    assert int(ref["max_num_nodes"]) == 200 and SO.maximum_num_nodes(150, 200) is None
    torch.manual_seed(2025)
    choice = SO.minimum_num_nodes(70, 300)
    assert np.array_equal(pos[:70][choice].numpy(), ref["min_pos_out"]) and int(ref["min_num_nodes"]) == 300
    assert SO.minimum_num_nodes(300, 300) is None
    assert np.array_equal(SO.normalize_pos(pos, 50).numpy(), ref["normalize_pos_out"])


def test_stitch_oracle_against_reference_run_vectors():
    """PINNED (as far as torch_scatter's absence allows): the reference's Interpolator.store_predictions +
    reduce_predicted_logits (myria3d/models/interpolation.py:94-121), run by oracle/gen_golden_ref.py with scatter_sum
    supplied as index_add_ (torch_scatter's CPU order), against the oracle's restatement: bit-exact, incl. the duplicated
    rows of `reduced_logits[idx_in_full_cloud]`."""
    import os
    from oracle import stitch_oracle as SO

    ref = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_sample_prep.npz"))
    logits, idx = torch.from_numpy(ref["stitch_logits"]), ref["stitch_idx"]
    red, idx_out = SO.reduce_predicted_logits([logits[:1400], logits[1400:2800], logits[2800:]],
                                              [idx[:1400], idx[1400:2800], idx[2800:]], int(ref["stitch_nb_points"]))
    assert np.array_equal(idx_out, ref["stitch_idx_out"])
    assert np.array_equal(red.numpy(), ref["stitch_reduced"])


def test_oracle_equals_reference_model_code():
    """PINNED: tests/golden/ref_model_standin.pt was produced by executing the reference's OWN model file
    (myria3d/models/modules/pyg_randla_net.py, unmodified) on stand-ins for the uninstallable PyG primitives
    (oracle/pyg_standin.py, oracle/gen_golden_ref_model.py).  The oracle restatement, run on the same seeds, must give
    bit-identical eval logits, train logits, loss, parameter gradients and BatchNorm buffers -- i.e. the same wiring,
    operator order, state-dict names and random-stream consumption (per-cloud randperm, dropout) as the reference file.
    Both kNN back-ends of the oracle (kd-tree like torch_cluster's CPU path, brute force) are held to it."""
    import os
    from oracle import gen_golden_ref_model as G

    gold = torch.load(os.path.join(os.path.dirname(__file__), "golden", "ref_model_standin.pt"))
    for name, c in gold["cases"].items():
        for method in ("kdtree", "brute"):
            out = G.run_case(lambda k: O.OracleRandLANet(9, 6, decimation=4, num_neighbors=k, return_logits=True,
                                                         knn_method=method), **c)
            g = gold[name]
            assert torch.equal(out["eval_logits"], g["eval_logits"]), (name, method)
            assert torch.equal(out["train_logits"], g["train_logits"]) and torch.equal(out["loss"], g["loss"])
            for n, v in g["grads_full"].items():
                assert torch.equal(out["grads"][n], v), n
            for n, v in g["grad_norms"].items():
                assert float(out["grads"][n].double().norm()) == float(v), n
            for n, v in g["buffers"].items():
                assert torch.equal(out["buffers"][n], v), n
