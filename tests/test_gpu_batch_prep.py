"""Batch preparation on the GPU (csrc/batch_prep.cu, myria3d_b200/batch_prep.py) against the CPU oracle
(oracle/batch_prep_oracle.py) replaying the same draws, the single-sample grid_sampling(), the reference-run fixture
(tests/golden/ref_batch_prep.npz) and the distributions of the draws."""
import os
import warnings

import numpy as np
import pytest
import torch

from oracle import batch_prep_oracle as BO
from oracle import sample_prep_oracle as SO
from tests.helpers import assert_close

pytestmark = pytest.mark.gpu
DEV = "cuda"
NAMES = ["Intensity", "ReturnNumber", "NumberOfReturns", "Red", "Green", "Blue", "Infrared", "rgb_avg", "ndvi"]
PRE = {3: 5, 4: 5, 0: 1, 66: 65, 100: 1, 101: 1}  # configs/dataset_description/20230601_lidarhd_pacasam_dataset.yaml
CLASSES = {1: "unclassified", 2: "ground", 5: "vegetation", 6: "building", 9: "water", 17: "bridge", 64: "lasting_above"}
CODES = [0, 1, 2, 3, 4, 5, 6, 9, 17, 64, 65, 66, 100, 101]


def _cfg(**kw):
    from myria3d_b200 import PrepConfig

    return PrepConfig(dict(PRE), dict(CLASSES), list(NAMES), **kw)


def _sample(n, seed, extent=(50.0, 50.0, 20.0), codes=None):
    from myria3d_b200 import Data

    g = torch.Generator().manual_seed(seed)
    pos = torch.rand(n, 3, generator=g) * torch.tensor(extent) + torch.tensor([1000.0, 2000.0, 100.0])
    pos = pos.float()
    x = torch.rand(n, len(NAMES), generator=g)
    x[:, 0] = torch.rand(n, generator=g) * 3000
    x[:, 7] = torch.rand(n, generator=g) * 60000
    if codes is None:
        y = torch.tensor(CODES)[torch.randint(0, len(CODES), (n,), generator=g)]
    else:
        y = torch.tensor(codes, dtype=torch.int64)
    idx = torch.randperm(200000, generator=g)[:n].sort().values
    return Data(pos=pos, x=x, y=y, idx_in_original_cloud=idx.numpy(), x_features_names=NAMES)


def _ragged(seed=0):
    """12 samples: 70 points (padded to 300), > 40 000 voxels (cut), one point left after the drop, dense samples whose
    0.25 m voxels merge, preprocessed codes and 65 / 66 artefacts everywhere."""
    s = [_sample(70, seed + 1), _sample(56000, seed + 2, extent=(50.0, 50.0, 30.0)),
         _sample(4, seed + 3, codes=[65, 66, 2, 66]), _sample(3000, seed + 4, extent=(4.0, 4.0, 2.0)),
         _sample(1200, seed + 5), _sample(2000, seed + 6, extent=(6.0, 6.0, 1.0)), _sample(800, seed + 7),
         _sample(5000, seed + 8, extent=(10.0, 10.0, 3.0)), _sample(350, seed + 9), _sample(600, seed + 10),
         _sample(150, seed + 11), _sample(2500, seed + 12, extent=(30.0, 30.0, 10.0))]
    return s


def _collate(samples):
    from myria3d_b200 import RawCollater

    return RawCollater()(samples).to(DEV, non_blocking=True)


def _oracle_batch(samples, mode, cfg, draws):
    """The oracle chain per sample with the GPU's draws, collated like prepare_batch."""
    from myria3d_b200 import Batch

    outs = []
    for b, d in enumerate(samples):
        ch = draws["choice"][b] if draws is not None else None
        outs.append(BO.prepare_sample(
            d.pos, d.x, d.y, torch.from_numpy(np.asarray(d.idx_in_original_cloud)), mode, cfg.classification_preprocessing_dict,
            cfg.classification_dict, cfg.x_features_names, cfg.subtile_width, cfg.grid_size, cfg.min_nodes, cfg.max_nodes,
            choice=None if ch is None else ch.cpu(), flip=draws["flip"][b].tolist() if draws is not None else (False, False),
            angle_deg=float(draws["angle_deg"][b]) if draws is not None else 0.0, rotate=bool(cfg.rotate_degrees)))
    sizes = [o["pos"].shape[0] for o in outs]
    ptr = torch.tensor(np.cumsum([0] + sizes), dtype=torch.int64)
    kw = dict(pos=torch.cat([o["pos"] for o in outs]), x=torch.cat([o["x"] for o in outs]), y=torch.cat([o["y"] for o in outs]),
              batch=torch.cat([torch.full((n,), i, dtype=torch.int64) for i, n in enumerate(sizes)]), ptr=ptr)
    if mode != "train":
        kw["copies"] = {k: torch.cat([o["copies"][k] for o in outs]) for k in outs[0]["copies"]}
        kw["idx_in_original_cloud"] = [o["idx_in_original_cloud"] for o in outs]
    return Batch(**kw)


def _compare(got, exp, mode):
    assert tuple(got.ptr_host) == tuple(exp.ptr.tolist()) and torch.equal(got.ptr.cpu(), exp.ptr)
    assert torch.equal(got.batch.cpu(), exp.batch) and torch.equal(got.y.cpu(), exp.y)
    assert_close(got.pos, exp.pos, atol=1e-6, rtol=3e-7, what=f"{mode} pos")
    assert_close(got.x, exp.x, atol=1e-6, rtol=3e-7, what=f"{mode} x")
    if mode != "train":
        assert set(got.copies) == set(exp.copies)
        for k in exp.copies:
            assert torch.equal(got.copies[k].cpu(), exp.copies[k]), k
        assert len(got.idx_in_original_cloud) == len(exp.idx_in_original_cloud)
        for a, b in zip(got.idx_in_original_cloud, exp.idx_in_original_cloud):
            assert torch.equal(a.cpu(), b)


@pytest.mark.parametrize("min_nodes", [300, 1])
@pytest.mark.parametrize("mode", ["train", "eval", "predict"])
def test_prepared_batch_equals_oracle_with_replayed_draws(lib, mode, min_nodes):
    """min_nodes = 1 keeps the one-point sample (train / eval) at one row: the n = 1 standardisation (NaN std -> 1)."""
    from myria3d_b200 import prepare_batch

    samples = _ragged()
    cfg = _cfg(rotate_degrees=180, min_nodes=min_nodes)
    got = prepare_batch(_collate(samples), mode, cfg, seed=11, counter=torch.tensor([3], device=DEV), return_draws=True)
    draws = got.draws
    sizes = np.diff(got.ptr_host)
    left = 3 if mode == "predict" else 1  # predict drops the raw code 65 only: [65, 66, 2, 66] keeps three points
    assert sizes[1] == 40000 and sizes[2] == max(left, min_nodes) and (sizes[0] == 300 or min_nodes == 1)
    assert (draws["choice"][0] is not None) == (min_nodes == 300) and draws["choice"][1] is not None
    _compare(got, _oracle_batch(samples, mode, cfg, draws), mode)
    if mode == "train":
        assert draws["flip"].any() and (draws["angle_deg"] != 0).all()
    else:
        assert not draws["flip"].any() and (draws["angle_deg"] == 0).all()


def test_pooled_samples_equal_single_sample_grid_sampling(lib):
    """GridSampling per sample bit-identical to grid_sampling() on that sample alone: pooled positions (CopySampledPos),
    majority labels, and the feature columns the standardisation leaves alone."""
    from myria3d_b200 import prepare_batch
    from myria3d_b200.sample_prep import grid_sampling

    samples = _ragged(seed=40)
    cfg = _cfg(min_nodes=1, max_nodes=10 ** 6)
    got = prepare_batch(_collate(samples), "eval", cfg)
    fp, ptr = got.copies["pos_copy"], [0]
    for a in got.idx_in_original_cloud:
        ptr.append(ptr[-1] + a.numel())
    keep_cols = [c for c in range(len(NAMES)) if NAMES[c] not in ("Intensity", "rgb_avg")]
    for b, d in enumerate(samples):
        o = got.ptr_host
        y = BO.target_transform(d.y, PRE, CLASSES)
        keep = BO.drop_points_by_class(y)
        p, f, l = grid_sampling(d.pos[keep].to(DEV), d.x[keep].to(DEV), y[keep].to(DEV), 0.25)
        assert torch.equal(fp[ptr[b]:ptr[b + 1]], d.pos[keep].to(DEV))
        assert torch.equal(got.copies["pos_sampled_copy"][o[b]:o[b + 1]], p), b
        assert torch.equal(got.y[o[b]:o[b + 1]], l), b
        assert torch.equal(got.x[o[b]:o[b + 1]][:, keep_cols], f[:, keep_cols]), b
    assert got.ptr_host[2] - got.ptr_host[1] > 40000  # the big sample pooled to more than the budget


def test_labels_drop_and_copies_against_the_reference_fixture(lib):
    """The reference's TargetTransform / DropPointsByClass / CopyFullPos / CopyFullPreparedTargets outputs, bit for bit."""
    from myria3d_b200 import Data, prepare_batch

    ref = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_batch_prep.npz"))
    names = [str(s) for s in ref["features"].tolist()]
    samples = [Data(pos=torch.from_numpy(ref[f"s{i}_pos"]), x=torch.from_numpy(ref[f"s{i}_x"]), y=torch.from_numpy(ref[f"s{i}_y"]),
                    idx_in_original_cloud=ref[f"s{i}_idx"], x_features_names=names) for i in range(int(ref["num_samples"]))]
    got = prepare_batch(_collate(samples), "eval", _cfg())
    exp_pos = np.concatenate([ref[f"s{i}_pos_copy"] for i in range(len(samples))])
    exp_y = np.concatenate([ref[f"s{i}_y_copy"] for i in range(len(samples))])
    assert np.array_equal(got.copies["pos_copy"].cpu().numpy(), exp_pos)
    assert np.array_equal(got.copies["transformed_y_copy"].cpu().numpy(), exp_y)
    for i, a in enumerate(got.idx_in_original_cloud):
        assert np.array_equal(a.cpu().numpy(), ref[f"s{i}_drop_idx"])
    assert got.ptr_host[4] - got.ptr_host[3] == 300  # the one-point sample, padded


def test_draw_distributions(lib):
    from scipy import stats

    from myria3d_b200 import prepare_batch

    # flips and angles over 4 000 samples
    samples = [_sample(6, 1000 + i, codes=[2, 2, 5, 6, 1, 9]) for i in range(4000)]
    cfg = _cfg(min_nodes=1, rotate_degrees=180)
    got = prepare_batch(_collate(samples), "train", cfg, seed=5, return_draws=True)
    flips = got.draws["flip"].double().cpu()
    sigma = (0.25 / 4000) ** 0.5
    assert ((flips.mean(0) - 0.5).abs() < 5 * sigma).all(), flips.mean(0)
    angles = got.draws["angle_deg"].cpu().numpy()
    assert angles.min() >= -180 and angles.max() <= 180
    assert stats.kstest(angles, "uniform", args=(-180, 360)).pvalue > 1e-3
    # budget draws
    samples = _ragged(seed=70)
    got = prepare_batch(_collate(samples), "train", _cfg(), seed=9, return_draws=True)
    cut = got.draws["choice"][1]
    assert cut.numel() == 40000 and cut.unique().numel() == 40000
    pad = got.draws["choice"][0].cpu()
    d = samples[0]  # its pooled size from the oracle chain, not from the draw
    y = BO.target_transform(d.y, PRE, CLASSES)
    keep = BO.drop_points_by_class(y)
    nv = SO.grid_sampling(d.pos[keep], d.x[keep], y[keep], 0.25)[0].shape[0]
    assert 0 < nv < 300 and pad.numel() == 300 and int(pad.min()) >= 0 and int(pad.max()) < nv
    counts = torch.bincount(pad, minlength=nv)
    assert counts.numel() == nv and int(counts.min()) >= 300 // nv


def test_same_seed_and_counter_give_the_same_batch(lib):
    from myria3d_b200 import prepare_batch

    raw = _collate(_ragged(seed=90))
    cfg = _cfg(rotate_degrees=180)
    ctr = torch.zeros(1, dtype=torch.int64, device=DEV)
    a = prepare_batch(raw, "train", cfg, seed=3, counter=ctr, return_draws=True)
    b = prepare_batch(raw, "train", cfg, seed=3, counter=ctr, return_draws=True)
    for k in ("pos", "x", "y", "batch", "ptr"):
        assert torch.equal(getattr(a, k), getattr(b, k)), k
    ctr += 1
    c = prepare_batch(raw, "train", cfg, seed=3, counter=ctr, return_draws=True)
    assert not torch.equal(a.draws["angle_deg"], c.draws["angle_deg"])
    assert not torch.equal(a.draws["choice"][1], c.draws["choice"][1])
    assert not torch.equal(a.pos, c.pos)


def test_errors(lib):
    from myria3d_b200 import RawCollater, prepare_batch

    cfg = _cfg()
    with pytest.raises(TypeError, match=r"\[7, 8\]"):
        prepare_batch(_collate([_sample(50, 1), _sample(4, 2, codes=[1, 7, 8, 2])]), "train", cfg)
    # a code the preprocessing maps to a code classification_dict lacks: both codes are named
    with pytest.raises(TypeError, match=r"raw codes \[3\] \(after classification_preprocessing_dict: \[42\]\)"):
        prepare_batch(_collate([_sample(4, 2, codes=[1, 3, 2, 2])]), "train", _cfg().__class__(
            {3: 42}, dict(CLASSES), list(NAMES)))
    with pytest.raises(TypeError, match="outside"):
        prepare_batch(_collate([_sample(4, 2, codes=[1, 300, 2, 2])]), "eval", cfg)
    with pytest.raises(ValueError, match=r"\[1\]"):
        prepare_batch(_collate([_sample(50, 1), _sample(3, 2, codes=[65, 66, 65])]), "eval", cfg)
    with pytest.raises(ValueError, match="32 bits"):
        prepare_batch(_collate([_sample(50, 3, extent=(1.0e5, 1.0e5, 20.0))]), "train", cfg)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        prepare_batch(RawCollater(pin_memory=False)([_sample(50, 1)]), "train", cfg)
    # predict mode ignores the class dicts and drops the raw code 65 only
    got = prepare_batch(_collate([_sample(5, 4, codes=[7, 65, 66, 200, 7])]), "predict", _cfg(min_nodes=1))
    assert got.copies["pos_copy"].shape[0] == 4 and "transformed_y_copy" not in got.copies


def test_one_synchronising_call_per_batch(lib):
    from myria3d_b200 import prepare_batch

    raw = _collate(_ragged(seed=120))
    cfg = _cfg(rotate_degrees=180)
    for mode in ("train", "eval", "predict"):
        prepare_batch(raw, mode, cfg)  # warm-up: label table, allocator
        torch.cuda.synchronize()
        prev = torch.cuda.get_sync_debug_mode()
        torch.cuda.set_sync_debug_mode("warn")
        try:
            with warnings.catch_warnings(record=True) as w:
                warnings.simplefilter("always")
                prepare_batch(raw, mode, cfg, return_draws=True)
        finally:
            torch.cuda.set_sync_debug_mode(prev)
        syncs = [str(x.message) for x in w if "synchroniz" in str(x.message).lower()]
        assert len(syncs) <= 1, (mode, syncs)


def test_model_steps_on_prepared_batches(lib):
    """Model.training_step on a train batch and Model.validation_step on an eval batch: logits of the GPU-prepared batch
    and of the oracle-prepared batch (same draws) agree; the eval loss is computed on transformed_y_copy."""
    from myria3d_b200 import Model, prepare_batch

    torch.manual_seed(0)
    model = Model(neural_net_class_name="B200RandLANet",
                  neural_net_hparams=dict(num_features=9, num_classes=7, num_neighbors=16, decimation=4, return_logits=True),
                  criterion=torch.nn.CrossEntropyLoss(ignore_index=65), interpolation_k=10, num_workers=1).to(DEV)
    samples = [_sample(n, 300 + i) for i, n in enumerate([700, 1500, 70, 2400])]
    cfg = _cfg(rotate_degrees=180)
    for mode, step in (("train", model.training_step), ("eval", model.validation_step)):
        got = prepare_batch(_collate(samples), mode, cfg, seed=1, return_draws=True)
        exp = _oracle_batch(samples, mode, cfg, got.draws).to(DEV)
        model.train() if mode == "train" else model.eval()
        torch.manual_seed(42)
        out_gpu = step(got, 0)
        torch.manual_seed(42)
        out_ref = step(exp, 0)
        assert_close(out_gpu["logits"], out_ref["logits"], atol=1e-5, what=f"{mode} logits")
        assert torch.equal(out_gpu["targets"], out_ref["targets"])
        if mode == "eval":
            assert torch.equal(out_gpu["targets"], got.copies["transformed_y_copy"])
            assert out_gpu["logits"].shape[0] == got.copies["pos_copy"].shape[0]
        assert torch.isfinite(out_gpu["loss"]) and abs(float(out_gpu["loss"]) - float(out_ref["loss"])) < 1e-5


def test_raw_collater_in_dataloader_workers_after_cuda_init(lib):
    """The documented switch-over: CUDA is initialised in the main process, DataLoader workers run RawCollater (no
    pinning there), the DataLoader pins in the main process, and prepare_batch consumes the result."""
    from myria3d_b200 import prepare_batch

    torch.zeros(1, device=DEV)  # initialise CUDA before the workers fork
    from myria3d_b200 import RawCollater

    samples = _ragged(seed=150)[2:8]
    loader = torch.utils.data.DataLoader(samples, batch_size=3, num_workers=2, collate_fn=RawCollater(), pin_memory=True)
    cfg = _cfg()
    seen = 0
    for b, raw in enumerate(loader):
        assert raw.pos.is_pinned() and raw.y.is_pinned() and len(raw.idx_in_original_cloud) == 3
        got = prepare_batch(raw.to(DEV, non_blocking=True), "eval", cfg, return_draws=True)
        part = samples[3 * b:3 * b + 3]
        _compare(got, _oracle_batch(part, "eval", cfg, got.draws), "eval")
        seen += 1
    assert seen == 2
