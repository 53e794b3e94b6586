"""Batch preparation, CPU side: the oracle (oracle/batch_prep_oracle.py) against vectors made by the reference's own
transforms.py (tests/golden/ref_batch_prep.npz), the label table of PrepConfig, and argument validation of the
b200_batch_prep_* entry points (which happens before any CUDA call)."""
import os
import re
from ctypes import c_void_p

import numpy as np
import pytest
import torch

from oracle import batch_prep_oracle as BO

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "ref_batch_prep.npz")


@pytest.fixture(scope="module")
def ref():
    return np.load(GOLDEN)


def _dicts(ref):
    pre = dict(zip(ref["pre_keys"].tolist(), ref["pre_vals"].tolist()))
    classes = {int(c): str(c) for c in ref["class_codes"].tolist()}
    return pre, classes, [str(s) for s in ref["features"].tolist()]


def test_oracle_equals_reference_transforms_bit_for_bit(ref):
    pre, classes, names = _dicts(ref)
    raw_codes = np.concatenate([ref[f"s{i}_y"] for i in range(int(ref["num_samples"]))])
    assert {0, 3, 4, 65, 66} <= set(raw_codes.tolist())
    for i in range(int(ref["num_samples"])):
        y = torch.from_numpy(ref[f"s{i}_y"])
        t = BO.target_transform(y, pre, classes)
        assert torch.equal(t, torch.from_numpy(ref[f"s{i}_target"])), i
        keep = BO.drop_points_by_class(t)
        pos = torch.from_numpy(ref[f"s{i}_pos"])[keep]
        assert torch.equal(pos, torch.from_numpy(ref[f"s{i}_pos_copy"])), i
        assert torch.equal(t[keep], torch.from_numpy(ref[f"s{i}_y_copy"])), i
        assert np.array_equal(ref[f"s{i}_idx"][keep.numpy()], ref[f"s{i}_drop_idx"]), i
        x = torch.from_numpy(ref[f"s{i}_x"])[keep]
        assert torch.equal(x, torch.from_numpy(ref[f"s{i}_drop_x"])), i
        p = BO.nullify_lowest_z(pos)
        assert torch.equal(p, torch.from_numpy(ref[f"s{i}_nullify"])), i
        p = BO.normalize_pos(p, 50)
        assert torch.equal(p, torch.from_numpy(ref[f"s{i}_normalize"])), i
        f = BO.standardize_rgb_and_intensity(x, names)
        assert torch.equal(f, torch.from_numpy(ref[f"s{i}_standardize"])), i


def test_fixture_covers_clamp_and_single_point(ref):
    """The +-3 std clamp (in standardised space, so values above 3 survive) and the n = 1 NaN std -> 1.0 path."""
    pre, classes, names = _dicts(ref)
    std = ref["s1_standardize"]
    i_col, rgb_col = names.index("Intensity"), names.index("rgb_avg")
    x = torch.from_numpy(ref["s1_drop_x"])
    lim = np.float32(3) * (torch.log(x[:, i_col] + 1).std() + 1e-6).numpy()
    assert lim > 3.0 and np.abs(std[:, i_col]).max() == pytest.approx(float(lim), rel=1e-6)  # the outliers sit on the clamp
    assert np.abs(std[:, rgb_col]).max() > 3.0  # not clamped to +-3
    assert ref["s3_standardize"].shape[0] == 1
    assert ref["s3_standardize"][0, i_col] == 0.0 and ref["s3_standardize"][0, rgb_col] == 0.0


def test_unknown_code_raises_type_error_like_the_reference(ref):
    pre, classes, _ = _dicts(ref)
    assert int(ref["unknown_raises"]) == 1
    with pytest.raises(TypeError, match=r"\[7, 8\]"):
        BO.target_transform(torch.from_numpy(ref["unknown_y"]), pre, classes)


def test_label_table_matches_target_transform(ref):
    from myria3d_b200.batch_prep import PrepConfig

    pre, classes, names = _dicts(ref)
    cfg = PrepConfig.from_dataset_description({"classification_preprocessing_dict": pre, "classification_dict": classes,
                                              "d_in": 9, "num_classes": 7}, names)
    lut = cfg.label_table()
    assert len(lut) == 256 and lut[65] == 65 and lut[66] == 65 and lut[0] == 0 and lut[3] == lut[4] == 2 and lut[7] == -1
    codes = torch.tensor([c for c in range(256) if lut[c] >= 0])
    assert torch.equal(torch.tensor([lut[c] for c in codes.tolist()]), BO.target_transform(codes, pre, classes))
    for c in range(256):
        if lut[c] < 0:
            with pytest.raises(TypeError):
                BO.target_transform(torch.tensor([c]), pre, classes)


def test_batch_prep_entry_points_validate_arguments(lib):
    """Null pointers, bad sizes and an unknown mode: B200_E_INVALID with a message, before any CUDA call."""
    P = c_void_p(256)  # never dereferenced: validation rejects the call first
    err = lambda: lib.b200_last_error().decode()  # noqa: E731
    assert lib.b200_batch_prep_stats_len(12) == 9 + 24

    args = [P, P, 9, P, P, P, 4, 1000, P, 0.25, P, P, P, P, P, P, P, None]
    assert lib.b200_batch_prep_compact(3, *args) == 1 and "unknown mode" in err()
    assert lib.b200_batch_prep_compact(0, None, *args[1:]) == 1 and "null pointer" in err()
    bad = list(args)
    bad[8] = None  # no label table in train mode
    assert lib.b200_batch_prep_compact(0, *bad) == 1 and "lut" in err()
    bad = list(args)
    bad[6] = 0  # no samples
    assert lib.b200_batch_prep_compact(0, *bad) == 1 and "bad sizes" in err()
    bad = list(args)
    bad[8 + 1] = 0.0  # grid size
    assert lib.b200_batch_prep_compact(1, *bad) == 1 and "bad sizes" in err()

    assert lib.b200_batch_prep_voxelize(P, None, P, P, P, 4, P, P, None) == 1 and "null pointer" in err()
    assert lib.b200_batch_prep_voxelize(P, P, P, P, P, 0, P, P, None) == 1 and "bad sizes" in err()
    assert lib.b200_batch_prep_pool(P, P, P, 4, 100, P, None, P, 9, P, 7, P, P, P, None) == 1 and "null pointer" in err()
    assert lib.b200_batch_prep_pool(P, P, P, 4, 100, P, P, P, 9, P, 300, P, P, P, None) == 1 and "bad sizes" in err()
    assert lib.b200_batch_prep_budget_draw(None, P, 3, 10, 0, None, P, P, P, P, None) == 1 and "null pointer" in err()
    assert lib.b200_batch_prep_budget_draw(P, P, -1, 10, 0, None, P, P, P, P, None) == 1 and "bad sizes" in err()

    fin = [P, P, 9, P, P, 4, P, P, P, 0, 7, 0.04, 0.5, 0.0, 0, None, P, P, P, P, P, P, P, P, P, P, P, None, None]
    assert lib.b200_batch_prep_finalize(7, *fin) == 1 and "unknown mode" in err()
    assert lib.b200_batch_prep_finalize(-1, *fin) == 1 and "unknown mode" in err()
    bad = list(fin)
    bad[0] = None
    assert lib.b200_batch_prep_finalize(0, *bad) == 1 and "null pointer" in err()
    bad = list(fin)
    bad[20] = None  # pos_sampled_copy is required in eval / predict
    assert lib.b200_batch_prep_finalize(1, *bad) == 1 and "copies" in err()
    bad = list(fin)
    bad[26] = None  # transformed_y_copy is required in eval
    assert lib.b200_batch_prep_finalize(1, *bad) == 1 and "target copy" in err()
    bad = list(fin)
    bad[10] = 0  # Intensity and rgb_avg in the same column
    assert lib.b200_batch_prep_finalize(0, *bad) == 1 and "bad sizes" in err()


def test_header_declares_the_batch_prep_flags():
    from myria3d_b200 import _lib, batch_prep

    header = open(os.path.join(os.path.dirname(os.path.dirname(__file__)), "include", "b200randla.h")).read()
    flags = {k: int(v) for k, v in re.findall(r"#define B200_BATCH_PREP_E_(\w+) (\d+)", header)}
    assert flags == {"UNKNOWN_CODE": batch_prep.E_UNKNOWN_CODE, "CODE_RANGE": batch_prep.E_CODE_RANGE,
                     "VOXEL_OVERFLOW": batch_prep.E_VOXEL_OVERFLOW}
    assert _lib.ABI_VERSION == 6
    assert {n for n in _lib.EXPORTED_SYMBOLS if n.startswith("b200_batch_prep_")} == {
        "b200_batch_prep_stats_len", "b200_batch_prep_compact", "b200_batch_prep_voxelize", "b200_batch_prep_pool",
        "b200_batch_prep_budget_draw", "b200_batch_prep_finalize"}


def test_raw_collater_and_prepare_batch_reject_cpu_tensors():
    from myria3d_b200 import Data, PrepConfig, RawCollater, prepare_batch

    names = ["Intensity", "rgb_avg"]
    samples = [Data(pos=torch.rand(n, 3), x=torch.rand(n, 2), y=torch.full((n,), 2), idx_in_original_cloud=np.arange(n),
                    x_features_names=names) for n in (5, 3)]
    raw = RawCollater(pin_memory=False)(samples)
    assert raw.ptr.tolist() == [0, 5, 8] and raw.x_features_names == names and len(raw.idx_in_original_cloud) == 2
    assert raw.idx_in_original_cloud_flat.tolist() == [0, 1, 2, 3, 4, 0, 1, 2]
    cfg = PrepConfig({}, {1: "a", 2: "b"}, names)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        prepare_batch(raw, "train", cfg)
    with pytest.raises(ValueError, match="unknown mode"):
        prepare_batch(raw, "test", cfg)


def test_unknown_code_message_names_raw_and_preprocessed_codes():
    from myria3d_b200.batch_prep import PrepConfig, unknown_codes_message

    cfg = PrepConfig({3: 42, 4: 5}, {1: "a", 5: "b"}, ["Intensity", "rgb_avg"])
    msg = unknown_codes_message(cfg, [3, 7])
    assert "raw codes [3, 7]" in msg and "after classification_preprocessing_dict: [7, 42]" in msg
    assert "outside the LAS code range" in unknown_codes_message(cfg, [], True)


def test_raw_collater_does_not_pin_inside_dataloader_workers(monkeypatch):
    """Pinning needs a CUDA context, which a forked worker of an initialised process cannot create."""
    from myria3d_b200 import Data, RawCollater

    calls = []
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self, *a, **k: calls.append(1) or self)
    monkeypatch.setattr(torch.utils.data, "get_worker_info", lambda: object())
    samples = [Data(pos=torch.rand(4, 3), x=torch.rand(4, 2), y=torch.full((4,), 2)) for _ in range(2)]
    RawCollater()(samples)
    assert calls == []
    monkeypatch.setattr(torch.utils.data, "get_worker_info", lambda: None)
    RawCollater()(samples)
    assert calls


def test_raw_collater_batches_come_back_from_dataloader_workers():
    """Batches collated in worker processes are pickled to the main process: Batch must survive the round trip."""
    import pickle

    from myria3d_b200 import Data, RawCollater

    names = ["Intensity", "rgb_avg"]
    samples = [Data(pos=torch.rand(n, 3), x=torch.rand(n, 2), y=torch.full((n,), 2), idx_in_original_cloud=np.arange(n),
                    x_features_names=names) for n in (4, 5, 6, 7)]
    b = pickle.loads(pickle.dumps(RawCollater(pin_memory=False)(samples[:2])))
    assert b.ptr.tolist() == [0, 4, 9] and "y" in b and b.x_features_names == names
    loader = torch.utils.data.DataLoader(samples, batch_size=2, num_workers=2, collate_fn=RawCollater())
    got = [(r.ptr.tolist(), r.idx_in_original_cloud_flat.tolist()) for r in loader]
    assert got == [([0, 4, 9], [0, 1, 2, 3, 0, 1, 2, 3, 4]), ([0, 6, 13], list(range(6)) + list(range(7)))]
