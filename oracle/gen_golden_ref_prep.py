"""Golden vectors of the batch preparation produced by the REFERENCE'S OWN transforms (run in the build container, where
/root/reference exists): myria3d/pctl/transforms/transforms.py is loaded unmodified over the stand-ins of
gen_golden_ref.py, and ``TargetTransform`` (with the dicts of configs/dataset_description/20230601_lidarhd_pacasam_dataset.yaml),
``DropPointsByClass``, ``CopyFullPos``, ``CopyFullPreparedTargets``, ``NullifyLowestZ``, ``NormalizePos`` and
``StandardizeRGBAndIntensity`` run on seeded raw samples.  The samples hold the raw codes 0, 3, 4, 65 and 66, intensity
outliers (the +-3 std clamp) and a sample left with one point (the NaN std path).  GridSampling, Center, the flips and the
rotation come from torch_geometric, which is not installable here: they stay restated in oracle/batch_prep_oracle.py.

    python oracle/gen_golden_ref_prep.py   ->  tests/golden/ref_batch_prep.npz

TEST INFRASTRUCTURE: nothing in the product imports this; the GPU box never runs it (no /root/reference there)."""
import logging
import os
import sys
import types

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle.gen_golden_ref import REF, _Data, _load  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "ref_batch_prep.npz")
PREPROCESSING = {3: 5, 4: 5, 0: 1, 66: 65, 100: 1, 101: 1}
CLASSES = {1: "unclassified", 2: "ground", 5: "vegetation", 6: "building", 9: "water", 17: "bridge", 64: "lasting_above"}
FEATURES = ["Intensity", "ReturnNumber", "NumberOfReturns", "Red", "Green", "Blue", "Infrared", "rgb_avg", "ndvi"]
CODES = np.array([0, 1, 2, 3, 4, 5, 6, 9, 17, 64, 65, 66, 100, 101])


class _DataIn(_Data):  # `key in data` as torch_geometric's Data
    def __contains__(self, k):
        return k in self.__dict__


def raw_samples():
    """Seeded raw samples: (pos, x, y, idx_in_original_cloud)."""
    g = np.random.default_rng(31)
    out = []
    for i, n in enumerate([400, 1000, 300, 5, 500]):
        pos = np.stack([g.random(n) * 50 + 1000.0, g.random(n) * 50 + 2000.0, g.random(n) * 20 + 100.0], 1).astype(np.float32)
        x = g.random((n, len(FEATURES))).astype(np.float32)
        x[:, 0] = (g.random(n) * 3000).astype(np.float32)          # Intensity
        x[:, 7] = (g.random(n) * 60000).astype(np.float32)         # rgb_avg
        if i == 1:
            x[:7, 0] = np.float32(1e9)                               # outliers beyond 3 std after the log
            x[:7, 7] = np.float32(1e7)
        y = CODES[g.integers(0, len(CODES), n)].astype(np.int64)
        if i == 3:
            y[:] = [65, 66, 2, 65, 66]                               # one point left
        idx = np.sort(g.choice(100000, n, replace=False)).astype(np.int64)
        out.append((pos, x, y, idx))
    return out


def main():
    tg, tgd, tgt = types.ModuleType("torch_geometric"), types.ModuleType("torch_geometric.data"), types.ModuleType("torch_geometric.transforms")
    tgd.Data, tgt.BaseTransform = _DataIn, object
    m3, m3u, m3uu = types.ModuleType("myria3d"), types.ModuleType("myria3d.utils"), types.ModuleType("myria3d.utils.utils")
    m3uu.get_logger = logging.getLogger
    m3u.utils = m3uu
    tr = _load(os.path.join(REF, "myria3d/pctl/transforms/transforms.py"), "ref_transforms",
               {"torch_geometric": tg, "torch_geometric.data": tgd, "torch_geometric.transforms": tgt,
                "myria3d": m3, "myria3d.utils": m3u, "myria3d.utils.utils": m3uu})
    target = tr.TargetTransform(PREPROCESSING, CLASSES)
    out = {"features": np.array(FEATURES), "pre_keys": np.array(list(PREPROCESSING)), "pre_vals": np.array(list(PREPROCESSING.values())),
           "class_codes": np.array(list(CLASSES))}
    for i, (pos, x, y, idx) in enumerate(raw_samples()):
        d = _DataIn(pos=torch.from_numpy(pos), x=torch.from_numpy(x), y=torch.from_numpy(y), idx_in_original_cloud=idx,
                    x_features_names=list(FEATURES), num_nodes=len(y))
        out[f"s{i}_pos"], out[f"s{i}_x"], out[f"s{i}_y"], out[f"s{i}_idx"] = pos, x, y, idx
        d = target(d)
        out[f"s{i}_target"] = d.y.numpy().copy()
        d = tr.DropPointsByClass()(d)
        d = tr.CopyFullPos()(d)
        d = tr.CopyFullPreparedTargets()(d)
        out[f"s{i}_drop_idx"] = np.asarray(d.idx_in_original_cloud)
        out[f"s{i}_pos_copy"] = d.copies["pos_copy"].numpy()
        out[f"s{i}_y_copy"] = d.copies["transformed_y_copy"].numpy()
        out[f"s{i}_drop_x"] = d.x.numpy().copy()
        d = tr.NullifyLowestZ()(d)
        out[f"s{i}_nullify"] = d.pos.numpy().copy()
        d = tr.NormalizePos(subtile_width=50)(d)
        out[f"s{i}_normalize"] = d.pos.numpy().copy()
        d = tr.StandardizeRGBAndIntensity()(d)
        out[f"s{i}_standardize"] = d.x.numpy().copy()
    out["num_samples"] = np.array(i + 1)
    bad = _DataIn(y=torch.tensor([1, 7, 2, 8]), num_nodes=4)
    try:
        target(bad)
        out["unknown_raises"] = np.array(0)
    except TypeError:
        out["unknown_raises"] = np.array(1)
    out["unknown_y"] = bad.y.numpy()
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
