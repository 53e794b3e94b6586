"""CPU oracle of the batched train / eval / predict preparation (myria3d_b200/batch_prep.py) -- TEST INFRASTRUCTURE,
never imported by the product.  Restates, per sample and in the reference's order (pctl/datamodule/hdf5.py:76-89),

* ``TargetTransform``, ``DropPointsByClass``, ``CopyFullPos``, ``CopyFullPreparedTargets``, ``CopySampledPos``,
  ``NullifyLowestZ``, ``NormalizePos``, ``StandardizeRGBAndIntensity``  (myria3d/pctl/transforms/transforms.py) with the
  reference's own torch operations -- pinned bit for bit by tests/golden/ref_batch_prep.npz (oracle/gen_golden_ref_prep.py
  runs the reference's transforms.py on the same inputs);
* ``GridSampling`` and ``Center`` as in sample_prep_oracle.py (PyG 2.4 restated; Center with an fp64 mean), and the
  statistics of ``StandardizeRGBAndIntensity`` in fp64 like the library (``stats64``; the reference's fp32 form is the
  one the fixture pins);
* ``MinimumNumNodes`` / ``MaximumNumNodes`` / ``RandomFlip`` / ``RandomRotate`` with REPLAYED draws (the row choice, the
  flip bits, the angle), because the library's Philox stream cannot equal Python's ``random`` / torch's CPU generator.
  RandomRotate(d, axis=2) follows PyG 2.4: ``M = [[cos, sin, 0], [-sin, cos, 0], [0, 0, 1]]`` (cos / sin of the angle in
  radians, rounded to fp32) and ``pos @ M.T`` through LinearTransformation.  The angle is uniform on [-d, d], so ``M`` and
  ``M.T`` give the same distribution; this convention is the one the library implements."""
import math
from typing import Dict, Optional, Sequence

import numpy as np
import torch

from oracle import sample_prep_oracle as SO

ARTEFACT = 65


def target_transform(y: torch.Tensor, preprocessing_dict: Dict[int, int], classification_dict: Dict[int, str]) -> torch.Tensor:
    """TargetTransform.transform: preprocessing map, then the rank in classification_dict (65 -> 65); TypeError naming
    the offending codes when a code maps to nothing."""
    pre = np.array([preprocessing_dict.get(int(c), int(c)) for c in y.tolist()], dtype=np.int64)
    rank = {code: i for i, code in enumerate(classification_dict.keys())}
    rank[ARTEFACT] = ARTEFACT
    bad = sorted({int(c) for c in pre if int(c) not in rank})
    if bad:
        raise TypeError(f"unknown classification codes {bad}")
    return torch.LongTensor([rank[int(c)] for c in pre])


def drop_points_by_class(y: torch.Tensor) -> torch.Tensor:
    """DropPointsByClass: the keep mask (rows whose label is not 65)."""
    return torch.logical_not(torch.isin(y, ARTEFACT))


def nullify_lowest_z(pos: torch.Tensor) -> torch.Tensor:
    pos = pos.clone()
    pos[:, 2] = pos[:, 2] - pos[:, 2].min()
    return pos


def normalize_pos(pos: torch.Tensor, subtile_width: float = 50) -> torch.Tensor:
    return pos * (1 / (subtile_width / 2))


def standardize_channel(channel_data: torch.Tensor, clamp_sigma: int = 3) -> torch.Tensor:
    mean = channel_data.mean()
    std = channel_data.std() + 10**-6
    if torch.isnan(std):
        std = 1.0
    standard = (channel_data - mean) / std
    clamp = clamp_sigma * std
    return torch.clamp(input=standard, min=-clamp, max=clamp)


def standardize_channel64(channel_data: torch.Tensor, clamp_sigma: int = 3) -> torch.Tensor:
    """standardize_channel with the library's fp64 statistics (mean and unbiased std accumulated in fp64, then rounded
    to fp32).  It differs from the reference's fp32 reductions by round-off, except on a constant channel: there std is
    1e-6 and the reference's fp32 mean round-off (v - mean != 0) is amplified a million times, where fp64 gives 0."""
    d = channel_data.double()
    mean64 = d.mean()
    std = torch.tensor(float(((d - mean64) ** 2).sum() / (d.numel() - 1)) ** 0.5 if d.numel() > 1 else float("nan"),
                       dtype=torch.float32) + 10**-6
    if torch.isnan(std):
        std = 1.0
    standard = (channel_data - mean64.float()) / std
    clamp = clamp_sigma * std
    return torch.clamp(input=standard, min=-clamp, max=clamp)


def standardize_rgb_and_intensity(x: torch.Tensor, x_features_names: Sequence[str], stats64: bool = False) -> torch.Tensor:
    std = standardize_channel64 if stats64 else standardize_channel
    x = x.clone()
    idx = list(x_features_names).index("Intensity")
    x[:, idx] = torch.log(x[:, idx] + 1)
    x[:, idx] = std(x[:, idx])
    idx = list(x_features_names).index("rgb_avg")
    x[:, idx] = std(x[:, idx])
    return x


def center64(pos: torch.Tensor) -> torch.Tensor:
    """Center with the library's fp64 accumulation of the mean."""
    return pos - pos.double().mean(dim=0).float()


def random_flip(pos: torch.Tensor, axis: int, flip: bool) -> torch.Tensor:
    pos = pos.clone()
    if flip:
        pos[..., axis] = -pos[..., axis]
    return pos


def random_rotate_z(pos: torch.Tensor, degree: float) -> torch.Tensor:
    rad = math.pi * degree / 180.0
    s, c = math.sin(rad), math.cos(rad)
    m = torch.tensor([[c, s, 0.0], [-s, c, 0.0], [0.0, 0.0, 1.0]], dtype=torch.float32)
    return pos @ m.t()


def prepare_sample(pos, x, y, idx, mode: str, preprocessing_dict, classification_dict, x_features_names,
                   subtile_width=50, grid_size=0.25, min_nodes=300, max_nodes=40000,
                   choice: Optional[torch.Tensor] = None, flip=(False, False), angle_deg: float = 0.0,
                   rotate: bool = False, stats64: bool = True) -> dict:
    """The ``mode`` chain on one raw sample with the draws given.  Returns pos, x, y and, in eval / predict, the copies
    and idx_in_original_cloud.  ``stats64``: StandardizeRGBAndIntensity with the library's fp64 statistics (False: the
    reference's fp32 torch reductions)."""
    pos, x = pos.float(), x.float()
    y = y.long() if y is not None else None
    out = {}
    if mode != "predict":
        y = target_transform(y, preprocessing_dict, classification_dict)
    if y is not None:
        keep = drop_points_by_class(y)
        pos, x, y = pos[keep], x[keep], y[keep]
        if idx is not None:
            idx = idx[keep]
    if pos.shape[0] == 0:
        raise ValueError("sample has no point left after DropPointsByClass")
    copies = {}
    if mode != "train":
        copies["pos_copy"] = pos.clone()
        if mode == "eval":
            copies["transformed_y_copy"] = y.clone()
    yy = y if y is not None else torch.zeros(pos.shape[0], dtype=torch.int64)
    pos_g, x_g, y_g, _ = SO.grid_sampling(pos, x, yy, grid_size)
    n = pos_g.shape[0]
    s = min(max(n, min_nodes), max_nodes)
    if s != n:
        assert choice is not None and choice.numel() == s, "the budget draw must be replayed"
        pos_g, x_g, y_g = pos_g[choice], x_g[choice], y_g[choice]
    if mode != "train":
        copies["pos_sampled_copy"] = pos_g.clone()
    p = center64(pos_g)
    p = nullify_lowest_z(p)
    p = normalize_pos(p, subtile_width)
    f = standardize_rgb_and_intensity(x_g, x_features_names, stats64)
    if mode == "train":
        p = random_flip(p, 0, bool(flip[0]))
        p = random_flip(p, 1, bool(flip[1]))
        if rotate:
            p = random_rotate_z(p, float(angle_deg))
    out.update(pos=p, x=f, y=y_g)
    if mode != "train":
        out["copies"] = copies
        if idx is not None:
            out["idx_in_original_cloud"] = idx
    return out

