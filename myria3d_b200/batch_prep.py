"""Train / eval / predict batch preparation on the GPU: myria3d's sample transform chain
(``configs/datamodule/transforms/``: ``preparations/points_budget.yaml``, ``normalizations/default.yaml``,
``augmentations/{light,heavy}.yaml``), run on a whole raw batch instead of per sample in the DataLoader workers.

=========  ==================================================================================================
mode       chain (the reference's order, ``pctl/datamodule/hdf5.py:76-89``)
=========  ==================================================================================================
train      TargetTransform, DropPointsByClass, GridSampling, MinimumNumNodes, MaximumNumNodes, Center,
           NullifyLowestZ, NormalizePos, StandardizeRGBAndIntensity, RandomFlip(x), RandomFlip(y), [RandomRotate]
eval       TargetTransform, DropPointsByClass, CopyFullPos, CopyFullPreparedTargets, GridSampling, Min, Max,
           CopySampledPos, Center, NullifyLowestZ, NormalizePos, StandardizeRGBAndIntensity
predict    DropPointsByClass, CopyFullPos, GridSampling, Min, Max, CopySampledPos, Center, the three normalizations
=========  ==================================================================================================

The workers return raw samples (no transforms), :class:`RawCollater` concatenates them, the batch moves to the GPU and
:func:`prepare_batch` runs the chain as the kernels of ``csrc/batch_prep.cu``, with one device-to-host read per batch
(the per-sample voxel counts and error flags).  Random draws (budget rows, flips, rotation angles) come from the
library's Philox stream keyed by ``seed`` and the device ``counter``; the reference draws from Python's ``random`` and
torch's CPU generator, so the distributions match, not the streams.  There is no CPU fallback.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Any, Dict, List, Optional, Sequence

import torch
from torch import Tensor

from . import _lib
from .data import Batch
from .ops import _call, _need_cuda, _p, _stream

MODES = {"train": 0, "eval": 1, "predict": 2}
ARTEFACT_CODE = 65  # COMMON_CODE_FOR_ALL_ARTEFACTS, pctl/transforms/transforms.py:13
E_UNKNOWN_CODE, E_CODE_RANGE, E_VOXEL_OVERFLOW = 1, 2, 4  # B200_BATCH_PREP_E_* of include/b200randla.h
_KEPT = 9  # stats[9 + b]: rows kept by DropPointsByClass; stats[9 + B + b]: voxels after GridSampling


@dataclass
class PrepConfig:
    """Parameters of the chain.  The defaults are those of ``points_budget.yaml``, ``normalizations/default.yaml`` and
    ``augmentations/light.yaml``; ``flip_p=None`` disables the flips, ``rotate_degrees=180`` adds the rotation of
    ``augmentations/heavy.yaml``."""

    classification_preprocessing_dict: Dict[int, int]
    classification_dict: Dict[int, str]
    x_features_names: Sequence[str]
    subtile_width: float = 50
    grid_size: float = 0.25
    min_nodes: int = 300
    max_nodes: int = 40000
    flip_p: Optional[float] = 0.5
    rotate_degrees: Optional[float] = None
    _luts: Dict[Any, Tensor] = field(default_factory=dict, init=False, repr=False, compare=False)

    @classmethod
    def from_dataset_description(cls, description: Dict[str, Any], x_features_names: Sequence[str], **kwargs) -> "PrepConfig":
        """From a ``configs/dataset_description/*.yaml`` dict (``classification_preprocessing_dict``,
        ``classification_dict``; other keys ignored)."""
        return cls(dict(description["classification_preprocessing_dict"]), dict(description["classification_dict"]),
                   list(x_features_names), **kwargs)

    def label_table(self) -> List[int]:
        """``TargetTransform`` as a table over the LAS codes 0..255: rank in ``classification_dict`` of
        ``preprocessing_dict.get(code, code)``, 65 for 65 (dropped next), -1 for a code neither dict maps."""
        rank = {code: i for i, code in enumerate(self.classification_dict.keys())}
        rank[ARTEFACT_CODE] = ARTEFACT_CODE
        return [rank.get(self.classification_preprocessing_dict.get(c, c), -1) for c in range(256)]

    def _lut(self, device) -> Tensor:
        key = str(device)
        if key not in self._luts:
            self._luts[key] = _h2d(self.label_table(), torch.int32, device)
        return self._luts[key]


class RawCollater:
    """Collate raw samples (``Data`` with ``pos``, ``x``, ``y`` raw codes, optional ``idx_in_original_cloud``, and
    ``x_features_names``) as the DataLoader workers return them when the datamodule has no transforms.  Tensors are
    concatenated; ``x_features_names`` is kept once, ``idx_in_original_cloud`` as a list (as myria3d's collater does)
    and, concatenated, as ``idx_in_original_cloud_flat`` for the GPU.

    ``pin_memory=True`` pins the batch only when the collater runs in the main process.  In a DataLoader worker it does
    not: a forked worker of a process that has initialised CUDA cannot create a CUDA context, and tensors sent back from
    a worker land in shared memory anyway.  With workers, pass ``pin_memory=True`` to the DataLoader instead; it pins
    each batch in the main process through ``Batch.pin_memory``."""

    def __init__(self, pin_memory: bool = True):
        self.pin_memory = pin_memory

    def __call__(self, data_list: List[Any]) -> Batch:
        data_list = [d for d in data_list if d is not None]
        if not data_list:
            return None
        sizes = [int(d.pos.shape[0]) for d in data_list]
        ptr = [0]
        for n in sizes:
            ptr.append(ptr[-1] + n)
        out: Dict[str, Any] = {
            "pos": torch.cat([torch.as_tensor(d.pos, dtype=torch.float32) for d in data_list]),
            "x": torch.cat([torch.as_tensor(d.x, dtype=torch.float32) for d in data_list]),
            "ptr": torch.tensor(ptr, dtype=torch.int64),
        }
        if getattr(data_list[0], "y", None) is not None:
            out["y"] = torch.cat([torch.as_tensor(d.y).to(torch.int64) for d in data_list])
        names = getattr(data_list[0], "x_features_names", None)
        if names is not None:
            out["x_features_names"] = list(names)
        if getattr(data_list[0], "idx_in_original_cloud", None) is not None:
            idx = [d.idx_in_original_cloud for d in data_list]
            out["idx_in_original_cloud"] = idx
            out["idx_in_original_cloud_flat"] = torch.cat([torch.as_tensor(i).to(torch.int64) for i in idx])
        if self.pin_memory and torch.utils.data.get_worker_info() is None and torch.cuda.is_available():
            for k, v in out.items():
                if isinstance(v, Tensor):
                    out[k] = v.pin_memory()
        return Batch(**out)


def unknown_codes_message(cfg: PrepConfig, raw_codes: List[int], out_of_range: bool = False) -> str:
    """TargetTransform's error for codes that map to no class: the raw LAS codes found in the batch and, as the
    reference reports them, the same codes after ``classification_preprocessing_dict``."""
    what = []
    if raw_codes:
        pre = sorted({cfg.classification_preprocessing_dict.get(c, c) for c in raw_codes})
        what.append(f"raw codes {raw_codes} (after classification_preprocessing_dict: {pre})")
    if out_of_range:
        what.append("values outside the LAS code range 0..255")
    return (f"prepare_batch: classification {' and '.join(what)} map to no class of classification_dict "
            f"{list(cfg.classification_dict)} (classification_preprocessing_dict {cfg.classification_preprocessing_dict})")


def _h2d(values, dtype, device) -> Tensor:
    """Host list -> device tensor through pinned memory, without synchronising."""
    return torch.tensor(values, dtype=dtype).pin_memory().to(device, non_blocking=True)


def _get(batch, key):
    return getattr(batch, key) if key in batch else None


def prepare_batch(raw_batch, mode: str, cfg: PrepConfig, seed: int = 0, counter: Optional[Tensor] = None,
                  return_draws: bool = False) -> Batch:
    """Run the ``mode`` chain (``"train"``, ``"eval"`` or ``"predict"``) on a raw batch already on the GPU.

    Returns a :class:`~myria3d_b200.data.Batch` with ``x``, ``pos``, ``y`` (int64), ``batch``, ``ptr`` and the host
    tuple ``ptr_host``; in eval and predict mode also ``copies`` (``pos_copy``, ``pos_sampled_copy`` and, in eval,
    ``transformed_y_copy``) and ``idx_in_original_cloud`` (a list of per-sample device tensors) when the raw batch has
    ``idx_in_original_cloud_flat``.  ``counter`` (device int64, optional) is read, never written: advance it between
    batches for fresh draws.  With ``return_draws=True`` the batch carries ``draws``: ``flip`` (bool ``[B, 2]``),
    ``angle_deg`` (fp64 ``[B]``) and ``choice`` (per sample, the budget rows as int64 indices into the pooled sample,
    or ``None`` when the budget kept every row), enough to replay the batch.

    Raises ``TypeError`` for labels that neither class dict maps (or outside 0..255), ``ValueError`` for a sample that
    DropPointsByClass empties or whose voxel ids do not fit in 32 bits."""
    if mode not in MODES:
        raise ValueError(f"prepare_batch: unknown mode {mode!r} (expected one of {sorted(MODES)})")
    m = MODES[mode]
    pos, x, ptr = raw_batch.pos, raw_batch.x, raw_batch.ptr
    y, idx = _get(raw_batch, "y"), _get(raw_batch, "idx_in_original_cloud_flat")
    _need_cuda(pos, x, ptr, y, idx, counter)
    if y is None and mode != "predict":
        raise ValueError(f"prepare_batch: {mode} mode needs the labels y")
    names = list(_get(raw_batch, "x_features_names") or cfg.x_features_names)
    col_i, col_rgb = names.index("Intensity"), names.index("rgb_avg")
    pos = pos.float().contiguous()
    x = x.float().contiguous()
    ptr = ptr.to(torch.int64).contiguous()
    y = y.to(torch.int64).contiguous() if y is not None else None
    idx = idx.to(torch.int64).contiguous() if idx is not None else None
    dev, n, cx, nb = pos.device, pos.shape[0], x.shape[1], ptr.numel() - 1
    lib = _lib.load()
    e32 = lambda k: torch.empty(k, dtype=torch.int32, device=dev)  # noqa: E731

    # (a) - (d): everything sized from the raw batch
    lut = cfg._lut(dev) if mode != "predict" else None
    pos_c, x_c = torch.empty(n, 3, device=dev), torch.empty(n, cx, device=dev)
    y_c = torch.empty(n, dtype=torch.int64, device=dev) if y is not None else None
    idx_c = torch.empty(n, dtype=torch.int64, device=dev) if idx is not None else None
    key, val, kt, vt, run_start = e32(n), e32(n), e32(n), e32(n), e32(n)
    stats = e32(int(lib.b200_batch_prep_stats_len(nb)))
    _call("b200_batch_prep_compact", m, _p(pos), _p(x), cx, _p(y), _p(idx), _p(ptr), nb, n, _p(lut), float(cfg.grid_size),
          _p(pos_c), _p(x_c), _p(y_c), _p(idx_c), _p(key), _p(val), _p(stats), _stream())
    _call("b200_batch_prep_voxelize", _p(key), _p(val), _p(kt), _p(vt), _p(ptr), nb, _p(run_start), _p(stats), _stream())
    pos_p, x_p = torch.empty(n, 3, device=dev), torch.empty(n, cx, device=dev)
    y_p = torch.empty(n, dtype=torch.int64, device=dev) if y is not None else None
    num_classes = len(cfg.classification_dict) if mode != "predict" else 256
    _call("b200_batch_prep_pool", _p(val), _p(run_start), _p(ptr), nb, n, _p(stats), _p(pos_c), _p(x_c), cx, _p(y_c),
          num_classes, _p(pos_p), _p(x_p), _p(y_p), _stream())

    # the one device-to-host read of the batch: flags, kept rows, voxel counts (and the raw ptr)
    st = torch.cat([stats.to(torch.int64), ptr]).cpu().tolist()
    raw_ptr = st[-(nb + 1):]
    kept, voxels = st[_KEPT:_KEPT + nb], st[_KEPT + nb:_KEPT + 2 * nb]
    if st[0] & (E_UNKNOWN_CODE | E_CODE_RANGE):
        codes = [c for c in range(256) if st[1 + (c >> 5)] & (1 << (c & 31))]
        raise TypeError(unknown_codes_message(cfg, codes, bool(st[0] & E_CODE_RANGE)))
    empty = [b for b in range(nb) if kept[b] == 0]
    if empty:
        raise ValueError(f"prepare_batch: sample(s) {empty} have no point left after DropPointsByClass")
    if st[0] & E_VOXEL_OVERFLOW:
        raise ValueError(f"prepare_batch: a sample's GridSampling({cfg.grid_size}) voxel ids do not fit in 32 bits")

    # budget sizes, segments of the permutation draws, output layout -- on the host, no further sync
    sizes, choice_off, seg_off, seg_ids = [], [], [0], []
    for b, v in enumerate(voxels):
        s = min(max(v, cfg.min_nodes), cfg.max_nodes)
        sizes.append(s)
        if s == v:
            choice_off.append(-1)
            continue
        choice_off.append(seg_off[-1])
        reps = math.ceil(s / v) if v < s else 1
        for r in range(reps):
            seg_off.append(seg_off[-1] + v)
            seg_ids += [b, r]  # (sample, repetition): two words of the Philox key / counter
    out_ptr, full_ptr = [0], [0]
    for b in range(nb):
        out_ptr.append(out_ptr[-1] + sizes[b])
        full_ptr.append(full_ptr[-1] + kept[b])
    nseg, total = len(seg_ids) // 2, seg_off[-1]
    host = _h2d(choice_off + out_ptr + full_ptr + seg_off, torch.int64, dev)
    choice_off_d, out_ptr_d = host[:nb], host[nb:2 * nb + 1]
    full_ptr_d, seg_off_d = host[2 * nb + 1:3 * nb + 2], host[3 * nb + 2:]
    pk, perm, pkt, ppt = e32(max(total, 1)), e32(max(total, 1)), e32(max(total, 1)), e32(max(total, 1))
    if nseg:
        _call("b200_batch_prep_budget_draw", _p(seg_off_d), _p(_h2d(seg_ids, torch.int32, dev)), nseg, total,
              seed & 0xFFFFFFFFFFFFFFFF, _p(counter), _p(pk), _p(perm), _p(pkt), _p(ppt), _stream())

    # (f) finalize into the collated outputs
    mo = out_ptr[-1]
    pos_o, x_o = torch.empty(mo, 3, device=dev), torch.empty(mo, cx, device=dev)
    y_o = torch.empty(mo, dtype=torch.int64, device=dev) if y is not None else None
    batch_o = torch.empty(mo, dtype=torch.int64, device=dev)
    copies: Dict[str, Tensor] = {}
    if mode != "train":
        copies["pos_copy"] = torch.empty(full_ptr[-1], 3, device=dev)
        copies["pos_sampled_copy"] = torch.empty(mo, 3, device=dev)
        if mode == "eval":
            copies["transformed_y_copy"] = torch.empty(full_ptr[-1], dtype=torch.int64, device=dev)
    draws = torch.empty(nb, 3, dtype=torch.float64, device=dev) if return_draws else None
    augment = mode == "train"
    flip_p = float(cfg.flip_p) if augment and cfg.flip_p is not None else -1.0
    rotate = float(cfg.rotate_degrees) if augment and cfg.rotate_degrees else 0.0
    scale = 1 / (cfg.subtile_width / 2)  # NormalizePos.scaling_factor, applied in fp32
    _call("b200_batch_prep_finalize", m, _p(pos_p), _p(x_p), cx, _p(y_p), _p(ptr), nb, _p(perm), _p(choice_off_d),
          _p(out_ptr_d), col_i, col_rgb, scale, flip_p, rotate, seed & 0xFFFFFFFFFFFFFFFF, _p(counter), _p(pos_o), _p(x_o),
          _p(y_o), _p(batch_o), _p(copies.get("pos_sampled_copy")), _p(pos_c), _p(y_c), _p(stats), _p(full_ptr_d),
          _p(copies.get("pos_copy")), _p(copies.get("transformed_y_copy")), _p(draws), _stream())

    out: Dict[str, Any] = dict(x=x_o, pos=pos_o, y=y_o, batch=batch_o, ptr=out_ptr_d, ptr_host=tuple(out_ptr))
    if mode != "train":
        out["copies"] = copies
        if idx_c is not None:
            out["idx_in_original_cloud"] = [idx_c[raw_ptr[b]:raw_ptr[b] + kept[b]] for b in range(nb)]
    if return_draws:
        out["draws"] = {
            "flip": draws[:, :2] != 0,
            "angle_deg": draws[:, 2],
            "choice": [None if choice_off[b] < 0 else perm[choice_off[b]:choice_off[b] + sizes[b]].to(torch.int64)
                       for b in range(nb)],
        }
    return Batch(**out)
