"""Minimal stand-ins for ``torch_geometric.data.Data`` / ``Batch`` as produced by myria3d's
``GeometricNoneProofCollater`` (``myria3d/pctl/dataloader/dataloader.py:19-32``): attribute bags with
``x, pos, y, batch, ptr`` (+ ``copies``, ``idx_in_original_cloud``), ``in`` and ``.to()``.

When torch_geometric is installed the real classes work unchanged with :class:`myria3d_b200.model.Model`;
these exist so the hot path can be driven (tests, bench, smoke) on a box without PyG.
"""
from __future__ import annotations

from typing import Any, Dict, Iterable, List, Optional

import torch
from torch import Tensor


class Data:
    def __init__(self, **kwargs: Any):
        self.__dict__["_store"] = dict(kwargs)

    def __getattr__(self, key: str) -> Any:
        # .get: while unpickling (DataLoader workers send batches to the main process) the store is not there yet and
        # pickle probes for __setstate__, which must then be an AttributeError
        store = self.__dict__.get("_store", {})
        if key in store:
            return store[key]
        raise AttributeError(key)

    def __setattr__(self, key: str, value: Any) -> None:
        self.__dict__["_store"][key] = value

    def __contains__(self, key: str) -> bool:
        return key in self.__dict__["_store"] and self.__dict__["_store"][key] is not None

    def keys(self) -> List[str]:
        return list(self.__dict__["_store"].keys())

    @property
    def num_nodes(self) -> int:
        return int(self.pos.shape[0])

    def to(self, device, non_blocking: bool = False):
        """Move every tensor (also inside ``copies``).  The host copy of ``ptr`` travels along as ``ptr_host`` (a
        tuple): consumers that need the batch layout on the host (``GraphedTrainStep``, ``B200RandLANet`` with
        ``static_ptr_host``) then never read the device ``ptr`` back."""
        store = self.__dict__["_store"]
        if "ptr_host" not in store and isinstance(store.get("ptr"), Tensor) and not store["ptr"].is_cuda:
            store["ptr_host"] = tuple(int(v) for v in store["ptr"].tolist())

        def move(v):
            if isinstance(v, Tensor):
                return v.to(device, non_blocking=non_blocking)
            if isinstance(v, dict):
                return {k: move(u) for k, u in v.items()}
            return v

        return type(self)(**{k: move(v) for k, v in self.__dict__["_store"].items()})

    def pin_memory(self):
        def pin(v):
            if isinstance(v, Tensor):
                return v.pin_memory()
            if isinstance(v, dict):
                return {k: pin(u) for k, u in v.items()}
            return v

        return type(self)(**{k: pin(v) for k, v in self.__dict__["_store"].items()})


class Batch(Data):
    @classmethod
    def from_data_list(cls, data_list: Iterable[Data]) -> "Batch":
        """Concatenate samples; ``batch`` / ``ptr`` like PyG's collater."""
        data_list = [d for d in data_list if d is not None]
        out: Dict[str, Any] = {}
        sizes = [d.num_nodes for d in data_list]
        tensor_keys = [k for k in data_list[0].keys() if isinstance(getattr(data_list[0], k), Tensor) and k != "batch"]
        for k in tensor_keys:
            out[k] = torch.cat([getattr(d, k) for d in data_list], dim=0)
        out["batch"] = torch.cat([torch.full((n,), i, dtype=torch.int64) for i, n in enumerate(sizes)])
        ptr = [0]
        for n in sizes:
            ptr.append(ptr[-1] + n)
        out["ptr"] = torch.tensor(ptr, dtype=torch.int64)
        if "copies" in data_list[0]:
            keys = data_list[0].copies.keys()
            out["copies"] = {k: torch.cat([d.copies[k] for d in data_list], dim=0) for k in keys}
        if "idx_in_original_cloud" in data_list[0]:
            out["idx_in_original_cloud"] = [d.idx_in_original_cloud for d in data_list]
        return cls(**out)

    @property
    def num_graphs(self) -> int:
        return int(self.ptr.numel() - 1)
