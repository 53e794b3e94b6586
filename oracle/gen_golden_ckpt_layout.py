"""The file layout of the reference's SHIPPED Lightning checkpoint, without its bulk (tests/golden/ref_ckpt_layout.npz).

    python -m oracle.gen_golden_ckpt_layout [path/to/proto151_V2.0_epoch_100_Myria3DV3.1.0.ckpt]

TEST INFRASTRUCTURE.  The checkpoint (13.6 MB) is a torch zip archive: one pickle (``data.pkl``, 89 KB: Lightning 1.5
metadata, omegaconf hyper-parameters, torchmetrics callbacks, the ``model.*`` state dict, Adam state) plus one raw file per
tensor storage.  The fixture keeps the pickle and the ``version`` record verbatim and, per storage file, its byte count
and the ``model.*`` entry whose bytes it holds (tests/golden/randla_trained_ckpt.pt already carries those weights).  Every
other storage (Adam moments, metric states) is zero-filled on rebuild.  The rebuilt archive is read by the same loader a
user calls on the real file (``myria3d_b200.ckpt.load_lightning_checkpoint``), so the stub unpickler meets the real pickle.
"""
from __future__ import annotations

import os
import sys
import tempfile
import zipfile

import numpy as np
import torch

from myria3d_b200.ckpt import load_lightning_checkpoint, net_state_dict
from oracle.gen_golden_ckpt import CKPT

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "ref_ckpt_layout.npz")


def rebuild_checkpoint(layout: str, state_dict, out: str) -> None:
    """Write a torch zip archive at ``out`` from the fixture ``layout`` and the weights ``state_dict`` (prefix stripped)."""
    lay = np.load(layout)
    prefix = str(lay["prefix"])
    with zipfile.ZipFile(out, "w", zipfile.ZIP_STORED) as z:
        z.writestr(f"{prefix}/data.pkl", lay["data_pkl"].tobytes())
        for key, n, src in zip(lay["storage_keys"].tolist(), lay["storage_nbytes"].tolist(), lay["storage_source"].tolist()):
            blob = state_dict[src].contiguous().numpy().tobytes() if src else bytes(n)
            assert len(blob) == n, (key, src)
            z.writestr(f"{prefix}/data/{key}", blob)
        z.writestr(f"{prefix}/version", lay["version"].tobytes())


def main(path: str = CKPT):
    sd = net_state_dict(load_lightning_checkpoint(path))
    by_bytes = {}
    for name, t in sd.items():
        by_bytes.setdefault(t.contiguous().numpy().tobytes(), name)
    golden = torch.load(os.path.join(ROOT, "tests", "golden", "randla_trained_ckpt.pt"))["state_dict"]
    assert golden.keys() == sd.keys() and all(torch.equal(golden[k], v) for k, v in sd.items())

    zf = zipfile.ZipFile(path)
    names = [i.filename for i in zf.infolist()]
    prefix = names[0].split("/")[0]
    assert names[0] == f"{prefix}/data.pkl" and names[-1] == f"{prefix}/version"
    keys, nbytes, source = [], [], []
    for n in names[1:-1]:
        assert n.startswith(f"{prefix}/data/"), n
        blob = zf.read(n)
        keys.append(n[len(prefix) + 6:])
        nbytes.append(len(blob))
        source.append(by_bytes.get(blob, ""))
    np.savez_compressed(OUT, prefix=np.array(prefix), data_pkl=np.frombuffer(zf.read(names[0]), np.uint8),
                        version=np.frombuffer(zf.read(names[-1]), np.uint8), storage_keys=np.array(keys),
                        storage_nbytes=np.array(nbytes, np.int64), storage_source=np.array(source))
    with tempfile.TemporaryDirectory() as d:
        rebuild_checkpoint(OUT, golden, os.path.join(d, "rebuilt.ckpt"))
        back = net_state_dict(load_lightning_checkpoint(os.path.join(d, "rebuilt.ckpt")))
    assert back.keys() == sd.keys() and all(torch.equal(back[k], v) for k, v in sd.items())
    print(f"wrote {OUT}: {os.path.getsize(OUT) / 1e3:.0f} KB; {len(keys)} storages, "
          f"{sum(1 for s in source if s)} of them hold model.* entries")


if __name__ == "__main__":
    main(*sys.argv[1:])
