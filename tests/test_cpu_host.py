"""CPU tests of the host side: C-ABI library loads and exports every declared symbol, host logic
(BatchNorm fold, decimation bookkeeping, model zoo, Data/Batch), loud failure without a GPU."""
import os
import re

import pytest
import torch

from oracle import randla_oracle as O
from tests.helpers import assert_close, rand_cloud

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_header_symbol(lib):
    from myria3d_b200 import _lib

    header = open(os.path.join(ROOT, "include", "b200randla.h")).read()
    declared = set(re.findall(r"\b(b200_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.EXPORTED_SYMBOLS), declared ^ set(_lib.EXPORTED_SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), f"{name} not exported by libb200randla.so"
    assert lib.b200_abi_version() == _lib.ABI_VERSION == int(re.search(r"#define B200_ABI_VERSION (\d+)", header).group(1))
    assert lib.b200_last_error() == b"" or isinstance(lib.b200_last_error(), bytes)
    assert lib.b200_launch_count() >= 0


def test_library_rejects_bad_arguments_without_gpu(lib):
    """Argument validation happens before any CUDA call: error code + message, no crash."""
    from myria3d_b200 import _lib

    rc = lib.b200_knn(None, None, 0, None, None, 0, 0, 0, 16, 16, None, None, None)
    assert rc == 1 and b"null pointer" in lib.b200_last_error()
    with pytest.raises(ValueError):
        _lib.check(rc, "b200_knn")
    rc = lib.b200_lfa_fwd(None, None, None, None, None, None, None, 10, 16, 16, None)
    assert rc == 1
    # train-mode BatchNorm backward in one call: statistics, `red` and the output gradient are required
    rc = lib.b200_affine_act_bwd(None, None, 0.2, None, None, None, None, None, None, None, None, None, None, None, None, None,
                                 None, None, None, None, 100, 32, None)
    assert rc == 1 and b"b200_affine_act_bwd" in lib.b200_last_error()
    assert lib.b200_set_option(b"no_such_option", 1) == 1 and b"unknown option" in lib.b200_last_error()
    assert lib.b200_get_option(b"no_such_option") == -1


def test_no_cpu_fallback():
    from myria3d_b200 import B200RandLANet, ops

    net = B200RandLANet(9, 6)
    x, pos, batch, ptr = rand_cloud([20], seed=0)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        net(x, pos, batch, ptr)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.linear(torch.rand(4, 4), torch.rand(4, 4))


def test_fold_encoder_equals_linear_plus_batchnorm():
    """BN-moment trick (SURVEY.md App. D-7/D-8): folded affine map of q=(p_i,p_j,dist) == Linear(10->h) +
    train-mode BatchNorm over all edges, values AND gradients AND running statistics (pure torch, CPU).  The unfolded
    layers run in fp64: the Linear bias gradient is exactly zero under train-mode BatchNorm, and in fp32 torch leaves a
    residue of up to 4x the tolerance there that depends on how many threads sum the batch statistics."""
    from myria3d_b200.randla_net import SharedMLP, fold_encoder

    _, pos, _, ptr = rand_cloud([60, 7], seed=4)
    ei = O.knn_graph(pos, 16, ptr.tolist(), "brute")
    j, i = ei
    d = pos[j] - pos[i]
    dist = torch.sqrt((d * d).sum(1, keepdim=True))
    r = torch.cat([pos[i], pos[j], d, dist], 1)
    q = torch.cat([pos[i], pos[j], dist], 1)
    e = q.shape[0]
    qd = q.double()
    moments = torch.cat([torch.tensor([float(e)], dtype=torch.float64), qd.sum(0), (qd.t() @ qd).flatten()])

    for training in (True, False):
        ref = O.SharedMLP([10, 8])
        g = torch.Generator().manual_seed(1)
        bn = ref.norms[0].module
        bn.weight.data.uniform_(0.5, 1.5, generator=g), bn.bias.data.uniform_(-0.5, 0.5, generator=g)
        bn.running_mean.uniform_(-0.3, 0.3, generator=g), bn.running_var.uniform_(0.5, 1.5, generator=g)
        enc = SharedMLP([10, 8])
        enc.load_state_dict(ref.state_dict())
        ref.double()
        ref.train(training), enc.train(training)
        ref.act = False  # compare pre-activation
        z_ref = ref(r.double())
        w, b = fold_encoder(enc, moments, e, training)
        z = q @ w.t() + b
        assert_close(z, z_ref, atol=2e-5, what="folded encoder output")
        go = torch.randn(e, 8, generator=g)
        z_ref.backward(go.double())
        z.backward(go)
        for (n1, p1), (_, p2) in zip(enc.named_parameters(), ref.named_parameters()):
            assert_close(p1.grad, p2.grad, atol=2e-4, rtol=2e-4, what=f"fold grad {n1}")
        for (n1, b1), (_, b2) in zip(enc.named_buffers(), ref.named_buffers()):
            assert_close(b1, b2, atol=1e-6, rtol=1e-5, what=f"fold buffer {n1}")


def test_decimation_bookkeeping_and_errors():
    from myria3d_b200.randla_net import B200RandLANet, _Level, decimation_indices, decimation_sizes

    assert decimation_sizes([0, 12800, 12850, 12851], 4) == [0, 3200, 3212, 3213]
    with pytest.raises(ValueError, match="decimation_factor"):
        decimation_sizes([0, 10], 0)
    torch.manual_seed(3)
    idx, new_ptr = decimation_indices([0, 50, 53], 4, torch.device("cpu"))
    torch.manual_seed(3)
    idx_ref, ptr_ref = O.decimation_indices([0, 50, 53], 4)
    assert torch.equal(idx, idx_ref) and new_ptr == ptr_ref  # same RNG stream as the reference's loop
    lvl = _Level([0, 50, 53], torch.device("cpu"))
    assert lvl.max_n == 50 and lvl.num_edges(16) == 50 * 16 + 3 * 3
    with pytest.raises(ValueError):
        B200RandLANet(9, 6, num_neighbors=64)


def test_model_zoo_and_wrapper_surface():
    from myria3d_b200 import MODEL_ZOO, B200RandLANet, Model, get_neural_net_class

    assert get_neural_net_class("B200RandLANet") is B200RandLANet
    assert get_neural_net_class("RandLANet") is B200RandLANet  # substring match like models/model.py:26-28
    with pytest.raises(KeyError):
        get_neural_net_class("PyGRandLANet")  # the stock name keeps selecting the reference class
    m = Model(neural_net_class_name="B200RandLANet", neural_net_hparams=dict(num_features=2, num_classes=7),
              criterion=torch.nn.CrossEntropyLoss(ignore_index=65), lr=1e-3,
              optimizer=lambda params, lr: torch.optim.Adam(params, lr=lr), lr_scheduler=None, monitor="val/loss")
    assert isinstance(m.model, B200RandLANet) and m.model.fc0.weight.shape == (32, 2)
    assert all(k.startswith("model.") for k in m.state_dict() if "criterion" not in k)
    assert isinstance(m.configure_optimizers(), torch.optim.Adam)
    t = m._get_batch_tensor_by_enumeration([torch.zeros(3, 3), torch.zeros(2, 3)])
    assert t.tolist() == [0, 0, 0, 1, 1]
    for name in ("forward", "training_step", "validation_step", "test_step", "predict_step", "configure_optimizers"):
        assert callable(getattr(m, name))


def test_data_batch_standins():
    from myria3d_b200 import Batch, Data

    ds = [Data(x=torch.rand(n, 9), pos=torch.rand(n, 3), y=torch.zeros(n, dtype=torch.long)) for n in (5, 3)]
    b = Batch.from_data_list(ds + [None])  # None-proof like GeometricNoneProofCollater
    assert b.ptr.tolist() == [0, 5, 8] and b.batch.tolist() == [0] * 5 + [1] * 3 and b.num_graphs == 2
    assert "copies" not in b and "x" in b
    b.copies = {"pos_copy": torch.rand(4, 3)}
    assert "copies" in b and b.to("cpu").copies["pos_copy"].shape == (4, 3)


def test_state_dict_keys_match_oracle():
    from myria3d_b200 import B200RandLANet

    a = B200RandLANet(9, 7).state_dict()
    b = O.OracleRandLANet(9, 7).state_dict()
    assert list(a.keys()) == list(b.keys())
    assert all(a[k].shape == b[k].shape and a[k].dtype == b[k].dtype for k in a)


def test_fused_decimation_is_a_valid_draw():
    """One batched draw: right counts per cloud, no duplicates, indices stay inside their cloud, random order."""
    from myria3d_b200.randla_net import _Level, decimation_sizes, fused_decimation_indices

    ptr = [0, 1000, 1003, 1004, 3004]
    lvl = _Level(ptr, torch.device("cpu"))
    new_ptr = decimation_sizes(ptr, 4)
    torch.manual_seed(0)
    idx = fused_decimation_indices(lvl, new_ptr)
    assert idx.numel() == new_ptr[-1] == 250 + 1 + 1 + 500
    for b in range(4):
        part = idx[new_ptr[b]:new_ptr[b + 1]]
        assert ((part >= ptr[b]) & (part < ptr[b + 1])).all()
        assert part.unique().numel() == part.numel()
    assert not torch.equal(idx[:250], idx[:250].sort().values)  # not sorted: order is random too
    idx2 = fused_decimation_indices(lvl, new_ptr)
    assert not torch.equal(idx, idx2)
    # uniformity: every point of cloud 0 is kept ~ 1/4 of the time
    hits = torch.zeros(1000)
    for _ in range(200):
        hits[fused_decimation_indices(lvl, new_ptr)[:250]] += 1
    assert abs(float(hits.mean()) - 50.0) < 1e-6 and float(hits.std()) < 9.0


def test_synthetic_workload_matches_the_oracle_copy():
    """bench.py draws its tiles from myria3d_b200.synthetic (no oracle import on the GPU arm); the CPU reference arm and
    the tests use the oracle's copy: same seeds must give the same tensors, bit for bit."""
    import torch

    from myria3d_b200 import synthetic as S
    from oracle import randla_oracle as O

    for a, b in zip(S.synthetic_batch([700, 33], seed=4242), O.synthetic_batch([700, 33], seed=4242)):
        assert torch.equal(a, b)


def test_product_never_imports_the_oracle():
    """The package, bench.py's GPU arm and the scripts must not depend on oracle/ (test infrastructure)."""
    import pathlib
    import re as _re

    root = pathlib.Path(__file__).resolve().parents[1]
    for path in list((root / "myria3d_b200").glob("*.py")):
        assert not _re.search(r"^\s*(from|import)\s+oracle", path.read_text(), _re.M), path
    bench = (root / "bench.py").read_text()
    hits = [m.start() for m in _re.finditer(r"^\s*(from|import)\s+oracle", bench, _re.M)]
    # cpu_reference() / cpu_reference_predict() only: the cpu_baseline leg and --impl reference (configs B/E and D)
    assert len(hits) == 2
    for h in hits:
        owner = [m.group(1) for m in _re.finditer(r"^def (\w+)", bench[:h], _re.M)][-1]
        assert owner in ("cpu_reference", "cpu_reference_predict"), owner


def test_fused_decimation_many_clouds_uses_wide_keys():
    """More than 32 clouds: the (cloud id, random bits) key no longer fits 31 bits -> int64 keys, same guarantees."""
    from myria3d_b200.randla_net import _Level, decimation_sizes, fused_decimation_indices

    sizes = [37 + (i % 5) for i in range(40)]
    ptr = [0]
    for n in sizes:
        ptr.append(ptr[-1] + n)
    lvl = _Level(ptr, torch.device("cpu"))
    new_ptr = decimation_sizes(ptr, 4)
    shift, take, bits = lvl.decimation_tables(new_ptr)
    assert shift.dtype == torch.int64 and bits == 31
    idx = fused_decimation_indices(lvl, new_ptr)
    for b in range(40):
        part = idx[new_ptr[b]:new_ptr[b + 1]]
        assert part.numel() == max(1, sizes[b] // 4)
        assert ((part >= ptr[b]) & (part < ptr[b + 1])).all() and part.unique().numel() == part.numel()
    small = _Level([0, 10, 30], torch.device("cpu"))
    s32, _, bits32 = small.decimation_tables(decimation_sizes([0, 10, 30], 4))
    assert s32.dtype == torch.int32 and bits32 == 30 and int(s32.max()) == 1 << 30


def test_scratch_arena_hands_out_zeroed_disjoint_slices():
    """ops._ScratchArena (small zero-initialised reduction buffers of the backward pass): aligned disjoint slices, None when
    full (callers then fall back to torch.zeros), one clear per reset."""
    from myria3d_b200.ops import _ScratchArena

    a = _ScratchArena(torch.device("cpu"), nbytes=256)
    x = a.take(5, torch.float64)   # 40 -> 48 bytes
    y = a.take(3, torch.float32)   # 12 -> 16 bytes
    assert x.dtype == torch.float64 and x.numel() == 5 and y.numel() == 3 and a.off == 64
    assert x.data_ptr() % 16 == 0 and y.data_ptr() % 16 == 0 and y.data_ptr() - x.data_ptr() == 48
    x.fill_(7.0), y.fill_(3.0)
    assert a.take(100, torch.float32) is None  # would overflow: no partial hand-out
    assert a.off == 64
    a.reset()
    assert a.off == 0 and not a.buf.any()
    z = a.take(5, torch.float64)
    assert z.data_ptr() == x.data_ptr() and not z.any()


def test_header_is_plain_c():
    """include/b200randla.h is the drop-in boundary: it must compile as C99 (no C++-isms, no torch types) without
    warnings, and link against the built library from a C translation unit."""
    import pathlib
    import subprocess
    import tempfile

    root = pathlib.Path(__file__).resolve().parents[1]
    lib_dir = root / "myria3d_b200"
    src = ('#include "b200randla.h"\n'
           "int main(void) { return (b200_abi_version() == B200_ABI_VERSION && b200_last_error() != 0) ? 0 : 1; }\n")
    with tempfile.TemporaryDirectory() as d:
        c = pathlib.Path(d) / "t.c"
        c.write_text(src)
        subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-fsyntax-only",
                        f"-I{root / 'include'}", str(c)], check=True)
        exe = pathlib.Path(d) / "t"
        r = subprocess.run(["gcc", "-std=c99", f"-I{root / 'include'}", str(c), "-o", str(exe), f"-L{lib_dir}",
                            "-lb200randla", f"-Wl,-rpath,{lib_dir}"], capture_output=True, text=True)
        if r.returncode == 0:  # linking needs the CUDA runtime the library depends on to be resolvable here
            assert subprocess.run([str(exe)]).returncode == 0


def test_checkpoint_unpickler_does_not_resolve_code_globals(tmp_path):
    """ADVICE r1: the stub unpickler whitelists tensor-rebuilding helpers and plain containers only; a pickle that
    names builtins.eval / os.system gets inert stubs (nothing is executed) while tensors still load."""
    import pickle

    from myria3d_b200.ckpt import _StubUnpickler, load_lightning_checkpoint

    class Evil:
        def __reduce__(self):
            return (eval, ("__import__('os').system('echo pwned > %s')" % (tmp_path / "pwned"),))

    import io

    blob = pickle.dumps({"x": Evil(), "n": 3})
    out = _StubUnpickler(io.BytesIO(blob)).load()
    assert out["n"] == 3 and not (tmp_path / "pwned").exists()
    path = tmp_path / "c.ckpt"
    torch.save({"state_dict": {"model.fc0.weight": torch.ones(2, 3)}, "evil": Evil(), "epoch": 1}, path)
    ck = load_lightning_checkpoint(str(path))
    assert torch.equal(ck["state_dict"]["model.fc0.weight"], torch.ones(2, 3)) and ck["epoch"] == 1
    assert not (tmp_path / "pwned").exists()


def test_b200_options_env_is_applied_by_the_binding():
    """``B200_OPTIONS=key=value,...`` is read by the PYTHON binding and applied through the public b200_set_option (the
    library itself reads no environment); defaults: TMA row kernels on (7), one-launch BatchNorm backward off; an unknown
    key fails loudly at load time."""
    import subprocess
    import sys

    code = ("from myria3d_b200 import _lib; l = _lib.load(); "
            "print(l.b200_get_option(b'tma_rows'), l.b200_get_option(b'bn_backward_fused'), l.b200_get_option(b'tensor_core_paths'))")
    env = dict(os.environ, PYTHONPATH=ROOT)
    env.pop("B200_OPTIONS", None)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr
    assert out.stdout.split() == ["7", "0", "31"]
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT,
                         env=dict(env, B200_OPTIONS="tma_rows=3, bn_backward_fused=1"))
    assert out.returncode == 0, out.stderr
    assert out.stdout.split() == ["3", "1", "31"]
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, env=dict(env, B200_OPTIONS="no_such_option=1"))
    assert out.returncode != 0 and "unknown option" in out.stderr


def test_bench_dump_outputs_formats_and_size_limit(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 / float64 .npy files, and above the size limit the same fixed, seeded sample of
    rows of every output with the most rows (row numbers in sample_rows.npy), identical from call to call."""
    import numpy as np

    import bench

    monkeypatch.setattr(bench, "DUMP_LIMIT", 4096)
    outs = {"loss": torch.tensor(0.5), "probas": torch.rand(1000, 3), "preds": torch.arange(1000),
            "stats": torch.rand(7, dtype=torch.float64)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), outs)
    got = {p.stem: np.load(p) for p in (tmp_path / "a").glob("*.npy")}
    assert sorted(got) == ["loss", "preds", "probas", "sample_rows", "stats"]
    assert sum(a.nbytes for a in got.values()) <= 4096
    assert got["loss"].dtype == np.float32 and got["loss"].tolist() == [0.5]
    assert got["stats"].dtype == np.float64 and np.array_equal(got["stats"], outs["stats"].numpy())
    rows = got["sample_rows"].astype(np.int64)
    assert 0 < len(rows) < 1000 and (np.diff(rows) > 0).all()
    assert got["probas"].dtype == np.float32 and np.array_equal(got["probas"], outs["probas"].numpy()[rows])
    assert got["preds"].dtype == np.float64 and np.array_equal(got["preds"], rows)
    for name, a in got.items():
        assert np.array_equal(np.load(tmp_path / "b" / f"{name}.npy"), a)
