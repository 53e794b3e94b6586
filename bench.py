#!/usr/bin/env python
"""bench.py -- points/sec (fwd+bwd) of the RandLA-Net hot path on N x B200 (BASELINE.json metric).

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps 5 --warmup 2       # the reference's CPU path (oracle port)
    python bench.py --steps 20 --dump-outputs DIR               # + the last timed step's outputs as DIR/*.npy

One "step" = one pass of the hot path over one synthetic batch: forward + CrossEntropyLoss +
backward (+ one flat NCCL gradient all-reduce when N > 1) + Adam update, on BASELINE.json configs[1]:
full RandLA-Net (4 down / 4 up), K=16, 16 tiles x 12 800 points per GPU (weak scaling).

Prints ONE JSON line (rank 0).  `value` is timed with inputs resident in HBM; `e2e` goes through the
public `Model.training_step` with pinned HOST batches (H2D copies and the loss read-back inside the
timed region); `roofline` is the dominant library kernel timed live with CUDA events in a separate
profiling pass; `cpu_baseline` is the CPU oracle (the reference's PyTorch path restated) on a bounded
sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import torch
import torch.distributed as dist
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "points/sec (fwd+bwd) RandLA-Net 12800-pt tiles"


def metric_name(args) -> str:
    """BASELINE.json's metric for the default workload; the other configs say what they measure."""
    if args.config == "D":
        return "points/sec (predict path) RandLA-Net 40960-pt tiles"
    if args.config == "E":
        return "points/sec (fwd+bwd) RandLA-Net 65536-pt tiles, K=32"
    return METRIC
UNIT = "points/s"
NUM_FEATURES, NUM_CLASSES, K_NEIGHBORS, DECIMATION = 9, 6, 16, 4
LR = 0.003933  # configs/model/default.yaml:21-24


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--tiles", type=int, default=16, help="tiles per GPU per step (BASELINE configs[1]: 16)")
    ap.add_argument("--points", type=int, default=12800, help="points per tile")
    ap.add_argument("--cpu-tiles", type=int, default=4, help="tiles per step of the bounded CPU sample")
    ap.add_argument("--cpu-steps", type=int, default=5)
    ap.add_argument("--profile-steps", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--eager", action="store_true", help="launch every kernel from Python instead of replaying the step graph")
    ap.add_argument("--torch-adam", action="store_true", help="use torch.optim.Adam(fused=True) instead of FlatAdam")
    ap.add_argument("--decimation-rng", choices=["fused", "reference"], default="fused",
                    help="fused: one batched random draw per level; reference: per-cloud torch.randperm like the reference")
    ap.add_argument("--kernel-report", default=None, help="write the per-kernel table (JSON) here")
    ap.add_argument("--config", choices=["B", "D", "E"], default="B",
                    help="BASELINE.json workload: B = configs[1]/[2] (default: 16 x 12 800-pt tiles, K=16, train step); "
                         "E = configs[4] (4 x 65 536-pt tiles per GPU, K=32, train step); D = configs[3] (inference-only "
                         "predict path: 50 x 40 960-pt tiles per batch, k=10 interpolation to the 60 000-pt windows, stitch)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0) as DIR/<name>.npy, for comparing two builds "
                         "output for output (the inputs are seeded: the same arguments give the same inputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl b200)")
    global K_NEIGHBORS
    if args.config == "E":
        K_NEIGHBORS = 32
        args.tiles, args.points = 4, 65536
        args.cpu_tiles, args.cpu_steps = 1, 2
    elif args.config == "D":
        args.tiles, args.points = 50, 40960
        args.cpu_tiles, args.cpu_steps = 1, 2
    return args


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------ synthetic data
def host_batch(tiles: int, points: int, seed: int):
    """Synthetic 50 m x 50 m Lidar-HD-like tiles (SURVEY.md 8d) as a pinned host Batch."""
    from myria3d_b200 import Batch, Data
    from myria3d_b200.synthetic import synthetic_tile

    datas = []
    for t in range(tiles):
        x, pos, y = synthetic_tile(points, seed + t, NUM_FEATURES, NUM_CLASSES)
        datas.append(Data(x=x, pos=pos, y=y))
    return Batch.from_data_list(datas)


# ------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.gpu_index)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        try:
            rows = [r.strip().split(", ") for r in open(self.path).read().strip().splitlines() if r.strip()]
            sm = sorted(float(r[1]) for r in rows if len(r) >= 9)
            if sm:
                out["sm_mhz"] = sm[len(sm) // 2]
                out["sm_max_mhz"] = max(float(r[2]) for r in rows if len(r) >= 9)
                out["samples"] = len(sm)
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for i, nm in enumerate(names):
                    if any(r[5 + i].strip().lower() == "active" for r in rows if len(r) >= 9):
                        out["reasons"].append(nm)
            os.unlink(self.path)
        except Exception:
            pass
        return out


# ------------------------------------------------------------------------------ roofline table
def algorithmic_bytes(name: str, a):
    """Compulsory HBM bytes of one library call (SURVEY.md 8d; fp32 values, int32 neighbour ids)."""
    if name == "b200_lfa_fwd":
        n, c, kt = a
        return n * (6 * c + 12 + 4 * kt)
    if name == "b200_lfa_bwd":
        _ws, n, c, kt = a
        return n * (8 * c + 12 + 4 * kt)
    if name == "b200_knn":
        nx, ny, _clouds, _maxq, k, kt = a
        return nx * 12 + ny * (12 + 4 * kt)
    if name == "b200_knn_grid":
        nx, ny, _clouds, _mx, _my, k, kt, _ws = a
        return nx * 12 + ny * (12 + 4 * kt)
    if name == "b200_edge_moments":
        n, kt = a
        return n * (12 + 4 * kt)
    if name == "b200_linear_fwd":
        _ld1, c1, _ld2, c2, n, cout = a
        return 4 * n * (c1 + c2 + cout)
    if name == "b200_linear_bwd_input":
        _l1, c1, _l2, c2, _ws, n, cout = a
        return 4 * n * (c1 + c2 + cout)
    if name == "b200_linear_bwd_weight":
        _l1, c1, _l2, c2, _ws, n, cout = a
        return 4 * n * (c1 + c2 + cout)
    if name == "b200_affine_act_fwd":
        n, c = a
        return 4 * n * c * 2
    if name == "b200_affine_act_bwd_reduce":
        n, c = a
        return 4 * n * c * 3
    if name == "b200_affine_act_bwd_apply":
        n, c = a
        return 4 * n * c * 4
    if name in ("b200_gather_rows", "b200_scatter_rows_add"):
        n, c = a
        return n * (8 * c + 8)
    if name == "b200_knn_interp_fwd":
        ny, c, k, kt, _ld = a
        return ny * (8 * c + 8 * kt)
    if name == "b200_knn_interp_bwd":
        _ld, ny, c, k, kt = a
        return ny * (8 * c + 8 * kt)
    return 0


def algorithmic_flops(name: str, a):
    """fp32 flops of one library call in the reference formulation (SURVEY.md 8d: LFA per centre K*(2*10*c/2 + 2c^2) forward;
    backward = score recompute + dF + dW contractions (6c^2 per edge) + encoder forward/backward)."""
    if name == "b200_lfa_fwd":
        n, c, kt = a
        return n * kt * (10 * c + 2 * c * c)
    if name == "b200_lfa_bwd":
        _ws, n, c, kt = a
        return n * kt * (20 * c + 6 * c * c)
    if name == "b200_linear_fwd":
        _l1, c1, _l2, c2, n, cout = a
        return 2 * n * (c1 + c2) * cout
    if name == "b200_linear_bwd_input":
        _l1, c1, _l2, c2, _ws, n, cout = a
        return 2 * n * (c1 + c2) * cout
    if name == "b200_linear_bwd_weight":
        _l1, c1, _l2, c2, _ws, n, cout = a
        return 2 * n * (c1 + c2) * cout
    return 0


def make_roofline(table, clocks, dev, args, ms_per_step):
    """The `roofline` object of the bench line from the per-kernel table (dominant library call first)."""
    import torch

    peak, peak_src = peaks()
    roof = None
    if table:
        top = table[0]
        lib_ms = sum(g["ms"] for g in table)
        traffic, traffic_src = ncu_traffic(top["name"], tuple(top["args"]))
        flops = algorithmic_flops(top["name"], tuple(top["args"]))
        sm_max = (clocks or {}).get("sm_max_mhz") or 1965
        fma_peak = torch.cuda.get_device_properties(dev).multi_processor_count * 128 * 2 * sm_max * 1e6 / 1e12
        tfs = flops / (top["ms_per_launch"] * 1e-3) / 1e12
        roof = {"bound": "hbm", "kernel": top["name"], "kernel_args": top["args"],
                "achieved": top["gbs"], "peak": peak, "unit": "GB/s", "frac": top["gbs"] / peak,
                "traffic": traffic, "traffic_source": traffic_src,
                # the same launch against the fp32 FMA pipe (SMs x 128 lanes x 2 x max clock): the fused LFA kernels are
                # ALU-bound long before they are HBM-bound (DESIGN.md section 6)
                "fp32_fma": {"flops": flops, "achieved": tfs, "peak": fma_peak, "unit": "TFLOP/s",
                             "frac": tfs / fma_peak if fma_peak else None},
                "peak_source": peak_src, "launch_ms": top["ms_per_launch"],
                "share_of_library_time": top["ms"] / lib_ms if lib_ms > 0 else None,
                "library_ms_per_step": lib_ms,
                # the next library calls by time, same definition of `achieved` (algorithmic bytes / CUDA-event time)
                "also": [{"kernel": g["name"], "kernel_args": g["args"], "launch_ms": g["ms_per_launch"],
                          "achieved": g["gbs"], "frac": g["gbs"] / peak,
                          "traffic": ncu_traffic(g["name"], tuple(g["args"]))[0]}
                         for g in table[1:9] if g["alg_bytes"] > 0]}
        report = args.kernel_report
        if report:
            with open(report, "w") as f:
                json.dump({"ms_per_step": ms_per_step, "kernels": table}, f, indent=1)
    return roof


def ncu_traffic(name: str, a):
    """dram bytes per launch of this kernel/shape from the committed single-kernel ncu capture, else None."""
    try:
        path = os.path.join(ROOT, "profiles", "ncu_traffic_r02.json")
        if not os.path.exists(path):
            path = os.path.join(ROOT, "profiles", "ncu_traffic_r01.json")
        with open(path) as f:
            entries = json.load(f)["entries"]
    except Exception:
        return None, None
    named = {}
    if name == "b200_lfa_bwd":
        named = dict(zip(("ws", "n", "c", "kt"), a))
    elif name == "b200_lfa_fwd":
        named = dict(zip(("n", "c", "kt"), a))
    elif name == "b200_knn_grid":
        named = dict(zip(("nx", "ny", "clouds", "mx", "my", "k", "kt", "ws"), a))
    for e in entries:
        if e["kernel"] == name and all(named.get(k) == v for k, v in e["match"].items()):
            return int(e["dram_bytes"]), e["source"]
    return None, None


def kernel_table(records):
    groups = {}
    for name, ints, ms in records:
        g = groups.setdefault((name, ints), {"name": name, "args": list(ints), "launches": 0, "ms": 0.0})
        g["launches"] += 1
        g["ms"] += ms
    rows = sorted(groups.values(), key=lambda g: -g["ms"])
    for g in rows:
        g["ms_per_launch"] = g["ms"] / g["launches"]
        g["alg_bytes"] = algorithmic_bytes(g["name"], tuple(g["args"]))
        g["gbs"] = g["alg_bytes"] / (g["ms_per_launch"] * 1e-3) / 1e9 if g["ms_per_launch"] > 0 else 0.0
    return rows


# ------------------------------------------------------------------------------ training state of the timed steps
def _state_tensors(model, opt) -> list:
    """Every tensor a training step updates: parameters, BatchNorm buffers, optimizer state."""
    ts = [p.data for p in model.parameters()] + list(model.buffers())
    ts += [getattr(opt, a) for a in ("flat_params", "exp_avg", "exp_avg_sq", "step_count") if hasattr(opt, a)]
    return ts + [v for st in opt.state.values() for v in st.values() if isinstance(v, torch.Tensor)]


def training_state(model, opt) -> dict:
    """A copy of the training state, keyed by storage range."""
    return {(t.data_ptr(), t.numel(), t.dtype): t.clone() for t in _state_tensors(model, opt)}


def restore_training_state(model, opt, state: dict) -> None:
    """Put back a ``training_state`` copy in place (a captured step graph keeps its addresses).  Optimizer state created
    after the copy (torch.optim.Adam's, on its first step) goes back to zero, as it was before that step."""
    with torch.no_grad():
        for t in _state_tensors(model, opt):
            saved = state.get((t.data_ptr(), t.numel(), t.dtype))
            if saved is None:
                t.zero_()
            else:
                t.copy_(saved)


# ------------------------------------------------------------------------------ --dump-outputs
DUMP_LIMIT = 64 << 20  # bytes of all dumped arrays together


def dump_outputs(out_dir: str, outputs: dict) -> None:
    """``out_dir/<name>.npy`` per output: float64 and integer outputs as float64 (exact), the others as float32.  Above
    DUMP_LIMIT in all, the outputs with the most rows are cut to one fixed, seeded sample of rows (the same rows for
    each of them, their row numbers in ``sample_rows.npy``)."""
    import numpy as np

    arrays = {}
    for name, t in outputs.items():
        a = np.atleast_1d(t.detach().cpu().numpy())
        wide = a.dtype == np.float64 or np.issubdtype(a.dtype, np.integer)
        arrays[name] = a.astype(np.float64 if wide else np.float32)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        n = max(a.shape[0] for a in arrays.values())
        big = [k for k, a in arrays.items() if a.shape[0] == n]
        rest = total - sum(arrays[k].nbytes for k in big)
        keep = (DUMP_LIMIT - rest) // (sum(arrays[k].nbytes // n for k in big) + 8)
        assert keep > 0, "the outputs do not fit --dump-outputs' size limit"
        rows = np.sort(np.random.default_rng(0).choice(n, size=keep, replace=False))
        arrays = {k: (a[rows] if k in big else a) for k, a in arrays.items()}
        arrays["sample_rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a))


# ------------------------------------------------------------------------------ CPU reference arm
def cpu_reference(tiles: int, points: int, steps: int, warmup: int):
    """The reference's CPU PyTorch path (oracle port): train-mode fwd + CE + bwd + Adam, kd-tree kNN."""
    from oracle import randla_oracle as O

    cores = os.cpu_count() or 1
    torch.manual_seed(12345)
    net = O.OracleRandLANet(NUM_FEATURES, NUM_CLASSES, decimation=DECIMATION, num_neighbors=K_NEIGHBORS,
                            return_logits=True)
    net.train()
    opt = torch.optim.Adam(net.parameters(), lr=LR)
    x, pos, y, batch, ptr = O.synthetic_batch([points] * tiles, seed=12345, num_features=NUM_FEATURES,
                                              num_classes=NUM_CLASSES)

    def step():
        opt.zero_grad()
        logits = net(x, pos, batch, ptr)
        loss = F.cross_entropy(logits, y, ignore_index=65)
        loss.backward()
        opt.step()
        return float(loss.detach())

    # "all the host threads it can use": torch's intra-op pool is NOT monotone in the thread count on
    # many-core hosts (the [N, c] ops here are small), so take the fastest of a few pool sizes.
    candidates = sorted({min(cores, t) for t in (8, 16, 32)})  # >32 threads measured 10-25x SLOWER on the 128-core box
    best_t, best_dt = candidates[0], float("inf")
    torch.set_num_threads(candidates[0])
    step()  # lazy initialisation (first call is several times slower)
    for t in candidates:
        torch.set_num_threads(t)
        step()
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        if dt < best_dt:
            best_t, best_dt = t, dt
    torch.set_num_threads(best_t)

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return {"value": tiles * points / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{tiles} tiles x {points} pts per step, {warmup} warm-up + {steps} timed steps, "
                      f"oracle/randla_oracle.py (pure torch CPU + scipy cKDTree, 1 kNN worker); "
                      f"{best_t} torch threads = fastest of {candidates} on a {cores}-core host",
            "ms_per_step": dt * 1e3}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.config == "D":
        res = cpu_reference_predict(args.cpu_tiles, args.points, min(args.steps, 3), 1)
    else:
        res = cpu_reference(args.cpu_tiles, args.points, args.steps if args.config == "B" else min(args.steps, 3),
                            max(args.warmup, 1) if args.config == "B" else 1)
    line = {
        "impl": "reference", "metric": metric_name(args), "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, max(int(args.gpus), 1), "reference"), "impl_detail": impl_detail(args, "reference"),
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world, impl="b200"):
    """`config`: the WORKLOAD, identical in the b200 and the reference arm (the driver compares the two lines)."""
    which = {"B": "configs[1]" + ("/[2]" if world > 1 else ""), "E": "configs[4]", "D": "configs[3]"}[args.config]
    per_tile = FULL_POINTS if args.config == "D" else args.points
    return {
        "workload": f"RandLA-Net full (4 down/4 up), K={K_NEIGHBORS}, {args.points} pts/tile, batch={args.tiles}/GPU "
                    f"(BASELINE {which})",
        "num_features": NUM_FEATURES, "num_classes": NUM_CLASSES, "global_batch_tiles": args.tiles * world,
        "points_per_step": args.tiles * per_tile * world, "parallelism": f"dp{world}",
        "l2": "GPU arm: 256 MiB buffer rewritten between timed steps (outside the event pairs), rotating input batches; "
              "CPU arm: not applicable",
    }


def impl_detail(args, impl="b200"):
    """How this arm runs the workload (kept out of `config` so that both arms print the same `config`)."""
    if args.config == "D":
        step = ("inference only: eval forward + k=10 interpolation of the logits to the 60 000-point windows + sliding-window "
                "stitch (scatter-sum, softmax, argmax, entropy); value counts FULL-cloud points")
        if impl == "reference":
            step += f"; reference CPU path on a bounded sample of {args.cpu_tiles} window(s) per step"
        return {"step": step}
    return {
        "optimizer": ("torch.optim.Adam (CPU)" if impl == "reference" else
                      "torch.optim.Adam(fused)" if getattr(args, "torch_adam", False) else "FlatAdam (b200_adam_flat)"),
        "step": "fwd + CrossEntropyLoss + bwd + flat NCCL grad all-reduce (N>1) + Adam; "
                + ("reference CPU path: eager PyTorch, bounded sample of "
                   f"{args.cpu_tiles} tiles per step" if impl == "reference" else
                   ("eager launches" if args.eager else "whole step replayed as one CUDA graph (GraphedTrainStep)")),
        "decimation_rng": "per-cloud torch.randperm" if impl == "reference" else args.decimation_rng,
        **({} if impl == "reference" else {
            "timed_state": "every resident timed step trains the seeded initial weights and optimizer state (put back "
                           "outside the event pairs), so what it computes depends on its arguments only"}),
    }


# ------------------------------------------------------------------------------ config D: predict path
FULL_POINTS = 60000   # points of a 50 m window before the 40 960-point budget (docs/source/background/general_design.md:42)
WINDOW_STRIDE = 45000  # consecutive windows share 15 000 points of the stitched cloud (sliding-window overlap)
CLASSES = {1: "unclassified", 2: "ground", 6: "building", 9: "water", 17: "bridge", 64: "lasting_above"}


def predict_batch(tiles: int, sub: int, seed: int, first_point: int = 0):
    """Host batch of `tiles` receptive fields as myria3d's predict dataloader yields them: the sub-sampled cloud the
    network sees, `copies` with the full-resolution positions, `idx_in_original_cloud` for the stitch."""
    import numpy as np

    from myria3d_b200 import Batch, Data
    from myria3d_b200.synthetic import synthetic_tile

    g = torch.Generator().manual_seed(seed)
    datas = []
    for w in range(tiles):
        x, pos, y = synthetic_tile(FULL_POINTS, seed=seed + w, num_features=NUM_FEATURES, num_classes=NUM_CLASSES)
        keep = torch.randperm(FULL_POINTS, generator=g)[:sub]
        d = Data(x=x[keep], pos=pos[keep], y=y[keep])
        d.copies = {"pos_copy": pos, "pos_sampled_copy": pos[keep]}
        lo = first_point + w * WINDOW_STRIDE
        d.idx_in_original_cloud = np.arange(lo, lo + FULL_POINTS, dtype=np.int64)
        datas.append(d)
    return Batch.from_data_list(datas), first_point + WINDOW_STRIDE * (tiles - 1) + FULL_POINTS


def cpu_reference_predict(tiles: int, sub: int, steps: int, warmup: int):
    """The reference's CPU predict path (oracle port): eval forward, k=10 interpolation to the full window
    (models/model.py:86-98), scatter-sum stitch + softmax + argmax + entropy (models/interpolation.py:98-166)."""
    from oracle import randla_oracle as O

    torch.manual_seed(12345)
    torch.set_num_threads(min(os.cpu_count() or 1, 16))
    net = O.OracleRandLANet(NUM_FEATURES, NUM_CLASSES, decimation=DECIMATION, num_neighbors=K_NEIGHBORS, return_logits=True).eval()
    batch, nb = predict_batch(tiles, sub, 12345)
    ptr_y = [0]
    for a in batch.idx_in_original_cloud:
        ptr_y.append(ptr_y[-1] + len(a))
    idx = torch.cat([torch.from_numpy(a) for a in batch.idx_in_original_cloud])

    def step():
        with torch.no_grad():
            logits = net(batch.x, batch.pos, batch.batch, batch.ptr)
            full = O.knn_interpolate(logits, batch.copies["pos_sampled_copy"], batch.copies["pos_copy"],
                                     [int(v) for v in batch.ptr], ptr_y, 10)
            red = torch.zeros(nb, NUM_CLASSES).index_add_(0, idx, full)
            probas = red[idx].softmax(1)
            return probas.argmax(1), torch.distributions.Categorical(probs=probas).entropy()

    for _ in range(max(warmup, 1)):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return {"value": tiles * FULL_POINTS / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{tiles} windows of {FULL_POINTS} pts ({sub} after sub-sampling) per step, {warmup} warm-up + {steps} "
                      "timed steps, oracle eval forward + kd-tree k=10 interpolation + torch scatter stitch",
            "ms_per_step": dt * 1e3}


def run_b200_predict(args):
    """BASELINE configs[3]: inference only.  A step = one predict batch: eval forward on `tiles` receptive fields of
    `points` points, k=10 interpolation of the logits to every point of the 60 000-point windows, sliding-window stitch.
    Multi-GPU = independent replicas on different tiles (no collective on the data path)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import datetime

        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))
    from myria3d_b200 import Model, _lib, ops
    from myria3d_b200.build import build_library
    from myria3d_b200.interpolation import Interpolator

    if rank == 0:
        build_library()
    if world > 1:
        dist.barrier()
    _lib.check(_lib.load().b200_check_device(), "b200_check_device")
    torch.manual_seed(12345)
    model = Model(neural_net_class_name="B200RandLANet",
                  neural_net_hparams=dict(num_features=NUM_FEATURES, num_classes=NUM_CLASSES, num_neighbors=K_NEIGHBORS,
                                          decimation=DECIMATION, return_logits=True),
                  criterion=torch.nn.CrossEntropyLoss(ignore_index=65), interpolation_k=10, num_workers=1).to(dev).eval()
    model.model.decimation_rng = "fused"
    n_rot = 2
    host, nb_points = [], 0
    for r in range(n_rot):
        b, nb_points = predict_batch(args.tiles, args.points, 5000 + 1000 * rank + 100 * r)
        host.append(b.pin_memory())
    resident = [b.to(dev) for b in host]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    h2d = sum(t.numel() * t.element_size() for t in (host[0].x, host[0].pos, host[0].batch, host[0].ptr,
                                                     host[0].copies["pos_copy"], host[0].copies["pos_sampled_copy"]))
    out_host = torch.empty(args.tiles * FULL_POINTS, dtype=torch.int64).pin_memory()

    def step(batch):
        with torch.no_grad():
            _, logits = model.forward(batch)  # network + k=10 interpolation on the GPU (SURVEY 8f-1)
            itp = Interpolator(interpolation_k=10, classification_dict=CLASSES)
            itp.store_predictions(logits, batch.idx_in_original_cloud)
            reduced, idx, _ = itp._reduce(nb_points)
            return ops.stitch_finalize(reduced, idx, want_logits=False)  # probas, preds, entropy per prediction

    copy_stream = torch.cuda.Stream(device=dev)

    def upload(b):  # pinned host batch -> device on the copy stream (what a prefetching predict DataLoader does)
        with torch.cuda.stream(copy_stream):
            d = b.to(dev, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return d, ev

    last = {}  # --dump-outputs: the outputs of the last timed resident step

    def timed(kind, steps):
        evs = []
        pending = upload(host[0]) if kind == "e2e" else None
        torch.cuda.synchronize()
        for s in range(steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            if kind == "resident":
                res = step(resident[s % n_rot])
                if args.dump_outputs is not None and s + 1 == steps:
                    last["res"] = res
                del res  # freed before the next step, as the outputs of a discarded call are
            else:
                # every timed iteration holds one full-batch H2D copy (the NEXT batch's, running under this batch's
                # kernels), this batch's compute and the read-back of its predicted classes
                d, ev = pending
                torch.cuda.current_stream().wait_event(ev)
                res = step(d)
                pending = upload(host[(s + 1) % n_rot])
                out_host.copy_(res[2], non_blocking=True)  # predicted classes of the batch's points back to the host
                torch.cuda.current_stream().synchronize()
                del d
            e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs)

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for s in range(max(args.warmup, 3)):
        step(resident[s % n_rot])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = _lib.launch_count()
    total_ms = max_over_ranks(timed("resident", args.steps))
    launches = (_lib.launch_count() - l0) // max(args.steps, 1)
    dumped = None
    if rank == 0 and args.dump_outputs is not None:
        _, probas, preds, entropy = last.pop("res")
        dumped = {"probas": probas.cpu(), "preds": preds.cpu(), "entropy": entropy.cpu()}
    if world > 1:
        dist.barrier()
    e2e_ms = max_over_ranks(timed("e2e", args.steps))
    clocks = sampler.stop() if rank == 0 else None
    table = []
    if rank == 0 and args.profile_steps > 0:  # per-kernel pass (CUDA events around every library call) for `roofline`
        prof = _lib.KernelProfiler()
        _lib.PROFILER = prof
        for s in range(args.profile_steps):
            step(resident[s % n_rot])
        _lib.PROFILER = None
        torch.cuda.synchronize()
        table = kernel_table([(n, i, ms_ / 1.0) for n, i, ms_ in prof.summary()])
        for g in table:
            g["ms"] /= args.profile_steps
            g["launches"] //= args.profile_steps
    if rank == 0:
        pts = args.tiles * FULL_POINTS
        ms = total_ms / args.steps
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            res = cpu_reference_predict(args.cpu_tiles, args.points, args.cpu_steps, 1)
            cpu = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")}
        cfg = workload_config(args, world)
        line = {"metric": "points/sec (predict path) RandLA-Net 40960-pt tiles", "value": pts * world / (ms * 1e-3), "unit": UNIT,
                "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
                "impl_detail": impl_detail(args), "clocks": clocks,
                "gpu_launches": int(launches),
                "e2e": {"value": pts * world / (e2e_ms / args.steps * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                        "d2h_bytes_per_step": int(out_host.numel() * 8), "ms_per_step": e2e_ms / args.steps},
                "roofline": make_roofline(table, clocks, dev, args, ms), "cpu_baseline": cpu}
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()

# ------------------------------------------------------------------------------ B200 arm
def run_b200(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import datetime

        # a collective that cannot complete (one rank died) aborts after 3 minutes instead of NCCL's default 10
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))

    from myria3d_b200 import Model, _lib
    from myria3d_b200.build import build_library
    from myria3d_b200.graphed import GraphedTrainStep
    from myria3d_b200.parallel import FlatGradAllReducer, broadcast_module_state

    if rank == 0:
        build_library()
    if world > 1:
        dist.barrier()
    lib = _lib.load()
    _lib.check(lib.b200_check_device(), "b200_check_device")

    torch.manual_seed(12345)
    model = Model(neural_net_class_name="B200RandLANet",
                  neural_net_hparams=dict(num_features=NUM_FEATURES, num_classes=NUM_CLASSES, num_neighbors=K_NEIGHBORS,
                                          decimation=DECIMATION, return_logits=True),
                  criterion=torch.nn.CrossEntropyLoss(ignore_index=65), lr=LR).to(dev)
    model.train()
    broadcast_module_state(model)
    reducer = FlatGradAllReducer(model)
    if args.torch_adam:
        opt = torch.optim.Adam(model.parameters(), lr=LR, capturable=not args.eager, fused=True)
    else:
        from myria3d_b200.optim import FlatAdam

        opt = FlatAdam(model, lr=LR, reducer=reducer)  # torch.optim.Adam arithmetic, one kernel over flat buffers
    model.model.decimation_rng = args.decimation_rng
    initial = training_state(model, opt)
    graphed = None if args.eager else GraphedTrainStep(model, opt, reducer, decimation_rng=args.decimation_rng)

    n_rot = 4
    host = [host_batch(args.tiles, args.points, 12345 + 1000 * rank + 100 * r).pin_memory() for r in range(n_rot)]
    resident = [b.to(dev) for b in host]
    h2d_bytes = sum(t.numel() * t.element_size() for t in (host[0].x, host[0].pos, host[0].y, host[0].batch, host[0].ptr))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    points_per_step = args.tiles * args.points

    def train_step(batch):
        if graphed is not None:
            return graphed(batch)
        return eager_step(batch)

    eager_out = {}

    def eager_step(batch):
        reducer.zero_grad()
        out = model.training_step(batch, 0)
        out["loss"].backward()
        reducer.all_reduce()
        opt.step()
        if args.dump_outputs is not None:
            eager_out.update(loss=out["loss"].detach(), logits=out["logits"].detach(), targets=out["targets"])
        return out["loss"]

    def timed(kind: str, steps: int):
        evs = []
        for s in range(steps):
            if kind == "resident":
                restore_training_state(model, opt, initial)
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            if kind == "resident":
                train_step(resident[s % n_rot])
            elif graphed is not None:
                # the public loop of GraphedTrainStep: pinned host batch in, loss out; the NEXT batch's host->device copy is
                # started right behind the replay (prefetch) and overlaps with it -- one H2D copy per timed iteration
                loss = graphed(host[s % n_rot])
                graphed.prefetch(host[(s + 1) % n_rot])
                loss.item()  # device -> host read of the step's result
            else:
                b = host[s % n_rot].to(dev, non_blocking=True)
                loss = train_step(b)
                loss.item()  # device -> host read of the step's result
            e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs)  # ms

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v: float) -> float:
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- warm-up, then the resident-input measurement
    for s in range(max(args.warmup, 3)):
        train_step(resident[s % n_rot])
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    def launches_now():
        return graphed.library_launches if graphed is not None else _lib.launch_count()

    launches0 = launches_now()
    barrier()
    ncu_range = os.environ.get("B200_NCU_RANGE") == "1"  # `ncu --profile-from-start off`: capture the timed steps only
    if ncu_range:
        torch.cuda.profiler.start()
    total_ms = timed("resident", args.steps)
    if ncu_range:
        torch.cuda.profiler.stop()
    barrier()
    launches = (launches_now() - launches0) // max(args.steps, 1)
    total_ms = max_over_ranks(total_ms)
    dumped = None
    if rank == 0 and args.dump_outputs is not None:
        # what the caller of the last timed step receives (GraphedTrainStep.last_outputs)
        outs = graphed.last_outputs(resident[(args.steps - 1) % n_rot]) if graphed is not None else eager_out
        dumped = {k: outs[k].cpu() for k in ("loss", "logits", "targets")}
    # ---- end-to-end through Model.training_step with host batches
    for s in range(2):
        train_step(host[s % n_rot].to(dev, non_blocking=True)).item()
    if graphed is not None:
        graphed.prefetch(host[0])  # what the previous iteration of a running loop would have done
    barrier()
    e2e_ms = timed("e2e", args.steps)
    barrier()
    e2e_ms = max_over_ranks(e2e_ms)
    clocks = sampler.stop() if rank == 0 else None

    # ---- per-kernel pass (CUDA events around every library call) for the roofline object
    table = []
    if args.profile_steps > 0:
        # every rank runs the eager steps (they contain the gradient all-reduce); rank 0 records the launches
        prof = _lib.KernelProfiler() if rank == 0 else None
        _lib.PROFILER = prof
        for s in range(args.profile_steps):
            eager_step(resident[s % n_rot])  # eager: CUDA events around every library call
        _lib.PROFILER = None
        torch.cuda.synchronize()
    if rank == 0 and args.profile_steps > 0:
        recs = prof.summary()
        table = kernel_table([(n, i, ms / 1.0) for n, i, ms in recs])
        for g in table:
            g["ms"] /= args.profile_steps
            g["launches"] //= args.profile_steps
    if world > 1:
        dist.barrier()

    if rank == 0:
        ms_per_step = total_ms / args.steps
        value = points_per_step * world / (ms_per_step * 1e-3)
        e2e_val = points_per_step * world / (e2e_ms / args.steps * 1e-3)
        roof = make_roofline(table, clocks, dev, args, ms_per_step)
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            res = cpu_reference(args.cpu_tiles, args.points, args.cpu_steps, 2)
            cpu = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")}
        line = {
            "metric": metric_name(args), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args, world),
            "impl_detail": impl_detail(args),
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": 4,
                    "ms_per_step": e2e_ms / args.steps,
                    "loop": ("loss = step(host_batch); step.prefetch(next_host_batch); loss.item() -- every timed iteration "
                             "holds one pinned-host -> device copy of a full batch (the next step's, overlapping the replay) "
                             "and the loss read-back" if graphed is not None else
                             "batch.to(device); eager step; loss.item()")},
            "roofline": roof, "cpu_baseline": cpu,
        }
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    elif args.config == "D":
        run_b200_predict(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
