"""Batch preparation benchmark: GPU prepare_batch (train and eval modes) against the CPU oracle chain on the same raw
batch, plus the training step on the prepared batch.  Prints one JSON line.

    python scripts/prep_bench.py [--samples 10] [--points 30000] [--iters 50] [--threads N] [--out FILE]
    python scripts/prep_bench.py --profile [--out FILE]     # per-kernel breakdown (torch.profiler), a run of its own

The raw samples follow SURVEY.md section 6 (a 50 m x 50 m Lidar HD sample: about 30 000 raw points, about 12 500 after
GridSampling(0.25)): pulses land around 8 000 footprints on a gently sloped ground with a few vegetation and roof
returns above, so the 0.25 m voxels merge as they do on real tiles.  GPU times are CUDA events around whole
prepare_batch calls (each ends with its one device-to-host read), median over --iters after a warm-up; CPU times are
the oracle chain (oracle/batch_prep_oracle.py, PyG's GridSampling restated in torch) on every sample, with the GPU's
draws replayed, at 1 thread and at --threads threads.  The batch's working set (about 30 MB of raw rows plus the
scratch buffers) fits the B200's 126 MB L2, so a 256 MB buffer is overwritten before every timed call (outside the
timed region): the GPU times are for a batch that starts in HBM, as a freshly transferred batch does.

--profile times the same calls under torch.profiler (CUDA activity) and reports, per kernel name, the device time per
prepare_batch call, with the sum of kernel time and the wall time of the profiled calls, so that the share of launch
gaps and of the one host read can be read off."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NAMES = ["Intensity", "ReturnNumber", "NumberOfReturns", "Red", "Green", "Blue", "Infrared", "rgb_avg", "ndvi"]
PRE = {3: 5, 4: 5, 0: 1, 66: 65, 100: 1, 101: 1}  # configs/dataset_description/20230601_lidarhd_pacasam_dataset.yaml
CLASSES = {1: "unclassified", 2: "ground", 5: "vegetation", 6: "building", 9: "water", 17: "bridge", 64: "lasting_above"}


def lidar_sample(n, seed):
    from myria3d_b200 import Data

    g = np.random.default_rng(seed)
    foot = g.random((8000, 2)) * 50.0
    k = g.integers(0, len(foot), n)
    xy = foot[k] + g.normal(0.0, 0.03, (n, 2))
    ground = 0.02 * xy[:, 0] + 0.01 * xy[:, 1]
    above = g.random(n) < 0.12
    z = ground + np.abs(g.normal(0.0, 0.02, n)) + above * g.random(n) * 12.0
    pos = np.stack([xy[:, 0] + 1000.0, xy[:, 1] + 2000.0, z + 100.0], 1).astype(np.float32)
    x = g.random((n, 9)).astype(np.float32)
    x[:, 0] = g.random(n).astype(np.float32) * 3000
    x[:, 7] = g.random(n).astype(np.float32) * 60000
    y = np.where(above, g.choice([3, 4, 5, 6], n), g.choice([2, 2, 2, 0, 1, 66, 65], n)).astype(np.int64)
    return Data(pos=torch.from_numpy(pos), x=torch.from_numpy(x), y=torch.from_numpy(y),
                idx_in_original_cloud=np.arange(n, dtype=np.int64), x_features_names=NAMES)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name()
    except Exception:
        return torch.cuda.get_device_name()


_FLUSH = None


def flush_l2():
    global _FLUSH
    if _FLUSH is None:
        _FLUSH = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device="cuda")  # 256 MB > 126 MB of L2
    _FLUSH.zero_()


def time_gpu(fn, iters):
    times = []
    for _ in range(iters):
        flush_l2()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        e.synchronize()
        times.append(s.elapsed_time(e))
    return float(np.median(times)), float(np.min(times))


def time_oracle(samples, mode, cfg, draws, threads):
    from oracle import batch_prep_oracle as BO

    torch.set_num_threads(threads)
    t0 = time.perf_counter()
    for b, d in enumerate(samples):
        ch = draws["choice"][b]
        BO.prepare_sample(d.pos, d.x, d.y, torch.from_numpy(d.idx_in_original_cloud), mode, PRE, CLASSES, NAMES,
                          choice=None if ch is None else ch.cpu(), flip=draws["flip"][b].tolist(),
                          angle_deg=float(draws["angle_deg"][b]), rotate=False)
    return (time.perf_counter() - t0) * 1e3


def profile(raw, cfg, counter, iters):
    """Device time per prepare_batch call and kernel name, from torch.profiler."""
    from torch.profiler import ProfilerActivity
    from torch.profiler import profile as tprofile

    from myria3d_b200 import prepare_batch

    out = {}
    for mode in ("train", "eval"):
        for _ in range(5):
            prepare_batch(raw, mode, cfg, seed=1, counter=counter)
        torch.cuda.synchronize()
        with tprofile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            t0 = time.perf_counter()
            for _ in range(iters):
                prepare_batch(raw, mode, cfg, seed=1, counter=counter)
            torch.cuda.synchronize()
            wall = (time.perf_counter() - t0) * 1e3 / iters
        kernels = {}
        for ev in prof.key_averages():
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = getattr(ev, "cuda_time_total", 0.0)
            if t and ev.device_type == torch.autograd.DeviceType.CUDA:
                kernels[ev.key[:60]] = round(t / iters, 2)
        out[f"{mode}_kernels_us_per_call"] = dict(sorted(kernels.items(), key=lambda kv: -kv[1]))
        out[f"{mode}_kernel_sum_us_per_call"] = round(sum(kernels.values()), 2)
        out[f"{mode}_wall_ms_per_call_profiled"] = round(wall, 4)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=10)
    ap.add_argument("--points", type=int, default=30000)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--threads", type=int, default=min(8, os.cpu_count() or 1))
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile", action="store_true", help="per-kernel breakdown only (torch.profiler)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prep_bench.py measures the GPU path: no CUDA device")

    from myria3d_b200 import Model, PrepConfig, RawCollater, prepare_batch
    from myria3d_b200.build import build_library

    build_library()
    samples = [lidar_sample(args.points + 37 * i, 100 + i) for i in range(args.samples)]
    raw = RawCollater()(samples).to("cuda", non_blocking=True)
    cfg = PrepConfig(PRE, CLASSES, NAMES)
    counter = torch.zeros(1, dtype=torch.int64, device="cuda")
    res = {"bench": "prep_bench", "gpu": gpu_info(), "samples": args.samples, "raw_points": int(raw.pos.shape[0])}
    if args.profile:
        res["profile"] = profile(raw, cfg, counter, args.iters)
        return _emit(res, args.out)
    res["l2"] = "256 MB overwritten before every timed GPU call"
    for mode in ("train", "eval"):
        for _ in range(5):
            prepare_batch(raw, mode, cfg, seed=1, counter=counter)
        med, best = time_gpu(lambda: prepare_batch(raw, mode, cfg, seed=1, counter=counter), args.iters)
        res[f"gpu_{mode}_ms_median"], res[f"gpu_{mode}_ms_min"] = round(med, 4), round(best, 4)
    batch = prepare_batch(raw, "train", cfg, seed=1, counter=counter, return_draws=True)
    res["prepared_points"] = int(batch.ptr_host[-1])
    res["prepared_points_per_sample_mean"] = float(np.mean(np.diff(batch.ptr_host)))
    for mode in ("train", "eval"):
        draws = prepare_batch(raw, mode, cfg, seed=1, counter=counter, return_draws=True).draws
        for th in sorted({1, args.threads}):
            time_oracle(samples[:1], mode, cfg, {k: v[:1] for k, v in draws.items()}, th)  # warm-up
            res[f"cpu_oracle_{mode}_ms_threads{th}"] = round(time_oracle(samples, mode, cfg, draws, th), 2)

    # the training step on the prepared batch (forward + loss + backward, Model.training_step)
    model = Model(neural_net_class_name="B200RandLANet",
                  neural_net_hparams=dict(num_features=9, num_classes=7, num_neighbors=16, decimation=4, return_logits=True),
                  criterion=torch.nn.CrossEntropyLoss(ignore_index=65), interpolation_k=10, num_workers=1).cuda()
    model.train()

    def step():
        out = model.training_step(batch, 0)
        out["loss"].backward()

    for _ in range(5):
        step()
    med, best = time_gpu(step, args.iters)
    res["train_step_ms_median"], res["train_step_ms_min"] = round(med, 4), round(best, 4)
    _emit(res, args.out)


def _emit(res, out):
    line = json.dumps(res)
    print(line)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
