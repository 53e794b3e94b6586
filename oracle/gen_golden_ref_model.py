"""Golden vectors from the REFERENCE'S OWN MODEL CODE: myria3d/models/modules/pyg_randla_net.py is loaded from
/root/reference and executed unmodified on top of oracle/pyg_standin.py (stand-ins for the uninstallable torch_geometric /
torch_cluster / torch_scatter primitives it imports).  What this pins: the reference file's wiring, operator order,
parameter names (strict state-dict load), random-stream consumption (per-cloud randperm draws, dropout) and the
train / eval switches -- everything in the file itself.  What it cannot pin: PyG's own kernels (not installable).

    python oracle/gen_golden_ref_model.py    ->  tests/golden/ref_model_standin.pt  (~120 KB)

tests/test_cpu_oracle.py::test_oracle_equals_reference_model_code re-runs the ORACLE on the same seeds and demands
bit-identical logits, loss, gradients and BatchNorm buffers."""
import importlib.util
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import pyg_standin, randla_oracle as O  # noqa: E402

REF_FILE = "/root/reference/myria3d/models/modules/pyg_randla_net.py"
OUT = os.path.join(ROOT, "tests", "golden", "ref_model_standin.pt")
CASES = {"two_clouds": dict(sizes=[700, 300], k=16, seed=5), "ragged_k8": dict(sizes=[260, 40, 3, 120], k=8, seed=6)}


def load_reference_model_module():
    stubs = pyg_standin.modules()
    saved = {k: sys.modules.get(k) for k in stubs}
    sys.modules.update(stubs)
    try:
        spec = importlib.util.spec_from_file_location("ref_pyg_randla_net", REF_FILE)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


# Intra-op threads of every run: torch sums train-mode BatchNorm statistics in one partial per thread, so the bits of the
# train step (which the test demands exactly) depend on the count.  tests/golden/ref_model_standin.pt was made with 8.
THREADS = 8


def run_case(make_net, sizes, k, seed):
    """One eval forward + one train step under fixed seeds and THREADS threads; ``make_net`` builds either
    implementation."""
    threads = torch.get_num_threads()
    torch.set_num_threads(THREADS)
    try:
        return _run_case(make_net, sizes, k, seed)
    finally:
        torch.set_num_threads(threads)


def _run_case(make_net, sizes, k, seed):
    torch.manual_seed(seed)
    init = O.OracleRandLANet(9, 6, num_neighbors=k, return_logits=True)  # the common initial state
    g = torch.Generator().manual_seed(seed + 1)
    for m in init.modules():
        if isinstance(m, torch.nn.BatchNorm1d):
            m.weight.data.uniform_(0.7, 1.3, generator=g)
            m.bias.data.uniform_(-0.2, 0.2, generator=g)
            m.running_mean.uniform_(-0.2, 0.2, generator=g)
            m.running_var.uniform_(0.6, 1.4, generator=g)
    net = make_net(k)
    net.load_state_dict(init.state_dict(), strict=True)
    x, pos, y, batch, ptr = O.synthetic_batch(sizes, seed=seed)
    out = {}
    net.eval()
    torch.manual_seed(seed + 2)
    with torch.no_grad():
        out["eval_logits"] = net(x, pos, batch, ptr).clone()
    net.train()
    torch.manual_seed(seed + 3)
    logits = net(x, pos, batch, ptr)
    loss = F.cross_entropy(logits, y, ignore_index=65)
    loss.backward()
    out["train_logits"], out["loss"] = logits.detach().clone(), loss.detach().clone()
    out["grads"] = {n: p.grad.clone() for n, p in net.named_parameters()}
    out["buffers"] = {n: b.clone() for n, b in net.named_buffers()}
    return out


def main():
    ref = load_reference_model_module()
    golden = {}
    for name, c in CASES.items():
        golden[name] = run_case(lambda k: ref.PyGRandLANet(9, 6, decimation=4, num_neighbors=k, return_logits=True), **c)
        # keep the fixture small: full logits, every gradient's norm + the full gradients of a few layers
        g = golden[name].pop("grads")
        golden[name]["grad_norms"] = {n: v.double().norm() for n, v in g.items()}
        golden[name]["grads_full"] = {n: g[n] for n in ("fc0.weight", "block1.lfa1.mlp_attention.lins.0.weight",
                                                        "block3.lfa2.mlp_encoder.lins.0.weight", "fp2.nn.lins.0.weight",
                                                        "fc_classif.weight", "block4.mlp2.norms.0.module.weight")}
    golden["cases"] = CASES
    torch.save(golden, OUT)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
