"""CUDA-graph step (GraphedTrainStep) vs the eager step: same losses, parameters move identically."""
import copy

import pytest
import torch

from oracle import randla_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _model(seed=0):
    from myria3d_b200 import Model

    torch.manual_seed(seed)
    return Model(neural_net_class_name="B200RandLANet",
                 neural_net_hparams=dict(num_features=9, num_classes=6, num_neighbors=16, decimation=4, return_logits=True),
                 criterion=torch.nn.CrossEntropyLoss(ignore_index=65), lr=1e-3).to(DEV).train()


def _batch(sizes, seed):
    from myria3d_b200 import Batch, Data

    datas = []
    for i, n in enumerate(sizes):
        x, pos, y = O.synthetic_tile(n, seed + i)
        datas.append(Data(x=x, pos=pos, y=y))
    return Batch.from_data_list(datas)


def test_graphed_forward_matches_eager(lib):
    """The loss a replay reports == the eager training_step loss at the same parameters, same decimation
    subsets (dropout disabled so the two Philox consumers cannot differ)."""
    from myria3d_b200.graphed import GraphedTrainStep
    from myria3d_b200.parallel import FlatGradAllReducer

    m = _model(1)
    m.model.mlp_classif.dropout = [0.0, 0.0]
    opt = torch.optim.Adam(m.parameters(), lr=1e-3, capturable=True)
    step = GraphedTrainStep(m, opt, FlatGradAllReducer(m))
    b = _batch([900, 400], 3).pin_memory()
    step(b)  # capture (3 eager warm-up steps) + first replay
    key = tuple(b.ptr.tolist())
    for _ in range(3):
        snap = copy.deepcopy(m)  # parameters before the replay
        loss_g = float(step(b))
        cap = step._captured[key]
        snap.model.injected_decimation_idx = [t.clone() for t in cap.idx_static]
        out = snap.training_step(b.to(DEV), 0)
        assert abs(float(out["loss"].detach()) - loss_g) < 1e-4, (float(out["loss"].detach()), loss_g)
    assert step.library_launches >= 4 * 200


def test_graphed_step_trains(lib):
    """Loss decreases over replays on a fixed batch; one graph per layout; e2e from pinned host memory."""
    from myria3d_b200.graphed import GraphedTrainStep

    m = _model(2)
    opt = torch.optim.Adam(m.parameters(), lr=3e-3, capturable=True)
    step = GraphedTrainStep(m, opt)
    b = _batch([700, 700], 5).pin_memory()
    first = float(step(b))
    for _ in range(30):
        last = float(step(b))
    assert last < first, (first, last)
    assert len(step._captured) == 1
    b2 = _batch([500, 300, 200], 9)
    step(b2.to(DEV))
    assert len(step._captured) == 2
    assert torch.isfinite(step.last_outputs(b2)["logits"]).all()


def test_flat_adam_matches_torch_adam(lib):
    """b200_adam_flat == torch.optim.Adam on the same gradients over several steps (parameters as flat views)."""
    from myria3d_b200.optim import FlatAdam

    torch.manual_seed(0)
    # (no BatchNorm right after a Linear: that Linear's bias has a mathematically zero gradient, whose fp32 noise Adam
    # normalises to +-lr steps -- any two Adam implementations diverge there by O(lr))
    net_a = torch.nn.Sequential(torch.nn.Linear(9, 33), torch.nn.Tanh(), torch.nn.Linear(33, 7)).to(DEV)
    net_b = copy.deepcopy(net_a)
    opt_a = torch.optim.Adam(net_a.parameters(), lr=3e-3, betas=(0.9, 0.999), eps=1e-8)
    opt_b = FlatAdam(net_b, lr=3e-3)
    for s in range(5):
        x = torch.randn(64, 9, device=DEV)
        for net, opt in ((net_a, opt_a), (net_b, opt_b)):
            opt.zero_grad()
            net(x).square().mean().backward()
            opt.step()
    for pa, pb in zip(net_a.parameters(), net_b.parameters()):
        assert torch.allclose(pa, pb, atol=1e-6, rtol=1e-5), float((pa - pb).abs().max())
    assert int(opt_b.step_count) == 5


def test_capture_trains_the_first_batch_exactly_once(lib):
    """ADVICE r1: warm-up + capture used to run 3 real optimizer steps (+ the replay) on the batch that triggers a
    capture.  Now the capture runs on a snapshot: after the first call the parameters, Adam state, BatchNorm running
    statistics and counters are those of ONE eager step."""
    from myria3d_b200.graphed import GraphedTrainStep
    from myria3d_b200.optim import FlatAdam
    from myria3d_b200.parallel import FlatGradAllReducer

    torch.manual_seed(7)
    m = _model(3)
    m.model.mlp_classif.dropout = [0.0, 0.0]  # the two paths would consume the dropout Philox stream differently
    m.model.decimation_rng = "fused"
    ref = copy.deepcopy(m)
    b = _batch([800, 300], 11)

    red = FlatGradAllReducer(m)
    opt = FlatAdam(m, lr=2e-3, reducer=red)
    step = GraphedTrainStep(m, opt, red)
    loss_g = float(step(b.pin_memory()))

    red_r = FlatGradAllReducer(ref)
    opt_r = FlatAdam(ref, lr=2e-3, reducer=red_r)
    red_r.zero_grad()
    out = ref.training_step(b.to(DEV), 0)
    out["loss"].backward()
    opt_r.step()

    assert abs(float(out["loss"]) - loss_g) < 1e-5
    assert int(opt.step_count) == 1 == int(opt_r.step_count)
    for (n1, p1), (_, p2) in zip(m.named_parameters(), ref.named_parameters()):
        if n1.endswith("bias") and "norms" not in n1:
            # a Linear bias in front of a train-mode BatchNorm has a mathematically zero gradient: Adam turns its fp32
            # noise into +-lr steps in either implementation.  ONE step of at most lr each: |difference| <= 2 lr
            assert float((p1 - p2).abs().max()) <= 2.01 * 2e-3, n1
            continue
        # first Adam step = lr * g / (|g| + eps): +-lr wherever |g| >> eps, noise-sensitive only for ~1e-8 gradients.
        # A second training pass on this batch would move every weight by another ~lr = 2e-3
        # (an element whose gradient is fp32 noise around zero may step the other way in the two runs: <= 2 lr apart)
        d = (p1 - p2).abs().flatten()
        assert float(d.max()) <= 2.01 * 2e-3 and float(d.float().quantile(0.99)) <= 5e-5, (n1, float(d.max()), float(d.median()))
    for (n1, b1), (_, b2) in zip(m.named_buffers(), ref.named_buffers()):
        assert torch.allclose(b1.float(), b2.float(), atol=1e-6, rtol=1e-5), n1  # num_batches_tracked == 1, running stats


def test_graph_cache_is_bounded_and_keyed_on_the_host_layout(lib):
    """LRU of ``max_graphs`` layouts; one-off layouts run eagerly until seen ``capture_after`` times; the layout key is
    the HOST ptr (two device ``ptr`` tensors at a recycled address with different contents must not share a graph)."""
    from myria3d_b200.graphed import GraphedTrainStep

    m = _model(4)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3, capturable=True)
    step = GraphedTrainStep(m, opt, max_graphs=2, capture_after=1)
    b1, b2, b3 = _batch([400, 200], 1), _batch([300, 300], 2), _batch([200, 400], 3)
    assert torch.isfinite(step(b1)) and len(step._captured) == 0      # first sight: eager
    assert torch.isfinite(step.last_outputs(b1)["logits"]).all()
    step(b1)
    assert list(step._captured) == [tuple(b1.ptr.tolist())]             # second sight: captured
    step(b2), step(b2), step(b3), step(b3)
    assert list(step._captured) == [tuple(b2.ptr.tolist()), tuple(b3.ptr.tolist())]  # b1 evicted
    # same total size, different boundaries, device-only ptr: keyed on the contents, not on the storage address
    d2, d3 = b2.to(DEV), b3.to(DEV)
    assert step._layout_key(d2) != step._layout_key(d3)


def test_flat_adam_checkpoint_and_scheduler(lib):
    """ADVICE r1: FlatAdam.state_dict() carries the moments and the step; the learning rate is a device scalar, so a
    scheduler acts on a captured graph without re-capturing."""
    from myria3d_b200.optim import FlatAdam

    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(9, 17), torch.nn.Tanh(), torch.nn.Linear(17, 3)).to(DEV)
    opt = FlatAdam(net, lr=1e-2)
    x = torch.randn(32, 9, device=DEV)
    for _ in range(3):
        opt.zero_grad()
        net(x).square().mean().backward()
        opt.step()
    sd = copy.deepcopy(opt.state_dict())
    assert int(sd["flat_adam"]["step"]) == 3 and float(sd["flat_adam"]["exp_avg"].abs().sum()) > 0
    net2 = copy.deepcopy(net)
    opt2 = FlatAdam(net2, lr=1e-2)
    opt2.load_state_dict(sd)
    for o, n_ in ((opt, net), (opt2, net2)):
        o.zero_grad()
        n_(x).square().mean().backward()
        o.step()
    for pa, pb in zip(net.parameters(), net2.parameters()):
        assert torch.equal(pa, pb)  # resumed run == uninterrupted run, bit for bit
    # scheduler through the device scalar, under a captured graph
    sched = torch.optim.lr_scheduler.StepLR(opt, step_size=1, gamma=0.0)  # lr -> 0 after one scheduler step
    g = torch.cuda.CUDAGraph()
    opt.zero_grad()
    net(x).square().mean().backward()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        opt.step()
    torch.cuda.current_stream().wait_stream(side)
    with torch.cuda.graph(g):
        opt.step()
    sched.step()
    opt.sync_lr()
    before = [p.detach().clone() for p in net.parameters()]
    g.replay()
    torch.cuda.synchronize()
    for p, q in zip(net.parameters(), before):
        assert torch.equal(p, q), "the captured update ignored the scheduler's lr = 0"
    # moving the module after the optimizer was built is detected
    net.float()  # no-op cast keeps the views
    assert opt.check_param_views()
    for p in net.parameters():
        p.data = p.data.clone()
    with pytest.raises(RuntimeError, match="flat parameter buffer"):
        opt.step()


def test_autograd_path_is_used_without_a_flat_reducer(lib):
    """ADVICE r1 (high): direct accumulation into ``p.grad`` is opt-in (FlatGradAllReducer's buffer only).  With plain
    ``.grad`` tensors -- torch DDP, gradient accumulation, ``zero_grad(set_to_none=False)`` -- every parameter
    gradient goes through its AccumulateGrad node, so DDP's reducer hooks fire; checked with a 1-rank DDP wrapper and
    ``accumulate_grad_batches = 2`` (configs/experiment/RandLaNet_base_run_FR-MultiGPU.yaml:9-13 uses 3)."""
    import os
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel as DDP

    m = _model(5)
    m.model.mlp_classif.dropout = [0.0, 0.0]
    ref = copy.deepcopy(m)
    b1, b2 = _batch([500, 200], 21).to(DEV), _batch([300, 300], 22).to(DEV)
    fired = []
    w = m.model.block2.lfa1.mlp_attention.lins[0].weight  # its gradient comes out of the fused LFA backward
    acc = w.expand_as(w).grad_fn.next_functions[0][0]
    acc.register_hook(lambda *a: fired.append(1))

    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29533")
    dist.init_process_group("nccl", rank=0, world_size=1)
    try:
        ddp = DDP(m, device_ids=[0])
        for t in (m, ref):
            t.model.injected_decimation_idx = None
        torch.manual_seed(1)
        with ddp.no_sync():
            ddp.module.training_step(b1, 0)["loss"].backward()
        n_after_first = len(fired)
        out = ddp(b2)  # DDP's forward arms the reducer; Model.forward returns (targets, logits)
        torch.nn.functional.cross_entropy(out[1], out[0], ignore_index=65).backward()
        assert n_after_first == 1 and len(fired) == 2, "AccumulateGrad did not run on the second micro-batch"
        g_ddp = {n: p.grad.clone() for n, p in m.named_parameters()}
    finally:
        dist.destroy_process_group()
    # the same two micro-batches without DDP (same seed -> the same per-cloud randperm subsets): identical accumulation
    ref.zero_grad()
    torch.manual_seed(1)
    ref.training_step(b1, 0)["loss"].backward()
    t, lg = ref(b2)
    torch.nn.functional.cross_entropy(lg, t, ignore_index=65).backward()
    params = dict(ref.named_parameters())
    for n, p in params.items():
        scale = float(p.grad.abs().max()) + 1e-12
        if ".lins." in n and n.endswith(".bias") and n.replace("lins.", "norms.").replace(".bias", ".module.weight") in params:
            # a Linear bias in front of train-mode BatchNorm has an exactly zero gradient: both sides are fp32 round-off
            # (~1e-6, the size of the absolute floor) of sums over the rows that make the Linear's weight gradient
            scale = float(params[n[:-len("bias")] + "weight"].grad.abs().max())
        assert float((g_ddp[n] - p.grad).abs().max()) <= 1e-4 * scale + 1e-6, n  # (+ fp32 noise of zero gradients)


def test_prefetch_feeds_the_next_replay(lib):
    """GraphedTrainStep.prefetch: the next (pinned) host batch is copied on a side stream while a step runs; the step
    called with that batch object then trains on exactly its data (static inputs == the batch), an unrelated batch object
    of the same layout falls back to the direct copy, and the loss of a prefetched step equals the eager loss."""
    from myria3d_b200.graphed import GraphedTrainStep
    from myria3d_b200.parallel import FlatGradAllReducer

    m = _model(5)
    m.model.mlp_classif.dropout = [0.0, 0.0]
    opt = torch.optim.Adam(m.parameters(), lr=1e-3, capturable=True)
    step = GraphedTrainStep(m, opt, FlatGradAllReducer(m))
    b1, b2, b3 = (_batch([700, 500], s).pin_memory() for s in (11, 12, 13))
    assert step.prefetch(b1) is False  # nothing captured yet: a no-op
    step(b1)
    key = tuple(b1.ptr.tolist())
    cap = step._captured[key]
    assert step.prefetch(b2) is True
    snap = copy.deepcopy(m)
    loss2 = float(step(b2))  # consumes the staged copy
    torch.cuda.synchronize()
    for k in ("x", "pos", "y", "batch"):
        assert torch.equal(cap.static[k].cpu(), getattr(b2, k)), k
    snap.model.injected_decimation_idx = [t.clone() for t in cap.idx_static]
    out = snap.training_step(b2.to(DEV), 0)
    assert abs(float(out["loss"].detach()) - loss2) < 1e-4
    # prefetch b3, but call with b1: the staged copy must not be used
    step.prefetch(b3)
    step(b1)
    torch.cuda.synchronize()
    assert torch.equal(cap.static["pos"].cpu(), b1.pos)
    step(b3)  # now the staged copy of b3 is consumed
    torch.cuda.synchronize()
    assert torch.equal(cap.static["x"].cpu(), b3.x)
    # a running loop: prefetch behind every replay
    step.prefetch(b1)
    for cur, nxt in ((b1, b2), (b2, b3), (b3, b1)):
        loss = step(cur)
        step.prefetch(nxt)
        assert torch.isfinite(loss).item()
        assert torch.equal(cap.static["y"].cpu(), cur.y)


def test_scratch_arena_is_clean_after_a_graph_replay(lib):
    """The replay of a captured step leaves its reduction sums in the arena slices it was captured with -- possibly beyond
    the extent of the pass that ran last from Python (another, smaller layout).  Consumers that never pass through
    ``B200RandLANet.forward`` (a bare LocalFeatureAggregation, ``ops.cross_entropy``) must still be handed zeros: the
    arena is cleared up to its high-water mark, and a reported replay makes the next eager ``take()`` clear it first
    (found by running test_lfa_module_parity after the graph tests: fp64 sums read back as fp32 gave 1e27 gradients)."""
    from myria3d_b200 import ops

    dev = torch.device(DEV)
    ops._zeros_scratch(8, torch.float32, dev)  # make sure the arena exists
    arena = ops._ARENAS[ops._arena_key(dev)]
    ops.reset_scratch(dev)
    big = ops._zeros_scratch(5000, torch.float64, dev)  # the extent of a large captured layout ...
    ops.reset_scratch(dev)
    small = ops._zeros_scratch(16, torch.float32, dev)  # ... then a small pass: Python's offset is far below it
    assert arena.off < arena.hw
    big.fill_(70.245)  # what a replay of the large graph leaves behind
    ops.mark_scratch_dirty(dev)
    t = ops._zeros_scratch(64, torch.float32, dev)
    u = ops._zeros_scratch(3000, torch.float64, dev)
    torch.cuda.synchronize()
    assert float(t.abs().max()) == 0.0 and float(u.abs().max()) == 0.0
    assert not arena.dirty
    # reset() always clears up to the high-water mark
    u.fill_(1.0)
    ops.reset_scratch(dev)
    v = ops._zeros_scratch(5000, torch.float64, dev)
    assert float(v.abs().max()) == 0.0
    del small
