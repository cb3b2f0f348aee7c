"""Data-parallel IKFlow training (cppflow_b200/ikflow_training.py: tree_levels, local_schedule, IkflowTrainer with
micro_batches and process_group; csrc/k_flow_train.cu: cppflow_flow_train_batch_rows, cppflow_flow_grad_tree_reduce,
cppflow_flow_train_apply).

CPU: the statement of the tree order against a float64 sum and the subtree alignment of every (W, M) with S <= 16,
and the rejected configurations.  One GPU: sharded draws, the reduction kernel against tree_sum, the M = 1 sharded
step against the one-call step, the micro-batched gradient against fp64 autograd over the global batch, skipped
steps, save / load and no host synchronisation.  Several GPUs (skipped when fewer exist): the ranks' weights against
each other and against one GPU at the same shard count, and a resume on one GPU from a multi-GPU checkpoint."""
import datetime

import numpy as np
import pytest
import torch

from oracle import ikflow_train as OT

DEV = "cuda:0"
POW2 = [1, 2, 4, 8, 16]


def _params():
    from cppflow_b200.ikflow import IkflowModelParameters

    return IkflowModelParameters(nb_nodes=2, dim_latent_space=9, coeff_fn_config=2, coeff_fn_internal_size=128,
                                 softflow_enabled=True)


def _trainer(device=DEV, **kw):
    from cppflow_b200.ikflow_training import IkflowTrainer
    from cppflow_b200.robot import get_robot

    kw.setdefault("batch_size", 256)
    return IkflowTrainer(get_robot("panda"), _params(), seed=kw.pop("seed", 3), n_data=20000, device=device, **kw)


# ----------------------------------------------------------------------------------------------------------- CPU


def test_local_schedule_is_a_binary_counter():
    from cppflow_b200.ikflow_training import local_schedule

    assert local_schedule(1) == [("grad", 0, 0)]
    assert local_schedule(4) == [("grad", 0, 0), ("grad", 1, 1), ("add", 0), ("grad", 2, 1), ("grad", 3, 2),
                                 ("add", 1), ("add", 0)]
    for M in POW2:
        ops = local_schedule(M)
        assert max(op[2] for op in ops if op[0] == "grad") + 1 == M.bit_length()  # log2(M) + 1 buffers
        assert sum(op[0] == "add" for op in ops) == M - 1


@pytest.mark.parametrize("W,M", [(W, M) for W in POW2 for M in POW2 if W * M <= 16])
def test_tree_order_statement(W, M):
    """Which shard pairs are summed, and when: replaying local_schedule on shard ranges gives the pairs of
    tree_levels(M) as soon as both halves exist; a rank's partial is an aligned subtree of tree_levels(S), whose top
    log2(W) levels combine whole ranks in rank order; the float32 result is T(g) bit for bit and near the float64 sum."""
    from cppflow_b200.ikflow_training import local_schedule, tree_levels, tree_sum

    S = W * M
    levels = tree_levels(S)
    nodes = {(a, b) for lv in levels for pair in lv for (a, b) in pair} | {(0, S)}
    # the local schedule on ranges
    stack, pairs = [], []
    for op in local_schedule(M):
        if op[0] == "grad":
            assert op[2] == len(stack)
            stack.append((op[1], op[1] + 1))
        else:
            left, right = stack[op[1]], stack[op[1] + 1]
            assert op[1] == len(stack) - 2 and left[1] == right[0] and left[1] - left[0] == right[1] - right[0]
            assert pairs == [] or right[1] >= pairs[-1][1][1]  # merged as soon as the right half is complete
            pairs.append((left, right))
            stack[op[1]:] = [(left[0], right[1])]
    assert stack == [(0, M)]
    assert sorted(pairs) == sorted(p for lv in tree_levels(M) for p in lv)
    for r in range(W):  # subtree alignment
        assert M == 1 or (r * M, (r + 1) * M) in nodes
    for lv in levels[len(tree_levels(M)):]:
        for (a, b), (c, d) in lv:
            assert a % M == 0 and b % M == 0 and c % M == 0 and d % M == 0
    # values: per rank through the schedule, then the top of the tree over ranks, in float32
    rng = np.random.default_rng(S * 31 + W)
    g = (rng.standard_normal((S, 257)) * np.exp(rng.uniform(-8, 8, (S, 1)))).astype(np.float32)
    partials = []
    for r in range(W):
        buf = [None] * M.bit_length()
        for op in local_schedule(M):
            if op[0] == "grad":
                buf[op[2]] = g[r * M + op[1]].copy()
            else:
                buf[op[1]] = (buf[op[1]] + buf[op[1] + 1]).astype(np.float32)
        partials.append(buf[0])
    got = tree_sum(partials) * np.float32(1.0 / S)
    assert got.dtype == np.float32
    assert np.array_equal(got, tree_sum(list(g)) * np.float32(1.0 / S))
    ref = g.astype(np.float64).sum(0) / S
    scale = np.abs(g.astype(np.float64)).sum(0) / S
    assert np.all(np.abs(got - ref) <= 4 * np.log2(2 * S) * np.finfo(np.float32).eps * scale)


def test_rejected_configurations(tmp_path, monkeypatch):
    from cppflow_b200 import _lib
    from cppflow_b200.ikflow_training import IkflowTrainer, local_schedule, tree_levels
    from cppflow_b200.robot import get_robot

    rob = get_robot("panda")
    for m in (0, 3, 6):
        with pytest.raises(ValueError, match="power of two"):
            IkflowTrainer(rob, _params(), batch_size=256, micro_batches=m, device="cpu")
        with pytest.raises(ValueError, match="power of two"):
            local_schedule(m)
    with pytest.raises(ValueError, match="power of two"):
        tree_levels(12)
    with pytest.raises(ValueError, match="multiple of 128"):
        IkflowTrainer(rob, _params(), batch_size=200, micro_batches=2, device="cpu")
    import torch.distributed as dist

    monkeypatch.setattr(dist, "get_world_size", lambda group=None: 3)
    monkeypatch.setattr(dist, "get_rank", lambda group=None: 0)
    with pytest.raises(ValueError, match="3 ranks"):
        IkflowTrainer(rob, _params(), batch_size=256, process_group=object(), device="cpu")
    monkeypatch.undo()
    # a checkpoint of S = 4 shards of 256 rows: another S or B is another run
    path = str(tmp_path / "ck.pt")
    torch.save({"shards": 4, "batch_size": 256, "hyper": {}}, path)
    for kw, msg in ((dict(micro_batches=2), "4 shards"), (dict(micro_batches=8), "4 shards"),
                    (dict(batch_size=512), "256 rows per shard")):
        with pytest.raises(ValueError, match=msg):
            IkflowTrainer.load(path, device="cpu", **kw)
    # the library's reduction: n a power of two <= 32, aligned multiples of 4
    lib = _lib.load()
    for n, length, stride, msg in ((3, 64, 64, b"power of two"), (64, 64, 64, b"power of two"), (2, 62, 64, b"multiples"),
                                   (2, 64, 32, b"stride >= len")):
        assert lib.cppflow_flow_grad_tree_reduce(256, n, length, stride, 1.0, 256, None) == -1
        assert msg in lib.cppflow_last_error()
    assert lib.cppflow_flow_grad_tree_reduce(260, 2, 64, 64, 1.0, 256, None) == -1
    assert b"aligned" in lib.cppflow_last_error()


# ----------------------------------------------------------------------------------------------------------- GPU


@pytest.mark.gpu
def test_sharded_draw_is_the_rows_of_one_draw():
    from cppflow_b200 import ops

    tr = _trainer(batch_size=1024)
    tr.counters[2] = 5  # the key's step
    idx, noise = torch.empty(1024, dtype=torch.int64, device=DEV), torch.empty((1024, 11), device=DEV)
    tr.draw_batch(idx, noise)
    x, cond = tr.x.clone(), tr.cond.clone()
    for first, n in ((0, 128), (128, 256), (384, 512), (896, 128)):
        xs, cs = torch.empty((n, 9), device=DEV), torch.empty((n, 8), device=DEV)
        i2, n2 = torch.empty(n, dtype=torch.int64, device=DEV), torch.empty((n, 11), device=DEV)
        ops.flow_train_batch(tr.desc, tr.data_q, tr.data_poses, tr.seed, tr.softflow_noise_scale, xs, cs, i2, n2,
                             first_row=first)
        sl = slice(first, first + n)
        assert torch.equal(xs, x[sl]) and torch.equal(cs, cond[sl]) and torch.equal(i2, idx[sl])
        assert torch.equal(n2, noise[sl])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 4, 8, 16, 32])
def test_tree_reduce_kernel_is_tree_sum(n):
    from cppflow_b200 import ops
    from cppflow_b200.ikflow_training import tree_sum

    g = torch.Generator(device=DEV).manual_seed(n)
    length, stride = 64 * 1001, 64 * 1003
    buf = torch.randn((n, stride), generator=g, device=DEV) * torch.exp(8 * torch.randn((n, 1), generator=g, device=DEV))
    buf[0, 7] = float("inf")
    buf[-1, 9] = float("nan")
    slices = buf[:, :length]
    scale = 1.0 / 3.0
    want = tree_sum([slices[i] for i in range(n)]) * torch.tensor(scale, dtype=torch.float32)
    out = ops.flow_grad_tree_reduce(slices, torch.empty(length, device=DEV), scale)
    assert torch.equal(out.isnan(), want.isnan()) and torch.equal(out.nan_to_num(), want.nan_to_num())
    ops.flow_grad_tree_reduce(slices, buf[0, :length], scale)  # in place on slice 0
    assert torch.equal(buf[0, :length].nan_to_num(), want.nan_to_num())


def _state(tr):
    return [tr.params_flat, tr.adam_m, tr.adam_v, tr.counters, tr.loss_history(),
            *(t for t in tr.bf16.values() if t is not None)]


def _assert_same(a, b):
    for x, y in zip(_state(a), _state(b), strict=True):
        assert torch.equal(x, y)


def _sharded_m1(**kw):
    """The data-parallel step at S = 1 (one NO_UPDATE step, the tree, apply) on one GPU"""
    tr = _trainer(**kw)
    tr._sharded = True
    tr._init_shards()
    return tr


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
def test_one_shard_equals_the_one_call_step(graph):
    a, b = _trainer(use_graph=graph), _sharded_m1(use_graph=graph)
    for tr in (a, b):
        tr.step(5)
    _assert_same(a, b)
    assert a.counters.tolist() == [5, 0, 5]


def _global_batch(tr):
    """The S B rows of the current step drawn at once"""
    from cppflow_b200 import ops

    n = tr.shards * tr.batch_size
    x, cond = torch.empty((n, 9), device=DEV), torch.empty((n, 8), device=DEV)
    ops.flow_train_batch(tr.desc, tr.data_q, tr.data_poses, tr.seed, tr.softflow_noise_scale, x, cond)
    return x, cond


@pytest.mark.gpu
@pytest.mark.parametrize("M", [2, 4])
def test_micro_batched_gradient_against_fp64_autograd(M):
    """G of S = M shards of 512 rows against fp64 autograd over the S x 512 rows, with the bound of
    tests/test_ikflow_training.py::test_gradient_parity_with_autograd (twice torch's bf16 autocast error)"""
    from cppflow_b200.ikflow_training import split_tables, unpack
    from oracle import ikflow as OF

    tr = _trainer(batch_size=512, micro_batches=M, seed=5)
    x, cond = _global_batch(tr)
    tr._exchange(tr._local_partial())
    P = tr._P
    G, loss = tr._G[:P].clone(), tr._G[P].item()
    one_loss, one = tr.loss_and_grad(x, cond)
    shard_losses = [tr.loss_and_grad(x[j * 512:(j + 1) * 512], cond[j * 512:(j + 1) * 512])[0].item() for j in range(M)]

    def glow(dtype):
        p = tr.params
        net = OF.Glow(tr.robot.actuated_joints_limits, 9, p.nb_nodes, p.coeff_fn_internal_size, p.coeff_fn_config,
                      p.rnvp_clamp, p.softflow_enabled)
        net.load_state_dict(tr.state_dict())
        return net.to(DEV, dtype)

    def grads(net, xx, cc, bf16, autocast):
        net.zero_grad()
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
            loss_ = OT.nll(*OT.forward_with_logdet(net, xx, cc, bf16=bf16))
        loss_.backward()
        return loss_.item(), {k: p.grad.detach().double().cpu() for k, p in net.named_parameters()}

    l64, ref = grads(glow(torch.float64), x.double(), cond.double(), True, False)
    _, torch_bf16 = grads(glow(torch.float32), x, cond, False, True)
    got, got_one = (unpack(split_tables(v, tr.params), tr.params) for v in (G, one))
    for k, r in ref.items():
        rel = ((got[k].double() - r).norm() / r.norm()).item()
        rel_one = ((got_one[k].double() - r).norm() / r.norm()).item()
        rel_t = ((torch_bf16[k] - r).norm() / r.norm()).item()
        cos = torch.nn.functional.cosine_similarity(got[k].double().reshape(1, -1), r.reshape(1, -1)).item()
        print(f"M={M} {k}: rel L2 {rel:.2e} (one call {rel_one:.2e}, torch bf16 autocast {rel_t:.2e}), cos {cos:.6f}")
        assert rel <= 2 * rel_t, k
        assert cos >= 0.999, k
    # the loss is the global mean: of the shard losses in fp64, and of the fp64 model's NLL
    want = float(np.mean(np.array(shard_losses, dtype=np.float64)))
    print(f"M={M}: loss {loss:.7f}, mean of shard losses {want:.7f}, one call {one_loss.item():.7f}, fp64 {l64:.7f}")
    assert abs(loss - want) <= 1e-6 * max(1.0, abs(want))
    assert abs(loss - l64) < 1e-3 * max(1.0, abs(l64))


@pytest.mark.gpu
def test_a_nan_in_one_shard_skips_the_step():
    tr = _trainer(micro_batches=4)
    tr.step(2)
    draw = tr._draw_shard

    def poisoned(j):
        draw(j)
        if j == 2:
            tr.cond[17, 4] = float("nan")

    tr._draw_shard = poisoned
    before = [t.clone() for t in _state(tr)[:3]] + [tr.bf16["w_in"].clone()]
    tr.step(1)
    assert tr.counters.tolist() == [2, 1, 3] and tr.steps_skipped.item() == 1
    for x, y in zip(before, _state(tr)[:3] + [tr.bf16["w_in"]]):
        assert torch.equal(x, y)
    assert torch.isnan(tr.loss_history()[-1])


@pytest.mark.gpu
def test_micro_batched_save_load_graph_and_no_sync(tmp_path):
    from cppflow_b200.ikflow_training import IkflowTrainer

    a, g = _trainer(micro_batches=4), _trainer(micro_batches=4, use_graph=True)
    assert a.hyper["lr_decay_steps"] == round(2_500_000 / (4 * 256))
    for tr in (a, g):
        tr.step(4)
    _assert_same(a, g)
    path = str(tmp_path / "ck.pt")
    a.save(path)
    assert torch.load(path, weights_only=False)["shards"] == 4
    a.step(3)
    r = IkflowTrainer.load(path, device=DEV)
    assert r.micro_batches == 4 and r.hyper == a.hyper
    r.step(3)
    _assert_same(a, r)
    assert a.loss_history().numel() == 7 and torch.isfinite(a.loss_history()).all()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        a.step(2)
        g.step(2)
    finally:
        torch.cuda.set_sync_debug_mode(0)


# ---------------------------------------------------------------------------------------------------- several GPUs


def _dp_worker(rank, W, M, K, save_at, use_graph, out):
    """One rank of a W-GPU run: K steps at M micro-batches per rank, rank 0 writing a checkpoint after save_at steps;
    every rank writes its final state."""
    import torch.distributed as dist

    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"file://{out}/rendezvous", rank=rank, world_size=W,
                            timeout=datetime.timedelta(minutes=3), device_id=torch.device("cuda", rank))
    try:
        tr = _trainer(device=f"cuda:{rank}", micro_batches=M, process_group=dist.group.WORLD, use_graph=use_graph)
        if save_at:
            tr.step(save_at)
            tr.save(f"{out}/ck.pt")
        tr.step(K - save_at)
        torch.cuda.synchronize()
        torch.save([t.cpu() for t in _state(tr)], f"{out}/rank{rank}.pt")
    finally:
        dist.destroy_process_group()


def _spawn(tmp_path, W, M, K, save_at=0, use_graph=False):
    import torch.multiprocessing as mp

    if torch.cuda.device_count() < W:
        pytest.skip(f"needs {W} GPUs, {torch.cuda.device_count()} present")
    mp.spawn(_dp_worker, args=(W, M, K, save_at, use_graph, str(tmp_path)), nprocs=W, join=True)
    return [torch.load(f"{tmp_path}/rank{r}.pt") for r in range(W)]


@pytest.mark.gpu
@pytest.mark.parametrize("W", [2, 4, 8])
@pytest.mark.parametrize("M", [1, 2])
def test_ranks_match_one_gpu_at_the_same_shard_count(tmp_path, W, M):
    K = 4
    ranks = _spawn(tmp_path, W, M, K, use_graph=M == 1)
    one = _trainer(micro_batches=W * M)
    one.step(K)
    want = [t.cpu() for t in _state(one)]
    for r, got in enumerate(ranks):
        for x, y in zip(got, want, strict=True):
            assert torch.equal(x, y), r


@pytest.mark.gpu
@pytest.mark.parametrize("W", [2, 4, 8])
def test_multi_gpu_checkpoint_resumes_on_one_gpu(tmp_path, W):
    from cppflow_b200.ikflow_training import IkflowTrainer

    k, K = 2, 5
    ranks = _spawn(tmp_path, W, 1, K, save_at=k)
    r = IkflowTrainer.load(f"{tmp_path}/ck.pt", device=DEV)
    assert r.micro_batches == W and r.shards == W
    r.step(K - k)
    for x, y in zip(ranks[0], [t.cpu() for t in _state(r)], strict=True):
        assert torch.equal(x, y)
