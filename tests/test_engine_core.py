"""engine.StudentTrainer, the step core the GCN, GraphSAGE and multi-GPU engines share: the flat-buffer layout of the
parameter tables, graph capture / replay and state_dict round trips on the SAGE engine, and the multi-GPU engines'
refusal of an auxiliary loss."""
import pytest
import torch

import efficient_gnns_b200  # noqa: F401
from efficient_gnns_b200.engine import GCNStudentTrainer
from efficient_gnns_b200.engine_sage import SAGEStudentTrainer
from efficient_gnns_b200.sparse import SparseTensor
from efficient_gnns_b200.synthetic import skewed_edges
from oracle import graph as og

# state-dict key -> (offset into the flat parameter / gradient / Adam buffers, shape).  The multi-GPU engines exchange the
# gradient buffer by position and Adam's state is positional, so these offsets are part of the engines' contract.
GCN_LAYOUT = {
    (128, 256, 256, 40): {
        "convs.0.weight": (0, (128, 256)),
        "convs.0.bias": (32768, (256,)),
        "bns.0.weight": (33024, (256,)),
        "bns.0.bias": (33280, (256,)),
        "convs.1.weight": (33536, (256, 256)),
        "convs.1.bias": (99072, (256,)),
        "bns.1.weight": (99328, (256,)),
        "bns.1.bias": (99584, (256,)),
        "convs.2.weight": (99840, (256, 40)),
        "convs.2.bias": (110080, (40,)),
    },
    (64, 64, 40): {
        "convs.0.weight": (0, (64, 64)),
        "convs.0.bias": (4096, (64,)),
        "bns.0.weight": (4160, (64,)),
        "bns.0.bias": (4224, (64,)),
        "convs.1.weight": (4288, (64, 40)),
        "convs.1.bias": (6848, (40,)),
    },
}
SAGE_LAYOUT = {
    (128, 256, 256, 40): {
        "convs.0.lin_l.weight": (0, (256, 128)),
        "convs.0.lin_l.bias": (32768, (256,)),
        "convs.0.lin_r.weight": (33024, (256, 128)),
        "bns.0.weight": (65792, (256,)),
        "bns.0.bias": (66048, (256,)),
        "convs.1.lin_l.weight": (66304, (256, 256)),
        "convs.1.lin_l.bias": (131840, (256,)),
        "convs.1.lin_r.weight": (132096, (256, 256)),
        "bns.1.weight": (197632, (256,)),
        "bns.1.bias": (197888, (256,)),
        "convs.2.lin_l.weight": (198144, (40, 256)),
        "convs.2.lin_l.bias": (208384, (40,)),
        "convs.2.lin_r.weight": (208424, (40, 256)),
    },
    (64, 64, 40): {
        "convs.0.lin_l.weight": (0, (64, 64)),
        "convs.0.lin_l.bias": (4096, (64,)),
        "convs.0.lin_r.weight": (4160, (64, 64)),
        "bns.0.weight": (8256, (64,)),
        "bns.0.bias": (8320, (64,)),
        "convs.1.lin_l.weight": (8384, (40, 64)),
        "convs.1.lin_l.bias": (10944, (40,)),
        "convs.1.lin_r.weight": (10984, (40, 64)),
    },
}


@pytest.mark.parametrize("dims", [(128, 256, 256, 40), (64, 64, 40)])
@pytest.mark.parametrize("engine,expected", [(GCNStudentTrainer, GCN_LAYOUT), (SAGEStudentTrainer, SAGE_LAYOUT)])
def test_parameter_table_keeps_the_flat_buffer_layout(engine, expected, dims):
    layout = engine.param_layout(list(dims))
    assert {key: (off, shape) for key, (off, shape, _) in layout.items()} == expected[dims]


def graph_and_inputs(n=3000, e=20_000, dims=(32, 64, 64, 8), seed=1):
    ei = skewed_edges(n, e, seed)
    row, col, _ = og.to_sparse_adj_t(ei.numpy(), n)
    r, c = og.to_symmetric(row, col, n)
    adj = SparseTensor(row=torch.from_numpy(r).cuda(), col=torch.from_numpy(c).cuda(), sparse_sizes=(n, n), is_sorted=True)
    g = torch.Generator().manual_seed(seed + 9)
    x = torch.randn(n, dims[0], generator=g).cuda()
    y = torch.randint(0, dims[-1], (n,), generator=g).cuda()
    t = (torch.randn(n, dims[-1], generator=g) * 2).cuda()
    idx = torch.randperm(n, generator=g)[: n // 2].sort().values.cuda()
    return adj, (x, y, idx, t)


@pytest.mark.gpu
def test_sage_capture_with_key_replays_the_eager_steps():
    """The second input-buffer set of the double-buffered end-to-end loop (key=1) drives the SAGE engine too."""
    dims = [32, 64, 64, 8]
    adj, args = graph_and_inputs(dims=dims)
    eager = SAGEStudentTrainer(adj, dims, dropout=0.5, lr=0.01, seed=1)
    want = [eager.train_step(*args).clone() for _ in range(3)]
    tr = SAGEStudentTrainer(adj, dims, dropout=0.5, lr=0.01, seed=1)
    tr.capture(*args, warmup=1, key=1)
    tr.reset_parameters(1)                   # capture() ran warm-up steps
    got = [tr.replay(1).clone() for _ in range(3)]
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(got, want))
    assert torch.equal(tr.params, eager.params)


@pytest.mark.gpu
def test_sage_state_dict_round_trip_restores_running_statistics():
    dims = [32, 64, 64, 8]
    adj, args = graph_and_inputs(dims=dims)
    tr = SAGEStudentTrainer(adj, dims, dropout=0.5, lr=0.01, seed=1)
    for _ in range(3):
        tr.train_step(*args)
    fresh = SAGEStudentTrainer(adj, dims, dropout=0.5, lr=0.01, seed=2)
    fresh.load_state_dict(tr.state_dict())
    for l in range(tr.L - 1):
        assert torch.equal(fresh.running_mean[l], tr.running_mean[l]) and torch.equal(fresh.running_var[l], tr.running_var[l])
    x = args[0]
    assert torch.equal(fresh.forward(x, training=False), tr.forward(x, training=False))


@pytest.mark.gpu
def test_multi_gpu_engines_refuse_an_auxiliary_loss_before_any_launch():
    import os
    import socket
    import torch.distributed as dist
    from efficient_gnns_b200 import lib
    from efficient_gnns_b200.dist import ShardedGCNTrainer
    from efficient_gnns_b200.hybrid import HybridGCNTrainer
    if not dist.is_initialized():
        with socket.socket() as s:
            s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    dims = [32, 64, 64, 8]
    adj, (x, y, idx, t) = graph_and_inputs(dims=dims)
    engines = [HybridGCNTrainer(adj, dims, dropout=0.0, seed=4, exchange="null", _fake=(0, 2)),
               ShardedGCNTrainer(adj, dims, dropout=0.0, seed=4)]
    for tr in engines:
        inputs = tr.shard_inputs(x, y, idx, t)
        torch.cuda.synchronize()
        before = lib.launch_count()
        with pytest.raises(NotImplementedError):
            tr.train_step(*inputs, aux=lambda f: f.square().mean())
        assert lib.launch_count() == before
        assert int(tr.step_count.item()) == 0
