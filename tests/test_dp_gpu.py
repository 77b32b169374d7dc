"""Fused data-parallel optimiser step (ppb_dp_adam_step: reduce-scatter + Adam + all-gather over NVLink peer
memory) against the unfused path it replaces (gradient all-reduce, pyprob/nn/inference_network.py:296-333, then
optimizer.step(), :496 — here ppb_adam_step_dev, itself checked against torch.optim.Adam in test_network_gpu)."""
import os
import socket

import pytest
import torch

pytestmark = pytest.mark.gpu

N = 100003          # not a multiple of 4 * world: exercises the ragged slice tails
STEPS = 3


def _hyper(world, dev):
    return torch.tensor([1e-3, 0.9, 0.999, 1e-8, 1e-5, 1.0 / world], dtype=torch.float32, device=dev)


def _reference_steps(p, grads, world, dev):
    """grads: list over steps of the summed gradient.  Returns (p, m, v) after the unfused device Adam."""
    from pyprob_b200._lib import call, ptr
    p = p.clone()
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    state = torch.zeros(4, dtype=torch.int32, device=dev)
    hyper = _hyper(world, dev)
    for g in grads:
        call('ppb_adam_step_dev', ptr(p), ptr(g), ptr(m), ptr(v), p.numel(), ptr(hyper), ptr(state),
             torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return p, m, v


def test_peer_adam_single_rank_is_plain_adam(cuda):
    from pyprob_b200 import parallel
    dev = cuda
    gen = torch.Generator(device='cpu').manual_seed(5)
    p0 = torch.randn(N, generator=gen).to(dev)
    grads = [torch.randn(N, generator=gen).to(dev) for _ in range(STEPS)]
    want_p, want_m, want_v = _reference_steps(p0, grads, 1, dev)
    peer = parallel.PeerAdam(N, dev)
    peer.params.copy_(p0)
    m, v = torch.zeros(N, device=dev), torch.zeros(N, device=dev)
    state = torch.zeros(4, dtype=torch.int32, device=dev)
    hyper = _hyper(1, dev)
    for i, g in enumerate(grads):
        peer.grad[:N].copy_(g)
        peer.grad[N] = 2.5 + i
        peer.step(m, v, hyper, state, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert float(peer.grad[N]) == 2.5 + i
    assert not peer.timed_out()
    assert int(state.view(torch.int64)[0]) == STEPS
    assert torch.equal(peer.params, want_p)
    assert torch.equal(m, want_m) and torch.equal(v, want_v)
    peer.close()


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, use_graph):
    import torch.distributed as dist
    from pyprob_b200 import parallel
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device('cuda', rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=dev)
    gen = torch.Generator(device='cpu').manual_seed(11)
    p0 = torch.randn(N, generator=gen).to(dev)                               # same start on every rank
    all_grads = [[torch.randn(N, generator=gen) for _ in range(world)] for _ in range(STEPS)]
    # unfused path: NCCL all-reduce of the gradient, then Adam on the full arena
    summed = []
    for step in all_grads:
        g = step[rank].to(dev)
        dist.all_reduce(g)
        summed.append(g)
    want_p, want_m, want_v = _reference_steps(p0, summed, world, dev)

    peer = parallel.PeerAdam(N, dev)
    peer.params.copy_(p0)
    m, v = torch.zeros(N, device=dev), torch.zeros(N, device=dev)
    state = torch.zeros(4, dtype=torch.int32, device=dev)
    hyper = _hyper(world, dev)
    stage = torch.zeros(N + 1, device=dev)

    def one_step():
        peer.grad[:N + 1].copy_(stage)
        peer.step(m, v, hyper, state, torch.cuda.current_stream().cuda_stream)

    graph = None
    if use_graph:      # the step must survive capture + replay (the barrier epoch lives in device memory)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            stage[:N].copy_(all_grads[0][rank].to(dev))
            stage[N] = float(rank + 1)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side):
                one_step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        # capture does not execute: state is untouched
    for i, step in enumerate(all_grads):
        stage[:N].copy_(step[rank].to(dev))
        stage[N] = float(rank + 1) * (i + 1)
        if graph is not None:
            graph.replay()
        else:
            one_step()
        torch.cuda.synchronize()
        want_loss = sum(float(r + 1) * (i + 1) for r in range(world))
        assert float(peer.grad[N]) == want_loss, (float(peer.grad[N]), want_loss)
    dist.barrier()
    assert not peer.timed_out()
    lo = ((N + world * 4 - 1) // (world * 4)) * 4 * rank
    hi = min(N, lo + ((N + world * 4 - 1) // (world * 4)) * 4)
    if world == 2:      # a two-term sum has one order: bit-exact against NCCL + Adam
        assert torch.equal(peer.params, want_p)
        assert torch.equal(m[lo:hi], want_m[lo:hi]) and torch.equal(v[lo:hi], want_v[lo:hi])
    else:
        torch.testing.assert_close(peer.params, want_p, rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(m[lo:hi], want_m[lo:hi], rtol=1e-5, atol=1e-7)
    # optimiser state outside the owned slice is never touched
    if lo > 0:
        assert float(m[:lo].abs().max()) == 0.0
    # replicas are bit-identical
    mine = peer.params.clone()
    ref = mine.clone()
    dist.broadcast(ref, 0)
    assert torch.equal(mine, ref)
    graph = None
    peer.close()
    dist.barrier()
    torch.cuda.synchronize()
    os._exit(0)


@pytest.mark.parametrize('use_graph', [False, True])
def test_peer_adam_matches_allreduce_adam(use_graph):
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip('needs at least two GPUs on one NVLink node')
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, use_graph)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(180)
    for p in procs:
        if p.is_alive():
            p.kill()
            pytest.fail('worker did not finish')
        assert p.exitcode == 0


def _checkpoint_worker(rank, world, port, path):
    """Data-parallel training keeps the Adam moments of an element on its owning rank only; a checkpoint must hold all of
    them (ADVICE round 1): _full_optimizer_moments gathers the owned slices, save -> load restores the full arrays."""
    import torch.distributed as dist
    from pyprob_b200 import synthetic
    from pyprob_b200.network import InferenceNetworkLSTM
    from pyprob_b200.util import Optimizer
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device('cuda', rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=dev)
    net = synthetic.gum_network(lstm_dim=32, seed=0)
    net._optimizer_type, net._learning_rate_init, net._weight_decay = Optimizer.ADAM, 1e-3, 1e-5
    net._create_optimizer()
    net._learning_rate = 1e-3
    dist.broadcast(net._arena.data, 0)
    p0 = net._arena.data.clone()
    net._enable_peer_optimizer()
    n = net._arena.numel()
    gen = torch.Generator(device='cpu').manual_seed(3)
    all_grads = [[torch.randn(n, generator=gen) for _ in range(world)] for _ in range(STEPS)]
    summed = []
    for step in all_grads:
        g = step[rank].to(dev)
        dist.all_reduce(g)
        summed.append(g)
    want_p, want_m, want_v = _reference_steps(p0, summed, world, dev)
    for step in all_grads:
        net._arena.grad = step[rank].to(dev)
        net._peer_optimizer_step(torch.tensor(1.0, device=dev), world)
    m, v = net._full_optimizer_moments()
    tol = dict(rtol=0, atol=0) if world == 2 else dict(rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(m, want_m, **tol)
    torch.testing.assert_close(v, want_v, **tol)
    if rank == 0:
        net._save(path, (m, v))
        loaded = InferenceNetworkLSTM._load(path)
        assert torch.equal(loaded._exp_avg, m) and torch.equal(loaded._exp_avg_sq, v)
        assert loaded._optimizer_step == STEPS
        torch.testing.assert_close(loaded._arena.data, want_p, rtol=1e-5, atol=1e-6)
    dist.barrier()
    torch.cuda.synchronize()
    os._exit(0)


def test_checkpoint_holds_the_moments_of_every_rank(tmp_path):
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip('needs at least two GPUs on one NVLink node')
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    port = _free_port()
    procs = [ctx.Process(target=_checkpoint_worker, args=(r, world, port, str(tmp_path / 'dp.network'))) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(180)
    for p in procs:
        if p.is_alive():
            p.kill()
            pytest.fail('worker did not finish')
        assert p.exitcode == 0
