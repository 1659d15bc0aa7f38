"""GossipDataParallel / GossipTrainer on the nvlink KERNEL transport with N virtual ranks inside
ONE process on ONE GPU (``LocalWorld`` loop-back): the same world-simulation oracle as the
multi-process tests (tests/test_multigpu.py), but runnable on a single-GPU box -- SGP, D-PSGD,
Overlap-SGP, the peers_per_itr schedule swap and the graph-captured trainer all exercise the
flag / ack protocol between kernels that are co-resident on the same device."""
import gc

import pytest
import torch

import stochastic_gradient_push_b200 as sgp

import test_distributed_c10d as sim

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _no_device_sync_from_gc():
    """One host thread drives every virtual rank, so a rank's gossip kernel can spin until the host
    launches its in-neighbour's step.  A dropped GossipDataParallel is part of a reference cycle
    (its hooks hold it) and owns symmetric buffers whose release is a cudaFree, which waits for the
    whole device: if the cyclic collector freed one between those two launches, the host would
    wait on a kernel that waits on the host until the heartbeat timeout fired.  So collect while
    nothing spins, and keep the collector off while the virtual ranks run."""
    gc.collect()
    gc.disable()
    try:
        yield
    finally:
        gc.enable()
        gc.collect()


def _world(n, graph_name, ppi, overlap, fused, nesterov):
    from stochastic_gradient_push_b200.optim import FusedGossipSGD
    from stochastic_gradient_push_b200.parallel.distributed import GossipDataParallel
    from stochastic_gradient_push_b200.parallel.symmetric import LocalWorld
    dev = torch.device('cuda', 0)
    lw = LocalWorld(n)
    ranks = []
    for r in range(n):
        graph = getattr(sgp, graph_name)(r, n, peers_per_itr=ppi)
        net = sim._model(r).to(dev)
        model = GossipDataParallel(net, graph=graph, overlap=overlap, rank=r, world_size=n,
                                   heartbeat_timeout=20, symmetric_world=lw.view(r), transport='nvlink',
                                   grid=4, symmetric_name='loopback')
        assert model.transport == 'nvlink'
        if fused:
            opt = FusedGossipSGD(model, lr=sim.LR, momentum=sim.MU, weight_decay=sim.WD, nesterov=nesterov)
        else:
            opt = torch.optim.SGD(model.parameters(), lr=sim.LR, momentum=sim.MU, weight_decay=sim.WD,
                                  nesterov=nesterov)
        model.train()
        ranks.append((model, opt, torch.cuda.Stream(device=dev)))
    return ranks


def _load_step_kernels(dev):
    """Launch the kernels of a training step once before any gossip kernel can spin: a kernel's
    first launch may load it, and loading may wait for the whole device (the gossip kernels
    themselves are loaded when their engine is built, see sgp_preload_kernels)."""
    net = sim._model(0).to(dev)
    x, y = sim._batch(0, 0)
    for _ in range(2):          # the second backward accumulates into existing .grad buffers
        ((net(x.to(dev)) - y.to(dev)) ** 2).mean().backward()
    torch.cuda.synchronize()


def _run(n, graph_name, ppi, steps, overlap, fused, nesterov, ppi_switch=None):
    dev = torch.device('cuda', 0)
    _load_step_kernels(dev)
    ranks = _world(n, graph_name, ppi, overlap, fused, nesterov)
    for step in range(steps):
        if ppi_switch is not None and step == ppi_switch[0]:
            torch.cuda.synchronize()
            for model, _, s in ranks:
                with torch.cuda.stream(s):
                    model.update_gossiper('peers_per_itr', ppi_switch[1])
        for r, (model, opt, s) in enumerate(ranks):
            with torch.cuda.stream(s):
                x, y = sim._batch(r, step)
                loss = ((model(x.to(dev)) - y.to(dev)) ** 2).mean()
                loss.backward()
                opt.step()
                opt.zero_grad()
                if not overlap:
                    model.transfer_params()          # launches the fused kernel; peers follow on their streams
    for model, _, s in ranks:
        with torch.cuda.stream(s):
            model.sync_comms()
            model.unbias()
    torch.cuda.synchronize()
    out = []
    for model, _, _ in ranks:
        model.engine.check()
        out.append((sim._flat(model.module).cpu(), float(model.ps_weight)))
    return out


@pytest.mark.parametrize('graph_name,ppi,overlap,fused,nesterov', [
    ('NPeerDynamicDirectedExponentialGraph', 1, False, True, True),
    ('NPeerDynamicDirectedExponentialGraph', 1, False, False, True),
    ('DynamicDirectedExponentialGraph', 2, False, True, False),
    ('NPeerDynamicDirectedExponentialGraph', 1, True, True, False),
    # (overlap + an external torch.optim optimizer is covered by the multi-process test only: its
    # host-side numerator / de-bias scaling reads the device step, and those host syncs of one
    # virtual rank wait on kernels of ranks the single host thread has not launched yet)
    ('RingGraph', 1, False, True, True),
])
def test_loopback_world_matches_simulation(graph_name, ppi, overlap, fused, nesterov):
    n, steps = 4, 5
    out = _run(n, graph_name, ppi, steps, overlap, fused, nesterov)
    want, ws = sim._simulate(n, graph_name, ppi, steps, overlap, nesterov)
    for r in range(n):
        got, w = out[r]
        torch.testing.assert_close(got, want[r], rtol=1e-4, atol=1e-5)
        assert abs(w - ws[r]) < 1e-5


@pytest.mark.parametrize('overlap', [False, True])
def test_loopback_schedule_swap_on_peers_per_itr_change(overlap):
    n, steps = 4, 6
    out = _run(n, 'NPeerDynamicDirectedExponentialGraph', 1, steps, overlap, True, True, ppi_switch=(3, 2))
    want, ws = sim._simulate(n, 'NPeerDynamicDirectedExponentialGraph', 1, steps, overlap, True,
                             ppi_switch=(3, 2))
    for r in range(n):
        torch.testing.assert_close(out[r][0], want[r], rtol=1e-4, atol=1e-5)
        assert abs(out[r][1] - ws[r]) < 1e-5


@pytest.mark.parametrize('algo', ['sgp', 'osgp'])
def test_loopback_graphed_trainer_equals_eager(algo):
    """two virtual ranks, each with its own captured CUDA graph (forward + fused loss + backward +
    fused gossip kernel); replays of the two graphs run on two streams and handshake on device"""
    from stochastic_gradient_push_b200 import models
    from stochastic_gradient_push_b200.optim import FusedGossipSGD
    from stochastic_gradient_push_b200.parallel.distributed import GossipDataParallel
    from stochastic_gradient_push_b200.parallel.symmetric import LocalWorld
    from stochastic_gradient_push_b200.parallel.trainer import GossipTrainer
    dev = torch.device('cuda', 0)
    n, steps = 2, 7
    results = []
    for use_graph in (False, True):
        lw = LocalWorld(n)
        trainers = []
        for r in range(n):
            torch.manual_seed(7 + r)
            net = models.TinyConvNet().to(dev).to(memory_format=torch.channels_last)
            model = GossipDataParallel(net, graph=sgp.NPeerDynamicDirectedExponentialGraph(r, n),
                                       overlap=(algo == 'osgp'), rank=r, world_size=n, heartbeat_timeout=20,
                                       symmetric_world=lw.view(r), transport='nvlink', grid=4, symmetric_name='loopback')
            opt = FusedGossipSGD(model, lr=0.05, momentum=0.9, weight_decay=1e-4, nesterov=True)
            if use_graph:
                # the copy-engine gather needs one graph per (row, parity), captured on first use;
                # a capture synchronises the device, which virtual ranks sharing one GPU cannot do
                # mid-step -> this test exercises the kernel gather under graphs (the DMA gather
                # runs in the eager loop-back tests above and in the multi-process tests)
                model.engine._gather_dma_pref = False
                model.engine._refresh_in_peers()
            trainers.append(GossipTrainer(model, opt, amp_dtype=None, use_cuda_graph=use_graph, warmup_iters=10 ** 6))
        gens = [torch.Generator().manual_seed(100 + r) for r in range(n)]
        for s in range(steps):
            if use_graph and s == 2:
                # capture EVERY rank's graph before any replay: a capture synchronises the device,
                # which must not happen while another virtual rank's replay waits for our flags
                for tr in trainers:
                    with torch.cuda.stream(tr.stream):
                        tr._capture()
            for r, tr in enumerate(trainers):
                x = torch.randn(8, 3, 32, 32, generator=gens[r]).pin_memory()
                y = torch.randint(0, 10, (8,), generator=gens[r]).pin_memory()
                tr.step(x, y)
            torch.cuda.synchronize()
        for tr in trainers:
            tr.finish()
        results.append([(tr.model.arena.flat.cpu().clone(), tr.engine.device_step) for tr in trainers])
        assert all((tr.graph is not None) == use_graph for tr in trainers)
    eager, graphed = results
    for r in range(n):
        torch.testing.assert_close(graphed[r][0], eager[r][0], rtol=1e-4, atol=1e-5)
        assert graphed[r][1] == eager[r][1] == steps
