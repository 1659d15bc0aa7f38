"""Fused gossip step and Overlap-SGP gather kernels vs an fp64 oracle, at sizes where their control
flow actually runs.

A CTA of the step kernels owns chunks b, b+G, b+2G, ... of the arena and cuts them into K segments;
phase 1 (SGD + publish) and phase 2 (pull + mix) interleave segment by segment, and the TMA-fed
kernels keep a ring of bulk copies in flight.  With at most one chunk per CTA only the last segment
carries data and no ring completes a lap.  So here numel = CHUNK * (grid * m + r) with 0 < r < grid:
CTAs own m or m + 1 chunks, and the cases together give CTAs with 0, 1, < K, == K, K + 1 and many
chunks, for K in {1, 2, 4, 7, 15} (15 = SGP_SEQ_STRIDE - 1, the most a step can publish).

Every buffer the kernels address through their arguments (z, grad, momentum, shadow, grad2) is a view
into an allocation with a whole chunk of NaN on either side.  Those bands must stay bit-identical:
a chunk index that runs past the arena in the last segment or the last CTA shows up there.

Loop-back layout: n <= 4 virtual ranks on one GPU, one stream each.  The ranks spin on each other's
flags, so every CTA of every rank must be resident at once; each test asserts n * grid <= max_grid
before its first launch.  (No more than 4 ranks: more streams than the default number of hardware
queues can put one rank's kernel behind another's on the same queue.)
"""
import functools
import gc

import pytest
import torch

import stochastic_gradient_push_b200 as sgp
from stochastic_gradient_push_b200.ops import oracle

pytestmark = pytest.mark.gpu

CHUNK = 4096
BAND = CHUNK                     # NaN sentinel elements on each side of every kernel-visible buffer
TOL = dict(rtol=1e-5, atol=1e-5)
LR, MU, WD = 0.1, 0.9, 1e-4

NPDDE = sgp.NPeerDynamicDirectedExponentialGraph
# column-stochastic but not doubly stochastic: push-sum weights drift away from 1, so the numerator
# scaling (z * w), the de-bias (/ w) and in_numerator=True all change the result
SELF_W = functools.partial(sgp.SelfWeightedMixing, self_weight=[0.3, 0.5, 0.6, 0.45])


@pytest.fixture(params=[True, False], ids=['pipe', 'regs'])
def pipe(request):
    """the full gossip step as the warp-specialised TMA kernel (sgp_step_pipe_kernel) or as the
    register-staged one (sgp_step_kernel)"""
    return request.param


@pytest.fixture(autouse=True)
def _no_gc_while_ranks_spin():
    """Dropping an engine frees symmetric memory, and that waits for the whole device.  One host
    thread launches every rank, so a free between two ranks' launches would wait for a kernel that
    waits for the next launch.  Collect while nothing spins, and not during a test."""
    gc.collect()
    gc.disable()
    try:
        yield
    finally:
        gc.enable()
        gc.collect()


class _Guarded(object):
    """`numel` elements between two NaN bands of BAND elements each (whole chunks, so the view keeps
    the 16-byte alignment the vector and TMA accesses need)"""

    def __init__(self, numel, dtype, dev):
        self.whole = torch.full((numel + 2 * BAND,), float('nan'), dtype=dtype, device=dev)
        self.view = self.whole[BAND:BAND + numel]
        self._bands0 = self._bands().clone()

    def _bands(self):
        bits = self.whole.view(torch.int16 if self.whole.dtype == torch.bfloat16 else torch.int32)
        return torch.cat([bits[:BAND], bits[-BAND:]])

    def intact(self):
        return torch.equal(self._bands(), self._bands0)


class _World(object):
    """n loop-back ranks.  bf16=True: bf16 gradient + bf16 shadow + fp32 grad2, the layout of
    bf16-compute training; otherwise one fp32 gradient.  grid=None: max_grid // n.

    The grid is set on the engines after they are built: an engine clamps it to the chunk count,
    while the kernels are written for CTAs that own no chunk too."""

    def __init__(self, pipe, n, numel, graph_cls, ppi=1, mixing_cls=None, grid=None, segments=4,
                 bf16=False, overlap=False, gather_grid=4):
        from stochastic_gradient_push_b200.ops.peer_mix import GossipEngine
        from stochastic_gradient_push_b200.parallel.symmetric import LocalWorld
        dev = torch.device('cuda', 0)
        torch.manual_seed(0)
        self.graph_cls, self.ppi = graph_cls, ppi
        self.mixing_cls = mixing_cls or sgp.UniformMixing
        lw = LocalWorld(n)
        self.engines, self.grad2s, self.guards = [], [], []
        self.streams = [torch.cuda.Stream(device=dev) for _ in range(n)]
        for r in range(n):
            graph = graph_cls(r, n, peers_per_itr=ppi)
            z = _Guarded(numel, torch.float32, dev)
            grad = _Guarded(numel, torch.bfloat16 if bf16 else torch.float32, dev)
            mom = _Guarded(numel, torch.float32, dev)
            z.view.normal_()
            mom.view.normal_()
            bufs = [z, grad, mom]
            shadow = grad2 = None
            if bf16:
                shadow = _Guarded(numel, torch.bfloat16, dev)
                grad2 = _Guarded(numel, torch.float32, dev)
                shadow.view.zero_()
                bufs += [shadow, grad2]
            e = GossipEngine(lw.view(r), z.view, graph, self.mixing_cls(graph, dev), grad=grad.view,
                             momentum=mom.view, shadow=shadow.view if bf16 else None,
                             with_residual=overlap, grid=grid, gather_grid=gather_grid, timeout_s=10.0,
                             name='scale', segments=segments)
            if bf16:
                e.set_sgd_buffers(grad.view, mom.view, grad2.view)
            e.ctx.set_pipe(pipe)
            assert e.ctx.segments() == segments
            self.engines.append(e)
            self.grad2s.append(grad2.view if bf16 else None)
            self.guards.append(bufs)
        self.max_grid = self.engines[0].max_grid
        self.grid = self.max_grid // n if grid is None else grid
        for e in self.engines:
            e.grid = self.grid
        # co-residency: a rank whose CTAs cannot all be resident next to the other ranks' would spin
        # until the heartbeat; that is a mistake in the test, so fail before anything is launched
        assert n * self.grid <= self.max_grid, \
            '%d ranks x grid %d cannot be co-resident (max_grid %d)' % (n, self.grid, self.max_grid)

    def oracle_graphs(self):
        n = len(self.engines)
        gs = [self.graph_cls(r, n, peers_per_itr=self.ppi) for r in range(n)]
        return gs, [self.mixing_cls(g, 'cpu') for g in gs]

    def new_grads(self):
        """fresh random gradients; returns grad + grad2 per rank in fp64"""
        gs = []
        for e, g2 in zip(self.engines, self.grad2s):
            e.grad.normal_()
            g = e.grad.double()
            if g2 is not None:
                g2.normal_()
                g = g + g2.double()
            gs.append(g)
        return gs

    def set_hyper(self, nesterov, grad_scale, do_sgd=True):
        for e in self.engines:
            e.set_hyper(LR, MU, WD, nesterov, do_sgd=do_sgd, grad_scale=grad_scale)

    def check(self, i, steps_done, z, m, psw, zeroed):
        e = self.engines[i]
        e.check()
        assert e.device_step == steps_done
        torch.testing.assert_close(e.z.double(), z, **TOL)
        torch.testing.assert_close(e.momentum.double(), m, **TOL)
        assert abs(e.ps_weight - psw) < 1e-6, (e.ps_weight, psw)
        if zeroed:
            assert not bool((e.grad != 0).any()), 'gradient not cleared'
            if self.grad2s[i] is not None:
                assert not bool((self.grad2s[i] != 0).any()), 'grad2 not cleared'
        if e.shadow is not None:
            assert torch.equal(e.shadow.view(torch.int16), e.z.bfloat16().view(torch.int16)), \
                'shadow != z.bfloat16()'
        for name, b in zip(('z', 'grad', 'momentum', 'shadow', 'grad2'), self.guards[i]):
            assert b.intact(), 'rank %d: guard band of %s overwritten' % (i, name)


def _sgd(x, g, m, grad_scale, nesterov):
    """the kernel's order: (grad + grad2) * grad_scale, then SGD-momentum on the numerator"""
    return oracle.sgd_momentum(x, g * grad_scale, m, LR, MU, WD, nesterov)


def _run_mix(w, steps, grad_scale, nesterov, in_numerator=False):
    n = len(w.engines)
    ogs, oms = w.oracle_graphs()
    zs = [e.z.double() for e in w.engines]
    ms = [e.momentum.double() for e in w.engines]
    ws = [1.0] * n
    w.set_hyper(nesterov, grad_scale)
    for step in range(steps):
        gs = w.new_grads()
        torch.cuda.synchronize()
        for e, s in zip(w.engines, w.streams):
            with torch.cuda.stream(s):
                e.mix(sgd=True, in_numerator=in_numerator)
        torch.cuda.synchronize()
        xs = []
        for i in range(n):
            x, ms[i] = _sgd(zs[i] if in_numerator else zs[i] * ws[i], gs[i], ms[i], grad_scale, nesterov)
            xs.append(x)
        xs, ws = oracle.mix_columns(xs, ws, ogs, oms)
        oracle.rotate_all(ogs)
        zs = [x / wt for x, wt in zip(xs, ws)]
        for i in range(n):
            w.check(i, step + 1, zs[i], ms[i], ws[i], zeroed=True)


# chunks per CTA are m (CTAs r..grid-1) and m + 1 (CTAs 0..r-1)
MIX_CASES = [
    # graph, ppi, mixing, grid, m, r, K, bf16 (+shadow +grad2), grad_scale, nesterov, in_numerator
    pytest.param(NPDDE, 1, None, 16, 0, 5, 4, False, 1.0, True, False, id='npdde1-chunks0or1-K4'),
    pytest.param(NPDDE, 2, None, 8, 3, 3, 4, True, 0.25, False, False, id='npdde2-chunks3or4-K4-bf16'),
    pytest.param(sgp.RingGraph, 1, SELF_W, 8, 7, 5, 7, False, 0.25, True, False, id='ring-chunks7or8-K7'),
    pytest.param(sgp.DynamicBipartiteExponentialGraph, 1, None, 6, 2, 1, 2, True, 1.0, True, False,
                 id='bipartite-chunks2or3-K2-bf16'),
    pytest.param(NPDDE, 2, SELF_W, 4, 40, 3, 15, False, 0.25, False, True, id='npdde2-chunks40or41-K15-numer'),
    pytest.param(NPDDE, 1, SELF_W, 8, 5, 2, 1, True, 0.25, True, False, id='npdde1-chunks5or6-K1-bf16'),
]


@pytest.mark.parametrize('graph_cls,ppi,mixing_cls,grid,m,r,K,bf16,grad_scale,nesterov,in_numerator',
                         MIX_CASES)
def test_fused_mix_matches_fp64_oracle(pipe, graph_cls, ppi, mixing_cls, grid, m, r, K, bf16, grad_scale,
                                       nesterov, in_numerator):
    w = _World(pipe, 4, CHUNK * (grid * m + r), graph_cls, ppi, mixing_cls, grid, K, bf16)
    # two full periods and one more step: both outbox parities and the WAR ack fence (step >= 2) run
    _run_mix(w, max(5, 2 * w.engines[0].period + 1), grad_scale, nesterov, in_numerator)


OVERLAP_CASES = [
    # gather, ppi (in-neighbours), grid, m, r, K, bf16 (+shadow +grad2), grad_scale
    pytest.param('dma', 1, 8, 5, 3, 4, False, 0.25, id='copy-engine-gather-K4'),
    pytest.param('tma', 2, 8, 6, 5, 7, True, 0.25, id='tma-gather-K7-bf16'),
    pytest.param('regs', 2, 6, 3, 2, 15, False, 1.0, id='register-gather-K15'),
]


@pytest.mark.parametrize('gather,ppi,grid,m,r,K,bf16,grad_scale', OVERLAP_CASES)
def test_overlap_publish_gather_fold_matches_fp64_oracle(pipe, gather, ppi, grid, m, r, K, bf16, grad_scale):
    """Overlap-SGP: publish(sgd, fold) on the main stream, gather() on a side stream, the residual of
    step k folded at step k+1, and a final local(fold) flush.  gather_grid 4: each gather CTA walks
    a dozen or more chunks per in-neighbour, so the TMA gather's 6-stage ring wraps several times."""
    n, steps, nesterov = 4, 6, False
    w = _World(pipe, n, CHUNK * (grid * m + r), NPDDE, ppi, None, grid, K, bf16, overlap=True, gather_grid=4)
    for e in w.engines:
        e._gather_dma_pref = gather == 'dma'
        e._refresh_in_peers()
        assert e.gather_dma == (gather == 'dma')
    side = [torch.cuda.Stream() for _ in range(n)]
    ogs, oms = w.oracle_graphs()
    zs = [e.z.double() for e in w.engines]
    ms = [e.momentum.double() for e in w.engines]
    ws = [1.0] * n
    res = [torch.zeros_like(z) for z in zs]
    wres = [0.0] * n
    for step in range(steps):
        gs = w.new_grads()
        w.set_hyper(nesterov, grad_scale, do_sgd=step > 0)      # no gradient yet at the first step
        torch.cuda.synchronize()
        for e, s in zip(w.engines, w.streams):
            with torch.cuda.stream(s):
                e.publish(sgd=True, fold=True)
        torch.cuda.synchronize()
        for e, s in zip(w.engines, side):
            with torch.cuda.stream(s):
                e.gather(tma=gather == 'tma')
        torch.cuda.synchronize()
        pub, pubw = [], []
        for i in range(n):
            x = zs[i] * ws[i]
            if step > 0:
                x, ms[i] = _sgd(x, gs[i], ms[i], grad_scale, nesterov)
            pub.append(x + res[i])
            pubw.append(ws[i] + wres[i])
        cols = [oms[j].scalar_weights(ogs[j].get_peers()[0]) for j in range(n)]
        for i in range(n):
            zs[i] = pub[i] / pubw[i]
            ws[i] = cols[i][0] * pubw[i]
            _, ins = ogs[i].get_peers()
            res[i] = sum(cols[j][1][i] * pub[j] for j in ins)
            wres[i] = sum(cols[j][1][i] * pubw[j] for j in ins)
        oracle.rotate_all(ogs)
        for i, e in enumerate(w.engines):
            w.check(i, step + 1, zs[i], ms[i], ws[i], zeroed=step > 0)
            torch.testing.assert_close(e.residual.double() * e.res_scale, res[i], **TOL)
            assert abs(e.res_weight - wres[i]) < 1e-6, (e.res_weight, wres[i])
    # flush: fold the last residual without publishing
    w.set_hyper(nesterov, grad_scale, do_sgd=False)
    for e in w.engines:
        e.local(sgd=False, fold=True)
    torch.cuda.synchronize()
    for i in range(n):
        w.check(i, steps, (zs[i] * ws[i] + res[i]) / (ws[i] + wres[i]), ms[i], ws[i] + wres[i], zeroed=False)


@functools.lru_cache(maxsize=None)
def _resnet50_arena_numel():
    from stochastic_gradient_push_b200 import models
    from stochastic_gradient_push_b200.utils.arena import FlatArena
    with torch.device('meta'):
        return FlatArena(list(models.resnet50().parameters())).total


def test_fused_mix_at_resnet50_size(pipe):
    """2 ranks at the training size and grid (ResNet-50 arena, ~6240 chunks, half the co-resident
    grid each): bf16 gradient + shadow + fp32 grad2, grad_scale != 1, default segments"""
    numel = _resnet50_arena_numel()
    w = _World(pipe, 2, numel, NPDDE, bf16=True)
    print('max_grid %d, grid %d, numel %d (%d chunks)' % (w.max_grid, w.grid, numel, numel // CHUNK))
    assert w.engines[0].ctx.segments() == 4
    _run_mix(w, 3, grad_scale=0.3, nesterov=True)
