#!/usr/bin/env python
"""
bench.py -- ResNet-50 gossip-SGD throughput (BASELINE.json headline metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--algo sgp|osgp|dpsgd|ar]
                    [--batch-size B] [--impl ours|reference] [--dump-outputs DIR]

N > 1 is launched by the driver as
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N \
        --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
(one rank per GPU; RANK / LOCAL_RANK / WORLD_SIZE / MASTER_* come from the env).

What is timed (our arm):
  * `value`  : K replays of the captured training step -- forward + fused softmax-xent /
    prec@1 / prec@5 + backward + ONE fused sm_100a kernel (SGD-momentum + push-sum publish +
    P2P pull over NVLink + mix + de-bias) -- inputs resident on the device, CUDA events on
    the launching stream, barrier + synchronize on both sides, max over ranks.  Whole-job
    images/s.  Default precision = the reference arm's: fp32 activations / weights / master
    parameters with TF32 tensor-core convolution math (`--dtype fp32`).
  * `e2e`    : the same K steps through the public API (`GossipTrainer.step`) with the
    step's inputs copied from pinned host memory every step (prefetch stream) and the
    step's results (loss, prec@1, prec@5 = 12 bytes, what the reference loop reads back
    with three `.item()` calls) copied to pinned host memory every step.
  * `secondary`: the same two numbers for bf16 compute at the same batch and for the
    reference's per-GPU batch of 32, clearly labelled (never the headline).
Synthetic 3x224x224 fp32 images, random-init ResNet-50 (no network / datasets).
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--algo', default='sgp', choices=['sgp', 'osgp', 'dpsgd', 'ar', 'adpsgd'])
    ap.add_argument('--batch-size', '--batch_size', dest='batch_size', type=int, default=256,
                    help='per-agent batch; 256 = every shipped job script of the reference '
                         '(job_scripts/submit_*.sh: --batch_size 256 per gossip agent); one agent '
                         'per B200 here')
    ap.add_argument('--dtype', default='fp32', choices=['bf16', 'fp32'],
                    help='fp32 (default): fp32 activations / weights with TF32 tensor-core convolutions, '
                         'the precision of the reference arm; bf16: reported as a labelled secondary line')
    ap.add_argument('--secondary', action='store_true',
                    help='also measure the secondary lines when --gpus > 1 (default: single-GPU runs only)')
    ap.add_argument('--no-secondary', action='store_true',
                    help='skip the secondary (other precision / per-GPU batch 32) measurements')
    ap.add_argument('--model', default='resnet50')
    ap.add_argument('--ppi', type=int, default=1)
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--autocast', action='store_true',
                    help='bf16 via torch.autocast instead of the bf16 shadow-weight twin')
    ap.add_argument('--ar-transport', default='auto', choices=['auto', 'nvls', 'p2p', 'nccl'],
                    help='AllReduce-SGD data plane: NVLS multimem kernel (auto when supported), the '
                         'one-shot P2P kernel, or NCCL all-reduce + fused SGD')
    ap.add_argument('--adpsgd-rounds', type=int, default=4,
                    help='AD-PSGD: bilateral rounds a rank may start per applied gradient (0 = unbounded)')
    ap.add_argument('--skip-e2e', action='store_true')
    ap.add_argument('--skip-local', action='store_true',
                    help='skip the gossip-disabled re-measurement behind `exposed_comm` (N > 1)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the K timed replays behind `value`, write what the last one computed '
                         '(rank 0) as float32 DIR/<name>.npy: metrics = [loss, prec@1, prec@5], logits, '
                         'bn_buffers (running statistics) and params (a fixed seeded sample of the '
                         'updated parameters); inputs are seeded, so two builds can be compared '
                         'array by array')
    args = ap.parse_args()
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs needs --impl ours')
    return args


# --------------------------------------------------------------------------- #
# clocks sampling (B200_PROFILING.md recipe)
# --------------------------------------------------------------------------- #
class ClockSampler(object):
    QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '--query-gpu=' + self.QUERY, '--format=csv,noheader,nounits',
                 '-lms', '100', '-i', str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None,
                'sm_max_mhz': max(mx) if mx else None,
                'power_w_max': max(power) if power else None,
                'samples': len(sm), 'reasons': sorted(reasons)}


# --------------------------------------------------------------------------- #
def _build(args, dtype, bs, rank, world, dev):
    """model + trainer for one measured configuration"""
    import torch
    import stochastic_gradient_push_b200 as sgp
    from stochastic_gradient_push_b200 import models
    from stochastic_gradient_push_b200.optim import FusedGossipSGD
    from stochastic_gradient_push_b200.parallel.distributed import GossipDataParallel
    from stochastic_gradient_push_b200.parallel.trainer import GossipTrainer

    amp = torch.bfloat16 if dtype == 'bf16' else None
    torch.manual_seed(1 + rank)
    net = models.MODEL_ZOO[args.model]()
    models.init_imagenet_in_1hr(net)
    net = net.to(dev).to(memory_format=torch.channels_last)
    lr = 0.1 * bs * world / 256
    if args.algo == 'ar':
        from stochastic_gradient_push_b200.parallel.allreduce import AllReduceDataParallel, ARTrainer
        model = AllReduceDataParallel(net, transport=args.ar_transport)
        trainer = ARTrainer(model, lr=lr, momentum=0.9, weight_decay=1e-4, nesterov=True,
                            amp_dtype=amp, use_cuda_graph=not args.no_graph)
        return net, model, trainer, 'all-reduce (%s)' % model.transport
    if args.algo == 'adpsgd':
        from stochastic_gradient_push_b200.parallel.ad_psgd import BilatGossipDataParallel, make_bilat_trainer
        model = BilatGossipDataParallel(net, rank=rank, world_size=world,
                                        graph_class=sgp.DynamicBipartiteExponentialGraph,
                                        mixing_class=sgp.UniformMixing, lr=lr, momentum=0.9,
                                        weight_decay=1e-4, nesterov=True, verbose=False,
                                        heartbeat_timeout=60, max_rounds_per_update=(args.adpsgd_rounds or None))
        trainer = make_bilat_trainer(model, lr, amp_dtype=amp, use_cuda_graph=not args.no_graph)
        model.train()
        model.enable_gossip()
        return net, model, trainer, 'dynamic bipartite exponential (bilateral)'
    if args.algo == 'dpsgd':
        graph = sgp.RingGraph(rank, world, peers_per_itr=args.ppi)
        graph_name = 'static ring'
    else:
        graph = sgp.NPeerDynamicDirectedExponentialGraph(rank, world, peers_per_itr=args.ppi)
        graph_name = 'n-peer dynamic directed exponential'
    model = GossipDataParallel(net, graph=graph, push_sum=(args.algo != 'dpsgd'),
                               overlap=(args.algo == 'osgp'), rank=rank, world_size=world,
                               verbose=False, heartbeat_timeout=60,
                               compute_dtype=(torch.bfloat16 if (amp is not None and not args.autocast)
                                              else None))
    opt = FusedGossipSGD(model, lr=lr, momentum=0.9, weight_decay=1e-4, nesterov=True)
    trainer = GossipTrainer(model, opt, amp_dtype=amp, use_cuda_graph=not args.no_graph)
    return net, model, trainer, graph_name


DUMP_MAX_ELEMS = 1 << 22          # per array: 16 MB of float32, so a dump stays well under 64 MB


def _dump_sample(flat):
    """``flat`` itself, or a fixed seeded sample of DUMP_MAX_ELEMS of its elements (sorted indices,
    the same for every run with the same sizes)."""
    import numpy as np
    import torch
    if flat.numel() <= DUMP_MAX_ELEMS:
        return flat
    idx = np.sort(np.random.default_rng(0).choice(flat.numel(), DUMP_MAX_ELEMS, replace=False))
    return flat.index_select(0, torch.from_numpy(idx).to(flat.device))


def dump_outputs(out_dir, net, trainer):
    """What the last training step handed its caller, as float32 ``out_dir/<name>.npy``."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    logits = trainer.static_out.detach().float()
    arrays = {
        'metrics': trainer.static_metrics.detach().float(),          # [loss, prec@1 %, prec@5 %]
        'logits': logits if logits.numel() <= DUMP_MAX_ELEMS else _dump_sample(logits.reshape(-1)),
        'bn_buffers': _dump_sample(torch.cat([b.detach().reshape(-1).float() for b in net.buffers()
                                              if b.is_floating_point()])),
        'params': _dump_sample(torch.cat([p.detach().reshape(-1).float() for p in net.parameters()])),
    }
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), t.cpu().numpy().astype(np.float32))


def measure(args, dtype, bs, K, W, rank, world, dev, sample_clocks, dump_dir=None):
    """One configuration: W warm-up steps, K device-timed replays (`value`), then K steps through
    the public API with H2D of the inputs and D2H of [loss, prec@1, prec@5] every step (`e2e`).
    ``dump_dir``: write what the last of the K timed replays computed there (rank 0)."""
    import torch
    import torch.distributed as dist
    from stochastic_gradient_push_b200.ops import native

    net, model, trainer, graph_name = _build(args, dtype, bs, rank, world, dev)
    # synthetic data: a small pool of pinned host batches (the loader's output)
    g = torch.Generator().manual_seed(1234 + rank)
    pool = [(torch.randn(bs, 3, 224, 224, generator=g).pin_memory(),
             torch.randint(0, 1000, (bs,), generator=g).pin_memory()) for _ in range(4)]
    h2d_bytes = pool[0][0].numel() * 4 + pool[0][1].numel() * 8

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up: eager iterations, graph capture, a few replays ------------
    n_warm = max(W, 5)
    if args.algo == 'osgp' and world > 1 and getattr(model.engine, 'gather_dma', False):
        # copy-engine gather: one captured graph per (schedule row, outbox parity); visit them all
        # before the timed region (a capture inside it would be timed as a multi-100-ms "step")
        n_warm += 2 * model.engine.period + 1
    for i in range(n_warm):
        trainer.step(*pool[i % len(pool)])
    sync_all()
    launches_per_step = trainer.own_launches_per_step

    # ---- device-only timed region -------------------------------------------
    sampler = ClockSampler(dev.index) if (rank == 0 and sample_clocks) else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record(trainer.stream)
    for i in range(K):
        trainer.step_resident()
    e1.record(trainer.stream)
    sync_all()
    clocks = sampler.stop() if sampler else None
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = ms.item()
    value = bs * world * K / (ms / 1e3)
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, net, trainer)

    # ---- end-to-end timed region (public API, H2D + D2H every step) ---------
    e2e = None
    if not args.skip_e2e:
        trainer.prefetch(*pool[0])
        sync_all()
        e0.record(trainer.stream)
        slots = []
        for i in range(K):
            nxt = pool[(i + 1) % len(pool)]
            slots.append(trainer.step(None, None, nxt[0], nxt[1]))
        e1.record(trainer.stream)
        sync_all()
        rows = [trainer.metrics_ring[s].tolist() for s in slots]      # D2H results, all K read
        ms2 = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
        ms2 = ms2.item()
        e2e = {'value': round(bs * world * K / (ms2 / 1e3), 2), 'unit': 'images/s',
               'ms_per_step': round(ms2 / K, 4),
               'h2d_bytes_per_step': h2d_bytes, 'd2h_bytes_per_step': 12,
               'per_step_results': 'loss, prec@1, prec@5 (as the reference loop, gossip_sgd.py:394-407)',
               'last_loss': round(rows[-1][0], 4), 'last_prec1': round(rows[-1][1], 3),
               'last_prec5': round(rows[-1][2], 3)}
    trainer.finish()
    rounds = int(model.rounds_completed) if args.algo == 'adpsgd' else None

    # ---- exposed communication: the same step with gossip switched off (every rank trains alone,
    # SGD-only fused kernel), timed the same way on the same GPUs right after -- the difference is
    # what gossip costs per step after all overlap (kernel time + waiting for the in-neighbours)
    exposed = None
    if world > 1 and args.algo != 'ar' and not args.skip_local and sample_clocks:   # (main measurement only)
        g_gossip = trainer.graph
        if args.algo == 'adpsgd':
            g_local = g_gossip               # the captured graph is forward/backward only

            def switch(gossip_on):
                model.enable_gossip() if gossip_on else model.disable_gossip()
        else:
            model.gossip_enable = False
            trainer.graph = None
            trainer._eager_steps = 0
            for i in range(5):               # eager warm-up + capture of the gossip-free step
                trainer.step(*pool[i % len(pool)])
            g_local = trainer.graph

            def switch(gossip_on):
                if not gossip_on and model.gossip_enable:
                    trainer.finish()         # land the deferred SGD / gathered residual (overlap) first
                model.gossip_enable = gossip_on
                trainer.graph = g_gossip if gossip_on else g_local

        def timed(gossip_on):
            switch(gossip_on)
            for i in range(2):
                trainer.step_resident()
            sync_all()
            e0.record(trainer.stream)
            for i in range(K):
                trainer.step_resident()
            e1.record(trainer.stream)
            sync_all()
            t = torch.tensor([e0.elapsed_time(e1)], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return t.item() / K

        # A B A B: alternate so that clock / thermal drift hits both arms alike
        with_g, without = [], []
        for _ in range(2):
            without.append(timed(False))
            with_g.append(timed(True))
        g_ms, l_ms = sum(with_g) / 2, sum(without) / 2
        exposed = {'ms_per_step': round(g_ms - l_ms, 4), 'with_gossip_ms_per_step': round(g_ms, 4),
                   'local_only_ms_per_step': round(l_ms, 4),
                   'runs_ms': {'with_gossip': [round(v, 4) for v in with_g], 'local_only': [round(v, 4) for v in without]},
                   'how': 'same captured step with gossip switched off (SGD-only kernel; every rank trains '
                          'alone), same GPUs, K steps each, alternated local/gossip/local/gossip, max over ranks'}
        switch(True)
        trainer.finish()
    if args.algo == 'adpsgd':
        model.shutdown()
    res = {'value': round(value, 2), 'ms_per_step': round(ms / K, 4), 'e2e': e2e, 'clocks': clocks,
           'exposed_comm': exposed, 'gossip_rounds': rounds,
           'launches_per_step': launches_per_step, 'graph_name': graph_name,
           'native_ops': native.describe_paths() if hasattr(native, 'describe_paths') else None}
    del trainer, model, net, pool
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    return res


DTYPE_LABEL = {'fp32': 'fp32 (fp32 activations/weights/master, TF32 tensor-core conv math = the '
                       "reference's cuDNN default)",
               'bf16': 'bf16 (bf16 NHWC activations + conv math, fp32 master weights / BN / gossip)'}


def run_ours(args):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from stochastic_gradient_push_b200 import models
    from stochastic_gradient_push_b200.ops import fused_bn as _fb

    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
        dist.barrier()
    torch.backends.cudnn.benchmark = True
    # the reference's defaults: TF32 inside cuDNN convolutions, full fp32 for matmul (the classifier)
    torch.backends.cudnn.allow_tf32 = True

    bs, K, W = args.batch_size, args.steps, args.warmup
    main = measure(args, args.dtype, bs, K, W, rank, world, dev, sample_clocks=True,
                   dump_dir=args.dump_outputs)
    # secondary, clearly labelled lines: the other precision at the headline batch, and the
    # reference's per-GPU batch (32 images per GPU in its 8-GPU-per-node job scripts), where the
    # gossip step is a larger share of the iteration
    secondary = {}
    # (multi-GPU runs measure the headline configuration only -- one model / one symmetric-memory
    # rendezvous per process; pass --secondary to force the extra lines there.  Batch-32 and bf16
    # multi-GPU numbers: profiles/bench_r2_n2_*_bs32_*, profiles/bench_n8_sgp_bs32_r2_fp32.json)
    if not args.no_secondary and (world == 1 or args.secondary):
        other = 'bf16' if args.dtype == 'fp32' else 'fp32'
        for key, (dt, b) in (('%s_bs%d' % (other, bs), (other, bs)), ('%s_bs32' % args.dtype, (args.dtype, 32))):
            if (dt, b) == (args.dtype, bs):
                continue
            r = measure(args, dt, b, K, W, rank, world, dev, sample_clocks=False)
            secondary[key] = {'dtype': DTYPE_LABEL[dt], 'per_gpu_batch': b, 'value': r['value'],
                              'unit': 'images/s', 'ms_per_step': r['ms_per_step'],
                              'e2e_value': r['e2e']['value'] if r['e2e'] else None,
                              'e2e_ms_per_step': r['e2e']['ms_per_step'] if r['e2e'] else None}

    if rank == 0:
        out = {
            'metric': 'resnet50_%s_images_per_sec' % args.algo, 'value': main['value'],
            'unit': 'images/s', 'n_gpus': world, 'steps': K, 'warmup': W,
            'ms_per_step': main['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': DTYPE_LABEL[args.dtype], 'data': 'synthetic', 'impl': 'ours',
            'config': {'model': args.model, 'algorithm': args.algo, 'graph': main['graph_name'],
                       'peers_per_itr': args.ppi, 'per_gpu_batch': bs, 'global_batch': bs * world,
                       'image': '3x224x224', 'parallelism': 'dp%d-gossip' % world,
                       'master_weights': 'fp32 flat arena', 'layout': 'NHWC',
                       'compute_path': ('fp32 activations and weights; TF32 tcgen05 / cuDNN convolutions'
                                        if args.dtype == 'fp32' else
                                        ('autocast' if (args.autocast or args.algo == 'ar') else
                                         'bf16 shadow weights written by the gossip kernel')),
                       'cuda_graph': not args.no_graph,
                       'conv1x1': ('tcgen05 GEMM (TMA/TMEM, kind::%s), BN statistics and skip gradient '
                                   'fused into its epilogues' % ('tf32' if args.dtype == 'fp32' else 'f16')
                                   if _fb.USE_TCGEN05_CONV1X1 else 'library'),
                       'loss': 'fused softmax-xent + prec@1/5 kernel inside the captured step',
                       'l2': 'per-step working set (activations+weights > 1 GB) exceeds the '
                             '126 MB L2; no explicit flush'},
            'clocks': main['clocks'], 'e2e': main['e2e'], 'exposed_comm': main['exposed_comm'],
            'gossip_rounds_completed_rank0': main['gossip_rounds'],
            'gpu_launches': (main['launches_per_step'] or 0) * K,
            'gpu_launches_per_step': main['launches_per_step'],
            'secondary': secondary,
        }
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def relaunch_under_torchrun(args):
    """`python bench.py --gpus N` without a launcher: start one rank per GPU ourselves."""
    import socket
    sock = socket.socket()
    sock.bind(('127.0.0.1', 0))
    port = sock.getsockname()[1]
    sock.close()
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node',
           str(args.gpus), '--master-addr', '127.0.0.1', '--master-port', str(port),
           os.path.abspath(__file__)] + sys.argv[1:]
    sys.exit(subprocess.call(cmd))


def main():
    args = parse()
    if args.gpus > 1 and 'RANK' not in os.environ:
        relaunch_under_torchrun(args)
    if args.impl == 'reference':
        sys.path.insert(0, os.path.join(ROOT, 'baseline'))
        try:
            import run_reference
        except Exception as e:       # pragma: no cover
            print(json.dumps({'impl': 'reference', 'unavailable': 'shim import failed: %r' % e}))
            return
        try:
            run_reference.main(args)
        except SystemExit:
            raise
        except Exception as e:
            import traceback
            traceback.print_exc()
            if int(os.environ.get('RANK', 0)) == 0:
                print(json.dumps({'impl': 'reference',
                                  'unavailable': 'reference run failed: %s' % str(e)[:200]}))
        return
    run_ours(args)


if __name__ == '__main__':
    main()
