#!/usr/bin/env python
"""Headline benchmark: synthetic ResNet-50 training throughput with hvd.DistributedOptimizer — the reference's own
benchmark (examples/pytorch/pytorch_synthetic_benchmark.py: torchvision-shape resnet50, SGD, op=Average, fixed random
batch) — device-timed, max over ranks.  Also drives BERT-large / GPT-2-medium and the allreduce bandwidth sweep
(`--model bert-large|gpt2-medium`, `--bench allreduce`).

    python bench.py                               # 1 GPU
    torchrun --nproc-per-node 8 bench.py --gpus 8 # 8 GPUs, one process per GPU

Prints ONE JSON line on rank 0 (see the contract in the task description).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def parse():
    p = argparse.ArgumentParser()
    p.add_argument('--gpus', type=int, default=1)
    p.add_argument('--steps', type=int, default=30)
    p.add_argument('--warmup', type=int, default=5)
    p.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    p.add_argument('--model', default='resnet50', choices=['resnet50', 'bert-large', 'gpt2-medium'])
    p.add_argument('--bench', default='train', choices=['train', 'allreduce'])
    p.add_argument('--batch-size', type=int, default=None, help='per-GPU batch (default: 64 resnet50, 8 bert-large seq 512, 4 gpt2-medium seq 1024)')
    p.add_argument('--seq-len', type=int, default=None)
    p.add_argument('--no-fused-optimizer', action='store_true')
    p.add_argument('--op', default='average', choices=['average', 'adasum'])
    p.add_argument('--fp32', action='store_true', help='disable bf16 autocast')
    p.add_argument('--bucket-wire-dtype', default=None, choices=['bf16', 'fp16'],
                   help='experimental: reduce the fp32 gradient buckets as bf16/fp16 (registered shadow buckets)')
    p.add_argument('--no-cuda-graph', action='store_true', help='eager forward/backward with gradient hooks instead of hvd.GraphedStep')
    p.add_argument('--bucket-cap-mb', type=float, default=32, help='size of the zero-copy gradient buckets')
    p.add_argument('--parity', action='store_true', help="the stock reference benchmark's configuration: fp32 (no TF32, no autocast), eager "
                   'hook-driven step, unfused optimizer — what `--impl reference` would run, for a same-config comparison')
    p.add_argument('--no-extras', action='store_true', help='skip extra.bert_large / extra.allreduce_busbw / extra.checks')
    p.add_argument('--sizes', default=None, help='allreduce sweep: comma separated byte sizes')
    p.add_argument('--dtype', default='fp32', help='allreduce sweep dtype: fp32|bf16|fp16')
    p.add_argument('--dump-outputs', default=None, metavar='DIR',
                   help='after the timed steps, write what the last timed training step computed (loss, and a fixed sample of '
                        'the updated parameters and of the reduced gradients) as DIR/<name>.npy, to compare two builds; '
                        'inputs are seeded, and resnet50 without --parity computes bit-identical outputs run to run')
    args = p.parse_args()
    if args.steps < 1:
        p.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'ours' or args.bench != 'train'):
        p.error('--dump-outputs applies to the training benchmark of this implementation')
    return args


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []
        self.thread = None

    def start(self):
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q, '--format=csv,noheader,nounits',
                                          '-lms', '200'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=3)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for l in self.lines:
            f = [x.strip() for x in l.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx, 'samples': len(sm), 'reasons': sorted(reasons)}


def reference_arm(args):
    """The unmodified reference cannot be installed offline (see DESIGN.md 'Reference install attempt'):
    third_party/{gloo,flatbuffers,boost,eigen,lbfgs,HTTPRequest} are empty and there is no MPI.

    The check looks for the reference's OWN native torch binding under baseline/_ref (never through `import horovod`: this
    repository ships a drop-in `horovod` namespace that resolves to horovod_b200).  Should a build ever be present, the
    reference's stock benchmark program runs against it, untouched, and its own "Total img/sec" line is reported."""
    import glob
    import re
    import subprocess
    if int(os.environ.get('RANK', '0')) != 0:
        return 0  # one JSON line for the whole job
    ref = os.path.join(ROOT, 'baseline', '_ref')
    native = glob.glob(os.path.join(ref, 'horovod', 'torch', 'mpi_lib_v2*.so'))
    if not native:
        print(json.dumps({'impl': 'reference', 'unavailable':
                          'horovod 0.28.1 does not build offline: third_party/gloo (and flatbuffers/boost/eigen/lbfgs) '
                          'submodules are empty in /root/reference and no MPI is installed (cmake: add_subdirectory '
                          'third_party/gloo has no CMakeLists.txt); baseline/_ref holds no horovod/torch/mpi_lib_v2*.so'}))
        return 0
    script = '/root/reference/examples/pytorch/pytorch_synthetic_benchmark.py'
    env = dict(os.environ, PYTHONPATH=ref + os.pathsep + os.environ.get('PYTHONPATH', ''))
    cmd = [sys.executable, '-m', 'horovod.runner.launch', '-np', str(args.gpus), sys.executable, script, '--model', 'resnet50',
           '--batch-size', str(args.batch_size or 64), '--num-warmup-batches', str(max(args.warmup, 3)),
           '--num-batches-per-iter', str(args.steps), '--num-iters', '1']
    try:
        out = subprocess.run(cmd, env=env, cwd=ref, capture_output=True, text=True, timeout=1800)
        m = re.search(r'Total img/sec on \d+ GPU\(s\): ([0-9.]+)', out.stdout)
        if out.returncode != 0 or not m:
            raise RuntimeError((out.stderr or out.stdout)[-300:])
        value = float(m.group(1))
    except Exception as e:  # noqa: BLE001
        print(json.dumps({'impl': 'reference', 'unavailable': 'reference build present but its benchmark did not run: %s' % str(e)[:200]}))
        return 0
    print(json.dumps({'impl': 'reference', 'metric': 'resnet50_synthetic_images_per_sec', 'value': value, 'unit': 'img/s',
                      'n_gpus': args.gpus, 'steps': args.steps, 'warmup': max(args.warmup, 3),
                      'ms_per_step': 1e3 * (args.batch_size or 64) * args.gpus / value, 'higher_is_better': True, 'scaling': 'weak',
                      'vs_baseline': None, 'dtype': 'fp32', 'data': 'synthetic',
                      'config': {'model': 'resnet50', 'global_batch': (args.batch_size or 64) * args.gpus, 'parallelism': 'dp%d' % args.gpus,
                                 'program': 'examples/pytorch/pytorch_synthetic_benchmark.py (stock, host-timed)'}}))
    return 0


def build_model(args, torch):
    from horovod_b200 import models
    if args.model == 'resnet50':
        bs = args.batch_size or 64
        model = models.resnet50().cuda().to(memory_format=torch.channels_last)

        def make_batch(device):
            x = torch.randn(bs, 3, 224, 224, device=device)
            y = torch.randint(0, 1000, (bs,), device=device)
            return (x, y)

        def step_fn(batch):
            x, y = batch
            x = x.contiguous(memory_format=torch.channels_last)
            return torch.nn.functional.cross_entropy(model(x), y)

        return model, make_batch, step_fn, bs, None, 'images/sec'
    if args.model == 'bert-large':
        bs = args.batch_size or 8
        seq = args.seq_len or 512
        model = models.bert_large().cuda()

        def make_batch(device):
            ids = torch.randint(0, 30522, (bs, seq), device=device)
            labels = torch.where(torch.rand(bs, seq, device=device) < 0.15, ids, torch.full_like(ids, -100))
            nsp = torch.randint(0, 2, (bs,), device=device)
            return (ids, labels, nsp)

        def step_fn(batch):
            ids, labels, nsp = batch
            return model(ids, labels=labels, next_sentence_label=nsp)

        return model, make_batch, step_fn, bs, seq, 'samples/sec'
    bs = args.batch_size or 4
    seq = args.seq_len or 1024
    model = models.gpt2_medium().cuda()

    def make_batch(device):
        ids = torch.randint(0, 50257, (bs, seq), device=device)
        return (ids,)

    def step_fn(batch):
        return model(batch[0], labels=batch[0])

    return model, make_batch, step_fn, bs, seq, 'samples/sec'


DUMP_SAMPLE = 1 << 22  # elements per sampled output: 16 MiB of float32 each, well under 64 MiB for all dumped arrays


def _reduced_grad(opt, p, torch):
    """p's gradient as the optimizer applied it: a bucket reduced in a wire dtype (--bucket-wire-dtype) keeps the reduced
    values in its bf16 / fp16 shadow, which the fused update reads directly, so p.grad still holds the local gradient."""
    bucket = getattr(opt, '_p_to_bucket', {}).get(p)
    if bucket is not None and bucket.get('shadow') is not None:
        return bucket['shadow_views'][p]
    return p.grad if p.grad is not None else torch.zeros_like(p)


def _step_outputs(model, opt, loss, torch):
    """What a caller of the training step holds after it: the loss, the updated parameters and the reduced gradients.
    Parameters and gradients are flattened in model.parameters() order and sampled at fixed, seeded positions."""
    params = torch.cat([p.detach().float().reshape(-1) for p in model.parameters()])
    grads = torch.cat([_reduced_grad(opt, p, torch).detach().float().reshape(-1) for p in model.parameters()])
    n = params.numel()
    if n > DUMP_SAMPLE:
        idx = torch.randint(n, (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values.to(params.device)
        params, grads = params[idx], grads[idx]
    return {'loss': loss.detach().float().reshape(()).cpu().numpy(), 'params': params.cpu().numpy(), 'grads': grads.cpu().numpy()}


def _time_train(args, model_name, steps, warmup, hvd, torch, sample_clocks, keep_outputs=False):
    """One training configuration: device-timed arm (inputs resident) and end-to-end arm (per-step pinned H2D input copy +
    D2H loss read).  Returns a dict (with keep_outputs, under 'outputs' what the last device-timed step computed); frees
    the model before returning."""
    from horovod_b200.data import DevicePrefetcher
    rank, size, local_rank = hvd.rank(), hvd.size(), hvd.local_rank()
    margs = argparse.Namespace(**vars(args))
    margs.model = model_name
    if model_name != args.model:
        margs.batch_size, margs.seq_len = None, None
    torch.manual_seed(0)  # same weights and batch on every run with the same arguments, so runs can be compared output for output
    model, make_batch, step_fn, bs, seq, unit = build_model(margs, torch)
    use_bf16 = not args.fp32
    eager = args.no_cuda_graph or args.parity
    lr_scaler = size if args.op == 'average' else 1
    if model_name == 'resnet50':
        base_opt = torch.optim.SGD(model.parameters(), lr=0.01 * lr_scaler, momentum=0.9)
    else:
        base_opt = torch.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=0.01)
    op = hvd.Average if args.op == 'average' else hvd.Adasum
    kw = {}
    if op == hvd.Average:
        kw = {'bucket_cap_mb': args.bucket_cap_mb,
              'bucket_wire_dtype': {'bf16': torch.bfloat16, 'fp16': torch.float16, None: None}[args.bucket_wire_dtype]}
    opt = hvd.DistributedOptimizer(base_opt, named_parameters=model.named_parameters(), op=op,
                                   fused=not (args.no_fused_optimizer or args.parity), **kw)
    hvd.broadcast_parameters(model.state_dict(), root_rank=0)
    hvd.broadcast_optimizer_state(opt, root_rank=0)
    model.train()

    dev_batch = make_batch('cuda')  # fixed synthetic batch on the device (as the reference benchmark does)
    host_batch = tuple(t.cpu().pin_memory() for t in dev_batch)  # the e2e arm copies this every step
    h2d_bytes = sum(t.numel() * t.element_size() for t in host_batch)

    def fwd(*batch):
        with torch.autocast('cuda', dtype=torch.bfloat16, enabled=use_bf16):
            return step_fn(batch)

    # the whole step — forward, backward and (multi-GPU) the gradient buckets' allreduce kernels, overlapped with backward
    # on a forked stream — is ONE CUDA graph; step() then applies the fused update.  Falls back to the eager hook-driven
    # step if capture is impossible (e.g. the Adasum optimizer's per-parameter steps).
    graphed = hvd.GraphedStep(fwd, opt, dev_batch, enabled=not eager)
    comm_nodes = len(getattr(opt, '_buckets', [])) if graphed.comm_in_graph else 0

    def timed(nsteps, e2e):
        hvd.barrier()
        torch.cuda.synchronize()
        k0 = hvd.runtime_stats()['kernel_launches']
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = None
        if e2e:
            # every step: host -> device copy of that step's inputs from pinned memory on the prefetcher's copy stream (the
            # copy of step i+1 overlaps the compute of step i) and a device -> host copy of the step's loss into pinned
            # memory; the host reads the loss of step i-2 while step i is issued (a training loop logs, it does not stall on
            # .item(): with a one-step lag the host could never run ahead of the device and its launch time — ~2 ms of
            # Python for BERT-large's 400 parameters — would be exposed), and every outstanding loss before the clock stops
            class _Loader:
                def __len__(self):
                    return nsteps

                def __iter__(self):
                    for _ in range(nsteps):
                        yield host_batch
            pf = DevicePrefetcher(_Loader(), device=f'cuda:{local_rank}', depth=2)
            ring = [(torch.zeros(1, dtype=torch.float32).pin_memory(), torch.cuda.Event()) for _ in range(3)]
            inflight = []  # (pinned buffer, event) of the steps whose loss copy has been issued but not read yet
            for i, batch in enumerate(pf):
                if len(inflight) == 2:  # the host stays at most two steps ahead of the device
                    buf, ev = inflight.pop(0)
                    ev.synchronize()
                    last = float(buf[0])
                loss = graphed(*batch)
                buf, ev = ring[i % 3]
                buf.copy_(loss.detach().float().reshape(1), non_blocking=True)
                ev.record()
                inflight.append((buf, ev))
            for buf, ev in inflight:
                ev.synchronize()
                last = float(buf[0])
            assert pf.h2d_bytes == h2d_bytes * nsteps
        else:
            for _ in range(nsteps):
                last = graphed(*dev_batch)
        e1.record()
        torch.cuda.synchronize()
        hvd.barrier()
        ms = e0.elapsed_time(e1)
        k1 = hvd.runtime_stats()['kernel_launches']
        t = torch.tensor([ms], dtype=torch.float64)
        ms = hvd.allreduce(t, op=hvd.Max, name='bench.ms').item()  # max over ranks
        return ms, (k1 - k0) + nsteps * comm_nodes, last

    for _ in range(max(3, warmup)):
        graphed(*dev_batch)
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank) if (rank == 0 and sample_clocks) else None
    if sampler:
        sampler.start()
    ms, launches, last = timed(steps, e2e=False)
    clocks = sampler.stop() if sampler else None
    outputs = _step_outputs(model, opt, last, torch) if keep_outputs else None
    for _ in range(2):
        graphed(*tuple(t.cuda(non_blocking=True) for t in host_batch))
    e2e_ms, _, last_loss = timed(steps, e2e=True)

    # every rank must hold bit-identical parameters after the run (each applied the same reduced gradients)
    flat = torch.cat([p.detach().float().reshape(-1) for p in model.parameters()])
    digest = torch.stack([flat.double().sum(), flat.double().abs().sum(), flat[::997].double().pow(2).sum()]).cpu()
    dmin = hvd.allreduce(digest, op=hvd.Min, name='bench.digest.min.' + model_name)
    dmax = hvd.allreduce(digest, op=hvd.Max, name='bench.digest.max.' + model_name)
    params_identical = bool(torch.equal(dmin, dmax)) and bool(torch.isfinite(digest).all())

    global_batch = bs * size
    out = {
        'model': model_name, 'unit': unit, 'value': round(global_batch * steps / (ms / 1e3), 2), 'ms_per_step': round(ms / steps, 3),
        'e2e_value': round(global_batch * steps / (e2e_ms / 1e3), 2), 'e2e_ms_per_step': round(e2e_ms / steps, 3),
        'h2d_bytes_per_step': h2d_bytes, 'last_loss': last_loss, 'gpu_launches': int(launches), 'clocks': clocks,
        'global_batch': global_batch, 'per_gpu_batch': bs, 'seq_len': seq, 'params_identical_across_ranks': params_identical,
        'cuda_graph': bool(graphed.captured), 'cuda_graph_fallback': graphed.fallback_reason,
        'allreduce_in_graph': bool(graphed.comm_in_graph), 'gradient_buckets': len(getattr(opt, '_buckets', [])),
        'optimizer': 'SGD(momentum=0.9)' if model_name == 'resnet50' else 'AdamW', 'outputs': outputs,
    }
    del graphed, opt, base_opt, model, dev_batch, host_batch
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    return out


def _nccl_group(torch, hvd):
    """torch.distributed NCCL process group next to the hvd runtime (the reference's data path IS ncclAllReduce:
    ops/nccl_operations.cc:256): bootstrapped through the same c10d store hvd.init() used, never a second server."""
    import torch.distributed as dist
    if dist.is_initialized():
        return dist
    from horovod_b200.common.basics import _EmbeddedRendezvous
    # NCCL prints its version banner on stdout at communicator creation: this program's stdout carries exactly one JSON
    # line, so library chatter goes to stderr while the group (and its first collective) come up
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        if _EmbeddedRendezvous.stores:
            store = dist.PrefixStore('bench_nccl', _EmbeddedRendezvous.stores[-1])
            dist.init_process_group('nccl', store=store, rank=hvd.rank(), world_size=hvd.size(),
                                    device_id=torch.device('cuda', hvd.local_rank()))
            warm = torch.ones(1024, device='cuda')
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        else:
            return None
    except Exception as e:  # noqa: BLE001
        sys.stderr.write('bench: NCCL comparison arm unavailable: %s\n' % e)
        return None
    finally:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)
    return dist


def _busbw_extra(args, hvd, torch):
    """allreduce bus bandwidth, ordinary cudaMalloc tensors, DEFAULT configuration of this library next to ncclAllReduce
    (torch.distributed NCCL) in the same job; device-timed, max over ranks, values checked."""
    size = hvd.size()
    dist = _nccl_group(torch, hvd)
    rows = []
    for nbytes in (4 << 10, 256 << 10, 4 << 20, 64 << 20, 512 << 20):
        n = nbytes // 4
        x = torch.ones(n, device='cuda')
        iters = max(4, min(50, int(2e9 // max(nbytes, 1 << 20))))
        row = {'bytes': nbytes}
        for arm in ('ours', 'nccl'):
            if arm == 'nccl' and dist is None:
                continue
            call = (lambda: hvd.allreduce_(x, op=hvd.Sum, name='bw.%d' % nbytes)) if arm == 'ours' else (lambda: dist.all_reduce(x))
            x.fill_(1.0)
            call()
            torch.cuda.synchronize()
            ok = bool((x[:8] == size).all() and (x[-8:] == size).all())
            for _ in range(2):
                call()
            hvd.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                call()
            e1.record()
            torch.cuda.synchronize()
            ms = hvd.allreduce(torch.tensor([e0.elapsed_time(e1) / iters], dtype=torch.float64), op=hvd.Max, name='bw.ms').item()
            row[arm + '_us'] = round(ms * 1e3, 1)
            row[arm + '_busbw_gbs'] = round(nbytes / (ms / 1e3) / 1e9 * 2 * (size - 1) / size, 1)
            row[arm + '_correct'] = ok
        rows.append(row)
        del x
    return {'dtype': 'fp32', 'tensors': 'plain cudaMalloc (unregistered), in place, blocking loop', 'rows': rows,
            'roofline_gbs_per_direction': 900}


def _checks_extra(hvd, torch):
    """Closed-form allreduce on every kernel path of the data plane, in the bench process (multi-GPU correctness the
    driver can see): small (one-shot), medium (two-shot / NVLS), large plain (software pipeline), registered zero-copy,
    and a collective captured as a CUDA-graph node."""
    size, rank = hvd.size(), hvd.rank()
    exp_sum = float(sum(range(1, size + 1)))
    res = {}

    def run(name, tensor, fn):
        tensor.fill_(float(rank + 1))
        fn(tensor)
        torch.cuda.synchronize()
        res[name] = bool((tensor == exp_sum).all().item())

    run('oneshot_4KiB', torch.empty(1024, device='cuda'), lambda t: hvd.allreduce_(t, op=hvd.Sum, name='chk.a'))
    run('twoshot_or_nvls_8MiB', torch.empty(2 << 20, device='cuda'), lambda t: hvd.allreduce_(t, op=hvd.Sum, name='chk.b'))
    run('pipelined_96MiB_plain', torch.empty(24 << 20, device='cuda'), lambda t: hvd.allreduce_(t, op=hvd.Sum, name='chk.c'))
    run('bf16_16MiB', torch.empty(8 << 20, device='cuda', dtype=torch.bfloat16), lambda t: hvd.allreduce_(t, op=hvd.Sum, name='chk.d'))
    if hvd.symm_available():
        z = hvd.symm_empty(4 << 20, dtype=torch.float32)
        run('zero_copy_16MiB_registered', z, lambda t: hvd.allreduce_(t, op=hvd.Sum, name='chk.e'))
        g = torch.cuda.CUDAGraph()
        z.fill_(0)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            hvd.captured_allreduce_(z, op=hvd.Sum)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        with torch.cuda.graph(g):
            hvd.captured_allreduce_(z, op=hvd.Sum)
        run('cuda_graph_node_16MiB', z, lambda t: g.replay())
    ag = hvd.allgather(torch.full((3,), float(rank), device='cuda'), name='chk.ag')
    res['allgather'] = bool((ag.view(size, 3)[:, 0].cpu() == torch.arange(size, dtype=torch.float32)).all())
    rs = hvd.reducescatter(torch.ones(size * 4, 5, device='cuda') * (rank + 1), op=hvd.Sum, name='chk.rs')
    res['reducescatter'] = bool((rs == exp_sum).all().item()) and tuple(rs.shape) == (4, 5)
    a2a = hvd.alltoall(torch.arange(size * 4, device='cuda', dtype=torch.float32) + 1000 * rank, name='chk.a2a')
    exp_a2a = torch.cat([torch.arange(rank * 4, rank * 4 + 4, dtype=torch.float32) + 1000 * r for r in range(size)]).cuda()
    res['alltoall'] = bool(torch.equal(a2a, exp_a2a))
    b = torch.full((1 << 20,), float(rank), device='cuda')
    hvd.broadcast_(b, root_rank=size - 1, name='chk.bc')
    res['broadcast'] = bool((b == size - 1).all().item())
    flags = torch.tensor([1.0 if v else 0.0 for v in res.values()])
    agree = hvd.allreduce(flags, op=hvd.Min, name='chk.all')
    return {k: bool(agree[i] > 0) for i, k in enumerate(res)}


def train_bench(args):
    import torch
    import horovod_b200.torch as hvd

    t_start = time.time()
    if args.op == 'adasum':
        # the GPU Adasum kernels work inside the symmetric buffer: make it hold the largest single delta (GPT-2's 206 MB wte)
        os.environ.setdefault('HVD_SYMM_BUFFER_BYTES', str(256 << 20))
    hvd.init()
    rank, size = hvd.rank(), hvd.size()
    torch.cuda.set_device(hvd.local_rank())
    # convolution algorithms from cuDNN's heuristics, deterministic ones only, so that two runs with the same arguments
    # compute the same steps: benchmark mode picks algorithms by timing them, and the pick differs from run to run.  It is
    # not faster here (ResNet-50, batch 64, bf16, one B200 at 1000 W, alternating runs: 4229 / 4236 img/s benchmark mode,
    # 4281 / 4412 img/s heuristics + deterministic).  --parity keeps the stock benchmark's benchmark mode.
    torch.backends.cudnn.benchmark = args.parity
    torch.backends.cudnn.deterministic = not args.parity
    torch.backends.cuda.matmul.allow_tf32 = not args.parity
    torch.backends.cudnn.allow_tf32 = not args.parity
    if args.parity:
        args.fp32 = True  # the stock reference benchmark: fp32, eager hooks, unfused optimizer, batch 64
    main = _time_train(args, args.model, args.steps, args.warmup, hvd, torch, sample_clocks=True,
                       keep_outputs=bool(args.dump_outputs) and rank == 0)
    if main['outputs'] is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in main['outputs'].items():
            np.save(os.path.join(args.dump_outputs, name + '.npy'), a)
    extra = {}
    if not args.no_extras:
        try:
            if size > 1:
                extra['checks'] = _checks_extra(hvd, torch)
                extra['allreduce_busbw'] = _busbw_extra(args, hvd, torch)
            if args.model == 'resnet50' and args.op == 'average' and time.time() - t_start < 240:
                # the second model of the BASELINE metric, same timing rules, fewer steps to bound the run
                b = _time_train(args, 'bert-large', min(args.steps, 20), 3, hvd, torch, sample_clocks=False)
                extra['bert_large'] = {'metric': 'bert-large synthetic pretraining throughput (whole job)', 'value': b['value'], 'unit': b['unit'],
                                       'ms_per_step': b['ms_per_step'], 'steps': min(args.steps, 20), 'warmup': 3, 'dtype': 'bf16' if not args.fp32 else 'fp32',
                                       'e2e': {'value': b['e2e_value'], 'ms_per_step': b['e2e_ms_per_step'], 'h2d_bytes_per_step': b['h2d_bytes_per_step'],
                                               'd2h_bytes_per_step': 4},
                                       'config': {'global_batch': b['global_batch'], 'per_gpu_batch': b['per_gpu_batch'], 'seq_len': b['seq_len'],
                                                  'optimizer': b['optimizer'], 'cuda_graph': b['cuda_graph'], 'allreduce_in_graph': b['allreduce_in_graph'],
                                                  'gradient_buckets': b['gradient_buckets']},
                                       'gpu_launches': b['gpu_launches'], 'params_identical_across_ranks': b['params_identical_across_ranks']}
        except Exception as e:  # noqa: BLE001 - the headline number must survive a failing extra
            extra['error'] = '%s: %s' % (type(e).__name__, str(e)[:300])
    extra.setdefault('checks', {})['params_identical_across_ranks'] = main['params_identical_across_ranks']
    if rank == 0:
        out = {
            'metric': f'{args.model} synthetic training throughput, hvd.DistributedOptimizer op={args.op} (whole job)',
            'value': main['value'], 'unit': main['unit'], 'n_gpus': size, 'steps': args.steps, 'warmup': max(3, args.warmup),
            'ms_per_step': main['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'bf16' if not args.fp32 else ('fp32' if args.parity else 'fp32(tf32)'),
            'data': 'synthetic (random images/tokens, random-init weights)', 'impl': 'ours',
            'config': {'model': args.model, 'global_batch': main['global_batch'], 'per_gpu_batch': main['per_gpu_batch'],
                       'seq_len': main['seq_len'], 'parallelism': f'dp{size}', 'optimizer': main['optimizer'],
                       'fused_optimizer': not (args.no_fused_optimizer or args.parity), 'grad_dtype': 'fp32',
                       'bucket_wire_dtype': args.bucket_wire_dtype or 'fp32', 'bucket_cap_mb': args.bucket_cap_mb,
                       'parity_mode': bool(args.parity),
                       'cudnn': {'benchmark': torch.backends.cudnn.benchmark, 'deterministic': torch.backends.cudnn.deterministic},
                       'cuda_graph': main['cuda_graph'], 'cuda_graph_fallback': main['cuda_graph_fallback'],
                       'allreduce_in_graph': main['allreduce_in_graph'], 'gradient_buckets': main['gradient_buckets'],
                       'l2': 'per-step working set (activations + 100+ MB of gradients) exceeds the 126 MB L2; no explicit flush',
                       'gpu_backend': hvd.gpu_backend_info(), 'tunables': hvd.tunable_params()},
            'clocks': main['clocks'],
            'e2e': {'value': main['e2e_value'], 'unit': main['unit'], 'ms_per_step': main['e2e_ms_per_step'],
                    'h2d_bytes_per_step': main['h2d_bytes_per_step'], 'd2h_bytes_per_step': 4, 'last_loss': main['last_loss'],
                    'loss_read': 'async D2H into pinned memory every step, read by the host two steps later'},
            'gpu_launches': main['gpu_launches'],
            'extra': extra,
        }
        print(json.dumps(out), flush=True)
    try:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception:  # noqa: BLE001
        pass
    hvd.shutdown()
    return 0


def allreduce_bench(args):
    """Bus bandwidth sweep: busBW = algBW * 2(N-1)/N, device-timed, max over ranks."""
    import torch
    import horovod_b200.torch as hvd

    hvd.init()
    rank, size = hvd.rank(), hvd.size()
    torch.cuda.set_device(hvd.local_rank())
    dt = {'fp32': torch.float32, 'bf16': torch.bfloat16, 'fp16': torch.float16}[args.dtype]
    sizes = [int(s) for s in args.sizes.split(',')] if args.sizes else [1 << p for p in range(10, 31, 2)]
    rows = []
    for nbytes in sizes:
        n = max(1, nbytes // torch.tensor([], dtype=dt).element_size())
        x = torch.randn(n, device='cuda').to(dt)
        iters = max(5, min(200, int(2e9 // max(nbytes, 1 << 16))))
        for _ in range(5):
            hvd.allreduce_(x, op=hvd.Sum, name=f'sweep.{nbytes}')
        hvd.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            hvd.allreduce_(x, op=hvd.Sum, name=f'sweep.{nbytes}')
        e1.record()
        torch.cuda.synchronize()
        ms = hvd.allreduce(torch.tensor([e0.elapsed_time(e1) / iters], dtype=torch.float64), op=hvd.Max, name='sweep.ms').item()
        alg = nbytes / (ms / 1e3) / 1e9
        rows.append({'bytes': nbytes, 'us': round(ms * 1e3, 2), 'algbw_gbs': round(alg, 2),
                     'busbw_gbs': round(alg * 2 * (size - 1) / max(size, 1), 2)})
    if rank == 0:
        best = max(r['busbw_gbs'] for r in rows) if rows else 0.0
        print(json.dumps({'metric': 'allreduce bus bandwidth sweep', 'value': best, 'unit': 'GB/s (peak busBW)', 'n_gpus': size,
                          'higher_is_better': True, 'dtype': args.dtype, 'impl': 'ours', 'rows': rows,
                          'config': {'gpu_backend': hvd.gpu_backend_info(), 'tunables': hvd.tunable_params(),
                                     'roofline_gbs_per_dir': 900, 'measured_peer_copy_gbs': 770}}), flush=True)
    hvd.shutdown()
    return 0


def main():
    args = parse()
    if args.impl == 'reference':
        return reference_arm(args)
    if args.bench == 'allreduce':
        return allreduce_bench(args)
    return train_bench(args)


if __name__ == '__main__':
    sys.exit(main())
