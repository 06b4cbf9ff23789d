"""Single-GPU checks of the public API (world size 1) + smoke()."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def hvd():
    import horovod_b200.torch as hvd
    hvd.init()
    torch.cuda.set_device(0)
    yield hvd
    hvd.shutdown()


def test_topology_discovered(hvd):
    topo = hvd.gpu_topology()
    assert "device 0/" in topo and "sm_100" in topo.replace("sm_10 0", "sm_100"), topo


def test_allreduce_world1_uses_native_scale_kernel(hvd):
    before = hvd.runtime_stats()['kernel_launches']
    t = torch.randn(1 << 20, device='cuda')
    out = hvd.allreduce(t, op=hvd.Sum, prescale_factor=2.0)
    torch.cuda.synchronize()
    torch.testing.assert_close(out, t * 2)
    assert hvd.runtime_stats()['kernel_launches'] > before


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16, torch.int32])
def test_collectives_world1(hvd, dtype):
    t = (torch.arange(4096, device='cuda') % 7).to(dtype)
    assert torch.equal(hvd.allreduce(t, op=hvd.Sum), t)
    assert torch.equal(hvd.allgather(t), t)
    assert torch.equal(hvd.broadcast(t, 0), t)
    assert torch.equal(hvd.alltoall(t), t)
    assert torch.equal(hvd.reducescatter(t, op=hvd.Sum), t)


@pytest.mark.parametrize("opt_name", ["sgd", "adamw"])
def test_fused_optimizer_matches_torch(hvd, opt_name):
    torch.manual_seed(0)
    def make():
        torch.manual_seed(0)
        return torch.nn.Sequential(torch.nn.Linear(64, 128), torch.nn.GELU(), torch.nn.Linear(128, 10)).cuda()
    m1, m2 = make(), make()
    if opt_name == "sgd":
        o1 = torch.optim.SGD(m1.parameters(), lr=0.1, momentum=0.9, weight_decay=1e-4, nesterov=True)
        o2 = torch.optim.SGD(m2.parameters(), lr=0.1, momentum=0.9, weight_decay=1e-4, nesterov=True)
    else:
        o1 = torch.optim.AdamW(m1.parameters(), lr=1e-2, weight_decay=0.05)
        o2 = torch.optim.AdamW(m2.parameters(), lr=1e-2, weight_decay=0.05)
    o2 = hvd.DistributedOptimizer(o2, named_parameters=m2.named_parameters(), fused=True)
    before = hvd.runtime_stats()['kernel_launches']
    for step in range(5):
        x = torch.randn(32, 64, device='cuda', generator=torch.Generator(device='cuda').manual_seed(step))
        for m, o in ((m1, o1), (m2, o2)):
            o.zero_grad()
            m(x).square().mean().backward()
            o.step()
    for a, b in zip(m1.parameters(), m2.parameters()):
        torch.testing.assert_close(a, b, rtol=2e-4, atol=2e-5)
    assert hvd.runtime_stats()['kernel_launches'] > before


def _small_cnn():
    torch.manual_seed(3)
    return torch.nn.Sequential(torch.nn.Conv2d(3, 8, 3, padding=1), torch.nn.BatchNorm2d(8), torch.nn.ReLU(),
                               torch.nn.AdaptiveAvgPool2d(1), torch.nn.Flatten(), torch.nn.Linear(8, 5)).cuda()


@pytest.mark.parametrize("fused", [False, True])
def test_graphed_step_matches_eager(hvd, fused):
    """hvd.GraphedStep (forward+backward as one CUDA graph replay, reduction + update after it) follows the same
    trajectory as the eager hook-driven step."""
    xs = [torch.randn(16, 3, 12, 12, device='cuda') for _ in range(6)]
    ys = [torch.randint(0, 5, (16,), device='cuda') for _ in range(6)]
    ref = _small_cnn()
    ropt = torch.optim.SGD(ref.parameters(), lr=0.05, momentum=0.9)
    for x, y in zip(xs, ys):
        ropt.zero_grad()
        torch.nn.functional.cross_entropy(ref(x), y).backward()
        ropt.step()
    model = _small_cnn()
    opt = hvd.DistributedOptimizer(torch.optim.SGD(model.parameters(), lr=0.05, momentum=0.9), named_parameters=model.named_parameters(),
                                   fused=fused)
    bn_before = model[1].running_mean.clone()
    step = hvd.GraphedStep(lambda x, y: torch.nn.functional.cross_entropy(model(x), y), opt, (xs[0], ys[0]), warmup_iters=2)
    assert step.captured, step.fallback_reason
    # the capture warm-up ran forward passes (BatchNorm statistics moved) but applied no update; realign the BN buffers
    model[1].running_mean.copy_(bn_before)
    model[1].running_var.fill_(1.0)
    model[1].num_batches_tracked.zero_()
    losses = [step(x, y).item() for x, y in zip(xs, ys)]
    assert step.replays == 6 and all(l == l for l in losses)
    for (n, a), (_, b) in zip(model.named_parameters(), ref.named_parameters()):
        torch.testing.assert_close(a, b, rtol=2e-4, atol=2e-5, msg=lambda m, n=n: f'{n}: {m}')
    torch.testing.assert_close(model[1].running_mean, ref[1].running_mean, rtol=1e-4, atol=1e-5)
    # eager fallback keeps working on the same object type
    eager = hvd.GraphedStep(lambda x, y: torch.nn.functional.cross_entropy(model(x), y), opt, (xs[0], ys[0]), enabled=False)
    assert not eager.captured and eager.fallback_reason == 'disabled'


def test_smoke_entry():
    import __graft_entry__ as g
    g.smoke()


def test_bench_dump_outputs_are_reproducible(tmp_path):
    """`bench.py --dump-outputs DIR` writes the last timed step's loss / parameter sample / gradient sample as float32 .npy,
    under 64 MB in all, and a second run with the same arguments writes the same arrays bit for bit."""
    import os
    import subprocess
    import sys
    import numpy as np
    from conftest import REPO
    dumps = []
    for run in ('a', 'b'):
        d = tmp_path / run
        r = subprocess.run([sys.executable, os.path.join(REPO, 'bench.py'), '--gpus', '1', '--steps', '2', '--warmup', '0',
                            '--no-extras', '--dump-outputs', str(d)], cwd=REPO, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        assert sorted(os.listdir(d)) == ['grads.npy', 'loss.npy', 'params.npy']
        assert sum(f.stat().st_size for f in d.iterdir()) < 64 << 20
        dumps.append({n: np.load(d / (n + '.npy')) for n in ('loss', 'params', 'grads')})
    a, b = dumps
    assert a['loss'].shape == () and a['params'].shape == a['grads'].shape == (1 << 22,)
    assert all(x.dtype == np.float32 and np.isfinite(x).all() for x in a.values())
    assert np.abs(a['grads']).max() > 0
    for n in a:
        assert np.array_equal(a[n], b[n]), n
