"""Unit tests of framework-neutral helpers: async data loader, ray strategy/discovery logic (without ray), stores."""
import pytest

from horovod_b200.data import AsyncDataLoaderMixin, BaseDataLoader
from horovod_b200.ray import strategy
from horovod_b200.ray.elastic import RayHostDiscovery
from horovod_b200.spark.common.store import LocalStore, Store


class _Loader(BaseDataLoader):
    def __init__(self, n, fail_at=None):
        self.n, self.fail_at = n, fail_at

    def __len__(self):
        return self.n

    def _iterate(self):
        for i in range(self.n):
            if self.fail_at == i:
                raise ValueError('boom')
            yield i


class _AsyncLoader(AsyncDataLoaderMixin, _Loader):
    pass


def test_async_loader_epochs_and_errors():
    l = _AsyncLoader(async_loader_queue_size=4, n=10)
    assert list(l) == list(range(10))
    assert list(l) == list(range(10))  # second epoch
    l.close_async_loader()
    sync = _AsyncLoader(async_loader_queue_size=0, n=5)
    assert list(sync) == list(range(5))
    bad = _AsyncLoader(async_loader_queue_size=2, n=5, fail_at=3)
    with pytest.raises(ValueError):
        list(bad)
    bad.close_async_loader()


def test_ray_rank_assignment_and_discovery():
    from horovod_b200.runner.cluster_job import assign_slots
    from horovod_b200.runner.mesh_run import create_slot_env_vars
    envs = [create_slot_env_vars(s) for s in assign_slots(['a', 'b', 'a', 'b', 'b'])]
    assert [e['HOROVOD_RANK'] for e in envs] == ['0', '2', '1', '3', '4']
    assert envs[4]['HOROVOD_LOCAL_RANK'] == '2' and envs[4]['HOROVOD_CROSS_SIZE'] == '1' and envs[4]['HOROVOD_CROSS_RANK'] == '0'
    assert envs[1]['HOROVOD_CROSS_RANK'] == '1' and envs[0]['HOROVOD_LOCAL_SIZE'] == '2'
    assert strategy.pack_bundles(3, 2) == ([{'CPU': 2}] * 3, 'PACK')
    from horovod_b200.ray import RayExecutor
    ex = RayExecutor(RayExecutor.create_settings(), num_hosts=2, num_workers_per_host=4, cpus_per_worker=2, use_gpu=True)
    b, st, wb, wr = ex._placement()
    assert b == [{'CPU': 8, 'GPU': 4}] * 2 and st == 'STRICT_SPREAD' and wb == [0, 0, 0, 0, 1, 1, 1, 1] and wr[0] == {'CPU': 2, 'GPU': 1}
    bundles, strat = strategy.colocated_bundles(2, 4, cpus_per_worker=2, gpus_per_worker=1)
    assert bundles == [{'CPU': 8, 'GPU': 4}] * 2 and strat == 'STRICT_SPREAD'
    nodes = [{'alive': True, 'NodeManagerAddress': 'n1', 'Resources': {'CPU': 16, 'GPU': 8}},
             {'alive': True, 'NodeManagerAddress': 'n2', 'Resources': {'CPU': 4}},
             {'alive': False, 'NodeManagerAddress': 'n3', 'Resources': {'CPU': 64, 'GPU': 8}}]
    d = RayHostDiscovery(use_gpu=True, cpus_per_slot=2, gpus_per_slot=1, nodes_fn=lambda: nodes)
    assert d.find_available_hosts_and_slots() == {'n1': 8}
    assert RayHostDiscovery(nodes_fn=lambda: nodes).find_available_hosts_and_slots() == {'n1': 16, 'n2': 4}


def test_local_store(tmp_path):
    s = Store.create(str(tmp_path))
    assert isinstance(s, LocalStore)
    ck = s.get_checkpoint_path('run1')
    s.write(ck, b'abc')
    assert s.exists(ck) and s.read(ck) == b'abc'
    assert s.get_logs_path('run1').endswith('runs/run1/logs') and s.get_train_data_path(3).endswith('intermediate_train_data.3')
    from horovod_b200.spark.common.store import FilesystemStore
    remote = Store.create('hdfs://namenode:8020/x/y')  # lazily bound pyarrow.fs filesystem
    assert isinstance(remote, FilesystemStore) and remote.get_run_path('r') == 'hdfs://namenode:8020/x/y/runs/r'


def test_utils_timing_helpers():
    from horovod_b200.utils import ClockSampler, device_timer, measured_peaks
    lines = ['1965, 1965, 612.3, Not Active, Not Active, Not Active, Not Active',
             '1410, 1965, 998.1, Not Active, Not Active, Not Active, Active',
             'garbage', '1965, 1965, 700.0, Not Active, Not Active, Not Active, Not Active']
    s = ClockSampler.summarise(lines)
    assert s == {'sm_mhz': 1965.0, 'sm_max_mhz': 1965.0, 'samples': 3, 'reasons': ['sw_power_cap']}
    assert ClockSampler.summarise([])['sm_mhz'] is None
    with device_timer() as t:
        sum(range(1000))
    assert t.ms is not None and t.ms >= 0
    assert isinstance(measured_peaks(), dict)


def test_ops_package_surface():
    import horovod_b200.ops as ops
    assert ops.sim.DTYPE_CODE[__import__('torch').bfloat16] == 10 and ops.sim.TWOSHOT == 1
    assert callable(ops.fused_sgd_step) and callable(ops.fused_adam_step) and callable(ops.symm_empty)


def test_common_util_availability_helpers():
    import torch
    from horovod_b200.common import util
    assert util.extension_available('torch') and not util.extension_available('definitely_not_a_framework')
    assert util.gloo_built() and util.nccl_built() and not util.mpi_built() and not util.ddl_built() and not util.ccl_built()
    assert util.gpu_available() == torch.cuda.is_available()
    assert util.check_installed_version('torch', torch.__version__)
    with pytest.warns(UserWarning, match='built against'):
        assert not util.check_installed_version('torch', '0.0.0')
    with pytest.raises(RuntimeError):
        util.check_installed_version('torch', '0.0.0', exception=RuntimeError('x'))

    class Ops:
        Average, Sum = 0, 1
    f = util.get_average_backwards_compatibility_fun(Ops)
    assert f(None, None) == Ops.Average and f(None, False) == Ops.Sum and f(Ops.Sum, None) == Ops.Sum
    with pytest.raises(ValueError):
        f(Ops.Sum, True)
    with util.env(HVD_T_X='1'):
        import os
        assert os.environ['HVD_T_X'] == '1'
    assert 'HVD_T_X' not in __import__('os').environ
    assert util.split_list([1, 2, 3, 4, 5], 2) == [[1, 2, 3], [4, 5]] and util.num_rank_is_power_2(8) and not util.num_rank_is_power_2(6)


def test_bench_reference_arm_reports_unavailable():
    """`bench.py --impl reference` must print ONE JSON line with impl=reference and exit 0 — and must not be fooled by the
    drop-in `horovod` namespace of this repository."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--gpus', '1', '--steps', '2', '--warmup', '3'],
                       cwd=root, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith('{')][-1]
    rec = json.loads(line)
    assert rec['impl'] == 'reference' and ('unavailable' in rec or 'value' in rec)
    if 'unavailable' in rec:
        assert 'mpi_lib_v2' in rec['unavailable'] or 'does not build offline' in rec['unavailable']


def test_bench_rejects_bad_arguments():
    """bench.py refuses a run with no timed step, and --dump-outputs outside the training benchmark of this library."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for extra, msg in ((['--steps', '0'], '--steps must be at least 1'),
                       (['--dump-outputs', 'out', '--impl', 'reference'], '--dump-outputs applies to'),
                       (['--dump-outputs', 'out', '--bench', 'allreduce'], '--dump-outputs applies to')):
        r = subprocess.run([sys.executable, os.path.join(root, 'bench.py')] + extra, cwd=root, capture_output=True, text=True,
                           timeout=120)
        assert r.returncode == 2 and msg in r.stderr, (extra, r.stderr[-2000:])
        assert not os.path.exists(os.path.join(root, 'out'))


def test_every_hvd_knob_is_documented():
    """docs/knobs.md lists every HVD_* environment variable the sources read."""
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    names = set()
    for base, _, files in os.walk(os.path.join(root, 'horovod_b200')):
        if '__pycache__' in base or os.sep + 'build' in base:
            continue
        for f in files:
            if f.endswith(('.cc', '.h', '.cu', '.cuh', '.py')):
                with open(os.path.join(base, f), errors='ignore') as fh:
                    names |= set(re.findall(r'["\'](HVD_[A-Z0-9_]+)["\']', fh.read()))
    doc = open(os.path.join(root, 'docs', 'knobs.md')).read()
    missing = sorted(n for n in names if n not in doc and not n.startswith('HVD_TEST_'))
    assert not missing, 'undocumented knobs: %s' % missing


def test_gpu_numa_cpu_list_from_sysfs(tmp_path):
    """NUMA binding helper (SURVEY C14: pin near the GPU's NUMA node): PCI address -> numa_node -> cpulist, on a fake sysfs."""
    from horovod_b200.common.util import _parse_cpulist, bind_to_gpu_numa, gpu_numa_cpus
    d = tmp_path
    (d / 'bus/pci/devices/0000:1b:00.0').mkdir(parents=True)
    (d / 'devices/system/node/node1').mkdir(parents=True)
    (d / 'bus/pci/devices/0000:1b:00.0/numa_node').write_text('1\n')
    (d / 'devices/system/node/node1/cpulist').write_text('56-59,112\n')
    assert gpu_numa_cpus(0, 0x1b, 0, str(d)) == {56, 57, 58, 59, 112}
    assert gpu_numa_cpus(0, 0x1c, 0, str(d)) is None            # unknown device
    (d / 'bus/pci/devices/0000:1b:00.0/numa_node').write_text('-1\n')
    assert gpu_numa_cpus(0, 0x1b, 0, str(d)) is None            # no NUMA information
    assert _parse_cpulist('0-2,8,10-11') == {0, 1, 2, 8, 10, 11}
    assert bind_to_gpu_numa(0, str(d)) is None                   # no GPU here: never touches the affinity


def test_fused_step_validation_is_pure_and_falls_back_cleanly(native_built):
    """DistributedOptimizer(fused=True) on parameters the fused kernels cannot take (CPU tensors): the eligibility pass must
    not touch any optimizer state, and the wrapped optimizer's own step() must then run exactly once (round-1 advisor
    finding: the old code mutated momentum buffers / Adam step counts before bailing out and left '_hvd_init' in state_dict)."""
    import copy

    import torch

    import horovod_b200.torch as hvd
    from horovod_b200.torch.optimizer import _fused_plan
    hvd.init()
    try:
        for make in (lambda ps: torch.optim.SGD(ps, lr=0.1, momentum=0.9), lambda ps: torch.optim.AdamW(ps, lr=0.01)):
            torch.manual_seed(0)
            model = torch.nn.Linear(6, 3)
            ref = copy.deepcopy(model)
            opt = hvd.DistributedOptimizer(make(model.parameters()), named_parameters=model.named_parameters(), fused=True)
            ropt = make(ref.parameters())
            for step in range(3):
                x = torch.randn(4, 6, generator=torch.Generator().manual_seed(step))
                for m, o in ((model, opt), (ref, ropt)):
                    o.zero_grad()
                    m(x).square().mean().backward()
                assert _fused_plan(opt) is None            # CPU parameters: not eligible ...
                before = {k: v for k, v in opt.state_dict()['state'].items()}
                assert _fused_plan(opt) is None and opt.state_dict()['state'].keys() == before.keys()  # ... and nothing was touched
                opt.step()
                ropt.step()
            for a, b in zip(model.parameters(), ref.parameters()):
                torch.testing.assert_close(a, b)           # stepped exactly once per step()
            for st in opt.state_dict()['state'].values():
                assert '_hvd_init' not in st
    finally:
        hvd.shutdown()
