"""Numerics of the sm_100a P2P kernels on ONE GPU: N simulated ranks = N buffers + N concurrently running kernels
(csrc/common/sim_api.cc).  Reference: plain PyTorch fp32/fp64 math of the same op."""
import ctypes
import itertools

import pytest
import torch

pytestmark = pytest.mark.gpu

DT = {torch.uint8: 0, torch.int8: 1, torch.int16: 3, torch.int32: 4, torch.int64: 5, torch.float16: 6, torch.float32: 7,
      torch.float64: 8, torch.bfloat16: 10}
ONESHOT, TWOSHOT = 0, 1
SUM, MIN, MAX, PROD = 1, 3, 4, 5


def _lib():
    from horovod_b200.common.basics import load_library
    lib = load_library()
    lib.hvd_sim_allreduce.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int64),
                                      ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64), ctypes.c_int,
                                      ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                      ctypes.c_double, ctypes.c_int, ctypes.POINTER(ctypes.c_float)]
    lib.hvd_sim_allgather.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.POINTER(ctypes.c_uint64),
                                      ctypes.POINTER(ctypes.c_uint64), ctypes.c_int]
    return lib


def sim_allreduce(ins, outs, dtype, wire, op, variant, ctas, pre=1.0, post=1.0, repeats=1):
    """ins/outs: [nranks][ntensors] CUDA tensors."""
    lib = _lib()
    n, t = len(ins), len(ins[0])
    counts = (ctypes.c_int64 * t)(*[x.numel() for x in ins[0]])
    ip = (ctypes.c_uint64 * (n * t))(*[x.data_ptr() for r in ins for x in r])
    op_ = (ctypes.c_uint64 * (n * t))(*[x.data_ptr() for r in outs for x in r])
    ms = ctypes.c_float(0)
    rc = lib.hvd_sim_allreduce(n, 0, t, counts, ip, op_, DT[dtype], DT[wire], op, variant, ctas, pre, post, repeats,
                               ctypes.byref(ms))
    assert rc == 0, f"sim allreduce failed with code {rc}"
    return ms.value


def _make(n, sizes, dtype, seed=0):
    g = torch.Generator(device='cuda').manual_seed(seed)
    ins = []
    for r in range(n):
        row = []
        for s in sizes:
            if dtype.is_floating_point:
                row.append((torch.randn(s, device='cuda', generator=g, dtype=torch.float32)).to(dtype))
            else:
                row.append(torch.randint(-5 if dtype != torch.uint8 else 0, 6, (s,), device='cuda', generator=g).to(dtype))
        ins.append(row)
    return ins


SIZES = [1, 17, 1000, 12345, (1 << 18) + 3]


@pytest.mark.parametrize("n", [2, 4, 8])
@pytest.mark.parametrize("variant", [ONESHOT, TWOSHOT])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_sum_float(n, variant, dtype):
    ins = _make(n, SIZES, dtype)
    outs = [[torch.empty_like(x) for x in row] for row in ins]
    sim_allreduce(ins, outs, dtype, dtype, SUM, variant, ctas=8, post=1.0 / n)
    for i in range(len(SIZES)):
        ref = torch.stack([ins[r][i].float() for r in range(n)]).sum(0) / n
        tol = 1e-5 if dtype == torch.float32 else 2e-2
        for r in range(n):
            torch.testing.assert_close(outs[r][i].float(), ref, rtol=tol, atol=tol)


@pytest.mark.parametrize("n", [2, 8])
@pytest.mark.parametrize("variant", [ONESHOT, TWOSHOT])
@pytest.mark.parametrize("dtype", [torch.int32, torch.int64, torch.uint8, torch.int8, torch.float64])
def test_sum_other_dtypes(n, variant, dtype):
    ins = _make(n, [5, 4099, 70001], dtype)
    outs = [[torch.empty_like(x) for x in row] for row in ins]
    sim_allreduce(ins, outs, dtype, dtype, SUM, variant, ctas=4)
    for i in range(3):
        ref = torch.stack([ins[r][i].to(torch.float64 if dtype == torch.float64 else torch.int64) for r in range(n)]).sum(0).to(dtype)
        for r in range(n):
            assert torch.equal(outs[r][i], ref) if dtype != torch.float64 else torch.allclose(outs[r][i], ref)


@pytest.mark.parametrize("op", [MIN, MAX, PROD])
@pytest.mark.parametrize("variant", [ONESHOT, TWOSHOT])
def test_min_max_product(op, variant):
    n = 4
    ins = _make(n, [33, 5000], torch.float32)
    outs = [[torch.empty_like(x) for x in row] for row in ins]
    sim_allreduce(ins, outs, torch.float32, torch.float32, op, variant, ctas=4)
    for i in range(2):
        st = torch.stack([ins[r][i] for r in range(n)])
        ref = st.min(0).values if op == MIN else st.max(0).values if op == MAX else st.prod(0)
        for r in range(n):
            torch.testing.assert_close(outs[r][i], ref, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("wire", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("variant", [ONESHOT, TWOSHOT])
def test_wire_compression_fused_cast(wire, variant):
    """fp32 gradients, 16-bit on the wire, fp32 accumulation: cast fused into pack/unpack."""
    n = 8
    ins = _make(n, [1000, 100003], torch.float32)
    outs = [[torch.empty_like(x) for x in row] for row in ins]
    sim_allreduce(ins, outs, torch.float32, wire, SUM, variant, ctas=8, pre=0.5, post=2.0 / n)
    for i in range(2):
        ref = torch.stack([(ins[r][i] * 0.5).to(wire).float() for r in range(n)]).sum(0) * (2.0 / n)
        for r in range(n):
            torch.testing.assert_close(outs[r][i], ref, rtol=2e-2, atol=2e-2)


def test_inplace_and_unaligned_views():
    """In-place (out == in) on tensors that are unaligned slices of a larger buffer (scalar path)."""
    n = 4
    bases = [torch.randn(50000, device='cuda') for _ in range(n)]
    ins = [[b[1:1 + 777], b[1001:1001 + 40001]] for b in bases]
    ref = [torch.stack([ins[r][i].clone() for r in range(n)]).sum(0) for i in range(2)]
    sim_allreduce(ins, ins, torch.float32, torch.float32, SUM, TWOSHOT, ctas=8)
    for i in range(2):
        for r in range(n):
            torch.testing.assert_close(ins[r][i], ref[i], rtol=1e-5, atol=1e-5)


def test_many_small_tensors_and_repeats():
    """A fused response like a real gradient set: hundreds of tensors, tiny to large; repeated (epoch reuse, ping-pong)."""
    n = 8
    sizes = [64, 256, 2048, 1, 3, 512 * 512, 1000, 7] * 20
    ins = _make(n, sizes, torch.float32)
    outs = [[torch.empty_like(x) for x in row] for row in ins]
    for variant in (ONESHOT, TWOSHOT):
        sim_allreduce(ins, outs, torch.float32, torch.float32, SUM, variant, ctas=16, repeats=5)
        for i in (0, 3, 5, len(sizes) - 1):
            ref = torch.stack([ins[r][i] for r in range(n)]).sum(0)
            for r in (0, n - 1):
                torch.testing.assert_close(outs[r][i], ref, rtol=1e-5, atol=1e-5)


def test_sim_allgather_exchange():
    lib = _lib()
    n, nbytes = 8, 1 << 20
    ins = [torch.randint(0, 255, (nbytes,), device='cuda', dtype=torch.uint8) for _ in range(n)]
    outs = [torch.empty(n * nbytes, device='cuda', dtype=torch.uint8) for _ in range(n)]
    ip = (ctypes.c_uint64 * n)(*[x.data_ptr() for x in ins])
    op_ = (ctypes.c_uint64 * n)(*[x.data_ptr() for x in outs])
    assert lib.hvd_sim_allgather(n, 0, nbytes, ip, op_, 8) == 0
    ref = torch.cat(ins)
    for r in range(n):
        assert torch.equal(outs[r], ref)


def test_sim_allgather_exchange_tma_variant():
    """The cp.async.bulk (UBLKCP) variant of the exchange kernel: ragged sizes (16 B-aligned bulk part + byte tail) and an
    unaligned destination (falls back to the vector path inside the same kernel).  Runs in a subprocess because the
    variant is selected once per process (HVD_EXCHANGE_TMA)."""
    import os, subprocess, sys, textwrap
    code = textwrap.dedent('''
        import ctypes, torch
        from horovod_b200.common.basics import load_library
        lib = load_library()
        lib.hvd_sim_allgather.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.POINTER(ctypes.c_uint64),
                                          ctypes.POINTER(ctypes.c_uint64), ctypes.c_int]
        for n, nbytes, shift in ((8, 1 << 20, 0), (4, (1 << 18) + 13, 0), (2, 100000, 3), (2, 7, 0)):
            ins = [torch.randint(0, 255, (nbytes,), device='cuda', dtype=torch.uint8) for _ in range(n)]
            bufs = [torch.zeros(n * nbytes + 64, device='cuda', dtype=torch.uint8) for _ in range(n)]
            outs = [b[shift:shift + n * nbytes] for b in bufs]
            ip = (ctypes.c_uint64 * n)(*[x.data_ptr() for x in ins])
            op_ = (ctypes.c_uint64 * n)(*[x.data_ptr() for x in outs])
            for rep in range(3):
                assert lib.hvd_sim_allgather(n, 0, nbytes, ip, op_, 8) == 0
            ref = torch.cat(ins)
            for r in range(n):
                assert torch.equal(outs[r], ref), (n, nbytes, shift, r)
        print('TMA EXCHANGE OK')
    ''')
    from conftest import REPO
    p = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, HVD_EXCHANGE_TMA='1', PYTHONPATH=REPO),
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=300)
    assert p.returncode == 0 and 'TMA EXCHANGE OK' in p.stdout.decode(), p.stdout.decode()[-3000:]


@pytest.mark.parametrize("slots", ["2", "16"])
def test_pipelined_allreduce_variant_in_simulation(slots):
    """kPipelined (role-specialised CTAs, chunk ring in the symmetric buffer, packed / reduced / unpack_done counters) with
    the P2P reduce stage on 2 / 4 / 8 simulated ranks; 64 KiB chunks and a 2-slot ring force many ring wrap-arounds."""
    import os, subprocess, sys, textwrap
    code = textwrap.dedent('''
        import torch
        from horovod_b200.ops import sim
        PIPELINED = 3
        for n in (2, 4, 8):
            for dtype, tol in ((torch.float32, 1e-5), (torch.bfloat16, 2e-2)):
                sizes = [1, 100003, 17, 262144 + 5, 4096]
                g = torch.Generator(device='cuda').manual_seed(n)
                ins = [[torch.randn(s, device='cuda', generator=g).to(dtype) for s in sizes] for _ in range(n)]
                outs = [[torch.empty_like(t) for t in row] for row in ins]
                for rep in range(3):  # the chunk counters keep running across launches
                    sim.allreduce(ins, outs, op=sim.SUM, variant=PIPELINED, ctas=16, prescale=0.5, postscale=2.0 / n)
                    for i in range(len(sizes)):
                        ref = torch.stack([ins[r][i].float() * 0.5 for r in range(n)]).sum(0) * (2.0 / n)
                        for r in range(n):
                            torch.testing.assert_close(outs[r][i].float(), ref, rtol=tol, atol=tol)
            big = [[torch.ones(3 << 20, device='cuda')] for _ in range(n)]   # 12 MiB: ~190 chunks
            sim.allreduce(big, big, op=sim.SUM, variant=PIPELINED, ctas=32)
            assert all(float(b[0][0]) == n and float(b[0][-1]) == n and float(b[0].min()) == n for b in big)
        print('PIPELINED OK')
    ''')
    from conftest import REPO
    p = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, HVD_PIPE_SLOTS=slots, HVD_PIPE_CHUNK_BYTES='65536',
                                                              HVD_KERNEL_TIMEOUT_SECONDS='20', PYTHONPATH=REPO),
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=600)
    assert p.returncode == 0 and 'PIPELINED OK' in p.stdout.decode(), p.stdout.decode()[-3000:]


def test_pack_reduce_bandwidth_smoke():
    """Not a benchmark: just checks a 64 MiB fused buffer moves at a sane rate on one GPU (all 'peers' are local HBM)."""
    n = 2
    ins = _make(n, [16 << 20], torch.float32)
    outs = [[torch.empty_like(x) for x in row] for row in ins]
    sim_allreduce(ins, outs, torch.float32, torch.float32, SUM, TWOSHOT, ctas=32, repeats=2)
    ms = sim_allreduce(ins, outs, torch.float32, torch.float32, SUM, TWOSHOT, ctas=32, repeats=5) / 5
    assert ms < 50.0, ms


def _adasum_ref(vecs):
    """fp64 oracle: pairwise adaptive sum in the VHDD tree order (reference ops/adasum/adasum.h:344-435)."""
    if len(vecs) == 1:
        return vecs[0]
    h = len(vecs) // 2
    a, b = _adasum_ref(vecs[:h]), _adasum_ref(vecs[h:])
    dot, na, nb = (a * b).sum(), (a * a).sum(), (b * b).sum()
    ac = 1 - dot / (2 * na) if na > 0 else 1.0
    bc = 1 - dot / (2 * nb) if nb > 0 else 1.0
    return ac * a + bc * b


@pytest.mark.parametrize("n", [2, 4, 8])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_adasum_kernels_vs_fp64_oracle(n, dtype):
    lib = _lib()
    lib.hvd_sim_adasum.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int64),
                                   ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64), ctypes.c_int, ctypes.c_int,
                                   ctypes.c_double, ctypes.c_double]
    sizes = [5, 1000, 33333, 64]
    ins = _make(n, sizes, dtype, seed=3)
    # tensor 3: identical on every rank (parallel vectors -> result equals the input)
    for r in range(n):
        ins[r][3].copy_(ins[0][3])
    outs = [[torch.empty_like(x) for x in row] for row in ins]
    t = len(sizes)
    counts = (ctypes.c_int64 * t)(*sizes)
    ip = (ctypes.c_uint64 * (n * t))(*[x.data_ptr() for r in ins for x in r])
    op_ = (ctypes.c_uint64 * (n * t))(*[x.data_ptr() for r in outs for x in r])
    rc = lib.hvd_sim_adasum(n, 0, t, counts, ip, op_, DT[dtype], 8, 1.0, 1.0)
    assert rc == 0, rc
    tol = 1e-4 if dtype == torch.float32 else 3e-2
    for i in range(t):
        ref = _adasum_ref([ins[r][i].double() for r in range(n)])
        for r in range(n):
            torch.testing.assert_close(outs[r][i].double(), ref, rtol=tol, atol=tol)
    torch.testing.assert_close(outs[0][3].double(), ins[0][3].double(), rtol=tol, atol=tol)
