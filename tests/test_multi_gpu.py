"""Multi-GPU entry points of the C-ABI (include/pffft/pffft_b200.h, SURVEY 8e): single process, one plan per GPU, ONE
broadcast of the plan tables (NCCL), batch sharded in contiguous ranges, no other inter-GPU traffic.  Runs on whatever the
box has: the 1-GPU case exercises the same code with a one-element communicator; the >= 2-GPU cases skip otherwise."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, uniform

pytestmark = pytest.mark.gpu


def _ngpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("want", [1, 0])
def test_host_batch_sharded_over_the_gpus_vs_reference(pf, ref, R, want):
    N, batch = 1024, 4096 + 3
    rng = np.random.default_rng(want)
    x = uniform(rng, batch * 2 * N).reshape(batch, 2 * N)
    m = pf.Multi(N, pf.PFFFT_COMPLEX, want)
    assert m.ngpus == (1 if want == 1 else _ngpus())
    assert m.backend in (("single",) if m.ngpus == 1 else ("nccl", "memcpy_peer"))
    y = np.empty_like(x); z = np.empty_like(x)
    m.transform_batch(x, y, batch, 0, 1)
    m.transform_batch(y, z, batch, 1, 1)
    idx = sorted({0, 1, batch // m.ngpus - 1, min(batch // m.ngpus, batch - 1), batch // 2, batch - 1})   # both sides of a shard boundary
    w = ref.transform_batch(N, 1, x[idx], 0, True)
    assert max(R.relmax(y[i], w[j]) for j, i in enumerate(idx)) <= 1e-5
    assert R.relmax(z, x * N) <= 1e-5
    m.close()


def test_device_resident_shards_and_bit_identical_gpus(pf, ref, R):
    import torch
    N = 4096
    m = pf.Multi(N, pf.PFFFT_REAL, 0)
    G = m.ngpus
    xs, ys, nb = [], [], []
    gen = torch.Generator(device="cuda:0"); gen.manual_seed(N)
    base = torch.rand((64, N), generator=gen, device="cuda:0") * 2 - 1
    for g in range(G):
        xs.append(base.to("cuda:%d" % g))
        ys.append(torch.empty_like(xs[-1]))
        nb.append(64)
    m.transform_shards(xs, ys, nb, 0, 1)
    m.synchronize()
    y0 = ys[0].cpu().numpy()
    for g in range(1, G):
        assert np.array_equal(ys[g].cpu().numpy(), y0), "GPU %d differs from GPU 0" % g     # same tables, same kernels
    w = ref.transform_batch(N, 0, base[:3].cpu().numpy(), 0, True)
    assert max(R.relmax(y0[i], w[i]) for i in range(3)) <= 1e-5
    m.close()


def test_rank_style_broadcast_entry_points(pf):
    """one-process-per-GPU flavour: id creation works wherever NCCL loads; a 1-rank broadcast is a no-op"""
    import ctypes as C
    buf = (C.c_char * 128)()
    rc = pf.lib.pffftb_nccl_unique_id(buf)
    with pf.Setup(1024, 1) as s:
        assert pf.lib.pffftb_setup_broadcast_tables(s.handle, buf, 0, 1) == 0
        if rc == 0 and _ngpus() >= 1:
            # a real communicator of size 1: ncclCommInitRank + ncclBroadcast on this GPU
            os.environ["PFFFT_B200_FORCE_NCCL_1RANK"] = "1"
            try:
                assert pf.lib.pffftb_setup_broadcast_tables(s.handle, buf, 0, 1) == 0, pf.last_error()
            finally:
                del os.environ["PFFFT_B200_FORCE_NCCL_1RANK"]
        x = np.zeros(2048, np.float32); x[0] = 1
        y = s.transform_batch(x, 0, True)
        assert np.allclose(y[0::2], 1) and np.allclose(y[1::2], 0)          # tables intact after the broadcast


def test_c_example_runs_on_all_gpus(tmp_path):
    exe = str(tmp_path / "multi_gpu_c2c")
    r = subprocess.run(["gcc", "-std=c99", "-I" + os.path.join(ROOT, "include", "pffft"), os.path.join(ROOT, "examples", "multi_gpu_c2c.c"),
                        "-L" + os.path.join(ROOT, "pffft_b200"), "-lpffft_b200", "-Wl,-rpath," + os.path.join(ROOT, "pffft_b200"), "-lm", "-o", exe],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    r = subprocess.run([exe, "0", "13"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
    assert r.returncode == 0, r.stdout
    assert "bit-identical: yes" in r.stdout
