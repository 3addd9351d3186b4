"""Tiled Stockham pipeline on hardware (pffft_b200/csrc/ts_kernels.cuh): oracle parity for every stage kind, batches that
recycle the L2-resident ring slots many times, in-place calls, concurrent streams on one plan, float and double."""
import numpy as np
import pytest

from conftest import uniform

pytestmark = pytest.mark.gpu
TOL = {np.dtype(np.float32): 1e-5, np.dtype(np.float64): 1e-12}


def _numpy_forward(x, N, tr):
    x = x.astype(np.float64)
    if tr == 1:
        W = np.fft.fft(x[0::2] + 1j * x[1::2])
        return np.stack([W.real, W.imag], -1).ravel()
    X = np.fft.rfft(x)
    w = np.stack([X.real[:-1], X.imag[:-1]], -1).ravel()
    w[1] = X.real[-1]
    return w


@pytest.fixture()
def ts_on(monkeypatch):
    monkeypatch.setenv("PFFFT_B200_TS", "1")


# cores: 2 passes (8192 .. 65536, mixed radices), 3 passes, closing small radix (384000 = 240 x 160 x 10)
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("tr", [1, 0])
@pytest.mark.parametrize("core", [8192, 12288, 16384, 20480, 36864, 61440, 65536, 131072, 196608, 384000])
def test_every_mode_vs_reference(pf, ref, R, ts_on, core, tr, dtype):
    import torch
    dtype = np.dtype(dtype)
    N = core if tr == 1 else 2 * core
    if pf.pffft_is_valid_size(N, tr) != 1:
        pytest.skip("size")
    rng = np.random.default_rng(core * 2 + tr)
    per = 2 * core
    batch = 3
    x = uniform(rng, batch * per, dtype).reshape(batch, per)
    pow2 = (N & (N - 1)) == 0
    tol_ref = TOL[dtype] if (pow2 or dtype == np.float32) else 5e-7      # reference double path: float radix-3/5 constants
    with pf.Setup(N, tr, dtype) as s:
        assert s.kernel.startswith(("ts_", "tsw_")), s.kernel
        xd = torch.from_numpy(x).cuda()
        fo = s.transform_batch(xd, 0, True)
        fz = s.transform_batch(xd, 0, False)
        bo = s.transform_batch(fo, 1, True)
        bz = s.transform_batch(fz, 1, False)
        ro = s.zreorder_batch(fz, 0)
        inpl = xd.clone(); s.transform_batch(inpl, 0, True, out=inpl)
        torch.cuda.synchronize()
        assert torch.equal(ro, fo), "ordered != zreorder(unordered)"
        assert torch.equal(inpl, fo), "in place != out of place"
        fo_, fz_, bo_, bz_ = [t.cpu().numpy() for t in (fo, fz, bo, bz)]
    wo = ref.transform_batch(N, tr, x, 0, True, dtype)
    wz = ref.transform_batch(N, tr, x, 0, False, dtype)
    for b in range(batch):
        assert R.relmax(fo_[b], _numpy_forward(x[b], N, tr)) <= TOL[dtype], (s.kernel, b)
        assert R.relmax(fo_[b], wo[b]) <= tol_ref and R.relmax(fz_[b], wz[b]) <= tol_ref
        assert R.relmax(bo_[b], x[b] * N) <= 10 * TOL[dtype] and R.relmax(bz_[b], x[b] * N) <= 10 * TOL[dtype]


@pytest.mark.parametrize("tr,core,batch", [(1, 16384, 3000), (0, 16384, 1500), (1, 65536, 700), (1, 8192, 5000), (1, 1 << 20, 40)])
def test_ring_slots_recycled_many_times(pf, ref, R, ts_on, tr, core, batch):
    """batches far larger than the ring (2*lag+1 transforms): every slot is overwritten many times while neighbours are still
    being consumed.  Sampled transforms against the reference, every transform by round trip."""
    import torch
    N = core if tr == 1 else 2 * core
    per = 2 * core
    g = torch.Generator(device="cuda"); g.manual_seed(core + tr)
    x = torch.rand((batch, per), generator=g, device="cuda") * 2 - 1
    with pf.Setup(N, tr) as s:
        y = s.transform_batch(x, 0, True)
        z = s.transform_batch(y, 1, True)
        torch.cuda.synchronize()
        err = float(((z / N - x) ** 2).sum(dim=1).max().item())
        assert err <= N * 1e-7, (s.kernel, err)
        idx = np.unique(np.concatenate([np.arange(8), np.arange(batch - 8, batch), np.random.default_rng(1).integers(0, batch, 48)]))
        ti = torch.from_numpy(idx).cuda()
        xs, ys = x[ti].cpu().numpy(), y[ti].cpu().numpy()
    want = ref.transform_batch(N, tr, xs, 0, True)
    assert max(R.relmax(ys[i], want[i]) for i in range(idx.size)) <= 1e-5


def test_two_streams_share_one_plan(pf, ref, R, ts_on):
    """the rings and counters of a plan serve one launch at a time: calls from two streams are ordered by the plan's event"""
    import torch
    N = 32768
    g = torch.Generator(device="cuda"); g.manual_seed(N)
    x1 = torch.rand((64, 2 * N), generator=g, device="cuda") * 2 - 1
    x2 = torch.rand((64, 2 * N), generator=g, device="cuda") * 2 - 1
    y1 = torch.empty_like(x1); y2 = torch.empty_like(x2)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    with pf.Setup(N, 1) as s:
        for _ in range(4):
            pf.lib.pffftb_set_stream(s.handle, s1.cuda_stream)
            pf.pffftb_transform_batch(s.handle, x1, y1, 64, 0, 1)
            pf.lib.pffftb_set_stream(s.handle, s2.cuda_stream)
            pf.pffftb_transform_batch(s.handle, x2, y2, 64, 0, 1)
        torch.cuda.synchronize()
        pf.lib.pffftb_set_stream(s.handle, None)
    for x, y in ((x1, y1), (x2, y2)):
        w = ref.transform_batch(N, 1, x[[0, 63]].cpu().numpy(), 0, True)
        g = y[[0, 63]].cpu().numpy()
        assert max(R.relmax(g[i], w[i]) for i in range(2)) <= 1e-5


# ---- opt-in variants of the pipeline (round 2b): warp-sized work items (tsw_kernels.cuh) and the cp.async input prefetch
@pytest.mark.parametrize("variant", ["tsw", "prefetch"])
@pytest.mark.parametrize("tr,core,batch", [(1, 16384, 300), (1, 65536, 40), (0, 16384, 60), (1, 131072, 6), (1, 8192, 500)])
def test_opt_in_pipeline_variants(pf, ref, R, ts_on, monkeypatch, variant, tr, core, batch):
    """same plans, other kernels: results against the reference on sampled transforms, every transform by round trip"""
    import torch
    if variant == "tsw":
        monkeypatch.setenv("PFFFT_B200_TSW", "1")
    else:
        monkeypatch.setenv("PFFFT_B200_TS_MINB", "3"); monkeypatch.setenv("PFFFT_B200_TS_PRE", "1")
    N = core if tr == 1 else 2 * core
    per = 2 * core
    g = torch.Generator(device="cuda"); g.manual_seed(core + tr + 11)
    x = torch.rand((batch, per), generator=g, device="cuda") * 2 - 1
    with pf.Setup(N, tr) as s:
        assert s.kernel.startswith("tsw_" if variant == "tsw" else "ts_"), s.kernel
        y = s.transform_batch(x, 0, True)
        yz = s.transform_batch(x, 0, False)
        z = s.transform_batch(y, 1, True)
        zz = s.transform_batch(yz, 1, False)
        torch.cuda.synchronize()
        assert float((z / N - x).abs().max()) <= N * 1e-7 and float((zz / N - x).abs().max()) <= N * 1e-7
        for b in (0, batch // 2, batch - 1):
            xb = x[b].cpu().numpy()
            assert R.relmax(y[b].cpu().numpy(), ref.transform(N, tr, xb, 0, True)) <= 1e-5, (s.kernel, b)
            assert R.relmax(yz[b].cpu().numpy(), ref.transform(N, tr, xb, 0, False)) <= 1e-5, (s.kernel, b)
