#!/usr/bin/env python
"""bench.py -- headline benchmark: batched 1-D FFTs/s at N=1024 complex fp32 (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One step = one pass of the hot path over one synthetic batch: `batch` forward transforms followed by
`batch` backward transforms (BASELINE configs[1] "N=1024 complex fp32 fwd+inv, batch=1M"; the reference's own
benchmark iteration is also fwd+bwd, benchmarks/bench_pffft.c:1008-1014).  Per-GPU batch is fixed
(weak scaling); ranks never communicate inside the timed region (one NCCL broadcast of the plan tables before it).

Prints ONE JSON line (rank 0).  Keys follow the driver contract; see DESIGN.md section "Measurement".
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N = 1024
BYTES_PER_FFT = 2 * N * 2 * 4          # 8 KiB read + 8 KiB written (SURVEY 8d: algorithmic bytes / transform)
# dram__bytes_read.sum + dram__bytes_write.sum of ONE `ncu --set full` capture of the forward kernel, per transform:
# (2.147577 + 2.097573) GB over a 262144-transform launch (profiles/r01_ncu_full_c1024.txt; re-captured in round 2 with the
# same result, profiles/r02_ncu_c1024.txt: 2.147574 + 2.098634 GB).
# STATIC: bench.py scales the committed capture to the units of its own launch and labels it so ("traffic_kind");
# it is evidence that traffic ~= algorithmic bytes, not a measurement of this run (ncu cannot run inside a timed bench).
NCU_DRAM_BYTES_PER_FFT = (2.147577e9 + 2.097573e9) / 262144
FLOPS_PER_FFT = 5 * N * 10             # 5 N log2 N (bench_pffft.c:1021)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=1 << 20, help="transforms per GPU per pass (default 2^20)")
    ap.add_argument("--e2e-batch", type=int, default=1 << 17, help="transforms per e2e step (host buffers)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target wall time of the cpu_baseline leg")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs (a fixed sample of rows) to DIR/forward.npy, DIR/backward.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_ROWS = 2048                       # 2 x 2048 transforms x 8 KiB = 32 MiB of outputs


def dump_outputs(d, y, z):
    """forward (y) and backward (z) outputs of the same seeded sample of rows, float32, one (rows, 2N) array each"""
    import torch
    os.makedirs(d, exist_ok=True)
    rows = np.sort(np.random.default_rng(0).choice(y.shape[0], min(y.shape[0], DUMP_ROWS), replace=False))
    idx = torch.from_numpy(rows).to(y.device)
    for name, t in (("forward", y), ("backward", z)):
        np.save(os.path.join(d, name + ".npy"), t.index_select(0, idx).cpu().numpy())


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        inside = [ln for ts, ln in self.lines if t0 is None or (t0 - 0.03 <= ts <= t1 + 0.03)]
        window = "timed region"
        if not inside:                       # sampler slower than the region: fall back to every sample of the run
            inside, window = [ln for _, ln in self.lines], "whole run (no sample landed inside the timed region)"
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "window": window}


# ------------------------------------------------------------------------------------------------ CPU legs
def host_llc_bytes():
    """total last-level cache of the host (sum over the distinct L3 instances sysfs lists), 0 when unknown"""
    seen, total = set(), 0
    base = "/sys/devices/system/cpu"
    try:
        for cpu in os.listdir(base):
            d = os.path.join(base, cpu, "cache", "index3")
            if not (cpu.startswith("cpu") and cpu[3:].isdigit() and os.path.isdir(d)):
                continue
            ident = open(os.path.join(d, "shared_cpu_list")).read().strip()
            if ident in seen:
                continue
            seen.add(ident)
            sz = open(os.path.join(d, "size")).read().strip()
            mult = {"K": 1 << 10, "M": 1 << 20, "G": 1 << 30}.get(sz[-1].upper(), 1)
            total += int(sz[:-1] if sz[-1].isalpha() else sz) * mult
    except Exception:
        return 0
    return total


def cpu_sample_transforms():
    """transforms per CPU pass: the working set (8 KiB in + 8 KiB out each) is >= 4x the host's total LLC so the
    reference streams from DRAM like the GPU streams from HBM (2^16 = 1 GiB at least, 2^19 = 8 GiB at most)"""
    llc = host_llc_bytes()
    n = 1 << 16
    while n * 2 * BYTES_PER_FFT // 2 < 4 * llc and n < (1 << 19):
        n <<= 1
    return n, llc


def cpu_reference_rate(seconds_target, fwd_inv=True):
    """FFTs/s of the reference's own CPU implementation (oracle/_ref, unmodified pffft built with
    -O3 -march=haswell) on all host cores, through oracle/libcpubench.so: threads share one PFFFT_Setup
    and each calls pffft_transform_ordered one vector at a time on its slice of a DRAM-resident batch."""
    from oracle import ref as R
    bench_so = os.path.join(ROOT, "oracle", "libcpubench.so")
    if not (R.have_ref() and os.path.exists(bench_so)):
        return None
    lib = C.CDLL(bench_so)
    lib.cpu_bench_transform.restype = C.c_double
    lib.cpu_bench_transform.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_long, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint]
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    path = R.REF_SO.encode()
    sample, llc = cpu_sample_transforms()              # >= 2^16 transforms (512 MiB in + 512 MiB out) and >= 4x LLC
    per_pass = 2 if fwd_inv else 1
    t1 = lib.cpu_bench_transform(path, N, 1, sample, cores, 1, 1 if fwd_inv else 0, 1, 1234)
    if t1 <= 0:
        return None
    iters = max(1, min(64, int(seconds_target / max(t1, 1e-3))))
    t = lib.cpu_bench_transform(path, N, 1, sample, cores, iters, 1 if fwd_inv else 0, 1, 1234)
    if t <= 0:
        return None
    rate = sample * per_pass * iters / t
    t_one = lib.cpu_bench_transform(path, N, 1, 1 << 13, 1, 4, 1 if fwd_inv else 0, 1, 1234)
    rate1 = (1 << 13) * per_pass * 4 / t_one if t_one > 0 else None
    return {"value": rate, "unit": "FFT/s", "cores": cores, "kind": "reference",
            "sample": "%d x N=1024 cplx fp32 %s (inverse in place on the just-written vector, as a per-vector caller would), "
                      "ordered, %d passes, %d threads sharing one PFFFT_Setup, uniform(-1,1); working set %.2f GiB = %.1fx host LLC (%.0f MiB)"
                      % (sample, "fwd+inv" if fwd_inv else "fwd", iters, cores, sample * BYTES_PER_FFT / 2**30,
                         (sample * BYTES_PER_FFT / llc) if llc else float("nan"), llc / 2**20),
            "single_thread_value": rate1, "seconds": t, "sample_transforms": sample, "host_llc_bytes": llc}


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path, all host threads (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    t0 = time.time()
    per_step = []
    total = max(1, args.steps)
    # each step = a bounded sample of the workload; whole run stays within a couple of minutes
    budget = min(8.0, 90.0 / (total + max(1, args.warmup)))
    for _ in range(max(1, args.warmup)):
        cpu_reference_rate(min(1.0, budget))
    res = None
    for _ in range(total):
        res = cpu_reference_rate(budget)
        if res is None:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libpffft_ref.so or oracle/libcpubench.so missing"}))
            return 0
        per_step.append(res["value"])
    value = float(np.median(per_step))
    sample = res["sample_transforms"]
    line = {
        "impl": "reference", "metric": "batched FFTs/sec at N=1024 cplx fp32 (fwd+inv)", "value": value, "unit": "FFT/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * (2 * sample) / value, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "C2: N=1024 complex fp32 fwd+inv, ordered; bounded sample of %d transforms per step on the host CPU (>= 4x LLC)" % sample},
        "cpu_baseline": {"value": value, "unit": "FFT/s", "cores": res["cores"], "kind": "reference", "sample": res["sample"]},
        "e2e": {"value": value, "unit": "FFT/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gbs_algorithmic": value * BYTES_PER_FFT / 1e9, "gflops": value * FLOPS_PER_FFT / 1e9,
        "wall_s": time.time() - t0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------ GPU arm
class _CudaMem:
    """exposes a raw device allocation to torch through __cuda_array_interface__ (for the NCCL table broadcast)"""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist
    import pffft_b200 as pf

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this benchmark has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    batch = args.batch
    setup = pf.Setup(N, pf.PFFFT_COMPLEX)
    # multi-GPU: rank 0's tables are THE tables (bit-identical plans everywhere): one NCCL broadcast over NVLink
    table_broadcast = "none (1 GPU)"
    if world > 1:
        # the library's own collective (multi.cu): rank 0 makes an NCCL id, torch.distributed only carries its 128 bytes,
        # ncclCommInitRank + ncclBroadcast(root 0) of the tables run inside libpffft_b200.so
        idbuf = torch.zeros(128, dtype=torch.uint8)
        ok = torch.ones(1, device="cuda", dtype=torch.int32)
        if rank == 0:
            raw = (C.c_char * 128)()
            ok[0] = 1 if pf.lib.pffftb_nccl_unique_id(raw) == 0 else 0
            idbuf = torch.frombuffer(bytearray(raw.raw), dtype=torch.uint8).clone()
        idd = idbuf.cuda()
        dist.broadcast(idd, src=0)
        dist.broadcast(ok, src=0)
        done = torch.zeros(1, device="cuda", dtype=torch.int32)
        if int(ok.item()) == 1 and os.environ.get("PFFFT_B200_BENCH_TORCH_BCAST") is None:
            raw = (C.c_char * 128).from_buffer_copy(bytes(idd.cpu().numpy().tobytes()))
            done[0] = 1 if pf.lib.pffftb_setup_broadcast_tables(setup.handle, raw, rank, world) == 0 else 0
        dist.all_reduce(done, op=dist.ReduceOp.MIN)
        if int(done.item()) == 1:
            table_broadcast = "libpffft_b200 (ncclCommInitRank + ncclBroadcast root 0)"
        else:                                  # NCCL not loadable from the library on this box: same broadcast through torch
            tptr, tbytes = setup.tables()
            tables = torch.as_tensor(_CudaMem(tptr, tbytes), device="cuda")
            dist.broadcast(tables, src=0)
            table_broadcast = "torch.distributed (library NCCL unavailable: %s)" % pf.last_error()
        torch.cuda.synchronize()

    # synthetic batch, generated on the device: uniform(-1,1), seed 1234 + rank (SURVEY 8d)
    g = torch.Generator(device="cuda"); g.manual_seed(1234 + rank)
    x = torch.rand((batch, 2 * N), generator=g, device="cuda", dtype=torch.float32) * 2 - 1
    y = torch.empty_like(x)
    z = torch.empty_like(x)

    def step():
        pf.pffftb_transform_batch(setup.handle, x, y, batch, pf.PFFFT_FORWARD, 1)
        pf.pffftb_transform_batch(setup.handle, y, z, batch, pf.PFFFT_BACKWARD, 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(3, args.warmup)):
        step()
    barrier()
    # sanity inside the bench: the timed path computes transforms (round trip == N*x on a slice)
    err = ((z[:64] / N - x[:64]) ** 2).sum(dim=1).max().item()
    assert err <= N * 1e-7, "bench self-check failed: round trip error %g" % err

    launches0 = pf.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fwd_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    wall0 = time.time()
    ev0.record()
    for i in range(args.steps):
        fwd_ev[i][0].record()
        pf.pffftb_transform_batch(setup.handle, x, y, batch, pf.PFFFT_FORWARD, 1)
        fwd_ev[i][1].record()
        pf.pffftb_transform_batch(setup.handle, y, z, batch, pf.PFFFT_BACKWARD, 1)
    ev1.record()
    barrier()
    wall1 = time.time()
    launches = pf.launch_count() - launches0
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, y, z)
    ms = ev0.elapsed_time(ev1)
    fwd_ms = float(np.mean([a.elapsed_time(b) for a, b in fwd_ev]))
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = world * batch * 2 * args.steps / (ms * 1e-3)

    # ---- e2e: same metric through the C-ABI with HOST buffers (pinned, pffft_aligned_malloc), copies inside the timed region
    eb = args.e2e_batch
    nbytes = eb * 2 * N * 4
    hin = pf.lib.pffft_aligned_malloc(nbytes); hmid = pf.lib.pffft_aligned_malloc(nbytes); hout = pf.lib.pffft_aligned_malloc(nbytes)
    a_in = np.ctypeslib.as_array(C.cast(hin, C.POINTER(C.c_float)), shape=(eb * 2 * N,))
    a_mid = np.ctypeslib.as_array(C.cast(hmid, C.POINTER(C.c_float)), shape=(eb * 2 * N,))
    a_out = np.ctypeslib.as_array(C.cast(hout, C.POINTER(C.c_float)), shape=(eb * 2 * N,))
    rng = np.random.default_rng(1234 + rank)
    a_in[:] = rng.random(eb * 2 * N, dtype=np.float32) * 2 - 1

    def e2e_step():
        pf.pffftb_transform_batch(setup.handle, a_in, a_mid, eb, pf.PFFFT_FORWARD, 1)
        pf.pffftb_transform_batch(setup.handle, a_mid, a_out, eb, pf.PFFFT_BACKWARD, 1)

    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_err = float(np.max(np.abs(a_out[:2 * N * 8] / N - a_in[:2 * N * 8])))
    e2e_value = world * eb * 2 * e2e_steps / e2e_s
    for p in (hin, hmid, hout):
        pf.lib.pffft_aligned_free(p)

    if rank == 0:
        peak, peak_src = peaks()
        fwd_gbs = batch * BYTES_PER_FFT / (fwd_ms * 1e-3) / 1e9
        line = {
            "metric": "batched FFTs/sec at N=1024 cplx fp32 (fwd+inv)", "value": value, "unit": "FFT/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "C2: N=1024 complex fp32 fwd+inv (pffft_transform_ordered semantics), batch=%d per GPU" % batch,
                       "global_batch": world * batch, "parallelism": "batch-sharded x%d, no data-path collective" % world,
                       "l2": "inputs larger than L2 (%.1f GiB per pass, fwd x->y, inv y->z)" % (batch * 8192 / 2**30),
                       "kernel": setup.kernel, "table_broadcast": table_broadcast},
            "gflops": value * FLOPS_PER_FFT / 1e9,
            "gbs_algorithmic": value * BYTES_PER_FFT / 1e9,
            "roofline": {"bound": "hbm", "achieved": fwd_gbs, "peak": peak, "unit": "GB/s", "frac": fwd_gbs / peak,
                         "traffic": NCU_DRAM_BYTES_PER_FFT * batch if "ldg" in setup.kernel else None,
                         "traffic_kind": "static",
                         "traffic_source": "profiles/r02_ncu_c1024.txt = profiles/r01_ncu_full_c1024.txt (ncu --set full of this unchanged kernel, 2.1476 + 2.0986 GB per 262144 transforms in both rounds: per-transform DRAM bytes x this launch's transforms; not measured in this run)",
                         "kernel": setup.kernel + " (forward launch, %d transforms)" % batch,
                         "algorithmic_bytes_per_launch": batch * BYTES_PER_FFT, "ms_per_launch": fwd_ms,
                         "peak_source": peak_src,
                         "whole_step_frac": (value / world) * BYTES_PER_FFT / 1e9 / peak},
            "e2e": {"value": e2e_value, "unit": "FFT/s", "h2d_bytes_per_step": 2 * nbytes, "d2h_bytes_per_step": 2 * nbytes,
                    "batch_per_step": eb, "steps": e2e_steps, "max_abs_roundtrip_err": e2e_err,
                    "api": "pffftb_transform_batch with pinned host buffers from pffft_aligned_malloc (3-stream chunked pipeline)"},
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if not args.no_cpu and world == 1:
            cb = cpu_reference_rate(args.cpu_seconds)
            line["cpu_baseline"] = cb if cb else {"value": None, "unit": "FFT/s", "cores": 0, "kind": "reference",
                                                   "sample": "unavailable: oracle/_ref or libcpubench.so missing"}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
