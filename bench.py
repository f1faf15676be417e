#!/usr/bin/env python
"""Benchmark of the hot path: samples/sec of with_logabsdet_jacobian through an 8-layer Planar flow, D=128,
N=2^20 Float32 per GPU (BASELINE.json configs[1]) -- plus, in the same run and under the same clock, every other
BASELINE config as a sub-record (`configs`): C3 (6 x Radial, forward + inverse), C4 (RQS K=8, N=2^19 TOTAL sharded over
the ranks), C5 (RealNVP logpdf, N=2^22 TOTAL sharded, ending in the path's ONE collective, b2b_allreduce_sum_f64,
INSIDE the timed region), each with an in-run oracle check on a 1024-column sample.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input.  Prints ONE JSON line (rank 0).
  value      whole-job samples/s with the batch resident in HBM (CUDA events, max over ranks)
  e2e        same metric through the public API with HOST (pinned, NUMA-local) buffers: H2D + kernels + D2H per step
  roofline   dominant kernel (the fused chain kernel): algorithmic bytes per launch / measured launch time
  cpu_baseline  the C restatement of the reference CPU path (oracle/b2b_oracle.c) on the host cores
  configs    sub-records of the other BASELINE configs (same timing rules: CUDA events, max over ranks, >= 3 warm-ups)
--dump-outputs DIR also writes what the last timed headline step returned (see dump_outputs), so that two builds can be
compared output for output on the same seeded inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

D, NCOLS, NLAYERS = 128, 1 << 20, 8
METRIC = "samples/sec: with_logabsdet_jacobian through 8-layer Planar flow, D=128"
WORKLOAD = "Composed(8x PlanarLayer), D=128, N=2^20 per GPU, Float32 (BASELINE configs[1])"
CPU_SAMPLE_COLS = 1 << 18  # per step of the --impl reference arm
DUMP_COLS = 1 << 16  # columns of y that --dump-outputs writes: D x 2^16 Float32 = 32 MiB (+ 4 MiB of logjac)
f32 = np.float32


def planar_params(seed_base=100):
    """SURVEY §8(d) C2: per layer w,u ~ N(0,1)/sqrt(D), b ~ N(0,1), PCG64 seeds 100+layer."""
    out = []
    for l in range(NLAYERS):
        rng = np.random.Generator(np.random.PCG64(seed_base + l))
        w = (rng.standard_normal(D) / np.sqrt(D)).astype(np.float32)
        u = (rng.standard_normal(D) / np.sqrt(D)).astype(np.float32)
        b = rng.standard_normal(1).astype(np.float32)
        out.append((w, u, b))
    return out


def dump_outputs(out_dir, y, lj):
    """What a caller of the timed path receives from with_logabsdet_jacobian(flow, x), as Float32 .npy files:
    DIR/logjac.npy, all N values, and DIR/y.npy, the (D, DUMP_COLS) columns of y at the sorted indices
    np.sort(default_rng(0).choice(N, DUMP_COLS, replace=False)) -- y itself is 512 MiB."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    cols = torch.as_tensor(np.sort(np.random.default_rng(0).choice(NCOLS, DUMP_COLS, replace=False)), device=y.device)
    np.save(os.path.join(out_dir, "y.npy"), np.ascontiguousarray(y[:, cols].cpu().numpy(), dtype=f32))
    np.save(os.path.join(out_dir, "logjac.npy"), np.ascontiguousarray(lj.cpu().numpy(), dtype=f32))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def pick_threads(layers):
    """Host threads for the CPU restatement: the fastest of {all cores the process may use, 64, 32, 16, 8} on a small
    probe (with fresh outputs per layer the pass is page-fault / bandwidth bound, so more threads is not always faster)."""
    from oracle import oracle_c as C

    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = C.num_procs()
    avail = max(1, min(avail, C.num_procs()))
    rng = np.random.Generator(np.random.PCG64(2))
    probe = np.asfortranarray(rng.standard_normal((D, 1 << 15), dtype=np.float32))
    best_t, best = avail, float("inf")
    for t in sorted({avail, *[c for c in (64, 32, 16, 8) if c <= avail]}, reverse=True):
        C.planar_chain_fwd(layers, probe, nthreads=t)
        t0 = time.perf_counter()
        C.planar_chain_fwd(layers, probe, nthreads=t)
        dt = time.perf_counter() - t0
        if dt < best:
            best_t, best = t, dt
    return best_t


def cpu_baseline(nthreads=None, repeats=5, cols=NCOLS):
    """Times the C restatement of the reference CPU path on a bounded sample of the same workload."""
    from oracle import oracle_c as C

    layers = planar_params()
    nthreads = nthreads or pick_threads(layers)
    rng = np.random.Generator(np.random.PCG64(1))
    x = np.asfortranarray(rng.standard_normal((D, cols), dtype=np.float32))
    C.planar_chain_fwd(layers, x[:, : 1 << 12], nthreads=nthreads)  # warm-up (library load, threads)
    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        C.planar_chain_fwd(layers, x, nthreads=nthreads)
        best = min(best, time.perf_counter() - t0)
    return {
        "value": cols / best,
        "unit": "samples/s",
        "cores": int(nthreads),
        "kind": "port",
        "sample": f"{cols} of {NCOLS} columns, best of {repeats} passes; C/OpenMP restatement of the reference "
                  f"CPU pass structure (gemv pass + broadcast pass per layer), not the Julia package; thread count "
                  f"picked by a probe",
        "seconds_per_pass": best,
    }


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, reasons, mx = [], set(), None
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))
        return out


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  The reference is Julia and no
    Julia toolchain exists in this image, so this arm times the C restatement of its CPU path (oracle port)
    with all host threads.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle_c as C

    layers = planar_params()
    nthreads = pick_threads(layers)
    cols = CPU_SAMPLE_COLS
    rng = np.random.Generator(np.random.PCG64(1))
    x = np.asfortranarray(rng.standard_normal((D, cols), dtype=np.float32))
    for _ in range(max(args.warmup, 1)):
        C.planar_chain_fwd(layers, x[:, : 1 << 14], nthreads=nthreads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        C.planar_chain_fwd(layers, x, nthreads=nthreads)
    dt = time.perf_counter() - t0
    val = cols * args.steps / dt
    sample = f"{cols} of {NCOLS} columns per step; C/OpenMP restatement of the reference CPU path (oracle port)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample},
        "cpu_baseline": {"value": val, "unit": "samples/s", "cores": int(nthreads), "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ----------------------------------------------------------------------------------------------------------------------
# sub-records of the other BASELINE configs
# ----------------------------------------------------------------------------------------------------------------------
def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(a), np.linalg.norm(b), 1e-30))


def run_configs(B, torch, dist, world, rank, comm, peak, iters, warmup):
    """C3 / C4 / C5 under the same clock: device-resident CUDA-event timing (max over ranks), samples/s of the WHOLE job,
    fraction of the measured HBM roofline (algorithmic bytes of one fused pass per launch, SURVEY §8(d)), and an oracle
    check of the device result on a 1024-column sample (float64 restatement of the reference; outside the timed region)."""
    from oracle import oracle_np as O
    from bijectors_jl_b200.distributed import shard_columns

    out = {}
    gen = torch.Generator(device="cuda").manual_seed(77 + rank)

    def batch(Dd, N, scale=1.0):
        return (torch.randn((N, Dd), device="cuda", generator=gen) * scale).t()

    def timed(fn, n):
        for _ in range(max(warmup, 3)):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / n], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    def rec(name, n_total, ms, bytes_total, **extra):
        r = {"ms": ms, "samples_per_s": n_total / (ms * 1e-3), "achieved_gbs": bytes_total / (ms * 1e-3) / 1e9,
             "frac": bytes_total / (ms * 1e-3) / 1e9 / (peak * world), "n_total": int(n_total)}
        r.update(extra)
        out[name] = r

    def sample_cols(N, k=1024):
        return np.sort(np.random.default_rng(5).choice(N, min(k, N), replace=False))

    # ---- C3: 6 x Radial, D=64, N=2^20 per GPU (weak), forward + inverse ------------------------------------------
    Dd, N, L = 64, 1 << 20, 6
    ls, ols = [], []
    for l in range(L):
        r = np.random.Generator(np.random.PCG64(200 + l))
        a, be, z0 = r.standard_normal(1).astype(f32), r.standard_normal(1).astype(f32), r.standard_normal(Dd).astype(f32)
        ls.append(B.RadialLayer(a, be, z0))
        ols.append(O.Layer("radial", dict(alpha_raw=a, beta=be, z0=z0)))
    flow = B.Composed(*ls)
    x, y, lj = batch(Dd, N), B.colmajor_empty(Dd, N), torch.empty(N, device="cuda")
    ms = timed(lambda: B.run_chain(flow, x, y=y, logjac=lj), iters)
    cols = sample_cols(N)
    ct = torch.as_tensor(cols, device="cuda")
    yo, ljo = O.chain_forward(ols, x[:, ct].cpu().numpy().astype(np.float64))
    chk = {"y_rel_err": _rel(y[:, ct].cpu().numpy(), yo), "logjac_rel_err": _rel(lj[ct].cpu().numpy(), ljo)}
    rec("C3_radial6_D64_fwd", world * N, ms, world * N * 4 * (2 * Dd + 1), scaling="weak", oracle_check=chk,
        workload="Composed(6x RadialLayer), D=64, N=2^20 per GPU, forward")
    inv = B.inverse(flow)
    x2, lj2 = B.colmajor_empty(Dd, N), torch.empty(N, device="cuda")
    ms = timed(lambda: B.run_chain(inv, y, y=x2, logjac=lj2), iters)
    xo, ljio = O.chain_inverse(ols, y[:, ct].cpu().numpy().astype(np.float64))
    chk = {"x_rel_err": _rel(x2[:, ct].cpu().numpy(), xo), "logjac_rel_err": _rel(lj2[ct].cpu().numpy(), ljio)}
    rec("C3_radial6_D64_inverse", world * N, ms, world * N * 4 * (2 * Dd + 1), scaling="weak", oracle_check=chk,
        workload="inverse of the same chain applied to its output")
    del x, y, x2, lj, lj2
    torch.cuda.empty_cache()

    # ---- C4: RQS K=8, D=32, N=2^19 TOTAL sharded over the ranks (strong) ---------------------------------------
    Dd, Ntot, K = 32, 1 << 19, 8
    lo, hi = shard_columns(Ntot, rank, world)
    N = hi - lo
    r = np.random.Generator(np.random.PCG64(300))
    rqs = B.RationalQuadraticSpline(r.standard_normal((Dd, K)).astype(f32), r.standard_normal((Dd, K)).astype(f32),
                                    r.standard_normal((Dd, K - 1)).astype(f32), 3.0)
    W, H, Dv = rqs.knots()
    orqs = O.Layer("rqs", dict(widths=W, heights=H, derivs=Dv))
    # the shard (64 MiB / world per pass) is L2-sized: rotate over enough buffer pairs to exceed L2 (126 MB) twice over
    pair_bytes = 2 * N * Dd * 4
    nbuf = max(4, int(2 * 126e6 / pair_bytes) + 1)
    xs = [batch(Dd, N, 1.5) for _ in range(nbuf)]
    ys = [B.colmajor_empty(Dd, N) for _ in range(nbuf)]
    lj = torch.empty(N, device="cuda")

    # one shard of this pass is 5-40 us of GPU time -- less than the Python + driver launch path -- so the rotation over
    # the buffer pairs is captured once into a CUDA graph and replayed (the entry points are launch-only, capture-safe)
    def rot_f():
        for i in range(nbuf):
            B.run_chain(rqs, xs[i], y=ys[i], logjac=lj)

    g_f = B.GraphedCalls(rot_f)
    ms = timed(g_f, max(iters // 2, 3)) / nbuf
    del g_f
    B.run_chain(rqs, xs[0], y=ys[0], logjac=lj)
    cols = sample_cols(N)
    ct = torch.as_tensor(cols, device="cuda")
    yo, ljo = orqs.forward(xs[0][:, ct].cpu().numpy().astype(np.float64))
    chk = {"y_rel_err": _rel(ys[0][:, ct].cpu().numpy(), yo), "logjac_rel_err": _rel(lj[ct].cpu().numpy(), ljo)}
    rec("C4_rqs_K8_D32_fwd", Ntot, ms, Ntot * 4 * (2 * Dd + 1), scaling="strong", oracle_check=chk, cols_per_gpu=int(N),
        l2=f"rotating {nbuf} buffer pairs (> 2 x L2)", launch="CUDA graph of the rotation (one replay = nbuf launches)",
        workload="RationalQuadraticSpline K=8, D=32, N=2^19 total sharded by column")
    irqs = B.inverse(rqs)
    for i in range(nbuf):
        B.run_chain(rqs, xs[i], y=ys[i], logjac=lj)
    xr = [B.colmajor_empty(Dd, N) for _ in range(nbuf)]

    def rot_i():
        for i in range(nbuf):
            B.run_chain(irqs, ys[i], y=xr[i], logjac=lj)

    g_i = B.GraphedCalls(rot_i)
    ms = timed(g_i, max(iters // 2, 3)) / nbuf
    del g_i
    B.run_chain(irqs, ys[0], y=xr[0], logjac=lj)
    xo, ljio = orqs.inverse(ys[0][:, ct].cpu().numpy().astype(np.float64))
    chk = {"x_rel_err": _rel(xr[0][:, ct].cpu().numpy(), xo), "logjac_rel_err": _rel(lj[ct].cpu().numpy(), ljio)}
    rec("C4_rqs_K8_D32_inverse", Ntot, ms, Ntot * 4 * (2 * Dd + 1), scaling="strong", oracle_check=chk, cols_per_gpu=int(N),
        l2=f"rotating {nbuf} buffer pairs (> 2 x L2)")
    del xs, ys, xr, lj
    torch.cuda.empty_cache()

    # ---- C5: RealNVP 4 x (Coupling + BatchNorm), D=256, N=2^22 TOTAL sharded; logpdf + the ONE NCCL sum ---------
    Dd, Ntot = 256, 1 << 22
    lo, hi = shard_columns(Ntot, rank, world)
    N = hi - lo
    r = np.random.Generator(np.random.PCG64(400))
    ls, ols = [], []
    for l in range(4):
        first = l % 2 == 0
        idx1 = list(range(1, 129)) if first else list(range(129, 257))
        idx2 = list(range(129, 257)) if first else list(range(1, 129))
        Wc = (r.standard_normal((256, 128)) * 0.05 / np.sqrt(128)).astype(f32)
        cc = np.zeros(256, f32)
        ls.append(B.Coupling(B.AffineConditioner(Wc, cc), B.PartitionMask(Dd, idx1, idx2)))
        ols.append(O.Layer("coupling_affine", dict(idx1=np.asarray(idx1), idx2=np.asarray(idx2), W=Wc, c=cc)))
        bb, logs, m = (r.standard_normal(Dd) * 0.1).astype(f32), (r.standard_normal(Dd) * 0.1).astype(f32), (r.standard_normal(Dd) * 0.1).astype(f32)
        v = r.uniform(0.5, 1.5, Dd).astype(f32)
        ls.append(B.InvertibleBatchNorm(b=bb, logs=logs, m=m, v=v))
        ols.append(O.Layer("batchnorm", dict(bn=O.BatchNormParams(bb, logs, m, v, f32(1e-5), f32(0.1)))))
    flow = B.Composed(*ls)
    td = B.transformed(B.MvNormal(Dd), flow)
    yb = batch(Dd, N)
    xb, lj = B.colmajor_empty(Dd, N), torch.empty(N, device="cuda")
    ms = timed(lambda: B.run_chain(flow, yb, y=xb, logjac=lj), iters)
    launches = B.lib().b2b_last_launch_count()
    cols = sample_cols(N, 512)
    ct = torch.as_tensor(cols, device="cuda")
    yo, ljo = O.chain_forward(ols, yb[:, ct].cpu().numpy().astype(np.float64))
    chk = {"y_rel_err": _rel(xb[:, ct].cpu().numpy(), yo), "logjac_rel_err": _rel(lj[ct].cpu().numpy(), ljo)}
    # BatchNorm layers are folded into the coupling launches: 4 data passes, each reads D, writes D + logjac
    rec("C5_realnvp_D256_fwd", Ntot, ms, Ntot * 4 * (4 * (2 * Dd + 1) + 3), scaling="strong", oracle_check=chk,
        cols_per_gpu=int(N), launches=int(launches), data_passes=4,
        workload="4 x (affine Coupling + InvertibleBatchNorm), D=256, N=2^22 total sharded by column, with_logabsdet_jacobian")
    total = torch.zeros((), dtype=torch.float64, device="cuda")
    lp_holder = [None]

    def logpdf_step():
        _, lp_holder[0] = B.logpdf_sum(td, yb, out=total)
        if comm is not None:
            comm.allreduce_sum_(total.reshape(1))  # the path's ONE collective: ncclAllReduce(sum) of 8 bytes

    ms = timed(logpdf_step, iters)
    lpo = O.transformed_logpdf(ols, np.zeros(Dd), np.ones(Dd), yb[:, ct].cpu().numpy().astype(np.float64))
    chk = {"logpdf_rel_err": _rel(lp_holder[0][ct].cpu().numpy(), lpo)}
    # cross-check of the reduced total: Σ over ranks of the float64 sum of the per-column logpdf vector
    local = lp_holder[0].double().sum().reshape(1)
    if world > 1:
        dist.all_reduce(local, op=dist.ReduceOp.SUM)
    chk["total_rel_err_vs_vector_sum"] = abs(float(total) - float(local)) / max(abs(float(local)), 1e-30)
    # algorithmic bytes (SURVEY §8(d)): 4 coupling passes with the BatchNorm layers folded in (read D, write D, logjac
    # written once and read-modify-written three times) + the MvNormal pass (read D + logjac, write logpdf)
    rec("C5_realnvp_logpdf_sum", Ntot, ms, Ntot * 4 * (4 * (2 * Dd + 1) + 3 + (Dd + 2)), scaling="strong", oracle_check=chk,
        cols_per_gpu=int(N), total_logpdf=float(total),
        collective=("b2b_allreduce_sum_f64: one ncclAllReduce(sum) of 8 bytes per step, inside the timed region"
                    if comm is not None else "none (1 GPU)"),
        workload="logpdf(transformed(MvNormal(0, I), flow), y) + batch sum, N=2^22 total sharded by column")
    del yb, xb, lj
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--variant", type=int, default=0, help="kernel variant (0 auto, 1 v0 lane-group, 2 v1 interpreter, 3 unrolled planar)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the host-buffer leg (default min(steps, 10))")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-configs", action="store_true", help="skip the C3/C4/C5 sub-records")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--profile", action="store_true",
                    help="profiling runs (under ncu): only the warm-up and the timed headline steps, no JSON contract line")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write y and logjac of the last timed headline step to DIR/*.npy (rank 0; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path; --impl reference has other inputs")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    import bijectors_jl_b200 as B
    from bijectors_jl_b200 import interface as I
    from bijectors_jl_b200.distributed import Communicator, device_for_rank, numa_bind

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    # ranks are spread round-robin over the sockets (2 or 4 ranks on an 8-GPU box use GPUs of BOTH sockets): the
    # host-buffer leg is bound by host DRAM bandwidth per socket
    local = local_rank if args.no_numa else device_for_rank(local_rank)
    torch.cuda.set_device(local)
    # every rank next to its GPU: CPU affinity + preferred memory node BEFORE any pinned host allocation (the 8-rank
    # e2e leg of round 1 crossed the inter-socket link with half of its copies)
    try:
        affinity0 = os.sched_getaffinity(0)
    except AttributeError:
        affinity0 = None
    numa = {"node": -1, "cpus": 0, "bound": False}
    if not args.no_numa:
        try:
            node, ncpu = numa_bind(local)
            numa = {"node": node, "cpus": ncpu, "bound": node >= 0}
        except Exception as ex:  # best effort: an unexposed topology must not fail the bench
            numa["error"] = str(ex)[:200]
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert world == args.gpus or world == 1, (world, args.gpus)
    comm = Communicator() if world > 1 else None  # libb2b's own NCCL communicator (b2b_comm_init_rank)
    B.lib().b2b_set_kernel_variant(args.variant)
    steps, warmup = args.steps, max(args.warmup, 3)

    # ---- synthetic workload (identical on every rank: weak scaling, N columns per GPU) ------------------
    flow = B.Composed(*[B.PlanarLayer(w, u, b) for (w, u, b) in planar_params()])
    gen = torch.Generator(device="cuda").manual_seed(1234 + rank)
    x = torch.randn((NCOLS, D), device="cuda", generator=gen).t()  # D x N column-major, 512 MiB > L2
    y = B.colmajor_empty(D, NCOLS)
    lj = torch.empty(NCOLS, device="cuda")

    def step():
        B.run_chain(flow, x, y=y, logjac=lj)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(warmup):
        step()
    launches_per_step = B.lib().b2b_last_launch_count()
    sync_all()
    sampler = ClockSampler(local) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    sync_all()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms)
    clocks = sampler.stop() if sampler else None
    value = world * NCOLS * steps / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, y, lj)

    if args.profile:
        if rank == 0:
            print(json.dumps({"profile_run": True, "ms_per_step": ms_total / steps, "value": value}))
        if world > 1:
            dist.destroy_process_group()
        return

    # in-run oracle check of the headline result on a 1024-column sample (outside the timed region)
    from oracle import oracle_np as O

    cols = np.sort(np.random.default_rng(5).choice(NCOLS, 1024, replace=False))
    ct = torch.as_tensor(cols, device="cuda")
    olayers = [O.Layer("planar", dict(w=w, u=u, b=b)) for (w, u, b) in planar_params()]
    yo, ljo = O.chain_forward(olayers, x[:, ct].cpu().numpy().astype(np.float64))
    headline_check = {"y_rel_err": _rel(y[:, ct].cpu().numpy(), yo), "logjac_rel_err": _rel(lj[ct].cpu().numpy(), ljo)}

    # ---- same chain with HOST-resident parameters (the reference's own residency): b2b_planar_chain_hostparams_f32 -
    host_flow = B.Composed(*[lay.to("cpu") for lay in B.flatten(flow)])
    for _ in range(3):
        B.run_chain(host_flow, x, y=y, logjac=lj)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        B.run_chain(host_flow, x, y=y, logjac=lj)
    e1.record()
    torch.cuda.synchronize()
    ms_hostparams = e0.elapsed_time(e1) / steps

    # ---- per-layer launches (the reference's launch structure: 8 kernels, y and logjac round-trip HBM) ---
    layers = B.flatten(flow)

    def step_layerwise():
        B.run_chain(layers[0], x, y=y, logjac=lj)
        for lay in layers[1:]:
            B.run_chain(lay, y, y=y, logjac=lj, accumulate=True)

    for _ in range(2):
        step_layerwise()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        step_layerwise()
    e1.record()
    torch.cuda.synchronize()
    ms_layerwise = e0.elapsed_time(e1) / steps
    B.run_chain(flow, x, y=y, logjac=lj)  # restore the fused result for the e2e comparison below

    # ---- e2e: the public API with HOST buffers (pinned, NUMA-local), H2D + kernels + D2H inside the timed region -----
    e2e_steps = args.e2e_steps or min(steps, 10)
    xh = torch.empty((NCOLS, D), dtype=torch.float32, pin_memory=True).t()
    xh.copy_(x)
    for _ in range(2):
        yh, ljh = B.with_logabsdet_jacobian(flow, xh)
    sync_all()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        yh, ljh = B.with_logabsdet_jacobian(flow, xh)
    torch.cuda.synchronize()
    dt = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_value = world * NCOLS * e2e_steps / float(dt)
    assert torch.equal(ljh.cuda(), lj), "host-buffer path and device path disagree"
    del xh, yh, ljh, x, y, lj
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs, same run, same clock -------------------------------------------------------
    peak, peak_src = measured_peaks()
    configs = None
    if not args.no_configs:
        configs = run_configs(B, torch, dist, world, rank, comm, peak, iters=max(min(steps, 10), 5), warmup=3)

    if rank == 0:
        ms_step = ms_total / steps
        bytes_fused = NCOLS * 4 * (2 * D + 1)  # read column + write column + write logjac, once per chain launch
        achieved = bytes_fused / (ms_step * 1e-3) / 1e9
        bytes_layerwise = NCOLS * 4 * (NLAYERS * (2 * D + 1) + (NLAYERS - 1))
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                tj = json.load(open(tpath))
                traffic = tj.get("chain_kernel_dram_bytes_per_launch")
                traffic_src = tj.get("source")
            except Exception:
                traffic = None
        line = {
            "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "chain": "one fused chain launch per step (column read once, written once); parameters device-resident",
                       "l2": "inputs_larger_than_L2 (x, y 512 MiB each per GPU; L2 126 MB)",
                       "parallelism": f"columns sharded, {world} rank(s), no data-path collective",
                       "kernel_variant": args.variant, "numa": numa, "cuda_device_of_rank0": local},
            "gpu_launches": int(launches_per_step * steps),
            "oracle_check": headline_check,
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": int(NCOLS * D * 4),
                    "d2h_bytes_per_step": int(NCOLS * D * 4 + NCOLS * 4), "steps": e2e_steps,
                    "api": "with_logabsdet_jacobian(flow, pinned host D x N) -> b2b_chain_run_host_f32",
                    "host_pipeline": {"chunk_cols": I.HOST_CHUNK_COLS, "streams": I.HOST_STREAMS, "numa_node": numa["node"]},
                    # what the copies ask of the host memory system (DMA reads + writes of pinned DRAM, all ranks)
                    "host_dram_gbs": e2e_value * (2 * D * 4 + 4) / 1e9},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peak_src})",
                         "kernel": "planar_dev_kernel: fused 8-layer chain, 1 launch/step", "algorithmic_bytes_per_launch": bytes_fused,
                         "accounting": "chain-fused: 4*(2D+1) B/sample per launch"},
            "host_resident_parameters": {"ms_per_step": ms_hostparams, "samples_per_s": NCOLS / (ms_hostparams * 1e-3),
                                         "frac": NCOLS * 4 * (2 * D + 1) / (ms_hostparams * 1e-3) / 1e9 / peak,
                                         "api": "b2b_planar_chain_hostparams_f32 (parameters as kernel arguments)"},
            "per_layer_launches": {"ms_per_step": ms_layerwise, "samples_per_s": NCOLS / (ms_layerwise * 1e-3),
                                   "achieved_gbs": bytes_layerwise / (ms_layerwise * 1e-3) / 1e9,
                                   "frac": bytes_layerwise / (ms_layerwise * 1e-3) / 1e9 / peak,
                                   "accounting": "8 launches: 4*(L*(2D+1)+(L-1)) B/sample"},
            "clocks": clocks,
        }
        if configs is not None:
            line["configs"] = configs
        if world == 1 and not args.no_cpu:
            if affinity0 is not None:
                try:
                    os.sched_setaffinity(0, affinity0)  # the CPU baseline may use every host core again
                except Exception:
                    pass
            line["cpu_baseline"] = cpu_baseline()
        print(json.dumps(line))
    if comm is not None:
        comm.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
