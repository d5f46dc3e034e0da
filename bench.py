#!/usr/bin/env python
"""bench.py -- headline benchmark of the block-sparse matmul hot path on B200.

A "step" = one fprop + one bprop + one updat of BlocksparseMatMul over one synthetic
minibatch (BASELINE.json configs[1]: 4096x4096, block_size 32, bf16, N=4096 per GPU,
density 25 % unless --density is given).  Metric = effective TFLOP/s
= 3 * 2*nnz_blocks*bs^2*N / t  (the reference's own flop accounting, op.cc:102,182).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step returned (Y, DX, DW) as float32 DIR/{y,dx,dw}.npy (rank 0), so that
two builds can be compared output for output: inputs and layout are seeded, identical from run to run.  The files hold
at most 64 MB in all, so a larger output is cut to a fixed, seeded sample of its minibatch rows (DW: of its blocks).

N>1 is launched by torchrun (one rank per GPU): the minibatch axis is sharded (weak
scaling: every rank holds N=4096 columns), fprop/bprop need no communication and the
updat output dW (fp32 when N>1) is all-reduced with NCCL on a side stream, overlapping the
next step's fprop/bprop, with BSMM_SM_MARGIN SMs left free for the NCCL kernel (SURVEY.md 8e).

Besides the headline the JSON line carries (rank 0, skipped with --no-extras):
  check           max_rel_err / l2_err of Y, DX, DW taken from the TIMED buffers against the oracle (row/block sample)
  density_sweep   every op at 5/10/25/50/100 % density with frac_tensor_peak and frac_hbm_peak, cold and warm L2
  variants        the skewed Barabasi-Albert layout, feature_axis 0, block size 64, fp16 at the headline density
  cfg3 / cfg4     the block-sparse attention ops and the block-size sweep of BASELINE configs[2] / [3]
  cfg5_strong     BASELINE configs[4]: global N=32768 split over the ranks (strong scaling), per-rank N = 32768/world
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C = K = 4096
BS = 32
N_PER_GPU = 4096
SEED = 1236
DUMP_BYTES = 64 * 10 ** 6


def make_layout(density, cb=C // BS, kb=K // BS, seed=SEED):
    rng = np.random.default_rng(seed)
    lay = (rng.random((cb, kb)) < density).astype(np.int32)
    np.fill_diagonal(lay, 1)
    return lay


def bind_to_gpu_numa_node(index):
    """Pin this process to the CPUs local to GPU `index` (sysfs local_cpulist of its PCI device); returns the previous
    affinity mask, or None when the topology cannot be read (then nothing changes)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:                   # NVML pads the PCI domain to 8 hex digits, sysfs uses 4
            bus = bus[4:]
        with open("/sys/bus/pci/devices/%s/local_cpulist" % bus) as f:
            txt = f.read().strip()
        cpus = set()
        for part in txt.split(","):
            if "-" in part:
                lo, hi = part.split("-")
                cpus.update(range(int(lo), int(hi) + 1))
            elif part:
                cpus.add(int(part))
        old = os.sched_getaffinity(0)
        cpus &= old
        if not cpus or cpus == old:
            return None
        os.sched_setaffinity(0, cpus)
        return old
    except Exception:
        return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, source="fallback")


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled WHILE the timed region runs (NVML in-process, ~1 ms per sample;
    falls back to spawning nvidia-smi, ~0.3 s per sample, when pynvml is not importable)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout
        f = [x.strip() for x in out.strip().split(",")]
        if len(f) >= 6:
            self.max_mhz = float(f[1])
            mask = 0
            for bit, v in zip((0x8, 0x40, 0x20, 0x4), f[2:6]):
                if v.lower().startswith("active"):
                    mask |= bit
            self.rows.append((float(f[0]), mask))

    def run(self):
        while not self._halt.is_set():
            try:
                if self.nvml:
                    mhz = float(self.nvml.nvmlDeviceGetClockInfo(self.handle, self.nvml.NVML_CLOCK_SM))
                    mask = int(self.nvml.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                    self.rows.append((mhz, mask))
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._halt.wait(0.005 if self.nvml else 0.1)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(r[0] for r in self.rows)
        seen = 0
        for _, m in self.rows:
            seen |= m
        reasons = [name for bit, name in self.REASONS.items() if seen & bit]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": getattr(self, "max_mhz", None), "reasons": reasons,
                "samples": len(self.rows), "source": "nvml" if self.nvml else "nvidia-smi"}


def cpu_reference(density, axis, budget_s=20.0, steps=1):
    """The reference's path on the host cores: its NumPy checker math (blocksparse/matmul.py:353-419),
    restated BLAS-batched in oracle/bsmm_oracle.py, on a bounded column sample of the same workload."""
    from oracle.bsmm_oracle import MatmulOracle, fprop_fast, bprop_fast, updat_fast
    lay = make_layout(density)
    orc = MatmulOracle(lay, BS, axis)
    rng = np.random.default_rng(SEED)
    n = 1024                                 # columns of the 4096-wide minibatch timed per step (shrunk below for many steps)
    W = rng.normal(0, 0.01, orc.w_shape).astype(np.float32)
    X = rng.normal(0, 0.1, orc.i_shape(n)).astype(np.float32)
    E = rng.normal(0, 0.1, orc.o_shape(n)).astype(np.float32)
    fprop_fast(orc, X[:8] if axis else X[:, :8], W)       # warm BLAS

    def one_pass(x, e):
        fprop_fast(orc, x, W)
        bprop_fast(orc, e, W)
        updat_fast(orc, x, e)

    # NumPy's batched small matmuls do not scale monotonically with BLAS threads (64 threads were 3x slower than 1 on
    # the B200 host): probe a few thread counts on a quarter-size sample and keep the fastest, up to all host cores.
    ncpu = os.cpu_count() or 1
    threads, limiter = ncpu, None
    try:
        from threadpoolctl import threadpool_limits
        xs = X[:256] if axis else X[:, :256]
        es = E[:256] if axis else E[:, :256]
        best = None
        for th in sorted({1, 4, 8, 16, min(32, ncpu), ncpu}):
            if th > ncpu:
                continue
            with threadpool_limits(limits=th):
                t = time.perf_counter()
                one_pass(xs, es)
                t = time.perf_counter() - t
            if best is None or t < best[0]:
                best = (t, th)
        threads = best[1]
        limiter = threadpool_limits(limits=threads)
    except Exception:
        pass
    # `--impl reference --steps K`: every step is one pass over a column sample sized so that the K steps end within
    # ~2 minutes (the metric is a rate, so the sample size only changes BLAS efficiency a little); the default
    # cpu_baseline leg (steps == 1) keeps the 1024-column sample and repeats it 3 times.
    if steps > 3:
        xs = X[:128] if axis else X[:, :128]
        es = E[:128] if axis else E[:, :128]
        t = time.perf_counter()
        one_pass(xs, es)
        per_col = (time.perf_counter() - t) / 128
        n_fit = int(120.0 / (steps * per_col))
        n = max(64, min(1024, n_fit // 64 * 64))
        X = X[:n] if axis else X[:, :n]
        E = E[:n] if axis else E[:, :n]
    t0 = time.perf_counter()
    done = 0
    while done < steps or (time.perf_counter() - t0 < budget_s and done < 3):
        one_pass(X, E)
        done += 1
    dt = (time.perf_counter() - t0) / done
    if limiter is not None:
        limiter.restore_original_limits()
    flops = 3 * 2.0 * orc.blocks * BS * BS * n
    return {"value": flops / dt / 1e12, "unit": "TFLOP/s", "cores": int(threads), "kind": "port",
            "host_cores": ncpu,
            "sample": "fprop+bprop+updat on %d of %d minibatch columns, density %.2f, fp32 NumPy/BLAS (best of 1..%d threads), %d repeats" % (n, N_PER_GPU, density, ncpu, done),
            "ms_per_sample": dt * 1e3}, dt


def time_loop(torch, fn, reps, warm=3):
    for i in range(warm):
        fn(i)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(reps):
        fn(i)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def op_record(ms, flops, nbytes, pk, kernel=None):
    r = {"ms": ms, "tflops": flops / (ms * 1e-3) / 1e12, "frac_tensor_peak": flops / (ms * 1e-3) / 1e12 / pk["tf_burst"],
         "hbm_gbs": nbytes / (ms * 1e-3) / 1e9, "frac_hbm_peak": nbytes / (ms * 1e-3) / 1e9 / pk["hbm"]}
    if kernel:
        r["kernel"] = kernel
    return r


def time_three_ops(torch, _lib, bsmm, W, Xs, Es, pk, reps=20, warm_l2=False):
    """fprop / bprop / updat of one BlocksparseMatMul, each alone.  cold: rotating input sets (> L2); warm: same buffers."""
    n = len(Xs)
    N = Xs[0].numel() // bsmm.C
    fl = 2.0 * bsmm.blocks * bsmm.bsize ** 2 * N
    by = 2.0 * (bsmm.C * N + bsmm.K * N) + 2.0 * bsmm.blocks * bsmm.bsize ** 2
    out = {}
    pick = (lambda i: 0) if warm_l2 else (lambda i: i % n)
    for name, fn in [("fprop", lambda i: bsmm.fprop(Xs[pick(i)], W)), ("bprop", lambda i: bsmm.bprop(Es[pick(i)], W)),
                     ("updat", lambda i: bsmm.updat([Xs[pick(i)]], [Es[pick(i)]]))]:
        ms = time_loop(torch, fn, reps)
        out[name] = op_record(ms, fl, by, pk, _lib.last_kernel())
    return out


def check_against_oracle(torch, bsmm, lay, axis, W, X, E, y, dx, dw, n_rows=32, n_blocks=64):
    """Sample of the step's own outputs against the oracle (bounded CPU work, test infrastructure used as the checker)."""
    from oracle.bsmm_oracle import MatmulOracle
    orc = MatmulOracle(lay, bsmm.bsize, axis)
    N = X.shape[0] if axis else X.shape[1]
    rows = torch.as_tensor((np.arange(n_rows) * (N // n_rows) + np.arange(n_rows) % 5) % N, device=X.device)

    def sample(t):
        return (t.index_select(0, rows) if axis else t.index_select(1, rows)).float().cpu().numpy()

    def errs(got, ref):
        d = np.abs(np.asarray(got, dtype=np.float64) - ref)
        return {"max_rel_err": float(d.max() / np.abs(ref).mean()), "l2_err": float(np.sqrt((d * d).sum() / (ref * ref).sum()))}

    Wh = W.float().cpu().numpy()
    rng = np.random.default_rng(0)
    blk = np.sort(rng.choice(bsmm.blocks, size=min(n_blocks, bsmm.blocks), replace=False))
    ref_dw = orc.updat_blocks(X.float().cpu().numpy(), E.float().cpu().numpy(), blk)
    return {"fprop": errs(sample(y), orc.fprop(sample(X), Wh)), "bprop": errs(sample(dx), orc.bprop(sample(E), Wh)),
            "updat": errs(dw.index_select(0, torch.as_tensor(blk, device=dw.device)).float().cpu().numpy(), ref_dw),
            "sample": "%d minibatch rows (all features) for fprop/bprop, %d weight blocks (full minibatch) for updat; "
                      "oracle = NumPy restatement of matmul.py:353-419" % (n_rows, len(blk)),
            "tolerance": "l2_err <= 1e-2 (bf16)"}


def dump_outputs(torch, out_dir, arrays):
    """Save {name: (tensor, dim)} as float32 out_dir/<name>.npy, DUMP_BYTES in all.  A tensor larger than its even share
    keeps a fixed, seeded, sorted sample of its slices along `dim` (minibatch rows for Y / DX, blocks for DW)."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays) - 128                  # 128: the .npy header
    for name, (t, dim) in arrays.items():
        n = t.shape[dim]
        keep = min(n, share // (4 * (t.numel() // n)))
        if keep < n:
            idx = np.sort(np.random.default_rng(SEED).choice(n, keep, replace=False))
            t = t.index_select(dim, torch.as_tensor(idx, device=t.device))
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--density", type=float, default=0.25)
    ap.add_argument("--axis", type=int, default=1)
    ap.add_argument("--sweep", action="store_true", help="(kept for compatibility: the sweep is on by default)")
    ap.add_argument("--no-extras", action="store_true", help="headline only: no sweep / variants / cfg3 / cfg4 / cfg5 sub-records")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--sm-margin", type=int, default=None, help="SMs left free for NCCL when N>1 (default 8 at 2 GPUs, 12 beyond; BSMM_SM_MARGIN wins)")
    ap.add_argument("--blocking-allreduce", action="store_true", help="round-1 behaviour: all-reduce on the compute stream")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's Y, DX, DW to DIR/{y,dx,dw}.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    args.warmup = max(args.warmup, 3)

    config = {"workload": "BlocksparseMatMul %dx%d block_size=%d density=%.0f%% N=%d/GPU bf16 fprop+bprop+updat (BASELINE configs[1])"
                          % (C, K, BS, args.density * 100, N_PER_GPU),
              "feature_axis": args.axis, "layout_seed": SEED, "global_N": N_PER_GPU * world,
              "parallelism": "dp%d (N-sharded, all-reduce on dW)" % world,
              "l2": "inputs larger than L2: 3 rotating buffer sets (X,DY,Y,DX per set), 400+ MB"}

    if args.impl == "reference":
        if rank != 0:
            return
        cb, dt = cpu_reference(args.density, args.axis, steps=args.steps)
        line = {"impl": "reference", "metric": "effective TFLOP/s (2*nnz_blocks*bs^2*N, fprop+bprop+updat)", "value": cb["value"],
                "unit": "TFLOP/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config, "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    from blocksparse_b200 import dist as bdist
    margin = 0
    if world > 1 and not args.blocking_allreduce:
        # measured (profiles/r2_scaling.txt): 8 NCCL CTAs hide the 17 MB fp32 all-reduce at 2 GPUs, 8 GPUs need 12.  The margin is
        # 4 SMs LARGER than the CTAs NCCL may use: the persistent grids are dealt tiles statically, so a single CTA that finds
        # its SM taken runs as a second wave and doubles the kernel time (the bimodal 0.23 / 0.40 ms steps seen with zero slack)
        ctas = (8 if world <= 2 else 12)
        margin = bdist.reserve_sms_for_nccl(ctas + 4 if args.sm_margin is None else args.sm_margin,
                                            nccl_ctas=ctas if args.sm_margin is None else max(1, args.sm_margin - 4))
    import torch
    import torch.distributed as dist
    from blocksparse_b200 import BlocksparseMatMul, _lib

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        if args.blocking_allreduce:
            dist.init_process_group("nccl", device_id=dev)
        else:
            dist.init_process_group("nccl", device_id=dev, pg_options=bdist.nccl_options())
    dtype = torch.bfloat16
    lay = make_layout(args.density)
    bsmm = BlocksparseMatMul(lay, block_size=BS, feature_axis=args.axis)
    N = N_PER_GPU
    gen = torch.Generator(device=dev).manual_seed(SEED + rank)
    W = (torch.randn(bsmm.w_shape, generator=gen, device=dev) * 0.01).to(dtype)
    NSETS = 3
    Xs = [(torch.randn(bsmm.i_shape(N), generator=gen, device=dev) * 0.1).to(dtype) for _ in range(NSETS)]
    Es = [(torch.randn(bsmm.o_shape(N), generator=gen, device=dev) * 0.1).to(dtype) for _ in range(NSETS)]
    launches = [0]
    # N>1: the partial dW is produced in fp32 and summed in fp32 (8 bf16 partial sums would each be rounded to 8 bits of
    # mantissa); the reduction runs on a side stream and overlaps the next step's fprop/bprop (the reference's
    # AllreduceNccl pattern, src/nccl_op.cc:168,513), ordered before the next updat.
    dw_dtype = torch.float32 if world > 1 else None
    side = bdist.AllreduceStream(dev) if (world > 1 and not args.blocking_allreduce) else None
    config["dw_dtype"] = "fp32" if world > 1 else "bf16"
    config["allreduce"] = ("none (1 GPU)" if world == 1 else "blocking on the compute stream" if side is None else
                           "side stream, one reduction in flight, overlaps the next step's kernels; %d SMs left to NCCL (NCCL_MAX_CTAS=%s)"
                           % (margin, os.environ.get("NCCL_MAX_CTAS")))

    use_side = [side is not None]

    def make_step(op, w, xs, es):
        def step(i):
            x, e = xs[i % len(xs)], es[i % len(es)]
            y = op.fprop(x, w)
            dx = op.bprop(e, w)
            dw = op.updat([x], [e], dw_dtype=dw_dtype)
            launches[0] += 3
            if use_side[0]:
                # at most one reduction in flight: the previous one (whose consumer would be the optimizer) is ordered
                # before this one is issued, so it overlaps a whole step of fprop / bprop / updat
                side.wait()
                side.reduce(dw)
            else:
                bdist.allreduce_dw(dw)            # no-op at world size 1
            return y, dx, dw
        return step

    step = make_step(bsmm, W, Xs, Es)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, steps):
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        last = None
        for i in range(steps):
            last = step_fn(i)
        if side is not None:
            side.wait()
        ev1.record()
        barrier()
        t = torch.tensor([ev0.elapsed_time(ev1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps, last

    for i in range(args.warmup):
        step(i)
    if side is not None:
        side.wait()
    if side is not None:
        # Untimed settling + calibration.  Whether the NCCL kernel really runs BESIDE the persistent grids depends on where the
        # block scheduler places it, and the first process on a fresh box has shown a transient 3.5 ms/step state
        # (profiles/r2_scaling.txt).  Run 100 more untimed steps, then time both schemes for 20 steps each, agree across ranks
        # (max over ranks) and keep the faster one for the timed region.
        for i in range(100):
            step(i)
        side.wait()

        def trial(flag, n=20):
            use_side[0] = flag
            for i in range(3):
                step(i)
            side.wait()
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(n):
                step(i)
            side.wait()
            b.record()
            barrier()
            t = torch.tensor([a.elapsed_time(b) / n], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        t_block, t_side = trial(False), trial(True)
        use_side[0] = t_side <= t_block
        config["allreduce"] += "; calibrated before timing: overlapped %.4f ms/step, blocking %.4f ms/step -> %s" % (
            t_side, t_block, "overlapped" if use_side[0] else "blocking")
    kernels = {}
    bsmm.fprop(Xs[0], W); kernels["fprop"] = _lib.last_kernel()
    bsmm.bprop(Es[0], W); kernels["bprop"] = _lib.last_kernel()
    bsmm.updat([Xs[0]], [Es[0]]); kernels["updat"] = _lib.last_kernel()
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    launches[0] = 0
    ms_per_step, last = timed(step, args.steps)
    timed_samples = len(sampler.rows) if sampler else 0
    n_launches = launches[0]
    flops_step_gpu = 3 * 2.0 * bsmm.blocks * BS * BS * N
    value = flops_step_gpu * world / (ms_per_step * 1e-3) / 1e12

    # ---- correctness of what was just timed: the last step's outputs against the oracle (rank 0)
    check = None
    if rank == 0:
        li = (args.steps - 1) % NSETS
        y_l, dx_l, dw_l = last
        if world > 1:           # the all-reduced dW is the sum over ranks: check this rank's partial instead
            dw_l = bsmm.updat([Xs[li]], [Es[li]], dw_dtype=dw_dtype)
        check = check_against_oracle(torch, bsmm, lay, args.axis, W, Xs[li], Es[li], y_l, dx_l, dw_l)
        check["device_error"] = _lib.device_error()
        if args.dump_outputs:   # dW as the caller receives it (all-reduced when N>1)
            dump_outputs(torch, args.dump_outputs, {"y": (y_l, 0 if args.axis else 1), "dx": (dx_l, 0 if args.axis else 1),
                                                    "dw": (last[2], 0)})

    # ---- per-kernel timing (each kernel alone) for the roofline object: cold (rotating inputs > L2) and warm L2
    pk = peaks()
    cold = time_three_ops(torch, _lib, bsmm, W, Xs, Es, pk, reps=50)
    warm = time_three_ops(torch, _lib, bsmm, W, Xs, Es, pk, reps=50, warm_l2=True)
    per_op = {k: v["ms"] for k, v in cold.items()}
    clocks = None
    if sampler:                      # sampled from the start of the timed region to the end of the per-kernel loops
        clocks = sampler.stop()
        clocks["samples_in_timed_region"] = timed_samples
    flops_op = 2.0 * bsmm.blocks * BS * BS * N
    bytes_op = 2.0 * (C * N + K * N) + 2.0 * bsmm.blocks * BS * BS
    dom = max(per_op, key=per_op.get)
    tf = flops_op / (per_op[dom] * 1e-3) / 1e12
    gbs = bytes_op / (per_op[dom] * 1e-3) / 1e9
    ridge = pk["tf_burst"] * 1e12 / (pk["hbm"] * 1e9)
    if flops_op / bytes_op >= ridge:
        roof = {"bound": "tensor", "achieved": tf, "peak": pk["tf_burst"], "unit": "TFLOP/s", "frac": tf / pk["tf_burst"]}
    else:
        roof = {"bound": "hbm", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"]}
    traffic, traffic_src = None, None
    for tname in ("r2_traffic.json", "r1_traffic.json"):       # dram bytes per launch from the committed ncu --set full capture
        tpath = os.path.join(ROOT, "profiles", tname)
        if os.path.exists(tpath) and abs(args.density - 0.25) < 1e-9:
            traffic = json.load(open(tpath)).get(kernels[dom])
            if traffic is not None:
                traffic_src = "profiles/" + tname
                break
    roof.update({"kernel": "%s (%s)" % (dom, kernels[dom]), "traffic": traffic, "traffic_source": traffic_src,
                 "peak_source": pk["source"], "per_op_ms": per_op, "per_op_ms_warm_l2": {k: v["ms"] for k, v in warm.items()},
                 "per_op_tflops": {k: v["tflops"] for k, v in cold.items()},
                 "per_op_frac_tensor_peak": {k: v["frac_tensor_peak"] for k, v in cold.items()},
                 "per_op_frac_hbm_peak": {k: v["frac_hbm_peak"] for k, v in cold.items()},
                 "algorithmic_flops_per_launch": flops_op, "algorithmic_bytes_per_launch": bytes_op})

    # ---- end to end through the public API with HOST buffers (pinned), copies inside the timed region
    # pinned buffers are first-touched on the NUMA node the GPU hangs off (PCIe copies from the far socket run at about
    # half rate on these hosts); the affinity is restored afterwards
    old_affinity = bind_to_gpu_numa_node(dev.index if dev.index is not None else 0)
    hx = [torch.empty(bsmm.i_shape(N), dtype=dtype).pin_memory() for _ in range(2)]
    he = [torch.empty(bsmm.o_shape(N), dtype=dtype).pin_memory() for _ in range(2)]
    for h, s in zip(hx + he, Xs[:2] + Es[:2]):
        h.copy_(s)
    hy = torch.empty(bsmm.o_shape(N), dtype=dtype).pin_memory()
    hdx = torch.empty(bsmm.i_shape(N), dtype=dtype).pin_memory()
    hdw = torch.empty(bsmm.w_shape, dtype=dtype).pin_memory()
    w_param = W.clone().requires_grad_()
    if old_affinity is not None:
        os.sched_setaffinity(0, old_affinity)

    # Three streams pipeline consecutive steps (copies of step i+1 / i-1 overlap the kernels of step i, as a training
    # input pipeline would); every step still moves its own inputs H2D and its own results D2H inside the timed region.
    s_h2d, s_d2h = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    s_comp = torch.cuda.current_stream()
    dev_x = [torch.empty(bsmm.i_shape(N), dtype=dtype, device=dev) for _ in range(2)]
    dev_e = [torch.empty(bsmm.o_shape(N), dtype=dtype, device=dev) for _ in range(2)]
    comp_done = [None, None]
    d2h_done = [None, None]

    def e2e_step(i):
        j = i % 2
        with torch.cuda.stream(s_h2d):
            if comp_done[j] is not None:
                s_h2d.wait_event(comp_done[j])          # step i-2 no longer reads these device buffers
            dev_x[j].copy_(hx[j], non_blocking=True)
            dev_e[j].copy_(he[j], non_blocking=True)
            ready = torch.cuda.Event()
            ready.record(s_h2d)
        s_comp.wait_event(ready)
        x = dev_x[j].detach().requires_grad_()
        w_param.grad = None
        y = bsmm(x, w_param)
        y.backward(dev_e[j])
        bdist.allreduce_dw(w_param.grad)
        done = torch.cuda.Event()
        done.record(s_comp)
        comp_done[j] = done
        yd, dxd, dwd = y.detach(), x.grad, w_param.grad
        with torch.cuda.stream(s_d2h):
            s_d2h.wait_event(done)
            hy.copy_(yd, non_blocking=True)
            hdx.copy_(dxd, non_blocking=True)
            hdw.copy_(dwd, non_blocking=True)
            for t_ in (yd, dxd, dwd):
                t_.record_stream(s_d2h)
            fin = torch.cuda.Event()
            fin.record(s_d2h)
            d2h_done[j] = fin

    def e2e_drain():
        for ev in d2h_done:
            if ev is not None:
                s_comp.wait_event(ev)

    e2e_steps = max(3, min(args.steps, 30))
    for i in range(3):
        e2e_step(i)
    e2e_drain()
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(e2e_steps):
        e2e_step(i)
    e2e_drain()
    b.record()
    barrier()
    t = torch.tensor([a.elapsed_time(b) / e2e_steps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    h2d_b = int(hx[0].numel() * 2 + he[0].numel() * 2)
    d2h_b = int(hy.numel() * 2 + hdx.numel() * 2 + hdw.numel() * 2)
    e2e = {"value": flops_step_gpu * world / (e2e_ms * 1e-3) / 1e12, "unit": "TFLOP/s",
           "h2d_bytes_per_step": h2d_b, "d2h_bytes_per_step": d2h_b,
           "ms_per_step": e2e_ms, "host_buffers_numa_local": old_affinity is not None,
           "pcie_gbs": {"h2d_plus_d2h_per_step_over_time": (h2d_b + d2h_b) / (e2e_ms * 1e-3) / 1e9},
           "api": "BlocksparseMatMul.__call__ + autograd backward; pinned host buffers; H2D / kernels / D2H on three streams, double-buffered"}
    del hx, he, hy, hdx, hdw, dev_x, dev_e

    # ---- BASELINE configs[4]: strong scaling, global N = 32768 split over the ranks (all ranks take part)
    extras = {}
    if not args.no_extras:
        Ng = 32768
        n_loc = Ng // world
        reps = 1 if n_loc <= N else n_loc // N
        # the shard is `reps` concatenated copies of the 4096-row synthetic sets (fresh rows would only change the data)
        xs5 = [torch.cat([Xs[(j + r) % NSETS] for r in range(reps)], 0 if args.axis else 1) for j in range(2 if reps > 2 else NSETS)]
        es5 = [torch.cat([Es[(j + r) % NSETS] for r in range(reps)], 0 if args.axis else 1) for j in range(2 if reps > 2 else NSETS)]
        step5 = make_step(bsmm, W, xs5, es5)
        for i in range(3):
            step5(i)
        ms5, _ = timed(step5, 20)
        extras["cfg5_strong"] = {"global_N": Ng, "N_per_gpu": n_loc, "ms_per_step": ms5,
                                 "value": 3 * 2.0 * bsmm.blocks * BS * BS * Ng / (ms5 * 1e-3) / 1e12, "unit": "TFLOP/s",
                                 "note": "BASELINE configs[4] as written: fixed global minibatch; compare across --gpus runs"}
        del xs5, es5

    if rank == 0 and world == 1 and not args.no_extras:       # single-GPU sub-records: part of the N=1 line only
        from blocksparse_b200.layouts import barabasi_albert_layout
        sweep = {}
        for d in (0.05, 0.10, 0.25, 0.50, 1.00):
            b2 = BlocksparseMatMul(make_layout(d), block_size=BS, feature_axis=args.axis)
            W2 = (torch.randn(b2.w_shape, generator=gen, device=dev) * 0.01).to(dtype)
            r = time_three_ops(torch, _lib, b2, W2, Xs, Es, pk, reps=20)
            rw = time_three_ops(torch, _lib, b2, W2, Xs, Es, pk, reps=20, warm_l2=True)
            for k in r:
                r[k]["ms_warm_l2"] = rw[k]["ms"]
            r["nnz_blocks"] = b2.blocks
            sweep["%d%%" % round(d * 100)] = r
        extras["density_sweep"] = sweep
        var = {}
        b2 = BlocksparseMatMul(barabasi_albert_layout(C // BS, args.density, np.random.default_rng(SEED + 1)), block_size=BS, feature_axis=args.axis)
        W2 = (torch.randn(b2.w_shape, generator=gen, device=dev) * 0.01).to(dtype)
        var["barabasi_albert_skewed"] = dict(time_three_ops(torch, _lib, b2, W2, Xs, Es, pk), nnz_blocks=b2.blocks,
                                             max_col_blocks=int(b2.layout.sum(0).max()), mean_col_blocks=float(b2.layout.sum(0).mean()))
        b2 = BlocksparseMatMul(lay, block_size=BS, feature_axis=1 - args.axis)
        xt = [x.t().contiguous() for x in Xs]
        et = [e.t().contiguous() for e in Es]
        var["feature_axis_%d" % (1 - args.axis)] = dict(time_three_ops(torch, _lib, b2, W, xt, et, pk), nnz_blocks=b2.blocks)
        del xt, et
        b2 = BlocksparseMatMul(make_layout(args.density, C // 64, K // 64), block_size=64, feature_axis=args.axis)
        W2 = (torch.randn(b2.w_shape, generator=gen, device=dev) * 0.01).to(dtype)
        var["block_size_64"] = dict(time_three_ops(torch, _lib, b2, W2, Xs, Es, pk), nnz_blocks=b2.blocks)
        var["fp16"] = dict(time_three_ops(torch, _lib, bsmm, W.half(), [x.half() for x in Xs], [e.half() for e in Es], pk), nnz_blocks=bsmm.blocks)
        extras["variants"] = var
        # BASELINE configs[3]: block-size sweep at 20 % density, N = 2048
        cfg4 = {}
        x4 = [x[:2048].contiguous() if args.axis else x[:, :2048].contiguous() for x in Xs]
        e4 = [e[:2048].contiguous() if args.axis else e[:, :2048].contiguous() for e in Es]
        for bs4 in (8, 16, 32, 64):
            b2 = BlocksparseMatMul(make_layout(0.20, C // bs4, K // bs4, seed=1238), block_size=bs4, feature_axis=args.axis)
            W2 = (torch.randn(b2.w_shape, generator=gen, device=dev) * 0.01).to(dtype)
            cfg4["bs%d" % bs4] = dict(time_three_ops(torch, _lib, b2, W2, x4, e4, pk, reps=10), nnz_blocks=b2.blocks)
        extras["cfg4_block_size_sweep"] = {"config": "4096x4096 density 20%% N=2048 bf16 axis %d" % args.axis, "results": cfg4}
        del x4, e4
        extras["cfg3_attention"] = bench_attention(torch, _lib, dev, pk)
        extras["device_error_after_extras"] = _lib.device_error()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu, _ = cpu_reference(args.density, args.axis)

    if rank == 0:
        line = {"metric": "effective TFLOP/s (2*nnz_blocks*bs^2*N, fprop+bprop+updat)", "value": value, "unit": "TFLOP/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": config, "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks,
                "gpu_launches": n_launches, "kernels": kernels, "nnz_blocks": bsmm.blocks,
                "frac_density_scaled_tensor_peak": value / world / pk["tf_sust"], "check": check}
        line.update(extras)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def bench_attention(torch, _lib, dev, pk):
    """BASELINE configs[2]: heads 16, ctx 4096, bs 64, local+strided causal layout, batch 4, head_state 64, fp16."""
    from blocksparse_b200 import BlocksparseTransformer
    from blocksparse_b200.layouts import local_strided_layout
    batch, heads, hs, bs, nb = 4, 16, 64, 64, 64
    lay = local_strided_layout(nb)

    def causal(blk_shape, head_idx, qry_idx, key_idx, blk_idx):
        m = np.ones(blk_shape, dtype=bool)
        return np.tril(m) if qry_idx == key_idx else m

    bst = BlocksparseTransformer(lay, bs, heads=heads, mask_callback=causal)
    gen = torch.Generator(device=dev).manual_seed(0)
    Q, Kt, V, DY = ((torch.rand((batch, nb * bs, heads * hs), generator=gen, device=dev) * 2 - 1).half() for _ in range(4))
    scale = 1.0 / np.sqrt(hs)
    S = bst._nt(Q, Kt, torch.bfloat16)
    P = bst._softmax(S, scale, True, None, torch.float16)
    DP = bst._nt(DY, V, torch.float16)
    bh = batch * heads
    gemm_flops = 2.0 * bst.blocks * bs * bs * hs * bh
    sparse_bytes = bst.blocks * bs * bs * 2.0 * bh
    dense_bytes = nb * bs * hs * 2.0 * bh
    ops = [("nt", lambda i: bst._nt(Q, Kt, torch.bfloat16), gemm_flops, 2 * dense_bytes + sparse_bytes),
           ("masked_softmax", lambda i: bst._softmax(S, scale, True, None, torch.float16), 0.0, 2 * sparse_bytes),
           ("nn", lambda i: bst._xn(P, V, False), gemm_flops, sparse_bytes + 2 * dense_bytes),
           ("tn", lambda i: bst._xn(P, DY, True), gemm_flops, sparse_bytes + 2 * dense_bytes),
           ("softmax_grad", lambda i: bst._softmax_grad(DP, P, scale), 0.0, 3 * sparse_bytes)]
    if hasattr(bst, "attention"):
        ops.append(("fused_attention", lambda i: bst.attention(Q, Kt, V, scale=scale), 2 * gemm_flops, 4 * dense_bytes))
    out = {"config": "batch 4 heads 16 head_state 64 ctx 4096 bs 64, %d blocks, fp16 in / bf16 scores" % bst.blocks}
    for name, fn, fl, by in ops:
        ms = time_loop(torch, fn, 10)
        out[name] = op_record(ms, fl, by, pk, _lib.last_kernel())
    out["forward_chain_ms"] = out["nt"]["ms"] + out["masked_softmax"]["ms"] + out["nn"]["ms"]
    return out


if __name__ == "__main__":
    main()
