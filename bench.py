#!/usr/bin/env python
"""bench.py — ESKF iterations / second of the B200-native LINS IESKF update path.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W [--impl reference]`.
  * workload: BASELINE.json configs[2] "synthetic 1000-scan sequence, flat-ground map" — 1000 independent
    (scan pair, prior) units per GPU (configs[1], the real bag, is not available: no dataset, no network);
    a STEP = one pass of the whole iterated update (performIESKF, all iterations) over the 1000 resident units.
  * value  = ESKF iterations executed by all ranks per second, inputs already resident in HBM (device-timed
    with CUDA events on the launching stream, max over ranks); one fused kernel launch per step.
  * e2e    = the same metric through the reference-facing C-ABI call lins_gpu_ieskf_batch with HOST buffers
    (pack + H2D + kernel + D2H inside the timed region).
  * roofline = dominant kernel (the fused IESKF kernel).  It is instruction-issue bound (a search / f64-algebra kernel
    that lives in shared memory and L2), so `bound` is "issue": warp instructions per launch (committed ncu capture)
    / the launch duration measured live, against 148 SMs x 4 schedulers x the SM clock.  roofline_hbm is the same launch
    against MEASURED_PEAKS.json hbm_gbs (algorithmic bytes), roofline_jacobian the split Jacobian kernel (SURVEY.md §8(d) U1).
  * cpu_baseline = the CPU oracle (a port of the reference path: it cannot be compiled here), rows (i) one pinned thread,
    reference-faithful M x M gain, (ii) one thread, 18 x 18 form, (iii) all cores scan-parallel (both forms, best of a
    thread sweep), on bounded samples of GPU batch 0.
  * --impl reference: the oracle arm timed alone (rank 0 only under torchrun) on the first units of the SAME batch.
  * parity_sample: after the timed region, units of every resident batch are re-run through the oracle and compared.
  * --dump-outputs DIR: what the last timed step computed (rank 0's states, covariances, result records) as DIR/*.npy;
    the inputs are seeded, so two builds run with the same arguments can be compared output for output.
L2 hygiene: three different 1000-unit batches (3 x ~87 MB > 126 MB L2) are resident and used round-robin, so
no step finds its inputs in L2.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SCANS_PER_GPU = 1000
WORKLOAD = "config3: synthetic 1000-scan flat-ground sequence (BASELINE.json configs[2]), 16x1800 VLP-16, shipped exp_port.yaml params (num_iter 30)"


def pkg(name):
    return importlib.import_module("lins---lidar-inertial-slam_b200." + name)


NB = 3  # resident batches per GPU, used round-robin


def bench_config(n, world):
    """The `config` object of the JSON line — identical for both arms (--impl ours / reference)."""
    return {"workload": WORKLOAD, "scans_per_gpu_per_step": n, "unit_seeds": "1000 + 100000*rank + 10000*batch + unit",
            "l2": f"{NB} resident batches used round-robin ({NB} x ~84 MB > 126 MB L2)",
            "parallelism": f"scan-sharded x{world}, one pose all_gather after the last step" if world > 1 else "1 GPU"}


def host_info():
    model = "unknown"
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                model = ln.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return {"nproc": os.cpu_count() or 1, "cpu_model": model}


def bind_to_gpu_numa_node(local):
    """Pin this rank (and every thread it starts: the generator's, the library's pack pool) to the CPUs of the NUMA node its
    GPU hangs off, so that the host clouds — first touched by these threads — and the pinned staging are node-local to the
    GPU's PCIe root.  What a replay job with one rank per GPU does; returns a description for the JSON line."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return f"{bdf}: no NUMA affinity reported"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return f"{bdf}: node {node} has no allowed CPUs"
        os.sched_setaffinity(0, cpus)
        return f"GPU {local} ({bdf}) -> NUMA node {node}, {len(cpus)} CPUs"
    except (OSError, ValueError, AttributeError) as e:
        return f"not bound ({type(e).__name__})"


def host_memory_policy(interleave):
    """set_mempolicy(MPOL_INTERLEAVE over the online NUMA nodes) / (MPOL_DEFAULT) for what this process allocates from here
    on: what `numactl --interleave=all` does for a replay job's host clouds and the library's pinned staging.  The pack
    threads and the copy engines read them from both sockets; with first-touch placement the end-to-end rate depended on
    which socket the clouds happened to land on (measured on the 2-socket B200 host, 3 contexts x 21 pack threads:
    5.6-6.2 M it/s first-touch, 7.7-7.9 M interleaved).  The CPU arms keep the default policy (thread-private matrices)."""
    try:
        import ctypes
        nodes = []
        for part in open("/sys/devices/system/node/online").read().strip().split(","):
            a, _, b = part.partition("-")
            nodes += list(range(int(a), int(b or a) + 1))
        if len(nodes) < 2:
            return "one NUMA node"
        libc = ctypes.CDLL(None, use_errno=True)
        if interleave:
            mask = ctypes.c_ulong(sum(1 << n for n in nodes))
            rc = libc.syscall(ctypes.c_long(238), ctypes.c_long(3), ctypes.byref(mask), ctypes.c_ulong(max(nodes) + 2))  # x86-64 set_mempolicy, MPOL_INTERLEAVE
        else:
            rc = libc.syscall(ctypes.c_long(238), ctypes.c_long(0), None, ctypes.c_ulong(0))  # MPOL_DEFAULT
        if rc != 0:
            return f"set_mempolicy refused (errno {ctypes.get_errno()})"
        return f"host buffers interleaved over NUMA nodes {nodes}" if interleave else "default policy"
    except (OSError, ValueError, AttributeError) as e:
        return f"not interleaved ({type(e).__name__})"


def thread_sweep(cores):
    return sorted({max(1, cores // 4), max(1, cores // 2), cores})


def oracle_rate(ob, prm, batch, count, form, threads, pin_core=None):
    """iterations/s of the oracle over the first `count` units of `batch` (optionally with the process pinned to one core)."""
    old = None
    if pin_core is not None and hasattr(os, "sched_setaffinity"):
        old = os.sched_getaffinity(0)
        os.sched_setaffinity(0, {sorted(old)[pin_core % len(old)]})
    try:
        _, _, _, sec, its = ob.ieskf_batch(prm, batch, count=count, form=form, threads=threads, want_cov=True)
    finally:
        if old is not None:
            os.sched_setaffinity(0, old)
    return its / sec, its, sec


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.lines, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


def algorithmic_bytes(batch, iters):
    """Compulsory HBM bytes of one fused launch over `batch` (DESIGN.md §Kernels): every query / target point
    once per scan (16 B packed), prior in, posterior out, the correspondence IDs written every iteration
    (`iters` = per-scan iteration counts)."""
    ns = np.diff(batch.offsets["surf_flat"]).astype(np.int64)
    nc = np.diff(batch.offsets["corner_sharp"]).astype(np.int64)
    ts = np.diff(batch.offsets["surf_less_flat"]).astype(np.int64)
    tc = np.diff(batch.offsets["corner_less_sharp"]).astype(np.int64)
    per_scan = 16 * (ns + nc + ts + tc) + (20 + 324) * 8 + (20 + 324) * 8 + 64 + 4 * (3 * ns + 2 * nc) * np.asarray(iters, np.int64)
    return int(per_scan.sum())


def profiled(key, field="dram_bytes_per_launch"):
    """A per-launch figure of the named kernel from the committed `ncu --set full` capture of this same command
    (profiles/traffic.json, written by tools/ncu_summary.py); None when no capture is recorded."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return float(json.load(f)[key][field])
    except (OSError, KeyError, ValueError, TypeError):
        return None


def profiled_traffic(key):
    return profiled(key)


def jacobian_bytes(batch):
    """SURVEY.md §8(d) U1: 76 B per surf query + 56 B per corner query + 384 B per scan."""
    ns = int(batch.offsets["surf_flat"][-1]); nc = int(batch.offsets["corner_sharp"][-1])
    return 76 * ns + 56 * nc + 384 * batch.n


DUMP_MAX_BYTES = 64_000_000


def dump_outputs(out_dir, states, covs, res, max_bytes=DUMP_MAX_BYTES):
    """Write what lins_gpu_batch_download hands the caller of one step (posterior states, exit covariances and the fields
    of the 64-B result records) as out_dir/<name>.npy in float64, so that two builds can be compared output for output.
    Above max_bytes a fixed, seeded sample of the units is written (in unit order; scan_id names each one)."""
    arrays = {"state": states, "cov": covs, "scan_id": res["scan_id"], "iters": res["iters"], "flags": res["flags"], "pose": res["pose"]}
    n = len(res)
    row_bytes = sum(8 * (np.asarray(a).size // max(1, n)) for a in arrays.values())
    keep = (max_bytes - 1024 * len(arrays)) // row_bytes  # (room for the .npy headers)
    idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False)) if n > keep else np.arange(n)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64)[idx])
    return sorted(arrays)


def reference_arm(args, rank, world):
    """--impl reference: the CPU oracle (port of the reference path; the reference itself needs ROS/PCL/Eigen and
    cannot be built here), reference-faithful M x M gain, scan-parallel over the host cores (best of a thread sweep),
    on the first units of the SAME batch the GPU arm's rank 0 processes (seeds 1000...)."""
    if rank != 0:
        return
    from oracle import oracle_binding as ob
    synth = pkg("synth")
    hi = host_info()
    cores = hi["nproc"]
    sample = max(cores, min(256, 2 * cores))
    b = synth.generate("config3", n=sample, seed0=1000)  # = the first `sample` units of GPU batch 0 on rank 0
    prm = ob.LinsParams.shipped()
    for _ in range(max(1, min(args.warmup, 1))):
        ob.ieskf_batch(prm, b, count=min(sample, cores), form=ob.FORM_A, threads=cores, want_cov=False)
    sweep = {}
    for t in thread_sweep(cores):
        tot_it, tot_s = 0, 0.0
        for _ in range(args.steps):
            _, its, sec = oracle_rate(ob, prm, b, sample, ob.FORM_A, t)
            tot_it += its; tot_s += sec
        sweep[t] = (tot_it / tot_s, tot_s)
    best_t = max(sweep, key=lambda t: sweep[t][0])
    val, tot_s = sweep[best_t]
    out = {
        "impl": "reference", "metric": "ESKF iterations/sec", "value": val, "unit": "iterations/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot_s / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64 (f32 association)", "data": "synthetic",
        "config": bench_config(args.scans, world),
        "cpu_baseline": {"value": val, "unit": "iterations/s", "cores": best_t, "kind": "port", **hi,
                         "sample": f"first {sample} units of batch 0 (seeds 1000..{1000 + sample - 1}) x {args.steps} steps per thread count; reference-faithful MxM Kalman gain (StateEstimator.hpp:542-546), kd-tree 1-NN, scan-parallel std::thread",
                         "thread_sweep_iters_per_s": {str(t): v[0] for t, v in sweep.items()}},
        "e2e": {"value": val, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scans", type=int, default=SCANS_PER_GPU, help="units per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write rank 0's outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; the reference arm has none to write")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    capi, synth, defs = pkg("capi"), pkg("synth"), pkg("ctypes_defs")
    prm = defs.LinsParams.shipped()
    # (opt-in: measured on the 2-socket B200 host it LOWERED the 2-GPU e2e — 12.2 -> 9.8 M it/s with host pack, 7.7 -> 6.1 M
    # with raw DMA — because it halves the CPUs the rank's pack threads and copy threads may use)
    numa = bind_to_gpu_numa_node(local) if world > 1 and os.environ.get("LINS_NUMA_BIND", "0") == "1" else "not bound"
    # The replay job's host buffers are interleaved over the NUMA nodes (pack threads and copy engines read them from both
    # sockets).  Measured: 1 GPU 5.6-6.2 M it/s first-touch -> 7.7-7.9 M interleaved (five runs of five); 2 GPUs on one box,
    # one run each: 7.1 M first-touch, 7.5 M interleaved.  LINS_NUMA_INTERLEAVE=0 turns it off.
    if os.environ.get("LINS_NUMA_INTERLEAVE", "1") != "0":  # (the CPU legs below reset the policy)
        numa += "; " + host_memory_policy(True)
    # host threads each lins_gpu_batch_upload may use for packing: the cores are shared by `world` ranks x 3 contexts
    os.environ.setdefault("LINS_PACK_THREADS", str(max(2, min(32, (os.cpu_count() or 8) // (max(1, int(os.environ.get("LOCAL_WORLD_SIZE", world))) * 6)))))
    # a non-default torch stream: its handle is non-NULL, so the library launches on it (NULL would make the
    # library create its own stream and torch.cuda.Event would not see the kernels)
    stream = torch.cuda.Stream(device=local)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    # one stream per resident batch: consecutive steps touch different batches, so the persistent kernel of step k+1
    # moves onto the SMs that step k's last (longest) scans no longer occupy instead of waiting for the whole grid
    bstreams = [torch.cuda.Stream(device=local) for _ in range(NB)]

    # ---- inputs: 3 resident batches of `scans` units each; weak scaling = different seeds per rank ----------
    n = args.scans
    batches = [synth.generate("config3", n=n, seed0=1000 + 100000 * rank + 10000 * k) for k in range(NB)]
    ctxs = [capi.LinsGpu(prm, device=local, stream=bstreams[k].cuda_stream) for k in range(NB)]
    for c, b in zip(ctxs, batches):
        c.batch_upload(b)
    torch.cuda.synchronize()

    class _DevView:  # zero-copy torch view of the resident result records (64 B / scan)
        def __init__(self, ptr, nbytes):
            self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}

    res_views = []
    for c in ctxs:
        p, nn = c.batch_results_device()
        res_views.append(torch.as_tensor(_DevView(p, nn * 64), device=f"cuda:{local}"))

    gathered = [torch.empty(world * n * 64, dtype=torch.uint8, device=f"cuda:{local}") for _ in range(NB)] if world > 1 else None

    def step(k):
        j = k % NB
        with torch.cuda.stream(bstreams[j]):
            ctxs[j].batch_run()  # one fused kernel launch on that batch's stream

    def gather_poses():
        # the path's ONLY exchange (north_star: "NCCL gather of poses only at the end"): the 64-B result records of the
        # resident batches, once after the last step, each ordered after its batch's last kernel on that batch's stream
        if world > 1:
            for j in range(NB):
                with torch.cuda.stream(bstreams[j]):
                    dist.all_gather_into_tensor(gathered[j], res_views[j])

    for k in range(max(args.warmup, NB)):
        step(k)
    gather_poses()
    torch.cuda.synchronize()
    iters_per_batch, iters_per_scan = [], []
    for c in ctxs:
        _, _, res, _ = c.batch_download(states=False, covs=False)
        iters_per_batch.append(int(res["iters"].sum()))
        iters_per_scan.append(res["iters"].astype(np.int64))

    # ---- timed region: exactly K steps ----------------------------------------------------------------------
    launches0 = sum(c.launch_count() for c in ctxs)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
        time.sleep(0.3)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)  # the device is idle here; every batch stream starts after this event ...
    for st in bstreams:
        st.wait_event(e0)
    for k in range(args.steps):
        step(k)
    gather_poses()
    for st in bstreams:  # ... and the end event waits for all of them
        done = torch.cuda.Event()
        done.record(st)
        stream.wait_event(done)
    e1.record(stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clk = clocks.stop() if rank == 0 else None
    elapsed_ms = e0.elapsed_time(e1)
    # launches of consecutive steps overlap at their tails, so a per-launch event pair would also count the time a
    # launch waits for SMs: the effective duration per launch is the timed region divided by its launches
    kernel_ms = [elapsed_ms / args.steps] * args.steps
    launches = sum(c.launch_count() for c in ctxs) - launches0
    my_iters = sum(iters_per_batch[k % NB] for k in range(args.steps))
    t = torch.tensor([elapsed_ms, float(my_iters), float(launches)], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        elapsed_ms, total_iters, total_launches = float(tmax[0]), float(tsum[1]), int(tsum[2])
    else:
        total_iters, total_launches = float(my_iters), launches
    value = total_iters / (elapsed_ms * 1e-3)
    if args.dump_outputs and rank == 0:  # (before the e2e legs below re-use these contexts)
        so, co, res, _ = ctxs[(args.steps - 1) % NB].batch_download(states=True, covs=True)
        dump_outputs(args.dump_outputs, so, co, res)

    # ---- end to end through the C-ABI with host buffers (pack + H2D + kernel + D2H timed) ------------------------
    # The user-facing call is lins_gpu_ieskf_batch(ctx, host batch) -> host results (synchronous: pack, H2D, the
    # fused kernel, D2H).  A replay job keeps NB contexts busy from NB host threads (ctypes drops the GIL), so one
    # batch's packing / PCIe traffic overlaps another's kernel; every step still moves all its bytes both ways.
    import threading
    # calls in flight (each is synchronous).  Measured on the B200 box (128 host cores): 3 contexts 3.8 M it/s,
    # 6 contexts 2.1 M, 9 contexts 2.2 M — more host threads than that only contend
    NE = int(os.environ.get("LINS_E2E_CONTEXTS", "3"))
    # (a step is 2-4 ms: a short sample mostly times the start of the worker threads; 8 x steps keeps the spread under a few %)
    e2e_steps = max(NE, int(os.environ.get("LINS_E2E_STEPS", 8 * args.steps)))
    e2e_streams = [torch.cuda.Stream(device=local) for _ in range(max(0, NE - NB))]  # (kept alive until the end of main)
    e2e_ctxs = (ctxs + [capi.LinsGpu(prm, device=local, stream=st.cuda_stream) for st in e2e_streams])[:NE]
    # the replay job's host clouds are page-locked once (lins_gpu_host_register): the library then DMAs the raw 32-B
    # PointXYZI records straight from them and packs on the device — no host pass over the points (LINS_E2E_PINNED=0:
    # pageable clouds, packed by host threads into the library's pinned staging)
    e2e_pinned = os.environ.get("LINS_E2E_PINNED", "1") != "0"
    if e2e_pinned:
        for b in batches:
            capi.pin_batch(b)
    for c in e2e_ctxs:
        for b in batches:  # warm: each context's pinned staging grows to the largest batch before the timed region
            c.ieskf_batch(b)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e2e_counts = [0] * NE
    up0 = [c.batch_upload_stats() for c in e2e_ctxs]

    def e2e_worker(j):
        for k in range(j, e2e_steps, NE):
            _, _, res = e2e_ctxs[j].ieskf_batch(batches[k % NB])
            e2e_counts[j] += int(res["iters"].sum())

    workers = [threading.Thread(target=e2e_worker, args=(j,)) for j in range(NE)]
    t0 = time.perf_counter()
    for w in workers:
        w.start()
    for w in workers:
        w.join()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_iters = sum(e2e_counts)
    te = torch.tensor([e2e_s, float(e2e_iters)], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        a = te.clone(); dist.all_reduce(a, op=dist.ReduceOp.MAX)
        s = te.clone(); dist.all_reduce(s, op=dist.ReduceOp.SUM)
        e2e_s, e2e_iters = float(a[0]), float(s[1])
    if e2e_pinned:
        for b in batches:
            capi.unpin_batch(b)
    # the same job when the caller keeps its clouds as page-locked 16-byte (x, y, z, intensity) records
    # (lins_batch_desc.point_format = LINS_POINTS_PACKED16): one DMA per slice, no host pass, half the raw path's bytes
    pbatches = [b.packed16() for b in batches]
    for pb in pbatches:
        capi.pin_batch(pb)
    for c in e2e_ctxs:
        c.ieskf_batch(pbatches[0])
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    p16_counts = [0] * NE

    def p16_worker(j):
        for k in range(j, e2e_steps, NE):
            _, _, res = e2e_ctxs[j].ieskf_batch(pbatches[k % NB])
            p16_counts[j] += int(res["iters"].sum())

    workers = [threading.Thread(target=p16_worker, args=(j,)) for j in range(NE)]
    t0 = time.perf_counter()
    for w in workers:
        w.start()
    for w in workers:
        w.join()
    torch.cuda.synchronize()
    p16_s = time.perf_counter() - t0
    tp = torch.tensor([p16_s, float(sum(p16_counts))], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        a = tp.clone(); dist.all_reduce(a, op=dist.ReduceOp.MAX)
        s_ = tp.clone(); dist.all_reduce(s_, op=dist.ReduceOp.SUM)
        tp = torch.stack([a[0], s_[1]])
    e2e_p16 = float(tp[1]) / float(tp[0])
    for pb in pbatches:
        capi.unpin_batch(pb)
    del pbatches
    host_memory_policy(False)  # (the oracle legs below allocate thread-private matrices: first-touch placement)
    b0 = batches[0]
    pts = sum(int(b0.offsets[k][-1]) for k in b0.FIELDS)
    # caller-pinned clouds are split at run time between the pack threads (16 B / point over PCIe) and the copy engine (raw
    # 32 B / point, packed on the device): count what actually went which way in the timed region
    pack_threads = int(os.environ.get("LINS_PACK_THREADS", "8"))
    up1 = [c.batch_upload_stats() for c in e2e_ctxs]
    packed_pts = sum(b_[0] - a_[0] for a_, b_ in zip(up0, up1)); raw_pts = sum(b_[1] - a_[1] for a_, b_ in zip(up0, up1))
    raw_frac = raw_pts / max(1, packed_pts + raw_pts)
    upload_mode = (f"caller-pinned 32-B PointXYZI clouds: {100 * (1 - raw_frac):.0f} % of the points packed to 16 B by {pack_threads} host threads per context, "
                   f"{100 * raw_frac:.0f} % DMA'd raw and packed on the device (LINS_UPLOAD={os.environ.get('LINS_UPLOAD', 'default')})") if e2e_pinned else \
                  f"pageable 32-B PointXYZI clouds packed to 16 B by {pack_threads} host threads per context into pinned staging"
    h2d = int((16 * packed_pts + 32 * raw_pts) / max(1, e2e_steps)) + 4 * 4 * (n + 1) + n * (20 + 324) * 8
    d2h = n * ((20 + 324) * 8 + 64)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel + the split Jacobian kernel (rank 0, N-independent) ----------------------
    peak, peak_src = measured_peak()
    alg = float(np.mean([algorithmic_bytes(batches[k % NB], iters_per_scan[k % NB]) for k in range(args.steps)]))
    kms = float(np.mean(kernel_ms))
    achieved = alg / (kms * 1e-3) / 1e9
    kname = "lins_ieskf_kernel<MODE_IESKF> (fused de-skew + 1-NN + ring walks + residual/Jacobian fold + 6x6 gain solve, all iterations)"
    roofline_hbm = {"kernel": kname, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": profiled_traffic("fused"), "peak_source": peak_src, "algorithmic_bytes_per_launch": alg, "avg_launch_ms": kms,
                    "note": "secondary: the kernel is not bandwidth bound (per unit ~90 KB of compulsory bytes feed ~17 iterations of searches served from shared memory / L2)"}
    # the honest bound: instruction issue.  Warp instructions per launch come from the committed ncu capture of this
    # command (smsp__inst_executed.sum of one 1000-unit launch, scaled by the iterations this step really ran); the
    # duration is the live measurement above; the peak is one warp instruction per scheduler per cycle.
    inst = profiled("fused", "warp_instructions_per_launch")
    inst_iters = profiled("fused", "iterations_of_profiled_launch")
    sm_mhz = (clk or {}).get("sm_mhz") or 1965.0
    issue_peak = 148 * 4 * sm_mhz * 1e6 / 1e9  # G warp-instructions / s
    if inst:
        if inst_iters:
            inst = inst * float(np.mean(iters_per_batch)) / inst_iters
        issue_ach = inst / (kms * 1e-3) / 1e9
        roofline = {"kernel": kname, "bound": "issue", "achieved": issue_ach, "peak": issue_peak, "unit": "Gwarp-inst/s", "frac": issue_ach / issue_peak,
                    "traffic": profiled_traffic("fused"), "warp_instructions_per_launch": inst, "avg_launch_ms": kms,
                    "peak_source": f"148 SMs x 4 schedulers x {sm_mhz:.0f} MHz (1 warp instruction / scheduler / cycle)",
                    "note": "instruction-issue bound search + f64 algebra kernel; instruction count from profiles/traffic.json (ncu smsp__inst_executed.sum), duration measured live; HBM view in roofline_hbm"}
    else:
        roofline = dict(roofline_hbm, note="no committed instruction count: HBM view only")
    # Jacobian kernel: tile the resident batch past L2 and time the split kernel alone
    jb = batches[0].tile(5)
    jctx = capi.LinsGpu(prm, device=local, stream=stream.cuda_stream)
    jctx.batch_upload(jb); jctx.batch_run(); torch.cuda.synchronize()
    for _ in range(3):
        jctx.batch_jacobian_pass()
    torch.cuda.synchronize()
    ja, jb_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    ja.record()
    for _ in range(reps):
        jctx.batch_jacobian_pass()
    jb_.record(); torch.cuda.synchronize()
    jms = ja.elapsed_time(jb_) / reps
    jbytes = jacobian_bytes(jb)
    roofline_j = {"kernel": "lins_jacobian_kernel (SURVEY.md §8(d) unit U1, given correspondence IDs)", "bound": "hbm", "achieved": jbytes / (jms * 1e-3) / 1e9,
                  "peak": peak, "unit": "GB/s", "frac": jbytes / (jms * 1e-3) / 1e9 / peak, "traffic": profiled_traffic("jacobian"), "scans": jb.n, "avg_launch_ms": jms,
                  "algorithmic_bytes_per_launch": jbytes, "working_set_mb": (16 * sum(int(jb.offsets[k][-1]) for k in jb.FIELDS)) / 1e6}
    jctx.close()

    # ---- row F2 (SURVEY.md §8(f)): the mapping node's scan-to-map refinement, one 50-key-frame unit ---------------------
    mu = synth.generate_map_unit("config3", seed=40, n_keyframes=50, sigma_t=0.1, sigma_r=0.01)
    mctx = capi.LinsGpu(prm, device=local, stream=stream.cuda_stream)
    mctx.map_set(mu.corner_map, mu.surf_map)
    for _ in range(2):
        mctx.scan2map(mu.corner_last, mu.surf_last, mu.guess)
    torch.cuda.synchronize()
    mreps = 10
    t0 = time.perf_counter()
    for _ in range(mreps):
        mT, mrep = mctx.scan2map(mu.corner_last, mu.surf_last, mu.guess)  # synchronous: H2D of the features, <= 10 x (5-NN, fits, reduce, D2H, LM)
    mapping_ms = (time.perf_counter() - t0) * 1e3 / mreps
    nq_map = len(mu.corner_last) + len(mu.surf_last)
    dist_evals = (len(mu.corner_last) * len(mu.corner_map) + len(mu.surf_last) * len(mu.surf_map)) * mrep.iters
    mapping = {"what": "lins_gpu_scan2map (lidar_mapping_node.cpp:1635-1652): exact hashed-grid 5-NN + line / plane fits + the LM loop on the device (one D2H + one sync per call), host buffers in / out",
               "map_points": int(len(mu.corner_map) + len(mu.surf_map)), "feature_points": int(nq_map), "lm_iterations": int(mrep.iters),
               "converged": int(mrep.converged), "ms_per_call": mapping_ms, "brute_force_equivalent_distance_evaluations_per_s": dist_evals / (mapping_ms * 1e-3),
               "translation_error_m": {"before": float(np.abs(mu.guess[3:] - mu.truth[3:]).max()), "after": float(np.abs(mT[3:] - mu.truth[3:]).max())}}
    mctx.close()

    # ---- CPU baseline (rank 0, N = 1 only): oracle on the host cores, bounded samples of batch 0 ------------------------
    cpu = None
    extras = {}
    if world == 1 and not args.no_cpu_baseline:
        from oracle import oracle_binding as ob
        hi = host_info()
        cores = hi["nproc"]
        sample = max(cores, min(256, 2 * cores))
        sweepA, sweepB = {}, {}
        for t in thread_sweep(cores):
            sweepA[t] = oracle_rate(ob, prm, batches[0], sample, ob.FORM_A, t)[0]
            sweepB[t] = oracle_rate(ob, prm, batches[0], n, ob.FORM_B, t)[0]
        tA = max(sweepA, key=sweepA.get); tB = max(sweepB, key=sweepB.get)
        rate_i = oracle_rate(ob, prm, batches[0], 6, ob.FORM_A, 1, pin_core=0)[0]     # row (i): the north_star's ">= 50x" denominator
        rate_ii = oracle_rate(ob, prm, batches[0], 256, ob.FORM_B, 1, pin_core=0)[0]  # row (ii)
        cpu = {"value": sweepA[tA], "unit": "iterations/s", "cores": tA, "kind": "port", **hi,
               "sample": f"first {sample} units of batch 0; reference-faithful MxM gain (form A, StateEstimator.hpp:542-546), kd-tree 1-NN, best of {sorted(sweepA)} scan-parallel threads",
               "row_i_form_a_1thread_pinned_iters_per_s": rate_i, "row_ii_form_b_18x18_1thread_pinned_iters_per_s": rate_ii,
               "row_iii_form_b_18x18_allcores_iters_per_s": sweepB[tB], "row_iii_threads": tB,
               "thread_sweep_form_a": {str(t): v for t, v in sweepA.items()}, "thread_sweep_form_b": {str(t): v for t, v in sweepB.items()},
               "gpu_e2e_over_row_i": (e2e_iters / e2e_s) / rate_i}
        mo = ob.MapOracle()
        mo.set_map(mu.corner_map, mu.surf_map)
        t0 = time.perf_counter()
        moT, morep = mo.scan2map(mu.corner_last, mu.surf_last, mu.guess)
        mapping["cpu_port_bruteforce_ms_per_call"] = (time.perf_counter() - t0) * 1e3  # 1 thread, BRUTE-FORCE 5-NN (the oracle's exact search; NOT what the reference costs)
        # the reference searches with kd-trees (lidar_mapping_node.cpp:1368, :1475): a like-for-like CPU figure for the search part
        from scipy.spatial import cKDTree
        xyz = lambda c: np.stack([c["x"], c["y"], c["z"]], 1).astype(np.float64)  # noqa: E731
        t0 = time.perf_counter()
        tc_, ts_ = cKDTree(xyz(mu.corner_map)), cKDTree(xyz(mu.surf_map))
        t_build = time.perf_counter() - t0
        t0 = time.perf_counter()
        for _ in range(int(mrep.iters)):
            tc_.query(xyz(mu.corner_last), k=5); ts_.query(xyz(mu.surf_last), k=5)
        mapping["cpu_kdtree_search_ms_per_call"] = {"build": t_build * 1e3, "queries": (time.perf_counter() - t0) * 1e3, "what": "scipy cKDTree, 1 thread, 5-NN of every feature point x LM iterations (search only, no fits)"}
        mapping["max_abs_transform_diff_vs_cpu_port"] = float(np.abs(moT - mT).max())

        # ---- parity sample: units of every resident batch, as the timed steps left them, against the oracle ----------------
        nchk = 64
        worst, iters_equal, flags_equal, checked = 0.0, True, True, 0
        for c, bt in zip(ctxs, batches):
            c.batch_run(); c.sync()
            sg, _, rg, _ = c.batch_download(states=True, covs=False)
            idx = np.linspace(0, bt.n - 1, nchk).astype(int)
            so, _, ro, _, _ = ob.ieskf_batch(prm, bt.subset(idx), form=ob.FORM_B, threads=min(cores, nchk), want_cov=False)
            worst = max(worst, float(np.abs(sg[idx] - so).max()))
            iters_equal &= bool(np.array_equal(rg["iters"][idx], ro["iters"]))
            flags_equal &= bool(np.array_equal(rg["flags"][idx], ro["flags"]))
            checked += len(idx)
        extras["parity_sample"] = {"units": checked, "max_state_diff": worst, "iters_equal": iters_equal, "flags_equal": flags_equal,
                                   "oracle": "brute-force-equivalent kd-tree 1-NN, 18x18 form; tolerance 1e-7 (north_star 1e-4)"}

        # ---- config 4 (64 x 1024, SURVEY.md §8(d)) and the single-scan seam latency (config 1) ---------------------------
        b4 = synth.generate("config4", n=148, seed0=7000).tile(4)  # 4 units per SM: one per SM would time the slowest unit, not throughput
        c4 = capi.LinsGpu(prm, device=local, stream=stream.cuda_stream)
        c4.batch_upload(b4)
        for _ in range(2):
            c4.batch_run()
        c4.sync()
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record(stream)
        for _ in range(3):
            c4.batch_run()
        eb.record(stream); torch.cuda.synchronize()
        _, _, r4, _ = c4.batch_download(states=False, covs=False)
        ms4 = ea.elapsed_time(eb) / 3
        it4 = int(r4["iters"].sum())
        o4 = oracle_rate(ob, prm, b4, min(148, cores), ob.FORM_B, min(148, cores))[0]
        extras["config4"] = {"what": "BASELINE.json configs[3]: 64 x 1024 dense scans, 592 units (148 distinct scans x 4), one fused launch", "units": b4.n,
                             "queries_per_unit": float((b4.offsets["surf_flat"][-1] + b4.offsets["corner_sharp"][-1]) / b4.n),
                             "targets_per_unit": float((b4.offsets["surf_less_flat"][-1] + b4.offsets["corner_less_sharp"][-1]) / b4.n),
                             "ms_per_launch": ms4, "iterations": it4, "iterations_per_s": it4 / (ms4 * 1e-3),
                             "cpu_form_b_allcores_iterations_per_s": o4}
        c4.close()
        b1 = synth.generate("config1", n=1, seed0=1)
        u1 = b1.unit(0)
        c1 = capi.LinsGpu(prm, device=local, stream=stream.cuda_stream)
        c1.set_map(u1["surf_less_flat"], u1["corner_less_sharp"])
        lat, lat_upd, lat_dev = [], [], []
        sl, cl = u1["surf_less_flat"].copy(), u1["corner_less_sharp"].copy()
        for k in range(30):
            t0 = time.perf_counter()
            s1, _, rep1 = c1.ieskf(u1["surf_flat"], u1["corner_sharp"], u1["state"], u1["cov"])
            t1 = time.perf_counter()
            if k % 2 == 0:
                c1.L.lins_gpu_update_map(c1.h, sl.ctypes.data, len(sl), cl.ctypes.data, len(cl), s1.ctypes.data, None)  # in place, read back
            else:
                c1.update_map_device(u1["surf_less_flat"], u1["corner_less_sharp"])  # device posterior, no read-back, no sync
            t2 = time.perf_counter()
            c1.sync()
            c1.set_map(u1["surf_less_flat"], u1["corner_less_sharp"])
            sl[:] = u1["surf_less_flat"]; cl[:] = u1["corner_less_sharp"]
            if k >= 6:
                lat.append((t1 - t0) * 1e6)
                (lat_upd if k % 2 == 0 else lat_dev).append((t2 - t1) * 1e6)
        o1 = ob.Oracle(prm); o1.set_map(u1["surf_less_flat"], u1["corner_less_sharp"])
        t0 = time.perf_counter(); o1.ieskf(u1["surf_flat"], u1["corner_sharp"], u1["state"], u1["cov"], form=ob.FORM_A); tA1 = (time.perf_counter() - t0) * 1e6
        t0 = time.perf_counter(); o1.ieskf(u1["surf_flat"], u1["corner_sharp"], u1["state"], u1["cov"], form=ob.FORM_B); tB1 = (time.perf_counter() - t0) * 1e6
        extras["single_scan_latency_us"] = {"what": "config 1 through the drop-in seam (StateEstimator.hpp:435-463): lins_gpu_ieskf then lins_gpu_update_map, host buffers, synchronous",
                                            "ieskf_median": float(np.median(lat)), "update_map_median": float(np.median(lat_upd)),
                                            "update_map_device_resident_median": float(np.median(lat_dev)), "iterations": int(rep1.iters),
                                            "cpu_port_form_a_us": tA1, "cpu_port_form_b_us": tB1}
        c1.close()

    out = {
        "metric": "ESKF iterations/sec", "value": value, "unit": "iterations/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64 (f32 association)", "data": "synthetic",
        "config": bench_config(n, world),
        "iterations_per_step_rank0": float(np.mean(iters_per_batch)),
        "streams": f"one CUDA stream per resident batch ({NB}): consecutive steps overlap at their kernel tails; e2e = {NE} host threads, one context (and stream) each",
        "clocks": clk,
        "e2e": {"value": e2e_iters / e2e_s, "unit": "iterations/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps, "host_threads": NE, "numa": numa,
                "upload": upload_mode},
        "e2e_packed16": {"value": e2e_p16, "unit": "iterations/s", "h2d_bytes_per_step": 16 * pts + 4 * 4 * (n + 1) + n * (20 + 324) * 8,
                         "what": "same call, caller-pinned 16-byte (x, y, z, intensity) clouds (point_format = LINS_POINTS_PACKED16): not the reference's PointXYZI layout, shown beside the headline e2e"},
        "gpu_launches": int(total_launches),
        "roofline": roofline, "roofline_hbm": roofline_hbm, "roofline_jacobian": roofline_j, "mapping_refinement": mapping,
    }
    out.update(extras)
    if cpu:
        out["cpu_baseline"] = cpu
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
