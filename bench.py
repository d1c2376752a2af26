#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200 NTT + FRI engine (contract: task prompt section 4).

Metric (BASELINE.json): 128-bit field butterflies/sec on 2^20-point NTTs; FRI commit ms @ 2^20.
One "step" = one pass of the hot path over one batch: BATCH independent 2^20-point forward
NTTs (code/ntt.py:3-18) resident in HBM (BATCH * 16 MiB = 256 MiB > the 126 MB L2, so every
step streams from HBM).  butterflies := (n/2) * log2 n per transform.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

N > 1: one process per GPU, every rank transforms its own batch (weak scaling, no data-path
collective); time is the max over ranks.  --impl reference times the CPU oracle port
(oracle/stark_oracle.c, all host threads) on the same workload definition.
--dump-outputs DIR writes a fixed sample of rank 0's last timed step (see dump_outputs) so that
two builds can be compared output for output; the inputs are seeded, so they are the same every run.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True  # the tree may be read-only: no __pycache__ next to the imported modules
for _p in (os.path.join(ROOT, "stark-anatomy_b200"), os.path.join(ROOT, "oracle"), ROOT):
    if _p not in sys.path:
        sys.path.insert(0, _p)

LOG_N = 20
N = 1 << LOG_N
BATCH = 16
BUTTERFLIES_PER_NTT = (N // 2) * LOG_N  # 10 485 760
METRIC = "128-bit field butterflies/sec on 2^20 NTT"
UNIT = "butterflies/s"
FRI_ROUNDS = 12                 # Fri(ef 4, 64 colinearity tests).num_rounds() at 2^20 (fri.py:22-28)
FRI_COMPRESSIONS = 4193268      # leaves + inner nodes of the 12 trees (SURVEY 8d)
FRI_ALG_BYTES = 50315264        # sum_r 16 N_r read + 8 N_r folded written (SURVEY 8d)
WORKLOAD = "batch of %d independent 2^20-point forward NTTs over p=1+407*2^119 (configs[1] size, batched)" % BATCH
DUMP_SAMPLE = 1 << 20           # residues written by --dump-outputs: 32 MiB of limbs + 8 MiB of indices


def config_dict(world):
    """the workload description both arms print (identical keys and values, so the driver's same_config
    comparison holds); "parallelism" describes how the job is cut across the N GPUs of the launch"""
    return {"workload": WORKLOAD, "log_n": LOG_N, "batch_per_gpu": BATCH,
            "l2": "inputs larger than L2: %d MiB in + %d MiB out per step" % (BATCH * 16, BATCH * 16),
            "parallelism": "batch sharded across %d GPU(s), no collective in the timed region" % world}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True).start()
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def dump_outputs(out_dir, y):
    """Write a fixed, seeded sample of the batch `y` (BATCH * N residues, (lo, hi) int64 limb pairs) as
    ntt_out.npy: DUMP_SAMPLE x 4 float64, the 32-bit limbs of each residue, least significant first (float64
    holds them exactly), and ntt_out_index.npy: the flat index (transform * N + position) of each row."""
    import numpy as np
    import torch
    idx = np.sort(np.random.default_rng(0).choice(BATCH * N, DUMP_SAMPLE, replace=False))
    v = y[torch.from_numpy(idx).to(y.device)].cpu().numpy().view(np.uint64)
    limbs = np.stack([v[:, 0] & 0xFFFFFFFF, v[:, 0] >> 32, v[:, 1] & 0xFFFFFFFF, v[:, 1] >> 32], axis=1)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "ntt_out.npy"), limbs.astype(np.float64))
    np.save(os.path.join(out_dir, "ntt_out_index.npy"), idx.astype(np.float64))


def cpu_arm(steps, warmup, batch):
    """the CPU oracle port on all host threads; returns (butterflies/s, threads, seconds/step)"""
    import numpy as np
    import oracle as O
    rng = np.random.default_rng(0)
    x = np.stack([rng.integers(0, 1 << 64, size=(batch, N), dtype=np.uint64),
                  rng.integers(0, 0xCB80000000000000, size=(batch, N), dtype=np.uint64)], axis=2)
    w = O.primitive_nth_root(N)
    # torchrun exports OMP_NUM_THREADS=1: size the team ourselves.  The port is a cache-hostile recursion, so
    # more threads are not always faster on a two-socket host: one probe step per candidate team size, the
    # fastest one is used and reported as `cores` (every thread of that team works: transforms, recursion and
    # combine loops are OpenMP tasks)
    ncpu = os.cpu_count() or 1
    best = None
    for cand in sorted({ncpu, max(1, ncpu // 2), max(1, ncpu // 4), min(ncpu, batch)}, reverse=True):
        O.lib().so_set_threads(cand)
        O.ntt_batch_np(w, x[:min(batch, 4)])  # team start-up
        t0 = time.perf_counter()
        O.ntt_batch_np(w, x)
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, cand)
    O.lib().so_set_threads(best[1])
    threads = O.lib().so_num_threads()
    for _ in range(max(warmup - 1, 0)):
        O.ntt_batch_np(w, x)
    t0 = time.perf_counter()
    for _ in range(steps):
        O.ntt_batch_np(w, x)
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return batch * BUTTERFLIES_PER_NTT / dt, threads, dt


def cpu_fri_commit(reps=2):
    """the CPU oracle port of Fri.commit (fri.py:56-96) on the seed-1 2^20 codeword; the OpenMP team size is
    probed upwards from 8 threads and the fastest one is used (on the two-socket GPU hosts the whole machine is
    SLOWER than one socket's worth of threads on the narrow tree levels); returns (ms per commit, roots, threads)"""
    import numpy as np
    import oracle as O
    rng = np.random.default_rng(1)
    cw = np.stack([rng.integers(0, 1 << 64, size=N, dtype=np.uint64),
                   rng.integers(0, 0xCB80000000000000, size=N, dtype=np.uint64)], axis=1)
    w = O.primitive_nth_root(N)
    ncpu = os.cpu_count() or 1
    best = None
    for cand in sorted({c for c in (8, 16, 32, 64, 128, ncpu) if c <= ncpu} or {ncpu}):
        O.lib().so_set_threads(cand)
        O.merkle_root_np(cw[:1 << 12])  # team start-up
        t0 = time.perf_counter()
        O.fri_commit_np(cw, O.GENERATOR, w, 4, 64)
        dt = time.perf_counter() - t0
        if best is not None and dt > 1.3 * best[0]:
            break  # getting worse: larger teams are not tried
        if best is None or dt < best[0]:
            best = (dt, cand)
    O.lib().so_set_threads(best[1])
    t0 = time.perf_counter()
    for _ in range(reps):
        roots, _, _ = O.fri_commit_np(cw, O.GENERATOR, w, 4, 64)
    return (time.perf_counter() - t0) / reps * 1e3, roots, best[1]


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import __graft_entry__ as G
    G.build_oracle()
    value, threads, dt = cpu_arm(args.steps, args.warmup, BATCH)
    fri_ms, _, fri_threads = cpu_fri_commit()
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u128 mod p (CPU unsigned __int128)", "data": "synthetic",
        "config": config_dict(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "%d steps of %d x 2^20-point ntt, oracle/stark_oracle.c so_ntt_batch: OpenMP tasks, "
                                   "every transform AND the recursion / combine loops inside it are tasks, so all "
                                   "%d threads work although the batch is %d; the reference itself is single-threaded "
                                   "pure Python (5.5e4 butterflies/s, 6 700x slower than this port, BASELINE.md section 2)"
                                   % (args.steps, BATCH, threads, BATCH)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        # second half of BASELINE.json's metric, same arm: Fri.commit of a 2^20 codeword (12 rounds,
        # 4 193 268 blake2b compressions) on the CPU port, all threads
        "fri_commit_ms_2_20": fri_ms,
        "fri_commit": {"ms": fri_ms, "cores": fri_threads, "kind": "port", "compressions_per_s": FRI_COMPRESSIONS / (fri_ms * 1e-3),
                       "sample": "2 commits, oracle so_merkle_tree / so_fri_fold (OpenMP, fastest team size of 8..all "
                                 "threads); the reference's own "
                                 "Fri.commit takes 73 100 ms on one core (BASELINE.md section 2)"},
    }
    print(json.dumps(line))


def allgather_leg(eng, dist, rank, world, w, reps=20):
    """north_star's multi-GPU sentence on the clock: ONE batch of 16 x 2^20 transforms sharded over the N ranks
    (strong scaling: 16 / N transforms per rank) INCLUDING the assembly of the whole batch on every rank, for every
    assembly mode of sa_dist.sharded_ntt.  Device-timed (CUDA events around `reps` calls incl. the cross-rank fence),
    max over ranks; rank 0 checks transforms it does not own against the oracle."""
    import numpy as np
    import torch
    import oracle as O
    import sa_dist
    dev = eng.device
    g = torch.Generator(device=dev)
    g.manual_seed(4321)  # the SAME batch on every rank
    lo = torch.randint(-(1 << 63), (1 << 63) - 1, (BATCH * N,), dtype=torch.int64, device=dev, generator=g)
    hi = torch.randint(0, 0x4B80000000000000, (BATCH * N,), dtype=torch.int64, device=dev, generator=g)
    xg = torch.stack([lo, hi], dim=1).contiguous()
    del lo, hi
    res = {"batch": BATCH, "log_n": LOG_N, "bytes_received_per_rank": (world - 1) * (BATCH // world) * N * 16, "modes": {}}
    peers = None
    try:
        peers = sa_dist.PeerBuffers(BATCH * N)
    except Exception as exc:  # no CUDA IPC in this container: the NCCL modes still run
        res["peer_buffers_error"] = repr(exc)[:300]
    check = sorted({BATCH - 1, BATCH // 2, 0})
    want = {b: O.ntt_np(w, xg[b * N:(b + 1) * N].cpu().numpy().view(np.uint64), parallel=True) for b in check} if rank == 0 else {}
    stream = torch.cuda.current_stream()
    modes = ["nccl", "nccl-pipelined", "p2p-copy", "p2p-store", "p2p-push"]  # (the plain ones first: a fault in a peer mode cannot hide them)
    mcast = None
    if os.environ.get("SA_BENCH_NVLS") == "1":  # NVLS multicast stores (measured slower than unicast: opt-in)
        try:
            mcast = sa_dist.McastBuffers(BATCH * N)
            modes += ["nvls-store", "nvls-push"]
        except Exception as exc:
            res["mcast_buffers_error"] = repr(exc)[:300]
    for mode in modes:
        if mode.startswith("p2p") and peers is None:
            continue
        bufs = mcast if mode.startswith("nvls") else peers
        try:
            def call():
                return sa_dist.sharded_ntt(xg, LOG_N, w, assemble=mode, peers=bufs)
            for _ in range(3):
                full = call()
            torch.cuda.synchronize()
            dist.barrier()
            if rank == 0:
                got = full.cpu().numpy().view(np.uint64)
                for b in check:
                    assert (got[b * N:(b + 1) * N] == want[b]).all(), "assembled batch differs from the oracle (%s, %d)" % (mode, b)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            dist.barrier()
            ev0.record(stream)
            for _ in range(reps):
                full = call()
            ev1.record(stream)
            torch.cuda.synchronize()
            dist.barrier()
            t = torch.tensor([ev0.elapsed_time(ev1) / reps], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            res["modes"][mode] = {"ms_per_call": float(t.item())}
            del full
        except Exception as exc:
            res["modes"][mode] = {"error": repr(exc)[:300]}
            torch.cuda.synchronize()
    for b_ in (peers, mcast):
        if b_ is not None:
            try:
                b_.close()
            except Exception:
                pass
    ok = {m: v["ms_per_call"] for m, v in res["modes"].items() if "ms_per_call" in v}
    if ok:
        best = min(ok, key=ok.get)
        res.update({"mode": best, "ms_per_call": ok[best], "value": BATCH * BUTTERFLIES_PER_NTT / (ok[best] * 1e-3),
                    "unit": UNIT, "scaling": "strong (one 16 x 2^20 batch over all ranks, result assembled on every rank)",
                    "received_gbs_per_rank": res["bytes_received_per_rank"] / (ok[best] * 1e-3) / 1e9})
    return res


def run_ours(args):
    import numpy as np
    import torch
    import __graft_entry__ as G
    G._paths()
    import sa_engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist = None
    # stdout carries exactly ONE JSON line: everything else that writes to fd 1 during the run
    # (NCCL's version banner, library chatter) is pointed at stderr, the line goes to the saved fd
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    eng = sa_engine.get_engine()
    lib = eng.lib
    dev = eng.device
    peak, peak_src = measured_peaks()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- inputs resident in HBM: BATCH * 16 MiB, canonical residues, per-rank seed
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    lo = torch.randint(-(1 << 63), (1 << 63) - 1, (BATCH * N,), dtype=torch.int64, device=dev, generator=g)
    hi = torch.randint(0, 0x4B80000000000000, (BATCH * N,), dtype=torch.int64, device=dev, generator=g)
    x = torch.stack([lo, hi], dim=1).contiguous()  # hi limb < 2^63 < p's top limb: canonical
    y = torch.empty_like(x)
    import oracle as O
    O.lib().so_set_threads(os.cpu_count() or 1)  # torchrun exports OMP_NUM_THREADS=1
    w = O.primitive_nth_root(N)
    root = sa_engine._limbs(w)
    stream = torch.cuda.current_stream()

    def step():
        rc = lib.sa_ntt(y.data_ptr(), x.data_ptr(), LOG_N, root, 0, BATCH, ctypes.c_void_p(stream.cuda_stream))
        if rc != 0:
            raise RuntimeError("sa_ntt failed: %d %s" % (rc, lib.sa_last_error().decode()))

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    # spot parity check inside the bench: transform 0 of this rank against the oracle
    if rank == 0:
        want = O.ntt_np(w, x[:N].cpu().numpy().view(np.uint64), parallel=True)
        assert (y[:N].cpu().numpy().view(np.uint64) == want).all(), "bench output differs from the oracle"
    barrier()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    launches0 = lib.sa_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = lib.sa_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    ms_per_step = ms / args.steps
    value = world * BATCH * BUTTERFLIES_PER_NTT * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:  # (before the legs below reuse y)
        dump_outputs(args.dump_outputs, y)

    # ---- the chip's measured 128-bit butterfly rate (montmul + add + sub on registers, no memory):
    #      the compute roof this kernel actually lives under (profiles/r01_notes.md)
    int_peak = None
    if rank == 0:
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        iters, ilp, blocks, threads = 2000, 4, sms * 4, 256
        mb_ms = lib.sa_microbench(3, ilp, iters, blocks, threads)
        if mb_ms > 0:
            int_peak = iters * ilp * blocks * threads / (mb_ms * 1e-3)

    # ---- single-transform latency (device resident), for the record
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 50
    for i in range(3):  # (a lone transform may take its own launch shape: load and warm it outside the timed region)
        lib.sa_ntt(y[:N].data_ptr(), x[:N].data_ptr(), LOG_N, root, 0, 1, ctypes.c_void_p(stream.cuda_stream))
    torch.cuda.synchronize()
    ev2.record(stream)
    for i in range(reps):
        off = (i % BATCH) * N
        lib.sa_ntt(y[off:off + N].data_ptr(), x[off:off + N].data_ptr(), LOG_N, root, 0, 1,
                   ctypes.c_void_p(stream.cuda_stream))
    ev3.record(stream)
    torch.cuda.synchronize()
    single_us = ev2.elapsed_time(ev3) / reps * 1e3

    if os.environ.get("SA_BENCH_QUICK") == "1":  # kernel experiments (tools/gpu_*.sh): transform timings only
        if rank == 0:
            os.write(json_fd, (json.dumps({"quick": True, "ms_per_step": ms_per_step, "value": value,
                                           "single_ntt_us": single_us, "int_peak": int_peak,
                                           "lib": os.environ.get("SA_B200_LIB"),
                                           "env": {k: v for k, v in os.environ.items() if k.startswith("SA_NTT")}}) + "\n").encode())
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- e2e: the same step through the C-ABI host entry (pinned host buffers, H2D + D2H inside)
    # The host buffers come from the library's own allocator (sa_host_alloc: page-locked, placed on the NUMA
    # node of this rank's GPU, so eight ranks do not push half of their copies across the socket interconnect).
    nbytes = BATCH * N * 16
    p_in, p_out = lib.sa_host_alloc(nbytes), lib.sa_host_alloc(nbytes)
    assert p_in and p_out, lib.sa_last_error()
    hx = np.ctypeslib.as_array((ctypes.c_uint64 * (nbytes // 8)).from_address(p_in)).reshape(-1, 2)
    hy = np.ctypeslib.as_array((ctypes.c_uint64 * (nbytes // 8)).from_address(p_out)).reshape(-1, 2)
    hx[:] = x.cpu().numpy().view(np.uint64)
    hy[:] = 0
    e2e_steps = max(2, min(args.steps, 5))
    lib.sa_ntt_host(p_out, p_in, LOG_N, root, 0, BATCH, ctypes.c_void_p(stream.cuda_stream))
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        rc = lib.sa_ntt_host(p_out, p_in, LOG_N, root, 0, BATCH, ctypes.c_void_p(stream.cuda_stream))
        assert rc == 0
    torch.cuda.synchronize()
    e2e_s = torch.tensor([(time.perf_counter() - t0) / e2e_steps], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = world * BATCH * BUTTERFLIES_PER_NTT / float(e2e_s.item())
    if rank == 0:
        assert (hy[:N] == want).all(), "e2e output differs from the oracle"
    del hx, hy
    lib.sa_host_free(p_in)
    lib.sa_host_free(p_out)

    # ---- FRI commit ms @ 2^20 (second half of BASELINE.json's metric), rank 0 only, list API excluded:
    #      device-resident codeword, 12 fused rounds, host Fiat-Shamir on the 64-byte roots
    fri_ms = fri_cpu_ms = fri_const_ms = b2_peak = None
    if rank == 0:
        import hashlib
        import pickle
        cw = x[:N]
        omega0, off0 = w, O.GENERATOR
        rounds = O.fri_num_rounds(N, 4, 64)
        assert rounds == FRI_ROUNDS

        def fri_commit(constant=False):
            objs = []

            def on_root(r, root, want_alpha):  # the host side of fri.py:71-79 on a plain ProofStream
                objs.append(root)
                if not want_alpha:
                    return None
                return 12345678901234567890 if constant else O.sample(hashlib.shake_256(pickle.dumps(objs)).digest(32))
            eng.fri_commit(cw, rounds, off0, omega0, on_root)
            return objs
        fri_commit()
        torch.cuda.synchronize()
        reps = 5
        t0 = time.perf_counter()
        for _ in range(reps):
            roots = fri_commit()
        torch.cuda.synchronize()
        fri_ms = (time.perf_counter() - t0) / reps * 1e3
        t0 = time.perf_counter()
        for _ in range(reps):
            fri_commit(constant=True)  # the same ladder without the pickle + shake_256 of the challenge
        torch.cuda.synchronize()
        fri_const_ms = (time.perf_counter() - t0) / reps * 1e3
        O.lib().so_set_threads(min(32, os.cpu_count() or 1))
        t0 = time.perf_counter()
        oroots, _, _ = O.fri_commit_np(cw.cpu().numpy().view(np.uint64), off0, omega0, 4, 64)
        fri_cpu_ms = (time.perf_counter() - t0) * 1e3  # (the reference arm probes the team size; this is the check)
        assert roots == oroots, "FRI commit roots differ from the oracle"
        # blake2b-only roof: register-resident chains of node compressions, 1024 threads per SM
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        b2_iters, b2_blocks = 400, sms * 4
        b2_ms = lib.sa_microbench(4, 1, b2_iters, b2_blocks, 256)
        if b2_ms > 0:
            b2_peak = b2_iters * b2_blocks * 256 / (b2_ms * 1e-3)

    # ---- the Python list API of the drop-in, one 2^20 transform / one 2^20 Fri.commit:
    #      list[FieldElement] in (pack + upload) and, since round 2, a device-resident list out
    list_api_s = fri_list_api_s = list_api_dev = None
    if rank == 0 and world == 1:
        import sa_host
        import sa_marshal
        import sa_devlist
        import ntt as dropin_ntt
        import fri as dropin_fri
        field = sa_host.algebra.Field.main()
        FE = sa_host.algebra.FieldElement
        vals = sa_marshal.unpack(x[:N].cpu().numpy(), field, FE)
        wfe = FE(w, field)

        def timed(fn, reps=3):
            fn()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps):
                r = fn()
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) / reps, r
        list_api_s, outl = timed(lambda: dropin_ntt.ntt(wfe, vals))           # list in, device list out
        assert outl[12345].value == int(want[12345][0]) | (int(want[12345][1]) << 64)
        chain_s, back = timed(lambda: dropin_ntt.intt(wfe, dropin_ntt.ntt(wfe, outl)))  # device list in and out
        f = dropin_fri.Fri(field.generator(), wfe, N, 4, 64)
        fri_list_api_s, _ = timed(lambda: f.commit(vals, dropin_fri.ProofStream()))      # list in
        fri_dev_s, _ = timed(lambda: f.commit(outl, dropin_fri.ProofStream()))           # device list in
        sa_devlist.ENABLED = False
        plain_s, _ = timed(lambda: dropin_ntt.ntt(wfe, vals), reps=1)                     # round-1 behaviour
        sa_devlist.ENABLED = True
        list_api_dev = {"ntt_list_in_device_list_out_s": list_api_s, "ntt_plus_intt_device_lists_s": chain_s,
                        "fri_commit_list_in_s": fri_list_api_s, "fri_commit_device_list_in_s": fri_dev_s,
                        "ntt_list_in_list_out_s": plain_s,
                        "note": "2^20 elements; 'list in' packs 2^20 FieldElement objects and uploads 16 MiB, 'list out' "
                                "creates 2^20 objects; device lists (sa_devlist.DeviceCodeword) skip both"}

    # ---- SURVEY 8 a4-a6 at 2^16 points, device-resident inputs, one C call each (for the record)
    poly_ms = None
    if rank == 0 and world == 1:
        K16 = 1 << 16
        dom, pvals = x[:K16].contiguous(), x[K16:2 * K16].contiguous()

        def ev_ms(fn, reps=5):
            fn()
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a_.record(stream)
            for _ in range(reps):
                r = fn()
            b_.record(stream)
            torch.cuda.synchronize()
            return a_.elapsed_time(b_) / reps, r
        z_ms, _ = ev_ms(lambda: eng.zerofier(dom))
        i_ms, poly = ev_ms(lambda: eng.interpolate(dom, pvals))
        e_ms, back = ev_ms(lambda: eng.poly_eval(poly, dom))
        assert bool((back == pvals).all().item()), "interpolant does not take the prescribed values"
        poly_ms = {"points": K16, "fast_zerofier": z_ms, "fast_interpolate": i_ms, "fast_evaluate": e_ms,
                   "note": "sa_zerofier / sa_interpolate / sa_poly_eval on 2^16 random points: device subproduct tree, "
                           "walk down the transposed tree; the interpolant is checked against the values"}

    # ---- N > 1: the same batch sharded over the ranks WITH the assembly on every rank (every rank takes part)
    with_allgather = allgather_leg(eng, dist, rank, world, w) if dist is not None else None

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- CPU baseline on this box's host cores, bounded sample (a few seconds); N = 1 only
    cpu_value = cpu_threads = py_value = None
    if world == 1:
        cpu_value, cpu_threads, cpu_dt = cpu_arm(2, 1, BATCH)
        # the reference is pure Python: time the literal Python restatement of ntt.py:3-18 (oracle.py
        # py_ntt, ints instead of FieldElement objects) on one core at 2^12 as the same-run interpreter arm
        import random
        rng = random.Random(0)
        pn = 1 << 12
        pv = [rng.randrange(O.P) for _ in range(pn)]
        t0 = time.perf_counter()
        O.py_ntt(O.primitive_nth_root(pn), pv)
        py_value = (pn // 2) * 12 / (time.perf_counter() - t0)

    # roofline of the dominant kernel, ntt_tile_kernel<10>: two launches per step (column pass, row pass).
    # Algorithmic bytes (SURVEY 8d): 32 * n per transform = 64 / log2(n) bytes per butterfly; one launch does
    # half of a transform's butterfly levels, i.e. 16 * n * BATCH algorithmic bytes.  The four-step split itself
    # reads and writes the whole batch once per launch (32 * n * BATCH): reported beside it as the design's floor.
    launches_per_step = 2
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):  # dram bytes per launch from the committed ncu --set full capture
        with open(tpath) as f:
            traffic = json.load(f).get("dram_bytes_per_launch_mean")
    bytes_per_butterfly = 64.0 / LOG_N
    alg_bytes_per_launch = int(bytes_per_butterfly * BATCH * BUTTERFLIES_PER_NTT / launches_per_step)
    pass_bytes_per_launch = 32 * N * BATCH
    launch_s = ms_per_step * 1e-3 / launches_per_step
    achieved = alg_bytes_per_launch / launch_s / 1e9
    achieved_pass = pass_bytes_per_launch / launch_s / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u128 mod p (4x u32 limbs, Montgomery)", "data": "synthetic",
        "config": config_dict(world),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "kernel": "ntt_tile_kernel<10>", "launches_per_step": launches_per_step,
                     "algorithmic_bytes_per_launch": alg_bytes_per_launch, "peak_source": peak_src,
                     "two_pass_floor": {"bytes_per_launch": pass_bytes_per_launch, "achieved": achieved_pass,
                                        "frac": achieved_pass / peak,
                                        "why": "a 2^20 transform (16 MiB) does not fit on chip: the four-step split "
                                               "reads and writes the vector once per pass, 2x the algorithmic bytes; "
                                               "ncu traffic matches this floor (no other re-reads)"},
                     "note": "bound by the integer pipes, not HBM: 21 IMAD.WIDE per field product (4 fmaheavy cycles each) put "
                             "the floor at ~30 us per 2^20 transform = frac ~0.17 (DESIGN.md 3.2, profiles/r01_notes.md)"},
        "int_roofline": {"bound": "integer pipes (IMAD.WIDE / IADD3)", "achieved": value / world,
                         "peak": int_peak, "unit": "butterflies/s per GPU",
                         "frac": (value / world / int_peak) if int_peak else None,
                         "how": "peak = sa_microbench: register-resident montmul+add+sub loop, 4 independent "
                                "chains per thread, 1024 threads per SM, measured in this run"},
        "cpu_baseline": {"value": cpu_value, "unit": UNIT, "cores": cpu_threads, "kind": "port",
                         "sample": "2 steps of %d x 2^20 ntt with oracle/stark_oracle.c (OpenMP tasks: transforms, "
                                   "recursion and combine loops, so every one of the `cores` threads works); the "
                                   "reference's pure-Python ntt is 5.5e4 butterflies/s on 1 core (BASELINE.md)" % BATCH},
        "cpu_python": {"value": py_value, "unit": UNIT, "cores": 1, "kind": "port",
                       "sample": "oracle.py py_ntt at n = 2^12; the reference's own ntt measured 3.9e4-6.4e4 "
                                 "butterflies/s at 2^10..2^20 on one Xeon core (BASELINE.md section 2)"},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": BATCH * N * 16,
                "d2h_bytes_per_step": BATCH * N * 16, "api": "sa_ntt_host (C ABI, host buffers from sa_host_alloc)",
                "host_buffers": "page-locked, on the NUMA node of the rank's GPU (sa_host_alloc)"},
        "with_allgather": with_allgather,
        "gpu_launches": int(launches),
        "clocks": clocks,
        "single_ntt_us": single_us,
        "list_api_ntt_2_20_s": list_api_s, "list_api_fri_commit_2_20_s": fri_list_api_s,
        "list_api": list_api_dev,
        "poly_ops_2_16_ms": poly_ms,
        "fri_commit_ms_2_20": fri_ms, "fri_commit_cpu_port_ms_2_20": fri_cpu_ms,
        "fri_roofline": None if fri_ms is None else {
            "bound": "alu pipe (blake2b: 64-bit add / xor / rotate), not HBM",
            "achieved": FRI_COMPRESSIONS / (fri_ms * 1e-3), "peak": b2_peak, "unit": "blake2b compressions/s",
            "frac": (FRI_COMPRESSIONS / (fri_ms * 1e-3) / b2_peak) if b2_peak else None,
            "compressions_per_commit": FRI_COMPRESSIONS, "rounds": FRI_ROUNDS,
            "ms_with_python_challenge": fri_ms, "ms_with_constant_challenge": fri_const_ms,
            "hbm": {"algorithmic_bytes": FRI_ALG_BYTES, "achieved_gbs": FRI_ALG_BYTES / (fri_ms * 1e-3) / 1e9,
                    "frac": FRI_ALG_BYTES / (fri_ms * 1e-3) / 1e9 / peak,
                    "retained_tree_bytes": 64 * (4 * N - ((4 * N) >> FRI_ROUNDS))},
            "how": "peak = sa_microbench(4): register-resident chains of single-block blake2b node compressions, 1024 "
                   "threads per SM, measured in this run; achieved = 4 193 268 compressions (12 trees) / wall time of "
                   "sa_fri_commit on a device-resident 2^20 codeword incl. the per-round host Fiat-Shamir"},
    }
    sys.stdout.flush()
    os.write(json_fd, (json.dumps(line) + "\n").encode())
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a seeded sample of rank 0's last step output to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
