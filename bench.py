#!/usr/bin/env python
"""bench.py - headline measurement for the Boojum polynomial-commitment hot path on B200.

metric  : Goldilocks NTT G-elements/s (BASELINE.json metric, first half).  The second half, proof-generation seconds
          at 2^22 rows at N GPUs, is reported in the extra objects "prove" (configs[4]'s type parameters: Poseidon2 tree hasher +
          Poseidon (v1) sponge transcript) and "prove_non_recursive" (configs[3]: Blake2s tree + Blake2sTranscript) on a synthetic
          SHA-256-bench-shaped circuit (the real circuit needs the Rust synthesiser); the library's C++ driver bj_prove runs on
          one GPU or coset-sharded over a bj_comm (NCCL) on N; every timed proof is checked by the oracle's restated verifier
          after the timed region ("verified"), the witness H2D is reported beside it, and on N > 1 GPUs rank 0 also times the
          single-GPU proof in the same run ("strong_scaling_efficiency").  "merkle" reports configs[2]; "ntt_family" the inverse /
          LDE figures of configs[1]; "prove.cpu_baseline_s" the CPU port's stage times.
workload: BASELINE.json configs[1] "2^20-2^24 Goldilocks NTT/LDE sweep on 1xB200": one step = forward
          natural->bit-reversed NTT on coset 7 (benches/benchmarks.rs:541 uses coset 7) of five resident batches,
          n = 2^20..2^24 with 128/64/32/16/8 columns (1 GiB each, SURVEY.md 8(d) cfg 2), in place, through the
          C-ABI (bj_ntt_natural_to_bitreversed).  5 GiB of inputs >> 126 MB L2, so no L2 flush is needed.
value   : elements transformed per second, all ranks (columns shard across GPUs with no collective -> weak scaling).
e2e     : the same sweep through bj_ntt_natural_to_bitreversed_host: pinned HOST buffers, H2D + NTT + D2H per step.
roofline: dominant kernel ntt_pass_v2_kernel; algorithmic bytes = 16 B per element per transform (read once, write
          once; SURVEY.md 8(d)) / measured HBM copy peak (MEASURED_PEAKS.json, burst figure); `traffic` = DRAM bytes per launch
          from the committed ncu capture (profiles/ncu_traffic.json).
cpu_baseline / --impl reference: the oracle's restatement of the reference CPU algorithm (one serial NTT per column,
          columns spread over all host threads, src/cs/implementations/utils.rs:295-304) on a bounded sample.
--dump-outputs DIR: after the timed steps, a fixed sample of the batches as the last timed step left them (see dump_outputs),
          so that two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SIZES = [20, 21, 22, 23, 24]
BATCH_ELEMS_LOG = 27  # 1 GiB of u64 per size
COSET = 7
METRIC = "goldilocks_ntt_gelements_per_s"
DUMP_SAMPLES = 1 << 19  # elements per size written by --dump-outputs: 5 sizes x 2^19 x 16 B = 40 MiB


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], 0, None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        while not self._stop_evt.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                self.reasons |= int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                pass
            time.sleep(0.02)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        names = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
                 0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": [n for b, n in names.items() if self.reasons & b], "samples": len(s)}


def dump_outputs(out_dir, data, rank, world):
    """Writes out_dir/ntt_log<m>.npy (ntt_log<m>_rank<r>.npy on several GPUs) for every size m: the elements at fixed, seeded
    positions of that size's batch, as float64 [samples, 2] = (high 32 bits, low 32 bits) of each u64 so that every value is
    exact.  The positions depend only on m and the number of GPUs."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for m, t in data.items():
        flat = t.view(-1)
        idx = np.sort(np.random.default_rng(m).integers(0, flat.numel(), DUMP_SAMPLES // world))
        v = flat[torch.from_numpy(idx).to(flat.device)].cpu().numpy().view(np.uint64)
        pair = np.stack([v >> np.uint64(32), v & np.uint64(0xFFFFFFFF)], axis=1).astype(np.float64)
        np.save(os.path.join(out_dir, "ntt_log%d%s.npy" % (m, "_rank%d" % rank if world > 1 else "")), pair)


def run_reference(args, rank, world):
    """Reference arm: the oracle's restatement of the reference CPU path, all host threads, bounded sample."""
    if rank != 0:
        return
    import numpy as np
    from oracle import oracle as O
    # all host threads this process may use, also under torchrun (which exports OMP_NUM_THREADS=1 to its workers)
    O.lib().orc_set_threads(len(os.sched_getaffinity(0)))
    threads = O.num_threads()
    rng = np.random.default_rng(0)
    cols = {m: max(1, min(threads, 1 << (BATCH_ELEMS_LOG - m))) for m in SIZES}
    data = {m: O.random_field(rng, (cols[m], 1 << m)) for m in SIZES}
    elems = sum(cols[m] << m for m in SIZES)

    def step():
        for m in SIZES:
            a = data[m]
            O.lib().orc_ntt_n2b(a.ctypes.data_as(ctypes.c_void_p), m, cols[m], 1 << m, COSET)

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    val = elems / dt / 1e9
    sample = "per step: forward NTT coset 7, sizes 2^20..2^24, %d column(s) each (one serial NTT per column, %d threads)" % (
        cols[SIZES[0]], threads)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "Gelem/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": "ntt_forward_sweep_2^20..2^24_coset7 (bounded sample of the GPU arm's batches)"},
        "cpu_baseline": {"value": val, "unit": "Gelem/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "Gelem/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def host_cpu_quota():
    """CPUs this process may actually use: the affinity mask, capped by the cgroup CPU quota when one is set (a container
    that sees 128 logical CPUs but is throttled to a few cores runs 128 threads no faster than 8)."""
    allowed = len(os.sched_getaffinity(0))
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:                                  # cgroup v2
            q, period = f.read().split()
        if q != "max":
            quota = float(q) / float(period)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:                 # cgroup v1
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                period = float(f.read())
            if q > 0:
                quota = q / period
        except Exception:
            pass
    return allowed, quota


def cpu_baseline_sample():
    """BASELINE.md section 3: the oracle port (one serial radix-2 NTT per column, columns over a thread pool) on the box's host
    cores; rows for 8 threads (the reference bench pins Worker::new_with_num_threads(8), src/gadgets/sha256/mod.rs:307) and for
    every allowed core (Worker::new()), >= 15 s each, with and without the reference's per-stage twiddle recomputation +
    primitivity assert loop (utils.rs:107-110; serial)."""
    import numpy as np
    from oracle import oracle as O
    allowed = len(os.sched_getaffinity(0))
    m = 22
    n = 1 << m
    tab = np.zeros(n // 2 + 1, np.uint64)
    t0 = time.perf_counter()
    O.lib().orc_twiddles(tab.ctypes.data_as(ctypes.c_void_p), m, 0, 1)
    t_assert = time.perf_counter() - t0
    t0 = time.perf_counter()
    O.lib().orc_twiddles(tab.ctypes.data_as(ctypes.c_void_p), m, 0, 0)
    t_assert = max(0.0, t_assert - (time.perf_counter() - t0))
    rows = []
    for threads in sorted({min(8, allowed), allowed}):
        O.lib().orc_set_threads(threads)
        cols = 2 * threads if threads <= 8 else threads
        a = O.random_field(np.random.default_rng(1), (cols, n))
        O.lib().orc_ntt_n2b(a.ctypes.data_as(ctypes.c_void_p), m, cols, n, COSET)  # warm-up (page faults, OpenMP team)
        t0 = time.perf_counter()
        reps = 0
        while True:
            O.lib().orc_ntt_n2b(a.ctypes.data_as(ctypes.c_void_p), m, cols, n, COSET)
            reps += 1
            if time.perf_counter() - t0 > 15.0 or reps >= 200:
                break
        dt = time.perf_counter() - t0
        rows.append({"cores": threads, "value": round(reps * cols * n / dt / 1e9, 5),
                     "value_with_reference_twiddle_recompute": round(reps * cols * n / (dt + reps * t_assert) / 1e9, 5),
                     "sample": "%d x (%d columns of 2^22, forward NTT coset 7, tables built once per batch), %.1f s" % (reps, cols, dt)})
        del a
    best = max(rows, key=lambda r: r["value"])
    _, quota = host_cpu_quota()
    return {"value": best["value"], "unit": "Gelem/s", "cores": best["cores"], "kind": "port", "sample": best["sample"],
            "cgroup_cpu_quota_cores": quota, "rows": rows, "twiddle_assert_loop_s_per_stage_2^22": round(t_assert, 4),
            "note": "rows: 8 threads = Worker::new_with_num_threads(8) of the reference bench, all cores = Worker::new(); "
                    "value_with_reference_twiddle_recompute adds the serial assert loop of precompute_twiddles_for_fft per batch call"}


def cpu_prove_stage_baseline(log_n=22, total_cols=93, budget_cols=8):
    """CPU beside the proof seconds (BASELINE.md section 3 'Prove: seconds per stage'): the oracle port's witness-commit stage
    (LDE to 8 cosets + Poseidon2 leaf/node hashing, cap 16), one DEEP group over those columns and the FRI fold chain, for the
    2^22-row shape, all allowed host threads.  To stay within a bounded sample the LDE / tree / DEEP run over `budget_cols`
    columns and are scaled linearly to the circuit's 93 witness-oracle columns (both are linear in the column count)."""
    import numpy as np
    from oracle import oracle as O
    threads = len(os.sched_getaffinity(0))
    O.lib().orc_set_threads(threads)
    n, L = 1 << log_n, 8
    cols = min(budget_cols, total_cols)
    rng = np.random.default_rng(7)
    trace = O.random_field(rng, (cols, n))
    out = {}
    t0 = time.perf_counter()
    lde = O.lde(trace, 3)
    out["lde_s"] = time.perf_counter() - t0
    srcs = [lde[c].reshape(-1) for c in range(cols)]
    t0 = time.perf_counter()
    lh = O.merkle_leaf_hashes(srcs)
    O.merkle_nodes(lh, 16)
    out["poseidon2_tree_s"] = time.perf_counter() - t0
    acc0, acc1 = np.zeros(n * L, np.uint64), np.zeros(n * L, np.uint64)
    vals = [(int(v), 0) for v in O.random_field(rng, cols)]
    chs = [(int(v), int(w)) for v, w in O.random_field(rng, (cols, 2))]
    t0 = time.perf_counter()
    acc0, acc1 = O.deep_group(acc0, acc1, [(s_, None) for s_ in srcs], vals, chs, (12345, 678))
    out["deep_s"] = time.perf_counter() - t0
    roots = O.twiddles(log_n + 3, inverse=True)
    t0 = time.perf_counter()
    a, k, f0, f1 = (3, 5), O.inv(7), acc0, acc1
    while len(f0) > 16:
        f0, f1 = O.fri_fold(f0, f1, a, roots[: len(f0) // 2], k)
        a, k = O.ext_mul(a, a), O.mul(k, k)
    out["fri_folds_s"] = time.perf_counter() - t0
    scale = total_cols / cols
    est = scale * (out["lde_s"] + out["poseidon2_tree_s"] + out["deep_s"]) + out["fri_folds_s"]
    return {"cores": threads, "kind": "port", "measured_columns": cols, "scaled_to_columns": total_cols,
            "measured_s": {k_: round(v, 3) for k_, v in out.items()},
            "witness_commit_stage_s_scaled": round(scale * (out["lde_s"] + out["poseidon2_tree_s"]), 2),
            "deep_s_scaled": round(scale * out["deep_s"], 2), "fri_folds_s": round(out["fri_folds_s"], 2),
            "covered_stages_s_scaled": round(est, 2),
            "covers": "stage 1 (witness LDE + Poseidon2 oracle), one DEEP pass over the same columns, FRI folds (no FRI oracles); "
                      "not covered: stage 2, quotient, openings, queries, setup"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--prove-log-n", type=int, default=22, help="rows (log2) of the synthetic SHA-shaped proof; 0 disables")
    ap.add_argument("--dump-outputs", metavar="DIR", help="(b200 impl) write a fixed sample of the last timed step's outputs to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import era_boojum_b200 as bj
    from era_boojum_b200 import native

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    numa = "unchanged"
    if world > 1:
        # keep this rank's host threads (and, by first touch, its pinned staging buffers) on the CPU socket next to its GPU:
        # the end-to-end path moves 10 GiB per step per GPU through host memory
        try:
            import pynvml
            pynvml.nvmlInit()
            h_ = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
            words = pynvml.nvmlDeviceGetCpuAffinity(h_, (os.cpu_count() + 63) // 64)
            cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
            cpus &= set(os.sched_getaffinity(0))
            if cpus:
                os.sched_setaffinity(0, cpus)
                numa = "bound to the %d CPUs local to GPU %d" % (len(cpus), local_rank)
        except Exception as e:  # affinity is an optimisation only
            numa = "unchanged (%s)" % type(e).__name__
    torch.cuda.set_device(local_rank)
    dev = "cuda:%d" % local_rank
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(dev))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ctx = bj.Context.on_current_stream(local_rank)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    cols = {m: 1 << (BATCH_ELEMS_LOG - m) for m in SIZES}
    # synthetic resident inputs: uniform 63-bit values (valid lazy field elements), created before the timed region
    data = {m: torch.randint(0, 2**63 - 1, (cols[m], 1 << m), dtype=torch.int64, device=dev, generator=gen) for m in SIZES}
    elems_per_step = sum(cols[m] << m for m in SIZES)

    def step():
        for m in SIZES:
            ctx.fft_natural_to_bitreversed(data[m], COSET)

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    clocks = sampler.stop()
    launches = ctx.launch_count() - l0
    ms = e0.elapsed_time(e1) / args.steps
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = world * elems_per_step / (ms * 1e-3) / 1e9
    if args.dump_outputs:   # before the per-size breakdown below transforms the batches again
        dump_outputs(args.dump_outputs, data, rank, world)

    # per-size breakdown (device time, CUDA events, same stream), after the headline region
    sweep = {}
    for m in SIZES:
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(3):
            ctx.fft_natural_to_bitreversed(data[m], COSET)
        a1.record()
        torch.cuda.synchronize()
        t_ms = a0.elapsed_time(a1) / 3
        el = cols[m] << m
        sweep["2^%d" % m] = {"cols": cols[m], "ms": round(t_ms, 4), "gelem_s": round(el / t_ms / 1e6, 3),
                             "algo_gbs": round(16 * el / t_ms / 1e6, 1)}

    # the rest of the NTT family at 2^22 (SURVEY 8d cfg 2): inverse (natural -> natural, coset 7) and LDE to 2 / 4 / 8 cosets
    family = {}
    if not args.no_e2e:
        m = 22
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.ifft_natural_to_natural(data[m], COSET)
        a0.record()
        for _ in range(3):
            ctx.ifft_natural_to_natural(data[m], COSET)
        a1.record()
        torch.cuda.synchronize()
        t_ms = a0.elapsed_time(a1) / 3
        family["inverse_2^22"] = {"cols": cols[m], "ms": round(t_ms, 4), "gelem_s": round((cols[m] << m) / t_ms / 1e6, 3)}
        src = data[m][:8]
        for lde in (2, 4, 8):
            out_l = torch.empty((8, lde, 1 << m), dtype=torch.int64, device=dev)
            ctx.transform_raw_storages_to_lde(src, lde, out=out_l)
            a0.record()
            for _ in range(3):
                ctx.transform_raw_storages_to_lde(src, lde, out=out_l)
            a1.record()
            torch.cuda.synchronize()
            t_ms = a0.elapsed_time(a1) / 3
            family["lde%d_2^22" % lde] = {"cols": 8, "ms": round(t_ms, 4), "in_gelem_s": round((8 << m) / t_ms / 1e6, 3),
                                           "algo_gbs": round(8 * (1 + lde) * (8 << m) / t_ms / 1e6, 1)}
            del out_l

    peak, peak_kind = load_peaks()
    launches_per_step = launches / max(1, args.steps)
    algo_bytes_step = 16.0 * elems_per_step
    achieved = algo_bytes_step / (ms * 1e-3) / 1e9  # the step is ntt_pass_v2_kernel launches only
    roofline = {"bound": "hbm", "kernel": "ntt_pass_v2_kernel", "achieved": round(achieved, 1), "peak": peak,
                "peak_source": peak_kind + " hbm copy", "unit": "GB/s", "frac": round(achieved / peak, 4),
                "algo_bytes_per_launch": algo_bytes_step / max(1.0, launches_per_step),
                "avg_launch_ms": ms / max(1.0, launches_per_step), "traffic": None}
    try:
        # DRAM bytes per launch of the same kernel from the committed `ncu --set full` capture (not measured in this run):
        # bytes per element per launch of the capture x the elements one launch of this run processes
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            tr_ = json.load(f)
        # one launch = one pass over one whole resident batch of 2^BATCH_ELEMS_LOG elements
        elems_per_launch = float(1 << BATCH_ELEMS_LOG)
        roofline["traffic"] = round(tr_["dram_bytes_per_element_per_launch"] * elems_per_launch)
        roofline["traffic_over_algo"] = round(roofline["traffic"] / roofline["algo_bytes_per_launch"], 3)
        roofline["traffic_source"] = "profiles/ncu_traffic.json (%s)" % tr_.get("capture", "ncu --set full")
    except Exception:
        pass

    # end to end: pinned host buffers -> H2D -> NTT -> D2H through the host-buffer C-ABI entry point
    e2e = None
    if not args.no_e2e:
        host = {m: torch.empty((cols[m], 1 << m), dtype=torch.int64).pin_memory() for m in SIZES}
        for m in SIZES:
            host[m].copy_(data[m])
        torch.cuda.synchronize()

        def e2e_step():
            for m in SIZES:
                st = native.lib.bj_ntt_natural_to_bitreversed_host(ctx._h, ctypes.c_void_p(host[m].data_ptr()), m, cols[m], COSET)
                if st != 0:
                    raise bj.BoojumError(st, "host NTT failed")

        e2e_step()
        barrier()
        k = max(1, min(args.steps, 3))
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0.record()
        for _ in range(k):
            e2e_step()
        b1.record()
        barrier()
        e_ms = b0.elapsed_time(b1) / k
        if world > 1:
            t = torch.tensor([e_ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e_ms = float(t.item())
        e2e = {"value": round(world * elems_per_step / (e_ms * 1e-3) / 1e9, 4), "unit": "Gelem/s",
               "h2d_bytes_per_step": 8 * elems_per_step, "d2h_bytes_per_step": 8 * elems_per_step,
               "ms_per_step": round(e_ms, 3), "steps": k, "host_affinity": numa}
        if world > 1:   # every rank's CPU binding (the e2e path is host-memory bound: placement per rank matters)
            per_rank = [None] * world
            dist.all_gather_object(per_rank, numa)
            e2e["host_affinity_per_rank"] = per_rank
        del host

    out = {
        "metric": METRIC, "value": round(value, 4), "unit": "Gelem/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(ms, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": "ntt_forward_sweep_2^20..2^24_coset7", "sizes_log2": SIZES,
                   "columns_per_size": [cols[m] for m in SIZES], "resident_bytes_per_gpu": 8 * elems_per_step,
                   "l2": "inputs (5 GiB) larger than L2, no flush", "parallelism": "columns sharded x%d, no collective" % world},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "sweep": sweep, "ntt_family": family, "e2e": e2e,
    }
    # BASELINE configs[2]: Poseidon2 Merkle tree over 2^22 leaves x 100 columns (cap 16), device-resident columns
    if world == 1 and args.prove_log_n > 0:
        data = None
        torch.cuda.empty_cache()
        m_cols, m_log = 100, 22
        srcs = [torch.randint(0, 2**63 - 1, (1 << m_log,), dtype=torch.int64, device=dev, generator=gen) for _ in range(m_cols)]
        ctx.merkle_tree_construct(srcs, 16)
        torch.cuda.synchronize()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(3):
            tree = ctx.merkle_tree_construct(srcs, 16)
        c1.record()
        torch.cuda.synchronize()
        m_ms = c0.elapsed_time(c1) / 3
        perms = (1 << m_log) * ((m_cols + 7) // 8) + (1 << m_log) - 16
        out["merkle"] = {"workload": "poseidon2 tree, 2^22 leaves x 100 columns, cap 16", "ms": round(m_ms, 3),
                         "leaves_per_s": round((1 << m_log) / m_ms * 1e3), "gperms_per_s": round(perms / m_ms / 1e6, 4),
                         "algo_gbs": round(((8 * m_cols + 32) * (1 << m_log) + 96 * ((1 << m_log) - 16)) / m_ms / 1e6, 1)}
        del srcs, tree
    # second half of BASELINE.json's metric: proof generation seconds on the SHA-256-bench-shaped circuit (synthetic trace,
    # 60 general-purpose columns + 8 lookup sub-arguments of width 4, 3 gate types, quotient degree 4, LDE 8, cap 16, ~100-bit security)
    if args.prove_log_n > 0:
        data = None
        torch.cuda.empty_cache()
        from era_boojum_b200 import parallel, prover, synthetic
        comm, pctx = None, ctx
        if world > 1:
            # coset-sharded proving by the library's own C++ driver: rank r keeps the LDE cosets j = r (mod world) of every committed
            # polynomial; caps, the quotient cosets (one ncclAllGather), the openings and the query answers are exchanged through
            # a bj_comm over NCCL (csrc/comm.cu); torch.distributed only hands the 128-byte NCCL unique id to the ranks
            pctx = bj.Context.on_current_stream(local_rank)
            comm = bj.Comm.from_torch_distributed(pctx, dist, 8)
        variables, sigmas, constants, gates, Q, lk = synthetic.generate(pctx, args.prove_log_n, 60, seed=42, lookup=True)
        # SURVEY 8(d): "H2D of the witness reported separately" - the witness columns (variables + multiplicities) from pinned
        # host memory to the device, timed with CUDA events (the trace itself is generated on the device, so the copy is not
        # part of the proof seconds; seconds_with_witness_h2d adds it)
        wit = torch.cat([variables.reshape(variables.shape[0], -1), lk["multiplicities"].reshape(1, -1)], dim=0)
        host_w = torch.empty(wit.shape, dtype=torch.int64).pin_memory()
        host_w.copy_(wit)
        torch.cuda.synchronize()
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        wit.copy_(host_w, non_blocking=True)
        w0.record()
        wit.copy_(host_w, non_blocking=True)
        w1.record()
        torch.cuda.synchronize()
        h2d_witness_s = w0.elapsed_time(w1) * 1e-3
        h2d_witness_bytes = wit.numel() * 8
        del wit, host_w
        from oracle import verifier as OV   # checker only: runs on the finished proof, outside every timed region

        def prove_once(hasher, transcript):
            """one timed proof of the synthetic SHA-shaped circuit with the given tree hasher (H) and transcript (TR)"""
            cfg = prover.ProofConfig(fri_lde_factor=8, merkle_tree_cap_size=16, security_level=100, hasher=hasher, transcript=transcript)
            # the host driver is the library's own C++ (bj_setup_create / bj_prove), sharded over the communicator when world > 1;
            # the proof comes back as serde JSON
            setup = pctx.native_setup(sigmas, constants, gates, Q, cfg, lookup=lk)
            # the deliverable of the C-ABI is the proof as serde JSON text (what a Rust caller hands to serde_json::from_slice);
            # the timed region ends when bj_proof_to_json has filled the buffer, parsing it (here: Python) is reported apart
            run_prove = lambda tm: setup.prove(variables, lk["multiplicities"], timings=tm, as_json=True)
            run_prove(None)  # warm-up (tables, allocator)
            best = None
            for _ in range(2):  # two timed proofs, the faster one is reported (max over ranks each)
                barrier()
                stages = {}
                t0 = time.perf_counter()
                proof_text = run_prove(stages)
                torch.cuda.synchronize()
                secs = time.perf_counter() - t0
                if world > 1:
                    t = torch.tensor([secs] + [stages[k] for k in sorted(stages)], device=dev, dtype=torch.float64)
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                    secs = float(t[0].item())
                    stages = {k: float(v) for k, v in zip(sorted(stages), t[1:].tolist())}
                if best is None or secs < best[0]:
                    best = (secs, stages)
            secs, stages = best
            t0 = time.perf_counter()
            proof = json.loads(proof_text)
            parse_s = time.perf_counter() - t0
            # the timed proof itself is checked by the oracle's restatement of the reference verifier (rank 0; every rank of the
            # sharded prover returns the same proof)
            verified = None
            if rank == 0:
                t0 = time.perf_counter()
                try:
                    verified = bool(OV.verify(setup.vk(), proof))
                except AssertionError as e:
                    verified = False
                    sys.stderr.write("bench: the oracle verifier REJECTED the timed %s/%s proof: %r\n" % (hasher, transcript, e))
                verify_s = time.perf_counter() - t0
            res = {"rows_log2": args.prove_log_n, "seconds": round(secs, 4), "queries": len(proof["queries_per_fri_repetition"]),
                   "n_gpus": world, "tree_hasher": hasher, "transcript": transcript, "verified": verified,
                   "h2d_witness_s": round(h2d_witness_s, 4), "h2d_witness_bytes": h2d_witness_bytes,
                   "seconds_with_witness_h2d": round(secs + h2d_witness_s, 4), "proof_json_bytes": len(proof_text),
                   "python_json_parse_s": round(parse_s, 4),
                   "stages_s": {k: round(v, 4) for k, v in stages.items()}}
            if rank == 0:
                res["verifier_s"] = round(verify_s, 3)
            if hasattr(setup, "close"):
                setup.close()
            del setup, proof, proof_text
            torch.cuda.empty_cache()
            return res

        common = {"circuit": "synthetic sha256-bench-shaped: 60 gp columns + 8 lookup sub-arguments of width 4 (92 copy-permutation columns, 1 multiplicity column), ConstantsAllocator/Fma/Reduction<4>, Q=4, L=8, cap 16",
                  "scaling": "strong (one proof, LDE cosets sharded over the GPUs)" if world > 1 else "single GPU",
                  "driver": "bj_prove (host C++ in libboojum_b200.so%s); timed until the serde JSON text of the proof is in the caller's buffer" % (", coset-sharded over bj_comm / NCCL" if world > 1 else ""),
                  "note": "best of 2 timed proofs after one warm-up; the witness H2D (pinned host -> device, CUDA events) is reported as h2d_witness_s and added in seconds_with_witness_h2d; `verified` = the last timed proof accepted by oracle/verifier.py after the timed region; wall clock, max over ranks"}
        # BASELINE configs[4] = run_sha256_prover_recursive_mode_poseidon2 (src/gadgets/sha256/mod.rs:286-293): Poseidon2 tree hasher +
        # GoldilocksPoisedonTranscript (the Poseidon v1 sponge transcript); configs[3] = run_sha256_prover_non_recursive (:264-271):
        # Blake2s256 tree hasher + Blake2sTranscript
        out["prove"] = dict(common, **prove_once("poseidon2", "poseidon"))
        out["prove_non_recursive"] = dict(common, **prove_once("blake2s", "blake2s"))
        if world > 1:
            # strong scaling of the proof, measured in this run: rank 0 proves the same circuit alone (its own unsharded context)
            # while the other ranks wait; efficiency = t(1 GPU) / (N * t(N GPUs))
            single = {}
            if rank == 0:
                sctx = bj.Context.on_current_stream(local_rank)
                for key, (hasher, transcript) in (("prove", ("poseidon2", "poseidon")), ("prove_non_recursive", ("blake2s", "blake2s"))):
                    cfg1 = prover.ProofConfig(fri_lde_factor=8, merkle_tree_cap_size=16, security_level=100, hasher=hasher, transcript=transcript)
                    s1 = sctx.native_setup(sigmas, constants, gates, Q, cfg1, lookup=lk)
                    s1.prove(variables, lk["multiplicities"], as_json=True)
                    best1 = None
                    for _ in range(2):
                        torch.cuda.synchronize()
                        t0 = time.perf_counter()
                        s1.prove(variables, lk["multiplicities"], as_json=True)
                        torch.cuda.synchronize()
                        dt1 = time.perf_counter() - t0
                        best1 = dt1 if best1 is None else min(best1, dt1)
                    single[key] = best1
                    s1.close()
                    torch.cuda.empty_cache()
                sctx.close()
            barrier()
            if rank == 0:
                for key, t1 in single.items():
                    out[key]["single_gpu_seconds_same_run"] = round(t1, 4)
                    out[key]["speedup_vs_single_gpu"] = round(t1 / out[key]["seconds"], 2)
                    out[key]["strong_scaling_efficiency"] = round(t1 / out[key]["seconds"] / world, 3)
        del variables, sigmas, constants, lk
        if world == 1:
            try:
                # the production shape (not a BASELINE config; reported beside them): geometry of the reference's own vk.json / proof.json
                # - 155 columns under the copy permutation, its 11 gate evaluators incl. the Poseidon2 flattened gate behind the
                # 6-level selector tree (415 quotient terms), 8 lookups of width 3, quotient degree 8 over fri_lde_factor 2, cap 32
                torch.cuda.empty_cache()
                plog = min(20, args.prove_log_n)
                c = synthetic.generate_production_shaped(pctx, plog, seed=42)
                shapes = {}
                for hasher in ("poseidon2", "blake2s"):
                    cfg = prover.ProofConfig(fri_lde_factor=2, merkle_tree_cap_size=32, security_level=100, hasher=hasher, transcript=hasher)
                    setup = pctx.native_setup(c["sigmas"], c["constants"], c["gates"], c["quotient_degree"], cfg, lookup=c["lookup"],
                                              public_inputs=c["public_inputs"])
                    m = c["lookup"]["multiplicities"]
                    setup.prove(c["variables"], m, as_json=True)
                    best = None
                    for _ in range(2):
                        torch.cuda.synchronize()
                        stages = {}
                        t0 = time.perf_counter()
                        text = setup.prove(c["variables"], m, timings=stages, as_json=True)
                        torch.cuda.synchronize()
                        secs = time.perf_counter() - t0
                        if best is None or secs < best[0]:
                            best = (secs, stages, text)
                    try:
                        ok = bool(OV.verify(setup.vk(), json.loads(best[2])))
                    except AssertionError as e:
                        ok = False
                        sys.stderr.write("bench: the oracle verifier REJECTED the production-shaped %s proof: %r\n" % (hasher, e))
                    shapes[hasher] = {"seconds": round(best[0], 4), "verified": ok, "stages_s": {k: round(v, 4) for k, v in best[1].items()}}
                    setup.close()
                    torch.cuda.empty_cache()
                out["prove_production_shape"] = {
                    "circuit": "synthetic, geometry of the reference's vk.json fixture: 2^%d rows, 130 gp + 24 lookup + 1 boolean columns, 8 constants, "
                               "11 gates / 415 terms incl. Poseidon2FlattenedGate, quotient degree 8, fri_lde_factor 2, cap 32, 4 public inputs" % plog,
                    "note": "not a BASELINE config - the shape of a zkSync recursion-layer circuit; bj_prove on one GPU, best of 2 after a warm-up, verified",
                    "poseidon2_tree_and_transcript": shapes["poseidon2"], "blake2s_tree_and_transcript": shapes["blake2s"]}
                del c
            except Exception as e:      # an extra, never at the expense of the contract line
                out["prove_production_shape"] = {"error": repr(e)[:300]}
                sys.stderr.write("bench: production-shaped proof skipped: %r\n" % (e,))
    if rank == 0 and world == 1 and not args.no_cpu:
        out["cpu_baseline"] = cpu_baseline_sample()
        if args.prove_log_n > 0:
            cpb = cpu_prove_stage_baseline(args.prove_log_n)
            for key in ("prove", "prove_non_recursive"):
                if key in out:
                    out[key]["cpu_baseline_s"] = cpb if key == "prove" else {"see": "prove.cpu_baseline_s (Poseidon2 tree; the CPU port has no Blake2s tree)",
                                                                              "lde_s_scaled": round(cpb["measured_s"]["lde_s"] * cpb["scaled_to_columns"] / cpb["measured_columns"], 2)}
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
