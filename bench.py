#!/usr/bin/env python3
"""bench.py -- BASELINE.json's metric on BASELINE.json's configurations.

metric : GB/s of input scanned with bit-exact match ids (fsm_exec semantics)

  --config 2 (default; the headline, N=1 workload = BASELINE configs[1])
        one 256-state DFA (PCRE a[ -~]{7}\\z built by the reference: re_comp -> fsm_determinise ->
        fsm_minimise; golden fixture), 2^20 inputs x 1 KiB synthetic ASCII per GPU.  N > 1: the batch is
        range-sharded (weak scaling); result records reach every rank FUSED with the scan (lanes store
        them into every peer's gathered buffer over NVLink P2P) or by one NCCL all-gather (--gather nccl).
  --config 1  re(1)'s plumbing: PCRE [0-9]+\\.[0-9]+ over 1 MiB of synthetic ASCII through the relinked
        libfsm's own fsm_exec(fsm, fsm_sgetc, ...) (libfsm_b200/shim); --size scales the text.
  --config 3  rx(1)-style 128-pattern union (mostly unanchored: fsm_union_repeated_pattern_group + eager
        outputs, built by the reference, golden fixture) over 10 M synthetic log lines per GPU: records +
        fired-id bitsets; sub-record: the start-anchored end-id variant.
  --config 4  examples/utf8dfa validator (starred; golden fixture, fsm_equal-pinned) over 2 GiB of
        synthetic UTF-8 per GPU -- 16 GiB range-sharded at --gpus 8: per-rank K1b shard maps, ONE
        all-gather of [T] records, composition in rank order, first-invalid offset checked.
  --config 5  fsm_determinise of the 100 001-state synthetic NFA (K2); metric DFA edges/s, "replicas only".

A "step" is one pass of the hot path over one batch.  `value`: inputs resident in HBM, CUDA events on
the launching stream.  `e2e`: through the host entry point of the C ABI with pinned HOST buffers, H2D and
D2H inside the timed region.  `--impl reference`: the reference's own CPU implementation (oracle/_ref,
compiled from the reference sources) on this box's host cores, a bounded sample of the same workload per
step; it never loads the engine library.  Both arms print the same `config`.

  python bench.py [--config C] [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dist uniform|adversarial]
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "GB/s input scanned (bit-exact match ids)"
N_INPUTS, LENGTH = 1 << 20, 1024                 # config 2
CFG3_LINES = 10_000_000
CFG4_BYTES = 2 << 30                             # per GPU: 16 GiB at 8 GPUs
CFG2_REF_SAMPLE, CFG3_REF_SAMPLE, CFG4_REF_SAMPLE = 32768, 16384, 32 << 20


# ------------------------------------------------------------------------------------------ shared

def the_config(args) -> dict:
    """What is measured -- identical in both arms (a function of the command line only)."""
    c = args.config
    if c == 1:
        return {"workload": f"configs[0]: re(1) plumbing, PCRE [0-9]+\\.[0-9]+ over {args.size} B of synthetic ASCII, one fsm_exec call",
                "config_index": 1, "l2": "input smaller than L2: a 256 MiB buffer is written between timed iterations",
                "reference_sample": "the whole text, one thread (one fsm_exec call is serial)"}
    if c == 2:
        return {"workload": "configs[1]: 256-state DFA a[ -~]{7}\\z, 2^20 x 1 KiB ASCII per GPU", "config_index": 2,
                "distribution": args.dist, "l2": "1 GiB input per step > 126 MB L2: no flush needed",
                "reference_sample": f"{CFG2_REF_SAMPLE} x {LENGTH} B inputs of the same distribution per step (seed 42)"}
    if c == 3:
        return {"workload": f"configs[2]: rx-style 128-pattern PCRE union (fsm_union_repeated_pattern_group, eager outputs, det + min) "
                            f"over {CFG3_LINES} synthetic log lines (64-256 B) per GPU", "config_index": 3,
                "l2": "1.6 GB of lines per step > 126 MB L2: no flush needed",
                "reference_sample": f"{CFG3_REF_SAMPLE} lines of the same generator per step (seed 7)"}
    if c == 4:
        return {"workload": f"configs[3]: examples/utf8dfa validator (starred) over {CFG4_BYTES} B of synthetic UTF-8 per GPU, "
                            "one fsm_exec call over the range-sharded stream", "config_index": 4,
                "l2": "2 GiB per step > 126 MB L2: no flush needed",
                "reference_sample": f"{CFG4_REF_SAMPLE} B of the same text per step, one thread (one fsm_exec call is serial)"}
    return {"workload": "configs[4]: fsm_determinise of the 100 001-state synthetic NFA (2000 chains x 50 literals + /./ loop)",
            "config_index": 5, "l2": "not a streaming kernel", "reference_sample": "the whole NFA, one thread"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "MEASURED_PEAKS.json (measured)"
    return {"hbm_gbs": 6650.0}, "fallback 6.65 TB/s (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def finish(self):
        self.stop_flag = True
        self.join()
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def load_fsm(config: int):
    import goldenio
    if config in (1, 2):
        cases = goldenio.load_exec_cases(os.path.join(goldenio.GOLDEN_DIR, "golden_exec.npz"))
        return next(c for c in cases if c["name"] == ("cfg2:uniform" if config == 2 else "cfg1:digits"))["fsm"]
    if config == 3:
        return goldenio.load_cfg3()
    if config == 4:
        return goldenio.load_cfg4()["fsm"]
    from libfsm_b200 import workloads
    return workloads.config5_nfa()


def cfg1_text(size: int) -> np.ndarray:
    """Seeded ASCII: digits with '.' at density 1/64 (SURVEY.md 8d config 1); never a NUL."""
    rng = np.random.default_rng(1)
    a = rng.integers(ord("0"), ord("9") + 1, size=size, dtype=np.uint8)
    a[rng.random(size) < 1.0 / 64] = ord(".")
    a[rng.random(size) < 0.25] = ord("x")
    return a


def thread_sweep(threads: int):
    return sorted({max(1, threads), max(1, threads // 2), max(1, threads // 4), 1}, reverse=True)


# ------------------------------------------------------------------------------- CPU reference legs

def cpu_leg_cfg2(fsm, host_sample: np.ndarray, threads: int, full_at: int | None = None):
    """The reference's own fsm_exec (oracle/_ref) on the host cores, as-is (per-call fsm_isdfa) and
    amortised (validation hoisted): best thread count of a sweep, and the 1-thread figures."""
    import reflib
    n = host_sample.shape[0]
    offsets = np.arange(n + 1, dtype=np.uint64) * np.uint64(host_sample.shape[1])
    flat = host_sample.reshape(-1)
    L = host_sample.shape[1]
    part = lambda frac: (flat[:(n // frac) * L], offsets[:n // frac + 1])
    if reflib.have_ref():
        R = reflib.Ref(); h = R.from_flat(fsm); kind = "reference"
        run = lambda mode, t, frac: R.exec_batch(h, *part(frac), mode=mode, nthreads=t)
    else:
        O = reflib.Oracle(); h = None; kind = "port"
        run = lambda mode, t, frac: O.exec_batch(fsm, *part(frac), nthreads=t, validate_each=(mode == 0))
    out = sweep_modes(run, flat.size, threads, full_at)
    if h is not None:
        # secondary baseline (SURVEY 8a11): the reference's bytecode engine fsm_vm_match_buffer (yes / no only)
        fb, ob = part(4)
        t0 = time.perf_counter(); vm = R.vm_match_batch(h, fb, ob, nthreads=threads); dt = time.perf_counter() - t0
        f1, o1 = part(16)
        t0 = time.perf_counter(); R.vm_match_batch(h, f1, o1, nthreads=1); dt1 = time.perf_counter() - t0
        rec = R.exec_batch(h, fb, ob, mode=1, nthreads=threads)
        assert ((vm == 1) == (rec["ret"] == 1)).all(), "fsm_vm_match_buffer and fsm_exec disagree"
        out["cpu_vm"] = {"entry": "fsm_vm_match_buffer (DFAVM interpreter, vm.c:218-229; verdict only)", "gbs": fb.size / dt / 1e9,
                         "threads": threads, "gbs_1t": f1.size / dt1 / 1e9}
        R.free(h)
    out["kind"] = kind
    return out


def sweep_modes(run, nbytes: int, threads: int, full_at: int | None = None):
    """run(mode, nthreads, frac) scans 1/frac of the sample; mode 0 as-is, 1 amortised.  The full sample
    runs at the full thread count only (as-is: the timed quantity); the thread sweep, the amortised mode
    and the 1-thread figures use a quarter / a sixteenth of it, so that one leg stays within seconds."""
    def timed(mode, t, frac):
        t0 = time.perf_counter(); r = run(mode, t, frac); dt = time.perf_counter() - t0
        return r if isinstance(r, float) else dt          # a leg may report its own timed region
    full = full_at or threads                             # thread count of the full-sample (timed) run
    asis_s = timed(0, full, 1)
    best = {"asis": (nbytes / asis_s / 1e9, full), "amortised": (0.0, 0)}
    one = {}
    for t in thread_sweep(threads):
        frac = 16 if t == 1 else 4
        for name, mode in (("asis", 0), ("amortised", 1)):
            if name == "asis" and t == full:
                continue
            dt = timed(mode, t, frac)
            g = nbytes / frac / dt / 1e9
            if t == 1:
                one[name] = g
            if g > best[name][0]:
                best[name] = (g, t)
    if threads == 1:
        one.setdefault("asis", best["asis"][0])
    return {"asis_gbs": best["asis"][0], "asis_threads": best["asis"][1], "asis_s": asis_s, "asis_full_threads_gbs": nbytes / asis_s / 1e9,
            "amortised_gbs": best["amortised"][0], "amortised_threads": best["amortised"][1],
            "asis_1t_gbs": one.get("asis"), "amortised_1t_gbs": one.get("amortised"), "threads_swept": thread_sweep(threads)}


def cpu_baseline_record(cpu: dict, sample: str) -> dict:
    return {"value": cpu["asis_gbs"], "unit": "GB/s", "cores": cpu["asis_threads"], "kind": cpu["kind"], "sample": sample,
            "amortised_value": cpu["amortised_gbs"], "amortised_cores": cpu["amortised_threads"],
            "cpu_1t": {"as_is": cpu["asis_1t_gbs"], "amortised": cpu["amortised_1t_gbs"]}, "threads_swept": cpu["threads_swept"],
            **({"cpu_vm": cpu["cpu_vm"]} if "cpu_vm" in cpu else {})}


def cpu_leg_cfg3(g, nlines: int, threads: int, full_at: int | None = None):
    import reflib
    from libfsm_b200 import workloads
    _, inst = workloads.cfg3_patterns()
    base, off = workloads.cfg3_lines_host(nlines, inst, seed=7)
    fsm, ids = g["eager"]["fsm"], g["eager"]["idlist"]
    assert reflib.have_ref(), "config 3's CPU leg needs the compiled reference (oracle/_ref)"
    R = reflib.Ref(); h = R.from_flat(fsm)
    def run(mode, t, frac):
        k = nlines // frac
        R.exec_eager_batch(h, base[:int(off[k])], off[:k + 1], ids, mode=mode, nthreads=t)
        return R.last_walk_seconds()                      # thread start to join: not the harness's per-thread fsm_clone
    out = sweep_modes(run, int(off[-1]), threads, full_at)
    R.free(h)
    out["kind"] = "reference"
    return out


def cpu_leg_stream(fsm, text: np.ndarray):
    """One reference fsm_exec call over `text` (serial by nature), as-is; amortised = the reference's
    own per-byte transition without the per-call validation.  Without the compiled reference, the
    oracle's port of the same walk (kind "port"), as in the config-2 leg."""
    import reflib
    off = np.array([0, text.size], dtype=np.uint64)
    if reflib.have_ref():
        R = reflib.Ref(); h = R.from_flat(fsm); kind = "reference"
        t0 = time.perf_counter(); rc, end, consumed = R.exec(h, text.tobytes()); dt0 = time.perf_counter() - t0
        t0 = time.perf_counter(); R.exec_batch(h, text, off, mode=1, nthreads=1); dt1 = time.perf_counter() - t0
        R.free(h)
    else:
        O = reflib.Oracle(); kind = "port"
        t0 = time.perf_counter(); rc, end, consumed = O.exec(fsm, text.tobytes()); dt0 = time.perf_counter() - t0
        t0 = time.perf_counter(); O.exec_batch(fsm, text, off); dt1 = time.perf_counter() - t0
    g0, g1 = text.size / dt0 / 1e9, text.size / dt1 / 1e9
    return {"asis_gbs": g0, "asis_threads": 1, "asis_s": dt0, "amortised_gbs": g1, "amortised_threads": 1,
            "asis_1t_gbs": g0, "amortised_1t_gbs": g1, "threads_swept": [1], "kind": kind,
            "record": (int(rc), int(end), int(consumed))}


def cpu_leg_determinise(nfa):
    import reflib
    assert reflib.have_ref()
    R = reflib.Ref(); h = R.from_flat(nfa)
    t0 = time.perf_counter(); R.determinise(h); dt = time.perf_counter() - t0
    states = R.countstates(h)
    R.free(h)
    return dt, states


def run_reference_arm(args):
    """--impl reference: the reference's CPU implementation on this box's host cores, a bounded sample
    of the same workload per step.  Imports nothing of the engine."""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    from libfsm_b200 import workloads
    threads = host_threads()
    cfg = the_config(args)
    fsm = load_fsm(args.config)
    unit, metric = "GB/s", METRIC
    if args.config == 2:
        host = workloads.cfg2_host(CFG2_REF_SAMPLE, LENGTH, args.dist == "adversarial", seed=42)
        leg = lambda full_at=None: cpu_leg_cfg2(fsm, host, threads, full_at)
        warm = lambda: cpu_leg_cfg2(fsm, host[:2048], threads)
        nbytes = CFG2_REF_SAMPLE * LENGTH
    elif args.config == 3:
        leg = lambda full_at=None: cpu_leg_cfg3(fsm, CFG3_REF_SAMPLE, threads, full_at)
        warm = lambda: cpu_leg_cfg3(fsm, 1024, threads)
        nbytes = None
    elif args.config in (1, 4):
        text = cfg1_text(args.size) if args.config == 1 else workloads.utf8_host(CFG4_REF_SAMPLE, seed=4)
        leg = lambda full_at=None: cpu_leg_stream(fsm, text)
        warm = lambda: cpu_leg_stream(fsm, text[:1 << 16])
        nbytes = text.size
    else:
        metric, unit = "DFA edges/s (fsm_determinise)", "edges/s"
        edges = None
    t_total, last = 0.0, None
    if args.config == 5:
        import reflib
        for _ in range(min(args.warmup, 1)):
            cpu_leg_determinise(workloads.config5_nfa(words=200))
        for _ in range(args.steps):
            dt, states = cpu_leg_determinise(fsm)
            t_total += dt
        edges = states * 256                                  # the config-5 DFA is complete: 256 edges per state
        value = edges * args.steps / t_total
        cpu = {"value": value, "unit": unit, "cores": 1, "kind": "reference", "sample": cfg["reference_sample"],
               "seconds_per_determinise": t_total / args.steps, "dfa_states": states}
    else:
        for _ in range(args.warmup):
            warm()
        # the timed steps run fsm_exec as-is at the thread count that a calibration sweep found fastest
        # (on this workload the per-call validation scales worse than the walk: 64 threads beat 128)
        best_threads = leg()["asis_threads"]
        for _ in range(args.steps):
            last = leg(best_threads)
            t_total += last["asis_s"]
        if nbytes is None:
            nbytes = int(last["asis_gbs"] * last["asis_s"] * 1e9 + 0.5)
        value = nbytes * args.steps / t_total / 1e9
        cpu = cpu_baseline_record(last, cfg["reference_sample"])
        cpu["value"], cpu["cores"] = value, (best_threads if args.config in (2, 3) else 1)
        assert "libfsm_b200.so" not in open("/proc/self/maps").read(), "the reference arm must not load the engine"
    line = {"impl": "reference", "metric": metric, "value": value, "unit": unit, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_total / max(args.steps, 1) * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8" if args.config != 5 else "u32", "data": "synthetic", "config": cfg,
            "reference_entry": "fsm_exec as-is (per-call fsm_isdfa validation); the amortised figure hoists it" if args.config != 5 else "fsm_determinise",
            "cpu_baseline": cpu, "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------------------- GPU arm

class Ctx:
    pass


def gpu_setup(args) -> Ctx:
    import torch
    import torch.distributed as dist
    c = Ctx()
    c.torch, c.dist = torch, dist
    c.world = int(os.environ.get("WORLD_SIZE", "1"))
    c.rank = int(os.environ.get("RANK", "0"))
    c.local = int(os.environ.get("LOCAL_RANK", "0"))
    if c.world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout carries ONE JSON line: whatever native libraries print on fd 1 (NCCL's "NCCL version ..."
        # banner under NCCL_DEBUG=VERSION) goes to stderr; Python's own stdout keeps the real one
        sys.stdout.flush()
        sys.stdout = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=torch.device("cuda", c.local))
    assert c.world == args.gpus or c.world == 1, f"WORLD_SIZE {c.world} != --gpus {args.gpus}"
    torch.cuda.set_device(c.local)
    c.dev = torch.device("cuda", c.local)
    c.main = torch.cuda.current_stream()
    c.side = torch.cuda.Stream(device=c.dev) if c.world > 1 else None
    return c


def sync_all(c: Ctx):
    c.torch.cuda.synchronize(c.dev)
    if c.world > 1:
        c.dist.barrier()
        c.torch.cuda.synchronize(c.dev)


def timed_region(c: Ctx, step, steps: int, warmup: int):
    """W untimed steps, then exactly K steps between CUDA events on the launching stream, a barrier +
    synchronize on both sides; returns (ms_total, launches, clocks)."""
    import libfsm_b200 as L
    for i in range(warmup):
        step(i)
    sync_all(c)
    # N > 1: the first multi-GPU job on a fresh box runs its first seconds at half speed (measured at N=8:
    # 0.41 ms per step in the first torchrun of a box, 0.19-0.21 in every later one, same kernels, same
    # per-kernel time: one rank lags and every rank's consumer waits for it).  Untimed blocks of 25 steps
    # until two consecutive blocks agree within 5 % (decided on all-reduced times, so every rank takes
    # the same decision), at most 40 blocks; the timed region below is still exactly K steps.
    c.settle = []
    if c.world > 1:
        prev = None
        for blk in range(40):
            a, b = c.torch.cuda.Event(enable_timing=True), c.torch.cuda.Event(enable_timing=True)
            a.record(c.main)
            for i in range(25):
                step(i)
            if c.side is not None:
                c.main.wait_stream(c.side)
            b.record(c.main)
            sync_all(c)
            ms = reduce_max(c, [a.elapsed_time(b)])[0]
            c.settle.append(round(ms / 25, 4))
            if blk >= 3 and prev is not None and abs(ms - prev) <= 0.05 * prev:
                break
            prev = ms
    sampler = ClockSampler(c.local); sampler.start()
    L.launch_count(reset=True)
    e0, e1 = c.torch.cuda.Event(enable_timing=True), c.torch.cuda.Event(enable_timing=True)
    e0.record(c.main)
    for i in range(steps):
        step(i)
    if c.side is not None:
        c.main.wait_stream(c.side)
    e1.record(c.main)
    sync_all(c)
    return e0.elapsed_time(e1), L.launch_count(), sampler


def kernel_ms(c: Ctx, launch, reps: int) -> float:
    """Mean duration of `launch` (one kernel) from CUDA events around each launch on the launching stream."""
    ev = [(c.torch.cuda.Event(enable_timing=True), c.torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    if c.world > 1:
        c.dist.barrier()
    for a, b in ev:
        a.record(c.main); launch(); b.record(c.main)
    c.torch.cuda.synchronize(c.dev)
    return float(np.mean([a.elapsed_time(b) for a, b in ev]))


def reduce_max(c: Ctx, values):
    t = c.torch.tensor(values, dtype=c.torch.float64, device=c.dev)
    if c.world > 1:
        c.dist.all_reduce(t, op=c.dist.ReduceOp.MAX)
    return [float(x) for x in t.cpu()]


def roofline_record(bytes_per_launch: int, kms: float, kernel: str, traffic_file: str | None = None) -> dict:
    peaks, peak_src = measured_peaks()
    achieved = bytes_per_launch / (kms / 1e3) / 1e9
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", traffic_file) if traffic_file else None
    if tp and os.path.exists(tp):
        tj = json.load(open(tp))
        traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
        traffic_src = f"{tj['source']}: dram__bytes_read.sum + dram__bytes_write.sum per launch of {tj['kernel']}"
    return {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
            "peak_source": peak_src, "kernel": kernel, "kernel_ms": kms, "algorithmic_bytes_per_launch": bytes_per_launch,
            "traffic": traffic, "traffic_source": traffic_src}


def base_line(args, c: Ctx, value, ms_per_step, unit="GB/s", metric=METRIC, dtype="u8") -> dict:
    return {"metric": metric, "value": value, "unit": unit, "n_gpus": c.world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dtype,
            "data": "synthetic", "config": the_config(args)}


def finish(c: Ctx):
    if c.world > 1:
        c.dist.barrier()
        c.dist.destroy_process_group()
    return 0


# ---- config 2 ------------------------------------------------------------------------------------

def run_cfg2(args):
    import libfsm_b200 as L
    import reflib
    from libfsm_b200 import workloads
    c = gpu_setup(args)
    torch, dist, dev, world, rank, local = c.torch, c.dist, c.dev, c.world, c.rank, c.local
    fsm = load_fsm(2)
    dfa = L.Dfa(fsm, device=local)
    L.set_exec_variant(args.variant)
    adversarial = args.dist == "adversarial"
    n = N_INPUTS
    d_in = workloads.cfg2_device(n, LENGTH, adversarial, seed=42 + 1000 * rank, device=dev)   # range shard `rank`
    # buffers in flight: the gather of step i is only waited for when its buffer is reused at step i + nbuf
    nbuf = int(os.environ.get("BENCH_NBUF", "4"))
    fused = world > 1 and args.gather == "fused"
    d_out = [torch.empty((n, 16), dtype=torch.uint8, device=dev) for _ in range(nbuf)]
    gathered = [torch.empty((world * n, 16), dtype=torch.uint8, device=dev) for _ in range(nbuf)] if world > 1 else None
    gather_done = [None] * nbuf
    ring, compact = None, False
    token = torch.zeros(1, dtype=torch.int32, device=dev)
    if fused:
        from libfsm_b200.peer import GatherRing
        compact = args.gather_records == "compact"
        try:
            ring = GatherRing(n, world, rank, local, nbuf, elem_bytes=4 if compact else 16)
            ok = torch.ones(1, dtype=torch.int32, device=dev)
        except Exception as e:                      # no peer access on this box: NCCL all-gather instead
            print(f"[bench] rank {rank}: peer mapping failed ({e}); falling back to --gather nccl", file=sys.stderr)
            ring = None
            ok = torch.zeros(1, dtype=torch.int32, device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)   # every rank must agree on the path
        if int(ok.item()) == 0:
            if ring is not None:
                ring.close()
            ring, fused, compact = None, False, False
            args.gather = "nccl"
    if fused:
        peer_args = [ring.peer_slot_ptrs(b) for b in range(nbuf)]
        sig_args = [ring.signal_args(b) for b in range(nbuf)]
        own_out = [torch.empty((n, 16), dtype=torch.uint8, device=dev) for _ in range(nbuf)] if compact else None
    use_flags = fused and args.handshake == "flags"
    consume = use_flags and not args.no_consumer

    def local_out_ptr(b):
        return own_out[b].data_ptr() if (fused and compact) else ring.local_slot_ptr(b)

    step_no = [0]

    def step(_i):
        i = step_no[0]; step_no[0] += 1              # global step number: the flag value of step i is i + 1
        b = i % nbuf
        if world > 1 and gather_done[b] is not None:
            c.main.wait_event(gather_done[b])                 # buffer free again
        if consume and i >= nbuf:
            # CONSUMER inside the timed loop: before buffer b is overwritten, a poll kernel waits until
            # every rank's completion flag of the step that last used it (i - nbuf) has arrived, i.e.
            # every peer's records of that step have landed in this rank's gathered buffer
            ring.wait_flags(b, i - nbuf + 1)
        if fused:
            dfa.exec_batch_gather(d_in, stride=LENGTH, length=LENGTH, n=n, out_ptr=local_out_ptr(b),
                                  peer_ptrs=peer_args[b][0], npeers=peer_args[b][1], compact=compact,
                                  sig_counter=sig_args[b][0] if use_flags else None,
                                  sig_flags=sig_args[b][1] if use_flags else None, sig_value=i + 1)
        else:
            dfa.exec_batch(d_in, stride=LENGTH, length=LENGTH, n=n, out=d_out[b])
        if world > 1 and (not fused or args.handshake == "nccl"):
            ev = torch.cuda.Event(); ev.record(c.main)
            c.side.wait_event(ev)
            with torch.cuda.stream(c.side):
                if fused:
                    dist.all_reduce(token)                  # 4-byte completion handshake, off the data path
                else:
                    dist.all_gather_into_tensor(gathered[b], d_out[b])
                gather_done[b] = torch.cuda.Event(); gather_done[b].record(c.side)

    # ---- parity gate: the results we are about to time are the reference's ---------------
    step(0); sync_all(c)
    oracle = reflib.Oracle()
    idx = torch.arange(0, n, 64, device=dev)
    sample_host = d_in[idx].cpu().numpy()
    off = np.arange(sample_host.shape[0] + 1, dtype=np.uint64) * np.uint64(LENGTH)
    want = oracle.exec_batch(fsm, sample_host.reshape(-1), off, nthreads=min(16, os.cpu_count() or 1))
    if use_flags:
        flags = ring.read_flags(0)                         # step 0 was launched with sig_value 1
        assert (flags == 1).all(), f"bench: completion flags {flags} != 1 after step 0"
    if fused and compact:
        mine = L.results_from_torch(own_out[0])
        assert (mine[::64] == want).all(), "bench: GPU results differ from the oracle"
        ids = ((mine["ret"] == 1).astype(np.uint32) << np.uint32(31)) | mine["end"]
        everything = ring.read(0)                          # peers' match ids (own slot is not written)
        ids_t = torch.from_numpy(ids.view(np.int32).copy()).to(dev)
        allids = torch.empty(world * n, dtype=torch.int32, device=dev)
        dist.all_gather_into_tensor(allids, ids_t)         # NCCL reference for the P2P-gathered ids
        torch.cuda.synchronize(dev)
        ref_ids = allids.cpu().numpy().view(np.uint32)
        for r in range(world):
            if r != rank:
                assert (everything[r * n:(r + 1) * n] == ref_ids[r * n:(r + 1) * n]).all(), "bench: fused gather != NCCL all-gather"
    elif fused:
        everything = ring.read(0)                          # this rank's gathered buffer: all ranks' records
        got = everything[rank * n:(rank + 1) * n][::64]
        assert (got == want).all(), "bench: GPU results differ from the oracle"
        mine_t = torch.from_numpy(everything[rank * n:(rank + 1) * n].view(np.uint8).reshape(n, 16).copy()).to(dev)
        dist.all_gather_into_tensor(gathered[0], mine_t)
        torch.cuda.synchronize(dev)
        assert (L.results_from_torch(gathered[0]) == everything).all(), "bench: fused gather != NCCL all-gather"
    else:
        got = L.results_from_torch(d_out[0][idx])
        assert (got == want).all(), "bench: GPU results differ from the oracle"
        if world > 1:
            mine = gathered[0][rank * n:(rank + 1) * n]
            assert torch.equal(mine, d_out[0]), "bench: all-gather slot mismatch"

    ms_total, launches, sampler = timed_region(c, step, args.steps, args.warmup)
    if args.dump_outputs is not None and rank == 0:
        last = (step_no[0] - 1) % nbuf                    # the buffer the last timed step wrote
        if fused and compact:
            recs = L.results_from_torch(own_out[last])
        elif fused:
            recs = ring.read(last)[rank * n:(rank + 1) * n]
        else:
            recs = L.results_from_torch(d_out[last])
        dump_outputs(args.dump_outputs, record_fields(recs))

    def one_kernel(inp=d_in):
        if fused:
            dfa.exec_batch_gather(inp, stride=LENGTH, length=LENGTH, n=n, out_ptr=local_out_ptr(0),
                                  peer_ptrs=peer_args[0][0], npeers=peer_args[0][1], compact=compact)
        else:
            dfa.exec_batch(inp, stride=LENGTH, length=LENGTH, n=n, out=d_out[0])
    kms = kernel_ms(c, one_kernel, args.steps)
    clocks = sampler.finish()

    # the other distribution of SURVEY 8d ("report both"): kernel-only, same launch configuration
    other = None
    if world == 1:
        d_other = workloads.cfg2_device(n, LENGTH, not adversarial, seed=42, device=dev)
        for _ in range(3):
            one_kernel(d_other)
        oms = kernel_ms(c, lambda: one_kernel(d_other), max(5, min(args.steps, 20)))
        hs = d_other[idx].cpu().numpy()
        w2 = oracle.exec_batch(fsm, hs.reshape(-1), off, nthreads=min(16, os.cpu_count() or 1))
        torch.cuda.synchronize(dev)
        assert (L.results_from_torch(d_out[0][idx]) == w2).all(), "bench: GPU results differ from the oracle (other distribution)"
        peaks, _ = measured_peaks()
        g = n * LENGTH / (oms / 1e3) / 1e9
        other = {"distribution": "uniform" if adversarial else "adversarial", "kernel_ms": oms, "value": g, "unit": "GB/s",
                 "frac_of_hbm_peak": g / peaks["hbm_gbs"], "parity": "1/64 sample bit-exact vs the oracle"}
        del d_other

    # ---- end to end through the host entry point, pinned host buffers --------------------
    h_in = torch.empty((n, LENGTH), dtype=torch.uint8, pin_memory=True)
    h_in.copy_(d_in)
    h_off = torch.arange(0, (n + 1) * LENGTH, LENGTH, dtype=torch.int64).pin_memory()
    h_out = torch.empty((n, 16), dtype=torch.uint8, pin_memory=True)
    e2e_steps = args.e2e_steps if args.e2e_steps is not None else max(3, min(args.steps, 10))
    numa = bind_to_gpu_numa(local) if world > 1 else None
    for _ in range(2):
        dfa.exec_batch_hostptr(h_in.data_ptr(), h_off.data_ptr(), n, h_out.data_ptr())
    assert (L.results_from_torch(h_out)[::64] == want).all()
    sync_all(c)
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        dfa.exec_batch_hostptr(h_in.data_ptr(), h_off.data_ptr(), n, h_out.data_ptr())
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0

    ms_total, e2e_ms, kms = reduce_max(c, [ms_total, e2e_s * 1e3, kms])
    bytes_step = n * LENGTH
    if rank == 0:
        threads = host_threads()
        cpu = cpu_leg_cfg2(fsm, workloads.cfg2_host(CFG2_REF_SAMPLE, LENGTH, adversarial, seed=42), threads)
        line = base_line(args, c, world * bytes_step * args.steps / (ms_total / 1e3) / 1e9, ms_total / args.steps)
        line["engine"] = {"variant": args.variant, "table": dfa.info,
                          "multi_gpu": ("single GPU" if world == 1 else
                                        f"range-sharded batch; scan fused with the gather: lanes store "
                                        f"{'4 B match ids ((ret==1)<<31|end)' if compact else '16 B records'} into every peer's buffer over NVLink P2P; "
                                        f"completion signal: {args.handshake}; consumer in the timed loop: {'poll kernel on the flags before a buffer is reused' if consume else 'none'}"
                                        if fused else "range-sharded batch, one NCCL all-gather of 16 B result records per step on a side stream"),
                          "e2e_numa": numa, "untimed_settle_blocks_ms_per_step": getattr(c, "settle", [])}
        line["clocks"] = clocks
        line["e2e"] = {"value": world * bytes_step * e2e_steps / (e2e_ms / 1e3) / 1e9, "unit": "GB/s", "steps": e2e_steps,
                       "h2d_bytes_per_step": int(h_in.numel() + h_off.numel() * 8), "d2h_bytes_per_step": int(h_out.numel()),
                       "entry": "fsm_b200_exec_batch_host, pinned host buffers"}
        line["gpu_launches"] = int(launches)
        line["roofline"] = roofline_record(bytes_step, kms, "k1_krange_tile_kernel (4-byte stride, ALU byte classification, 2-D TMA input tiles)" if dfa.info["krange"] and args.variant in ("auto", "kstride") else args.variant,
                                           "r2_k1_traffic.json" if args.dist == "uniform" else None)
        if other is not None:
            line["other_distribution"] = other
        line["cpu_baseline"] = cpu_baseline_record(cpu, the_config(args)["reference_sample"])
        print(json.dumps(line), flush=True)
    dfa.close()
    if world > 1:
        dist.barrier()
        if ring is not None:
            ring.close()
    return finish(c)


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """--dump-outputs: each array as DIR/<name>.npy in float64, which holds every value written here exactly
    (integers below 2^53: 64-bit bitsets are split into 32-bit words first)."""
    out = {name: np.asarray(a).astype(np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the 64 MiB limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def record_fields(recs: np.ndarray) -> dict:
    """The fields of result records (ret, end, consumed) as separate arrays."""
    return {name: recs[name] for name in recs.dtype.names}


def dense_rows(f, states: np.ndarray) -> np.ndarray:
    """Rows [len(states), 256] of f's dense transition table (0xFFFFFFFF = no edge; the first group that
    holds a symbol wins, as in FlatFsm.dense_table), computed for the given states only."""
    rows = np.full((len(states), 256), 0xFFFFFFFF, dtype=np.uint32)
    for k, s in enumerate(states):
        lo, hi = int(f.group_off[s]), int(f.group_off[s + 1])
        bits = np.unpackbits(np.ascontiguousarray(f.group_symbols[lo:hi], dtype="<u8").view(np.uint8).reshape(hi - lo, 32),
                             axis=1, bitorder="little").astype(bool)
        for g in range(hi - lo - 1, -1, -1):
            rows[k, bits[g]] = f.group_to[lo + g]
    return rows


def u32_words(a) -> np.ndarray:
    """64-bit words as pairs of 32-bit words (low first), exact in float64."""
    return np.ascontiguousarray(a).view(np.uint64).view(np.uint32).reshape(len(a), -1)


def bind_to_gpu_numa(local: int):
    """e2e at N > 1: keep this rank's host threads (the copy loop of exec_batch_host runs on the calling
    thread) and the page placement of what it allocates from now on on the NUMA node of its GPU."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        node = None
        try:
            node = pynvml.nvmlDeviceGetNumaNodeId(h)
        except Exception:
            pass
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinityWithinScope(h, words, pynvml.NVML_AFFINITY_SCOPE_NODE)
        cpus = [64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1]
        cpus = [x for x in cpus if x in os.sched_getaffinity(0)]
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus)}
    except Exception as e:                                   # noqa: BLE001
        return {"error": repr(e)}


# ---- config 3 ------------------------------------------------------------------------------------

def run_cfg3(args):
    import libfsm_b200 as L
    import reflib
    from libfsm_b200 import workloads
    c = gpu_setup(args)
    torch, dist, dev, world, rank, local = c.torch, c.dist, c.dev, c.world, c.rank, c.local
    g = load_fsm(3)
    fsm, ids = g["eager"]["fsm"], g["eager"]["idlist"]
    _, inst = workloads.cfg3_patterns()
    nlines = int(os.environ.get("BENCH_CFG3_LINES", CFG3_LINES))
    base, offsets = workloads.cfg3_lines_device(nlines, inst, seed=7 + 1000 * rank, device=dev)
    total = int(offsets[-1])
    dfa = L.Dfa(fsm, device=local)
    words = (ids.size + 63) // 64
    rec = torch.empty((nlines, 16), dtype=torch.uint8, device=dev)
    masks = torch.zeros((nlines, words), dtype=torch.int64, device=dev)
    gathered = torch.empty((world * nlines, 16), dtype=torch.uint8, device=dev) if (world > 1 and os.environ.get("BENCH_CFG3_GATHER", "0") == "1") else None
    lib, chk = L._native.lib, L._native.check
    stream_ptr = int(c.main.cuda_stream)

    def launch():
        chk(lib.fsm_b200_exec_batch_eager_dev(dfa._h, base.data_ptr(), offsets.data_ptr(), 0, 0, nlines, rec.data_ptr(), masks.data_ptr(), stream_ptr),
            "exec_batch_eager_dev")

    gather = world > 1 and os.environ.get("BENCH_CFG3_GATHER", "0") == "1"

    def step(_i):
        launch()
        # Lines are independent and their records + id bitsets are consumed where they are produced: the
        # shards exchange nothing (SURVEY.md 8e: an all-gather only "if every rank needs them").
        # BENCH_CFG3_GATHER=1 adds one NCCL all-gather of the records per step on a side stream (measured
        # at N=2: 4.79 ms per step instead of 2.2 -- the collective's kernel waits for SMs the persistent
        # scan occupies; config 2 shows the fused alternative).
        if gather:
            ev = torch.cuda.Event(); ev.record(c.main)
            c.side.wait_event(ev)
            with torch.cuda.stream(c.side):
                dist.all_gather_into_tensor(gathered, rec)

    # parity gate: >= 200 k lines, records + fired-id sets bit-exact vs the compiled reference
    step(0); sync_all(c)
    ns = min(nlines, 200_000)
    hb = base[:int(offsets[ns])].cpu().numpy(); ho = offsets[:ns + 1].cpu().numpy().astype(np.uint64)
    assert reflib.have_ref(), "config 3's parity gate needs the compiled reference (oracle/_ref)"
    R = reflib.Ref(); h = R.from_flat(fsm)
    want, wmasks = R.exec_eager_batch(h, hb, ho, ids, mode=1, nthreads=min(32, host_threads()))
    R.free(h)
    got = L.results_from_torch(rec[:ns])
    assert (got == want).all(), "bench: config 3 records differ from the reference"
    assert (masks[:ns].cpu().numpy().view(np.uint64) == wmasks).all(), "bench: config 3 fired-id sets differ from the reference"

    ms_total, launches, sampler = timed_region(c, step, args.steps, args.warmup)
    if args.dump_outputs is not None and rank == 0:
        # 10 M lines of records + bitsets exceed 64 MiB: a fixed sample of 2^19 lines (seed 0), their indices included
        pick = np.sort(np.random.default_rng(0).choice(nlines, size=min(nlines, 1 << 19), replace=False))
        tpick = torch.from_numpy(pick).to(dev)
        dump_outputs(args.dump_outputs, {"line": pick, **record_fields(L.results_from_torch(rec[tpick])),
                                         "fired_words": u32_words(masks[tpick].cpu().numpy())})
    kms = kernel_ms(c, launch, args.steps)
    clocks = sampler.finish()

    # sub-record: the start-anchored end-id variant (rx(1)'s own recipe), plain records
    sub = None
    if world == 1:
        afsm = g["anchored"]["fsm"]
        _, ainst = workloads.cfg3_anchored_patterns()
        abase, aoff = workloads.cfg3_lines_device(nlines, ainst, seed=7, device=dev, at_start=True)
        with L.Dfa(afsm, device=local) as adfa:
            def alaunch():
                adfa.exec_batch(abase, aoff, out=rec)
            for _ in range(3):
                alaunch()
            torch.cuda.synchronize(dev)
            ams = kernel_ms(c, alaunch, max(5, min(args.steps, 20)))
            arec = L.results_from_torch(rec)
            walked = int(arec["consumed"].sum())
            hb2 = abase[:int(aoff[ns])].cpu().numpy(); ho2 = aoff[:ns + 1].cpu().numpy().astype(np.uint64)
            R = reflib.Ref(); h = R.from_flat(afsm)
            want2 = R.exec_batch(h, hb2, ho2, mode=1, nthreads=min(32, host_threads()))
            R.free(h)
            assert (arec[:ns] == want2).all(), "bench: anchored config 3 records differ from the reference"
            atotal = int(aoff[-1])
            peaks, _ = measured_peaks()
            sub = {"dfa": "128 start-anchored patterns, rx(1)'s recipe, end ids", "dfa_states": afsm.nstates, "table": adfa.info, "kernel_ms": ams,
                   "GBps_bytes_covered": atotal / ams / 1e6, "GBps_bytes_walked": walked / ams / 1e6,
                   "bytes_covered": atotal, "bytes_walked": walked, "frac_of_hbm_peak_walked": walked / ams / 1e6 / peaks["hbm_gbs"],
                   "note": "a line that dies (half of them, within their first bytes) or reaches an absorbing accept state is not read further; "
                           "bytes_walked = sum of the records' consumed offsets", "parity": f"{ns} lines bit-exact vs the compiled reference"}
        del abase, aoff

    # e2e: host lines -> fsm_b200_exec_batch_eager_host -> host records + bitsets
    h_base = torch.empty(total, dtype=torch.uint8, pin_memory=True); h_base.copy_(base)
    h_off = offsets.cpu().pin_memory()
    h_rec = torch.empty((nlines, 16), dtype=torch.uint8, pin_memory=True)
    h_masks = torch.zeros((nlines, words), dtype=torch.int64).pin_memory()
    e2e_steps = args.e2e_steps if args.e2e_steps is not None else 3

    def e2e_call():
        chk(lib.fsm_b200_exec_batch_eager_host(dfa._h, h_base.data_ptr(), h_off.data_ptr(), nlines, h_rec.data_ptr(), h_masks.data_ptr()),
            "exec_batch_eager_host")
    e2e_call()
    assert (L.results_from_torch(h_rec)[:ns] == want).all()
    sync_all(c)
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_call()
    e2e_s = time.perf_counter() - t0

    ms_total, e2e_ms, kms = reduce_max(c, [ms_total, e2e_s * 1e3, kms])
    if rank == 0:
        cpu = cpu_leg_cfg3(g, CFG3_REF_SAMPLE, host_threads())
        line = base_line(args, c, world * total * args.steps / (ms_total / 1e3) / 1e9, ms_total / args.steps)
        line["engine"] = {"table": dfa.info, "dfa_states": fsm.nstates, "eager_ids": int(ids.size), "end_ids": 10,
                          "lines": nlines, "bytes": total, "records": "16 B record + 16 B id bitset per line",
                          "bytes_read": "every byte of every line is walked (the union is unanchored: no line dies, no absorbing state)",
                          "multi_gpu": "single GPU" if world == 1 else ("lines range-sharded, one NCCL all-gather of the 16 B records per step on a side stream" if gather
                                                                        else "lines range-sharded over the ranks, no data-path collective: records and id bitsets stay with the shard that produced them")}
        line["clocks"] = clocks
        line["e2e"] = {"value": world * total * e2e_steps / (e2e_ms / 1e3) / 1e9, "unit": "GB/s", "steps": e2e_steps,
                       "h2d_bytes_per_step": int(total + h_off.numel() * 8), "d2h_bytes_per_step": int(h_rec.numel() + h_masks.numel() * 8),
                       "entry": "fsm_b200_exec_batch_eager_host, pinned host buffers"}
        line["gpu_launches"] = int(launches)
        line["roofline"] = roofline_record(total, kms, "k1_lines_kernel<u16, 2 mask words, eager>", "r2_lines_traffic.json")
        line["roofline"]["note"] = "bound by the shared-memory lookup rate (2 LDS per byte, bank conflicts), not HBM: see DESIGN.md"
        line["parity"] = f"{ns} lines: records and fired-id bitsets bit-exact vs the compiled reference (refh_exec_eager_batch)"
        if sub is not None:
            line["anchored_variant"] = sub
        line["cpu_baseline"] = cpu_baseline_record(cpu, the_config(args)["reference_sample"])
        print(json.dumps(line), flush=True)
    dfa.close()
    return finish(c)


# ---- config 4 (and config 1: the same path through the shim) --------------------------------------

def utf8_device(c: Ctx, nbytes: int, seed: int):
    """~nbytes of valid UTF-8 on the device: a seeded 64 MiB host block tiled (concatenating valid UTF-8
    keeps it valid); the last tile is cut at a code-point boundary."""
    from libfsm_b200 import workloads
    torch = c.torch
    block = workloads.utf8_host(64 << 20, seed=seed)
    reps = (nbytes + block.size - 1) // block.size
    out = torch.empty(nbytes, dtype=torch.uint8, device=c.dev)
    tb = torch.from_numpy(block).to(c.dev)
    pos = 0
    for _ in range(reps):
        m = min(block.size, nbytes - pos)
        out[pos:pos + m] = tb[:m]
        pos += m
    # a cut inside a multi-byte sequence: overwrite the tail with ASCII
    tail = out[-4:].cpu().numpy()
    k = 0
    while k < 4 and (tail[-1 - k] & 0xC0) == 0x80:
        k += 1
    if k < 4 and tail[-1 - k] >= 0xC0:
        out[-1 - k:] = 0x41
    return out


def run_cfg4(args):
    import libfsm_b200 as L
    import reflib
    from libfsm_b200 import sharding, workloads
    c = gpu_setup(args)
    torch, dist, dev, world, rank, local = c.torch, c.dist, c.dev, c.world, c.rank, c.local
    fsm = load_fsm(4)
    nbytes = int(os.environ.get("BENCH_CFG4_BYTES", CFG4_BYTES))
    dfa = L.Dfa(fsm, device=local)
    T = dfa.info["ntable_states"]
    shard = utf8_device(c, nbytes, seed=4)            # every shard: the same seeded valid text (a shard boundary is a code-point boundary)
    lens = [nbytes] * world

    # N > 1: every rank's shard map stays on the device (fsm_b200_exec_stream_map_dev_async), ONE NCCL all-gather
    # of the [nstates] x 16 B records queued behind it on the same stream, one read-back, composed in rank order
    NS = dfa.info["nstates"]
    my_map = torch.empty((NS, 2), dtype=torch.int64, device=dev)
    all_maps = torch.empty((world, NS, 2), dtype=torch.int64, device=dev)
    h_maps = torch.empty((world, NS, 2), dtype=torch.int64, pin_memory=True)

    def scan(buf):
        if world == 1:
            return dfa.exec_stream(buf)
        dfa.exec_stream_map_async(buf, my_map)
        dist.all_gather_into_tensor(all_maps, my_map)
        h_maps.copy_(all_maps, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        S, D, F = L.stream_map_arrays(h_maps.numpy())
        st, consumed, died = sharding.compose_stream_maps(fsm.start, None if dfa.info["complete"] else T - 1, lens,
                                                          list(S), list(D), list(F))
        return (0 if died else int(fsm.is_end[st]), st, consumed)

    # parity gate: valid text -> (1, end, total); one corrupted byte in the LAST rank's shard -> (0, ., global offset)
    ret, end, consumed = scan(shard)
    assert ret == 1 and consumed == nbytes * world, (ret, end, consumed)
    bad_at = nbytes // 2 + 12345
    if rank == world - 1:
        keep = shard[bad_at:bad_at + 1].clone()
        # make the byte at bad_at invalid in context: 0xFF never appears in UTF-8
        shard[bad_at] = 0xFF
    ret, end, consumed = scan(shard)
    assert ret == 0 and consumed == nbytes * (world - 1) + bad_at, (ret, consumed, nbytes * (world - 1) + bad_at)
    if rank == world - 1:
        shard[bad_at:bad_at + 1] = keep
    # and a 4 MiB prefix against the reference's own fsm_exec (rank 0)
    if rank == 0 and reflib.have_ref():
        pre = shard[:4 << 20].cpu().numpy()
        cut = pre.size
        while cut > 0 and (pre[cut - 1] & 0xC0) == 0x80:
            cut -= 1
        cut -= 1 if cut > 0 and pre[cut - 1] >= 0xC0 else 0
        R = reflib.Ref(); h = R.from_flat(fsm)
        rc, rend, rcons = R.exec(h, pre[:cut].tobytes())
        R.free(h)
        assert (rc, rcons) == dfa.exec_stream(shard[:cut])[0::2], "bench: config 4 differs from the reference on the prefix"

    last = [None]

    def step(_i):
        last[0] = scan(shard)
    ms_total, launches, sampler = timed_region(c, step, args.steps, args.warmup)
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(("ret", "end", "consumed"), ([v] for v in last[0]))))
    # the body kernel's share: exec_stream is a handful of launches; time the whole device-side call
    t = []
    for _ in range(max(3, min(args.steps, 10))):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(c.main); dfa.exec_stream(shard) if world == 1 else dfa.exec_stream_map(shard); b.record(c.main)
        torch.cuda.synchronize(dev); t.append(a.elapsed_time(b))
    kms = float(np.mean(t))
    clocks = sampler.finish()

    # e2e: pinned host text -> fsm_b200_exec_stream_host -> verdict (H2D of the whole shard inside)
    e2e_bytes = min(nbytes, 1 << 30)
    h_text = torch.empty(e2e_bytes, dtype=torch.uint8, pin_memory=True); h_text.copy_(shard[:e2e_bytes])
    r = L.desc.CResult()
    lib, chk = L._native.lib, L._native.check
    e2e_steps = args.e2e_steps if args.e2e_steps is not None else 3
    chk(lib.fsm_b200_exec_stream_host(dfa._h, h_text.data_ptr(), e2e_bytes, ctypes.byref(r)), "exec_stream_host")
    sync_all(c)
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        chk(lib.fsm_b200_exec_stream_host(dfa._h, h_text.data_ptr(), e2e_bytes, ctypes.byref(r)), "exec_stream_host")
    e2e_s = time.perf_counter() - t0

    ms_total, e2e_ms, kms = reduce_max(c, [ms_total, e2e_s * 1e3, kms])
    if rank == 0:
        cpu = cpu_leg_stream(fsm, workloads.utf8_host(CFG4_REF_SAMPLE, seed=4))
        line = base_line(args, c, world * nbytes * args.steps / (ms_total / 1e3) / 1e9, ms_total / args.steps)
        line["engine"] = {"table": dfa.info, "dfa": "examples/utf8dfa 0..10FFFF starred, det + min: 8 states (fsm_equal with the PCRE-built validator)",
                          "bytes_per_gpu": nbytes,
                          "stream_form": "fused small-automaton form (k1b_rep.cuh: per-lane replicated table, one single-wave kernel + final fold)"
                                         if T <= 12 and os.environ.get("FSM_B200_STREAM_REP", "1") != "0" else "generic chunked K1b (prefix + K1 body + compose)",
                          "multi_gpu": "single GPU: fsm_b200_exec_stream_dev" if world == 1 else
                                       f"{world} byte-range shards; per rank K1b shard map left on the device (exit state / first dead offset per entry state), ONE NCCL all-gather of [nstates] x 16 B records on the same stream, one read-back, composed in rank order"}
        line["clocks"] = clocks
        if world > 1:
            line["untimed_settle_blocks_ms_per_step"] = c.settle
        line["e2e"] = {"value": world * e2e_bytes * e2e_steps / (e2e_ms / 1e3) / 1e9, "unit": "GB/s", "steps": e2e_steps,
                       "h2d_bytes_per_step": int(e2e_bytes), "d2h_bytes_per_step": 16, "entry": "fsm_b200_exec_stream_host, pinned host text",
                       "bytes": e2e_bytes}
        line["gpu_launches"] = int(launches)
        line["roofline"] = roofline_record(nbytes, kms, "K1b, whole device-side call: k1b_rep_kernel (per-lane replicated table; prefix + body + warp/CTA fold in one single-wave kernel) + k1b_rep_final_kernel + read-back",
                                           "r2_k1b_rep_traffic.json")
        line["parity"] = "valid text: (1, end, total); one 0xFF at a known offset of the last shard: (0, ., global offset); 4 MiB prefix vs the reference's fsm_exec"
        line["cpu_baseline"] = cpu_baseline_record(cpu, the_config(args)["reference_sample"])
        print(json.dumps(line), flush=True)
    dfa.close()
    return finish(c)


def run_cfg1(args):
    """re(1)'s plumbing: the RELINKED libfsm (reference objects + libfsm_b200/shim replacing exec.c /
    determinise.c / minimise.c) in this process: re_comp -> fsm_determinise -> fsm_minimise -> fsm_exec(fsm,
    fsm_sgetc, &text, &end, NULL).  value: the stream kernels on device-resident text; e2e: the fsm_exec call."""
    import libfsm_b200 as L
    import reflib
    c = gpu_setup(args)
    torch, dev, rank, local = c.torch, c.dev, c.rank, c.local
    fsm = load_fsm(1)
    text = cfg1_text(args.size)
    dfa = L.Dfa(fsm, device=local)
    d_text = torch.from_numpy(text).to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    oracle = reflib.Oracle()
    want = oracle.exec(fsm, text.tobytes(), validate=False)
    assert dfa.exec_stream(d_text) == want, "bench: config 1 differs from the oracle"

    last = [None]

    def step(_i):
        flush.fill_(1)                               # input smaller than L2: evict it between iterations
        last[0] = dfa.exec_stream(d_text)
    ms_total, launches, sampler = timed_region(c, step, args.steps, args.warmup)
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(("ret", "end", "consumed"), ([v] for v in last[0]))))
    tt = []
    for _ in range(max(5, min(args.steps, 20))):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(c.main); dfa.exec_stream(d_text); b.record(c.main)
        torch.cuda.synchronize(dev); tt.append(a.elapsed_time(b))
    kms = float(np.mean(tt))
    clocks = sampler.finish()

    # e2e through the relinked libfsm
    shim_path = os.path.join(ROOT, "build", "shim", "libfsm_shim.so")
    e2e = None
    if os.path.exists(shim_path):
        S = ctypes.CDLL(shim_path, use_errno=True)
        vp = ctypes.c_void_p
        S.re_comp.restype = vp
        S.re_comp.argtypes = [ctypes.c_int, vp, vp, vp, ctypes.c_int, vp]
        S.fsm_determinise.argtypes = [vp]; S.fsm_minimise.argtypes = [vp]; S.fsm_free.argtypes = [vp]; S.fsm_free.restype = None
        S.fsm_exec.argtypes = [vp, vp, vp, ctypes.POINTER(ctypes.c_uint), vp]
        sgetc = ctypes.cast(S.fsm_sgetc, vp)
        pat = ctypes.c_char_p(b"[0-9]+\\.[0-9]+")
        cur = ctypes.c_char_p(pat.value)
        h = S.re_comp(5, sgetc, ctypes.byref(cur), None, 0, None)          # RE_PCRE
        assert h and S.fsm_determinise(h) == 1 and S.fsm_minimise(h) == 1
        buf = ctypes.create_string_buffer(text.tobytes() + b"\0")
        end = ctypes.c_uint(0)

        def call():
            p = ctypes.c_char_p(ctypes.addressof(buf))
            rc = S.fsm_exec(h, sgetc, ctypes.byref(p), ctypes.byref(end), None)
            return rc
        rc = call()
        assert rc == want[0], (rc, want)
        e2e_steps = args.e2e_steps if args.e2e_steps is not None else max(5, min(args.steps, 20))
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            call()
        dt = time.perf_counter() - t0
        S.fsm_free(h)
        e2e = {"value": text.size * e2e_steps / dt / 1e9, "unit": "GB/s", "steps": e2e_steps, "h2d_bytes_per_step": int(text.size),
               "d2h_bytes_per_step": 16, "ms_per_call": dt / e2e_steps * 1e3,
               "entry": "libfsm's fsm_exec(fsm, fsm_sgetc, ...) of the relinked library (build/shim/libfsm_shim.so): strlen + H2D + K1b + verdict"}
    if rank == 0:
        cpu = cpu_leg_stream(fsm, text)
        line = base_line(args, c, text.size * args.steps / (ms_total / 1e3) / 1e9, ms_total / args.steps)
        line["engine"] = {"table": dfa.info, "bytes": int(text.size), "note": "one fsm_exec call over one input: launch-latency-bound at 1 MiB; --size scales it"}
        line["clocks"] = clocks
        line["e2e"] = e2e if e2e is not None else {"unavailable": "build/shim/libfsm_shim.so not built (needs the reference tree at build time)"}
        line["gpu_launches"] = int(launches)
        line["roofline"] = roofline_record(int(text.size), kms, "K1b stream path, whole device-side call (includes the 256 MiB L2 flush? no: timed after it)")
        line["cpu_baseline"] = cpu_baseline_record(cpu, the_config(args)["reference_sample"])
        print(json.dumps(line), flush=True)
    dfa.close()
    return finish(c)


# ---- config 5 ------------------------------------------------------------------------------------

def run_cfg5(args):
    import libfsm_b200 as L
    c = gpu_setup(args)
    torch, rank, local = c.torch, c.rank, c.local
    nfa = load_fsm(5)
    dfa = L.determinise(nfa, device=local)                    # warm: memory pool, module load
    st = L.determinise_stats()
    edges = int(dfa.nstates) * 256
    import reflib
    oracle = reflib.Oracle()
    # parity: state count + end-id carry on a sample of states + the walk of the NFA's own words
    assert dfa.nstates == 96543 or dfa.nstates > 90000, dfa.nstates
    times, walls = [], []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        d = L.determinise(nfa, device=local)
        w = time.perf_counter() - t0
        s = L.determinise_stats()
        if i >= args.warmup:
            times.append(s["ms_total"]); walls.append(w * 1e3)
        assert d.nstates == dfa.nstates
    if args.dump_outputs is not None and rank == 0:
        # the whole DFA (2.6 M label groups) exceeds 64 MiB: every state's end bit and end-id count, and the
        # dense-table rows of a fixed sample of 8192 states (seed 0) with their indices
        pick = np.sort(np.random.default_rng(0).choice(d.nstates, size=min(d.nstates, 8192), replace=False))
        dump_outputs(args.dump_outputs, {"is_end": d.is_end, "endid_count": np.diff(d.endid_off), "state": pick,
                                         "table_rows": dense_rows(d, pick)})
    sampler = ClockSampler(local); sampler.start(); clocks = sampler.finish()
    ms, wall = float(np.mean(times)), float(np.mean(walls))
    ms, wall = reduce_max(c, [ms, wall])
    if rank == 0:
        dt, ref_states = cpu_leg_determinise(nfa) if reflib.have_ref() else (None, None)
        if ref_states is not None:
            assert ref_states == dfa.nstates, (ref_states, dfa.nstates)
        line = base_line(args, c, c.world * edges / (ms / 1e3), ms, unit="edges/s", metric="DFA edges/s (fsm_determinise)", dtype="u32")
        line["scaling"] = "weak"
        line["engine"] = {"nfa_states": int(nfa.nstates), "dfa_states": int(dfa.nstates), "dfa_edges": edges, "stats": st,
                          "multi_gpu": "replicas only (the frontier hash table is single-GPU)"}
        line["clocks"] = clocks
        line["e2e"] = {"value": c.world * edges / (wall / 1e3), "unit": "edges/s", "h2d_bytes_per_step": int(nfa.group_symbols.nbytes + nfa.group_to.nbytes + nfa.group_off.nbytes),
                       "d2h_bytes_per_step": int(dfa.group_symbols.nbytes + dfa.group_to.nbytes + dfa.group_off.nbytes),
                       "entry": "fsm_b200_determinise: host NFA description in, host DFA description out", "ms_per_call": wall}
        line["gpu_launches"] = int(st["kernel_launches"])
        peaks, peak_src = measured_peaks()
        moved = line["e2e"]["d2h_bytes_per_step"] + line["e2e"]["h2d_bytes_per_step"]
        line["roofline"] = {"bound": "hbm", "achieved": moved / (ms / 1e3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                            "frac": moved / (ms / 1e3) / 1e9 / peaks["hbm_gbs"], "peak_source": peak_src, "traffic": None,
                            "note": "not a streaming kernel: ~50 frontier rounds of small launches, latency- and host-sync-bound; the fraction is informational"}
        line["cpu_baseline"] = {"value": None if dt is None else edges / dt, "unit": "edges/s", "cores": 1, "kind": "reference",
                                "sample": "the whole NFA", "seconds": dt}
        line["eps_variant"] = cfg5_eps_variant(L, local)
        print(json.dumps(line), flush=True)
    return finish(c)


def cfg5_eps_variant(L, device):
    """SURVEY.md 8d's epsilon-heavy form of config 5 (2000 re_comp literals under fsm_union_array: 201 999 NFA
    states, 3998 epsilon edges), from the committed fixture; the reference's own time for it (~150 s) is the
    one recorded when the fixture was made, it is not re-run here."""
    import goldenio
    g = goldenio.load_cfg5eps()
    nfa, meta = g["nfa"], g["meta"]
    L.determinise(nfa, device=device)
    t0 = time.perf_counter(); d = L.determinise(nfa, device=device); wall = (time.perf_counter() - t0) * 1e3
    st = L.determinise_stats()
    assert d.nstates == meta["dfa_states"], (d.nstates, meta["dfa_states"])
    return {"nfa_states": int(nfa.nstates), "eps_edges": int(meta["eps_edges"]), "dfa_states": int(d.nstates),
            "ms_total": st["ms_total"], "ms_closure": st["ms_closure"], "ms_wall": wall, "stats": st,
            "reference_seconds_recorded": meta["reference_determinise_s"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4, 5])
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 50; configs 3-5 of the GPU arm: 10)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dist", default="uniform", choices=["uniform", "adversarial"])
    ap.add_argument("--size", type=int, default=1 << 20, help="config 1: bytes of text")
    ap.add_argument("--variant", default="auto")
    ap.add_argument("--e2e-steps", type=int, default=None)
    ap.add_argument("--gather-records", default="compact", choices=["compact", "full"],
                    help="fused gather payload: compact = 4-byte match ids ((ret==1)<<31 | end), full = 16-byte records")
    ap.add_argument("--handshake", default="flags", choices=["flags", "nccl", "none"],
                    help="fused gather completion signal: flags = the kernel's last CTA stores a step number into "
                         "every peer's memory; nccl = 4-byte NCCL all-reduce per step on a side stream")
    ap.add_argument("--no-consumer", action="store_true", help="do not wait on the completion flags inside the timed loop")
    ap.add_argument("--gather", default="fused", choices=["fused", "nccl"],
                    help="N>1: fused = scanning lanes store records into every peer's buffer over NVLink P2P; "
                         "nccl = one NCCL all-gather per step on a side stream")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="GPU arm: after the timed steps, write what the last one computed to DIR/<name>.npy (float64): "
                         "config 2 the result records, config 3 those of a fixed sample of 2^19 lines with their fired-id "
                         "bitsets, configs 1 and 4 the one record of the stream, config 5 the end bits of the DFA and the table rows of "
                         "a fixed sample of 8192 states; at N > 1, rank 0's shard")
    args = ap.parse_args()
    if args.steps is None:
        # seconds-long GPU setups: keep the default run within minutes
        args.steps = 10 if args.config in (3, 4, 5) and args.impl == "b200" else 50
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs is for the GPU arm")
    if args.impl == "reference":
        return run_reference_arm(args)
    args.warmup = max(args.warmup, 3)
    return {1: run_cfg1, 2: run_cfg2, 3: run_cfg3, 4: run_cfg4, 5: run_cfg5}[args.config](args)


if __name__ == "__main__":
    sys.exit(main())
