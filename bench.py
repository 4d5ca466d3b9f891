#!/usr/bin/env python3
"""bench.py -- BASELINE metric: GiB/s of haystack scanned (config 2: 5000 patterns, 4 GiB, DFA,
MatchKind::Standard overlapping) on N B200s, with roofline / cpu_baseline / e2e objects.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--hay-gib G] [--workload cfg2|cfg3|cfg4|cfg5]
                    [--impl reference] [--dump-outputs DIR]

Every timed loop (the workload's device-resident steps, its end-to-end steps and those of the extra
configs) runs exactly K steps.  --dump-outputs DIR writes the matches the last timed step of the
workload returned to its caller (see dump_outputs) so that two builds can be compared on the same
seeded inputs.

Our arm: every search goes through the C ABI of libacb200.so (ctypes).  N > 1: one process per GPU,
acg_comm_init + acg_find_overlapping_sharded (haystack slices, records stored into rank 0's buffer
over NVLink peer memory; NCCL for the counts / barrier) -- torch.distributed is only the launcher's
rendezvous, barrier and max-over-ranks reduction of the timings.
Reference arm (--impl reference): the reference's CPU loop (src/automaton.rs:1491-1534 over
src/dfa.rs:218-226) as restated in oracle/ (kind "port": no rustc in this image), on the host cores.
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
GIB = float(1 << 30)
DESC = {"cfg2": "5000 random 4-16B printable-ASCII patterns, DFA, MatchKind::Standard, find_overlapping_iter",
        "cfg3": "5000 patterns, ascii_case_insensitive, DFA, MatchKind::LeftmostFirst, find_iter",
        "cfg4": "50 literals (Teddy-active set), MatchKind::LeftmostFirst, find_iter",
        "cfg5": "100000 patterns, DFA, MatchKind::Standard, find_overlapping_iter"}


def load_workload_module():
    """aho-corasick_b200/workload.py loaded by path: the synthetic-input generator has no native
    dependency, and the reference arm must not load the product's shared library."""
    spec = importlib.util.spec_from_file_location("acb_workload", ROOT / "aho-corasick_b200" / "workload.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return json.loads(p.read_text())["hbm_gbs"], "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.samples, self.reasons, self._stop, self.index = [], set(), threading.Event(), index
        self.max_mhz = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for nme, v in zip(names, f[2:6]):
                    if v.lower().startswith("active"):
                        self.reasons.add(nme)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


def usable_cores():
    """Host threads this process can really run at once: the CPU count, cut by the affinity mask
    and by a cgroup CPU quota (a container on a 128-thread host may be limited to far fewer)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = Path(path).read_text().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]) + 0.5)))
            else:
                quota = int(txt[0])
                period = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read_text())
                if quota > 0:
                    n = min(n, max(1, int(quota / period + 0.5)))
            break
        except (OSError, ValueError, IndexError):
            continue
    return max(1, n)


def bind_to_gpu_numa_node(local_rank):
    """Run this rank (and first-touch its pinned buffers) on the CPUs of the GPU's NUMA node: with 8
    ranks on a two-socket host, host buffers on the far socket cut the H2D rate of a rank to a third."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local_rank)],
                             capture_output=True, text=True, timeout=10).stdout.strip()
        bus = out.lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        node = int(Path(f"/sys/bus/pci/devices/{bus}/numa_node").read_text())
        if node < 0:
            return None
        cpus = set()
        for part in Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        return None
    return None


DUMP_BYTES = 64_000_000 - 4096   # 64 MB in all, npy headers included
DUMP_SEED = 0xD0AC


def dump_outputs(out_dir, rec):
    """The match records (pid, start, end in global offsets, in the order the caller receives them)
    as float64 arrays -- exact, offsets stay far below 2^53 -- in out_dir/{pid,start,end}.npy, with
    out_dir/match_count.npy.  A list too large for DUMP_BYTES is cut to a fixed seeded sample of
    records, in order; out_dir/sample_index.npy then holds their positions in the full list."""
    import numpy as np
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    n = len(rec)
    arrays = {"match_count": np.array([n], dtype=np.float64)}
    if n * 3 * 8 > DUMP_BYTES:
        keep = DUMP_BYTES // (4 * 8)
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=keep, replace=False))
        rec = rec[idx]
        arrays["sample_index"] = idx.astype(np.float64)
    for k in ("pid", "start", "end"):
        arrays[k] = rec[k].astype(np.float64)
    for name, a in arrays.items():
        np.save(out_dir / f"{name}.npy", a)


def cpu_scan(o, hay, cores, back):
    """One pass of the oracle's overlapping DFA loop over `hay` on `cores` threads (slices with
    max_pattern_len-1 overlap; the C call releases the GIL).  Returns the match count."""
    from concurrent.futures import ThreadPoolExecutor
    n = hay.size
    if cores == 1:
        return o.scan_overlapping_count(hay)[0]
    bounds = [n * i // cores for i in range(cores + 1)]

    def work(i):
        # ownership by end offset: count in [lo, hi) minus what the overlap re-reports is not needed
        # for a throughput figure; the slices are scanned exactly as a sharded CPU run would scan them
        s = max(0, bounds[i] - back)
        return o.scan_overlapping_count(hay, span=(s, bounds[i + 1]))[0]
    with ThreadPoolExecutor(cores) as ex:
        return sum(ex.map(work, range(cores)))


def reference_arm(args):
    """The reference's own CPU path on the host cores (see the module docstring).  Every step scans
    the same bounded sample of the workload's haystack with all usable threads; the 1-thread figure
    (what the single-threaded reference does) is measured on the same bytes and reported beside it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, str(ROOT / "tests"))
    import numpy as np
    import oracle_py as O
    W = load_workload_module()
    wl = args.workload
    cfg = W.CONFIGS[wl]
    cores = usable_cores()
    sample = min(int(args.hay_gib * GIB), 256 << 20)   # same bytes on every box
    sample -= sample % 8
    pats = W.make_patterns(cfg["n_patterns"], cfg["pattern_seed"], alphabet=cfg["alphabet"])
    hay = np.empty(sample, dtype=np.uint8)
    W.make_config(wl, sample, out=hay)
    o = O.Oracle(pats, kind=O.KIND_DFA)
    back = max(len(p) for p in pats) - 1
    t0 = time.perf_counter()
    n1 = cpu_scan(o, hay, 1, back)
    one_thread = sample / GIB / (time.perf_counter() - t0)
    for _ in range(args.warmup):
        cpu_scan(o, hay, cores, back)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_scan(o, hay, cores, back)
    dt = (time.perf_counter() - t0) / args.steps
    val = sample / GIB / dt
    line = {"impl": "reference", "metric": "haystack_scan_throughput", "value": val, "unit": "GiB/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "same_config": False, "kind": "port",
            "config": {"workload": f"{wl}: {DESC[wl]}; bounded sample of the synthetic haystack",
                       "sample_bytes": sample,
                       "note": "C restatement of src/automaton.rs:1491-1534 over src/dfa.rs:218-226 (no rustc in "
                               "the image); the reference itself is single-threaded -- see one_thread_value"},
            "one_thread_value": one_thread, "matches_in_sample": n1,
            "cpu_baseline": {"value": val, "unit": "GiB/s", "cores": cores, "kind": "port",
                             "one_thread_value": one_thread,
                             "sample": f"first {sample >> 20} MiB of the {wl} haystack, {cores} threads "
                                       f"(slices with max_pattern_len-1 overlap); 1 thread on the same bytes: "
                                       f"{one_thread:.3f} GiB/s"},
            "e2e": {"value": val, "unit": "GiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


class Rig:
    """Process-wide state of our arm: ranks, device, the sharded communicator."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.numa = bind_to_gpu_numa_node(self.local) if self.world > 1 else None
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.comm = None
        if self.world > 1:
            if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
                os.environ["NCCL_DEBUG"] = "WARN"   # keep stdout to the single JSON line
            dist.init_process_group("nccl", device_id=self.dev)
            from aho_corasick_b200 import sharded as S
            uid = torch.zeros(S.COMM_ID_BYTES, dtype=torch.uint8, device=self.dev)
            if self.rank == 0:
                uid.copy_(torch.frombuffer(bytearray(S.unique_id()), dtype=torch.uint8))
            dist.broadcast(uid, 0)
            self.comm = S.Comm(bytes(uid.cpu().numpy().tobytes()), self.rank, self.world)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()

    def sum_over_ranks(self, v):
        t = self.torch.tensor([v], dtype=self.torch.int64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t)
        return int(t.item())


def run_workload(rig, args, wl, steps, warmup, want_e2e=True, check=True, dump_dir=None):
    """Device-resident and end-to-end throughput of one workload on rig.world GPUs; with dump_dir,
    rank 0 writes what the last timed step returned there (dump_outputs)."""
    import numpy as np
    import aho_corasick_b200 as ab
    from aho_corasick_b200 import sharded as S
    from aho_corasick_b200 import workload as W
    torch, world, rank, dev = rig.torch, rig.world, rig.rank, rig.dev
    cfg = W.CONFIGS[wl]
    overlapping = wl in ("cfg2", "cfg5")
    if world > 1 and not overlapping:
        raise SystemExit(f"{wl}: find_iter is not sharded; multi-GPU runs take cfg2 or cfg5")
    per_gpu = int(args.hay_gib * GIB)
    per_gpu -= per_gpu % 4096
    total = per_gpu * world  # weak scaling: the global haystack grows with the number of GPUs
    pats = W.make_patterns(cfg["n_patterns"], cfg["pattern_seed"], alphabet=cfg["alphabet"])
    b = ab.AhoCorasick.builder().kind(ab.AhoCorasickKind.DFA)
    if wl == "cfg3":
        b.ascii_case_insensitive(True).match_kind(ab.MatchKind.LeftmostFirst)
    if wl == "cfg4":
        b.match_kind(ab.MatchKind.LeftmostFirst)
    if args.device_fill or (wl == "cfg5" and not args.host_fill):
        b.device_fill(True)
    t0 = time.perf_counter()
    ac = b.build(pats).set_engine(args.engine)
    build_s = time.perf_counter() - t0
    if args.experiment:
        import ctypes
        ab._lib.acg_debug_set_experiment.argtypes = [ctypes.c_void_p, ctypes.c_uint32]
        assert ab._lib.acg_debug_set_experiment(ac._h, args.experiment) == 0
    # haystack slicing: this rank owns ends in (own_lo, own_hi] and reads from read_lo
    own_lo, own_hi, read_lo = S.slice_plan(0, total, world, ac.max_pattern_len())[rank]
    gen_lo = read_lo - read_lo % 4096
    n_local = own_hi - gen_lo
    n_alloc = n_local + (-n_local) % 8
    d_hay = torch.empty(n_alloc, dtype=torch.uint8, device=dev)
    W.torch_fill_config(wl, d_hay, pats, global_offset=gen_lo)
    torch.cuda.synchronize()
    span = (read_lo - gen_lo, own_hi - gen_lo)
    n_bytes = own_hi - own_lo  # bytes this rank is credited with (overlap re-reads are not)
    state = {"cap": max(1 << 20, n_bytes // 512)}
    state["out"] = torch.empty(state["cap"] * 24, dtype=torch.uint8, device=dev) if world == 1 and overlapping else None

    def step():
        """One pass of the hot path over this rank's slice.  N = 1: ordered matches left on the device
        (overlapping) or returned (find_iter).  N > 1: the sharded call -- scan, then every rank's
        records stored into rank 0's buffer.  Returns (matches, scan+order ms, gather ms)."""
        if world > 1:
            n, _, st, _ = rig.comm.find_overlapping(ac, d_hay.data_ptr(), n_local, gen_lo, (0, total))
            return n, st["scan_ms"] + st["order_ms"], st["gather_ms"], st
        while True:
            try:
                if overlapping:
                    n, ms = ac.find_overlapping_devout(d_hay.data_ptr(), n_local, span, own_lo - gen_lo, gen_lo,
                                                       state["out"].data_ptr(), state["cap"])
                else:
                    r, ms = ac.find_iter_dev_np(d_hay.data_ptr(), n_local, span)
                    n = len(r)
                    state["found"] = r
                return n, ms, 0.0, None
            except OverflowError as e:
                state["cap"] = int(e.args[0]) * 9 // 8 + 1024
                state["out"] = torch.empty(state["cap"] * 24, dtype=torch.uint8, device=dev)

    def stream_of_steps(k_steps):
        """N > 1, a stream of batches: step k + 1 begins before step k is waited for
        (acg_find_overlapping_sharded_begin / _wait), so its scan runs while a copy engine moves step
        k's records into rank 0's buffer.  Timed by CUDA events recorded by the library around the whole
        loop (acg_comm_mark).  Returns (matches, loop ms on this rank's device, per-step stats)."""
        args_b = (ac, d_hay.data_ptr(), n_local, gen_lo, (0, total))
        per_step = []
        rig.comm.mark(0)
        tk = rig.comm.begin(*args_b)
        for _k in range(1, k_steps):
            tk_next = rig.comm.begin(*args_b)
            n, _, sst = rig.comm.wait(tk)
            per_step.append(sst)
            tk = tk_next
        n, _, sst = rig.comm.wait(tk)
        per_step.append(sst)
        rig.comm.mark(1)
        return n, rig.comm.mark_elapsed_ms(), per_step

    # ---- device-resident throughput (inputs already in HBM) ----
    for _ in range(warmup):
        step()
    mode = "blocking"
    calib = None
    if world > 1 and not args.blocking_steps:
        # warm-up doubles as calibration: both forms of the step run `warmup` times untimed, the faster
        # (max over ranks) is the one the timed region uses
        n_cal = max(3, warmup)
        rig.barrier()
        b_ms = 0.0
        for _ in range(n_cal):
            _, ms, gms, _ = step()
            b_ms += ms + gms
        rig.barrier()
        stream_of_steps(2)  # first use allocates the staging buffer and the second workspace
        rig.barrier()
        _, p_ms, _ = stream_of_steps(n_cal)
        b_s, p_s = rig.max_over_ranks(b_ms / 1e3, p_ms / 1e3)
        calib = {"blocking_ms_per_step": b_s * 1e3 / n_cal, "stream_ms_per_step": p_s * 1e3 / n_cal, "steps": n_cal}
        if p_s < b_s:
            mode = "stream"
    rig.barrier()
    kernel_ms, scan_ms, gather_ms = [], [], []
    loop_ms = None
    with ClockSampler(rig.local) as clocks:
        t0 = time.perf_counter()
        if mode == "stream":
            cnt, loop_ms, per_step = stream_of_steps(steps)
            for sst in per_step:
                kernel_ms.append(sst["scan_ms"] + sst["order_ms"])
                scan_ms.append(sst["scan_ms"])
                gather_ms.append(sst["gather_ms"])
        else:
            for _ in range(steps):
                cnt, ms, gms, sst = step()
                st = ac.last_stats()
                kernel_ms.append(ms)
                scan_ms.append(sst["scan_ms"] if sst else st["scan_ms"])
                gather_ms.append(gms)
        rig.barrier()
        wall = time.perf_counter() - t0
    if dump_dir is not None and rank == 0:
        # N > 1: every rank's records in rank 0's buffer; N = 1: the ordered records left on the device
        # (overlapping) or the list returned (find_iter)
        if world > 1:
            last = rig.comm.fetch()
        elif overlapping:
            last = state["out"][: cnt * ab.MATCH_DTYPE.itemsize].cpu().numpy().view(ab.MATCH_DTYPE)
        else:
            last = state["found"]
        dump_outputs(dump_dir, last)
        del last
    stats = ac.last_stats()
    if mode == "stream":
        # one pair of CUDA events around the K overlapped steps, taken inside the library after the
        # device has drained (acg_comm_mark): the whole loop, nothing left out
        dev_s, wall = rig.max_over_ranks(loop_ms / 1e3, wall)
        stats = dict(stats)
        stats["scan_ms"], stats["order_ms"] = per_step[-1]["scan_ms"], per_step[-1]["order_ms"]
        stats["candidates"], stats["launches"] = per_step[-1]["candidates"], per_step[-1]["launches"]
    else:
        # CUDA-event times taken inside the library: scan + order on the search stream, and (N > 1) count
        # exchange + expand into rank 0's buffer + closing barrier on the communicator's stream
        dev_s, wall = rig.max_over_ranks((sum(kernel_ms) + sum(gather_ms)) / 1e3, wall)
    value = total * steps / GIB / dev_s
    total_matches = cnt if world > 1 else rig.sum_over_ranks(cnt)
    transport = rig.comm.transport() if world > 1 else None
    checked = None
    if world > 1 and check:
        # outside the timed region: every rank's segment of rank 0's buffer must be, record for record,
        # the list that rank obtains on its own through the single-GPU entry point, in global offsets
        loc, _ = ac.find_overlapping_iter_dev_np(d_hay.data_ptr(), n_local, span)
        loc = loc[loc["end"].astype(np.int64) > own_lo - gen_lo].copy()
        loc["start"] += gen_lo
        loc["end"] += gen_lo
        gathered = S.gather_to_rank0(loc, rig.dist, device=dev)
        if rank == 0:
            rec = rig.comm.fetch()
            assert len(rec) == total_matches == len(gathered), (len(rec), total_matches, len(gathered))
            for k in ("pid", "start", "end"):
                assert np.array_equal(rec[k], gathered[k]), f"gathered stream differs from the per-rank lists in {k}"
            assert bool(np.all(np.diff(rec["end"].astype(np.int64)) >= 0))
            checked = "record-for-record against each rank's single-GPU list"

    # ---- end to end through the host-buffer C-ABI call (host haystack, H2D + D2H inside) ----
    e2e = None
    if want_e2e and not args.no_e2e:
        e2e_bytes = span[1] - span[0]
        h_hay = torch.empty(e2e_bytes, dtype=torch.uint8, pin_memory=True)
        h_hay.copy_(d_hay[span[0]: span[1]])
        h_np = h_hay.numpy()

        def e2e_step(buf):
            if world > 1:
                n, _, _, out = rig.comm.find_overlapping(ac, buf.ctypes.data, buf.size, read_lo, (0, total),
                                                         on_device=False, host_out=True)
                return n if rank else len(out)
            r = (ac.try_find_overlapping_iter_np if overlapping else ac.try_find_iter_np)(buf)
            return len(r)
        for _ in range(2):
            n_e2e = e2e_step(h_np)
        rig.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            n_e2e = e2e_step(h_np)
        rig.barrier()
        (e2e_s,) = rig.max_over_ranks((time.perf_counter() - t0) / steps)
        e2e = {"value": world * e2e_bytes / GIB / e2e_s, "unit": "GiB/s", "h2d_bytes_per_step": e2e_bytes,
               "d2h_bytes_per_step": int(n_e2e * 24), "host_memory": "pinned",
               "call": "acg_find_overlapping_sharded(host slice)" if world > 1 else
                       ("acg_find_overlapping" if overlapping else "acg_find_iter"),
               "bytes_per_gpu_per_step": e2e_bytes}
        if world == 1 and not args.no_pageable:
            # the same call on ordinary (pageable) host memory: what a caller gets without cudaHostRegister
            p_np = np.empty(e2e_bytes, dtype=np.uint8)
            p_np[:] = h_np
            e2e_step(p_np)
            t0 = time.perf_counter()
            for _ in range(steps):
                e2e_step(p_np)
            e2e["pageable_value"] = e2e_bytes / GIB / ((time.perf_counter() - t0) / steps)
            del p_np
        del h_hay, h_np
    scan_s = sum(scan_ms) / len(scan_ms) / 1e3
    res = {"workload": wl, "value": value, "dev_s": dev_s, "wall": wall, "steps": steps, "matches": total_matches,
           "candidates": int(stats["candidates"]), "scan_ms": sum(scan_ms) / len(scan_ms),
           "order_ms": float(stats["order_ms"]), "gather_ms": sum(gather_ms) / len(gather_ms),
           "gather_ms_samples": [round(g, 4) for g in gather_ms] if world > 1 else None, "build_s": build_s,
           "engine": int(stats["engine"]), "launches": int(stats["launches"]), "achieved": n_bytes / scan_s / 1e9,
           "n_bytes": n_bytes, "per_gpu": per_gpu, "total": total, "e2e": e2e, "clocks": clocks.summary(),
           "table_bytes": ac.memory_usage(), "states": ac.state_len(), "transport": transport, "checked": checked,
           "device_fill": bool(args.device_fill or (wl == "cfg5" and not args.host_fill)),
           "step_mode": mode if world > 1 else "single", "calibration": calib}
    # CPU baseline on rank 0: the oracle's loop on a bounded sample of this rank's haystack
    if not args.no_cpu_baseline and rank == 0 and overlapping:
        sys.path.insert(0, str(ROOT / "tests"))
        import oracle_py as O
        sample = min(64 << 20, span[1] - span[0])
        o = O.Oracle(pats, kind=O.KIND_DFA)
        h = d_hay[span[0]: span[0] + sample].cpu().numpy()
        t0 = time.perf_counter()
        o.scan_overlapping_count(h)
        dt = time.perf_counter() - t0
        res["cpu_baseline"] = {"value": sample / GIB / dt, "unit": "GiB/s", "cores": 1, "kind": "port",
                               "sample": f"first {sample >> 20} MiB of rank 0's haystack, scalar DFA loop "
                                         "(src/automaton.rs:1491-1534 restated in oracle/), 1 thread"}
    del d_hay
    state["out"] = None
    torch.cuda.empty_cache()
    return res


TIMING = {
    "single": "CUDA events inside the library: scan + order on the search stream",
    "blocking": ("CUDA events inside the library: scan + order on the search stream + count exchange, expand into rank "
                 "0's buffer over peer memory and closing barrier on the communicator's stream; max over ranks"),
    "stream": ("one pair of CUDA events recorded by the library around the K overlapped steps (acg_comm_mark: device "
               "drained, event on the communicator's stream, before the first begin and after the last wait); max over "
               "ranks.  scan_ms / order_ms are per-step event times inside that loop; gather_ms is begin-of-exchange to "
               "records-landed of a step and runs beside the next step's scan (not additive)"),
}
SHARDING = {
    "blocking": "acg_find_overlapping_sharded: records stored into rank 0's buffer by the expand kernel",
    "stream": ("acg_find_overlapping_sharded_begin / _wait, two steps in flight: records expanded locally, then one "
               "copy-engine copy into rank 0's buffer while the next step scans"),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--hay-gib", type=float, default=4.0, help="haystack GiB per GPU (weak scaling)")
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--engine", type=int, default=0, help="0 auto, 1 walk, 2 prefilter")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--blocking-steps", action="store_true",
                    help="N > 1: time blocking acg_find_overlapping_sharded steps only (no begin / wait calibration)")
    ap.add_argument("--no-pageable", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the configs sub-object (cfg3/cfg4/cfg5 at N=1, cfg5 at N>1)")
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "cfg5"])
    ap.add_argument("--device-fill", action="store_true",
                    help="build the dense table on the GPU (acg_build_on_device) for every workload; cfg5 does by default")
    ap.add_argument("--host-fill", action="store_true", help="cfg5: build the dense table on the host")
    ap.add_argument("--experiment", type=int, default=0,
                    help="ACG_EXP_* flags (include/acb200_debug.h); 0 = default kernel")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the matches of the workload's last timed step to DIR/*.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must not be negative")
    if args.impl == "reference":
        return reference_arm(args)

    sys.path.insert(0, str(ROOT))
    rig = Rig(args)
    world, rank = rig.world, rig.rank
    wl = args.workload
    main_res = run_workload(rig, args, wl, args.steps, args.warmup, want_e2e=True, dump_dir=args.dump_outputs)
    extras = {}
    if not args.no_extras and not args.experiment and wl == "cfg2":
        # the other BASELINE configs, device-resident, so that the driver-run line carries them:
        # N = 1: cfg3, cfg4, cfg5 (4 GiB each); N > 1: cfg5 (100 000 patterns, N x 4 GiB: config 5 at N = 8)
        for x in (["cfg3", "cfg4", "cfg5"] if world == 1 else ["cfg5"]):
            saved = args.no_cpu_baseline
            args.no_cpu_baseline = True
            r = run_workload(rig, args, x, args.steps, 3, want_e2e=(x == "cfg5" and world > 1), check=True)
            args.no_cpu_baseline = saved
            extras[x] = r
    if rank != 0:
        if world > 1:
            rig.comm.close()
            rig.dist.destroy_process_group()
        return
    peak, which = peaks()
    kname = {1: "walk_overlapping_kernel", 2: "prefilter_kernel", 3: "seq_find_kernel"}

    def roofline(r):
        k = kname[r["engine"]]
        traffic, src = None, None
        tf = ROOT / "profiles" / "dram_traffic.json"
        if tf.exists():
            rec = json.loads(tf.read_text()).get(f"{r['workload']}:{k}")
            if rec:  # `ncu --set full` of this kernel (dram__bytes_read.sum + dram__bytes_write.sum per
                     # haystack byte of one launch), scaled to this launch's bytes; not measured by this run
                traffic, src = rec["dram_bytes_per_haystack_byte"] * r["n_bytes"], rec["source"]
        return {"bound": "hbm", "achieved": r["achieved"], "peak": peak, "unit": "GB/s", "frac": r["achieved"] / peak,
                "traffic": traffic, "traffic_source": src, "peak_source": which, "kernel": k,
                "algorithmic_bytes_per_launch": r["n_bytes"]}
    r = main_res
    line = {
        "metric": "haystack_scan_throughput", "value": r["value"], "unit": "GiB/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["dev_s"] / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic",
        "config": {"workload": f"{wl}: {DESC[wl]}; {r['per_gpu'] / GIB:g} GiB synthetic haystack per GPU, "
                               "~1 planted pattern per 4 KiB",
                   "haystack_bytes_per_gpu": r["per_gpu"], "global_haystack_bytes": r["total"],
                   "l2": "input per launch is far larger than the 126 MB L2",
                   "engine": kname[r["engine"]], "experiment": args.experiment, "device_fill": r["device_fill"],
                   "table_bytes": r["table_bytes"], "states": r["states"],
                   "sharding": (f"haystack slices, max_pattern_len-1 overlap, " + SHARDING[r["step_mode"]] +
                                f" ({r['transport']} transport), NCCL counts + barrier")
                               if world > 1 else "single GPU",
                   "numa_node": rig.numa},
        "matches": r["matches"], "matches_per_s": r["matches"] * args.steps / r["dev_s"],
        "candidates": r["candidates"], "scan_ms": r["scan_ms"], "order_ms": r["order_ms"], "gather_ms": r["gather_ms"],
        "timing": TIMING[r["step_mode"]],
        "step_mode": r["step_mode"], "step_mode_calibration": r["calibration"],
        "gather_ms_samples": r["gather_ms_samples"],
        "build_s": r["build_s"], "wall_ms_per_step": r["wall"] / args.steps * 1e3,
        "roofline": roofline(r),
        "gpu_launches": r["launches"] * args.steps,
        "clocks": r["clocks"],
    }
    if r["checked"]:
        line["gathered_stream_check"] = r["checked"]
    if r["e2e"]:
        line["e2e"] = r["e2e"]
    if "cpu_baseline" in r:
        line["cpu_baseline"] = r["cpu_baseline"]
    if extras:
        line["configs"] = {}
        for x, xr in extras.items():
            line["configs"][x] = {"workload": f"{x}: {DESC[x]}", "value": xr["value"], "unit": "GiB/s",
                                  "global_haystack_bytes": xr["total"], "scan_ms": xr["scan_ms"],
                                  "order_ms": xr["order_ms"], "gather_ms": xr["gather_ms"],
                                  "step_mode": xr["step_mode"], "step_mode_calibration": xr["calibration"],
                                  "ms_per_step": xr["dev_s"] / xr["steps"] * 1e3,
                                  "gather_ms_samples": xr["gather_ms_samples"], "matches": xr["matches"],
                                  "candidates": xr["candidates"], "build_s": xr["build_s"],
                                  "device_fill": xr["device_fill"], "states": xr["states"],
                                  "table_bytes": xr["table_bytes"], "roofline": roofline(xr),
                                  "clocks": xr["clocks"], "gathered_stream_check": xr["checked"]}
            if xr["e2e"]:
                line["configs"][x]["e2e"] = xr["e2e"]
    print(json.dumps(line), flush=True)
    if world > 1:
        rig.comm.close()
        rig.dist.destroy_process_group()


if __name__ == "__main__":
    main()
