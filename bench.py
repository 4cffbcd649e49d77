#!/usr/bin/env python
"""bench.py -- BWTS forward + inverse throughput on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload C1..C5]
    (N > 1: launched by torch.distributed.run, one rank per GPU)

Default workload = the north-star configurations:
    N = 1   C4: ONE 1 GiB synthetic DNA transform on one GPU (the largest single-GPU config);
            the line also carries `multi_block`, the C5 file on this one GPU (base of the scaling run)
    N > 1   C5: the multi-block file of 8 x 256 MiB independent blocks, dealt round-robin over
            the N GPUs (strong scaling: total work fixed).  Every rank transforms its own blocks;
            rank 0 additionally drives all N GPUs from ONE process through the library's own
            dealer, bwts_b200_{forward,inverse}_blocks(devices = 0..N-1)  (`dealer`).

A step = one pass of the hot path over the rank's blocks: forward BWTS, then inverse BWTS of
the result.  `value`: buffers resident in HBM, CUDA events, max over ranks.  `e2e`: the same
through the host-buffer C-ABI calls with pinned host memory, both copies inside the timed
region.  `e2e_cli` (N = 1): wall time of the drop-in tools `bin/mk_bwts in out && bin/unbwts out
back` on /dev/shm files (map_file input, fwrite output, process start and CUDA context included).
The forward output of every block is compared with the SHA-256 of what the unmodified reference
writes for the same input (tests/golden/fullsize.json) before anything is timed.

`--impl reference` times the reference's own CPU tools (oracle/_ref, built from the unmodified
sources; else the oracle port) on a bounded sample of the same workload.

`--dump-outputs DIR` writes what the device-resident path returned in its last timed step, the
forward and the inverse output of every block, as DIR/<workload>_<block>_{forward,inverse}.npy
(float32, 48 MiB in all; a longer block is sampled at fixed, seeded positions).  The inputs come
from a seeded generator, so two builds run with the same arguments can be compared file by file.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO / "tests"))

MB = 1e6
WORKLOADS = {
    # name: (generator kind, seed, bytes, description)                      BASELINE.json configs[i]
    "C1": ("random", 1, 1 << 20, "C1: 1 MiB uniform random bytes"),
    "C2": ("text", 2, 64 << 20, "C2: 64 MiB English-like order-2 Markov text"),
    "C3": ("tiled", 3, 256 << 20, "C3: 256 MiB 64 KiB-tiled text, one substitution per MiB"),
    "C4": ("dna", 4, 1 << 30, "C4: 1 GiB DNA (ACGT) with copied segments, one transform"),
    "C3F": ("fibonacci", 0, 256 << 20, "C3 stress: 256 MiB Fibonacci word"),
    "C6": ("dna", 6, 3 << 29, "C6: 1.5 GiB DNA (ACGT) with copied segments, one transform (above 2^30)"),
    # C5: a multi-block file of 8 x 256 MiB independent blocks (seeds 50..57) dealt over the ranks
    "C5": ("text", 50, 256 << 20, "C5: multi-block file, 8 x 256 MiB order-2 Markov text blocks"),
    # the same shape at an eighth of the size (pipeline diagnostics)
    "C5S": ("text", 50, 32 << 20, "C5 small: multi-block file, 8 x 32 MiB order-2 Markov text blocks"),
}
C5_BLOCKS = 8
MULTI = ("C5", "C5S")
DUMP_BYTES = 48 << 20  # --dump-outputs: all arrays of a run together, as float32
INVERSE_CLASSES = ("inv_tile_hist", "inv_lf_rank", "inv_walk", "inv_jump", "inv_scan", "inv_place")


def block_owner(block, ndev):
    """Round-robin dealing of independent blocks, the same rule as bwts_b200_*_blocks (run_blocks)."""
    return block % ndev


def plan_blocks(workload, rank, world):
    """(generator kind, seed, bytes, golden name) of every block this rank transforms in one step.
    C1..C4: one block per rank (weak scaling).  C5: 8 fixed blocks dealt round-robin (strong)."""
    kind, seed, n, _ = WORKLOADS[workload]
    if workload in MULTI:
        return [(kind, seed + b, n, f"{workload}_{b}") for b in range(C5_BLOCKS) if block_owner(b, world) == rank]
    return [(kind, seed + 100 * rank, n, workload if rank == 0 else None)]


def total_blocks(workload, world):
    return C5_BLOCKS if workload in MULTI else world


def default_workload(world):
    return "C4" if world == 1 else "C5"


_JSON_OUT = None


def claim_stdout():
    """Keep the real stdout for the one JSON line; whatever libraries print to fd 1 (NCCL's
    version banner, for one) goes to stderr instead."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
        sys.stdout = sys.stderr


def emit_json(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


def load_product():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bwts_b200", REPO / "bijective-bwt_b200" / "bwts_b200.py")
    mod = importlib.util.module_from_spec(spec)
    sys.modules["bwts_b200"] = mod
    spec.loader.exec_module(mod)
    return mod


def make_input(kind, seed, n):
    import helpers
    return helpers.Generator().make(kind, seed, n)


def make_inputs(plan):
    """generate the blocks side by side (the generator releases the GIL inside ctypes)"""
    if len(plan) == 1:
        return [make_input(*plan[0][:3])]
    with ThreadPoolExecutor(min(len(plan), os.cpu_count() or 1)) as ex:
        return list(ex.map(lambda p: make_input(*p[:3]), plan))


def golden_table():
    p = REPO / "tests" / "golden" / "fullsize.json"
    try:
        return json.loads(p.read_text())
    except Exception:
        return {}


def sha256_tensor(t):
    """SHA-256 of a uint8 torch tensor (host or device), 64 MiB at a time"""
    h = hashlib.sha256()
    step = 64 << 20
    for o in range(0, t.numel(), step):
        h.update(t[o:o + step].cpu().numpy().tobytes())
    return h.hexdigest()


def measured_peak():
    p = REPO / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons, sampled every 50 ms from before the warm-up on;
    stop() keeps the samples whose timestamps fall inside the timed regions."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.t0 = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def mark(self):
        """the timed region starts now"""
        self.t0 = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t1 = time.time()
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def digest(rows):
            sm, mx, reasons = [], [], set()
            for _, r in rows:
                try:
                    sm.append(float(r[1])); mx.append(float(r[2]))
                except Exception:
                    continue
                for name, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            sm.sort()
            return sm, mx, reasons

        inside = [x for x in self.rows if self.t0 is not None and self.t0 - 0.05 <= x[0] <= t1 + 0.1]
        sm, mx, reasons = digest(inside)
        window = "timed regions"
        if not sm:  # region shorter than the sampling period: report what was seen around it
            sm, mx, reasons = digest(self.rows)
            window = "whole run (timed region shorter than the sampling period)"
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "window": window, "reasons": sorted(reasons)}


# --------------------------------------------------------------------------- CPU arms

def ref_kind():
    import helpers
    return "reference" if helpers.ref_available() else "port"


def cpu_round_trip(data, kind):
    """forward + inverse of `data` on one host core; returns seconds (fwd, inv) and checks the round trip."""
    import helpers
    if kind == "reference":
        d = "/dev/shm" if os.path.isdir("/dev/shm") else None
        with tempfile.TemporaryDirectory(dir=d) as td:
            src, mid, back = Path(td) / "in", Path(td) / "mid", Path(td) / "back"
            src.write_bytes(data)
            t0 = time.perf_counter()
            subprocess.check_call([str(helpers.REF_DIR / "mk_bwts"), str(src), str(mid)])
            t1 = time.perf_counter()
            subprocess.check_call([str(helpers.REF_DIR / "unbwts"), str(mid), str(back)])
            t2 = time.perf_counter()
            assert back.read_bytes() == data, "reference round trip failed"
            fwd = mid.read_bytes()
    else:
        o = helpers.Oracle()
        t0 = time.perf_counter()
        fwd = o.forward(data)
        t1 = time.perf_counter()
        back = o.inverse(fwd)
        t2 = time.perf_counter()
        assert back == data, "oracle round trip failed"
    return t1 - t0, t2 - t1, fwd


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    kind_name, seed, n, desc = WORKLOADS[args.workload]
    kind = ref_kind()
    total = max(1, args.steps + args.warmup)
    # the reference tools run ~2.5 MB/s round trip on one core (one transform = one thread, the
    # reference has no parallelism); keep the whole `--steps K --warmup W` run near two minutes
    budget = int(2.5e6 * 110 / total)
    sample = 1 << 20
    while sample * 2 <= min(n, budget):
        sample *= 2
    if n <= budget:
        sample = n  # the whole block fits the arm's time budget: same bytes as the GPU arm
    nproc = os.cpu_count() or 1
    # the same blocks the GPU arm transforms in one step, run side by side on the host cores
    all_blocks = [blk for r in range(world) for blk in plan_blocks(args.workload, r, world)]
    datas = [d[:sample] for d in make_inputs(all_blocks)]
    blocks = len(datas)
    conc = min(blocks, nproc)

    def one_step():
        t0 = time.perf_counter()
        if conc == 1:
            for d in datas:
                cpu_round_trip(d, kind)
        else:
            with ThreadPoolExecutor(conc) as ex:
                list(ex.map(lambda d: cpu_round_trip(d, kind), datas))
        return time.perf_counter() - t0

    for _ in range(args.warmup):
        one_step()
    times = [one_step() for _ in range(args.steps)]
    sec = sum(times) / len(times)
    value = blocks * sample / MB / sec
    who = ("unmodified reference mk_bwts+unbwts (oracle/_ref; suffix sort = substitute SA-IS, not libdivsufsort)"
           if kind == "reference" else "oracle port")
    if sample == n:
        sample_desc = f"all {blocks} block(s) of {desc} at full size; {who}; {conc} process(es) at a time, 1 thread each"
        why = "full blocks: same bytes as the GPU arm"
    else:
        sample_desc = (f"first {sample >> 20} MiB of each of {blocks} block(s) of {desc}; {who}; "
                       f"{conc} process(es) at a time, 1 thread each")
        why = (f"a full {n >> 20} MiB block takes the single-threaded reference ~{n / 2.5e6:.0f} s per round trip; "
               f"{total} steps of it do not fit the arm's few-minute budget, so every step runs the first "
               f"{sample >> 20} MiB of each block (the reference's MB/s falls slowly with size, so this favours it)")
    line = {
        "impl": "reference", "metric": "bwts_round_trip_throughput", "value": value, "unit": "MB/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "strong" if args.workload in MULTI else "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": desc + ", forward + inverse round trip", "bytes_per_gpu": n * blocks // world,
                   "blocks": blocks, "sample_bytes": sample, "same_bytes_as_gpu_arm": sample == n, "sample_reason": why},
        "cpu_baseline": {"value": value, "unit": "MB/s", "cores": conc, "kind": kind, "sample": sample_desc},
        "e2e": {"value": value, "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit_json(line)


# --------------------------------------------------------------------------- GPU arm

def pin_to_gpu_numa_node(torch, local_rank):
    """Best effort: run this rank's host threads (and so its pinned allocations, first touch) on the
    NUMA node the GPU hangs off.  Returns what was found for the JSON line."""
    info = {"node": None, "cpus": None, "pinned": False}
    try:
        props = torch.cuda.get_device_properties(local_rank)
        bus = f"{props.pci_domain_id:04x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        node = int(Path(f"/sys/bus/pci/devices/{bus}/numa_node").read_text().strip())
        info["node"] = node
        if node < 0:
            return info
        cpulist = Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip()
        cpus = set()
        for part in cpulist.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        info["cpus"] = len(cpus)
        if cpus and cpus != os.sched_getaffinity(0):
            os.sched_setaffinity(0, cpus)
            info["pinned"] = True
    except Exception as e:  # containers often hide the topology
        info["error"] = type(e).__name__
    return info


class Blocks:
    """the blocks one rank owns: host (pinned) and device buffers, golden names"""

    def __init__(self, torch, dev, plan, pin=True):
        self.items = []
        datas = make_inputs(plan)
        for (k_, s_, n_, gname), data in zip(plan, datas):
            host_in = torch.frombuffer(bytearray(data), dtype=torch.uint8)
            if pin:
                host_in = host_in.pin_memory()
            self.items.append({
                "host_in": host_in, "n": n_, "golden": gname,
                "host_mid": torch.empty(n_, dtype=torch.uint8, pin_memory=pin),
                "host_back": torch.empty(n_, dtype=torch.uint8, pin_memory=pin),
                "d_in": host_in.to(dev), "d_mid": torch.empty(n_, dtype=torch.uint8, device=dev),
                "d_back": torch.empty(n_, dtype=torch.uint8, device=dev)})
        self.bytes = sum(b["n"] for b in self.items)


def absorb(st, acc):
    for name, c in st["classes"].items():
        a = acc.setdefault(name, {"launches": 0, "ms": 0.0, "bytes": 0.0})
        a["launches"] += c["launches"]; a["ms"] += c["ms"]; a["bytes"] += c["bytes"]


def device_resident(torch, ctx, blocks, stream, flush, steps, warmup, golden, agg=None, before_timed=None):
    """W warm-up + K timed forward+inverse passes over `blocks`, buffers in HBM.  Returns
    (total_ms over the K steps, fwd_ms/step, inv_ms/step, launches, last forward stats, last inverse
    stats, names of the golden hashes that were checked)."""
    sh = stream.cuda_stream
    dev = flush.device

    def step(acc=None):
        out = []
        for b in blocks.items:
            flush.zero_()
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e2 = torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            ctx.forward_device(b["d_in"].data_ptr(), b["n"], b["d_mid"].data_ptr(), sh)
            sf = ctx.stats()
            e1.record(stream)
            ctx.inverse_device(b["d_mid"].data_ptr(), b["n"], b["d_back"].data_ptr(), sh)
            si = ctx.stats()
            e2.record(stream)
            if acc is not None:
                absorb(sf, acc[0]); absorb(si, acc[1])
            out.append((e0, e1, e2, sf, si))
        return out

    def check_round_trip():
        for b in blocks.items:
            assert torch.equal(b["d_back"], b["d_in"]), "round trip lost data"

    checked = []
    for w in range(max(warmup, 1)):
        step()
        torch.cuda.synchronize(dev)
        if w == 0:  # correctness gate of the bench itself: round trip + the reference's own output hash
            check_round_trip()
            for b in blocks.items:
                g = golden.get(b["golden"]) if b["golden"] else None
                if g and g["n"] == b["n"]:
                    got = sha256_tensor(b["d_mid"])
                    assert got == g["fwd_sha256"], f"forward output of {b['golden']} differs from the reference's ({got})"
                    checked.append(b["golden"])
    if before_timed:
        before_timed()  # barrier + synchronize, clock sampler mark
    t_begin = torch.cuda.Event(enable_timing=True); t_end = torch.cuda.Event(enable_timing=True)
    t_begin.record(stream)
    evs, launches, last_f, last_i = [], 0, None, None
    for _ in range(steps):
        for e0, e1, e2, sf, si in step(agg):
            launches += sf["launches"] + si["launches"]
            evs.append((e0, e1, e2))
            last_f, last_i = sf, si
    t_end.record(stream)
    torch.cuda.synchronize(dev)
    total_ms = t_begin.elapsed_time(t_end)
    fwd_ms = sum(a.elapsed_time(b) for a, b, _ in evs) / steps
    inv_ms = sum(b.elapsed_time(c) for _, b, c in evs) / steps
    check_round_trip()
    return total_ms, fwd_ms, inv_ms, launches, last_f, last_i, checked


def dump_outputs(torch, blocks, names, out_dir, per_array):
    """--dump-outputs: d_mid (forward output) and d_back (inverse output) of every block as float32 .npy files.
    A block longer than `per_array` bytes is sampled: one byte out of every n // per_array, at an offset inside
    that stretch drawn from a fixed seed, so that every run of the same arguments reads the same positions."""
    import numpy as np
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for b, name in zip(blocks.items, names):
        n, idx = b["n"], None
        if n > per_array:
            stride = n // per_array
            pos = np.arange(per_array, dtype=np.int64) * stride + np.random.default_rng(0).integers(0, stride, per_array)
            idx = torch.from_numpy(pos).to(b["d_mid"].device)
        for what, t in (("forward", b["d_mid"]), ("inverse", b["d_back"])):
            np.save(out / f"{name}_{what}.npy", (t if idx is None else t[idx]).float().cpu().numpy())
    log(f"wrote {2 * len(names)} output array(s) to {out}")


def host_buffers(torch, ctx, blocks, steps, warmup):
    """the host-buffer C-ABI calls on pinned memory, one block at a time; returns (wall ms, device ms) per step"""
    copies = {"h2d_ms": 0.0, "d2h_ms": 0.0, "bytes": 0}

    def step(count=False):
        t0 = time.perf_counter()
        dev_ms = 0.0
        for b in blocks.items:
            ctx.forward_host_ptr(b["host_in"].data_ptr(), b["n"], b["host_mid"].data_ptr())
            sf = ctx.stats()
            ctx.inverse_host_ptr(b["host_mid"].data_ptr(), b["n"], b["host_back"].data_ptr())
            si = ctx.stats()
            dev_ms += sum(s["h2d_ms"] + s["total_ms"] + s["d2h_ms"] for s in (sf, si))
            if count:
                copies["h2d_ms"] += sf["h2d_ms"] + si["h2d_ms"]; copies["d2h_ms"] += sf["d2h_ms"] + si["d2h_ms"]
                copies["bytes"] += 2 * b["n"]
        return (time.perf_counter() - t0) * 1e3, dev_ms

    for _ in range(warmup):
        step()
    res = [step(True) for _ in range(steps)]
    for b in blocks.items:
        assert torch.equal(b["host_back"], b["host_in"]), "e2e round trip lost data"
    h2d_gbs = copies["bytes"] / (copies["h2d_ms"] * 1e-3) / 1e9 if copies["h2d_ms"] > 0 else 0.0
    d2h_gbs = copies["bytes"] / (copies["d2h_ms"] * 1e-3) / 1e9 if copies["d2h_ms"] > 0 else 0.0
    return sum(w for w, _ in res) / steps, sum(d for _, d in res) / steps, h2d_gbs, d2h_gbs


def blocks_call(torch, bwts, items, devices, steps, warmup, golden, pinned=True):
    """bwts_b200_forward_blocks + bwts_b200_inverse_blocks on the concatenation of `items` (equal
    sizes), host clock around both calls; per-block golden hashes checked on the forward output."""
    nb_, bl = len(items), items[0]["n"]
    cat_in = torch.cat([b["host_in"] for b in items])
    cat_mid = torch.empty_like(cat_in)
    cat_back = torch.empty_like(cat_in)
    if pinned:
        cat_in, cat_mid, cat_back = cat_in.pin_memory(), cat_mid.pin_memory(), cat_back.pin_memory()

    def step():
        t0 = time.perf_counter()
        bwts.blocks_ptr(0, cat_in.data_ptr(), nb_ * bl, bl, cat_mid.data_ptr(), devices=devices)
        t1 = time.perf_counter()
        bwts.blocks_ptr(1, cat_mid.data_ptr(), nb_ * bl, bl, cat_back.data_ptr(), devices=devices)
        return (time.perf_counter() - t0) * 1e3, (t1 - t0) * 1e3

    for _ in range(warmup):
        step()
    res = [step() for _ in range(steps)]
    assert torch.equal(cat_back, cat_in), "blocks call: round trip lost data"
    checked = []
    for i, b in enumerate(items):
        g = golden.get(b["golden"]) if b["golden"] else None
        if g and g["n"] == bl:
            got = sha256_tensor(cat_mid[i * bl:(i + 1) * bl])
            assert got == g["fwd_sha256"], f"blocks call: forward output of {b['golden']} differs from the reference's"
            checked.append(b["golden"])
    return sum(w for w, _ in res) / steps, sum(f for _, f in res) / steps, checked


def cli_round_trip(data, n, steps):
    """wall seconds of `bin/mk_bwts in out` and `bin/unbwts out back` on /dev/shm files: the best of `steps`
    timed round trips after one untimed one"""
    bindir = REPO / "bijective-bwt_b200" / "bin"
    d = "/dev/shm" if os.path.isdir("/dev/shm") else None
    with tempfile.TemporaryDirectory(dir=d) as td:
        src, mid, back = Path(td) / "in", Path(td) / "mid", Path(td) / "back"
        src.write_bytes(data)
        env = dict(os.environ)
        best = None
        for i in range(1 + steps):  # the untimed first run pages the binaries and the CUDA libraries in
            t0 = time.perf_counter()
            subprocess.check_call([str(bindir / "mk_bwts"), str(src), str(mid)], env=env)
            t1 = time.perf_counter()
            subprocess.check_call([str(bindir / "unbwts"), str(mid), str(back)], env=env)
            t2 = time.perf_counter()
            if i > 0 and (best is None or t2 - t0 < best[0] + best[1]):
                best = (t1 - t0, t2 - t1)
        ok = back.read_bytes() == data
        fwd_sha = hashlib.sha256(mid.read_bytes()).hexdigest()
    assert ok, "CLI round trip lost data"
    return best[0], best[1], fwd_sha


def roofline_block(agg_f, agg_i, total_ms, peak, peak_src, workload):
    """dominant class = the one with the largest summed time; fractions per direction"""
    allc = {}
    for acc in (agg_f, agg_i):
        for k, v in acc.items():
            a = allc.setdefault(k, {"launches": 0, "ms": 0.0, "bytes": 0.0})
            a["launches"] += v["launches"]; a["ms"] += v["ms"]; a["bytes"] += v["bytes"]
    if not allc:
        return None
    name, dom = max(allc.items(), key=lambda kv: kv[1]["ms"])
    achieved = dom["bytes"] / (dom["ms"] * 1e-3) / 1e9 if dom["ms"] > 0 else 0.0

    def frac(acc):
        ms = sum(v["ms"] for v in acc.values())
        by = sum(v["bytes"] for v in acc.values())
        return (by / (ms * 1e-3) / 1e9 / peak) if ms > 0 and peak else None

    traffic = None
    tp = REPO / "profiles" / "r02_traffic.json"
    if tp.exists():
        try:
            traffic = json.loads(tp.read_text()).get(workload, {}).get(name, {}).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    return {"bound": "hbm", "kernel": name, "how": "class with the largest summed CUDA-event time over the timed steps",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
            "traffic": traffic, "peak_source": peak_src, "launches": dom["launches"],
            "algorithmic_bytes_per_launch": dom["bytes"] / dom["launches"] if dom["launches"] else 0,
            "avg_launch_ms": dom["ms"] / dom["launches"] if dom["launches"] else 0,
            "share_of_step": dom["ms"] / total_ms if total_ms else None,
            "forward_frac": frac(agg_f), "inverse_frac": frac(agg_i),
            "round_trip_frac": frac(allc),
            "frac_note": "forward/inverse/round_trip_frac = sum of the classes' algorithmic bytes / sum of their "
                         "event times / peak (DESIGN.md section 4 states the per-element byte counts)"}


def run_gpu_arm(args, rank, local_rank, world):
    import torch
    bwts = load_product()
    if bwts.device_count() < 1:
        raise RuntimeError("bench.py: no CUDA device; the product has no CPU path")
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        # host-side group: ranks that sit out a leg wait on the CPU -- an NCCL barrier would park a spinning
        # kernel on their GPU while rank 0's dealer (another process) wants to run kernels on that same GPU
        host_group = dist.new_group(backend="gloo")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    numa = pin_to_gpu_numa_node(torch, local_rank)
    kind_name, seed, n, desc = WORKLOADS[args.workload]
    plan = plan_blocks(args.workload, rank, world)
    golden = golden_table()
    if args.bytes:
        n = args.bytes
        plan = [(k_, s_, n, None) for k_, s_, _, _ in plan]
    for kv in args.tune:
        k, v = kv.split(":")
        bwts.tune(int(k), int(v))
    ctx = bwts.Context(local_rank)
    ctx.reserve(n)
    t_setup = time.time()
    blocks = Blocks(torch, dev, plan)
    my_bytes = blocks.bytes
    log(f"rank {rank}: {len(blocks.items)} block(s), {my_bytes >> 20} MiB generated in {time.time() - t_setup:.1f} s")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    stream = torch.cuda.current_stream(dev)

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def host_barrier():
        torch.cuda.synchronize(dev)
        if dist:
            dist.barrier(group=host_group)

    sampler = ClockSampler(local_rank)
    sampler.start()
    agg_f, agg_i = {}, {}

    def before_timed():
        barrier()
        sampler.mark()

    # ---- W warm-up steps (with the parity gate), barrier, exactly K timed steps, barrier
    total_ms, fwd_ms, inv_ms, launches, last_f, last_i, checked = device_resident(
        torch, ctx, blocks, stream, flush, args.steps, args.warmup, golden, (agg_f, agg_i), before_timed)
    barrier()
    log(f"rank {rank}: device-resident {total_ms / args.steps:.2f} ms/step (fwd {fwd_ms:.2f}, inv {inv_ms:.2f}); golden checked: {checked}")

    # ---- end to end: the host-buffer C-ABI call, pinned host memory, both copies inside
    barrier()
    e2e_wall_ms, e2e_dev_ms, h2d_gbs, d2h_gbs = host_buffers(torch, ctx, blocks, args.steps, min(args.warmup, 2))

    # ---- several blocks per GPU: the block pipeline (bwts_b200_*_blocks: H2D of block b+1 |
    # transform of block b | D2H of block b-1), whole call timed on the host clock
    pipe_ms = None
    if len(blocks.items) > 1 and len({b["n"] for b in blocks.items}) == 1:
        barrier()
        pipe_ms, _, _ = blocks_call(torch, bwts, blocks.items, [local_rank], args.steps, min(args.warmup, 1), golden)
    clocks = sampler.stop()  # sampled across the timed regions (device-resident and end-to-end)
    if args.dump_outputs:  # d_mid / d_back still hold the last device-resident step
        names = [f"{args.workload}_{s_ - seed if args.workload in MULTI else rank}" for _, s_, _, _ in plan]
        per_array = DUMP_BYTES // 4 // (2 * total_blocks(args.workload, world))
        dump_outputs(torch, blocks, names, args.dump_outputs, per_array)
    barrier()

    # ---- max over ranks (times), sum over ranks (bytes)
    t = torch.tensor([total_ms, fwd_ms, inv_ms, e2e_wall_ms, e2e_dev_ms, pipe_ms or 0.0], dtype=torch.float64, device=dev)
    nb = torch.tensor([float(my_bytes), float(len(checked))], dtype=torch.float64, device=dev)
    # slowest rank's copy rates (min over ranks): the host side of the PCIe copies is what limits e2e scaling
    cp = torch.tensor([-h2d_gbs, -d2h_gbs], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(nb, op=dist.ReduceOp.SUM)
        dist.all_reduce(cp, op=dist.ReduceOp.MAX)
    h2d_min, d2h_min = (-x for x in cp.tolist())
    total_ms, fwd_ms, inv_ms, e2e_wall_ms, e2e_dev_ms, pipe_ms_max = t.tolist()
    job_bytes, golden_checked = nb.tolist()
    ms_per_step = total_ms / args.steps

    # ---- N > 1, multi-block file: rank 0 drives ALL N GPUs from one process through the library's
    # own dealer (run_blocks: one host thread + pipeline per device); the other ranks wait
    dealer = None
    if world > 1 and args.workload in MULTI and not args.no_dealer:
        host_barrier()  # every GPU is idle from here on; the other ranks wait in gloo, not on their GPU
        if rank == 0:
            allplan = [blk for r in range(world) for blk in plan_blocks(args.workload, r, world)]
            allplan.sort(key=lambda p: p[1])  # file order = block order = seed order
            items = [{"host_in": torch.frombuffer(bytearray(d), dtype=torch.uint8), "n": p[2], "golden": p[3]}
                     for p, d in zip(allplan, make_inputs(allplan))]
            d_ms, d_fwd_ms, d_checked = blocks_call(torch, bwts, items, list(range(world)), args.steps, 1, golden)
            fb = sum(b["n"] for b in items)
            dealer = {"value": fb / MB / (d_ms * 1e-3), "unit": "MB/s", "devices": world, "ms": d_ms, "forward_ms": d_fwd_ms,
                      "bytes": fb, "golden_checked": d_checked,
                      "how": "ONE process: bwts_b200_forward_blocks + bwts_b200_inverse_blocks(devices=0..N-1) on the whole "
                             "multi-block file in pinned host memory, host clock around both calls; per-block SHA-256 of "
                             "the forward output compared with the unmodified reference's"}
            del items
        host_barrier()

    if rank == 0:
        peak, peak_src = measured_peak()
        line = {
            "metric": "bwts_round_trip_throughput", "value": job_bytes / MB / (ms_per_step * 1e-3), "unit": "MB/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong" if args.workload in MULTI else "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": desc + ", forward + inverse round trip", "bytes_per_gpu": my_bytes,
                       "blocks": total_blocks(args.workload, world), "l2": "flushed between steps (256 MiB device memset inside the timed loop)",
                       "generator": f"bijective-bwt_b200/host/gen_input.c kind={kind_name} seed={seed}"
                                    + ("+block" if args.workload in MULTI else "+100*rank"),
                       "parallelism": f"independent blocks over {world} GPU(s), round-robin, no collective",
                       "parity": f"{int(golden_checked)} block(s): SHA-256 of the forward output == the unmodified reference's "
                                 "(tests/golden/fullsize.json), and inverse(forward(x)) == x, before the timed steps"},
            "forward_mbs": job_bytes / MB / (fwd_ms * 1e-3), "inverse_mbs": job_bytes / MB / (inv_ms * 1e-3),
            "forward_ms": fwd_ms, "inverse_ms": inv_ms,
            "e2e": {"value": job_bytes / MB / (e2e_dev_ms * 1e-3), "unit": "MB/s",
                    "h2d_bytes_per_step": 2 * my_bytes, "d2h_bytes_per_step": 2 * my_bytes,
                    "wall_value": job_bytes / MB / (e2e_wall_ms * 1e-3),
                    "h2d_gbs_slowest_rank": h2d_min, "d2h_gbs_slowest_rank": d2h_min, "numa_rank0": numa,
                    "how": "bwts_b200_forward_host + bwts_b200_inverse_host on pinned host buffers; CUDA events "
                           "from before the H2D copy to after the D2H copy (wall_value: host clock)"},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": roofline_block(agg_f, agg_i, total_ms, peak, peak_src, args.workload),
            "kernel_classes": {},
            "transform": {"factors": last_f["factors"], "longest_factor": last_f["longest_factor"],
                          "alphabet_bits": last_f["alphabet_bits"], "initial_depth": last_f["initial_depth"],
                          "doubling_rounds": last_f["rounds"], "radix_passes": last_f["radix_passes"],
                          "local_sort_rounds": last_f["local_rounds"], "cta_sort_rounds": last_f["cta_rounds"],
                          "live_sum": last_f["live_sum"], "cycles": last_i["factors"],
                          "splitters": last_i["splitters"], "unreached": last_i["unreached"],
                          "arena_bytes_per_input_byte": last_f.get("arena_bytes_per_byte")},
        }
        for direction, acc in (("forward", agg_f), ("inverse", agg_i)):
            for k, v in sorted(acc.items(), key=lambda kv: -kv[1]["ms"]):
                line["kernel_classes"][k] = {"direction": direction, "launches": v["launches"] // max(args.steps, 1),
                                             "ms_per_step": v["ms"] / args.steps,
                                             "gbs": (v["bytes"] / (v["ms"] * 1e-3) / 1e9) if v["ms"] > 0 else None}
        if pipe_ms is not None:
            # the headline end-to-end number of a multi-block workload is the pipelined call
            line["e2e"]["one_block_at_a_time_value"] = line["e2e"]["value"]
            line["e2e"]["value"] = job_bytes / MB / (pipe_ms_max * 1e-3)
            line["e2e"]["wall_value"] = line["e2e"]["value"]
            line["e2e"]["how"] = ("bwts_b200_forward_blocks + bwts_b200_inverse_blocks over all blocks of the rank, "
                                  "pinned host buffers, per-device pipeline H2D | transform | D2H; host clock around "
                                  "both calls (one_block_at_a_time_value: the per-block host-buffer calls, CUDA events)")
        if dealer:
            line["dealer"] = dealer
        if world == 1 and not args.no_cli and (REPO / "bijective-bwt_b200" / "bin" / "mk_bwts").exists():
            ctx.close()  # the tools are separate processes with their own workspace: give the HBM back first
            b0 = blocks.items[0]
            data0 = b0["host_in"].numpy().tobytes()
            tf, ti, fwd_sha = cli_round_trip(data0, b0["n"], args.steps)
            g = golden.get(b0["golden"]) if b0["golden"] else None
            if g and g["n"] == b0["n"]:
                assert fwd_sha == g["fwd_sha256"], "CLI forward output differs from the reference's"
            line["e2e_cli"] = {"value": b0["n"] / MB / (tf + ti), "unit": "MB/s", "forward_s": tf, "inverse_s": ti,
                               "how": "wall clock of `bin/mk_bwts in mid` + `bin/unbwts mid back` on /dev/shm files: process "
                                      "start, CUDA context, workspace allocation, map_file input, transform, fwrite output "
                                      f"(map_file.c:16-46 -> mk_bwts_sa.c:60, unbwts.c:173); best of {args.steps} runs "
                                      "after one untimed run"}
            del data0
        if world == 1 and not args.no_cpu:
            kind = ref_kind()
            b0 = blocks.items[0]
            sample = min(b0["n"], args.cpu_sample)
            data0 = b0["host_in"][:sample].numpy().tobytes()
            tf, ti, fwd = cpu_round_trip(data0, kind)
            # a full-size sample doubles as a parity check of the timed workload
            if sample == b0["n"]:
                assert bytes(b0["d_mid"].cpu().numpy()) == fwd, "GPU forward differs from the CPU baseline output"
            line["cpu_baseline"] = {
                "value": sample / MB / (tf + ti), "unit": "MB/s", "cores": 1, "kind": kind,
                "forward_mbs": sample / MB / tf, "inverse_mbs": sample / MB / ti,
                "sample": f"first {sample} bytes of the same block, forward + inverse, "
                          + ("unmodified reference mk_bwts + unbwts from oracle/_ref (suffix sort = substitute SA-IS, "
                             "not libdivsufsort), 1 thread (the reference has no parallelism)" if kind == "reference"
                             else "oracle port, 1 thread"),
                "host_cpus": os.cpu_count()}
            del data0
    # ---- N = 1 default run: the multi-block file on this one GPU (base of the 1/2/4/8 scaling run)
    if world == 1 and args.multi_block and args.workload not in MULTI:
        b0 = None
        del blocks
        torch.cuda.empty_cache()
        ctx.close()
        ctx = bwts.Context(local_rank)
        mplan = plan_blocks("C5", 0, 1)
        mb = Blocks(torch, dev, mplan)
        ms_total, mf, mi, _, _, _, mchecked = device_resident(torch, ctx, mb, stream, flush, args.steps, 1, golden)
        p_ms, _, pchecked = blocks_call(torch, bwts, mb.items, [local_rank], args.steps, 1, golden)
        line["multi_block"] = {
            "workload": WORKLOADS["C5"][3] + ", all 8 blocks on this one GPU",
            "value": mb.bytes / MB / (ms_total / args.steps * 1e-3), "unit": "MB/s", "forward_ms": mf, "inverse_ms": mi,
            "e2e_value": mb.bytes / MB / (p_ms * 1e-3), "golden_checked": sorted(set(mchecked) | set(pchecked)),
            "how": f"value: device-resident, CUDA events, 1 warm-up + {args.steps} steps; e2e_value: bwts_b200_*_blocks "
                   "pipeline on pinned host buffers, host clock"}
    if rank == 0:
        emit_json(line)
    ctx.close()
    if dist:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS),
                    help="default: C4 (1 GiB, one transform) on 1 GPU, C5 (8 x 256 MiB blocks) on N > 1")
    ap.add_argument("--bytes", type=int, default=0, help="override the block size (diagnostics only)")
    ap.add_argument("--cpu-sample", type=int, default=32 << 20, help="bytes of the block the CPU baseline runs")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-cli", action="store_true", help="skip the e2e_cli leg")
    ap.add_argument("--no-dealer", action="store_true", help="skip rank 0's in-process multi-GPU dealer leg")
    ap.add_argument("--no-multi-block", dest="multi_block", action="store_false",
                    help="N = 1: skip the C5-on-one-GPU leg")
    ap.add_argument("--tune", action="append", default=[], help="key:value for bwts_b200_tune (experiments)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the forward and inverse outputs of the last timed step to DIR/*.npy (GPU arm)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arm; --impl reference has none to write")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl != "reference" and world != args.gpus and world == 1 and args.gpus > 1:
        # not under torchrun: re-launch ourselves with one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29533", str(Path(__file__).resolve())] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.workload is None:
        args.workload = default_workload(max(world, args.gpus))
        args.default_workload = True
    else:
        args.default_workload = False
        args.multi_block = False  # the extra leg belongs to the default run only
    claim_stdout()
    if args.impl == "reference":
        run_reference_arm(args, rank, max(world, args.gpus, 1))
        return
    run_gpu_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
