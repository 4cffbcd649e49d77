"""Diagnostic (not a test): the FM-index (bwts_b200_fm_*) on the GPU, device-resident.

    python tests/gpu_fm_timing.py --out DIR [--warmup 3] [--steps 5] [--workloads C2,C4,C3F]

Per workload (bench.py's seeded inputs, tests/gpu_bwt_timing.py):
  * build: bwts_b200_fm_build_device (sample 32) against bwts_b200_sa_device and bwts_b200_divbwt_forward_device alone;
  * count: 2^20 patterns of 16, 64 and 256 bytes in one call, hits (substrings at random positions) and near misses
    (the same with the middle byte replaced by the byte at another random position), in patterns/s and pattern
    bytes/s;
  * locate: 2^20 single rows at random, at sample 8, 32 and 128, in rows/s;
  * index bytes per input byte at each of those sample rates.
Each figure is the median of --steps steps after --warmup warm-ups; the legs of one group run alternated inside each
step, timed with CUDA events around the call on the caller's stream, with per-launch events off.  Every count step
checks that every hit has a non-empty range.  DIR/fm_timing.json holds median, min and max per leg, the
GPU's name and its power limit."""
import argparse
import json
import statistics
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent))
import helpers  # noqa: E402
from gpu_bwt_timing import WORKLOADS, gpu_info  # noqa: E402

NPAT = 1 << 20


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--workloads", default="C2,C4,C3F")
    args = ap.parse_args()
    import torch
    bwts = helpers.load_product()
    gen = helpers.Generator()
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream(dev)
    s = stream.cuda_stream
    res = {"gpu": gpu_info(), "torch_gpu_name": torch.cuda.get_device_name(0), "warmup": args.warmup,
           "steps": args.steps, "npat": NPAT, "workloads": {}}

    def timed(box, name, fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        out = fn()
        e1.record(stream)
        e1.synchronize()
        box.setdefault(name, []).append(e0.elapsed_time(e1))
        return out

    def summary(t):
        return {"median_ms": statistics.median(t), "min_ms": min(t), "max_ms": max(t), "all_ms": t}

    with bwts.Context(0) as ctx:
        ctx.set_profile(False)
        for w in args.workloads.split(","):
            kind, seed, n = WORKLOADS[w]
            x = b"a" * n if kind is None else gen.make(kind, seed, n)
            d_x = torch.frombuffer(bytearray(x), dtype=torch.uint8).to(dev)
            torch.cuda.synchronize()
            rec = {"n": n, "kind": kind or "one byte", "seed": seed}
            # -- build
            d_sa = torch.empty(n, dtype=torch.int32, device=dev)
            d_u = torch.empty_like(d_x)
            box = {}
            for step in range(args.warmup + args.steps):
                if step == args.warmup:
                    box.clear()
                timed(box, "sa_device", lambda: ctx.sa_device(d_x.data_ptr(), n, d_sa.data_ptr(), s))
                timed(box, "divbwt_forward_device", lambda: ctx.divbwt_forward_device(d_x.data_ptr(), n, d_u.data_ptr(), s))
                timed(box, "fm_build_device", lambda: ctx.fm_build_device(d_x.data_ptr(), n, 32, s)).close()
            rec["build"] = {k: summary(v) for k, v in box.items()}
            del d_sa, d_u
            torch.cuda.empty_cache()
            # -- count
            g = torch.Generator(device=dev)
            g.manual_seed(11)
            fm = ctx.fm_build_device(d_x.data_ptr(), n, 32, s)
            rec["count"] = {}
            d_rng = torch.empty(2 * NPAT, dtype=torch.int32, device=dev)
            for m in (16, 64, 256):
                start = torch.randint(0, n - m, (NPAT,), device=dev, generator=g)
                j = torch.arange(m, device=dev)
                hits = d_x[start[:, None] + j].contiguous()
                miss = hits.clone()
                miss[:, m // 2] = d_x[torch.randint(0, n, (NPAT,), device=dev, generator=g)]
                off = torch.arange(NPAT + 1, dtype=torch.int64, device=dev) * m
                torch.cuda.synchronize()  # the inputs come from torch's stream, the calls run on `stream`
                box = {}
                for step in range(args.warmup + args.steps):
                    if step == args.warmup:
                        box.clear()
                    for name, P in (("hits", hits), ("misses", miss)):
                        timed(box, name, lambda: ctx.fm_count_device(fm, P.data_ptr(), NPAT * m, off.data_ptr(), NPAT,
                                                                     d_rng.data_ptr(), s))
                        if name == "hits":
                            assert bool((d_rng[1::2] > d_rng[0::2]).all()), (w, m)
                for name, t in box.items():
                    r = summary(t)
                    r["patterns_per_s"] = NPAT / (r["median_ms"] / 1e3)
                    r["pattern_bytes_per_s"] = NPAT * m / (r["median_ms"] / 1e3)
                    rec["count"][f"{name}_{m}"] = r
                del hits, miss, off
            fm.close()
            # -- locate and index size per sample rate
            rec["locate"], rec["index_bytes_per_byte"] = {}, {}
            rows = torch.randint(0, n, (NPAT,), device=dev, generator=g).to(torch.int32)
            d_rng = torch.stack([rows, rows + 1], 1).reshape(-1).contiguous()
            d_pos = torch.empty(NPAT, dtype=torch.int32, device=dev)
            torch.cuda.synchronize()
            for sample in (8, 32, 128):
                fm = ctx.fm_build_device(d_x.data_ptr(), n, sample, s)
                rec["index_bytes_per_byte"][sample] = fm.nbytes / n
                box = {}
                for step in range(args.warmup + args.steps):
                    if step == args.warmup:
                        box.clear()
                    timed(box, "locate", lambda: ctx.fm_locate_device(fm, d_rng.data_ptr(), NPAT, d_pos.data_ptr(),
                                                                       NPAT, s))
                r = summary(box["locate"])
                r["rows_per_s"] = NPAT / (r["median_ms"] / 1e3)
                rec["locate"][sample] = r
                fm.close()
            res["workloads"][w] = rec
            print(w, "build", {k: round(v["median_ms"], 2) for k, v in rec["build"].items()},
                  "count Mpat/s", {k: round(v["patterns_per_s"] / 1e6, 1) for k, v in rec["count"].items()},
                  "locate Mrows/s", {k: round(v["rows_per_s"] / 1e6, 1) for k, v in rec["locate"].items()},
                  "B/B", {k: round(v, 3) for k, v in rec["index_bytes_per_byte"].items()}, flush=True)
            del d_x, d_rng, d_pos, rows
            torch.cuda.empty_cache()
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "fm_timing.json").write_text(json.dumps(res, indent=1) + "\n")
    print("gpu:", res["gpu"])


if __name__ == "__main__":
    main()
