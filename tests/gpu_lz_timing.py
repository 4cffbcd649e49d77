"""Diagnostic (not a test): device-resident suffix array + LCP array (bwts_b200_sa_lcp_device) against the LPF array
(bwts_b200_lpf_device) and against the LZ77 parse (bwts_b200_lz77_device).

    python tests/gpu_lz_timing.py --out DIR [--warmup 2] [--steps 5] [--workloads C2,C4,C3F,all_a]

Inputs are those of tests/gpu_bwt_timing.py (bench.py's seeded workloads plus 64 MiB of one byte).  Each step runs
the three legs back to back on one context, so that drift on a shared machine touches them alike; each leg is timed
with CUDA events around the call on the caller's stream, with per-launch events off.  The LPF stage is the LPF leg
minus the SA + LCP leg, the parse the LZ77 leg minus the LPF leg.  One more LZ77 call with per-launch events on
records the emit class per kernel name.  DIR/lz_timing.json holds median, min and max per leg, the stage times, the
kernel breakdown, the GPU's name and its power limit."""
import argparse
import json
import statistics
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent))
import helpers  # noqa: E402
from gpu_bwt_timing import WORKLOADS, gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--workloads", default="C2,C4,C3F,all_a")
    args = ap.parse_args()
    import torch
    bwts = helpers.load_product()
    gen = helpers.Generator()
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream(dev)
    res = {"gpu": gpu_info(), "torch_gpu_name": torch.cuda.get_device_name(0), "warmup": args.warmup,
           "steps": args.steps, "workloads": {}}
    with bwts.Context(0) as ctx:
        ctx.set_profile(False)
        for w in args.workloads.split(","):
            kind, seed, n = WORKLOADS[w]
            x = b"a" * n if kind is None else gen.make(kind, seed, n)
            d_x = torch.frombuffer(bytearray(x), dtype=torch.uint8).to(dev)
            d_sa, d_lcp, d_lpf, d_prev = (torch.empty(n, dtype=torch.int32, device=dev) for _ in range(4))
            d_f = torch.empty((n, 2), dtype=torch.int32, device=dev)
            box, zs = {}, []

            def leg(name, fn):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                fn()
                e1.record(stream)
                e1.synchronize()
                box.setdefault(name, []).append(e0.elapsed_time(e1))

            s = stream.cuda_stream
            p = d_x.data_ptr()
            for step in range(args.warmup + args.steps):
                if step == args.warmup:
                    box.clear()
                leg("sa_lcp", lambda: ctx.sa_lcp_device(p, n, d_sa.data_ptr(), d_lcp.data_ptr(), s))
                leg("lpf", lambda: ctx.lpf_device(p, n, d_lpf.data_ptr(), d_prev.data_ptr(), s))
                leg("lz77", lambda: zs.append(ctx.lz77_device(p, n, d_f.data_ptr(), n, s)))
            assert len(set(zs)) == 1, (w, zs)
            rec = {"n": n, "kind": kind or "one byte", "seed": seed, "z": zs[0], "lpf_max": int(d_lpf.max())}
            for name, t in box.items():
                rec[name] = {"median_ms": statistics.median(t), "min_ms": min(t), "max_ms": max(t), "all_ms": t}
            med = {k: rec[k]["median_ms"] for k in box}
            rec["lpf_stage_ms"] = med["lpf"] - med["sa_lcp"]
            rec["parse_ms"] = med["lz77"] - med["lpf"]
            # the suffix sort alone: the LCP stage's kernels are separated out in the profiled call below
            ctx.set_profile(True)
            ctx.lz77_device(p, n, d_f.data_ptr(), n, s)
            torch.cuda.synchronize()
            st = ctx.stats()
            ctx.set_profile(False)
            rec["profiled"] = {"total_ms": st["total_ms"], "phases": st["phases"],
                               "emit_class": st["classes"].get("emit")}
            print(w, {k: round(v, 3) for k, v in med.items()}, "LPF stage %.3f ms, parse %.3f ms, z %d"
                  % (rec["lpf_stage_ms"], rec["parse_ms"], rec["z"]), flush=True)
            res["workloads"][w] = rec
            del d_x, d_sa, d_lcp, d_lpf, d_prev, d_f
            torch.cuda.empty_cache()
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "lz_timing.json").write_text(json.dumps(res, indent=1) + "\n")
    print("gpu:", res["gpu"])


if __name__ == "__main__":
    main()
