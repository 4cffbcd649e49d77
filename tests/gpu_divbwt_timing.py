"""Diagnostic (not a test): device-resident divbwt (libdivsufsort's end-of-text BWT) forward / inverse beside the
BWTS and classic BWT forward / inverse.

    python tests/gpu_divbwt_timing.py --out DIR [--warmup 3] [--steps 5] [--workloads C1,C2,C3,C3F,C4,all_a]

Inputs are those of tests/gpu_bwt_timing.py (bench.py's seeded workloads plus 64 MiB of one byte).  Each step
runs the six legs back to back on one context (BWTS, classic BWT and divbwt forward, then the three inverses of
those outputs), so that drift on a shared machine touches all legs alike; each leg is timed with CUDA events
around the call on the caller's stream.  Every step checks the three round trips.  DIR/divbwt_timing.json holds
median, min and max per leg, the GPU's name and its power limit."""
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
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
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
            d_s, d_b, d_d, d_back = (torch.empty_like(d_x) for _ in range(4))
            box = {}

            def leg(name, fn):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                r = fn()
                e1.record(stream)
                e1.synchronize()
                box.setdefault(name, []).append(e0.elapsed_time(e1))
                return r

            s = stream.cuda_stream
            for step in range(args.warmup + args.steps):
                if step == args.warmup:
                    box.clear()
                leg("bwts_forward", lambda: ctx.forward_device(d_x.data_ptr(), n, d_s.data_ptr(), s))
                p = leg("bwt_forward", lambda: ctx.bwt_forward_device(d_x.data_ptr(), n, d_b.data_ptr(), s))
                pd = leg("divbwt_forward", lambda: ctx.divbwt_forward_device(d_x.data_ptr(), n, d_d.data_ptr(), s))
                leg("bwts_inverse", lambda: ctx.inverse_device(d_s.data_ptr(), n, d_back.data_ptr(), s))
                ok_s = torch.equal(d_back, d_x)
                leg("bwt_inverse", lambda: ctx.bwt_inverse_device(d_b.data_ptr(), n, p, d_back.data_ptr(), s))
                ok_b = torch.equal(d_back, d_x)
                leg("divbwt_inverse", lambda: ctx.divbwt_inverse_device(d_d.data_ptr(), n, pd, d_back.data_ptr(), s))
                ok_d = torch.equal(d_back, d_x)
                assert ok_s and ok_b and ok_d, (w, step, ok_s, ok_b, ok_d)
            rec = {"n": n, "kind": kind or "one byte", "seed": seed, "bwt_primary": p, "divbwt_primary": pd}
            for name, t in box.items():
                rec[name] = {"median_ms": statistics.median(t), "min_ms": min(t), "max_ms": max(t),
                             "MBps_median": n / 1e6 / (statistics.median(t) / 1e3), "all_ms": t}
            res["workloads"][w] = rec
            print(w, {k: round(v["median_ms"], 3) for k, v in rec.items() if isinstance(v, dict)}, flush=True)
            del d_x, d_s, d_b, d_d, d_back
            torch.cuda.empty_cache()
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "divbwt_timing.json").write_text(json.dumps(res, indent=1) + "\n")
    print("gpu:", res["gpu"])


if __name__ == "__main__":
    main()
