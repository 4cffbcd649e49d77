"""Diagnostic (not a test): device-resident suffix array alone (bwts_b200_sa_device) against suffix array + LCP
array (bwts_b200_sa_lcp_device).

    python tests/gpu_sa_lcp_timing.py --out DIR [--warmup 3] [--steps 5] [--workloads C1,C2,C3,C3F,C4,all_a]

Inputs are those of tests/gpu_bwt_timing.py (bench.py's seeded workloads plus 64 MiB of one byte).  Each step runs
the two legs back to back on one context, so that drift on a shared machine touches both alike; each leg is timed
with CUDA events around the call on the caller's stream, with per-launch events off.  Every step checks that the
two suffix arrays agree.  One more call with per-launch events on records the forward's phase times and the emit
class (k_emit_sa and the k_lcp_* kernels; BWTS_B200_TRACE=1 lists them one by one).  DIR/sa_lcp_timing.json holds
median, min and max per leg, the LCP stage (the difference of the medians), the GPU's name and its power limit."""
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
            d_sa, d_sa2, d_lcp = (torch.empty(n, dtype=torch.int32, device=dev) for _ in range(3))
            box = {}

            def leg(name, fn):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                fn()
                e1.record(stream)
                e1.synchronize()
                box.setdefault(name, []).append(e0.elapsed_time(e1))

            s = stream.cuda_stream
            for step in range(args.warmup + args.steps):
                if step == args.warmup:
                    box.clear()
                leg("sa", lambda: ctx.sa_device(d_x.data_ptr(), n, d_sa.data_ptr(), s))
                leg("sa_lcp", lambda: ctx.sa_lcp_device(d_x.data_ptr(), n, d_sa2.data_ptr(), d_lcp.data_ptr(), s))
                assert torch.equal(d_sa, d_sa2), (w, step)
            rec = {"n": n, "kind": kind or "one byte", "seed": seed, "lcp_max": int(d_lcp.max()),
                   "lcp_mean": float(d_lcp.double().mean())}
            for name, t in box.items():
                rec[name] = {"median_ms": statistics.median(t), "min_ms": min(t), "max_ms": max(t),
                             "MBps_median": n / 1e6 / (statistics.median(t) / 1e3), "all_ms": t}
            lcp_ms = rec["sa_lcp"]["median_ms"] - rec["sa"]["median_ms"]
            rec["lcp_stage_ms"] = lcp_ms
            rec["lcp_stage_ns_per_byte"] = lcp_ms * 1e6 / n
            rec["lcp_stage_over_sa"] = lcp_ms / rec["sa"]["median_ms"]
            ctx.set_profile(True)
            ctx.sa_lcp_device(d_x.data_ptr(), n, d_sa2.data_ptr(), d_lcp.data_ptr(), s)
            st = ctx.stats()
            ctx.set_profile(False)
            rec["profiled"] = {"total_ms": st["total_ms"], "phases": st["phases"],
                               "emit_class": st["classes"].get("emit")}
            res["workloads"][w] = rec
            print(w, {k: round(v["median_ms"], 3) for k, v in rec.items() if isinstance(v, dict) and "median_ms" in v},
                  "lcp stage %.3f ms (%.2f ns/B, %.1f %% of SA)" % (lcp_ms, rec["lcp_stage_ns_per_byte"],
                                                                    100 * rec["lcp_stage_over_sa"]), flush=True)
            del d_x, d_sa, d_sa2, d_lcp
            torch.cuda.empty_cache()
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "sa_lcp_timing.json").write_text(json.dumps(res, indent=1) + "\n")
    print("gpu:", res["gpu"])


if __name__ == "__main__":
    main()
