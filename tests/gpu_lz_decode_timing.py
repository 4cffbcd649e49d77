"""Diagnostic (not a test): device-resident LZ77 decoding (bwts_b200_lz77_decode_device) of the greedy parse of each
workload, beside the parse itself (bwts_b200_lz77_device).

    python tests/gpu_lz_decode_timing.py --out DIR [--warmup 2] [--steps 5] [--workloads C2,C4,C3F,all_a]

Inputs are those of tests/gpu_bwt_timing.py (bench.py's seeded workloads plus 64 MiB of one byte).  The parse is made
once per workload; each step then times the parse and the decode with CUDA events around the call on the caller's
stream, with per-launch events off, and checks the decode against the input on the device.  One more decode with
per-launch events on records the rounds, live_sum and milliseconds per kernel class.  DIR/lz_decode_timing.json
holds median, min and max per leg, that breakdown, the GPU's name and its power limit."""
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
            d_f = torch.empty((n // 2 + 64, 2), dtype=torch.int32, device=dev)
            d_out = torch.empty(n, dtype=torch.uint8, device=dev)
            s = stream.cuda_stream
            box, zs = {}, []

            def leg(name, fn):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                fn()
                e1.record(stream)
                e1.synchronize()
                box.setdefault(name, []).append(e0.elapsed_time(e1))

            for step in range(args.warmup + args.steps):
                if step == args.warmup:
                    box.clear()
                leg("lz77", lambda: zs.append(ctx.lz77_device(d_x.data_ptr(), n, d_f.data_ptr(), d_f.shape[0], s)))
                d_out.fill_(0)
                torch.cuda.synchronize()
                leg("decode", lambda: ctx.lz77_decode_device(d_f.data_ptr(), zs[-1], n, d_out.data_ptr(), s))
                assert torch.equal(d_out, d_x), w
            assert len(set(zs)) == 1, (w, zs)
            rec = {"n": n, "kind": kind or "one byte", "seed": seed, "z": zs[0]}
            for name, t in box.items():
                rec[name] = {"median_ms": statistics.median(t), "min_ms": min(t), "max_ms": max(t), "all_ms": t}
            ctx.set_profile(True)
            ctx.lz77_decode_device(d_f.data_ptr(), zs[0], n, d_out.data_ptr(), s)
            torch.cuda.synchronize()
            st = ctx.stats()
            ctx.set_profile(False)
            rec["profiled"] = {"total_ms": st["total_ms"], "rounds": st["rounds"], "live_sum": st["live_sum"],
                               "phases": st["phases"], "classes": st["classes"]}
            print(w, "parse %.3f ms, decode %.3f ms (min %.3f, max %.3f), z %d, rounds %d, live_sum %d"
                  % (rec["lz77"]["median_ms"], rec["decode"]["median_ms"], rec["decode"]["min_ms"],
                     rec["decode"]["max_ms"], rec["z"], st["rounds"], st["live_sum"]),
                  {k: round(v["ms"], 3) for k, v in st["classes"].items()}, flush=True)
            res["workloads"][w] = rec
            del d_x, d_f, d_out
            torch.cuda.empty_cache()
    res["gpu_after"] = gpu_info()
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "lz_decode_timing.json").write_text(json.dumps(res, indent=1) + "\n")
    print("gpu:", res["gpu"])


if __name__ == "__main__":
    main()
