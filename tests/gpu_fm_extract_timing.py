"""Diagnostic (not a test): FM-index extract (bwts_b200_fm_extract_device) on the GPU, device-resident.

    python tests/gpu_fm_extract_timing.py --out DIR [--warmup 3] [--steps 5] [--workloads C2,C4,C3F]

Per workload (bench.py's seeded inputs, tests/gpu_bwt_timing.py) and per sample rate 8, 32 and 128:
  * snippets: 2^20 ranges of 64 bytes at random starts in one call, in output bytes/s;
  * whole: the range [0, n), beside bwts_b200_divbwt_inverse_device of the same text's divbwt (once per workload);
  * one: a single 64-byte range, which isolates the per-call work that does not depend on the ranges (the inverse
    table of the samples).
Each figure is the median of --steps steps after --warmup warm-ups, timed with CUDA events around the call on the
caller's stream with per-launch events off; a 512 MiB buffer is overwritten before every timed call, so no leg
starts with its index or table in L2.  After the timed steps one call per leg runs with per-launch events on and its
inv_scan (checks, scans, table) and inv_walk (walk) times are kept.  Every leg's output is checked against the text
once.  DIR/fm_extract_timing.json holds median, min and max per leg, the GPU's name and its power limit."""
import argparse
import json
import statistics
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent))
import helpers  # noqa: E402
from gpu_bwt_timing import WORKLOADS, gpu_info  # noqa: E402

NSNIP, SNIP = 1 << 20, 64


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
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    res = {"gpu": gpu_info(), "torch_gpu_name": torch.cuda.get_device_name(0), "warmup": args.warmup,
           "steps": args.steps, "snippets": [NSNIP, SNIP], "l2": "512 MiB overwritten before every timed call",
           "workloads": {}}

    def timed(box, name, fn):
        with torch.cuda.stream(stream):
            flush.fill_(len(box.get(name, [])) & 0xff)
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
        for w in args.workloads.split(","):
            kind, seed, n = WORKLOADS[w]
            x = b"a" * n if kind is None else gen.make(kind, seed, n)
            d_x = torch.frombuffer(bytearray(x), dtype=torch.uint8).to(dev)
            del x
            rec = {"n": n, "kind": kind or "one byte", "seed": seed, "samples": {}}
            g = torch.Generator(device=dev)
            g.manual_seed(17)
            start = torch.randint(0, n - SNIP, (NSNIP,), device=dev, generator=g, dtype=torch.int64)
            snip_rng = torch.stack([start, start + SNIP], 1).to(torch.int32).reshape(-1).contiguous()
            want_snip = d_x[start[:, None] + torch.arange(SNIP, device=dev)].reshape(-1)
            whole_rng = torch.tensor([0, n], dtype=torch.int32, device=dev)
            one_rng = torch.tensor([n // 2, n // 2 + SNIP], dtype=torch.int32, device=dev)
            d_out = torch.empty(max(n, NSNIP * SNIP), dtype=torch.uint8, device=dev)
            legs = {"snippets": (snip_rng, NSNIP, NSNIP * SNIP), "whole": (whole_rng, 1, n), "one": (one_rng, 1, SNIP)}
            torch.cuda.synchronize()
            # -- the inverse transform of the same text, for the whole-text leg
            d_u = torch.empty_like(d_x)
            ctx.set_profile(False)
            primary = ctx.divbwt_forward_device(d_x.data_ptr(), n, d_u.data_ptr(), s)
            box = {}
            for step in range(args.warmup + args.steps):
                if step == args.warmup:
                    box.clear()
                timed(box, "inverse_bw_transform", lambda: ctx.divbwt_inverse_device(d_u.data_ptr(), n, primary,
                                                                                      d_out.data_ptr(), s))
            stream.synchronize()
            assert torch.equal(d_out[:n], d_x), w
            rec["inverse_bw_transform"] = summary(box["inverse_bw_transform"])
            del d_u
            for sample in (8, 32, 128):
                fm = ctx.fm_build_device(d_x.data_ptr(), n, sample, s)
                r = {"index_bytes_per_byte": fm.nbytes / n}
                ctx.set_profile(False)
                box = {}
                for step in range(args.warmup + args.steps):
                    if step == args.warmup:
                        box.clear()
                    for name, (rng, nr, tot) in legs.items():
                        got = timed(box, name, lambda: ctx.fm_extract_device(fm, rng.data_ptr(), nr, d_out.data_ptr(),
                                                                             tot, s))
                        assert got == tot, (w, sample, name)
                        if step == 0:
                            stream.synchronize()
                            want = {"snippets": want_snip, "whole": d_x, "one": d_x[n // 2:n // 2 + SNIP]}[name]
                            assert torch.equal(d_out[:tot], want), (w, sample, name)
                ctx.set_profile(True)
                for name, (rng, nr, tot) in legs.items():
                    leg = summary(box[name])
                    leg["bytes_per_s"] = tot / (leg["median_ms"] / 1e3)
                    ctx.fm_extract_device(fm, rng.data_ptr(), nr, d_out.data_ptr(), tot, s)
                    st = ctx.stats()
                    leg["profiled_class_ms"] = {k: v["ms"] for k, v in st["classes"].items()}
                    r[name] = leg
                fm.close()
                rec["samples"][sample] = r
                print(w, "sample", sample, {k: round(r[k]["median_ms"], 3) for k in legs},
                      "ms; snippets GB/s", round(r["snippets"]["bytes_per_s"] / 1e9, 2),
                      "whole GB/s", round(r["whole"]["bytes_per_s"] / 1e9, 2), "classes(one)",
                      {k: round(v, 3) for k, v in r["one"]["profiled_class_ms"].items()}, flush=True)
            print(w, "inverse_bw_transform ms", round(rec["inverse_bw_transform"]["median_ms"], 3), flush=True)
            res["workloads"][w] = rec
            del d_x, d_out, start, snip_rng, want_snip
            torch.cuda.empty_cache()
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "fm_extract_timing.json").write_text(json.dumps(res, indent=1) + "\n")
    print("gpu:", res["gpu"])


if __name__ == "__main__":
    main()
