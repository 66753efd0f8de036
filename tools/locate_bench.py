"""Throughput of batched exact-match queries (Context.locate) against a resident index:
    python tools/locate_bench.py [--config 4] [--counts 1000000,10000000] [--lengths 20,32,100,1000] [--out FILE]

Builds the synthetic genome of the config (C4: 3.1 Gbp, index far larger than the 126 MB L2), then for every
(batch size, pattern length): half the patterns cut from the genome, half random ACGT; one warm-up call, then --reps timed
calls with counts only (max_hits=0) and --reps with positions (max_hits=--max-hits). Reports per call patterns/s, hits/s,
device time of the locate kernels (CUDA events on the library's stream: stats ms_locate), algorithmic bytes (stats
bytes_locate: 24 B per bisection step, 16 B per further 32 symbols compared, 8 B per reported position) and their share of
the 7.7 TB/s HBM roofline, plus a per-kernel split from one torch.profiler pass. Card name and power limit are read in the
same run. A combination whose pattern bytes exceed --max-bytes is skipped (host memory) and reported as such."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import asgart_b200 as ab  # noqa: E402

HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU (1,000 W card)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "sm_clock_max": clk}
    except Exception as e:  # noqa: BLE001
        return {"name": None, "error": str(e)}


def make_batch(strand: np.ndarray, n: int, L: int, rng) -> tuple:
    n_cut = n // 2
    starts = rng.integers(0, len(strand) - 1 - L, n_cut)
    buf = np.empty((n, L), dtype=np.uint8)
    for a in range(0, n_cut, 1 << 16):   # gather in pieces: bounded temporaries
        b = min(n_cut, a + (1 << 16))
        buf[a:b] = strand[starts[a:b, None] + np.arange(L)[None, :]]
    buf[n_cut:] = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, (n - n_cut, L), dtype=np.uint8)]
    return buf.reshape(-1), np.arange(n + 1, dtype=np.uint64) * L


def kernel_split(ctx, batch, max_hits):
    """device ms per kernel name over one call (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.locate(batch, max_hits=max_hits)
    out = {}
    for ev in prof.key_averages():
        name = ev.key
        if "locate" in name or "scan_" in name:
            short = name.split("(")[0].split("<")[0].replace("void ", "").replace("ab200::", "")
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            out[short] = round(out.get(short, 0.0) + t / 1e3, 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=4)
    ap.add_argument("--scale-n", type=int, default=0)
    ap.add_argument("--counts", default="1000000,10000000")
    ap.add_argument("--lengths", default="20,32,100,1000")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--max-hits", type=int, default=8)
    ap.add_argument("--max-bytes", type=float, default=4e9)
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if ab.device_count() <= 0:
        sys.exit("locate_bench: no CUDA device (asgart_b200 has no CPU path)")
    info = {"card": card(), "config": a.config}
    g, fr = ab.synth_genome(a.config, scale_n=a.scale_n, threads=os.cpu_count() or 8)
    prep = ab.Prepared.from_memory(ab.normalise(g, False), fr, f"synthC{a.config}.fa")
    strand = np.array(prep.strand)
    del g
    info["strand_bp"] = int(len(strand))
    rows = []
    out = open(a.out, "w") if a.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    with ab.Context(0) as ctx:
        ctx.load_strand(strand)
        ctx.build_index()
        info["index_bits"] = ctx.stats()["sa_index_bits"]
        emit({"run": info})
        rng = np.random.default_rng(1)
        for n in [int(float(x)) for x in a.counts.split(",")]:
            for L in [int(x) for x in a.lengths.split(",")]:
                if n * L > a.max_bytes:
                    emit({"n_patterns": n, "length": L, "skipped": f"{n * L} pattern bytes > --max-bytes {a.max_bytes:.0f}"})
                    continue
                batch = make_batch(strand, n, L, rng)
                rec = {"n_patterns": n, "length": L}
                for mode, mh in (("counts", 0), ("positions", a.max_hits)):
                    ctx.locate(batch, max_hits=mh)   # warm-up
                    reps = []
                    for _ in range(a.reps):
                        ctx.reset_stats()
                        t0 = time.perf_counter()
                        h = ctx.locate(batch, max_hits=mh)
                        wall = time.perf_counter() - t0
                        s = ctx.stats()
                        ms = s["ms_locate"]
                        reps.append({"wall_s": round(wall, 4), "device_ms": round(ms, 3),
                                     "patterns_per_s_device": round(n / (ms / 1e3)), "patterns_per_s_wall": round(n / wall),
                                     "hits": int(s["locate_hits"]), "hits_per_s_device": round(s["locate_hits"] / (ms / 1e3)),
                                     "alg_bytes": int(s["bytes_locate"]),
                                     "hbm_fraction": round(s["bytes_locate"] / (ms / 1e3) / HBM_BYTES_PER_S, 4)})
                    rec[mode] = {"max_hits": mh, "reps": reps, "matched_patterns": int((h.count > 0).sum()),
                                 "total_count": int(h.count.sum())}
                    if not a.no_profile:
                        rec[mode]["kernel_ms"] = kernel_split(ctx, batch, mh)
                emit(rec)
                rows.append(rec)
                del batch
    if out:
        out.close()


if __name__ == "__main__":
    main()
