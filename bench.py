#!/usr/bin/env python
"""bench.py — the hot path (SA build + LUT + probe search + arm automaton + post-steps) on synthetic genomes.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 1..5] [--scale-n BP] [--impl ours|reference]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

One JSON line on rank 0. A "step" = one whole pass of the path over the workload genome:
  value  (bp/s)  device-resident input: strand already in HBM, K x [build_index + search + post-steps], CUDA events on
                 the library's stream, max over ranks.
  e2e    (bp/s)  same through the C ABI with HOST buffers: K x [load_strand (H2D from pinned memory) + build_index +
                 search + post-steps + families D2H].
Workload (default, every N) = BASELINE.json configs[3], the configuration its metric is quoted on and the north-star
target: synthetic 3.1 Gbp 24-fragment human-genome-sized multiFASTA, -RC, k=20, g=100 (fits one B200: ~115 GB peak).
`--config 2` selects configs[1] (57 Mbp chrY-sized, -RC -S). N>1: the same genome (strong scaling); the index is built
by all GPUs together (sharded suffix-array build: key ranges per GPU, rank array in peer memory over NVLink, NCCL at the
phase boundaries and for the final exchange of SA pieces), then every GPU holds the whole index, probes are partitioned
by position and the stage-A partials are all-gathered (NCCL).
`--impl reference` times the reference algorithm on the host cores: the reference's own libdivsufsort64 (oracle/_ref) +
the oracle port of its Rust probe loop/automaton/post-steps (no Rust toolchain exists here), all host threads.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

CONFIG_FLAGS = {
    1: dict(),
    2: dict(reverse=True, complement=True, skip_masked=True),
    3: dict(reverse=True, complement=True, max_cardinality=500),
    4: dict(reverse=True, complement=True),
    5: dict(reverse=True, complement=True, probe_size=32, gap_size=200),
}
CONFIG_NAMES = {
    1: "C1 synthetic 10 Mbp single-FASTA, 40 planted direct pairs, direct only",
    2: "C2 synthetic 57 Mbp chrY-sized, planted direct+RC duplications, -RC -S",
    3: "C3 synthetic 250 Mbp chr1-sized, -RC, max_cardinality=500",
    4: "C4 synthetic 3.1 Gbp 24-fragment multiFASTA, -RC",
    5: "C5 cross-genome: two synthetic 1 Gbp 10-fragment genomes with shared planted segments, -RC, k=32, g=200",
}
FULL_N = {1: 10_000_000, 2: 57_227_415, 3: 248_956_422, 4: 3_088_269_832, 5: 2_000_000_000}
METRIC = "bp/s searched end-to-end (SA build + search + clustering; -RC, k=20, g=100)"


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled during the timed region."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def make_workload(config: int, scale_n: int):
    import asgart_b200 as ab
    flags = CONFIG_FLAGS[config]
    st = ab.RunSettings(**flags)
    threads = os.cpu_count() or 8
    if config == 5:     # `asgart A.fa B.fa`: the two genomes concatenated with a running offset (src/bin/asgart.rs:375-395)
        ga, fa = ab.synth_genome(5, part=0, scale_n=scale_n // 2, threads=threads)
        gb, fb = ab.synth_genome(5, part=1, scale_n=scale_n // 2, threads=threads)
        g = np.concatenate([ga, gb])
        fr = fa + [(nm, pos + len(ga), ln) for nm, pos, ln in fb]
        names = "synthC5_A.fa, synthC5_B.fa"
    else:
        g, fr = ab.synth_genome(config, scale_n=scale_n, threads=threads)
        names = f"synthC{config}.fa"
    prep = ab.Prepared.from_memory(ab.normalise(g, st.skip_masked), fr, names)
    return st, prep


def oracle_settings(st):
    import oracle
    return oracle.make_settings(probe_size=st.probe_size, gap_size=st.gap_size, min_length=st.min_duplication_length,
                                max_cardinality=st.max_cardinality, reverse=st.reverse, complement=st.complement,
                                skip_masked=st.skip_masked)


def oracle_workload(config: int, scale_n: int):
    """The workload as the REFERENCE side sees it: same generated bases, but normalisation table aside, the fragment
    map, the chunk list and the '$' come from the oracle's restatement of prepare_data (src/bin/asgart.rs:273-471) — used
    by the reference arm, cpu_baseline and tests/golden/make_families_golden.py, never by our arm."""
    import asgart_b200 as ab
    import oracle
    flags = CONFIG_FLAGS[config]
    st = ab.RunSettings(**flags)
    threads = os.cpu_count() or 8
    if config == 5:
        ga, fa = ab.synth_genome(5, part=0, scale_n=scale_n // 2, threads=threads)
        gb, fb = ab.synth_genome(5, part=1, scale_n=scale_n // 2, threads=threads)
        fr = fa + [(nm, pos + len(ga), ln) for nm, pos, ln in fb]
        g = np.concatenate([ga, gb])
        del ga, gb
        names = "synthC5_A.fa, synthC5_B.fa"
    else:
        g, fr = ab.synth_genome(config, scale_n=scale_n, threads=threads)
        names = f"synthC{config}.fa"
    g = ab.normalise(g, st.skip_masked)
    prep = oracle.Prepared.from_memory(g, fr, names)
    del g
    return st, prep


def searched_bp(prep) -> int:
    return int(sum(c[1] for c in prep.chunks))


DUMP_LIMIT_BYTES = 64 << 20


def _dump_rows(n: int, row_bytes: int, budget_bytes: int) -> np.ndarray:
    """All n row numbers, or a fixed seeded sample of them (in order) when n rows would exceed the byte budget."""
    if n * row_bytes <= budget_bytes:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, size=budget_bytes // row_bytes, replace=False))


def dump_families(out_dir: str, fam) -> None:
    """Write the families a caller of Context.search receives as <out_dir>/<field>.npy (float64; identity float32), so
    that two builds can be compared output for output. Positions stay exact in float64 (< 2^53). Above 64 MB in all, a
    fixed seeded sample of the family offsets (at most half the budget) and of the duplicons is written; fam_index.npy
    and sd_index.npy hold the row numbers written."""
    os.makedirs(out_dir, exist_ok=True)
    sds = fam.sds
    fields = ("left", "right", "left_length", "right_length", "identity", "reversed", "complemented")
    fam_rows = _dump_rows(len(fam.fam_offsets), 16, DUMP_LIMIT_BYTES // 2)           # offset + row number
    sd_rows = _dump_rows(len(sds), 8 * len(fields) + 4, DUMP_LIMIT_BYTES - 16 * len(fam_rows))   # identity is 4 B
    out = {"fam_offsets": np.asarray(fam.fam_offsets, dtype=np.float64)[fam_rows], "fam_index": fam_rows.astype(np.float64),
           "sd_index": sd_rows.astype(np.float64)}
    for f in fields:
        out[f] = sds[f][sd_rows].astype(np.float32 if f == "identity" else np.float64)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def golden(config: int):
    """tests/golden/families_c<config>.json: the oracle's digests of the full-size config, made offline on the CPU."""
    try:
        with open(os.path.join(ROOT, "tests", "golden", f"families_c{config}.json")) as f:
            return json.load(f)
    except Exception:
        return None


def workload_config(config: int, scale_n: int, st, strand_bp: int, bp: int, n_chunks: int):
    """The `config` object of the JSON line: the workload, identical for our arm and for --impl reference (which runs a
    bounded sample of it and says so in cpu_baseline.sample / sample_bp)."""
    return {"workload": CONFIG_NAMES[config], "strand_bp": strand_bp, "searched_bp": bp, "chunks": n_chunks,
            "flags": CONFIG_FLAGS[config], "probe_size": st.probe_size, "gap_size": st.gap_size,
            "min_duplication_length": st.min_duplication_length, "max_cardinality": st.max_cardinality,
            "scale_n": scale_n or None,
            "l2": "inputs larger than L2 (text + suffix array + sort buffers > 1 GB per step vs 126 MB L2); no flush needed"}


# ---------------------------------------------------------------------------------------------------- reference arm
def cpu_reference_pass(strand: np.ndarray, chunks, st, threads: int):
    """One pass of the reference algorithm on the CPU. The only place (with cpu_baseline) bench.py executes oracle/."""
    import oracle
    from asgart_b200.api import families_digest
    so = oracle_settings(st)
    kind = "reference" if oracle.ref() is not None else "port"
    t0 = time.perf_counter()
    sa = oracle.ref_divsufsort64(strand) if oracle.ref() is not None else oracle.suffix_array(strand)   # single thread, like build.rs builds it
    t1 = time.perf_counter()
    out = oracle.search(strand, sa, chunks, so, oracle.POST_ALL, threads=threads)
    t2 = time.perf_counter()
    f = out.families
    return {"seconds": t2 - t0, "sa_s": t1 - t0, "lut_s": out.seconds["lut"], "search_s": out.seconds["search"],
            "post_s": out.seconds["post"], "families": len(f.fam_offsets) - 1, "duplicons": len(f.fields), "sa_kind": kind,
            "families_sha256": families_digest(f.fam_offsets, f.fields, f.identity, f.flags)}


REF_SAMPLE_BP = 57_227_415      # the reference arm's sample per step: the workload's generator scaled to C2's length


def reference_sample_n(config: int, scale_n: int, passes: int) -> int:
    """Genome length the CPU arm runs per step: the whole workload when it is small enough, else the same generator
    scaled to REF_SAMPLE_BP (about 6-9 s per pass on 8-16 host cores), shrunk further when more than 25 passes are asked."""
    full_n = scale_n or FULL_N[config]
    cap = REF_SAMPLE_BP if passes <= 25 else max(2_000_000, REF_SAMPLE_BP * 25 // passes)
    return min(full_n, cap)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    full_n = args.scale_n or FULL_N[args.config]
    sample_n = args.ref_sample_bp or reference_sample_n(args.config, args.scale_n, args.steps + args.warmup)
    sample_n = min(sample_n, full_n)
    st, prep = oracle_workload(args.config, 0 if sample_n == FULL_N[args.config] else sample_n)   # chunker: the oracle's prepare_data
    strand = prep.strand
    bp = searched_bp(prep)
    for _ in range(args.warmup):
        cpu_reference_pass(strand, prep.chunks, st, cores)
    t0 = time.perf_counter()
    last = None
    for _ in range(args.steps):
        last = cpu_reference_pass(strand, prep.chunks, st, cores)
    dt = time.perf_counter() - t0
    value = bp * args.steps / dt
    g = golden(args.config) if not args.scale_n else None
    whole = sample_n == full_n
    if whole:
        full_bp, full_chunks = bp, len(prep.chunks)
    elif g:
        full_bp, full_chunks = g["searched_bp"], g["n_chunks"]
    else:
        full_bp, full_chunks = None, None
    sample = (f"{'whole workload' if whole else 'bounded sample of the workload'}: {len(strand) - 1} of {full_n} bp "
              f"(same generator and seeds, config C{args.config}{'' if whole else ', scaled'}), {bp} bp in {len(prep.chunks)} chunks cut by the "
              f"oracle's prepare_data; SA by the reference's libdivsufsort64 (1 thread, as build.rs builds it) + oracle port of the "
              f"Rust probe loop/automaton/post-steps ({cores} threads, one task per chunk; no rustc in this image)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "bp/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u8/int64", "data": "synthetic",
        "config": workload_config(args.config, args.scale_n, st, full_n, full_bp, full_chunks),
        "sample_bp": len(strand) - 1, "full_bp": full_n, "sample_fraction": (len(strand) - 1) / full_n,
        "cpu_baseline": {"value": value, "unit": "bp/s", "cores": cores, "kind": last["sa_kind"] if last else "port", "sample": sample,
                         "phases_s": {k: round(v, 3) for k, v in (last or {}).items() if k.endswith("_s")},
                         "families": last["families"] if last else None, "families_sha256": last["families_sha256"] if last else None},
        "e2e": {"value": value, "unit": "bp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if g:   # the one same-input CPU datapoint: the whole config, run offline by tests/golden/make_families_golden.py
        sec = g["oracle_seconds"]
        tot = sec["sa_divsufsort64_1thread"] + sec["lut"] + sec["search_automaton"] + sec["post"]
        line["offline_full_config"] = {"seconds": round(tot, 2), "bp_per_s": g["searched_bp"] / tot, "phases_s": sec,
                                       "families": g["families"], "families_sha256": g["families_sha256"],
                                       "source": f"tests/golden/families_c{args.config}.json"}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------- FASTA ingest
def fasta_bytes(seq: np.ndarray, frags, width: int = 60) -> np.ndarray:
    """The strand as a `width`-column multiFASTA, one record per fragment (numpy only: 3 GB in a few seconds)."""
    parts = []
    for name, pos, ln in frags:
        parts.append(np.frombuffer(f">{name} synthetic\n".encode(), dtype=np.uint8))
        body = seq[pos:pos + ln]
        full = ln // width * width
        rows = np.empty((ln // width, width + 1), dtype=np.uint8)
        rows[:, :width] = body[:full].reshape(-1, width)
        rows[:, width] = 10
        parts.append(rows.reshape(-1))
        if ln > full:
            parts.append(body[full:])
            parts.append(np.frombuffer(b"\n", dtype=np.uint8))
    return np.concatenate(parts)


def measure_ingest(ctx, prep, peak_gbs: float):
    """prepare_data on the device (SURVEY §8f row N1): the workload as a 60-column multiFASTA in pinned host memory ->
    strand + fragment map + chunks in HBM. Not part of `value` / `e2e` (the metric starts at the strand, like the
    reference's SearchDuplications step); reported next to them."""
    import torch
    fa = fasta_bytes(np.asarray(prep.strand)[:-1], prep.map)
    pinned = torch.empty(len(fa), dtype=torch.uint8).pin_memory()
    pinned.numpy()[:] = fa
    del fa
    view = pinned.numpy()
    best = None
    for _ in range(3):
        ctx.reset_stats()
        t0 = time.perf_counter()
        got = ctx.ingest([view], False, names=["bench.fa"])
        wall = (time.perf_counter() - t0) * 1e3
        s = ctx.stats()
        alg = 3 * s["ingest_bytes"] + (got.n1 - 1)          # three reads per file byte, one write per kept byte
        row = {"file_bytes": int(s["ingest_bytes"]), "records": int(s["ingest_records"]), "ms_wall": wall, "ms_h2d": s["ms_h2d"],
               "ms_scans": s["ms_ingest"], "ms_pack": s["ms_pack"], "scan_alg_GBps": alg / max(s["ms_ingest"], 1e-9) / 1e6,
               "gpu_launches": int(s["launches_total"])}
        row["scan_frac_of_hbm_peak"] = row["scan_alg_GBps"] / peak_gbs
        assert got.map == prep.map and got.chunks == [tuple(c) for c in prep.chunks] and got.n1 == len(prep.strand)
        if best is None or row["ms_wall"] < best["ms_wall"]:
            best = row
    return best


# ---------------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch

    import asgart_b200 as ab

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    # rank 0 generates the genome with all host threads; the others receive strand and chunks (NCCL broadcast)
    prep = None
    if rank == 0:
        st, prep = make_workload(args.config, args.scale_n)
        n1 = len(prep.strand)
        chunks = [tuple(c) for c in prep.chunks]
    else:
        st = ab.RunSettings(**CONFIG_FLAGS[args.config])
        n1, chunks = 0, None
    if dist is not None:
        box = [n1, chunks]
        dist.broadcast_object_list(box, src=0, device=dev)
        n1, chunks = box
    bp = int(sum(c[1] for c in chunks))
    pinned = torch.empty(n1, dtype=torch.uint8).pin_memory()
    if rank == 0:
        pinned.numpy()[:] = prep.strand
    if dist is not None:
        d_strand = pinned.to(dev) if rank == 0 else torch.empty(n1, dtype=torch.uint8, device=dev)
        dist.broadcast(d_strand, src=0)
        if rank != 0:
            pinned.copy_(d_strand)
        del d_strand
        torch.cuda.empty_cache()
    ctx = ab.Context(local)
    if args.index_bits:
        ctx.set_index_bits(args.index_bits)
    if dist is not None:
        from asgart_b200.dist import join_index_group
        join_index_group(ctx, dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()

    def search(post=ab.POST_ALL):
        if dist is None:
            return ctx.search(chunks, st, post)
        from asgart_b200.dist import sharded_search
        return sharded_search(ctx, chunks, st, post, dev)

    def step_resident():
        ctx.build_index()
        return search()

    def step_e2e():
        ctx.load_strand_ptr(pinned.data_ptr(), n1)
        ctx.build_index()
        return search()

    def timed(fn, steps):
        barrier()
        ctx.timer_start()
        t0 = time.perf_counter()
        fam = None
        for _ in range(steps):
            fam = fn()
        ms = ctx.timer_stop()
        barrier()
        wall = (time.perf_counter() - t0) * 1e3
        if dist is not None:
            t = torch.tensor([ms, wall], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall = float(t[0]), float(t[1])
        return ms, wall, fam

    # ---- device-resident value
    ctx.load_strand_ptr(pinned.data_ptr(), n1)
    for _ in range(args.warmup):
        step_resident()
    ctx.reset_stats()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms, wall, fam = timed(step_resident, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    stats = ctx.stats()
    if args.dump_outputs and rank == 0:
        dump_families(args.dump_outputs, fam)
    # ---- end to end through the C ABI with host buffers
    for _ in range(min(args.warmup, 3)):
        step_e2e()
    ctx.reset_stats()
    ms_e2e, wall_e2e, fam2 = timed(step_e2e, args.steps)
    stats_e2e = ctx.stats()
    assert fam2.digest() == fam.digest()
    digest = fam.digest()
    free_b, total_b = torch.cuda.mem_get_info(dev)     # the library's block cache only grows: what is in use now is the peak
    sa_bad = ctx.check_sa() if args.check_sa else None   # on-device sufcheck of this rank's copy of the index
    if dist is not None:
        t = torch.tensor([total_b - free_b, -1 if sa_bad is None else sa_bad], dtype=torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        peak_dev, sa_bad = int(t[0]), (None if int(t[1]) < 0 else int(t[1]))
    else:
        peak_dev = total_b - free_b
    g = golden(args.config) if not args.scale_n else None
    digest_ok = (digest == g["families_sha256"]) if g else None     # None: no full-size golden for this run (scaled workload)

    if rank == 0:
        peak, peak_src = peaks()
        K = args.steps
        # kernel families of the step: device ms (CUDA events on the library stream, accumulated over the K steps), launches
        # and ALGORITHMIC bytes (DESIGN.md section 4). The roofline block describes the family with the largest share.
        msd = stats["msd_levels"] > 0
        fams = {}

        def family(name, what, ms_tot, launches, nbytes):
            if launches and ms_tot > 0:
                fams[name] = {"what": what, "ms_per_step": ms_tot / K, "launches_per_step": launches / K, "ms_per_launch": ms_tot / launches,
                              "bytes_per_launch": nbytes / launches, "alg_GBps": nbytes / ms_tot / 1e6, "frac_of_hbm_peak": nbytes / ms_tot / 1e6 / peak,
                              "share_of_step": ms_tot / ms if ms else None}
        if msd:
            family("msd_local_kernel", "initial sort, finishing sort of the small buckets in shared memory (12 B read + 12 B written per suffix)",
                   stats["ms_msd_local"], stats["launches_msd_local"], stats["bytes_msd_local"])
            family("msd_scatter_kernel", "initial sort, 12-bit partition pass over (key, index) pairs, levels >= 1 (24 B per pair)",
                   stats["ms_sa_scatter_main"], stats["launches_sa_scatter_main"], stats["bytes_sa_scatter_main"])
            family("msd_scatter_kernel<text>", "initial sort, level 0: keys built from the text and partitioned (1 B read + 12 B written per suffix)",
                   stats["ms_msd_scatter0"], K, stats["bytes_msd_scatter0"])
            family("msd_hist_kernel", "initial sort, per-level digit histograms (1 B per suffix from the text, then 8 B per pair)",
                   stats["ms_msd_hist"], K * max(1, int(stats["msd_levels"])), stats["bytes_msd_hist"])
        else:
            family("rs_scatter_kernel", "initial sort (LSD form), stable 8-bit scatter pass (24 B per suffix)",
                   stats["ms_sa_scatter_main"], stats["launches_sa_scatter_main"], stats["bytes_sa_scatter_main"])
        family("probe_search_kernel", "k-mer probe search: LUT narrow + lock-step equal range + filters (SURVEY 8d gather bytes)",
               stats["ms_probe"], stats["launches_probe"], stats["bytes_probe"])
        family("gather_rank_kernel", "prefix doubling: rank[i + D] gathers (12 B per unsorted suffix and round)",
               stats["ms_sa_gather"], stats["launches_sa_gather"], stats["bytes_sa_gather"])
        top = max(fams, key=lambda k: fams[k]["ms_per_step"]) if fams else None
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if top and os.path.exists(tpath):
            try:
                tj_all = json.load(open(tpath))
                tj = tj_all.get("kernels", {}).get(top)
                # the capture must be of this very workload and launch pattern (same config, same launches per step)
                if tj and tj_all.get("config") == args.config and tj_all.get("strand_bp") == n1 - 1 and world == 1 \
                        and abs(tj["launches_per_step"] - fams[top]["launches_per_step"]) < 0.5:
                    traffic = tj["dram_bytes_per_launch"]
            except Exception:
                traffic = None
        roof = {"kernel": None, "bound": "hbm", "achieved": 0.0, "peak": peak, "unit": "GB/s", "frac": None, "traffic": None}
        if top:
            f = fams[top]
            roof = {"kernel": f"{top} ({f['what']})", "bound": "hbm", "achieved": f["alg_GBps"], "peak": peak, "unit": "GB/s",
                    "frac": f["frac_of_hbm_peak"], "traffic": traffic, "peak_source": peak_src, "bytes_per_launch": f["bytes_per_launch"],
                    "ms_per_launch": f["ms_per_launch"], "launches_per_step": f["launches_per_step"], "share_of_step": f["share_of_step"],
                    "note": ("largest share of the step among the kernel families (kernel_families lists all of them); msd_local_kernel works in "
                             "shared memory and is bound by instruction issue, not by HBM (profiles/r2_ncu_full_msd_v1.summary.txt)")}
        line = {
            "metric": METRIC, "value": bp * K / (ms * 1e-3), "unit": "bp/s", "n_gpus": world, "steps": K, "warmup": args.warmup,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u%d" % int(stats["sa_index_bits"]), "data": "synthetic",
            "config": workload_config(args.config, args.scale_n, st, n1 - 1, bp, len(chunks)),
            "parallelism": (f"index built by {world} GPUs together (suffix ranges by key, rank array in peer memory), "
                            f"then replicated; probe range x{world}" if world > 1 else "one GPU"),
            "timing": "CUDA events on the library stream around the K-step loop; wall clock agrees within ms_per_step_wall",
            "ms_per_step_wall": wall / K,
            "families_sha256": digest, "families_match_oracle_golden": digest_ok,
            "device_bytes_peak": peak_dev, "sa_check_violations": sa_bad,
            "clocks": clocks,
            "e2e": {"value": bp * K / (ms_e2e * 1e-3), "unit": "bp/s", "ms_per_step": ms_e2e / K,
                    "h2d_bytes_per_step": stats_e2e["h2d_bytes"] // K, "d2h_bytes_per_step": stats_e2e["d2h_bytes"] // K},
            "gpu_launches": int(stats["launches_total"]),
            "roofline": roof,
            "kernel_families": fams,
            "initial_sort": {"form": "msd" if msd else "lsd", "levels": int(stats["msd_levels"]), "ms_per_step": stats["ms_sa_sort"] / K},
            "phases_ms_per_step": {k: stats[k] / K for k in ("ms_sa_build", "ms_lut", "ms_search", "ms_automaton", "ms_post", "ms_d2h")},
            "counters_per_step": {k: stats[k] // K for k in ("n_probes", "n_searched", "n_skipped_n", "n_skipped_card", "n_matches")}
                                 | {"sa_rounds": stats["sa_rounds"], "families": fam.n_families, "duplicons": len(fam.sds)},
        }
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            full = n1 - 1
            sample_n = min(full, REF_SAMPLE_BP)
            # the CPU side gets its strand, fragment map and chunk list from the oracle's prepare_data, not from our library
            st2, prep2 = oracle_workload(args.config, args.scale_n if sample_n == full else sample_n)
            s_strand, s_chunks, s_bp = prep2.strand, prep2.chunks, searched_bp(prep2)
            r = cpu_reference_pass(s_strand, s_chunks, st, cores)
            line["cpu_baseline"] = {
                "value": s_bp / r["seconds"], "unit": "bp/s", "cores": cores, "kind": r["sa_kind"],
                "sample": (f"{'whole workload' if sample_n == full else 'scaled workload'}: {len(s_strand) - 1} bp, one pass; SA by the "
                           f"reference's libdivsufsort64 (1 thread, as build.rs builds it) + oracle port of the Rust probe "
                           f"loop/automaton/post-steps on {cores} threads over {len(s_chunks)} chunks (no rustc in this image)"),
                "phases_s": {k: round(v, 3) for k, v in r.items() if k.endswith("_s")}, "families": r["families"],
                "sample_bp": len(s_strand) - 1, "full_bp": full}
            if sample_n == full:    # same input on both sides: the digests must agree
                line["cpu_baseline"]["families_sha256"] = r["families_sha256"]
                line["cpu_baseline"]["families_match_gpu"] = r["families_sha256"] == digest
            if g:
                sec = g["oracle_seconds"]
                tot = sec["sa_divsufsort64_1thread"] + sec["lut"] + sec["search_automaton"] + sec["post"]
                line["cpu_baseline"]["offline_full_config"] = {
                    "seconds": round(tot, 2), "bp_per_s": g["searched_bp"] / tot, "cores": sec["threads"],
                    "source": f"tests/golden/families_c{args.config}.json (the whole config, run offline on the CPU container)"}
        try:    # the output side next to the path (SURVEY 8d: FASTA parse and JSON write are reported separately)
            t0 = time.perf_counter()
            js = prep.to_json(st, fam)
            line["json_write"] = {"ms": (time.perf_counter() - t0) * 1e3, "bytes": len(js), "where": "host (serde_json pretty layout, exporters.rs:12-25)"}
        except Exception as e:   # never lose the bench line over the report
            line["json_write"] = {"error": str(e)}
        if world == 1 and not args.no_ingest:
            line["ingest"] = measure_ingest(ctx, prep, peak)
        print(json.dumps(line), flush=True)
    if dist is not None:
        ctx.dist_shutdown()
    ctx.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", type=int, default=4, choices=[1, 2, 3, 4, 5])
    ap.add_argument("--scale-n", type=int, default=0, help="override the config's genome length (bp)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--index-bits", type=int, default=0, choices=[0, 32, 64], help="force the suffix-index width (0 = auto)")
    ap.add_argument("--check-sa", action="store_true", help="run the on-device sufcheck on every rank's index after the timed steps")
    ap.add_argument("--ref-sample-bp", type=int, default=0, help="--impl reference: genome length per step (0 = bounded default)")
    ap.add_argument("--no-ingest", action="store_true", help="skip the FASTA-ingest measurement (N=1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the families of the last step as DIR/<field>.npy, to compare two "
                         "builds of this project output for output (--impl ours only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what --impl ours computes")
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.warmup < 3:
            args.warmup = 3
        run_ours(args)


if __name__ == "__main__":
    main()
