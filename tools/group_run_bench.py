"""Wall-clock of a whole multi-device run: python tools/group_run_bench.py [--config 4] [--scale-n N] [--ns 1,2,4,8]
Writes the synthetic config as a 60-column multiFASTA (one record per fragment) to a temporary directory, then times
asgart_b200_run_files_devices (ingest on member 0, strand copies, group build, group search, JSON) on devices
0..N-1 for every N the machine has GPUs for, `--reps` times each. One JSON line per N: the wall times, the sha256 of the
JSON text (equal for every N), and the peak device memory of each GPU above what was in use before the run (sampled
with cudaMemGetInfo every few ms while the run is in flight; the library's block cache only grows until its contexts
are destroyed, so the last samples before the end hold the peak). The card name and power limit come with every line."""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import asgart_b200 as ab  # noqa: E402
from asgart_b200 import _lib  # noqa: E402
from tools.ingest_bench import fasta_bytes  # noqa: E402

CONFIG_FLAGS = {2: dict(reverse=True, complement=True, skip_masked=True), 3: dict(reverse=True, complement=True),
                4: dict(reverse=True, complement=True)}


def card_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout
        return [dict(zip(("index", "name", "power_limit", "max_sm_clock"), (x.strip() for x in line.split(","))))
                for line in out.strip().splitlines()]
    except (OSError, subprocess.TimeoutExpired):
        return []


class PeakSampler:
    """Largest (total - free) device memory of each GPU while the sampler runs, minus what was in use at its start."""

    def __init__(self, devices):
        import torch
        self.torch = torch
        self.devices = sorted(set(devices))
        self.base = {d: self.used(d) for d in self.devices}
        self.peak = dict(self.base)
        self.stop = threading.Event()
        self.thread = threading.Thread(target=self.loop, daemon=True)

    def used(self, d):
        free, total = self.torch.cuda.mem_get_info(d)
        return total - free

    def loop(self):
        while not self.stop.is_set():
            for d in self.devices:
                self.peak[d] = max(self.peak[d], self.used(d))
            time.sleep(0.002)

    def __enter__(self):
        self.thread.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.thread.join()

    def result(self):
        return {str(d): self.peak[d] - self.base[d] for d in self.devices}


def run(path, st, devices):
    L = _lib.load()
    arr = (_lib.Settings * 1)(st.to_c())
    dev = (C.c_int32 * len(devices))(*devices)
    err = C.c_char_p()
    t0 = time.perf_counter()
    p = L.asgart_b200_run_files_devices(path.encode(), arr, 1, dev, len(devices), None, C.byref(err))
    wall = time.perf_counter() - t0
    if not p:
        raise RuntimeError(err.value.decode() if err.value else "run failed")
    try:
        js = C.string_at(p)
    finally:
        L.asgart_b200_free_string(p)
    return wall, hashlib.sha256(js).hexdigest(), len(js)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=4, choices=sorted(CONFIG_FLAGS))
    ap.add_argument("--scale-n", type=int, default=0, help="override the config's genome length (bp)")
    ap.add_argument("--ns", default="1,2,4,8", help="member counts; those above the GPU count are reported as not measured")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--dir", default=tempfile.gettempdir(), help="where the FASTA file is written (removed at the end)")
    ap.add_argument("--out", default="", help="append the JSON lines to this file too")
    args = ap.parse_args()
    import torch
    n_gpus = torch.cuda.device_count()
    if n_gpus < 1:
        sys.exit("group_run_bench: no CUDA device")
    st = ab.RunSettings(**CONFIG_FLAGS[args.config])
    g, fr = ab.synth_genome(args.config, scale_n=args.scale_n, threads=os.cpu_count() or 8)
    fd, path = tempfile.mkstemp(suffix=f"_c{args.config}.fa", dir=args.dir)
    os.close(fd)
    try:
        fasta_bytes(g, fr).tofile(path)
        bp = len(g)
        del g
        cards = card_info()
        for n in (int(x) for x in args.ns.split(",")):
            line = {"tool": "group_run_bench", "config": args.config, "bp": bp, "settings": CONFIG_FLAGS[args.config], "n": n,
                    "cards": cards[:max(n, 1)]}
            if n > n_gpus:
                line["result"] = f"not measured: the machine has {n_gpus} GPU(s)"
            else:
                devices = list(range(n))
                walls, shas, peaks = [], set(), []
                for _ in range(args.reps):
                    with PeakSampler(devices) as ps:
                        wall, sha, nbytes = run(path, st, devices)
                    walls.append(round(wall, 3))
                    shas.add(sha)
                    peaks.append(ps.result())
                line.update(wall_s=walls, json_sha256=sorted(shas), json_bytes=nbytes,
                            device_bytes_peak={d: max(p[d] for p in peaks) for d in peaks[0]})
            print(json.dumps(line), flush=True)
            if args.out:
                with open(args.out, "a") as f:
                    f.write(json.dumps(line) + "\n")
    finally:
        os.unlink(path)


if __name__ == "__main__":
    main()
