#!/usr/bin/env python
"""bench.py -- BWT build throughput (Mbp/s) of the deBWT hot path on B200, next to the CPU reference.

Contract (one JSON line on stdout, printed by rank 0):
  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3] [--dump-outputs DIR]
  N > 1 is launched by the driver through torch.distributed.run (one rank per GPU).

Default workload: BASELINE.json configs[2], the 3.1 Gbp human-genome-sized sequence with interspersed repeat families
(24 records) -- the configuration the metric's north star is quoted on and the largest that fits one GPU.  The genome is
generated in HBM (debwt_b200/synth_gpu.py, bit-identical to the numpy generators of debwt_b200/synth.py).

A "step" is one pass of the whole hot path (2-bit pack -> 32-mer extraction -> LSD radix sort -> branch k-mer
detection -> branch codes -> segmented sort -> BWT emission) over the genome.
  value : input bases / device time, text already resident in HBM (CUDA events on the library's stream)
  e2e   : same metric through the public C-ABI call sequence with HOST buffers: pinned host text -> H2D -> build ->
          D2H of the packed BWT, every step
  roofline : the dominant kernel (onesweep_kernel, the radix-sort scatter pass): 16 B/key algorithmic per launch /
          mean launch time (CUDA events on the library's stream), against the measured HBM copy bandwidth
  cpu_baseline : the compiled reference (oracle/_ref/deBWT + Jellyfish stand-in) on a bounded prefix of the workload
  verify : outside the timed regions -- SHA-256 of the packed BWT against the committed value
          (tests/golden/workload_sha.json) and the GPU LF-inversion verifier (debwt_verify_*: the BWT inverted by
          its LF mapping must reproduce the input text)
--impl reference times the reference's own CPU implementation on a bounded prefix of the same workload.
--dump-outputs DIR writes the BWT of the last timed step (a seeded sample of its rows) to DIR; the workloads are seeded,
so two builds of the project run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "bwt_build_throughput"
UNIT = "Mbp/s"


# ------------------------------------------------------------------------------------------------
# workloads (BASELINE.json configs; SURVEY.md section 8d)
# ------------------------------------------------------------------------------------------------
class Workload:
    def __init__(self, name, desc, n_bases, n_records, device_text, host_prefix):
        self.name, self.desc, self.n_bases, self.n_records = name, desc, n_bases, n_records
        self.device_text = device_text      # (device ordinal) -> (torch.uint8 CUDA tensor holding T, seps np.uint64)
        self.host_prefix = host_prefix      # (max_bases) -> list of numpy records: a bounded prefix of the workload, on the CPU


def _host_text_to_device(records, device):
    import torch
    from debwt_b200 import api
    text, seps = api.join_records(records)
    return torch.from_numpy(text).to(torch.device("cuda", device)), seps


def _cut(records, max_bases):
    out, left = [], max_bases
    for r in records:
        if left <= 33:
            break
        out.append(r[:left])
        left -= out[-1].size
    return out


def workload(name: str) -> Workload:
    from debwt_b200 import synth

    def gpu(fn):
        def run(device):
            from debwt_b200 import synth_gpu
            return fn(synth_gpu, device)
        return run

    def c3_like(n, nrec, label):
        per = -(-n // nrec)
        return Workload(name, label, n, nrec, gpu(lambda g, d: g.config3(n, nrec, device=d)),
                        lambda m: _cut([synth.genome_like_prefix(n, 5, min(m, per))], m))

    def c4_like(base, ng, label):
        return Workload(name, label, base * ng, ng, gpu(lambda g, d: g.config4(base, ng, device=d)),
                        lambda m: _cut([synth.genome_like_prefix(base, 9, min(m, base))], m))

    if name == "c1":
        return Workload(name, "synthetic 4.6 Mbp random ACGT single sequence, k=32", 4_600_000, 1,
                        lambda d: _host_text_to_device(synth.config1(), d), lambda m: _cut(synth.config1(), m))
    if name == "c2":
        return Workload(name, "synthetic 100 Mbp sequence with planted repeats (5% copies of 10 kbp elements), k=32", 100_000_000, 1,
                        lambda d: _host_text_to_device(synth.config2(), d), lambda m: _cut(synth.config2(), m))
    if name == "c2s":
        return Workload(name, "synthetic 20 Mbp sequence with planted repeats (reduced C2, smoke only)", 20_000_000, 1,
                        lambda d: _host_text_to_device(synth.config2(20_000_000), d), lambda m: _cut(synth.config2(20_000_000), m))
    if name == "c3":
        return c3_like(3_100_000_000, 24, "synthetic 3.1 Gbp human-genome-sized sequence with interspersed repeat families "
                                          "(24 records), k=32")
    if name == "c3s":
        return c3_like(400_000_000, 4, "synthetic 400 Mbp genome with repeat families (reduced C3)")
    if name == "c4":
        return c4_like(300_000_000, 10, "collection of 10 synthetic 300 Mbp genomes at 0.1% SNP divergence (3 Gbp), k=32")
    if name == "c4s":
        return c4_like(10_000_000, 10, "10 synthetic 10 Mbp genomes at 0.1% divergence (reduced C4)")
    raise SystemExit(f"unknown workload {name}")


def common_config(w: Workload, world: int) -> dict:
    """identical in both arms (the driver compares the `config` objects)"""
    return {"workload": w.desc, "n_bases": w.n_bases, "n_records": w.n_records, "k": 32,
            "l2": "inputs larger than L2 (every step streams the whole text and key arrays through HBM)",
            "parallelism": "single GPU" if world == 1 else
                           "position split x%d, keys range-partitioned by sampled splitters, exchanged over NVLink" % world}


def expected_sha(name: str):
    p = os.path.join(ROOT, "tests", "golden", "workload_sha.json")
    try:
        return json.load(open(p)).get(name)
    except (OSError, ValueError):
        return None


DUMP_ROWS = 1 << 22     # BWT rows sampled by --dump-outputs: 12 B each (float64 row + float32 code), 48 MB at most


def dump_outputs(out_dir: str, words, sharp, dollar, n_rows: int) -> dict:
    """Writes the BWT a caller receives (packed words, '#' rows, '$' row) as float arrays that two builds can be
    compared with, output for output:
      sharp_rows.npy, dollar_row.npy : float64, every row (exact: rows < 2^53)
      bwt_rows.npy, bwt_codes.npy    : float64 row numbers and float32 symbol codes (0-3 = A,C,G,T, 4 = '#', 5 = '$') of
                                       DUMP_ROWS rows, one seeded pick from each of DUMP_ROWS equal slices of the BWT (all
                                       rows when there are fewer)"""
    import numpy as np
    words = np.asarray(words).view(np.uint64)
    if n_rows <= DUMP_ROWS:
        rows = np.arange(n_rows, dtype=np.uint64)
    else:
        edges = np.arange(DUMP_ROWS + 1, dtype=np.uint64) * np.uint64(n_rows) // np.uint64(DUMP_ROWS)
        rows = np.random.default_rng(20261020).integers(edges[:-1], edges[1:], dtype=np.uint64)
    codes = (words[rows >> np.uint64(5)] >> (np.uint64(62) - np.uint64(2) * (rows & np.uint64(31)))) & np.uint64(3)
    codes[np.isin(rows, sharp)] = 4
    codes[rows == np.uint64(dollar[0])] = 5
    arrays = {"sharp_rows": np.asarray(sharp).astype(np.float64), "dollar_row": np.asarray(dollar).astype(np.float64),
              "bwt_rows": rows.astype(np.float64), "bwt_codes": codes.astype(np.float32)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return {"dir": out_dir, "rows_sampled": int(rows.size), "rows": n_rows}


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock and throttle reasons DURING the timed region through NVML (in-process: spawning
    nvidia-smi in a loop perturbs the driver enough to slow the measured kernels down)."""

    def __init__(self, index: int, period_s: float = 0.02):
        self.index, self.period, self.rows, self.stop, self.thr, self.h = index, period_s, [], threading.Event(), None, None
        self.nv = None

    def __enter__(self):
        if os.environ.get("DEBWT_NO_CLOCKS"):
            return self
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)   # slow call: once, up front
            self.thr = threading.Thread(target=self._run, daemon=True)
            self.thr.start()
        except Exception:  # noqa: BLE001
            self.nv = None
        return self

    def _run(self):
        nv = self.nv
        while not self.stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                mx = self.max_mhz
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((sm, mx, rs))
            except Exception:  # noqa: BLE001
                pass
            self.stop.wait(self.period)

    def __exit__(self, *a):
        self.stop.set()
        if self.thr:
            self.thr.join(timeout=2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        reasons = sorted(k for k, bit in names.items() if any(r[2] & bit for r in self.rows))
        return {"sm_mhz": statistics.median(r[0] for r in self.rows), "sm_max_mhz": max(r[1] for r in self.rows),
                "reasons": reasons, "samples": len(self.rows)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except (KeyError, ValueError):
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(nk: int):
    """dram bytes of one onesweep launch from the committed `ncu --set full` capture (profiles/): the capture's own
    figure when it was taken at this key count, else scaled per key (and said so)"""
    for fn in ("r02_onesweep_traffic.json", "onesweep_traffic.json"):
        p = os.path.join(ROOT, "profiles", fn)
        if os.path.isfile(p):
            try:
                t = json.load(open(p))
            except ValueError:
                continue
            per_key = t.get("dram_bytes_per_key")
            if not per_key:
                continue
            exact = t.get("n_keys") == nk
            return per_key * nk, ("ncu capture at this size (profiles/%s)" % fn) if exact else \
                ("ncu capture at %s keys (profiles/%s: %.2f B/key), scaled to this launch" % (t.get("n_keys"), fn, per_key))
    return None, None


def roofline_block(nk, sweeps_per_step, per_launch_ms, sort_ms, text_bytes, who):
    peak, peak_src = measured_peak()
    achieved = 16.0 * nk / (per_launch_ms * 1e-3) / 1e9 if per_launch_ms > 0 else 0.0
    traffic, traffic_src = ncu_traffic(nk)
    phase = {}
    if sort_ms > 0:
        survey = 136.0 * nk / (sort_ms * 1e-3) / 1e9                    # SURVEY.md 8d: 8 B histogram sweep + 8 x 16 B
        moved = (128.0 * nk + text_bytes) / (sort_ms * 1e-3) / 1e9      # what moves: the histograms come from the packed text
        phase = {"ms": sort_ms, "survey_formula": {"bytes_per_key": 136, "achieved": survey, "frac": survey / peak},
                 "moved_bytes": {"bytes_per_key": 128 + text_bytes / max(nk, 1), "achieved": moved, "frac": moved / peak}}
    return {"bound": "hbm", "kernel": "onesweep_kernel (radix-sort scatter pass%s, %d launches/step)" % (who, sweeps_per_step),
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "frac_of_nominal_8000": achieved / 8000.0,
            "peak_source": peak_src, "algorithmic_bytes_per_launch": 16 * nk, "mean_launch_ms": per_launch_ms,
            "traffic": traffic, "traffic_source": traffic_src, "sort_phase": phase}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline
# ------------------------------------------------------------------------------------------------
def run_reference_sample(w: Workload, max_bases: int, threads: int):
    from debwt_b200 import synth
    from oracle import refrun
    if not refrun.available():
        raise RuntimeError("oracle/_ref is not built")
    sample = w.host_prefix(max_bases)
    nb = int(sum(r.size for r in sample))
    with tempfile.TemporaryDirectory() as d:
        fa = os.path.join(d, "sample.fa")
        synth.write_fasta(sample, fa)
        res = refrun.run_reference(fa, threads=threads, timeout=3600, scratch_root=d)
    return nb, res


def cpu_baseline_block(w: Workload, sample_bases: int):
    cores = os.cpu_count() or 1
    try:
        nb, res = run_reference_sample(w, sample_bases, cores)
        return {"value": nb / res.wall_s / 1e6, "unit": UNIT, "cores": cores, "kind": "reference", "same_input": nb == w.n_bases,
                "sample": f"oracle/_ref/deBWT -t {cores} -k 32 on the first {nb} bases of the workload ({w.n_bases} in all): "
                          f"{res.wall_s:.2f} s wall of which {res.standin_s:.2f} s in the Jellyfish stand-in "
                          f"(deBWT proper {nb / max(res.proper_s, 1e-9) / 1e6:.2f} Mbp/s)"}
    except Exception as e:  # noqa: BLE001
        return {"value": None, "unit": UNIT, "cores": cores, "kind": "reference", "sample": f"failed: {e}"}


def reference_arm(args, rank, world):
    """The reference's own CPU implementation (oracle/_ref/deBWT, all host threads) on a bounded prefix of the same
    workload, sized so that steps + warmup runs end within a few minutes."""
    if rank != 0:
        return
    w = workload(args.workload)
    cores = os.cpu_count() or 1
    runs = max(args.steps + args.warmup, 1)
    per_run_s = 170.0 / runs                                  # whole arm within ~3 minutes
    sample = int(min(w.n_bases, max(2_000_000, (per_run_s - 3.0) * 1.0e6)))   # ~1 Mbp/s + ~3 s fixed cost per run
    if args.ref_sample:
        sample = min(w.n_bases, args.ref_sample)
    times, standin = [], []
    nb = sample
    for i in range(runs):
        nb, res = run_reference_sample(w, sample, cores)
        if i >= args.warmup:
            times.append(res.wall_s); standin.append(res.standin_s)
    t = sum(times) / len(times)
    v = nb / t / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
            "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": common_config(w, world),
            "same_input": nb == w.n_bases,
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "reference", "same_input": nb == w.n_bases,
                             "sample": f"oracle/_ref/deBWT -t {cores} -k 32 on the first {nb} bases of the workload per step "
                                       f"({w.n_bases} in all; the reference needs ~16 B of RAM and ~36 B of temp files per distinct "
                                       f"32-mer); Jellyfish replaced by oracle/jellyfish_standin.c "
                                       f"({sum(standin) / len(standin):.2f} s of the {t:.2f} s per step)"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# file to file (SURVEY.md 8d "also report file-to-file")
# ------------------------------------------------------------------------------------------------
def file_to_file(h_text_np, seps, n_bases, device, expect_sha):
    """host/deBWT -o out in.fa: FASTA file -> the reference's three output files, wall clock of the whole process"""
    import numpy as np
    from debwt_b200 import synth
    exe = os.path.join(ROOT, "host", "deBWT")
    if not os.path.isfile(exe):
        return {"value": None, "note": "host/deBWT is not built"}
    root = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    with tempfile.TemporaryDirectory(dir=root) as d:
        fa, out = os.path.join(d, "w.fa"), os.path.join(d, "w.bwt")
        start, recs = 0, []
        for s in seps.tolist():
            recs.append(h_text_np[start:int(s)])
            start = int(s) + 1
        synth.write_fasta(recs, fa)
        fa_bytes = os.path.getsize(fa)
        t0 = time.perf_counter()
        r = subprocess.run([exe, "-o", out, "-g", str(device), fa], capture_output=True, text=True)
        wall = time.perf_counter() - t0
        if r.returncode != 0:
            return {"value": None, "note": "host/deBWT failed: " + r.stderr[-300:]}
        h = hashlib.sha256()
        with open(out, "rb") as f:
            for blk in iter(lambda: f.read(1 << 24), b""):
                h.update(blk)
        sha = h.hexdigest()
    return {"value": n_bases / wall / 1e6, "unit": UNIT, "wall_s": wall, "fasta_bytes": fa_bytes, "where": root or "tmp",
            "what": "host/deBWT -o out in.fa, whole process: create context, read + parse FASTA, H2D, build, D2H, write the three files",
            "bwt_sha256": sha, "sha_ok": (sha == expect_sha) if expect_sha else None, "stderr_tail": r.stderr.strip().splitlines()[-2:]}


# ------------------------------------------------------------------------------------------------
# our arm, one GPU
# ------------------------------------------------------------------------------------------------
def ours(args, rank, world, local_rank):
    import numpy as np
    import torch
    from debwt_b200 import api, binding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    w = workload(args.workload)
    t_gen = time.perf_counter()
    d_text, seps = w.device_text(local_rank)
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t_gen
    n = int(d_text.numel())
    n_bases = n - len(seps)
    assert n_bases == w.n_bases, (n_bases, w.n_bases)
    # pinned host staging for the end-to-end leg
    h_text = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    h_text.copy_(d_text)
    n_words = (n + 31) // 32
    h_out = torch.empty(n_words, dtype=torch.int64, pin_memory=True)
    torch.cuda.synchronize()

    b = api.BwtBuilder(device=local_rank, sort_config=args.sort_cfg, blue_grouping=int(os.environ.get("DEBWT_BLUE", "0")))

    def step_resident():
        b.set_text_device(d_text.data_ptr(), n, seps)
        b.build()
        return b.stats()

    def step_e2e():
        b.set_text_ptr(h_text.data_ptr(), n, seps)
        b.build()
        return b.result_into(h_out.data_ptr())

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step_resident()
    torch.cuda.synchronize()
    l0 = binding.lib().debwt_launch_count()
    with ClockSampler(local_rank) as clk:
        t0 = time.perf_counter()
        dev_ms, sort_ms, sweep_ms, sweeps, last = 0.0, 0.0, 0.0, 0, None
        for _ in range(args.steps):
            st = step_resident()
            dev_ms += st["ms_total"]; sort_ms += st["ms_sort"]; sweep_ms += st["ms_sort_sweeps"]; sweeps += st["sort_sweeps"]
            last = st
        torch.cuda.synchronize()
        wall_step = (time.perf_counter() - t0) * 1e3 / args.steps
    launches = int(binding.lib().debwt_launch_count() - l0)
    clocks = clk.summary()
    ms_dev = dev_ms / args.steps
    dumped = None
    if args.dump_outputs:                                 # before the e2e leg reuses h_out
        sharp, dollar = b.result_into(h_out.data_ptr())
        dumped = dump_outputs(args.dump_outputs, h_out.numpy(), sharp, dollar, n)

    for _ in range(2):
        step_e2e()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        sharp, dollar = step_e2e()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    e2e_stats = b.stats()

    # ---- verification, outside the timed regions ----
    sha = hashlib.sha256(h_out.numpy().tobytes()).hexdigest()
    want = expected_sha(w.name)
    verify = {"bwt_sha256": sha, "sha_expected": want, "sha_ok": (sha == want) if want else None}
    if not args.no_verify:
        try:
            bad, vms = b.verify(device_ptr=d_text.data_ptr(), n_symbols=n)
            verify.update({"lf_inversion_bad_rows": bad, "lf_inversion_ms": vms, "lf_inversion_ok": bad == 0,
                           "how": "debwt_verify_text_device: occ/C tables + LF mapping of the result on the GPU, list ranking by "
                                  "pointer jumping, every row's symbol compared with the input text"})
        except Exception as e:  # noqa: BLE001
            verify.update({"lf_inversion_ok": None, "lf_inversion_error": str(e)})
    nk = last["n_keys"]
    line = {
        "metric": METRIC, "value": n_bases / (ms_dev * 1e-3) / 1e6, "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": warm, "ms_per_step": ms_dev, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic (generated in HBM in %.2f s)" % t_gen,
        "config": common_config(w, world),
        "timing": "CUDA events on the library stream (debwt_stats.ms_total); wall per step %.3f ms" % wall_step,
        "clocks": clocks,
        "e2e": {"value": n_bases / (e2e_ms * 1e-3) / 1e6, "unit": UNIT, "h2d_bytes_per_step": n,
                "d2h_bytes_per_step": 8 * n_words + 8 * len(seps), "ms_per_step": e2e_ms,
                "ms_h2d": e2e_stats["ms_h2d"], "ms_build": e2e_stats["ms_total"], "ms_d2h": e2e_stats["ms_d2h"]},
        "gpu_launches": launches,
        "roofline": roofline_block(nk, sweeps // args.steps, sweep_ms / max(sweeps, 1), sort_ms / args.steps, n / 4.0, ""),
        "phases_ms": {k: last[k] for k in last if k.startswith("ms_")},
        "sizes": {k: last[k] for k in ("n_symbols", "n_keys", "n_branch", "n_blue", "n_codes", "n_special")},
        "hbm": {"arena_bytes": last["arena_bytes"], "arena_used_bytes": last["arena_used_bytes"],
                "bytes_per_base": last["arena_bytes"] / max(n_bases, 1)},
        "verify": verify,
        "bwt_sha256": sha,
    }
    if dumped:
        line["dump_outputs"] = dumped
    b.close()
    if not args.no_file_to_file:
        try:
            line["file_to_file"] = file_to_file(h_text.numpy(), seps, n_bases, local_rank, want or sha)
        except Exception as e:  # noqa: BLE001
            line["file_to_file"] = {"value": None, "note": f"failed: {e}"}
    if not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_block(w, args.cpu_sample)
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# our arm, N GPUs
# ------------------------------------------------------------------------------------------------
def ours_sharded_python(args, rank, world, local_rank):
    """(--orchestrator python: debwt_b200/dist.py, the CPU-testable harness)  N GPUs, one process per GPU: the text is split by position, keys are range-partitioned by sampled splitters and
    exchanged over NVLink (debwt_b200/dist.py).  Strong scaling: the same genome on N GPUs."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from debwt_b200 import api, binding, dist as D

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    comm = D.Comm()
    ops = D.CudaOps(local_rank, sort_cfg=args.sort_cfg or 8)
    ops.timed_main_sort = True
    w = workload(args.workload)
    t_gen = time.perf_counter()
    d_full, seps = w.device_text(local_rank)          # every rank generates the genome in its own HBM (milliseconds)
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t_gen
    n = int(d_full.numel())
    n_bases = n - len(seps)
    lo, hi = D.my_slice(n, comm)
    d_slice = d_full[lo:hi].clone() if hi > lo else torch.zeros(1, dtype=torch.uint8, device=d_full.device)
    if rank != 0 or args.no_verify:
        del d_full
        d_full = None
    h_slice = torch.empty(max(hi - lo, 1), dtype=torch.uint8, pin_memory=True)
    h_slice[:d_slice.numel()].copy_(d_slice)
    n_words = (n + 31) // 32
    h_out = torch.empty(n_words, dtype=torch.int64, pin_memory=True) if rank == 0 else None
    torch.cuda.empty_cache()

    def barrier():
        comm.barrier()
        torch.cuda.synchronize()

    stats = {}
    out = [None]

    def step(resident: bool):
        src = d_slice if resident else h_slice.to("cuda", non_blocking=True)
        out[0] = D.build_sharded(None, seps, comm, ops, stats, n_symbols=n, ascii_slice=src, fetch=False)
        if not resident and rank == 0:
            h_out.copy_(out[0][0], non_blocking=True)
        torch.cuda.synchronize()

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step(True)
    barrier()
    l0 = binding.lib().debwt_launch_count()
    sent0 = comm.bytes_sent
    sort_ms = sweep_ms = 0.0
    sweeps = 0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        t0 = time.perf_counter()
        ev0.record()
        for _ in range(args.steps):
            step(True)
            sort_ms += ops.sort_stats["ms"]; sweep_ms += ops.sort_stats["ms_sweeps"]; sweeps += ops.sort_stats["sweeps"]
        ev1.record()
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    dev_ms = ev0.elapsed_time(ev1) / args.steps
    launches = int(binding.lib().debwt_launch_count() - l0)
    sent_per_step = (comm.bytes_sent - sent0) / args.steps
    clocks = clk.summary()
    for _ in range(2):
        step(False)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step(False)
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    tt = torch.tensor([dev_ms, e2e_ms, wall_ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, wall_ms = (float(x) for x in tt.tolist())
    phases = None
    if args.profile_phases:                              # one extra, synchronised step: per-phase wall times on rank 0 (not a timing run)
        stats["profile"] = True
        step(True)
        phases = stats.get("phases_ms")
        stats["profile"] = False
    if rank == 0:
        sha = hashlib.sha256(h_out.numpy().tobytes()).hexdigest()
        want = expected_sha(w.name)
        verify = {"bwt_sha256": sha, "sha_expected": want, "sha_ok": (sha == want) if want else None}
        if not args.no_verify:
            try:
                bwt_t, sharp_t, dollar_t = out[0]
                sharp_np = sharp_t.cpu().numpy().view(np.uint64)
                bad, vms = api.verify_bwt_device(bwt_t.data_ptr(), n, sharp_np, int(dollar_t.cpu().numpy().view(np.uint64)[0]),
                                                 d_full.data_ptr(), device=local_rank)
                verify.update({"lf_inversion_bad_rows": bad, "lf_inversion_ms": vms, "lf_inversion_ok": bad == 0,
                               "how": "debwt_verify_bwt_device on rank 0: LF mapping of the stitched result, list ranking by pointer "
                                      "jumping, every row's symbol compared with the input text"})
            except Exception as e:  # noqa: BLE001
                verify.update({"lf_inversion_ok": None, "lf_inversion_error": str(e)})
        nk_loc = ops.sort_stats["n"]
        line = {
            "metric": METRIC, "value": n_bases / (dev_ms * 1e-3) / 1e6, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": dev_ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic (generated in HBM on every rank in %.2f s)" % t_gen,
            "config": common_config(w, world),
            "timing": "CUDA events on the torch stream around the steps, max over ranks; wall per step %.3f ms" % wall_ms,
            "exchange": {"path": "CUDA-IPC peer stores fused with the bucketing (NCCL for the small collectives)"
                         if os.environ.get("DEBWT_P2P", "1") != "0" and world > 1 else "torch.distributed all_to_all",
                         "keys_per_gpu": stats.get("keys_local"), "bytes_sent_rank0_per_step": sent_per_step},
            "clocks": clocks,
            "e2e": {"value": n_bases / (e2e_ms * 1e-3) / 1e6, "unit": UNIT, "h2d_bytes_per_step": n, "d2h_bytes_per_step": 8 * n_words,
                    "ms_per_step": e2e_ms},
            "gpu_launches": launches,
            "roofline": roofline_block(nk_loc, sweeps // max(args.steps, 1), sweep_ms / max(sweeps, 1), sort_ms / args.steps, 0.0,
                                       " on rank 0's key range"),
            "sizes": {k: stats.get(k) for k in ("n_symbols", "n_keys", "n_branch", "n_blue", "n_codes")},
            "verify": verify,
            "bwt_sha256": sha,
        }
        if phases:
            line["rank0_phases_ms_synchronised"] = phases
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def ours_shard(args, rank, world, local_rank):
    """N GPUs, one process per GPU, the sharded build behind the C ABI (csrc/shard.cu: debwt_shard_*): the text is split by
    position, keys are range-partitioned by sampled splitters and stored into their owner's memory over NVLink, every rank
    emits its own BWT segment.  Strong scaling: the same genome on N GPUs.  torch.distributed (NCCL) is only the bench's own
    barrier / max-over-ranks plumbing."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from debwt_b200 import api, binding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    tag = [f"b{os.environ.get('MASTER_PORT', '0')}_{os.getpid()}_{time.time_ns() & 0xffffff}"]
    if world > 1:
        dist.broadcast_object_list(tag, src=0)
    sh = api.Shard(local_rank, rank, world, tag[0], sort_config=args.sort_cfg)
    w = workload(args.workload)
    t_gen = time.perf_counter()
    d_full, seps = w.device_text(local_rank)          # every rank generates the genome in its own HBM (milliseconds)
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t_gen
    n = int(d_full.numel())
    n_bases = n - len(seps)
    lo, hi = sh.slice(n)
    d_slice = d_full[lo:hi].clone() if hi > lo else torch.zeros(1, dtype=torch.uint8, device=d_full.device)
    if rank != 0 or args.no_verify:
        del d_full
        d_full = None
    h_slice = torch.empty(max(hi - lo, 1), dtype=torch.uint8, pin_memory=True)
    h_slice[:d_slice.numel()].copy_(d_slice)
    n_words = (n + 31) // 32
    h_out = torch.empty(n_words, dtype=torch.int64, pin_memory=True) if rank == 0 else None
    torch.cuda.empty_cache()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warm = max(args.warmup, 3)
    for _ in range(warm):
        sh.build(d_slice.data_ptr(), True, n, seps)
    barrier()
    l0 = binding.lib().debwt_launch_count()
    dev_ms = sort_ms = sweep_ms = 0.0
    sweeps = 0
    with ClockSampler(local_rank) as clk:
        t0 = time.perf_counter()
        for _ in range(args.steps):
            sh.build(d_slice.data_ptr(), True, n, seps)
            st = sh.stats()
            dev_ms += st["ms_total"]; sort_ms += st["ms_sort"]; sweep_ms += st["ms_sort_sweeps"]; sweeps += st["sort_sweeps"]
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    dev_ms /= args.steps
    launches = int(binding.lib().debwt_launch_count() - l0)
    clocks = clk.summary()
    last = sh.stats()

    def step_e2e():
        sh.build(h_slice.data_ptr(), False, n, seps)
        return sh.result_into(h_out.data_ptr()) if rank == 0 else None
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        sd = step_e2e()
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    tt = torch.tensor([dev_ms, e2e_ms, wall_ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, wall_ms = (float(x) for x in tt.tolist())
    keys_local = torch.tensor([last["n_keys_local"]], device="cuda", dtype=torch.int64)
    kl = [torch.zeros_like(keys_local) for _ in range(world)]
    if world > 1:
        dist.all_gather(kl, keys_local)
    else:
        kl = [keys_local]
    if rank == 0:
        sha = hashlib.sha256(h_out.numpy().tobytes()).hexdigest()
        want = expected_sha(w.name)
        verify = {"bwt_sha256": sha, "sha_expected": want, "sha_ok": (sha == want) if want else None}
        if not args.no_verify:
            try:
                sharp_np, dollar_np = sd
                bad, vms = api.verify_bwt_device(sh.result_device_ptr(), n, sharp_np, int(dollar_np[0]), d_full.data_ptr(), device=local_rank)
                verify.update({"lf_inversion_bad_rows": bad, "lf_inversion_ms": vms, "lf_inversion_ok": bad == 0,
                               "how": "debwt_verify_bwt_device on rank 0: LF mapping of the stitched result, list ranking by pointer "
                                      "jumping, every row's symbol compared with the input text"})
            except Exception as e:  # noqa: BLE001
                verify.update({"lf_inversion_ok": None, "lf_inversion_error": str(e)})
        nk_loc = last["n_keys_local"]
        line = {
            "metric": METRIC, "value": n_bases / (dev_ms * 1e-3) / 1e6, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": dev_ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic (generated in HBM on every rank in %.2f s)" % t_gen,
            "config": common_config(w, world),
            "timing": "CUDA events on each rank's library stream around its whole build (debwt_shard_stats.ms_total), mean over the "
                      "steps, max over ranks; wall per step %.3f ms (max over ranks)" % wall_ms,
            "exchange": {"path": "debwt_shard_* (csrc/shard.cu): bucketing kernel stores into the owners' CUDA-IPC mapped buffers over "
                                 "NVLink; control data over a shared-memory communicator; no NCCL on the data path",
                         "keys_per_gpu": [int(x.item()) for x in kl]},
            "clocks": clocks,
            "e2e": {"value": n_bases / (e2e_ms * 1e-3) / 1e6, "unit": UNIT, "h2d_bytes_per_step": n, "d2h_bytes_per_step": 8 * n_words,
                    "ms_per_step": e2e_ms},
            "gpu_launches": launches,
            "roofline": roofline_block(nk_loc, sweeps // max(args.steps, 1), sweep_ms / max(sweeps, 1), sort_ms / args.steps, 0.0,
                                       " on rank 0's key range"),
            "sizes": {k: last[k] for k in ("n_symbols", "n_keys", "n_branch", "n_blue", "n_codes")},
            "hbm": {"arena_bytes_rank0": last["arena_bytes"]},
            "verify": verify,
            "bwt_sha256": sha,
        }
        print(json.dumps(line), flush=True)
    sh.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3")
    ap.add_argument("--sort-cfg", type=int, default=0, help="sort kernel configuration (0 = default)")
    ap.add_argument("--cpu-sample", type=int, default=12_000_000, help="bases of the workload the cpu_baseline leg runs")
    ap.add_argument("--ref-sample", type=int, default=0, help="bases per step of the --impl reference arm (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true", help="skip the LF-inversion verifier in the epilogue")
    ap.add_argument("--no-file-to-file", action="store_true")
    ap.add_argument("--no-clocks", action="store_true", help="do not sample clocks (to measure the sampler's own cost)")
    ap.add_argument("--profile-phases", action="store_true", help="sharded path: add rank 0's synchronised per-phase times")
    ap.add_argument("--orchestrator", default="c", choices=["c", "python"],
                    help="N > 1: the sharded build behind the C ABI (csrc/shard.cu) or the Python harness debwt_b200/dist.py")
    ap.add_argument("--sharded", action="store_true", help="use the sharded (multi-GPU) code path even at N=1")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="single-GPU path: write the BWT of the last timed step to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.no_clocks:
        os.environ["DEBWT_NO_CLOCKS"] = "1"
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and (args.impl != "ours" or world > 1 or args.sharded):
        ap.error("--dump-outputs is implemented for the single-GPU path only")
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return
    if (world > 1 or args.sharded) and args.orchestrator == "python":
        ours_sharded_python(args, rank, world, local_rank)
    elif world > 1 or args.sharded:
        ours_shard(args, rank, world, local_rank)
    else:
        ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
