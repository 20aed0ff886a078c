#!/usr/bin/env python
"""bench.py — candidate x sequence mismatch evaluations per second of the degenerate-primer candidate scan.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run, one rank/GPU)
    python bench.py --impl reference ...                     (the CPU arm: the reference's algorithm on the host cores)
    python bench.py ... --dump-outputs DIR                   (also save the last timed step's outputs, to compare builds)

Workload (BASELINE.json configs[3], the configuration the metric is quoted on): synthetic 10^6-sequence x 600-column
alignment (multiprime_b200/synth.py), k=18, degeneracy <= 256 (-n 8), <= 3 mismatches, other flags default.
One step = one full pass of the hot path over every window of the conserved region: entropy prefilter, window k-mer
extraction + haplotype tables, gates, base/dinucleotide tensors, seeds, the NN-array refinement walk with one
candidate scan per round, the per-sequence coverage bit vectors of the chosen primers, Tm, filters, self-dimer gate
-> the rows of the reference's .out TSV.  `value` counts exactly the evaluations the reference makes: (calls to
mis_primer_check) x (sequences), summed over windows, divided by the step time.
With N GPUs every rank holds n_seq sequences of the same synthetic family (weak scaling).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K, DNUM, DEG, VAR = 18, 8, 256, 3
PARAMS = dict(primer_length=K, coverage=0.8, number_of_dege_bases=DNUM, score_of_dege_bases=DEG, product_len=100,
              position="1,2,-1", variation=VAR, raw_entropy_threshold=3.6, distance=4, GC="0.2,0.7", nproc=1)
BYTES_PER_EVAL = K / 2 + 0.25      # SURVEY.md 8(d): one k-column window in 4-bit cells + 2 result bits
BYTES_PER_KMER = K / 2             # window passes: one k-column window in 4-bit cells per (window, sequence)
KERNELS = ("k_prefilter", "k_prefilter_sums", "k_hist", "k_hist_summary", "k_hist_match", "k_cscan", "k_cscan_plan",
           "k_cscan_special", "k_walk_round", "k_walk_advance", "k_walk_compact", "k_walk_seed", "k_peer_allreduce", "k_tm",
           "k_tm_sets", "k_dimer_pairs", "k_dimer_expand", "k_dimer_ends")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n-seq", type=int, default=1_000_000, help="sequences per GPU")
    ap.add_argument("--n-col", type=int, default=600)
    ap.add_argument("--cpu-sample-seqs", type=int, default=20000)
    ap.add_argument("--cpu-sample-windows", type=int, default=256,
                    help="windows of the single-core cpu_baseline leg (about 13 s of CPU work for the port)")
    ap.add_argument("--ref-sample-windows", type=int, default=32,
                    help="windows per step of --impl reference (raised to two per usable core)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--parity-seqs", type=int, default=1 << 18, help="rows of the untimed sharded-parity check (N>1)")
    ap.add_argument("--workload", default="scan", choices=["scan", "dimer"],
                    help="scan: the headline metric (default); dimer: BASELINE.json configs[4], all-pairs dimer grid")
    ap.add_argument("--primers", type=int, default=100_000, help="primers of the dimer workload")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (scan workload, --impl b200)")
    args = ap.parse_args()
    if args.dump_outputs and (args.workload != "scan" or args.impl != "b200"):
        ap.error("--dump-outputs applies to the scan workload of --impl b200")
    return args


def host_cores() -> int:
    """the cores this process may run on (cgroup / affinity aware: os.cpu_count() over-reports inside a lease)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


# ----------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """SM clock and throttle reasons during the timed region (B200_PROFILING.md), read through NVML in-process: spawning
    nvidia-smi five times a second initialises every GPU of the box each time and perturbs the ranks it shares them
    with; nvidia-smi is only the fallback when the NVML binding is missing"""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []            # (sm MHz, max MHz, [reason flags hw_slowdown, hw_thermal, sw_thermal, sw_power_cap])
        self.stop_flag = threading.Event()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle) if hasattr(n, "nvmlDeviceGetCurrentClocksEventReasons") \
            else n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        flags = [bool(r & 0x8), bool(r & 0x40), bool(r & 0x20), bool(r & 0x4)]
        self.rows.append((float(sm), float(mx), flags))

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
        f = [x.strip() for x in out.strip().split(",")]
        if len(f) >= 7:
            self.rows.append((float(f[0]), float(f[1]), [x.lower().startswith("active") for x in f[3:7]]))

    def run(self):
        while not self.stop_flag.is_set():
            try:
                if self.nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self.stop_flag.wait(0.05 if self.nvml is not None else 0.5)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(r[0] for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2][i] for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.rows[0][1], "reasons": reasons,
                "samples": len(self.rows), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def kernel_traffic():
    """DRAM bytes (read + write) per launch of the profiled kernels, from the committed `ncu --set full` captures"""
    path = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh)
    return {}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------------------
# CPU arm.  The reference is a set of Python scripts: in the build container (where /root/reference exists) the live
# NN_degenerate.get_primers is timed (kind "live"); on the GPU box, where the reference cannot travel, its restatement
# oracle/mp_oracle.py (kind "port", pinned to the live reference by tests/golden/) runs the same windows.
# ----------------------------------------------------------------------------------------------------------
_CPU_DATA = {}
REF_CORE = "/root/reference/scripts/multiPrime-core_V20.py"


def _oracle_window(p):
    """one window of the bounded sample through the oracle port; the alignment is inherited from the parent (fork)"""
    from oracle import mp_oracle as o
    prm = o.Params(k=K, dnum=DNUM, degeneracy=DEG, variation=VAR, entropy=3.6, gc="0.2,0.7", size=100, fraction=0.8,
                   coordinate="1,2,-1", away=4)
    trace = []
    o.design_window(_CPU_DATA["ids"], _CPU_DATA["seqs"], p, prm, 3.6, trace)
    return len(trace)


def _live_window(p):
    """one window through the live reference class (mis_primer_check calls counted by wrapping the method)"""
    app = _CPU_DATA["live"]
    calls = [0]
    orig = app.mis_primer_check

    def wrapped(*a):
        calls[0] += 1
        return orig(*a)

    app.mis_primer_check = wrapped
    try:
        app.get_primers(app.seq_dict, p)
        app.resQ.get()
    finally:
        app.mis_primer_check = orig
    return calls[0]


def cpu_prepare(n_seq: int, n_col: int, live: bool):
    from multiprime_b200 import synth
    from oracle import mp_oracle as o
    key = (n_seq, n_col, live)
    if _CPU_DATA.get("key") == key:
        return
    codes = synth.synth_codes(n_seq, n_col)
    ids, seqs = synth.seq_ids(n_seq), synth.codes_to_strings(codes)
    _CPU_DATA.clear()
    _CPU_DATA.update(key=key, ids=ids, seqs=seqs, region=o.region(seqs, 0.8))
    if live:
        import importlib.util
        import tempfile
        import warnings
        warnings.filterwarnings("ignore")
        spec = importlib.util.spec_from_file_location("mpcore_live", REF_CORE)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        tmp = tempfile.mkdtemp()
        fa = os.path.join(tmp, "in.fa")
        synth.write_fasta(fa, codes)
        _CPU_DATA["live"] = mod.NN_degenerate(seq_file=fa, primer_length=K, coverage=0.8, number_of_dege_bases=DNUM,
                                              score_of_dege_bases=DEG, product_len=100, position="1,2,-1",
                                              variation=VAR, raw_entropy_threshold=3.6, distance=4, GC="0.2,0.7",
                                              nproc=1, outfile=os.path.join(tmp, "x.out"))


def cpu_sample(n_seq: int, n_col: int, n_windows: int, procs: int, live: bool = False):
    """the CPU implementation over a bounded sample: the first n_seq synthetic sequences, n_windows windows spread over
    the region.  Returns (evals, seconds).  Windows are dealt to `procs` forked workers (the reference itself is
    single-process: its pool is inert, core:1143; this is the best case for the CPU side)."""
    cpu_prepare(n_seq, n_col, live)
    start, stop = _CPU_DATA["region"]
    all_pos = list(range(start, stop - K))
    pos = [all_pos[int(i * (len(all_pos) - 1) / max(1, n_windows - 1))] for i in range(n_windows)]
    fn = _live_window if live else _oracle_window
    t0 = time.perf_counter()
    if procs <= 1:
        calls = [fn(p) for p in pos]
    else:
        import multiprocessing as mp
        with mp.get_context("fork").Pool(procs) as pool:
            calls = pool.map(fn, pos, chunksize=1)
    dt = time.perf_counter() - t0
    return sum(calls) * n_seq, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    live = os.path.exists(REF_CORE)
    n_windows = max(args.ref_sample_windows, 2 * cores)            # keep every core busy
    procs = min(cores, n_windows)
    vals = []
    for i in range(args.warmup + args.steps):
        ev, dt = cpu_sample(args.cpu_sample_seqs, args.n_col, n_windows, procs, live)
        if i >= args.warmup:
            vals.append((ev, dt))
        if i == 0 and dt > 40:                                      # a slow host: one warm-up pass is enough
            args.warmup = 1
    per_step = [v[0] / v[1] for v in vals]
    value = statistics.median(per_step)
    sample = "%s, first %d synthetic sequences x %d windows spread over the region, %d worker processes on %d usable " \
             "cores; median of %d steps (min %.3g, max %.3g evals/s)" % (
                 "live reference multiPrime-core_V20.py NN_degenerate.get_primers" if live else
                 "oracle port (oracle/mp_oracle.py; the Python reference cannot travel to the GPU box)",
                 args.cpu_sample_seqs, n_windows, procs, cores, len(vals), min(per_step), max(per_step))
    line = {"impl": "reference", "metric": "candidate_x_sequence_evals_per_sec", "value": value, "unit": "evals/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000 * statistics.median(v[1] for v in vals),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": "synthetic MSA %dx%d k=%d d<=%d v<=%d (bounded sample)" %
                       (args.n_seq, args.n_col, K, DEG, VAR)},
            "cpu_baseline": {"value": value, "unit": "evals/s", "cores": procs, "kind": "reference" if live else "port",
                             "sample": sample},
            "e2e": {"value": value, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------
def sharded_parity(args, rank, local, world, comm, stream):
    """untimed strong-scaling check (N > 1): the SAME alignment once on one rank without a communicator and once
    sharded over all ranks with NCCL — rows and call traces must be identical"""
    import numpy as np
    import torch.distributed as dist
    from multiprime_b200 import core, synth
    n, L = args.parity_seqs, args.n_col
    codes = synth.synth_codes(n, L, seed=77)
    ids = synth.seq_ids(n)
    lo, hi = rank * n // world, (rank + 1) * n // world
    kw = dict(PARAMS)
    app = core.NN_degenerate(seq_file=None, outfile="", alignment=(ids[lo:hi], codes[lo:hi], np.full(hi - lo, L, np.int32)),
                             device=local, sidecars=False, stream=stream, comm=comm, row0=lo, **kw)
    pos = list(range(app.start_position, app.stop_position - K))
    got = sorted((r["row"], r["trace"]) for r in app.design(pos))
    app.close()
    out = None
    if rank == 0:
        one = core.NN_degenerate(seq_file=None, outfile="", alignment=(ids, codes, np.full(n, L, np.int32)), device=local,
                                 sidecars=False, stream=stream, **kw)
        want = sorted((r["row"], r["trace"]) for r in one.design(pos))
        one.close()
        out = {"sequences": n, "windows": len(pos), "rows": len(want), "equal": got == want}
    dist.barrier()
    return out


# columns of a row (the reference's .out TSV) that are numbers; 3 is the primer, 10 the Information column
ROW_COLUMNS = {"position": 0, "entropy_cover": 1, "entropy_total": 2, "degenerate_number": 4, "nonsense_number": 5,
               "coverage": 6, "mis_f_coverage": 7, "mis_r_coverage": 8, "tm": 9}
FILTER_FLAGS = {"GC_out_of_range": 1, "di_nucleotide": 2, "hairpin": 4}
DUMP_SAMPLE_SEQS = 1 << 14
DUMP_SAMPLE_BYTES = 48 << 20


def dump_outputs(out_dir, recs, app):
    """--dump-outputs: the rows of one step, sorted by position, as one float64 array per numeric column, the primers as
    4-bit base sets, and the Information column as GC content (-1 where the row holds only filter notes) and filter flags;
    the per-sequence F non-cover / R non-cover / gap-row bit vectors of every row as counts over all sequences of this
    rank and as the bits of a fixed seeded sample of sequences (the whole vectors are 375 KB per row at 10^6)"""
    import numpy as np
    from multiprime_b200.iupac import sets_of
    rows = sorted((r["row"] for r in recs), key=lambda row: row[0])
    out = {name: np.array([row[c] for row in rows], np.float64) for name, c in ROW_COLUMNS.items()}
    out["primer_sets"] = np.array([sets_of(row[3]) for row in rows], np.float32).reshape(len(rows), K)
    gc, flags = np.full(len(rows), -1.0), np.zeros(len(rows))
    for i, row in enumerate(rows):
        if not isinstance(row[10], str):
            gc[i] = row[10]
            continue
        for note in row[10].split("|"):              # "GC_out_of_range (0.72)", "di_nucleotide", "hairpin"
            flags[i] += FILTER_FLAGS[note.split(" ")[0]]
            if note.startswith("GC_out_of_range"):
                gc[i] = float(note.split("(")[1].rstrip(")"))
    out["gc"], out["filter_flags"] = gc, flags
    pos, bits = app.coverage_bits()                  # also windows whose primer the self-dimer test dropped
    at = {p: i for i, p in enumerate(pos.tolist())}
    bits = bits[[at[row[0]] for row in rows]]
    n_seq = app.n_local
    if n_seq % 32:                                   # bits past the last sequence are not part of the vectors
        bits[:, :, -1] &= np.uint32((1 << (n_seq % 32)) - 1)
    out["non_cover_counts"] = np.bitwise_count(bits).sum(axis=2, dtype=np.int64).astype(np.float64)
    n_sample = min(n_seq, DUMP_SAMPLE_SEQS, DUMP_SAMPLE_BYTES // (12 * max(1, len(rows))))
    seqs = np.sort(np.random.default_rng(0).permutation(n_seq)[:n_sample])
    out["sample_sequences"] = seqs.astype(np.float64)
    out["coverage_bits_sample"] = ((bits[:, :, seqs >> 5] >> (seqs & 31).astype(np.uint32)) & 1).astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def run_b200(args):
    from multiprime_b200 import core, synth

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    n_seq, n_col = args.n_seq, args.n_col
    # synthetic input first: the generator forks worker processes, which must happen before CUDA / NCCL threads exist
    codes = synth.synth_codes_parallel(n_seq, n_col, row0=rank * n_seq, procs=max(1, host_cores() // world))
    packed = core.pack4(codes)
    del codes
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pinned = torch.from_numpy(packed).pin_memory()
    packed_pinned = pinned.numpy()
    ids = synth.seq_ids(n_seq, rank * n_seq)
    stream = torch.cuda.current_stream().cuda_stream

    comm = None
    if world > 1:
        from multiprime_b200.comm import TorchComm
        comm = TorchComm(torch.device("cuda", local))

    def make_app():
        # sidecars=False: no JSON side files (they list sequence ids per uncovered haplotype and do not scale to 10^6
        # sequences); keep_bits=True: the per-sequence F / R non-cover and gap-row bit vectors of every chosen primer ARE
        # produced (in HBM, where the pairing step reads them)
        return core.NN_degenerate(seq_file=None, outfile="", packed=(ids, packed_pinned, n_col, None), device=local,
                                  sidecars=False, want_trace=False, keep_bits=True, stream=stream, comm=comm,
                                  row0=rank * n_seq, rows_on_rank0_only=True, **PARAMS)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    parity = sharded_parity(args, rank, local, world, comm, stream) if world > 1 else None

    app = make_app()
    positions = list(range(app.start_position, app.stop_position - K))
    h2d = packed_pinned.nbytes

    def step_resident():
        return app.design(positions)

    e2e_init = {}

    def step_e2e():
        a = make_app()                                  # H2D of the packed alignment + plane build + region
        for kk, vv in a.init_ms.items():
            e2e_init[kk] = e2e_init.get(kk, 0.0) + vv
        recs = a.design(list(range(a.start_position, a.stop_position - K)))
        a.close()
        return recs

    # a long-lived process (server, pipeline driver) does not want the cyclic GC to walk the 10^6 sequence ids and the
    # imported modules in the middle of a step (a full collection costs 100+ ms here): park everything allocated so far
    import gc
    gc.collect()
    gc.freeze()
    results = {}
    sampler = ClockSampler(local)
    for name, fn in (("value", step_resident), ("e2e", step_e2e)):
        for _ in range(args.warmup):
            fn()
        e2e_init.clear()
        app.ctx.profile_read(None)
        app.ctx.profile(name == "value")
        app.stats.update(evals=0, scan_calls=0, candidates=0, phase_ms={})
        launches0 = app.ctx.launches
        if name == "value":
            sampler.start()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t0 = time.perf_counter()
        recs = []
        per_step = []
        for _ in range(args.steps):
            ts = time.perf_counter()
            recs = fn()
            per_step.append(1000 * (time.perf_counter() - ts))
        e1.record()
        nrows = len(recs)
        if name == "value":
            last_recs = recs
        barrier()
        wall = time.perf_counter() - t0
        ms = max(e0.elapsed_time(e1), 0.0)
        ms = max(ms, 1000 * wall) if name == "e2e" else ms
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        results[name] = {"ms": float(t.item()), "rows": nrows,
                         "per_step": [round(min(per_step), 2), round(statistics.median(per_step), 2), round(max(per_step), 2)]}
        if name == "value":
            sampler.stop_flag.set()
            results["launches"] = app.ctx.launches - launches0
            results["prof"] = {kn: app.ctx.profile_read(kn) for kn in KERNELS}
            results["evals_per_step"] = app.stats["evals"] / args.steps
            results["scan_calls"] = app.stats["scan_calls"] / args.steps
            results["candidates"] = app.stats["candidates"] / args.steps
            results["phases"] = {k: round(v / args.steps, 2) for k, v in app.stats["phase_ms"].items()}
            app.ctx.profile(False)
    evals_all = float(results["evals_per_step"])      # already global: calls x (sequences of ALL shards)
    if world > 1:
        sys.stderr.write("rank %d phases ms/step: %s\n" % (rank, json.dumps(results["phases"])))
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_recs, app)
    ms_step = results["value"]["ms"] / args.steps
    value = evals_all / (ms_step / 1000)
    e2e_ms = results["e2e"]["ms"] / args.steps
    peak, peak_src = peaks()
    prof = results["prof"]
    traffic = kernel_traffic()

    def roofline_of(kn):
        ms, n, units = prof[kn]
        per_unit = BYTES_PER_EVAL if kn == "k_cscan" else BYTES_PER_KMER
        ach = units * per_unit / (ms / 1000) / 1e9 if ms > 0 else 0.0
        return {"bound": "hbm", "kernel": kn, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic.get(kn), "peak_source": peak_src, "launches": n,
                "avg_launch_ms": ms / max(1, n), "units_in_launches": units, "bytes_per_unit": per_unit,
                "ms_per_step": ms / args.steps}

    big = max(("k_prefilter", "k_hist", "k_cscan"), key=lambda kn: prof[kn][0])
    roof = roofline_of(big)
    roof["note"] = (
        "dominant kernel of the step by CUDA-event time. achieved = algorithmic bytes (SURVEY.md 8d: k/2 B per (window, "
        "sequence) k-mer for the window passes, k/2 + 0.25 B per candidate x sequence evaluation for the scan) / "
        "event-timed kernel time; traffic = dram read+write bytes of one launch (ncu --set full, profiles/). The "
        "algorithmic figure assumes no reuse: the window passes cut up to 32 windows out of every loaded word and the "
        "column scan re-reads plane rows from L2, so real DRAM traffic is far below it and a fraction above 1 is "
        "reuse, not a faster-than-HBM kernel; these kernels are bound by L2 atomics / integer issue (see profiles/README.md)")
    line = {
        "metric": "candidate_x_sequence_evals_per_sec", "value": value, "unit": "evals/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": "synthetic MSA %dx%d per GPU (multiprime_b200/synth.py seed 20240923), k=%d, -n %d -d %d "
                               "-v %d, %d windows, %d rows out" % (n_seq, n_col, K, DNUM, DEG, VAR, len(positions),
                                                                  results["value"]["rows"]),
                   "parallelism": "sequence shards x%d: windows owned round-robin (all-to-all of haplotype entries), "
                                  "all-reduce of the coverage-count vector per scan round" % world,
                   "l2": "inputs (2 x %.0f MB of bit-planes + GB-sized haplotype tables) exceed the 126 MB L2" %
                         (n_seq * n_col / 2 / 1e6),
                   "evals_per_step": evals_all, "scan_rounds_per_step": results["scan_calls"],
                   "scan_candidates_per_step": results["candidates"]},
        "clocks": sampler.summary(),
        "e2e": {"value": evals_all / (e2e_ms / 1000), "unit": "evals/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": int(results["value"]["rows"] * 120), "ms_per_step": e2e_ms,
                "host_ms_min_median_max": results["e2e"]["per_step"],
                "setup_ms_per_step": {kk: round(vv / args.steps, 2) for kk, vv in e2e_init.items()}},
        "host_ms_min_median_max": results["value"]["per_step"],
        "gpu_launches": int(results["launches"]),
        "roofline": roof,
        "roofline_scan": roofline_of("k_cscan"),
        "kernels": {"k_scan_ms_per_step": prof["k_cscan"][0] / args.steps,
                    "ms_per_step": {kn: round(prof[kn][0] / args.steps, 3) for kn in KERNELS}},
        "host_phases_ms_per_step": results["phases"],
    }
    if parity is not None:
        line["sharded_parity"] = parity
    if not args.no_cpu_baseline and world == 1:       # the CPU baseline is timed on rank 0 at N = 1 only
        live = os.path.exists(REF_CORE)
        evc, dtc = cpu_sample(args.cpu_sample_seqs, n_col, args.cpu_sample_windows, 1, live)
        line["cpu_baseline"] = {"value": evc / dtc, "unit": "evals/s", "cores": 1, "kind": "reference" if live else "port",
                                "sample": "%s, first %d synthetic sequences x %d windows, %.1f s" %
                                          ("multiPrime-core_V20.py" if live else "oracle/mp_oracle.py",
                                           args.cpu_sample_seqs, args.cpu_sample_windows, dtc)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_dimer(args):
    """secondary metric (BASELINE.json configs[4]): primer pairs per second of the all-pairs dimer grid (finDimer
    semantics, threshold 3.96) on P synthetic 18-mers with ~6 % two-fold positions.  The grid is a set of independent
    units: with N ranks the row bands are dealt round-robin and the sparse hit lists gathered (strong scaling)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from multiprime_b200 import _lib
    from multiprime_b200.dimer import dg_consts, loss_table
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    comm = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        from multiprime_b200.comm import TorchComm
        comm = TorchComm(torch.device("cuda", local))
    P = args.primers
    rng = np.random.default_rng(5)
    sets = (1 << rng.integers(0, 4, (P, 18))).astype(np.uint8)
    amb = rng.random((P, 18)) < 0.06
    sets[amb] |= (1 << rng.integers(0, 4, int(amb.sum()))).astype(np.uint8)
    sets_list = [row.tolist() for row in sets]
    ctx = _lib.Context.shared(local, torch.cuda.current_stream().cuda_stream)
    eng = _lib.Dimer(ctx, sets_list, 5, 18, True, loss_table(3.96), dg_consts())
    band = max(1, min(P, (1 << 25) // P * 8))
    bands = list(range(0, P, band))

    def step():
        hits = tested = 0
        for b, r0 in enumerate(bands):
            if b % world != rank:
                continue
            hi, hj, ho, hd, nt = eng.grid(r0, min(P, r0 + band), max_hits=1 << 24)
            hits += len(hi)
            tested += nt
        tot = np.array([hits, tested], np.int64)
        return comm.allreduce_sum(tot) if comm else tot

    for _ in range(min(args.warmup, 1)):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = ctx.launches
    t0 = time.perf_counter()
    for _ in range(args.steps):
        tot = step()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = float(t.item())
    pairs = P * (P + 1) // 2
    if rank == 0:
        print(json.dumps({"metric": "dimer_pairs_per_sec", "value": pairs * args.steps / dt, "unit": "pairs/s",
                          "n_gpus": world, "steps": args.steps, "warmup": min(args.warmup, 1),
                          "ms_per_step": 1000 * dt / args.steps, "higher_is_better": True, "scaling": "strong",
                          "vs_baseline": None, "dtype": "u64", "data": "synthetic",
                          "config": {"workload": "all-pairs dimer grid, %d synthetic 18-mers (~6%% two-fold positions), "
                                                 "threshold 3.96" % P, "pairs": pairs,
                                     "pairs_after_5mer_prefilter": int(tot[1]), "dimer_pairs": int(tot[0]),
                                     "parallelism": "row bands round-robin over %d ranks, hit counts all-reduced" % world},
                          "gpu_launches": int(ctx.launches - launches0)}))
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    if a.workload == "dimer":
        run_dimer(a)
    elif a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
