#!/usr/bin/env python3
"""bench.py -- headline benchmark of the gap-affine WFA hot path on B200.

  python bench.py --gpus N --steps K --warmup W            (our CUDA path)
  python bench.py --impl reference --gpus N --steps K ...  (the reference's CPU WFA, host cores)

Workload (BASELINE.json metric, SURVEY.md 8(d) cfg 4 headline sub-run): synthetic
10 kbp pairs, 5 % error, penalties x=2,o=3,e=1, `-e 3000`, exact, with CIGAR.
A step = one pass of the hot path (pack, score-bound, wavefront, traceback and CIGAR-text
kernels) over one batch of PAIRS_PER_GPU pairs per GPU.  Pairs shard across GPUs with no collective
(weak scaling: per-GPU batch fixed).

  value : alignments/s over all GPUs, batch resident in HBM, device time from CUDA
          events recorded on the launching stream, max over ranks.
  e2e   : same metric through the public C API exactly as an unmodified reference caller uses it
          (wfagpu_add_sequences ... wfagpu_align, no extension call): H2D of the ASCII from the aligner's
          own page-locked buffer, kernels, D2H of results + CIGAR text and the copy into results[i]
          are all inside the timed region.

Besides the contract keys the line carries (rank 0):
  roofline       the BINDING roof: instruction issue (cells counted by the kernel x 64 nominal thread
                 instructions / wavefront-kernel time against SMs x 128 lanes x sampled clock)
  roofline_hbm   the HBM figure (algorithmic bytes / kernel time against the measured copy bandwidth) + ncu traffic
  reference_gpu  the UNMODIFIED reference GPU binary (oracle/_ref/gpu, built for sm_100) on a sample of the same
                 workload on the same GPU: its own wall-time alignments/s and how many CIGARs are byte-identical
  configs        BASELINE configs 1-5 at their stated sizes through wfagpu_align, each with a parity sample
  envelope       cold first call, un-hinted provisioning, stale hint (with the pairs that were re-dispatched)
  e2e_pageable   launch_alignments on a buffer the caller malloc'ed itself (staged through pinned memory)
  e2e_inlib      (N > 1) ONE wfagpu_align call on rank 0 sharding N x the batch over the N GPUs in-library
  per_rank       per-rank step time, launch shape and re-dispatch count
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "wfa-gpu_b200", "python"))

METRIC = "alignments_per_s_10kbp_5pct_cigar"
UNIT = "alignments/s"
LENGTH, ERR, PEN, MAX_ERROR = 10000, 0.05, (2, 3, 1), 3000
PAIRS_PER_GPU = int(os.environ.get("WFAGPU_BENCH_PAIRS", 8192))
CPU_SAMPLE = int(os.environ.get("WFAGPU_BENCH_CPU_SAMPLE", 1536))
REF_STEP_PAIRS = int(os.environ.get("WFAGPU_BENCH_REF_PAIRS", 768))
REFGPU_SAMPLE = int(os.environ.get("WFAGPU_BENCH_REFGPU_SAMPLE", 2048))
SEED = 0xB2000004


def config(extra=None):
    c = {"workload": "cfg4-headline: 10 kbp pairs, 5% error, x=2,o=3,e=1, -e 3000, exact, CIGAR",
         "pairs_per_gpu_per_step": PAIRS_PER_GPU, "length": LENGTH, "error_rate": ERR,
         "penalties": list(PEN), "max_error": MAX_ERROR,
         "l2_policy": "inputs+arenas larger than L2 (164 MB ASCII + >10 GB ring-snapshot arena per step)"}
    if extra:
        c.update(extra)
    return c


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons during the timed region (B200_PROFILING.md's clocks line).

    Sampled through NVML inside this process (nvidia_ml_py): starting an nvidia-smi process every
    200 ms takes the driver lock for tens of milliseconds and showed up as idle gaps between the
    kernels of a step.  Falls back to nvidia-smi when NVML cannot be loaded."""

    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu = gpu
        self.rows = []          # (sm_mhz, sm_max_mhz, [reason names])
        self.stop_flag = threading.Event()
        self.nvml = None
        self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            idx = gpu
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    idx = int(vis.split(",")[gpu])
                except Exception:
                    idx = gpu
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def sample_nvml(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        bits = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        masks = [n.nvmlClocksEventReasonHwSlowdown, n.nvmlClocksEventReasonHwThermalSlowdown,
                 n.nvmlClocksEventReasonSwThermalSlowdown, n.nvmlClocksEventReasonSwPowerCap]
        self.rows.append((int(sm), int(mx), [self.NAMES[i] for i in range(4) if bits & masks[i]]))

    def sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        r = [x.strip() for x in out.split(",")]
        if len(r) >= 6 and r[0].isdigit():
            self.rows.append((int(r[0]), int(r[1]) if r[1].isdigit() else 0,
                              [self.NAMES[i] for i in range(4) if r[2 + i].lower().startswith("active")]))

    def run(self):
        while not self.stop_flag.is_set():
            try:
                if self.nvml:
                    self.sample_nvml()
                else:
                    self.sample_smi()
            except Exception:
                pass
            self.stop_flag.wait(0.1 if self.nvml else 0.5)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm = sorted(r[0] for r in self.rows)
        mx = [r[1] for r in self.rows if r[1]]
        reasons = sorted({x for r in self.rows for x in r[2]})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "source": "nvml" if self.nvml else "nvidia-smi"}


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    return rank, world, local


def shard_seed(rank):
    """Every rank aligns its own deterministic slice of the synthetic workload."""
    return SEED + 7919 * rank


def reduce_max(values, device=None):
    """Max over ranks of a list of floats (device time, wall time): the slowest rank sets the pace."""
    import torch
    import torch.distributed as dist
    t = torch.tensor(values, dtype=torch.float64, device=device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.tolist()


def aggregate_value(pairs_per_gpu, world, steps, t_max):
    """Whole-job throughput: all pairs of all ranks over the slowest rank's time."""
    return pairs_per_gpu * world * steps / t_max


def gather_per_rank(info, world):
    """[info of rank 0, ..., info of rank world-1] on every rank (plain python objects)."""
    if world == 1:
        return [info]
    import torch.distributed as dist
    out = [None] * world
    dist.all_gather_object(out, info)
    return out


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def algorithmic_bytes(a, n_ops_total):
    """SURVEY.md 8(d): ASCII read by pack + packed write + one packed read + metadata + result + bt chain."""
    total = 0
    for i in range(a.num_pairs):
        m = a.s.sequences_metadata[i]
        pl, tl = m.pattern_len, m.text_len
        total += (pl + tl) + 2 * ((pl + 3) // 4 + (tl + 3) // 4) + 48 + 20
    return total + 8 * ((n_ops_total + 15) // 16)


def cells_of_scores(lib, wfagpu, scores):
    import ctypes as C
    x, o, e = PEN
    md = MAX_ERROR * (max(x, o + e) + 1) + 16
    tab = (wfagpu.Step * (md + 1))()
    units = C.c_uint64()
    d_end = lib.wfagpu_build_step_table(x, o, e, MAX_ERROR, md, 0, tab, C.byref(units))
    cum = [0] * (d_end + 1)
    run = 0
    for d in range(d_end):
        if tab[d].kind in (1, 2):
            run += 2 * tab[d].n + 1
        cum[d] = run
    return sum(cum[min(s, d_end - 1)] for s in scores)


def measured_cells(gpu):
    """Cells the wavefront kernel really computes for one step of this workload: the same batch run
    once more in a child process with the kernel's per-pair cell counter switched on (untimed)."""
    try:
        env = dict(os.environ, WFAGPU_COUNT_CELLS="1", CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(gpu)))
        out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "perf_probe.py"), str(PAIRS_PER_GPU), str(LENGTH),
                              str(ERR), str(MAX_ERROR), "1", "1"], env=env, capture_output=True, text=True, timeout=300).stdout
        return int(json.loads(out.strip().splitlines()[-1])["cells"])
    except Exception:
        return 0


def make_aligner(wfagpu, seed, n, length, err_lo, err_hi, pen, max_error=None, cigar=True, band=None, width=None, batch=None):
    a = wfagpu.Aligner()
    a.add_synthetic(seed, n, length, err_lo, err_hi)
    assert a.initialize_parameters(*pen)
    if max_error is not None:
        a.options.max_error = max_error
    a.options.compute_cigar = cigar
    if band:
        a.options.band = band
        a.options.threads_per_block = width
    if batch:
        a.set_batch_size(batch)
    return a


def time_align(a, reps, warm=1):
    """Best wall time of `reps` wfagpu_align calls (after `warm` untimed ones) and the stats of the last."""
    for _ in range(warm):
        a.reset_results()
        a.align()
    best = None
    for _ in range(reps):
        a.reset_results()
        t0 = time.perf_counter()
        a.align()
        dt = time.perf_counter() - t0
        best = dt if best is None or dt < best else best
    return best, a.run_stats()


def gcells(a):
    return sum(a.s.sequences_metadata[i].pattern_len * a.s.sequences_metadata[i].text_len for i in range(a.num_pairs))


# ------------------------------------------------------------------ reference GPU binary (unmodified)
REF_GPU_BIN = os.path.join(ROOT, "oracle", "_ref", "gpu", "wfa.affine.gpu")


def run_reference_gpu(pairs, pen, max_error, cigar=True, extra=()):
    """-> ([(score, cigar)], the tool's own 'Wall time' seconds, total seconds) or None when the binary is missing."""
    if not os.path.exists(REF_GPU_BIN):
        return None
    with tempfile.TemporaryDirectory() as td:
        seq, out = os.path.join(td, "in.seq"), os.path.join(td, "out.txt")
        with open(seq, "w") as f:
            for p, t in pairs:
                f.write(">" + p + "\n<" + t + "\n")
        cmd = [REF_GPU_BIN, "-i", seq, "-g", "%d,%d,%d" % pen, "-e", str(max_error), "-o", out] + (["-x"] if cigar else []) + list(extra)
        t0 = time.time()
        pr = subprocess.run(cmd, capture_output=True, text=True)
        total = time.time() - t0
        if pr.returncode != 0:
            return None
        wall = None
        for line in (pr.stdout + pr.stderr).splitlines():
            if "Wall time" in line:
                try:
                    wall = float(line.split("Wall time:")[1].split("s")[0])
                except Exception:
                    pass
        res = []
        for line in open(out):
            parts = line.rstrip("\n").split("\t")
            if parts and parts[0] != "":
                res.append((-int(parts[0]), parts[1] if len(parts) > 1 else None))
        return res, wall, total


def reference_gpu_block(a):
    n = min(REFGPU_SAMPLE, a.num_pairs)
    pairs = [a.pair(i) for i in range(n)]
    r = run_reference_gpu(pairs, PEN, MAX_ERROR, cigar=True)
    if r is None:
        return {"unavailable": "oracle/_ref/gpu/wfa.affine.gpu missing or failed (built by `make -C oracle refgpu` where /root/reference exists)"}
    res, wall, total = r
    same = sum(1 for i in range(n) if res[i] == (a.error(i), a.cigar(i)))
    same_score = sum(1 for i in range(n) if res[i][0] == a.error(i))
    return {"impl": "unmodified reference GPU code (lib/kernels/*.cu built -gencode arch=compute_100,code=sm_100), its CLI defaults",
            "cmd": "wfa.affine.gpu -i sample.seq -g 2,3,1 -e 3000 -x -o out", "sample_pairs": n,
            "value": round(n / wall, 1) if wall else None, "unit": UNIT, "tool_wall_s": wall, "process_s": round(total, 2),
            "identical_cigars": f"{same}/{n}", "identical_scores": f"{same_score}/{n}",
            "note": "same GPU, outside every timed region; includes the tool's own H2D/D2H and its CPU fallback, like its published numbers"}


# ------------------------------------------------------------------ BASELINE configs 1-5 at stated size
def parity_sample(a, idx, pen, kind, orc, refcpu, max_error, band=None, width=None):
    """Compares the pairs `idx` with the checker; returns 'k/k identical (what)'."""
    ok = 0
    if kind == "cpu_wfa_score":
        P, T = [a.pair(i)[0] for i in idx], [a.pair(i)[1] for i in idx]
        errs, _ = refcpu.align_batch(P, T, *pen, cigar=False, threads=len(os.sched_getaffinity(0)))
        ok = sum(1 for j, i in enumerate(idx) if errs[j] == a.error(i))
        return f"{ok}/{len(idx)} scores == unmodified reference CPU WFA"
    for i in idx:
        p, t = a.pair(i)
        if band:
            r = orc.align(p, t, *pen, max_error, band=band, window=width, cigar=a.options.compute_cigar)
            if not r["finished"]:
                r = orc.align(p, t, *pen, 100000, cigar=a.options.compute_cigar)
        else:
            r = orc.align(p, t, *pen, 100000, cigar=a.options.compute_cigar)
        good = a.error(i) == r["distance"] and (not a.options.compute_cigar or a.cigar(i) == r["cigar"])
        ok += 1 if good else 0
    return f"{ok}/{len(idx)} identical to the oracle (score" + (" + CIGAR text)" if a.options.compute_cigar else ")")


def run_configs(wfagpu):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle import Oracle, RefCPU
    orc = Oracle()
    refcpu = RefCPU() if RefCPU.available() else None
    out = {}

    def release(a):
        """Every configuration starts from an empty device: pooled contexts keep their grown buffers (tens of GB of
        snapshot arenas after cfg 4), and a configuration that finds little free memory gets fewer resident CTAs."""
        a.destroy()
        wfagpu.load().wfagpu_device_close_all()

    def entry(a, dt, st, parity, extra=None):
        e = {"pairs": a.num_pairs, "e2e_alignments_per_s": round(a.num_pairs / dt, 1), "e2e_gcups": round(gcells(a) / dt / 1e9, 1),
             "wall_ms": round(dt * 1e3, 2), "redispatched": int(st["redispatched"]), "launches": int(st["launches"]),
             "failed_pairs": int(st["failed_pairs"]), "parity_sample": parity}
        if extra:
            e.update(extra)
        return e

    # cfg 1: 10 000 x 150 bp, 2 %, score + CIGAR (defaults of wfagpu_initialize_parameters)
    a = make_aligner(wfagpu, 0xB2000001, 10000, 150, 0.02, 0.02, PEN, cigar=True)
    dt, st = time_align(a, 3)
    out["cfg1_150bp_2pct_cigar"] = entry(a, dt, st, parity_sample(a, range(0, 10000, 100), PEN, "oracle", orc, refcpu, a.options.max_error))
    release(a)
    # cfg 2: 1 000 000 x 150 bp, 5 %, score only
    a = make_aligner(wfagpu, 0xB2000002, 1000000, 150, 0.05, 0.05, PEN, cigar=False)
    dt, st = time_align(a, 2)
    out["cfg2_150bp_5pct_score_1M"] = entry(a, dt, st, parity_sample(a, range(0, 1000000, 10007), PEN, "oracle", orc, refcpu, a.options.max_error))
    release(a)
    # cfg 3: 100 000 x 1 kbp, 10 %, exact with CIGAR, -e 300 (about 5 % of the pairs exceed it: re-dispatched on the GPU)
    a = make_aligner(wfagpu, 0xB2000003, 100000, 1000, 0.10, 0.10, PEN, max_error=300, cigar=True)
    dt, st = time_align(a, 2)
    out["cfg3_1kbp_10pct_cigar_e300"] = entry(a, dt, st, parity_sample(a, range(0, 100000, 2503), PEN, "oracle", orc, refcpu, 300))
    release(a)
    # cfg 4 at full size: 100 000 x 10 kbp in ONE wfagpu_align call, error ~ U[1 %, 5 %], exact vs -B 25 -t 512
    a = make_aligner(wfagpu, 0xB2000004, 100000, 10000, 0.01, 0.05, PEN, max_error=MAX_ERROR, cigar=True)
    dt, st = time_align(a, 1)
    exact = a.errors()
    out["cfg4_10kbp_1to5pct_cigar_exact_100k"] = entry(a, dt, st, parity_sample(a, range(0, 100000, 6251), PEN, "oracle", orc, refcpu, MAX_ERROR),
                                                        {"host_buffer_gb": round(a.s.sequences_buffer_len / 1e9, 2)})
    a.options.band = 25
    a.options.threads_per_block = 512
    dt, st = time_align(a, 1)
    banded = a.errors()
    recall = sum(1 for x, y in zip(exact, banded) if x == y) / len(exact)
    out["cfg4_10kbp_1to5pct_cigar_band25_w512_100k"] = entry(
        a, dt, st, parity_sample(a, range(0, 100000, 12503), PEN, "oracle", orc, refcpu, MAX_ERROR, band=25, width=512),
        {"banded_recall": round(recall, 5), "note": "recall = pairs whose banded score equals the exact score"})
    release(a)
    # cfg 5: 50 kbp, 15 %, CIGAR, first budget (8000) below every score: every pair is re-dispatched on the GPU
    n5 = int(os.environ.get("WFAGPU_BENCH_CFG5_PAIRS", 2500))     # BASELINE: 20 000 pairs over 8 GPUs
    a = make_aligner(wfagpu, 0xB2000005, n5, 50000, 0.15, 0.15, PEN, max_error=8000, cigar=True)
    dt, st = time_align(a, 1, warm=1)
    par = parity_sample(a, list(range(0, n5, max(1, n5 // 8)))[:8], PEN, "cpu_wfa_score", orc, refcpu, 8000) if refcpu else "reference CPU WFA not built"
    bad_cigar = 0
    pen = wfagpu.AffinePenalties(*PEN)
    for i in range(0, n5, max(1, n5 // 32)):
        p, t = a.pair(i)
        bad_cigar += 0 if a.L.wfagpu_check_result(p.encode(), len(p), t.encode(), len(t), pen, a.error(i), a.cigar(i).encode()) else 1
    out["cfg5_50kbp_15pct_cigar_redispatch"] = entry(a, dt, st, par, {"invalid_cigars_in_sample": bad_cigar,
                                                                      "note": f"{n5} pairs on one GPU = one GPU's share of BASELINE's 20 000 over 8; the reference GPU code cannot run it (int16 offsets)"})
    a.destroy()
    return out


DUMP_CIGAR_PAIRS = 256


def dump_outputs(path, lib, wfagpu, a, out, ops):
    """What the last timed step returned to its caller, as .npy files for comparing two builds output for output:
    distance.npy   every pair's score (float64),
    n_ops.npy      every pair's number of backtrace operations (float64),
    cigar_index.npy / cigar.npy   a fixed sample of DUMP_CIGAR_PAIRS pairs (seeded) and their CIGAR text as
                   character codes (float32, one row per pair, zero-padded)."""
    import ctypes as C
    import numpy as np
    os.makedirs(path, exist_ok=True)
    n = a.num_pairs
    np.save(os.path.join(path, "distance.npy"), np.array([out[i].distance for i in range(n)], dtype=np.float64))
    np.save(os.path.join(path, "n_ops.npy"), np.array([out[i].n_ops for i in range(n)], dtype=np.float64))
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(DUMP_CIGAR_PAIRS, n), replace=False))
    free = C.CDLL(None).free
    free.argtypes = [C.c_void_p]
    base = C.addressof(ops.contents)
    texts = []
    for i in idx:
        p, t = (s.encode() for s in a.pair(int(i)))
        cg = wfagpu.Cigar()
        words = C.cast(base + 4 * out[i].ops_off, C.POINTER(C.c_uint32))
        assert lib.wfagpu_ops_to_cigar(p, len(p), t, len(t), out[i].distance, words, out[i].n_ops, C.byref(cg))
        texts.append(C.string_at(cg.buffer) if cg.buffer else b"")
        free(cg.buffer)
    codes = np.zeros((len(idx), max(map(len, texts), default=0)), dtype=np.float32)
    for r, s in enumerate(texts):
        codes[r, :len(s)] = np.frombuffer(s, dtype=np.uint8)
    np.save(os.path.join(path, "cigar_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(path, "cigar.npy"), codes)


def envelope_block(wfagpu, a, local):
    """Operating envelope around the steady-state numbers: cold first call, un-hinted provisioning, stale hint."""
    out = {}
    # (1) a context that never saw a batch: first call = allocations + rings sized for -e 3000; second = steady state
    code = (
        "import sys,time,json; sys.path.insert(0,%r); import wfagpu\n"
        "a=wfagpu.Aligner(); a.add_synthetic(%d,%d,%d,%f,%f); a.initialize_parameters(2,3,1)\n"
        "a.options.max_error=%d; a.options.compute_cigar=True\n"
        "ts=[]\n"
        "for _ in range(3):\n"
        "    a.reset_results(); t0=time.perf_counter(); a.align(); ts.append(time.perf_counter()-t0)\n"
        "print(json.dumps({'ts':ts,'st':a.run_stats()}))\n") % (os.path.join(ROOT, "wfa-gpu_b200", "python"), SEED, PAIRS_PER_GPU, LENGTH, ERR, ERR, MAX_ERROR)
    for key, env in (("fresh_process", {}), ("no_hint", {"WFAGPU_NO_HINT": "1"}), ("no_hint_no_prebound", {"WFAGPU_NO_HINT": "1", "WFAGPU_NO_PREBOUND": "1"})):
        try:
            pr = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(local)), **env),
                                capture_output=True, text=True, timeout=600)
            r = json.loads(pr.stdout.strip().splitlines()[-1])
            out[key] = {"call_1_alignments_per_s": round(PAIRS_PER_GPU / r["ts"][0], 1), "call_2_alignments_per_s": round(PAIRS_PER_GPU / r["ts"][1], 1),
                        "call_3_alignments_per_s": round(PAIRS_PER_GPU / r["ts"][2], 1), "redispatched_last_call": int(r["st"]["redispatched"])}
        except Exception as e:                                                  # pragma: no cover
            out[key] = {"error": str(e)[:200]}
    out["fresh_process"]["note"] = ("call 1 = cold (CUDA context, buffer allocation); every call sizes its rings from the score bounds of its own "
                                    "pairs (bound kernel first, one host round trip per chunk)")
    out["no_hint"]["note"] = "WFAGPU_NO_HINT=1: nothing remembered between calls; the rings still follow the batch's own score bounds"
    out["no_hint_no_prebound"]["note"] = ("WFAGPU_NO_HINT=1 WFAGPU_NO_PREBOUND=1: the policy before bound-first provisioning -- rings for the full "
                                          "-e 3000 budget, one resident CTA less per SM")
    # (2) stale hint: a 2 % batch teaches the library small scores, then the 5 % batch arrives
    low = make_aligner(wfagpu, SEED + 1, PAIRS_PER_GPU, LENGTH, 0.02, 0.02, PEN, max_error=MAX_ERROR, cigar=True)
    low.align()
    a.reset_results()
    t0 = time.perf_counter()
    a.align()
    dt = time.perf_counter() - t0
    st = a.run_stats()
    out["stale_hint"] = {"alignments_per_s": round(a.num_pairs / dt, 1), "redispatched": int(st["redispatched"]),
                         "note": "the headline 5 % batch right after a 2 % batch (the remembered scores are ~650): the rings follow the bounds of "
                                 "the batch itself, nothing is re-dispatched"}
    # the other direction: the 2 % batch right after the 5 % batch, against its own steady state
    low.reset_results()
    t0 = time.perf_counter()
    low.align()
    dt_after = time.perf_counter() - t0
    low.reset_results()
    t0 = time.perf_counter()
    low.align()
    dt_steady = time.perf_counter() - t0
    out["stale_hint_high"] = {"alignments_per_s": round(low.num_pairs / dt_after, 1), "steady_alignments_per_s": round(low.num_pairs / dt_steady, 1),
                              "redispatched": int(low.run_stats()["redispatched"]),
                              "note": "a 2 % batch right after the 5 % batch (remembered scores ~1600: where bounding every pair does not pay, a "
                                      "128-pair sample of bounds detects the stale memory) next to the same call repeated"}
    low.destroy()
    a.reset_results()
    a.align()                                                                    # leave the hint as the headline batch wants it
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    import wfagpu

    rank, world, local = dist_setup(args.gpus)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: this framework has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = wfagpu.load()
    wfagpu.set_devices(str(local))
    # torchrun pins OMP_NUM_THREADS=1 per rank; the library's result loop may use this rank's share of the host cores
    wfagpu.set_host_threads(max(1, min(4, len(os.sched_getaffinity(0)) // max(1, world))))

    a = make_aligner(wfagpu, shard_seed(rank), PAIRS_PER_GPU, LENGTH, ERR, ERR, PEN, max_error=MAX_ERROR, cigar=True)
    gcells_total = gcells(a)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident hot path: `value` ----------------------
    rb = wfagpu.ResidentBatch(a, device=local, slot=0)
    rb.upload()
    plan = rb.plan(cigar=True)
    for _ in range(args.warmup):
        rb.align(plan)
        rb.wait()
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    t0 = time.perf_counter()
    dev_ms = 0.0
    align_ms = 0.0
    wf_ms = 0.0
    pending = 0
    for _ in range(args.steps):
        rb.align(plan)
        mp, ma = rb.wait()
        dev_ms += mp + ma
        align_ms += ma
        st_step = rb.stats()
        wf_ms += st_step["ms_wavefront"]           # CUDA events around the wavefront kernel on its stream
        pending += st_step["pending_pairs"]        # pairs the timed pass left to the (untimed) re-dispatch tier
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.summary()
    st = rb.stats()
    # every pair must have finished inside the timed passes: nothing of the step is hidden in download()
    assert pending == 0, f"{pending} pairs were left to the re-dispatch tier outside the timed region"
    launches_per_step = st["launches"]
    out, ops, used = rb.download()
    scores = [out[i].distance for i in range(rb.n)]
    n_ops_total = sum(out[i].n_ops for i in range(rb.n))
    assert all(out[i].status & 1 for i in range(rb.n)), "unfinished pairs in the benchmark batch"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, lib, wfagpu, a, out, ops)
    rb.release()

    t_max, wall_max = reduce_max([dev_ms / 1e3, wall], device="cuda")
    total_pairs = PAIRS_PER_GPU * world * args.steps
    value = aggregate_value(PAIRS_PER_GPU, world, args.steps, t_max)

    # ---------------- end to end through the public C API: `e2e` -------------
    # exactly what an unmodified reference caller does: no batch size set, no buffer registered
    assert a.host_buffer_pinned(), "wfagpu_initialize_aligner should hand out page-locked memory on a GPU box"
    for _ in range(max(1, min(args.warmup, 2))):
        a.reset_results()
        a.align()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        a.reset_results()
        a.align()
    barrier()
    e2e_s = time.perf_counter() - t0
    rs = a.run_stats()
    (t_e2e_max,) = reduce_max([e2e_s], device="cuda")
    e2e_value = total_pairs / t_e2e_max
    # the e2e answer must be the resident answer
    assert [a.error(i) for i in range(0, a.num_pairs, 97)] == scores[::97]

    per_rank = gather_per_rank({"rank": rank, "ms_per_step": round(dev_ms / args.steps, 3), "wavefront_ms": round(wf_ms / args.steps, 3),
                                "e2e_ms_per_step": round(e2e_s * 1e3 / args.steps, 3), "redispatched_e2e": int(rs["redispatched"]),
                                "n_cap": st["n_cap"], "cta_threads": st["cta_threads"], "ctas": st["ctas"], "d_end": st["d_end"],
                                "max_score": max(scores), "mean_score": round(sum(scores) / len(scores), 1)}, world)

    # ---------------- (N > 1) one wfagpu_align call sharding over the N GPUs in-library -------------
    e2e_inlib = None
    if world > 1:
        # every rank gives its device memory back first (pooled contexts keep ~40 GB of snapshot arenas per GPU)
        lib.wfagpu_device_close_all()
        barrier()
        try:
            store = dist.distributed_c10d._get_default_store()      # host-side wait: no NCCL kernel spins on the idle GPUs
        except Exception:                                            # pragma: no cover
            store = None
        if rank == 0:
            try:
                wfagpu.set_host_threads(len(os.sched_getaffinity(0)))     # the other ranks are idle now
                big = make_aligner(wfagpu, SEED + 31, PAIRS_PER_GPU * world, LENGTH, ERR, ERR, PEN, max_error=MAX_ERROR, cigar=True)
                wfagpu.set_devices(f"n:{world}")
                dt, bst = time_align(big, max(1, min(args.steps, 3)), warm=2)
                wfagpu.set_devices(str(local))
                e2e_inlib = {"value": round(big.num_pairs / dt, 1), "unit": UNIT, "pairs_per_call": big.num_pairs, "devices": int(bst["devices"]),
                             "h2d_bytes_per_call": int(bst["h2d_bytes"]), "d2h_bytes_per_call": int(bst["d2h_bytes"]),
                             "api": f"ONE wfagpu_align call from rank 0 with WFAGPU_DEVICES=n:{world}: chunks handed to one host thread per GPU, results in results[i]"}
                big.destroy()
            except Exception as e:                                        # pragma: no cover
                e2e_inlib = {"error": str(e)[:300]}
            # BASELINE config 5 at its stated size on N GPUs: 2500 pairs per GPU (20 000 on 8) of 50 kbp / 15 % in ONE call
            if not args.quick and not args.no_configs:
                try:
                    n5 = int(os.environ.get("WFAGPU_BENCH_CFG5_PAIRS", 2500)) * world
                    a5 = make_aligner(wfagpu, 0xB2000005, n5, 50000, 0.15, 0.15, PEN, max_error=8000, cigar=True)
                    wfagpu.set_devices(f"n:{world}")
                    dt5, st5 = time_align(a5, 1, warm=1)
                    wfagpu.set_devices(str(local))
                    pen5 = wfagpu.AffinePenalties(*PEN)
                    bad5 = 0
                    for i in range(0, n5, max(1, n5 // 32)):
                        p5, t5 = a5.pair(i)
                        bad5 += 0 if lib.wfagpu_check_result(p5.encode(), len(p5), t5.encode(), len(t5), pen5, a5.error(i), a5.cigar(i).encode()) else 1
                    e2e_inlib["cfg5_50kbp_15pct_cigar_redispatch"] = {
                        "pairs": n5, "devices": int(st5["devices"]), "e2e_alignments_per_s": round(n5 / dt5, 1), "e2e_gcups": round(gcells(a5) / dt5 / 1e9, 1),
                        "wall_ms": round(dt5 * 1e3, 1), "redispatched": int(st5["redispatched"]), "failed_pairs": int(st5["failed_pairs"]),
                        "invalid_cigars_in_sample": bad5, "note": "ONE wfagpu_align call sharded in-library; first budget 8000 below every score"}
                    a5.destroy()
                except Exception as e:                                    # pragma: no cover
                    e2e_inlib["cfg5_50kbp_15pct_cigar_redispatch"] = {"error": str(e)[:300]}
            if store is not None:
                store.set("wfagpu_inlib_done", "1")
        elif store is not None:
            store.wait(["wfagpu_inlib_done"])
        if store is None:
            dist.barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_kind = hbm_peak()
    alg_bytes = algorithmic_bytes(a, n_ops_total)
    k_ms = (wf_ms or align_ms) / args.steps      # dominant kernel: wfa_quad_kernel, its own launch duration
    achieved = alg_bytes / (k_ms / 1e3) / 1e9
    cells_unpruned = cells_of_scores(lib, wfagpu, scores)           # what the reference's kernels compute for these scores
    cells = measured_cells(local) or cells_unpruned                 # cells the wavefront kernel computed in one step
    sm = lib.get_cuda_SM_count(local)
    clk = (clocks["sm_mhz"] or 1965) * 1e6
    int_peak = sm * 128 * clk
    roofline = {"bound": "issue", "kernel": "wfa_quad_kernel<bt>", "cells_per_launch": cells, "cells_without_pruning": cells_unpruned,
                "nominal_instr_per_cell": 64, "achieved": round(cells * 64 / (k_ms / 1e3) / 1e12, 3), "peak": round(int_peak / 1e12, 3),
                "unit": "T thread-instr/s", "frac": round(cells * 64 / (k_ms / 1e3) / int_peak, 4),
                "peak_kind": f"{sm} SMs x 128 lanes x sampled SM clock", "kernel_ms": round(k_ms, 3),
                "step_kernels_ms": round(align_ms / args.steps, 3), "gcells_per_s": round(cells / (k_ms / 1e3) / 1e9, 3),
                # SURVEY 8(d) defines the work unit with the reference's growth model (cells_without_pruning):
                # the same time against that work -- above 1 means fewer cells than the reference computes
                "frac_of_reference_work": round(cells_unpruned * 64 / (k_ms / 1e3) / int_peak, 4),
                "traffic": None,
                "note": "integer SIMT path (no contraction, no tensor cores); SURVEY 8(d): 64 thread instructions per cell with backtrace"}
    roofline_hbm = {"bound": "hbm", "achieved": round(achieved, 2), "peak": peak, "peak_kind": peak_kind, "unit": "GB/s",
                    "frac": round(achieved / peak, 6), "algorithmic_bytes_per_launch": alg_bytes, "traffic": None,
                    "note": "compulsory HBM traffic is ~31 KB/pair: not the binding roof"}
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_file):
        try:
            tr = json.load(open(traffic_file))
            roofline_hbm["traffic"] = roofline["traffic"] = int(tr["dram_bytes_per_pair"] * PAIRS_PER_GPU)
            roofline_hbm["traffic_note"] = tr.get("note", "ncu dram bytes per pair (profiles/traffic.json) x pairs per launch")
        except Exception:
            pass

    line = {
        "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(t_max * 1e3 / args.steps, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int16", "data": "synthetic",
        "config": config({"parallelism": f"pairs sharded over {world} GPU(s), no collective"}),
        "gcups": round(gcells_total * world * args.steps / t_max / 1e9, 1),
        "wall_ms_per_step": round(wall_max * 1e3 / args.steps, 3),
        "e2e": {"value": round(e2e_value, 1), "unit": UNIT,
                "h2d_bytes_per_step": int(rs["h2d_bytes"]), "d2h_bytes_per_step": int(rs["d2h_bytes"]),
                "gcups": round(gcells_total * world * args.steps / t_e2e_max / 1e9, 1),
                "api": "wfagpu_align on the aligner's own buffer, as an unmodified reference caller uses it: no extension call, default batch size "
                       "(page-locked by wfagpu_initialize_aligner; H2D, kernels, CIGAR text printed on the GPU, D2H, copy into results[i])"},
        "gpu_launches": int(launches_per_step * args.steps),
        "pending_after_timed_pass": int(pending),
        "hint_note": "rings of a step are sized from the score bounds of its own pairs (bound kernel first); what earlier calls needed only decides whether bounding pays and the first-pass budget beyond -e; see envelope for cold / un-hinted / stale-memory numbers",
        "clocks": clocks, "roofline": roofline, "roofline_hbm": roofline_hbm, "per_rank": per_rank,
    }
    if e2e_inlib:
        line["e2e_inlib"] = e2e_inlib

    if world == 1 and not args.quick:
        # launch_alignments on a buffer the caller allocated itself (pageable): staged through the slots' pinned buffers
        import ctypes as C
        n = a.s.sequences_buffer_len
        copy = C.create_string_buffer(n)
        C.memmove(copy, a.s.sequences_buffer, n)
        best = None
        for i in range(3):
            a.reset_results()
            t0 = time.perf_counter()
            lib.launch_alignments(copy, n, a.s.sequences_metadata, a.s.results, a.s.alignment_options, False)
            dt = time.perf_counter() - t0
            if i and (best is None or dt < best):
                best = dt
        pst = a.run_stats()
        line["e2e_pageable"] = {"value": round(a.num_pairs / best, 1), "unit": UNIT, "staged": int(pst["staged"]),
                                "api": "launch_alignments(buffer malloc'ed by the caller): every chunk copied into page-locked staging by the worker's host threads, then DMA"}
        del copy
        line["reference_gpu"] = reference_gpu_block(a)
        if line["reference_gpu"].get("value"):
            line["reference_gpu"]["e2e_speedup_over_reference_gpu"] = round(e2e_value / line["reference_gpu"]["value"], 1)
        line["envelope"] = envelope_block(wfagpu, a, local)
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(a, CPU_SAMPLE)
        a.destroy()
        lib.wfagpu_device_close_all()
        if not args.no_configs:
            line["configs"] = run_configs(wfagpu)
    elif world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(a, CPU_SAMPLE)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def cpu_baseline(a, sample):
    """The reference's CPU path (WFA2-lib v2.3 through utils/wfa_cpu.c, compiled into oracle/_ref)
    on the first `sample` pairs of the workload, all host threads."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle import RefCPU, Oracle
    n = min(sample, a.num_pairs)
    pairs = [a.pair(i) for i in range(n)]
    if RefCPU.available():
        r = RefCPU()
        threads = len(os.sched_getaffinity(0))          # all host cores (torchrun pins OMP_NUM_THREADS=1)
        t0 = time.perf_counter()
        errs, _ = r.align_batch([p for p, _ in pairs], [t for _, t in pairs], *PEN, cigar=True, threads=threads)
        dt = time.perf_counter() - t0
        for i in range(0, n, 37):
            assert errs[i] == a.error(i), "CPU reference and GPU scores differ"
        return {"value": round(n / dt, 1), "unit": UNIT, "cores": threads, "kind": "reference",
                "sample": f"first {n} pairs of the workload, CIGAR, wavefront_memory_low, OpenMP static",
                "seconds": round(dt, 2)}
    o = Oracle()
    n = min(n, 24)
    t0 = time.perf_counter()
    for p, t in pairs[:n]:
        o.align(p, t, *PEN, MAX_ERROR)
    dt = time.perf_counter() - t0
    return {"value": round(n / dt, 2), "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"first {n} pairs, scalar restatement", "seconds": round(dt, 2)}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores."""
    rank, world, local = dist_setup(args.gpus)
    if rank != 0:
        return
    import wfagpu
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle import RefCPU, Oracle
    a = wfagpu.Aligner()
    a.add_synthetic(SEED, REF_STEP_PAIRS, LENGTH, ERR, ERR)
    pairs = [a.pair(i) for i in range(a.num_pairs)]
    P, T = [p for p, _ in pairs], [t for _, t in pairs]
    if RefCPU.available():
        r = RefCPU()
        threads, kind = len(os.sched_getaffinity(0)), "reference"
        step = lambda: r.align_batch(P, T, *PEN, cigar=True, threads=threads)
        n = len(P)
    else:
        o = Oracle()
        threads, kind, n = 1, "port", 8
        step = lambda: [o.align(p, t, *PEN, MAX_ERROR) for p, t in pairs[:n]]
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    v = n * args.steps / dt
    gc = sum(len(p) * len(t) for p, t in pairs[:n]) * args.steps / dt / 1e9
    sample = f"{n} pairs per step (bounded sample of the workload), CIGAR, all host threads"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(v, 1), "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt * 1e3 / args.steps, 2),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": config({"parallelism": f"pairs sharded over {world} GPU(s), no collective"}), "sample_pairs_per_step": n,
        "gcups": round(gc, 2),
        "cpu_baseline": {"value": round(v, 1), "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": round(v, 1), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE configs 1-5 block (N = 1 only)")
    ap.add_argument("--quick", action="store_true", help="headline numbers only (no reference GPU, envelope, configs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step (rank 0's batch) to DIR/*.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
