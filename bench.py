"""
bench.py -- headline benchmark of the quantum-inferno B200 time-frequency path.

Workload (BASELINE.json north_star): fused order-3 Gabor CWT + power + Shannon information/entropy, fp32 planes,
CH_PER_GPU channels x 2^24 samples @ 800 Hz per GPU (60 bands) -- 64 x 2^24 on 8 GPUs, weak scaling by channel with no
data-path collective.  A step is one pass of the hot path over that resident batch.  QI_BENCH_DTYPE=float64 times the
reference-precision (fp64) path on the same records instead.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py ... --dump-outputs DIR                          # also save the last timed step's outputs (.npy)
    python bench.py --impl reference ...                            # CPU port of the reference (oracle), host cores
    torchrun --nproc-per-node N bench.py --gpus N ...               # one rank per GPU

Rank 0 prints ONE JSON line (contract in the task statement):
  value        TFR cells/s over all GPUs, inputs resident in HBM, CUDA-event time, max over ranks
  e2e          same metric through the public API from pinned host memory (H2D of the records and D2H of the
               entropy / power summaries inside the timed region), over the same K steps
  roofline     dominant kernel (largest live CUDA-event share) against the measured HBM copy peak
  cpu_baseline the oracle timed on one host core (N = 1 only)
  check        results of the run compared OUTSIDE the timed region with the numpy oracle (single bands of channel 0
               at full size, the whole config[0]-sized call) and with an fp64 recomputation of the entropy from the
               planes; a failed comparison aborts the bench
  configs      device-timed secondary configurations run after the headline: BASELINE configs[3] share (order 6,
               8 ch x 2^22) and, for N > 1, configs[4]-shaped band sharding of ONE long record (order 12) with its single
               NCCL all-reduce of the total power
  dump_outputs (with --dump-outputs DIR) the files written to DIR: what the last timed step returned to its caller on
               rank 0, so that two builds run with the same arguments can be compared output for output
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FS = 800.0
ORDER = 3
LOG2_N = int(os.environ.get("QI_BENCH_LOG2N", "24"))
CH_PER_GPU = int(os.environ.get("QI_BENCH_CHANNELS", "8"))
DTYPE = os.environ.get("QI_BENCH_DTYPE", "float32")         # 'float32' (headline, SURVEY 8d) or 'float64'
HOST_CHUNKS = int(os.environ.get("QI_BENCH_HOST_CHUNKS", "4"))
METHOD = os.environ.get("QI_BENCH_METHOD", "auto")          # 'auto' = what the public API picks; 'exact' forces the FFT passes
SHARD_LOG2_N = int(os.environ.get("QI_BENCH_SHARD_LOG2N", "25"))
EXTRAS = os.environ.get("QI_BENCH_EXTRAS", "1") != "0"
CHECKS = os.environ.get("QI_BENCH_CHECKS", "1") != "0"
ITEM = {"float32": 4, "float64": 8}[DTYPE]
KERNEL_OF = {
    "multirate": {"fft_fwd": "mr_table_kernel+mr_pyramid3_kernel+mr_decimate_kernel",
                  "inv_first": "mr_level2k_kernel[levels>=1]+mr_expand_kernel<MID>",
                  "inv_mid": "mr_level2k_kernel[level 0]", "inv_last": "mr_expand_kernel<POWER_INFO>",
                  "info": "mr_info_rows_kernel"},
    "exact": {"fft_fwd": "fft_pass_kernel[forward]", "inv_first": "fft_pass_kernel[spectrum x response]",
              "inv_mid": "fft_pass_kernel[middle]", "inv_last": "fft_pass_kernel[slice + power]",
              "info": "shannon_kernel"}}
METRIC = "tfr_cells_per_s"
UNIT = "cells/s"


def alg_bytes_per_cell(n_bands):
    """SURVEY 8(d): power + information planes + the record's share."""
    return 2 * ITEM + ITEM / float(n_bands)


def workload_config(world, n_bands):
    """The `config` object of the JSON line -- identical for both arms (the reference arm times a bounded sample of it)."""
    return {"workload": f"north_star: N=3 Gabor CWT + power + info + entropy, {CH_PER_GPU} ch/GPU x 2^{LOG2_N} samples "
                        f"@ 800 Hz, {'fp32' if DTYPE == 'float32' else 'fp64'} planes",
            "channels_total": world * CH_PER_GPU, "bands": n_bands,
            "parallelism": f"channel-sharded x{world}, no data-path collective",
            "l2": "inputs (0.5 GB) and planes (64 GB) per step are far larger than L2; no flush needed"}


def csrc_sha():
    """Hash of the kernel sources: profiles/traffic.json is only quoted while it matches."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "quantum_inferno_b200", "csrc")
    for fn in sorted(os.listdir(d)):
        if fn.endswith((".cu", ".cuh", ".h")):
            h.update(fn.encode())
            h.update(open(os.path.join(d, fn), "rb").read())
    return h.hexdigest()[:16]


# ----------------------------------------------------------------------------- synthetic input (SURVEY 8d)
def synth_channel_numpy(n, chan):
    k = np.arange(n, dtype=np.float64)
    f_c = 60.0 * 2.0 ** ((chan % 12) / 12.0)
    dur = n / FS
    chirp = 0.5 * np.cos(2 * np.pi * (1.0 * k / FS + 0.5 * (199.0 / dur) * (k / FS) ** 2))
    noise = np.random.default_rng(1234 + chan).standard_normal(n) * 2.0 ** -4
    return np.cos(2 * np.pi * f_c / FS * k) + chirp + noise


def synth_batch_device(rt, n, chans, dtype="float32"):
    """Records made where they are consumed: tone and linear chirp by the library's device generator
    (qi_synth_chirp, float64 phase arithmetic), noise by torch's seeded device generator."""
    from quantum_inferno_b200 import _driver
    torch = rt.torch
    tdt = getattr(torch, dtype)
    out = torch.empty(len(chans), n, dtype=tdt, device=rt.device)
    dur = n / FS
    for i, c in enumerate(chans):
        f_c = 60.0 * 2.0 ** ((c % 12) / 12.0)
        tone = _driver.synth_chirp(n, "float64", 2 * np.pi * f_c / FS, rt=rt)[0]
        # cos(2 pi (t + 0.5 (199 / dur) t^2)), t = k / fs:  omega k + half_gamma (k / fs)^2
        chirp = _driver.synth_chirp(n, "float64", 2 * np.pi * 1.0 / FS, half_gamma=np.pi * 199.0 / dur, chirp_scale=FS,
                                    rt=rt)[0]
        g = torch.Generator(device=rt.device).manual_seed(1234 + c)
        noise = torch.randn(n, dtype=torch.float64, device=rt.device, generator=g) * 2.0 ** -4
        out[i] = (tone + 0.5 * chirp + noise).to(tdt)
    return out


def synth_batch_torch(torch, n, chans, dev, dtype="float32"):
    """Same records for the scripts under tools/ (which pass the torch module and a device)."""
    from quantum_inferno_b200 import _runtime
    with torch.cuda.device(dev):
        return synth_batch_device(_runtime.get_runtime(), n, chans, dtype)


# ----------------------------------------------------------------------------- CPU port (oracle) timing
def cpu_baseline_single(log2n=None):
    """~10-30 s of single-threaded CPU work on a bounded sample of the same workload."""
    from oracle import qi_oracle as orc
    log2n = int(os.environ.get("QI_BENCH_CPU_LOG2N", "20")) if log2n is None else log2n
    n = 1 << log2n
    x = synth_channel_numpy(n, 0)
    t0 = time.perf_counter()
    r = orc.cwt_power_entropy(ORDER, x, FS)
    dt = time.perf_counter() - t0
    cells = r["power"].shape[0] * n
    return {"value": cells / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"oracle/qi_oracle.cwt_power_entropy (numpy fp64 restatement of styx_cwt + tfr_info), channel 0, "
                      f"first 2^{log2n} samples ({cells // n} bands), {dt:.1f} s",
            "samples_per_s": n / dt}


_REF_CACHE = {}


def _oracle_band_job(args):
    """One band of one full-length record the way the reference computes it (styx_cwt.py:195 transforms the record once
    PER BAND: fftconvolve on the tiled signal), followed by |.|^2 and the information of that row."""
    chan, band, log2n = args
    from oracle import qi_oracle as orc
    n = 1 << log2n
    key = (chan, log2n)
    if key not in _REF_CACHE:
        _REF_CACHE.clear()
        _REF_CACHE[key] = (synth_channel_numpy(n, chan), orc.log_frequency_hz_from_fft_points(FS, n, ORDER))
    x, freq = _REF_CACHE[key]
    xf = np.fft.fft(x, 2 * n)
    row = orc.cwt_band(xf, ORDER, n, freq[band], FS)
    p = np.abs(row) ** 2
    s = float(p.sum())
    info = -np.log2(p / s + np.finfo(np.float64).eps)
    return n, float(np.sum(p / s * info))


def run_reference_arm(args):
    """bench.py --impl reference: the reference's CPU algorithm (numpy port -- the Python reference itself cannot travel
    to the GPU box) on the host cores, on the bench's own record shape.  A step = one band of a 2^LOG2_N-sample record
    per worker process (bands spread over the 60-band table of channel 0); cells/s = cells of those rows / wall time."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    log2n = int(os.environ.get("QI_BENCH_REF_LOG2N", str(LOG2_N)))
    n = 1 << log2n
    from oracle import qi_oracle as orc
    n_bands = len(orc.log_frequency_hz_from_fft_points(FS, n, ORDER))
    n_bands_config = len(orc.log_frequency_hz_from_fft_points(FS, 1 << LOG2_N, ORDER))
    # ~3 GB of fp64 work arrays per worker at 2^24 (record spectrum, atom, its spectrum, product)
    per_worker = 48 * (2 * n) * 1.25
    try:
        import psutil
        mem_cap = int(psutil.virtual_memory().available * 0.6 / per_worker)
    except Exception:                          # noqa: BLE001
        mem_cap = 8
    cores = max(1, min(os.cpu_count() or 1, int(os.environ.get("QI_BENCH_CPU_PROCS", "32")), mem_cap, n_bands))
    bands = [int(round(i * (n_bands - 1) / max(1, cores - 1))) for i in range(cores)]
    jobs = [(0, b, log2n) for b in bands]
    # single-thread figure first (BASELINE.md section 3: single-thread and all-core)
    _oracle_band_job(jobs[len(jobs) // 2])                       # builds the record, warms numpy's FFT plan
    t0 = time.perf_counter()
    _oracle_band_job(jobs[len(jobs) // 2])
    single = n / (time.perf_counter() - t0)
    with mp.get_context("fork").Pool(cores) as pool:
        for _ in range(max(1, min(args.warmup, 2))):
            pool.map(_oracle_band_job, jobs, chunksize=1)
        t0 = time.perf_counter()
        cells = 0
        for _ in range(args.steps):
            cells += sum(c for c, _ in pool.map(_oracle_band_job, jobs, chunksize=1))
        dt = time.perf_counter() - t0
    value = cells / dt
    sample = (f"{cores} worker processes x 1 band each of channel 0's 2^{log2n}-sample record per step (bands "
              f"{bands[0]}..{bands[-1]} of {n_bands}; numpy fp64 port of styx_cwt + |.|^2 + information, record FFT "
              f"repeated per band as the reference's fftconvolve on the tiled signal does); warm-up capped at 2 steps")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.gpus, n_bands_config),
            "samples_per_s": value / n_bands,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                             "single_thread_value": single, "host_cpus": os.cpu_count()},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(prefix="qi_clocks_", suffix=".csv")
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in open(self.path):
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2])); power.append(float(parts[3]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(power)),
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------- our arm
def _l2(a, b):
    return float(np.linalg.norm(np.asarray(a, dtype=np.float64) - b) / np.linalg.norm(b))


def checks_rank0(torch, cwt_entropy, x, power, info, r, n, n_bands):
    """Outside the timed region: the step's own outputs against the numpy oracle and an fp64 recomputation."""
    from oracle import qi_oracle as orc
    tol_l2 = 1e-4 if DTYPE == "float32" else 1e-10
    tol_bits = 1e-3 if DTYPE == "float32" else 1e-9
    out = {"tolerance_power_l2": tol_l2, "tolerance_entropy_bits": tol_bits}
    # (1) entropy of channel 0 recomputed in fp64 from the power plane the step wrote
    s = float(r.total_power[0].item())
    ent = 0.0
    eps = float(np.finfo(np.float64).eps)
    for b in range(n_bands):
        pdf = power[0, b].double() / s
        ent += float((pdf * -torch.log2(pdf + eps)).sum().item())
    got = float(r.entropy_bits()[0].item())
    out["entropy_bits_ch0"] = got
    out["entropy_bits_ch0_recomputed_fp64"] = ent
    assert abs(got - ent) < tol_bits, ("fused entropy differs from the fp64 recomputation", got, ent)
    # (2) single bands of channel 0 at full size against the oracle (band 0 is a record-long truncated atom)
    xh = x[0].double().cpu().numpy()
    xf = np.fft.fft(xh, 2 * n)
    freq = r.frequency_hz
    band_l2 = {}
    for b in (0, n_bands // 2):
        row = np.abs(orc.cwt_band(xf, ORDER, n, freq[b], FS)) ** 2
        band_l2[str(b)] = _l2(power[0, b].double().cpu().numpy(), row)
        assert band_l2[str(b)] < tol_l2, ("band power differs from the oracle", b, band_l2[str(b)])
        ref_info = -np.log2(row / s + eps)
        strong = row > 1e-2 * row.max()
        d_info = float(np.max(np.abs(info[0, b].double().cpu().numpy() - ref_info)[strong]))
        assert d_info < (1e-3 if DTYPE == "float32" else 1e-8), ("information plane differs from the oracle", b, d_info)
        band_l2[f"info_{b}"] = d_info
    out["oracle_band_power_l2"] = band_l2
    del xf
    # (3) BASELINE configs[0]: the whole call at 2^16 samples against the whole oracle
    n1 = 1 << 16
    x1 = synth_channel_numpy(n1, 0)
    ref = orc.cwt_power_entropy(ORDER, x1, FS)
    r1 = cwt_entropy.cwt_power_entropy(ORDER, torch.from_numpy(x1).to(x.device), FS, dtype=DTYPE)
    p1 = r1.power[0].double().cpu().numpy()
    out["config0_power_l2"] = _l2(p1, ref["power"])
    out["config0_per_band_l2_max"] = float(np.max(np.linalg.norm(p1 - ref["power"], axis=1) /
                                                  np.linalg.norm(ref["power"], axis=1)))
    out["config0_entropy_abs_diff_bits"] = abs(float(r1.entropy_bits()[0].item()) - ref["entropy_bits"])
    assert out["config0_per_band_l2_max"] < tol_l2 and out["config0_entropy_abs_diff_bits"] < tol_bits, out
    out["passed"] = True
    return out


DUMP_PLANE_BYTES = 24 << 20       # per [C, B, N] plane: power + info + the per-band arrays stay under 64 MB in all


def plane_sample_index(shape, itemsize, seed=0):
    """Flat indices of the cells of a [C, B, N] plane that --dump-outputs saves: None (the whole plane) when it fits
    DUMP_PLANE_BYTES, else a uniform sample drawn from a fixed seed (sorted, repeats dropped), so that two runs with the
    same arguments save the same cells."""
    total = int(np.prod(shape))
    k = DUMP_PLANE_BYTES // itemsize
    if total <= k:
        return None
    return np.unique(np.random.default_rng(seed).integers(0, total, size=k))


def dump_outputs(torch, r, out_dir):
    """Save what the step returned to its caller as out_dir/<name>.npy (float32 / float64): the per-band and
    per-record arrays whole, the power and information planes whole or as the sample of plane_sample_index."""
    os.makedirs(out_dir, exist_ok=True)
    idx = plane_sample_index(r.power.shape, r.power.element_size())
    arrays = {"frequency_hz": np.asarray(r.frequency_hz, dtype=np.float64), "band_power": r.band_power,
              "total_power": r.total_power, "band_entropy_bits": r.band_entropy_bits, "entropy_bits": r.entropy_bits()}
    if idx is None:
        arrays["power"], arrays["info"] = r.power, r.info
    else:
        flat = torch.from_numpy(idx).to(r.power.device)
        arrays["power"], arrays["info"] = r.power.reshape(-1)[flat], r.info.reshape(-1)[flat]
    nbytes = 0
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else a
        np.save(os.path.join(out_dir, name + ".npy"), a)
        nbytes += a.nbytes
    cells = int(np.prod(r.power.shape))
    return {"dir": out_dir, "files": sorted(n + ".npy" for n in arrays), "bytes": nbytes,
            "planes": "whole" if idx is None else
                      f"{len(idx)} of {cells} cells of the flattened {list(r.power.shape)} plane, drawn with "
                      "numpy default_rng(0) (bench.plane_sample_index)"}


def timed_calls(torch, fn, reps, dist, dev):
    """Device time per call (ms), max over ranks, after one untimed call."""
    fn()
    torch.cuda.synchronize(dev)
    if dist is not None:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        res = fn()
    e1.record()
    torch.cuda.synchronize(dev)
    t = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.float64, device=dev)
    mine = float(t.item())
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), mine, res


def secondary_configs(torch, rt, dist, rank, world, dev):
    """Device-timed secondary configurations (inputs resident, planes written), run after the headline buffers are freed."""
    from quantum_inferno_b200 import cwt_entropy, distributed
    out = {}
    # ---- BASELINE configs[3] share: order 6, 2^22-sample records, 8 channels per GPU (256 channels need 32 GPUs' worth)
    n4, c4 = 1 << 22, 8
    x4 = synth_batch_device(rt, n4, [rank * c4 + i for i in range(c4)])
    nb4 = len(cwt_entropy.scales.log_frequency_hz_from_fft_points(FS, n4, 6))
    p4 = torch.empty(c4, nb4, n4, dtype=torch.float32, device=dev)
    i4 = torch.empty_like(p4)
    ms, _, _ = timed_calls(torch, lambda: cwt_entropy.cwt_power_entropy(6, x4, FS, dtype="float32", out_power=p4, out_info=i4),
                           5, dist, dev)
    out["config3_share"] = {"workload": f"order 6 CWT + info/entropy, {c4} ch/GPU x 2^22 samples, {nb4} bands, fp32",
                            "ms_per_call": ms, "cells_per_s": world * c4 * nb4 * n4 / (ms * 1e-3)}
    del x4, p4, i4
    torch.cuda.empty_cache()
    if world == 1:
        return out
    # ---- BASELINE configs[4] shape: ONE long record, order 12, bands sharded over the ranks, one all-reduce of S
    n5 = 1 << SHARD_LOG2_N
    x5 = synth_batch_device(rt, n5, [1000])                       # same seed on every rank: the same record
    freq5 = cwt_entropy.scales.log_frequency_hz_from_fft_points(FS, n5, 12)
    nb5 = len(freq5)
    ar = distributed.sum_allreduce()

    # this rank's planes are allocated once and handed back to every timed call (like the headline's): the caching
    # allocator otherwise ping-pongs between two 30 GB sets and an occasional cudaMalloc lands inside the timed calls
    # (observed: 9 ms or 14 ms per call from one run to the next)
    first = distributed.cwt_power_entropy_band_sharded(12, x5, FS, allreduce=ar, dtype="float32")
    pw5, in5 = first.power, first.info
    del first

    def sharded():
        return distributed.cwt_power_entropy_band_sharded(12, x5, FS, allreduce=ar, dtype="float32", out_power=pw5,
                                                          out_info=in5)

    calls0 = ar.calls
    ms, mine, r5 = timed_calls(torch, sharded, 3, dist, dev)
    per_call = (ar.calls - calls0) // 4
    times = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
    dist.all_gather(times, torch.tensor([mine], dtype=torch.float64, device=dev))
    rank_ms = [float(t.item()) for t in times]
    ent = r5.entropy_bits().clone()
    dist.all_reduce(ent)                                          # verification only, outside the timed path
    b0, b1 = r5.band_slice
    shard = {"workload": f"one record of 2^{SHARD_LOG2_N} samples, order 12, {nb5} bands band-sharded over {world} GPUs, "
                         f"fp32 power + info planes", "ms_per_call": ms, "cells_per_s": nb5 * n5 / (ms * 1e-3),
             "allreduce_calls": int(per_call), "rank_ms": rank_ms,
             "cost_model_imbalance_max_over_mean": max(rank_ms) / (sum(rank_ms) / len(rank_ms)),
             "entropy_bits": float(ent[0].item())}
    if rank == 0:
        from oracle import qi_oracle as orc
        xh = x5[0].double().cpu().numpy()
        xf = np.fft.fft(xh, 2 * n5)
        row = np.abs(orc.cwt_band(xf, 12, n5, freq5[b0], FS)) ** 2
        shard["oracle_band_l2"] = {str(b0): _l2(r5.power[0, 0].double().cpu().numpy(), row)}
        assert shard["oracle_band_l2"][str(b0)] < 1e-4, shard
        del xf, row
    total_sharded = float(r5.total_power[0].item())
    del r5, pw5, in5
    torch.cuda.empty_cache()
    if rank == 0:
        # the same record unsharded on one GPU: entropy and total power must agree
        full = cwt_entropy.cwt_power_entropy(12, x5, FS, dtype="float32")
        shard["entropy_abs_diff_vs_unsharded"] = abs(float(full.entropy_bits()[0].item()) - shard["entropy_bits"])
        shard["total_power_rel_diff_vs_unsharded"] = abs(float(full.total_power[0].item()) - total_sharded) / total_sharded
        assert shard["entropy_abs_diff_vs_unsharded"] < 1e-3, shard
        del full
    torch.cuda.empty_cache()
    dist.barrier()
    out["config4_band_sharded"] = shard
    return out


def run_gpu_arm(args):
    # the contract is ONE JSON line on stdout: route anything libraries print to fd 1 (e.g. the NCCL banner) to stderr
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    import torch
    from quantum_inferno_b200 import _lib, _numa, _plan, _runtime, cwt_entropy

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU port)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # host placement: this rank's CPUs and pinned staging memory on the NUMA node of its GPU
    numa = _numa.bind_to_gpu_numa_node(local) if os.environ.get("QI_BENCH_NUMA", "1") != "0" else {"bound": False, "why": "off"}
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)
    rt = _runtime.get_runtime()
    lib = rt.lib

    n = 1 << LOG2_N
    chans = [rank * CH_PER_GPU + i for i in range(CH_PER_GPU)]
    x = synth_batch_device(rt, n, chans, DTYPE)                       # resident input, C*N*item bytes (> L2)
    freq = cwt_entropy.scales.log_frequency_hz_from_fft_points(FS, n, ORDER)
    n_bands = len(freq)
    tdt = getattr(torch, DTYPE)
    multirate = DTYPE == "float32" and METHOD != "exact"
    n_level0 = int(np.count_nonzero(_plan.multirate_bands(ORDER, n, freq, FS, "norm")[0]["level"] == 0))
    cells_per_step_gpu = CH_PER_GPU * n_bands * n
    power = torch.empty(CH_PER_GPU, n_bands, n, dtype=tdt, device=dev)
    info = torch.empty_like(power)

    def step(src, **kw):
        return cwt_entropy.cwt_power_entropy(ORDER, src, FS, dtype=DTYPE, out_power=power, out_info=info,
                                             method=METHOD, **kw)

    def sync_all():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        r = step(x)
    sync_all()

    # ---- timed region: K steps, inputs resident in HBM
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    lib.qi_profile_enable(1)
    launches0 = lib.qi_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    for _ in range(args.steps):
        r = step(x)
    e1.record()
    sync_all()
    elapsed_ms = e0.elapsed_time(e1)
    launches = lib.qi_launch_count() - launches0
    lib.qi_profile_enable(0)
    cat_ms = (np.zeros(_lib.QI_N_CATEGORIES), np.zeros(_lib.QI_N_CATEGORIES, dtype=np.int64))
    lib.qi_profile_read(cat_ms[0].ctypes.data, cat_ms[1].ctypes.data)
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    # before the end-to-end steps below write the same planes again
    dumped = dump_outputs(torch, r, args.dump_outputs) if args.dump_outputs and rank == 0 else None

    # ---- end to end through the public API: pinned host records -> H2D -> kernels -> D2H of the summaries, K steps
    x_host = torch.empty(CH_PER_GPU, n, dtype=tdt, pin_memory=True)
    x_host.copy_(x)
    step(x_host, host_chunks=HOST_CHUNKS)
    sync_all()
    # the box's plain pinned-host -> HBM bandwidth for the same buffer: the floor of any end-to-end number
    xd_probe = torch.empty_like(x)
    e0.record()
    xd_probe.copy_(x_host, non_blocking=True)
    e1.record()
    sync_all()
    h2d_gbps = x_host.numel() * ITEM / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del xd_probe
    e0.record()
    d2h = 0
    for _ in range(args.steps):
        rr = step(x_host, host_chunks=HOST_CHUNKS)
        outs = [rr.band_entropy_bits.cpu(), rr.band_power.cpu(), rr.total_power.cpu()]
        d2h = sum(o.numel() * o.element_size() for o in outs)
    e1.record()
    sync_all()
    clocks = sampler.stop() if rank == 0 else None
    t2 = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_ms = float(t2.item()) / args.steps

    # ---- correctness of what was just timed (rank 0; the others wait), then the secondary configurations
    check = None
    if CHECKS and rank == 0:
        r = step(x)
        check = checks_rank0(torch, cwt_entropy, x, power, info, r, n, n_bands)
    if dist is not None:
        dist.barrier()
    del power, info, x_host, r, rr
    x = None
    torch.cuda.empty_cache()
    extras = secondary_configs(torch, rt, dist, rank, world, dev) if (EXTRAS and DTYPE == "float32") else {}

    if rank == 0:
        ms_per_step = elapsed_ms / args.steps
        value = world * cells_per_step_gpu / (ms_per_step * 1e-3)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except (OSError, ValueError):
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "6650 GB/s (of fallback)"
        bpc = alg_bytes_per_cell(n_bands)
        # dominant kernel = the category with the largest summed device time in the timed region
        dom = int(np.argmax(cat_ms[0]))
        dom_name = _lib.CATEGORY_NAMES[dom]
        dom_launches = int(cat_ms[1][dom])
        dom_avg_ms = float(cat_ms[0][dom] / max(1, dom_launches))
        # cells the dominant category's launches process per step: the expand launches of the multirate path write the
        # bands of level >= 1 only (the level-0 rows are written by the level-0 convolution + the information pass)
        dom_cells_step = cells_per_step_gpu
        if multirate and dom_name == "inv_last":
            dom_cells_step = CH_PER_GPU * (n_bands - n_level0) * n
        cells_per_launch = dom_cells_step * args.steps / max(1, dom_launches)
        achieved = bpc * cells_per_launch / (dom_avg_ms * 1e-3) / 1e9
        traffic, traffic_note = None, "no ncu capture on record"
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            key = "multirate" if multirate else ("exact" if DTYPE == "float32" else "float64")
            if tj.get("csrc_sha") == csrc_sha():
                per_step = tj[key].get(dom_name + "_per_step")
                if per_step is not None:                      # bytes of the category per STEP -> per launch like `achieved`
                    traffic = per_step * args.steps / max(1, dom_launches)
                    traffic_note = tj[key].get("_note", "")
            else:
                traffic_note = "profiles/traffic.json was captured from other kernel sources (csrc hash differs): not quoted"
        except (OSError, ValueError, KeyError):
            pass
        path = "multirate" if multirate else "exact"
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if DTYPE == "float32" else "f64", "data": "synthetic (device-generated: qi_synth_chirp + seeded noise)",
            "config": workload_config(world, n_bands),
            "algorithm": path,
            "samples_per_s": world * CH_PER_GPU * n / (ms_per_step * 1e-3),
            "roofline": {"bound": "hbm", "kernel": KERNEL_OF[path].get(dom_name, dom_name),
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src,
                         "avg_launch_ms": dom_avg_ms, "launches": dom_launches,
                         "cells_per_launch": cells_per_launch, "alg_bytes_per_cell": bpc,
                         "step_frac": bpc * cells_per_step_gpu / (ms_per_step * 1e-3) / 1e9 / peak,
                         "category_ms_per_step": {nm: float(ms) / args.steps for nm, ms in zip(_lib.CATEGORY_NAMES, cat_ms[0])}},
            "cpu_baseline": cpu_baseline_single() if world == 1 else None,
            "e2e": {"value": world * cells_per_step_gpu / (e2e_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": int(CH_PER_GPU * n * ITEM), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_ms, "steps": args.steps, "h2d_gbps_measured": h2d_gbps,
                    "h2d_floor_ms": CH_PER_GPU * n * ITEM / (h2d_gbps * 1e9) * 1e3, "numa": numa,
                    "note": f"public API cwt_entropy.cwt_power_entropy(host_chunks={HOST_CHUNKS}) on pinned host records (H2D of the "
                            "next channel group overlaps the kernels of the current one); the planes (64 GB per step) stay "
                            "in HBM for the consumers of SURVEY 8(f)3, the entropy / band-power / total-power summaries "
                            "are read back"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "check": check,
            "configs": extras,
        }
        if dumped is not None:
            line["dump_outputs"] = dumped
        json_out.write(json.dumps(line) + "\n")
        json_out.flush()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, save what the last one computed as DIR/<name>.npy (rank 0's channels; "
                         "the planes as a fixed sample, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs saves the outputs of the CUDA path (--impl b200)")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
