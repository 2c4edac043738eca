#!/usr/bin/env python
"""bench.py -- headline benchmark of the barcode-assignment hot path.

Workload (BASELINE.json configs[1], SURVEY.md section 8d "config 2"): synthetic 10 M x 150 bp
single-end reads per GPU, 96 barcodes of 24 nt with injected indels/mismatches,
:semiglobal with the reference's default options.  A "step" = one pass of the hot
path over the whole 10 M-read batch.

  value : reads/s, whole job, reads already resident in HBM (kernels only)
  e2e   : reads/s through the C ABI with HOST (pinned) buffers: H2D of every batch,
          kernels, D2H of the per-read results, all inside the timed region
  --impl reference : the reference's CPU algorithm (oracle port, all host threads)
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
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

READ_LEN = 150
N_BARCODES = 96
BARCODE_LEN = 24
SEED = 0x42444D58  # "BDMX"
CU_PER_READ = N_BARCODES * BARCODE_LEN * READ_LEN          # full-matrix cell updates (SURVEY 8d)
OPS_PER_READ = 17 * N_BARCODES * ((BARCODE_LEN + 31) // 32) * READ_LEN   # algorithmic int-ops (SURVEY 8d)
BYTES_PER_READ = READ_LEN + 4 + 20                         # sequence + offset in, bdx_result out
CHUNK = 4000                                               # reference chunk_size (core.jl:521)
# DRAM traffic of the dominant kernel from the committed `ncu --set full` capture
# (profiles/r01g_kernels_ncu_summary.txt: k_filter<1,3,0,1>, 4 M-read step, 516 667 reads through the
# automaton): dram__bytes_read.sum 164.03 MB + dram__bytes_write.sum 16.11 MB.  Per read that is 2x the
# algorithmic 174 B: worklist-scattered 150-byte reads touch 6 32-byte sectors, offsets / PassOut one each.
NCU_FILTER_DRAM_BYTES_PER_READ = (164.026880e6 + 16.110336e6) / 516667
# the same for k_seed_var's complete level, the kernel that now takes those reads in config 2
# (profiles/r02_kernels_ncu_summary.txt: 4 M-read step, 746 917 reads: 222.07 MB read + 21.04 MB written)
NCU_SEEDVAR_DRAM_BYTES_PER_READ = (222.070016e6 + 21.044992e6) / 746917
# k_seed (config 2 runs one level of it), per read of its input (same capture: 2 155 000 reads left by the
# prefilter; 497.53 MB read + 37.23 MB written)
NCU_SEED_DRAM_BYTES_PER_READ = (497.526784e6 + 37.233920e6) / 2155000
DUMP_SAMPLE = 1_000_000      # reads whose results --dump-outputs writes: 5 x 4 MB of float32 + 8 MB of indices


def make_config():
    import bdx_b200 as bdx
    rng = np.random.default_rng(SEED)
    alpha = np.frombuffer(b"ACGT", dtype=np.uint8)
    bcs = [bytes(alpha[rng.integers(0, 4, BARCODE_LEN)]).decode() for _ in range(N_BARCODES)]
    return bdx.DemuxConfig(bc_seqs=bcs, bc_lengths_no_N=[BARCODE_LEN] * N_BARCODES,
                           ids=[f"bc{i:03d}" for i in range(N_BARCODES)])


def synth_spec(first_read: int):
    from bdx_b200 import capi
    return capi.SynthSpec(seed=SEED, first_read=first_read, read_len=READ_LEN, plant_permille=900,
                          start_lo=1, start_hi=120, n_permille_x10=50, set2_mode=0, end_lo=0, end_hi=0)


def numpy_reads(cfg, n, seed):
    """CPU stand-in for the device generator (same distribution, used only when no GPU is visible)."""
    import synth
    rng = np.random.default_rng(seed)
    reads = synth.random_reads(rng, n, cfg.bc_seqs, min_len=READ_LEN, plant=0.9, start_hi=119, n_prob=0.005)
    blob = np.frombuffer(b"".join(reads), dtype=np.uint8).copy()
    off = np.arange(n + 1, dtype=np.int64) * READ_LEN
    return blob, off


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed regions (B200_PROFILING.md).  One nvidia-smi process
    runs from before the warm-up (its start-up takes longer than a short timed region); only the samples that
    arrive inside a marked window [begin(), end()] are kept."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines, self.windows, self._t0 = index, None, [], [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def begin(self):
        self._t0 = time.perf_counter()

    def end(self):
        if self._t0 is not None:
            self.windows.append((self._t0, time.perf_counter()))
            self._t0 = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            if not any(a <= ts <= b for a, b in self.windows):
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons),
                "windows": "device-resident timed region + e2e timed region"}


def bind_to_gpu_numa_node(local: int):
    """Pin this rank's threads (and with them its pinned host allocations, which the kernel places on the local
    node) to the NUMA node the GPU hangs off: H2D / D2H of several ranks then do not cross the socket
    interconnect.  Best effort; returns a short description for the JSON line."""
    if os.environ.get("BDX_NUMA_BIND", "1") == "0":
        return "off"
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(local)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dev = bus.lower()
        if len(dev.split(":")[0]) == 8:          # nvml prints an 8-digit domain, sysfs uses 4
            dev = dev[4:]
        node = int(open(f"/sys/bus/pci/devices/{dev}/numa_node").read())
        if node < 0:
            return "gpu has no NUMA node"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return f"node {node}: none of its cpus allowed"
        os.sched_setaffinity(0, cpus)
        return f"node {node} ({len(cpus)} cpus)"
    except Exception as exc:
        return f"unavailable ({type(exc).__name__})"


def dump_outputs(out_dir, res):
    """Writes the per-read results `res` (bdx_result records) as <out_dir>/<field>.npy in float32 (every field is a
    small integer, exact in float32) for a fixed, seeded sample of DUMP_SAMPLE reads, and <out_dir>/read_index.npy
    (float64) with the indices of those reads.  The reads come from a seeded generator, so two builds run with the
    same arguments can be compared file for file."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(res)
    idx = np.arange(n) if n <= DUMP_SAMPLE else np.sort(np.random.default_rng(SEED).choice(n, DUMP_SAMPLE, replace=False))
    np.save(os.path.join(out_dir, "read_index.npy"), idx.astype(np.float64))
    for f in res.dtype.names:
        np.save(os.path.join(out_dir, f"{f}.npy"), res[f][idx].astype(np.float32))


def oracle_rate(cfg, blob, off64, threads):
    """reads/s of the oracle port over (blob, off64) with `threads` workers, chunked like
    the reference (4000 reads per task)."""
    import orc
    o = orc.Oracle(cfg)
    n = len(off64) - 1
    spans = [(a, min(a + CHUNK, n)) for a in range(0, n, CHUNK)]

    def work(span):
        a, b = span
        sub_off = off64[a:b + 1] - off64[a]
        o.classify(blob[off64[a]:off64[b]], sub_off)
        return b - a

    t0 = time.perf_counter()
    if threads == 1:
        done = sum(work(s) for s in spans)
    else:
        with ThreadPoolExecutor(threads) as ex:
            done = sum(ex.map(work, spans))
    dt = time.perf_counter() - t0
    return done / dt, dt


def sample_reads_host(cfg, n_sample, rank=0):
    """n_sample reads of the workload's distribution, on the host, as (uint8 blob, int64 offsets).  numpy only:
    the reference arm maps no library of this repository other than the oracle it times."""
    blob, off = numpy_reads(cfg, n_sample, SEED)
    return blob, off, "numpy generator (same distribution as the device generator: 90 % planted, P(k edits) of SURVEY 8d)"


def calibrate_sample(cfg, threads, seconds, lo=20000, hi=2_000_000):
    blob, off, _ = sample_reads_host(cfg, 8000)
    r1, _ = oracle_rate(cfg, blob, off, 1)
    n = int(r1 * threads * seconds * 0.8)
    n = max(lo, min(hi, n))
    return (n + CHUNK - 1) // CHUNK * CHUNK, r1


STATED_READS = {"3": 50_000_000, "4": 50_000_000, "5s": 200_000_000, "5h": 200_000_000, "5e": 200_000_000}
CONFIG_BATCH = 10_000_000          # reads per device batch (offsets are int32: a batch stays below 2^31 bytes)


def measure_config(key, cfg, sp, name, total_reads, rank, world, local, parity_seconds, parity_reads):
    """One BASELINE.json config at its stated size: `total_reads` reads of READ_LEN bases, sharded contiguously
    over the ranks (SURVEY.md section 8d), generated on the device batch by batch (not timed) and classified
    device-resident (timed with CUDA events on the library's compute stream).  Rank 0 checks the first reads of
    its shard against the multi-threaded oracle."""
    import torch
    import torch.distributed as dist
    import bdx_b200 as bdx
    from bdx_b200 import capi
    import bench_configs
    import orc

    per_rank = total_reads // world
    first = rank * per_rank
    B = min(CONFIG_BATCH, per_rank)
    config = capi.Config(cfg)
    st = capi.Stream(config, device=local, max_reads=0, max_bytes=0)
    ext = torch.cuda.ExternalStream(st.cuda_stream, device=torch.device("cuda", local))
    d_seq = torch.empty(B * READ_LEN, dtype=torch.uint8, device="cuda")
    d_off = torch.empty(B + 1, dtype=torch.int32, device="cuda")
    d_res = torch.empty(B * bdx.RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    res_i32 = d_res.view(torch.int32).view(-1, 5)

    def gen(k, nb):
        spec = capi.SynthSpec(seed=bench_configs.SEED, first_read=first + k * B, read_len=READ_LEN, plant_permille=900,
                              n_permille_x10=50, **sp)
        st.synth_device(spec, nb, d_seq.data_ptr(), d_off.data_ptr())
        st.sync()

    # warm-up on the first batch (also what the parity check looks at)
    nb0 = min(B, per_rank)
    gen(0, nb0)
    for _ in range(2):
        st.classify_device(d_seq.data_ptr(), d_off.data_ptr(), nb0, d_res.data_ptr())
    st.sync()
    parity = None
    if rank == 0:
        o = orc.Oracle(cfg)
        k = parity_reads
        if not k:                      # as many reads as the oracle finishes in about parity_seconds on this host
            probe = 4000 if len(cfg.bc_seqs) < 1000 else 800
            blob = d_seq[:probe * READ_LEN].cpu().numpy()
            t0 = time.perf_counter()
            o.classify_mt(blob, np.arange(probe + 1, dtype=np.int64) * READ_LEN)
            rate = probe / (time.perf_counter() - t0)
            k = int(max(20_000, min(1_000_000, rate * parity_seconds)))
        k = min(k, nb0)
        blob = d_seq[:k * READ_LEN].cpu().numpy()
        got = np.frombuffer(d_res[:k * bdx.RESULT_DTYPE.itemsize].cpu().numpy().tobytes(), dtype=bdx.RESULT_DTYPE)
        t0 = time.perf_counter()
        want = o.classify_mt(blob, np.arange(k + 1, dtype=np.int64) * READ_LEN)
        dt = time.perf_counter() - t0
        ok = all((got[f] == want[f]).all() for f in ("status", "bc1", "bc2", "keep_start", "keep_end"))
        parity = {"reads_checked": k, "bit_exact": bool(ok), "oracle_reads_per_s": k / dt, "oracle_threads": os.cpu_count()}
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms, matched, ambiguous, launches = 0.0, 0, 0, 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    done = 0
    k = 0
    while done < per_rank:
        nb = min(B, per_rank - done)
        if k > 0 or nb != nb0:
            gen(k, nb)
        l0 = st.launch_count
        e0.record(ext)
        st.classify_device(d_seq.data_ptr(), d_off.data_ptr(), nb, d_res.data_ptr())
        e1.record(ext)
        st.sync()
        ms += e0.elapsed_time(e1)
        launches += st.launch_count - l0
        stt = res_i32[:nb, 0]
        matched += int((stt == 0).sum().item())
        ambiguous += int((stt == 2).sum().item())
        done += nb
        k += 1
    # one more pass over the last batch with per-stage CUDA events and the work counters (not timed above)
    st.profile(True)
    st.work_counters(reset=True)
    st.classify_device(d_seq.data_ptr(), d_off.data_ptr(), nb, d_res.data_ptr())
    stage_ms = {k2: v[0] for k2, v in st.profile_read_stages().items() if v[1]}
    st.profile(False)
    wc = st.work_counters(reset=True)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([matched, ambiguous, launches], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    st.close()
    del d_seq, d_off, d_res
    secs = float(t.item()) * 1e-3
    reads = per_rank * world
    out = {"workload": name, "reads": reads, "reads_per_gpu": per_rank, "sharding": "contiguous shards, no data-path collective",
           "scaling": "strong", "reads_per_sec": reads / secs, "gcups": reads / secs * bench_configs.cell_updates(cfg) / 1e9,
           "seconds": secs, "matched_fraction": int(cnt[0].item()) / reads, "ambiguous_fraction": int(cnt[1].item()) / reads,
           "gpu_launches": int(cnt[2].item()), "parity": parity,
           "last_batch": {"reads": nb, "stage_ms": stage_ms,
                          "reads_by_path": {"prefilter": wc[0], "seed": wc[1], "automaton": wc[2]},
                          "verified_hit_columns": wc[3]}}
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = make_config()
    threads = os.cpu_count() or 1
    per_step_s = 6.0
    n_sample, r1 = calibrate_sample(cfg, threads, per_step_s)
    blob, off, how = sample_reads_host(cfg, n_sample)
    times = []
    for i in range(args.warmup + args.steps):
        _, dt = oracle_rate(cfg, blob, off, threads)
        if i >= args.warmup:
            times.append(dt)
    total = sum(times)
    value = n_sample * len(times) / total
    line = {
        "impl": "reference", "metric": "reads_per_sec", "value": value, "unit": "reads/s",
        "gcups": value * CU_PER_READ / 1e9, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": f"config2: RATE over a {n_sample}-read sample of the 10M x {READ_LEN}bp job (a CPU step over all "
                               f"10M reads would take minutes), {N_BARCODES} barcodes x {BARCODE_LEN}nt, :semiglobal defaults",
                   "sample_reads": n_sample,
                   "note": "C restatement of BioDemuX.jl classification.jl (oracle port), all host threads; "
                           "Julia is not installed in this image so the reference itself cannot run"},
        "cpu_baseline": {"value": value, "unit": "reads/s", "cores": threads, "kind": "port",
                         "sample": f"{n_sample} reads per step; {how}", "single_thread_reads_per_s": r1},
        "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def run_ours(args):
    import torch
    import torch.distributed as dist
    import bdx_b200 as bdx
    from bdx_b200 import capi

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path")
    numa = bind_to_gpu_numa_node(local) if world > 1 else "single rank: not bound"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n = args.reads
    cfg = make_config()
    config = capi.Config(cfg, debug=args.debug_flags)
    stream = capi.Stream(config, device=local, max_reads=args.e2e_batch, max_bytes=args.e2e_batch * READ_LEN)
    ext = torch.cuda.ExternalStream(stream.cuda_stream, device=torch.device("cuda", local))

    d_seq = torch.empty(n * READ_LEN, dtype=torch.uint8, device="cuda")
    d_off = torch.empty(n + 1, dtype=torch.int32, device="cuda")
    d_res = torch.empty(n * bdx.RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    stream.synth_device(synth_spec(rank * n), n, d_seq.data_ptr(), d_off.data_ptr())
    stream.sync()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        stream.classify_device(d_seq.data_ptr(), d_off.data_ptr(), n, d_res.data_ptr())

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # ---- device-resident: value + roofline of the dominant kernel -------------------------
    for _ in range(args.warmup):
        step()
    stream.sync()
    peak_ops = capi.C.c_double()
    capi._check(stream.lib.bdx_int_alu_peak(local, capi.C.byref(peak_ops)))
    barrier()
    sampler.begin()
    stream.profile(True)
    stream.path_counters(reset=True)
    l0 = stream.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ext)
    for _ in range(args.steps):
        step()
    e1.record(ext)
    stream.sync()
    barrier()
    sampler.end()
    ms = e0.elapsed_time(e1)
    launches = stream.launch_count - l0
    stages = stream.profile_read_stages()
    filt_ms, filt_n = stages["k_filter"]
    stream.profile(False)
    (pre_reads, seed_reads, auto_reads, hit_cols, sv_in_reads, seed_qmers, seed_ver_cols, sv_positions,
     sv_filter_diags) = stream.work_counters(reset=True)
    auto_per_launch = auto_reads / max(filt_n, 1)       # reads that actually ran the DP automaton
    clocks = None
    if args.no_e2e and rank == 0:
        clocks = sampler.stop()
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * n * args.steps / (ms_max * 1e-3)

    # ---- sanity on the timed results (parity proper lives in tests/) -----------------------
    res = np.frombuffer(d_res.cpu().numpy().tobytes(), dtype=bdx.RESULT_DTYPE)
    matched = int((res["status"] == 0).sum())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res)

    if args.no_e2e:
        if rank == 0:
            filt_s = filt_ms * 1e-3 / max(filt_n, 1)
            print(json.dumps({"value": value, "ms_per_step": ms_max / args.steps, "kernel_ms": filt_s * 1e3,
                              "matched_fraction": matched / n, "peak_Tops": peak_ops.value / 1e12,
                              "achieved_Tops": OPS_PER_READ * auto_per_launch / filt_s / 1e12,
                              "prefilter_fraction": pre_reads / max(pre_reads + seed_reads + auto_reads, 1),
                              "seed_fraction": seed_reads / max(pre_reads + seed_reads + auto_reads, 1), "clocks": clocks,
                              "stage_ms_per_step": {k: v[0] / args.steps for k, v in stages.items() if v[1]}}))
        stream.close()
        return

    # ---- e2e through the C ABI with host buffers ------------------------------------------
    B = args.e2e_batch
    nb = n // B
    h_seq = torch.empty(n * READ_LEN, dtype=torch.uint8, pin_memory=True)
    h_seq.copy_(d_seq)
    h_off = torch.empty(B + 1, dtype=torch.int32, pin_memory=True)
    h_off.copy_(d_off[:B + 1])
    torch.cuda.synchronize()
    seq_np, off_np = h_seq.numpy(), h_off.numpy()
    e2e_matched = 0

    DEPTH = int(os.environ.get("BDX_E2E_DEPTH", "4"))  # batches kept in flight (BDX_MAX_IN_FLIGHT = 4)

    def submit_bytes(k):
        stream.submit(seq_np[k * B * READ_LEN:(k + 1) * B * READ_LEN], off_np, tag=k, pinned=True)

    def e2e_steps(n_steps, submit=submit_bytes):
        """n_steps passes over the workload as ONE pipeline of batches: every batch is copied H2D from pinned
        host memory, classified, its results copied D2H and read by the host; DEPTH batches are in flight,
        the pipeline is drained at the end (inside the timed region), not between steps."""
        nonlocal e2e_matched
        m = 0
        queued = 0
        for _ in range(n_steps):
            for k in range(nb):
                submit(k)
                queued += 1
                if queued == DEPTH:
                    _, r = stream.fetch(copy=False)
                    m += int(np.count_nonzero(r["bc1"]))      # the host reads every result record
                    queued -= 1
        while queued:
            _, r = stream.fetch(copy=False)
            m += int(np.count_nonzero(r["bc1"]))
            queued -= 1
        e2e_matched = m

    e2e_steps(max(1, min(args.warmup, 2)))
    # what the host link gives a plain pinned H2D copy of one batch (the e2e path's own bound)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d_probe = torch.empty(B * READ_LEN, dtype=torch.uint8, device="cuda")
    d_probe.copy_(h_seq[:B * READ_LEN], non_blocking=True)
    torch.cuda.synchronize()
    # (one pass over the WHOLE pinned workload, like a step of the pipeline: on virtualised hosts a copy that cycles
    # over a few hundred MB runs up to twice as fast as one that streams gigabytes -- DMA address translation)
    p0.record()
    for k in range(nb):
        d_probe.copy_(h_seq[k * B * READ_LEN:(k + 1) * B * READ_LEN], non_blocking=True)
    p1.record()
    torch.cuda.synchronize()
    pcie_h2d_gbs = nb * B * READ_LEN / (p0.elapsed_time(p1) * 1e-3) / 1e9
    # the same copy issued by ALL ranks at once (barrier first): what the box's host memory / PCIe complex gives N
    # GPUs together is the ceiling the N-GPU e2e number has to be read against
    barrier()
    p0.record()
    for k in range(2 * nb):
        d_probe.copy_(h_seq[(k % nb) * B * READ_LEN:(k % nb + 1) * B * READ_LEN], non_blocking=True)
    p1.record()
    torch.cuda.synchronize()
    conc = torch.tensor([2 * nb * B * READ_LEN / (p0.elapsed_time(p1) * 1e-3) / 1e9], dtype=torch.float64, device="cuda")
    conc_all = [conc.clone() for _ in range(world)]
    if world > 1:
        dist.all_gather(conc_all, conc)
    conc_per_rank = [float(x.item()) for x in conc_all]
    del d_probe
    barrier()
    sampler.begin()                           # second sampling window: the e2e timed region
    t0 = time.perf_counter()
    e2e_steps(args.steps)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    sampler.end()
    if rank == 0:
        clocks = sampler.stop()
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * nb * B * args.steps / float(t.item())
    assert e2e_matched == args.steps * int((res["status"][:nb * B] == 0).sum()), "e2e and device-resident results disagree"

    # ---- the same pipeline fed with 4-bit packed reads (bdx_submit_packed4_pinned): half the H2D bytes.  The reads
    # are packed once, outside the timed region -- packing is what a reader does INSTEAD of copying the sequence
    # bytes into the staging buffer (bdx_pack_reads4 runs at memcpy speed; its rate is reported) ----
    e2e_packed = None
    if not args.no_packed:
        h_packed = torch.empty(n * READ_LEN // 2 + 16, dtype=torch.uint8, pin_memory=True)
        packed_np = h_packed.numpy()
        tp = time.perf_counter()
        for k in range(nb):
            config.pack4(seq_np[k * B * READ_LEN:(k + 1) * B * READ_LEN], packed_np[k * B * READ_LEN // 2:(k + 1) * B * READ_LEN // 2])
        pack_gbs = nb * B * READ_LEN / (time.perf_counter() - tp) / 1e9

        def submit_packed(k):
            stream.submit_packed4(packed_np[k * B * READ_LEN // 2:(k + 1) * B * READ_LEN // 2], off_np, tag=k, pinned=True)

        e2e_steps(1, submit_packed)
        barrier()
        t0 = time.perf_counter()
        e2e_steps(args.steps, submit_packed)
        torch.cuda.synchronize()
        tpk = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tpk, op=dist.ReduceOp.MAX)
        assert e2e_matched == args.steps * int((res["status"][:nb * B] == 0).sum()), "packed e2e and device-resident results disagree"
        e2e_packed = {"value": world * nb * B * args.steps / float(tpk.item()), "unit": "reads/s",
                      "h2d_bytes_per_step": nb * (B * READ_LEN // 2 + 4 * (B + 1)),
                      "d2h_bytes_per_step": nb * B * bdx.RESULT_DTYPE.itemsize,
                      "api": "bdx_submit_packed4_pinned / bdx_fetch_view", "host_pack_gbs_one_thread": pack_gbs,
                      "note": "reads packed to 4-bit codes by the reader (bdx_pack_reads4, outside the timed region: it replaces "
                              "the reader's copy into the staging buffer); results identical to the byte input"}
        del h_packed

    # ---- one host process driving all GPUs of the job through bdx_pool (the Julia host's shape, core.jl:454-466):
    # rank 0 deals the batches round-robin over the ranks' devices while the other ranks wait ----
    pool_line = None
    if not args.no_pool:
        barrier()
        if rank == 0:
            devs = list(range(world))
            pool = capi.Pool(config, devs, streams_per_device=2, max_reads=B, max_bytes=B * READ_LEN)
            cap = len(devs) * 2 * 3

            readers = ThreadPoolExecutor(4)       # the host still reads every result record (numpy drops the GIL)

            def pool_pass(n_steps):
                counts, queued = [], 0
                for _ in range(n_steps):
                    for k in range(nb):
                        pool.submit(seq_np[k * B * READ_LEN:(k + 1) * B * READ_LEN], off_np, tag=k, pinned=True)
                        queued += 1
                        if queued == cap:
                            _, r = pool.fetch(copy=False)
                            counts.append(readers.submit(lambda v: int(np.count_nonzero(v["bc1"])), r))
                            queued -= 1
                while queued:
                    _, r = pool.fetch(copy=False)
                    counts.append(readers.submit(lambda v: int(np.count_nonzero(v["bc1"])), r))
                    queued -= 1
                return sum(c.result() for c in counts)

            pool_pass(1)
            for dv in devs:
                torch.cuda.synchronize(dv)
            t0 = time.perf_counter()
            m = pool_pass(args.steps)
            for dv in devs:
                torch.cuda.synchronize(dv)
            dtp = time.perf_counter() - t0
            assert m == args.steps * int((res["status"][:nb * B] == 0).sum())
            pool_line = {"n_gpus": world, "reads_per_sec": args.steps * nb * B / dtp, "streams_per_device": 2,
                         "batches_in_flight": cap, "api": "bdx_pool_submit_pinned / bdx_pool_fetch_view, ONE host process and "
                         "thread, one pinned copy of the workload on rank 0's NUMA node"}
            pool.close()
            torch.cuda.set_device(local)
        barrier()

    # ---- N > 1: the one collective of the path -- DemuxStats counters summed over GPUs ------
    stats_ms = None
    if world > 1:
        scfg = capi.Config(cfg, want_stats=True)
        sst = capi.Stream(scfg, device=local, max_reads=0, max_bytes=0)
        ns = min(n, 1_000_000)
        d_det = torch.empty(2 * ns * bdx.DETAIL_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
        sst.classify_device(d_seq.data_ptr(), d_off.data_ptr(), ns, d_res.data_ptr(), d_det.data_ptr())
        sst.sync()
        L = scfg.layout.total_len

        class _DevBuf:  # zero-copy torch view of the stream's device counters
            __cuda_array_interface__ = {"shape": (L,), "typestr": "<i8", "version": 2,
                                        "data": (sst.stats_device_ptr, False)}

        counters = torch.as_tensor(_DevBuf(), device="cuda")
        torch.cuda.synchronize()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        dist.all_reduce(counters, op=dist.ReduceOp.SUM)
        c1.record()
        torch.cuda.synchronize()
        stats_ms = c0.elapsed_time(c1)
        assert int(counters[0].item()) == world * ns
        sst.close()

    # ---- the data-dependence of the headline on record: the same workload with NO barcode planted, i.e. every read
    # has to run the full-range automaton (k_filter) to prove "no barcode" ----
    floor = None
    if not args.no_floor:
        nf = min(n, 2_000_000)
        fspec = synth_spec(rank * n)
        fspec.plant_permille = 0
        stream.synth_device(fspec, nf, d_seq.data_ptr(), d_off.data_ptr())
        stream.sync()
        for _ in range(2):
            stream.classify_device(d_seq.data_ptr(), d_off.data_ptr(), nf, d_res.data_ptr())
        stream.sync()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(ext)
        for _ in range(args.steps):
            stream.classify_device(d_seq.data_ptr(), d_off.data_ptr(), nf, d_res.data_ptr())
        f1.record(ext)
        stream.sync()
        tf = torch.tensor([f0.elapsed_time(f1) / args.steps], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tf, op=dist.ReduceOp.MAX)
        floor = {"reads_per_sec": world * nf / (float(tf.item()) * 1e-3), "reads_per_gpu": nf,
                 "workload": "config2 reads with plant_permille = 0: no read carries a barcode, all of them run the "
                             "full-range automaton (the rate when nothing can be short-cut)"}
    # ---- BASELINE.json configs 3, 4, 5 at their stated sizes (device-resident, sharded over the ranks).  Each is timed
    # as one pass over its stated read count (the whole job is the unit those configs are quoted in), not per --steps ----
    others = None
    if not args.no_configs:
        import bench_configs
        del d_seq, d_off, d_res
        torch.cuda.empty_cache()
        others = {}
        for key, (ocfg, sp, name) in bench_configs.configs().items():
            if args.configs and key not in args.configs:
                continue
            total = int(STATED_READS[key] * args.config_scale)
            total -= total % world
            others[key] = measure_config(key, ocfg, sp, name, total, rank, world, local, args.parity_seconds,
                                         args.parity_reads)

    if rank == 0:
        hbm_peak = None
        try:
            hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
            hbm_src = "MEASURED_PEAKS.json"
        except Exception:
            hbm_peak, hbm_src = 6650.0, "fallback (B200_PROFILING.md)"
        # ---- roofline of the DOMINANT kernel of the step (the stage with the most CUDA-event time).  All candidates
        # are bound by integer-ALU issue, not by HBM (1.5 GB of reads per step is 0.2 ms of HBM time).  Their
        # algorithmic units, counted on the device (bdx_stream_work_counters) and priced in int-ops (DESIGN.md 4.5):
        #   k_filter              17 x barcodes x columns for every read that ran the full-range automaton (SURVEY 8d)
        #   k_seed (levels 1-2)    8 x q-mers probed (rolling-hash step + bitmap test) + 17 x window columns verified
        #   k_seed_var (complete) 24 x (read, position) pairs scanned (a 5-mer code, two table look-ups)
        #                         + 10 x diagonals the 3-gram filter tested + 17 x window columns verified
        # The seed kernels do far LESS arithmetic than the automaton they replace -- that is their point -- so their
        # fraction of the ALU peak is small by construction; the reads they decide would have cost 244 800 int-ops
        # each in k_filter, which is reported next to it as the survey-convention figure.
        stage_names = {"k_seed_deep": "k_seed_var (complete level)", "k_seed": "k_seed"}
        dom = max((k for k in stages if stages[k][1]), key=lambda k: stages[k][0])
        dom_ms, dom_n = stages[dom]
        dom_s = dom_ms * 1e-3 / max(dom_n, 1)             # average duration of one launch of it
        if dom == "k_filter":
            units = OPS_PER_READ * auto_reads / max(dom_n, 1)
            dom_reads = auto_reads / max(dom_n, 1)
            traffic = NCU_FILTER_DRAM_BYTES_PER_READ * dom_reads
            how = "17 int-ops x 96 barcodes x 150 columns x reads that ran the automaton (device counter)"
        elif dom == "k_seed_deep":
            units = (24.0 * sv_positions + 10.0 * sv_filter_diags + 17.0 * hit_cols) / max(dom_n, 1)
            dom_reads = sv_in_reads / max(dom_n, 1)           # what k_prefilter and k_seed's levels left: it decides nearly all
            traffic = NCU_SEEDVAR_DRAM_BYTES_PER_READ * dom_reads
            how = ("24 int-ops x (read, position) pairs scanned + 10 x 3-gram-filter diagonals + 17 x window columns verified "
                   "(device counters bdx_stream_work_counters[7], [8], [3])")
        elif dom == "k_seed":
            units = (8.0 * seed_qmers + 17.0 * seed_ver_cols) / max(dom_n, 1)
            dom_reads = (n - pre_reads / max(stages["k_prefilter"][1], 1)) if stages.get("k_prefilter", (0, 0))[1] else n
            traffic = NCU_SEED_DRAM_BYTES_PER_READ * dom_reads
            how = ("8 int-ops x q-mers probed + 17 x window columns verified, average of its launches "
                   "(device counters bdx_stream_work_counters[5], [6]); reads_per_launch = the first level's input")
        else:
            units, dom_reads, traffic, how = None, None, None, "no algorithmic unit defined for this stage"
        achieved_ops = units / dom_s if units and dom_s > 0 else 0.0
        roof = {"bound": "int_alu", "achieved": achieved_ops / 1e12, "peak": peak_ops.value / 1e12, "unit": "Tint-op/s",
                "frac": achieved_ops / peak_ops.value if peak_ops.value else None,
                "kernel": stage_names.get(dom, dom), "kernel_ms": dom_s * 1e3, "kernel_share_of_step": dom_ms / ms if ms else None,
                "algorithmic_unit": how,
                "stage_ms_per_step": {k: v[0] / args.steps for k, v in stages.items() if v[1]},
                "reads_by_path_per_step": {"prefilter": pre_reads / args.steps, "seed_kernels": seed_reads / args.steps,
                                           "automaton": auto_reads / args.steps},
                "peak_source": "bdx_int_alu_peak: LOP3/IADD3 chains measured live on this GPU (dual-pipe issue peak)"}
        roof["traffic"] = traffic
        roof["traffic_unit"] = ("DRAM bytes per launch: ncu dram__bytes_read.sum + dram__bytes_write.sum per read of this kernel "
                                "(profiles/r02_kernels_ncu_summary.txt) x its reads per launch here")
        roof["reads_per_launch"] = dom_reads
        roof["work_units_per_step"] = {k: v / args.steps for k, v in {
            "k_seed_qmers_probed": seed_qmers, "k_seed_columns_verified": seed_ver_cols,
            "k_seed_var_positions_scanned": sv_positions, "k_seed_var_filter_diagonals": sv_filter_diags,
            "k_seed_var_columns_verified": hit_cols, "k_seed_var_input_reads": sv_in_reads}.items()}
        if dom in ("k_seed_deep", "k_seed"):
            roof["survey_convention"] = {"achieved": OPS_PER_READ * dom_reads / dom_s / 1e12 if dom_s > 0 else None,
                                         "what": "244 800 int-ops (the full 96 x 150 matrix, SURVEY 8d) per read this kernel decides / its "
                                                 "time: what the lane-per-barcode automaton would have had to do for the same reads"}
        hbm_gbs = BYTES_PER_READ * (dom_reads or 0) / dom_s / 1e9 if dom_s > 0 else 0.0
        step_gbs = BYTES_PER_READ * n / (ms_max / args.steps * 1e-3) / 1e9
        roof["hbm"] = {"achieved": hbm_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_gbs / hbm_peak, "peak_source": hbm_src,
                       "bytes_per_read": BYTES_PER_READ, "what": "the dominant kernel: algorithmic bytes of ITS reads / its time",
                       "whole_step_gbs": step_gbs}
        # the lane-per-barcode automaton where it still dominates: config 5 :semiglobal (1 536 barcodes)
        if others and "5s" in others and "k_filter" in others["5s"]["last_batch"]["stage_ms"]:
            lb = others["5s"]["last_batch"]
            ops5 = 17 * 1536 * READ_LEN
            a5 = ops5 * lb["reads_by_path"]["automaton"] / (lb["stage_ms"]["k_filter"] * 1e-3)
            roof["k_filter_on_config5"] = {"achieved": a5 / 1e12, "frac": a5 / peak_ops.value if peak_ops.value else None,
                                           "kernel_ms": lb["stage_ms"]["k_filter"], "reads": lb["reads_by_path"]["automaton"],
                                           "ops_per_read": ops5, "share_of_its_step": lb["stage_ms"]["k_filter"] / sum(lb["stage_ms"].values())}
        line = {
            "metric": "reads_per_sec", "value": value, "unit": "reads/s", "gcups": value * CU_PER_READ / 1e9,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32",
            "data": "synthetic",
            "config": {"workload": f"config2: {n} x {READ_LEN}bp reads per GPU, {N_BARCODES} barcodes x "
                                   f"{BARCODE_LEN}nt, :semiglobal defaults (max_error_rate 0.2, unit costs)",
                       "reads_per_gpu": n, "l2": "inputs (1.5 GB of reads per step) exceed the 126 MB L2",
                       "matched_fraction": matched / n, "e2e_batch_reads": B},
            "roofline": roof,
            "e2e": {"value": e2e_value, "unit": "reads/s", "h2d_bytes_per_step": nb * (B * READ_LEN + 4 * (B + 1)),
                    "d2h_bytes_per_step": nb * B * bdx.RESULT_DTYPE.itemsize,
                    "api": f"bdx_submit_pinned / bdx_fetch_view, {DEPTH} batches in flight",
                    "h2d_gbs_achieved": e2e_value / world * (READ_LEN + 4) / 1e9, "numa_binding_rank0": numa,
                    "h2d_gbs_plain_memcpy": pcie_h2d_gbs,
                    "h2d_gbs_concurrent_per_rank": conc_per_rank, "h2d_gbs_concurrent_aggregate": sum(conc_per_rank),
                    "reads_per_sec_at_concurrent_h2d_ceiling": sum(conc_per_rank) * 1e9 / (READ_LEN + 4),
                    # weak scaling gives every rank the same reads: the job ends with the rank whose link is slowest
                    "reads_per_sec_at_slowest_rank_h2d": world * min(conc_per_rank) * 1e9 / (READ_LEN + 4),
                    "bound": "host link: every read is 154 B of H2D; a bare pinned cudaMemcpyAsync of the same "
                             "bytes runs at h2d_gbs_plain_memcpy on this box"},
            "gpu_launches": launches, "clocks": clocks,
        }
        if stats_ms is not None:
            line["stats_allreduce_ms"] = stats_ms
        if e2e_packed is not None:
            line["e2e_packed"] = e2e_packed
        if pool_line is not None:
            line["pool_single_process"] = pool_line
        if floor is not None:
            line["floor"] = floor
        if others is not None:
            line["configs"] = others
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            n_sample, r1 = calibrate_sample(cfg, threads, 12.0)
            blob = seq_np[:n_sample * READ_LEN]
            off64 = np.arange(n_sample + 1, dtype=np.int64) * READ_LEN
            rate, dt = oracle_rate(cfg, blob, off64, threads)
            line["cpu_baseline"] = {"value": rate, "unit": "reads/s", "cores": threads, "kind": "port",
                                    "sample": f"first {n_sample} reads of the same workload, {dt:.1f} s, "
                                              f"chunks of {CHUNK}; C restatement of classification.jl "
                                              "(Julia unavailable in image)",
                                    "gcups": rate * CU_PER_READ / 1e9, "single_thread_reads_per_s": r1}
        print(json.dumps(line))
    stream.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=10_000_000, help="reads per GPU (config 2: 10 M)")
    ap.add_argument("--e2e-batch", type=int, default=500_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="device-resident timing only (kernel experiments)")
    ap.add_argument("--debug-flags", type=int, default=0, help="BDX_DEBUG_* (kernel experiments only)")
    ap.add_argument("--no-floor", action="store_true", help="skip the no-barcode (all-automaton) rate")
    ap.add_argument("--no-packed", action="store_true", help="skip the 4-bit packed-input e2e leg")
    ap.add_argument("--no-pool", action="store_true", help="skip the single-process bdx_pool leg")
    ap.add_argument("--no-configs", action="store_true", help="skip BASELINE.json configs 3 / 4 / 5")
    ap.add_argument("--configs", nargs="*", default=None, help="subset of 3 4 5s 5h 5e")
    ap.add_argument("--config-scale", type=float, default=1.0, help="fraction of the stated read counts (1.0 = 50 M / 50 M / 200 M)")
    ap.add_argument("--parity-seconds", type=float, default=15.0, help="oracle time per config for the parity sample")
    ap.add_argument("--parity-reads", type=int, default=0, help="parity sample size per config (0 = by --parity-seconds)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the CUDA path's per-read results of the last timed step (rank 0's reads; a seeded "
                         f"sample of {DUMP_SAMPLE} of them) to DIR/<field>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the CUDA path's results; it does not apply to --impl reference")
    if args.reads % args.e2e_batch:
        args.e2e_batch = args.reads
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
