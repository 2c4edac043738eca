#!/usr/bin/env python
"""Search-window input (bdx_submit_windows) against the whole-read inputs, on three workloads: config 3 (dual,
150-base reads, 1:40 / end-39:end), 3 kb reads with one 1:120 range, and the same reads with 1:120 / end-119:end.

Per workload: device-resident reads/s; end-to-end reads/s of a pinned pipeline with four batches in flight for
byte, packed4, window and window + packed4 input; host-to-device bytes per read; a bare pinned H2D copy rate;
bdx_window_reads on one host core; and whether the windowed results equal the device-resident ones on every
timed batch.  --profile instead times k_expand_windows with torch.profiler against a device-to-device copy of the
same bytes (a run of its own: tracing slows the host).  Inputs are larger than the 126 MB L2.  Prints one JSON line.
Usage: python tools/bench_windows.py [--steps 3] [--profile]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
SEED = 0x57494E44


def workloads():
    import bdx_b200 as bdx
    import bench_configs
    R = bdx.parse_dynamic_range
    rng = np.random.default_rng(SEED)
    cfg3, sp3, _ = bench_configs.configs()["3"]
    b1, b2 = bench_configs.barcodes(rng, 96, 24, 24), bench_configs.barcodes(rng, 96, 24, 24)
    single = bdx.DemuxConfig(bc_seqs=b1, bc_lengths_no_N=[24] * 96, ids=[f"a{i}" for i in range(96)],
                             ref_search_range=R("1:120"))
    dual = bdx.DemuxConfig(bc_seqs=b1, bc_lengths_no_N=[24] * 96, ids=[f"a{i}" for i in range(96)], is_dual=True,
                           bc_seqs2=b2, bc_lengths_no_N2=[24] * 96, ids2=[f"b{i}" for i in range(96)],
                           ref_search_range=R("1:120"), ref_search_range2=R("end-119:end"))
    long_sp = dict(start_lo=1, start_hi=90, set2_mode=1, end_lo=0, end_hi=90)
    # name: (config, read length, reads, batch, synth plant spec)
    return {"config3_150bp": (cfg3, 150, 4_000_000, 100_000, sp3),
            "long3kb_1:120": (single, 3000, 400_000, 50_000, dict(long_sp, set2_mode=0)),
            "long3kb_dual_1:120_end-119:end": (dual, 3000, 400_000, 50_000, long_sp)}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def run(name, spec, args, torch):
    import bdx_b200 as bdx
    from bdx_b200 import capi
    cfg, L, n, B, sp = spec
    n = n // args.scale // B * B if args.scale > 1 else n
    config = capi.Config(cfg)
    st = capi.Stream(config, device=0, max_reads=B, max_bytes=B * L)
    ext = torch.cuda.ExternalStream(st.cuda_stream)
    d_seq = torch.empty(n * L + 16, dtype=torch.uint8, device="cuda")
    d_off = torch.empty(n + 1, dtype=torch.int32, device="cuda")
    d_res = torch.empty(n * bdx.RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    st.synth_device(capi.SynthSpec(seed=SEED, first_read=0, read_len=L, plant_permille=900, n_permille_x10=50, **sp),
                    n, d_seq.data_ptr(), d_off.data_ptr())
    st.classify_device(d_seq.data_ptr(), d_off.data_ptr(), n, d_res.data_ptr())
    st.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ext)
    for _ in range(args.steps):
        st.classify_device(d_seq.data_ptr(), d_off.data_ptr(), n, d_res.data_ptr())
    e1.record(ext)
    st.sync()
    device_rate = n * args.steps / (e0.elapsed_time(e1) * 1e-3)
    ref = np.frombuffer(d_res.cpu().numpy().tobytes(), dtype=bdx.RESULT_DTYPE)

    h_seq = torch.empty(n * L, dtype=torch.uint8, pin_memory=True)
    h_seq.copy_(d_seq[:n * L])
    torch.cuda.synchronize()
    seq = h_seq.numpy()
    off = (np.arange(B + 1, dtype=np.int32) * L)
    t = time.perf_counter()
    win_all, win_off_all = config.window_reads(seq, np.arange(n + 1, dtype=np.int64).astype(np.int32) * L)
    window_reads_s = time.perf_counter() - t
    w = int(win_off_all[1])                                   # window bytes per read (every read has length L)
    win_off = np.ascontiguousarray(win_off_all[:B + 1])

    def pinned(a):
        p = torch.empty(a.size, dtype=torch.uint8, pin_memory=True)
        p.numpy()[:] = a
        return p

    h_win = pinned(win_all)
    h_pk = pinned(config.pack4(seq))
    h_wpk = pinned(config.pack4(win_all))
    h_off = torch.from_numpy(off).pin_memory()
    h_woff = torch.from_numpy(win_off).pin_memory()
    arrays = dict(seq=seq, win=h_win.numpy(), pk=h_pk.numpy(), wpk=h_wpk.numpy(), off=h_off.numpy(),
                  woff=h_woff.numpy())
    nb = n // B
    modes = {
        "bytes": (L + 4, lambda k: st.submit(arrays["seq"][k * B * L:(k + 1) * B * L], arrays["off"], tag=k, pinned=True)),
        "packed4": (L / 2 + 4, lambda k: st.submit_packed4(arrays["pk"][k * B * L // 2:(k + 1) * B * L // 2],
                                                             arrays["off"], tag=k, pinned=True)),
        "windows": (w + 8, lambda k: st.submit_windows(arrays["win"][k * B * w:(k + 1) * B * w], arrays["woff"],
                                                       arrays["off"], pinned=True, tag=k)),
        "windows_packed4": (w / 2 + 8, lambda k: st.submit_windows(arrays["wpk"][k * B * w // 2:(k + 1) * B * w // 2],
                                                                   arrays["woff"], arrays["off"], packed4=True,
                                                                   pinned=True, tag=k)),
    }
    got = np.zeros(nb * B, dtype=bdx.RESULT_DTYPE)
    got_bytes, rec = got.view(np.uint8), bdx.RESULT_DTYPE.itemsize

    def pipeline(submit, steps):
        """Every result record is copied out as raw bytes (a field-wise structured copy would bound the pipeline)."""
        queued = 0
        for _ in range(steps):
            for k in range(nb):
                submit(k)
                queued += 1
                if queued == 4:
                    tag, r = st.fetch(copy=False)
                    got_bytes[tag * B * rec:(tag + 1) * B * rec] = r.view(np.uint8)
                    queued -= 1
        while queued:
            tag, r = st.fetch(copy=False)
            got_bytes[tag * B * rec:(tag + 1) * B * rec] = r.view(np.uint8)
            queued -= 1

    if args.profile:
        return profile(name, st, modes, pipeline, d_seq, B, L, w, nb, torch)
    e2e, equal = {}, {}
    for mode, (bpr, submit) in modes.items():
        pipeline(submit, 1)
        got[:] = 0
        t = time.perf_counter()
        pipeline(submit, args.steps)
        dt = time.perf_counter() - t
        e2e[mode] = {"reads_per_s": round(nb * B * args.steps / dt), "h2d_bytes_per_read": bpr}
        equal[mode] = bool((got == ref[:nb * B]).all())
    d_probe = torch.empty(B * L, dtype=torch.uint8, device="cuda")
    e0.record()
    for k in range(nb):
        d_probe.copy_(h_seq[k * B * L:(k + 1) * B * L], non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    copy_gbs = nb * B * L / (e0.elapsed_time(e1) * 1e-3) / 1e9
    link_bound = copy_gbs * 1e9 / (w + 8)
    target = 0.8 * min(device_rate, link_bound)
    out = {"reads": nb * B, "read_len": L, "batch": B, "window_bytes_per_read": w,
           "device_resident_reads_per_s": round(device_rate), "e2e": e2e,
           "results_equal_device_resident": equal, "pinned_h2d_copy_GBps": round(copy_gbs, 2),
           "windowed_target_reads_per_s": round(target),
           "windowed_target_met": e2e["windows"]["reads_per_s"] >= target,
           "window_reads_per_core": {"reads_per_s": round(n / window_reads_s),
                                     "input_GBps": round(n * L / window_reads_s / 1e9, 2)}}
    st.close()
    config.close()
    return out


def profile(name, st, modes, pipeline, d_seq, B, L, w, nb, torch):
    """k_expand_windows per batch against a device-to-device copy of one batch (the same working-set size: for
    config 3 a batch, and the four slots' buffers it cycles through, fit the 126 MB L2, so both are L2 rates there) and
    against a copy of the whole input (larger than L2: the HBM rate)."""
    from torch.profiler import ProfilerActivity, profile as tprofile
    src = torch.empty(B * L, dtype=torch.uint8, device="cuda")
    dst = torch.empty(B * L, dtype=torch.uint8, device="cuda")
    src.copy_(d_seq[:B * L])
    whole = torch.empty(nb * B * L, dtype=torch.uint8, device="cuda")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    whole.copy_(d_seq[:nb * B * L])
    e0.record()
    for _ in range(3):
        whole.copy_(d_seq[:nb * B * L])
    e1.record()
    torch.cuda.synchronize()
    hbm_copy_gbps = 3 * 2 * nb * B * L / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del whole
    out = {"batch_output_MB": round(B * L / 1e6, 1), "batch_fits_l2": 4 * B * (L + w) < 126e6,
           "whole_input_d2d_GBps": round(hbm_copy_gbps, 1)}
    for mode in ("windows", "windows_packed4"):
        pipeline(modes[mode][1], 1)
        torch.cuda.synchronize()
        with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
            pipeline(modes[mode][1], 1)
            for _ in range(nb):
                dst.copy_(src)
            torch.cuda.synchronize()
        ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        k = [e.device_time for e in ev if "k_expand_windows" in e.name]
        c = [e.device_time for e in ev if "Memcpy DtoD" in e.name or "Memcpy Device to Device" in e.name]
        moved = B * (w if mode == "windows" else w / 2) + B * L + 8 * (B + 1)   # window in, offsets in, batch out
        k_us, c_us = float(np.median(k or [np.nan])), float(np.median(c or [np.nan]))
        out[mode] = {"k_expand_windows_us": round(k_us, 1), "launches": len(k), "bytes_moved": int(moved),
                     "GBps": round(moved / k_us / 1e3, 1), "d2d_copy_us": round(c_us, 1),
                     "d2d_GBps": round(2 * B * L / c_us / 1e3, 1)}
        out[mode]["ratio_to_d2d"] = round(out[mode]["GBps"] / out[mode]["d2d_GBps"], 3)
        out[mode]["ratio_to_whole_input_d2d"] = round(out[mode]["GBps"] / hbm_copy_gbps, 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--scale", type=int, default=1, help="divide the read counts (quick runs; below L2 size)")
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--only", nargs="*", default=None)
    args = ap.parse_args()
    import torch
    torch.cuda.set_device(0)
    line = {"bench": "windows" + ("_profile" if args.profile else ""), "gpu": gpu_info(), "steps": args.steps}
    for name, spec in workloads().items():
        if args.only and name not in args.only:
            continue
        line[name] = run(name, spec, args, torch)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
