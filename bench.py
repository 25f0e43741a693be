#!/usr/bin/env python
"""bench.py -- DEFLATE level-6 compress + inflate throughput (GB/s of uncompressed bytes) on B200.

One "step" = one pass of the hot path over one batch of synthetic input:
    deflate leg : config C3 -- raw Deflater level 6 on 1024 x 256 KiB Silesia-mix buffers
    inflate leg : config C2 -- raw Inflater on 256 x 1 MiB text buffers pre-deflated (level 6) by the oracle
value = (uncompressed bytes of both legs) / (device time of both legs), inputs resident in HBM, CUDA events.
e2e   = the same step through the LIBRARY'S host-buffer call: b200z_pipeline_submit / _collect (include/b200z.h) on plain
        host pointers into pinned host memory -- staging, H2D of every input byte, kernels, D2H of exactly the produced bytes
        and the hand-over to the caller's buffers all inside the timed region, one submit + one collect per leg and step
        (depth 2: the upload of step i+1 and the download of step i-1 overlap step i's kernels, inside the library).
With --gpus N > 1 (torchrun, one rank per GPU) every rank runs the same shape on its own buffers (weak scaling; --scaling
strong splits ONE C3 + C2 batch over the ranks by bytes instead), the static Huffman tables are broadcast once over NCCL,
and rank 0 reports total units / max-over-ranks time.
--impl reference times the CPU restatement of the reference (oracle/, all host threads) on the SAME buffers and mix.
--steps K times K steps (resident, end to end and per kernel); --dump-outputs DIR writes what the last resident step computed
to DIR as .npy files (the inputs are generated from fixed seeds, so two builds can be compared output for output).
--config c4 / c5 run BASELINE.json's configs 4 (one 2 GiB log stream through GZipOutputStream's bytes) and 5 (level x size
grid); they print their own JSON line and are not the driver's bench line.
"""
import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

METRIC = "DEFLATE level-6 compress + inflate GB/s (uncompressed) at 1/2/4/8 B200 vs C# ref"
N_DEFLATE, SZ_DEFLATE = 1024, 262144      # C3
N_INFLATE, SZ_INFLATE = 256, 1 << 20       # C2


def _gen_deflate(i):
    from sharpziplib_b200 import datagen
    return datagen.silesia_mix(i, SZ_DEFLATE, config=3)


def _gen_inflate(i):
    from sharpziplib_b200 import datagen
    return datagen.text_buffer(i, SZ_INFLATE, config=2)


def make_inputs(rank, n_def, n_inf, workers):
    """(list of deflate inputs, list of inflate originals) as numpy uint8 arrays; buffer indices are offset per rank"""
    from concurrent.futures import ProcessPoolExecutor
    di = [rank * N_DEFLATE + i for i in range(n_def)]
    ii = [rank * N_INFLATE + i for i in range(n_inf)]
    if workers > 1:
        with ProcessPoolExecutor(max_workers=workers) as ex:
            d = list(ex.map(_gen_deflate, di, chunksize=8))
            t = list(ex.map(_gen_inflate, ii, chunksize=2))
    else:
        d = [_gen_deflate(i) for i in di]
        t = [_gen_inflate(i) for i in ii]
    return d, t


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md recipe)"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    """threads the reference arm may really use: logical CPUs, capped by the affinity mask and the cgroup CPU quota"""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, int(q / per + 0.5)))
        except Exception:
            pass
    return n


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def captured_traffic(kernel, small):
    """dram bytes (read + write) of one launch of `kernel` on this workload, from the committed ncu --set full capture"""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if small or not os.path.exists(p):
        return None, None
    j = json.load(open(p))
    if j.get("kernel") != kernel:
        return None, None
    return int(j["dram_bytes_per_launch"]), j.get("source")


INFLATE_KERNELS = ("k_wrap", "k_find", "k_find3", "k_seglist", "k_dec1", "k_chain", "k_dec2", "k_resolve", "k_inflate")


def dotnet_probe():
    """is there a .NET / mono runtime to run the real SharpZipLib with (tools/csharp_harness)?  Probed, not assumed."""
    found = {t: shutil.which(t) for t in ("dotnet", "mono", "csc", "mcs")}
    return {"found": {k: v for k, v in found.items() if v}, "any": any(found.values())}


class CpuSample:
    """the oracle (C++ restatement of the reference) on the step's own buffers; only the C calls are timed"""

    def __init__(self, d_inputs, comp_inf, inf_caps):
        import oracle_lib as O
        self.dj = O.BatchJob(0, [a.tobytes() for a in d_inputs], level=6)
        self.ij = O.BatchJob(1, comp_inf, out_caps=[c + 64 for c in inf_caps])
        self.ud = int(self.dj.lens.sum())
        self.ui = int(sum(inf_caps))

    def run(self, threads):
        t0 = time.perf_counter()
        self.dj.run(threads)
        t1 = time.perf_counter()
        self.ij.run(threads)
        t2 = time.perf_counter()
        return {"value": (self.ud + self.ui) / (t2 - t0) / 1e9, "deflate_gbs": self.ud / (t1 - t0) / 1e9,
                "inflate_gbs": self.ui / (t2 - t1) / 1e9, "seconds": t2 - t0}


def workload_name(n_def, n_inf):
    return "C3 deflate L6 %dx256KiB + C2 inflate %dx1MiB per GPU" % (n_def, n_inf)


def run_reference(args, rank, world, out):
    """--impl reference: the reference's CPU algorithm on all host threads, on the GPU arm's own step: the same generators,
    the same 1024 + 256 buffers, the same 1:1 mix of the legs, whatever the thread count.  The C# original cannot run here:
    neither this image nor the GPU boxes have a .NET / mono runtime (profiles/r02_probe_gpu_box.txt; probed again below), so
    the arm is the line-faithful C++ restatement under oracle/ (kind "port")."""
    if rank != 0:
        return
    import oracle_lib as O
    O.build()
    threads = host_threads()
    n_def = N_DEFLATE // (8 if args.small else 1)
    n_inf = N_INFLATE // (8 if args.small else 1)
    d, t = make_inputs(0, n_def, n_inf, min(threads, 32))
    comp = O.batch(0, [a.tobytes() for a in t], level=6, threads=threads)
    job = CpuSample(d, comp, [a.size for a in t])
    for _ in range(args.warmup):
        job.run(threads)
    times, last = [], None
    for _ in range(args.steps):
        last = job.run(threads)
        times.append(last["seconds"])
    ub = n_def * SZ_DEFLATE + n_inf * SZ_INFLATE
    val = ub * len(times) / sum(times) / 1e9
    sample = "the whole step: %d x 256 KiB deflate L6 + %d x 1 MiB inflate, %d threads" % (n_def, n_inf, threads)
    probe = dotnet_probe()
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000 * sum(times) / len(times), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload_name(n_def, n_inf), "sample": sample},
            "cpu_baseline": {"value": val, "unit": "GB/s", "cores": threads, "kind": "port", "sample": sample,
                             "dotnet": probe,
                             "note": "C++ restatement of SharpZipLib's managed path (oracle/); the C# harness is tools/csharp_harness"},
            "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "deflate_gbs": last["deflate_gbs"], "inflate_gbs": last["inflate_gbs"], "gpu_launches": 0}
    out.write(json.dumps(line) + "\n")
    out.flush()


def _claim_stdout():
    """Libraries (NCCL's version banner, torchrun children) may print to fd 1; the contract is ONE JSON line on stdout.
    Everything else is redirected to stderr and the JSON line is written to the saved descriptor."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(saved, "w")


def _dist_setup(rank, local_rank, world):
    import torch
    import torch.distributed as dist
    import sharpziplib_b200 as z
    from sharpziplib_b200.sharding import broadcast_static_tables
    torch.cuda.set_device(local_rank)
    z.init(local_rank)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))
        broadcast_static_tables(dist, device=torch.device("cuda", local_rank))  # the path's only collective
    return dist


def _max_over_ranks(dist, world, ms, dev):
    import torch
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    return ms


def main():
    out = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200z", choices=["b200z", "reference"])
    ap.add_argument("--config", default="bench", choices=["bench", "c4", "c5", "multi"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--small", action="store_true", help="1/8 size workload for quick checks (not a bench value)")
    ap.add_argument("--no-probe", dest="no_probe", action="store_true", help="(accepted for older command lines; no effect)")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world, out)
        return
    if args.config == "c4":
        run_c4(args, rank, local_rank, world, out)
        return
    if args.config == "c5":
        run_c5(args, rank, local_rank, world, out)
        return
    if args.config == "multi":
        run_multi(args, rank, out)
        return
    run_bench(args, rank, local_rank, world, out)


DUMP_SEED, DUMP_DEFLATE_STREAMS, DUMP_INFLATE_STREAMS = 20240601, 32, 4


def dump_outputs(dirname, dplan, iplan, d_dout, d_dlen, d_dst, d_iout, d_ilen, d_ist, d_iused):
    """What the two plans handed their caller in the last step, as DIR/<name>.npy: every stream's output length, status and
    (inflate) input bytes consumed in float64, and the output bytes of a fixed, seeded sample of streams (32 compressed, 4
    inflated; back to back in stream order) in float32 -- at most 55 MB, so that two builds can be compared output for output."""
    rng = np.random.default_rng(DUMP_SEED)
    dlen, ilen = d_dlen.cpu().numpy(), d_ilen.cpu().numpy()
    dpick = np.sort(rng.choice(dlen.size, min(DUMP_DEFLATE_STREAMS, dlen.size), replace=False))
    ipick = np.sort(rng.choice(ilen.size, min(DUMP_INFLATE_STREAMS, ilen.size), replace=False))

    def streams(d_buf, offsets, lens, pick):
        return np.concatenate([d_buf[int(offsets[i]):int(offsets[i] + lens[i])].cpu().numpy() for i in pick]).astype(np.float32)
    arrays = {"deflate_out_len": dlen, "deflate_status": d_dst.cpu().numpy(), "deflate_sample_streams": dpick,
              "deflate_out_sample": streams(d_dout, dplan.out_offsets, dlen, dpick),
              "inflate_out_len": ilen, "inflate_status": d_ist.cpu().numpy(), "inflate_in_used": d_iused.cpu().numpy(),
              "inflate_sample_streams": ipick, "inflate_out_sample": streams(d_iout, iplan.out_offsets, ilen, ipick)}
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def run_bench(args, rank, local_rank, world, out):
    import torch
    import oracle_lib as O
    import sharpziplib_b200 as z
    from sharpziplib_b200.sharding import partition_by_bytes
    dist = _dist_setup(rank, local_rank, world)
    n_def = N_DEFLATE // (8 if args.small else 1)
    n_inf = N_INFLATE // (8 if args.small else 1)
    ncpu = host_threads()
    workers = max(1, min(32, ncpu // max(1, world)))
    strong = args.scaling == "strong" and world > 1
    t_setup = time.time()
    if strong:
        # ONE batch for the whole job, cut by cumulative bytes (sharding.partition_by_bytes); this rank's share
        d_all, t_all = make_inputs(0, n_def, n_inf, workers)
        a, b = partition_by_bytes([x.size for x in d_all], world)[rank]
        d_np = d_all[a:b]
        a, b = partition_by_bytes([x.size for x in t_all], world)[rank]
        t_np = t_all[a:b]
        n_def, n_inf = len(d_np), len(t_np)
    else:
        d_np, t_np = make_inputs(rank, n_def, n_inf, workers)
    O.build()
    comp = O.batch(0, [a.tobytes() for a in t_np], level=6, threads=max(1, ncpu // max(1, world)))
    setup_s = time.time() - t_setup

    # ---- plans and resident device buffers ---------------------------------------------------------------
    dplan = z.DeflatePlan([a.size for a in d_np], level=6)
    iplan = z.InflatePlan([len(c) for c in comp], [a.size for a in t_np])
    dev = torch.device("cuda", local_rank)
    h = np.zeros(dplan.in_bytes, dtype=np.uint8)
    for o, a in zip(dplan.in_offsets, d_np):
        h[o:o + a.size] = a
    d_din = torch.from_numpy(h).to(dev)
    h = np.zeros(iplan.in_bytes, dtype=np.uint8)
    for o, c in zip(iplan.in_offsets, comp):
        h[o:o + len(c)] = np.frombuffer(c, dtype=np.uint8)
    d_iin = torch.from_numpy(h).to(dev)
    del h
    d_dout = torch.empty(dplan.out_bytes, dtype=torch.uint8, device=dev)
    d_iout = torch.empty(iplan.out_bytes, dtype=torch.uint8, device=dev)
    d_dlen = torch.zeros(n_def, dtype=torch.int64, device=dev)
    d_dst = torch.zeros(n_def, dtype=torch.int32, device=dev)
    d_ilen = torch.zeros(n_inf, dtype=torch.int64, device=dev)
    d_ist = torch.zeros(n_inf, dtype=torch.int32, device=dev)
    d_iused = torch.zeros(n_inf, dtype=torch.int64, device=dev)
    U_def = sum(a.size for a in d_np)
    U_inf = sum(a.size for a in t_np)
    C_inf = sum(len(c) for c in comp)

    # The two legs are independent: the inflate leg runs on a second stream next to the ENCODE half of the deflate leg
    # (the SEARCH half's CTAs take a whole SM's shared memory).
    s_leg = torch.cuda.Stream(device=dev)
    ev_leg0, ev_leg1 = torch.cuda.Event(), torch.cuda.Event()

    def step_resident(overlap=True):
        cur = torch.cuda.current_stream()
        if not overlap:
            dplan.run(d_din, d_dout, d_dlen, d_dst)
            iplan.run(d_iin, d_iout, d_ilen, d_ist, None, d_iused)
            return
        dplan.run(d_din, d_dout, d_dlen, d_dst, stages=z.STAGE_SEARCH)
        ev_leg0.record(cur)
        s_leg.wait_event(ev_leg0)
        iplan.run(d_iin, d_iout, d_ilen, d_ist, None, d_iused, stream=s_leg)
        ev_leg1.record(s_leg)
        dplan.run(d_din, d_dout, d_dlen, d_dst, stages=z.STAGE_ENCODE)
        cur.wait_event(ev_leg1)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = _max_over_ranks(dist, world, e0.elapsed_time(e1), dev)
        barrier()
        return ms

    for _ in range(max(3, args.warmup)):
        step_resident()
    torch.cuda.synchronize()
    # ---- parity of what is being timed (not in the timed region) -------------------------------------------
    C_def = int(d_dlen.sum().item())
    assert int((d_dst != 0).sum().item()) == 0 and int((d_ist != 0).sum().item()) == 0, "device status != OK"
    lens = d_dlen.cpu().numpy()
    outb = d_dout.cpu().numpy()
    for i in range(0, n_def, max(1, n_def // 16)):
        ref = O.deflate(d_np[i].tobytes(), level=6)
        got = outb[dplan.out_offsets[i]:dplan.out_offsets[i] + lens[i]].tobytes()
        assert got == ref, "deflate parity failed for buffer %d" % i
    io = d_iout.cpu().numpy()
    for i in range(n_inf):  # every inflated stream, byte for byte
        assert np.array_equal(io[iplan.out_offsets[i]:iplan.out_offsets[i] + t_np[i].size], t_np[i]), "inflate mismatch %d" % i
    del outb, io
    inflate_stats = iplan.stats()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_total = timed(step_resident, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:  # before the per-kernel timing below runs the plans again
        dump_outputs(args.dump_outputs, dplan, iplan, d_dout, d_dlen, d_dst, d_iout, d_ilen, d_ist, d_iused)
    ms_step = ms_total / args.steps
    units_t = torch.tensor([float(U_def + U_inf)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(units_t)
    units = float(units_t.item())
    value = units / (ms_step / 1e3) / 1e9

    # ---- per-kernel device times for the roofline (separate steps, events between kernels) -------------------
    dplan.set_timing(True)
    iplan.set_timing(True)
    acc = {}
    reps = args.steps
    for _ in range(reps):
        step_resident(overlap=False)  # one kernel at a time: these are per-kernel durations
        torch.cuda.synchronize()
        for k, v in list(dplan.timings().items()) + list(iplan.timings().items()):
            acc[k] = acc.get(k, 0.0) + v / reps
    dplan.set_timing(False)
    iplan.set_timing(False)
    t_inf = sum(v for k, v in acc.items() if k in INFLATE_KERNELS)
    t_def = sum(v for k, v in acc.items() if k not in INFLATE_KERNELS)
    dom = max(acc, key=acc.get)
    peak, peak_src = peaks()
    alg_bytes = (C_inf + U_inf) if dom in INFLATE_KERNELS else (U_def + C_def)
    achieved = alg_bytes / (acc[dom] / 1e3) / 1e9
    traffic, traffic_src = captured_traffic(dom, args.small)
    legs = {"deflate": {"ms": t_def, "algorithmic_bytes": U_def + C_def, "gbs": (U_def + C_def) / (t_def / 1e3) / 1e9 if t_def else None},
            "inflate": {"ms": t_inf, "algorithmic_bytes": C_inf + U_inf, "gbs": (C_inf + U_inf) / (t_inf / 1e3) / 1e9 if t_inf else None}}
    for v in legs.values():
        v["frac_of_peak"] = v["gbs"] / peak if v["gbs"] else None
    # the device buffers of the resident measurement are not needed any more
    del d_dout, d_iout, d_din, d_iin
    torch.cuda.empty_cache()

    # ---- end to end through the library's host-buffer pipelines ----------------------------------------------------
    # Plain host pointers: every input stream lies in pinned host memory (one tensor per leg, streams back to back) and every
    # output goes to its own pinned region; the library sees only addresses and sizes.
    def pinned_concat(arrs):
        t = torch.empty(sum(len(a) for a in arrs) + 64, dtype=torch.uint8).pin_memory()
        ptrs, pos = [], 0
        for a in arrs:
            n = len(a)
            t[pos:pos + n] = torch.frombuffer(bytearray(a), dtype=torch.uint8) if isinstance(a, (bytes, bytearray)) else torch.from_numpy(a)
            ptrs.append(t.data_ptr() + pos)
            pos += n
        return t, ptrs

    h_din, din_ptrs = pinned_concat(d_np)
    h_iin, iin_ptrs = pinned_concat(comp)
    dcaps = np.array([z.lib().b200z_deflate_bound(int(a.size)) + 16 for a in d_np], dtype=np.int64)
    icaps = np.array([a.size for a in t_np], dtype=np.int64)
    h_dout = torch.empty(int(dcaps.sum()) + 64, dtype=torch.uint8).pin_memory()
    h_iout = torch.empty(int(icaps.sum()) + 64, dtype=torch.uint8).pin_memory()
    dout_off = np.concatenate([[0], np.cumsum(dcaps)[:-1]]).astype(np.int64)
    iout_off = np.concatenate([[0], np.cumsum(icaps)[:-1]]).astype(np.int64)
    P = z.Pipeline
    din_p, iin_p = P.pointers(din_ptrs), P.pointers(iin_ptrs)
    dout_p = P.pointers([h_dout.data_ptr() + int(o) for o in dout_off])
    iout_p = P.pointers([h_iout.data_ptr() + int(o) for o in iout_off])
    dpipe = P.deflate([a.size for a in d_np], level=6, depth=2)
    ipipe = P.inflate([len(c) for c in comp], icaps, depth=2)
    e2e_d2h = [0]

    def e2e_collect():
        dpipe.collect(dout_p, dcaps)
        ipipe.collect(iout_p, icaps)
        e2e_d2h[0] = int(dpipe.out_len.sum()) + int(ipipe.out_len.sum()) + 28 * (n_def + n_inf)

    def e2e_steps(k):
        """k steps: submit(step i) before collect(step i-1); the last step is collected before the clock stops"""
        for i in range(k):
            dpipe.submit(din_p)
            ipipe.submit(iin_p)
            if i > 0:
                e2e_collect()
        e2e_collect()

    def timed_host(fn, k):
        barrier()
        t0 = time.perf_counter()
        fn(k)
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3
        ms = _max_over_ranks(dist, world, ms, dev)
        barrier()
        return ms

    e2e_steps(3)  # warm-up
    # what came back through the library is checked too
    assert int(np.count_nonzero(dpipe.status)) == 0 and int(np.count_nonzero(ipipe.status)) == 0
    hd = h_dout.numpy()
    for i in range(0, n_def, max(1, n_def // 8)):
        got = hd[dout_off[i]:dout_off[i] + int(dpipe.out_len[i])].tobytes()
        assert got == O.deflate(d_np[i].tobytes(), level=6), "e2e deflate parity failed for buffer %d" % i
    hi = h_iout.numpy()
    for i in range(0, n_inf, max(1, n_inf // 8)):
        assert np.array_equal(hi[iout_off[i]:iout_off[i] + t_np[i].size], t_np[i]), "e2e inflate mismatch %d" % i
    n_e2e = args.steps
    ms_e2e = timed_host(e2e_steps, n_e2e) / n_e2e
    e2e_val = units / (ms_e2e / 1e3) / 1e9
    # the same call on PAGEABLE host memory (what a caller that never pinned anything hands over): staged by the library
    pg_din = [np.array(a, copy=True) for a in d_np]
    pg_iin = [np.frombuffer(bytearray(c), dtype=np.uint8) for c in comp]
    pg_dout = np.empty(int(dcaps.sum()) + 64, dtype=np.uint8)
    pg_iout = np.empty(int(icaps.sum()) + 64, dtype=np.uint8)
    din_p, iin_p = P.pointers([a.ctypes.data for a in pg_din]), P.pointers([a.ctypes.data for a in pg_iin])
    dout_p = P.pointers([pg_dout.ctypes.data + int(o) for o in dout_off])
    iout_p = P.pointers([pg_iout.ctypes.data + int(o) for o in iout_off])
    e2e_steps(2)
    ms_pg = timed_host(e2e_steps, args.steps) / args.steps
    dpipe.close()
    ipipe.close()
    del h_din, h_iin, h_dout, h_iout, pg_dout, pg_iout

    # ---- the streaming handles (what DeflaterOutputStream / InflaterInputStream callers get) -------------------------
    handles = None
    if rank == 0:
        import io as _io
        blob = b"".join(a.tobytes() for a in d_np[:16 if args.small else 256])  # 4 MiB / 64 MiB of the deflate leg's buffers as one stream
        defl = z.Deflater(6, True)
        write_gbs = []
        for attempt in range(2):  # the second stream goes through the same Deflater after Reset(), as ZipOutputStream's entries do
            if attempt:
                defl.Reset()
            sink = _io.BytesIO()
            t0 = time.perf_counter()
            s = z.DeflaterOutputStream(sink, defl, bufferSize=65536)
            for o in range(0, len(blob), 1 << 20):  # DeflaterOutputStream.Write in 1 MiB writes
                s.Write(blob[o:o + (1 << 20)])
            s.Finish()
            t1 = time.perf_counter()
            write_gbs.append(len(blob) / (t1 - t0) / 1e9)
            raw = sink.getvalue()
            assert raw == O.deflate(blob, level=6), "DeflaterOutputStream bytes differ from the oracle's"

        def read_back(buffer_size, limit):
            r = z.InflaterInputStream(_io.BytesIO(raw), z.Inflater(True), bufferSize=buffer_size)
            back = bytearray()
            t = time.perf_counter()
            while len(back) < limit:
                chunk = r.read(1 << 16)
                if not chunk:
                    break
                back += chunk
            dt = time.perf_counter() - t
            assert bytes(back) == blob[:len(back)] and len(back) >= limit, "InflaterInputStream round trip failed"
            return len(back) / dt / 1e9
        small_part = min(len(blob), 4 << 20)
        handles = {"deflater_output_stream_1MiB_writes_gbs": write_gbs[1],
                   "deflater_output_stream_first_stream_gbs": write_gbs[0],  # with the handle's one-time allocations
                   # the reference's default buffer (InflaterInputStream.cs:358: 4096 bytes per Fill), first 4 MiB of the stream
                   "inflater_input_stream_4KiB_feeds_gbs": read_back(4096, small_part),
                   # the same class with its bufferSize constructor argument (:346) at 1 MiB, the whole stream
                   "inflater_input_stream_1MiB_feeds_gbs": read_back(1 << 20, len(blob)),
                   "bytes": len(blob), "bytes_4KiB_feeds": small_part}

    # ---- CPU baseline: the oracle on one host core, the whole step once ------------------------------------------------
    cpu = None
    if rank == 0:
        r = CpuSample(d_np, comp, [a.size for a in t_np]).run(1)
        cpu = {"value": r["value"], "unit": "GB/s", "cores": 1, "kind": "port",
               "sample": "the whole step once: %d x 256 KiB deflate L6 + %d x 1 MiB inflate, single thread, %.1f s" % (n_def, n_inf, r["seconds"]),
               "deflate_gbs": r["deflate_gbs"], "inflate_gbs": r["inflate_gbs"], "host_cores": ncpu, "dotnet": dotnet_probe(),
               "note": "C++ restatement of SharpZipLib's managed path (oracle/); the C# harness for a box with .NET is tools/csharp_harness"}
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "config": {"workload": workload_name(N_DEFLATE // (8 if args.small else 1), N_INFLATE // (8 if args.small else 1)) if not strong
                       else "ONE C3 + C2 batch split over %d GPUs by bytes (rank 0: %d + %d buffers)" % (world, n_def, n_inf),
                       "l2": "inputs (256 MiB + 77 MiB compressed per step) exceed the 126 MB L2; no flush needed",
                       "parity": "before timing: deflate bytes == oracle on 16 buffers, every inflated stream == original; e2e outputs checked again",
                       "ratio_deflate": U_def / max(1, C_def), "ratio_inflate": U_inf / max(1, C_inf), "setup_s": setup_s,
                       "inflate_pipeline": inflate_stats},
            "deflate_gbs": U_def / (t_def / 1e3) / 1e9 if t_def else None,
            "inflate_gbs": U_inf / (t_inf / 1e3) / 1e9 if t_inf else None,
            "kernels_ms": acc, "legs": legs,
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes": alg_bytes},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_val, "unit": "GB/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": int(U_def + C_inf),
                    "d2h_bytes_per_step": int(e2e_d2h[0]),
                    "pageable_host_memory": {"value": units / (ms_pg / 1e3) / 1e9, "ms_per_step": ms_pg},
                    "how": "b200z_pipeline_submit + b200z_pipeline_collect per leg and step on host pointers into pinned memory (depth 2, "
                           "the library's own streams / staging / packed D2H); host clock around %d steps + the last collect, device idle "
                           "on both sides; pageable_host_memory: the same calls on malloc'ed buffers (staged through the library's pinned slots)" % n_e2e},
            "handles": handles,
            "gpu_launches": int(dplan.launches + iplan.launches) * args.steps,
            "gpu_launches_per_step": int(dplan.launches + iplan.launches),
            "clocks": clocks,
        }
        out.write(json.dumps(line) + "\n")
        out.flush()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_c4(args, rank, local_rank, world, out):
    """BASELINE.json config 4: GZipOutputStream end to end (CRC32 + deflate) on ONE 2 GiB synthetic log stream, 1 x B200.
    The stream goes through the library's host call with wrap = GZIP (header, raw level-6 stream, CRC-32, ISIZE = 0x80000000);
    the bytes are compared with the oracle's for the whole stream (the reference's DeflaterEngine is serial: one host
    thread, ~80 s) and inflated back by zlib.  A single stream does not shard: other ranks idle ("replicas only")."""
    import zlib
    import torch
    import oracle_lib as O
    import sharpziplib_b200 as z
    from sharpziplib_b200 import datagen
    if rank != 0:
        return
    torch.cuda.set_device(local_rank)
    z.init(local_rank)
    size = (256 << 20) if args.small else (2048 << 20)
    t0 = time.time()
    d = datagen.log_stream(size)
    gen_s = time.time() - t0
    P = z.Pipeline
    pipe = P.deflate([size], level=6, wrap=2, depth=1)
    h_in = torch.from_numpy(d).pin_memory()
    cap = np.array([z.lib().b200z_deflate_bound(size) + 64], dtype=np.int64)
    h_out = torch.empty(int(cap[0]), dtype=torch.uint8).pin_memory()
    inp, outp = P.pointers([h_in.data_ptr()]), P.pointers([h_out.data_ptr()])
    times = []
    for it in range(1 + max(2, min(args.steps, 3))):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pipe.submit(inp)
        pipe.collect(outp, cap)
        times.append(time.perf_counter() - t0)
    clen = int(pipe.out_len[0])
    gz = h_out[:clen].numpy().tobytes()
    isize = int.from_bytes(gz[-4:], "little")
    crc = int.from_bytes(gz[-8:-4], "little")
    ok_crc = crc == (zlib.crc32(d) & 0xFFFFFFFF)
    ok_hdr = gz[:10] == bytes([0x1F, 0x8B, 8, 0, 0, 0, 0, 0, 0, 0xFF])
    back_ok = hashlib.sha256(zlib.decompress(gz, 31)).digest() == hashlib.sha256(d).digest()
    t0 = time.time()
    ref = O.deflate(d, level=6)  # the whole stream through the restated DeflaterEngine
    oracle_s = time.time() - t0
    parity = gz[10:-8] == ref
    e2e_s = float(np.median(times[1:]))
    line = {"config": "c4", "workload": "one %d MiB log stream, GZipOutputStream bytes (CRC32 + deflate L6), host memory to host memory" % (size >> 20),
            "bytes": size, "gzip_bytes": clen, "ratio": size / clen, "e2e_ms": e2e_s * 1e3, "e2e_gbs": size / e2e_s / 1e9,
            "isize": "0x%08X" % isize, "isize_ok": isize == (size & 0xFFFFFFFF), "crc_ok": bool(ok_crc), "header_ok": bool(ok_hdr),
            "inflates_to_input": bool(back_ok), "parity_whole_stream_vs_oracle": bool(parity), "oracle_seconds": oracle_s,
            "oracle_gbs_one_thread": size / oracle_s / 1e9, "gen_s": gen_s, "n_gpus": 1}
    out.write(json.dumps(line) + "\n")
    out.flush()


def run_c5(args, rank, local_rank, world, out):
    """BASELINE.json config 5: Deflater level 1 / 6 / 9 x buffer size 4 KiB .. 64 MiB, 256 MiB per point and GPU, device time
    through the plan API with parity against the oracle on EVERY distinct buffer of every point."""
    import torch
    import oracle_lib as O
    import sharpziplib_b200 as z
    from sharpziplib_b200 import datagen
    dist = _dist_setup(rank, local_rank, world)
    dev = torch.device("cuda", local_rank)
    O.build()
    peak, _ = peaks()
    threads = max(1, host_threads() // max(1, world))
    per_point = (32 << 20) if args.small else (256 << 20)
    points = []
    for level in (1, 6, 9):
        for sz in (4 << 10, 16 << 10, 64 << 10, 256 << 10, 1 << 20, 4 << 20, 16 << 20, 64 << 20):
            if args.small and sz > (4 << 20):
                continue
            nb = max(4 if sz >= (64 << 20) else 1, per_point // sz)
            uniq = min(nb, 64 if sz <= (1 << 20) else (16 if sz <= (4 << 20) else 4))  # distinct buffers (class mix), tiled over the batch
            bufs = [datagen.silesia_mix(rank * 64 + i, sz, config=5) for i in range(uniq)]
            plan = z.DeflatePlan([sz] * nb, level=level)
            h = np.zeros(plan.in_bytes, dtype=np.uint8)
            for i, o in enumerate(plan.in_offsets):
                h[o:o + sz] = bufs[i % uniq]
            din = torch.from_numpy(h).to(dev)
            dout = torch.empty(plan.out_bytes, dtype=torch.uint8, device=dev)
            dl = torch.zeros(nb, dtype=torch.int64, device=dev)
            ds = torch.zeros(nb, dtype=torch.int32, device=dev)
            plan.run(din, dout, dl, ds)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 2
            e0.record()
            for _ in range(reps):
                plan.run(din, dout, dl, ds)
            e1.record()
            torch.cuda.synchronize()
            ms = _max_over_ranks(dist, world, e0.elapsed_time(e1) / reps, dev)
            assert int(ds.abs().sum()) == 0
            lens = dl.cpu().numpy()
            ob = dout.cpu().numpy()
            refs = O.batch(0, [b.tobytes() for b in bufs], level=level, threads=threads)
            ok = all(ob[plan.out_offsets[i]:plan.out_offsets[i] + lens[i]].tobytes() == refs[i] for i in range(uniq))
            C = float(lens.sum())
            points.append({"level": level, "size": sz, "buffers_per_gpu": nb, "distinct_checked": uniq, "ms": ms,
                           "gbs": world * nb * sz / ms / 1e6, "hbm_gbs": world * (nb * sz + C) / ms / 1e6,
                           "frac_of_peak": (nb * sz + C) / ms / 1e6 / peak, "ratio": nb * sz / C, "parity": bool(ok)})
            plan.close()
            del din, dout, ob
            torch.cuda.empty_cache()
    if rank == 0:
        out.write(json.dumps({"config": "c5", "n_gpus": world, "scaling": "weak", "peak_gbs": peak, "points": points,
                              "all_parity": all(p["parity"] for p in points)}) + "\n")
        out.flush()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_multi(args, rank, out):
    """ONE host process, 1 .. all visible GPUs: the C3 batch (1024 x 256 KiB, level 6) and the C2 batch (256 x 1 MiB) through
    b200z_deflate_batch_multi / b200z_inflate_batch_multi on pinned host memory -- strong scaling through the C-ABI, host
    clock around whole calls (staging, H2D, kernels, packed D2H, hand-over), outputs compared with the oracle / originals."""
    import torch
    import oracle_lib as O
    import sharpziplib_b200 as z
    if rank != 0:
        return
    z.init(0)
    ndev = z.lib().b200z_device_count()
    n_def = N_DEFLATE // (8 if args.small else 1)
    n_inf = N_INFLATE // (8 if args.small else 1)
    ncpu = host_threads()
    d_np, t_np = make_inputs(0, n_def, n_inf, max(1, min(32, ncpu)))
    O.build()
    comp = O.batch(0, [a.tobytes() for a in t_np], level=6, threads=ncpu)
    refs = O.batch(0, [a.tobytes() for a in d_np[::max(1, n_def // 32)]], level=6, threads=ncpu)

    def pinned(arrs):
        t = torch.empty(sum(len(a) for a in arrs) + 64, dtype=torch.uint8).pin_memory()
        ptrs, pos = [], 0
        for a in arrs:
            n = len(a)
            t[pos:pos + n] = torch.frombuffer(bytearray(a), dtype=torch.uint8) if isinstance(a, (bytes, bytearray)) else torch.from_numpy(a)
            ptrs.append(t.data_ptr() + pos)
            pos += n
        return t, ptrs

    P = z.Pipeline
    h_din, din_ptrs = pinned(d_np)
    h_iin, iin_ptrs = pinned(comp)
    dlens = np.array([a.size for a in d_np], dtype=np.int64)
    clens = np.array([len(c) for c in comp], dtype=np.int64)
    dcaps = np.array([z.lib().b200z_deflate_bound(int(a.size)) + 16 for a in d_np], dtype=np.int64)
    icaps = np.array([a.size for a in t_np], dtype=np.int64)
    h_dout = torch.empty(int(dcaps.sum()) + 64, dtype=torch.uint8).pin_memory()
    h_iout = torch.empty(int(icaps.sum()) + 64, dtype=torch.uint8).pin_memory()
    dout_off = np.concatenate([[0], np.cumsum(dcaps)[:-1]]).astype(np.int64)
    iout_off = np.concatenate([[0], np.cumsum(icaps)[:-1]]).astype(np.int64)
    din_p, iin_p = P.pointers(din_ptrs), P.pointers(iin_ptrs)
    dout_p = P.pointers([h_dout.data_ptr() + int(o) for o in dout_off])
    iout_p = P.pointers([h_iout.data_ptr() + int(o) for o in iout_off])
    dl, il, iu = np.zeros(n_def, dtype=np.int64), np.zeros(n_inf, dtype=np.int64), np.zeros(n_inf, dtype=np.int64)
    dck, ick = np.zeros(n_def, dtype=np.uint32), np.zeros(n_inf, dtype=np.uint32)
    dst, ist = np.zeros(n_def, dtype=np.int32), np.zeros(n_inf, dtype=np.int32)
    L = z.lib()
    U_def, U_inf = int(dlens.sum()), int(icaps.sum())
    rows = []
    nd = 1
    while nd <= ndev:
        dv = np.arange(nd, dtype=np.int32)

        def step():
            rc = L.b200z_deflate_batch_multi(dv.ctypes.data, nd, din_p, dlens.ctypes.data, n_def, 6, 0, 0, 0, dout_p, dcaps.ctypes.data,
                                             dl.ctypes.data, dck.ctypes.data, dst.ctypes.data)
            assert rc == 0, rc
            rc = L.b200z_inflate_batch_multi(dv.ctypes.data, nd, iin_p, clens.ctypes.data, n_inf, 0, iout_p, icaps.ctypes.data, il.ctypes.data,
                                             iu.ctypes.data, ick.ctypes.data, ist.ctypes.data)
            assert rc == 0, rc
        for _ in range(2):
            step()
        hd = h_dout.numpy()
        for k, i in enumerate(range(0, n_def, max(1, n_def // 32))):
            assert hd[dout_off[i]:dout_off[i] + int(dl[i])].tobytes() == refs[k], "deflate parity, %d devices, buffer %d" % (nd, i)
        hi = h_iout.numpy()
        for i in range(0, n_inf, max(1, n_inf // 16)):
            assert np.array_equal(hi[iout_off[i]:iout_off[i] + t_np[i].size], t_np[i]), "inflate, %d devices, stream %d" % (nd, i)
        reps = max(3, min(args.steps, 5))
        t0 = time.perf_counter()
        for _ in range(reps):
            step()
        dt = (time.perf_counter() - t0) / reps
        rows.append({"devices": nd, "ms_per_step": dt * 1e3, "gbs": (U_def + U_inf) / dt / 1e9})
        nd *= 2
    for r in rows:
        r["efficiency_vs_1"] = r["gbs"] / (rows[0]["gbs"] * r["devices"])
    out.write(json.dumps({"config": "multi", "workload": workload_name(n_def, n_inf).replace(" per GPU", " in all (strong scaling)"),
                          "how": "one host process, b200z_*_batch_multi on pinned host memory, synchronous calls (no overlap between steps), host clock",
                          "host_threads": ncpu, "rows": rows}) + "\n")
    out.flush()
    z.lib().b200z_release_cached()


if __name__ == "__main__":
    main()
