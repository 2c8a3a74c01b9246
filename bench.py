#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native fastp hot path.

A "step" is one pass of the per-read operator chain over one batch of synthetic 2x150 bp read pairs
(BASELINE.json configs[2]: PE, overlap adapter trimming + --correction) that is already resident in
HBM.  N GPUs: every rank processes its own shard of the same size (weak scaling, no data-path
collective) and the int64 counter block is all-reduced (NCCL sum) once per step.

  python bench.py --gpus N --steps K --warmup W            # this framework
  python bench.py --impl reference ...                     # the reference's own CPU code (oracle/_ref)

Prints ONE JSON line (rank 0).  torch is plumbing only (device memory, streams, torch.distributed).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TRUSEQ_R1 = "AGATCGGAAGAGCACACGTCTGAACTCCAGTCA"
TRUSEQ_R2 = "AGATCGGAAGAGCGTCGTGTAGGGAAAGAGTGT"
READ_LEN, STRIDE = 150, 160
BYTES_PER_PAIR = 4 * READ_LEN + 32          # SURVEY.md 8(d): 4*L in + two 16-byte fp_read_result out
SEED = 42


# BASELINE.json configs -> bench workloads.  configs[0] (testdata, CPU plumbing) is a parity test, not a bench line.
WORKLOADS = {
    "pe150_overlap_correction": dict(cfg="configs[2]", paired=1, L=150, S=160, units=100_000_000, profile=1),
    "pe150_full":               dict(cfg="configs[3]", paired=1, L=150, S=160, units=125_000_000, profile=1),
    "se150_cut_right_polyg":    dict(cfg="configs[1]", paired=0, L=150, S=160, units=10_000_000, profile=1),
    "pe250_overrep":            dict(cfg="configs[4]", paired=1, L=250, S=256, units=12_500_000, profile=3),
}
OVERREP_PRESCAN_UNITS = 8192        # > 151*10000 / 250 reads: what Evaluator::computeOverRepSeq looks at (evaluator.cpp:83)


def metric_string(paired, L):
    """ONE string for both arms (the driver divides the two lines only when `metric` matches)."""
    return (f"{'pairs' if paired else 'reads'} per second, {L} bp {'PE' if paired else 'SE'} synthetic FASTQ"
            + (" (1 pair = 2 reads: reads_per_s = 2 x value)" if paired else ""))


def bytes_per_unit(paired, L):
    return (4 * L + 32) if paired else (2 * L + 16)     # SURVEY.md 8(d)


def workload_params(capi, lib, name, overrep=None):
    """fp_params of the named BASELINE.json config.  overrep = (candidates1, candidates2) for pe250_overrep."""
    if name == "pe150_overlap_correction":      # configs[2]
        return capi.default_params(1, lib=lib, correction_enabled=1)
    if name == "pe150_full":                    # configs[3]
        return capi.default_params(1, lib=lib, cut_right=1, polyg_enabled=1, polyx_enabled=1, correction_enabled=1,
                                   adapter_seq_r1=TRUSEQ_R1, adapter_seq_r2=TRUSEQ_R2)
    if name == "se150_cut_right_polyg":         # configs[1]
        return capi.default_params(0, lib=lib, cut_right=1, polyg_enabled=1, adapter_enabled=0)
    if name == "pe250_overrep":                 # configs[4]: -p, sampling 20 (options.h:71-80), candidates from the host pre-scan
        c1, c2 = overrep if overrep is not None else ([], [])
        return capi.default_params(1, lib=lib, overrep_enabled=1, overrep_sampling=20, seq_len1=250, seq_len2=250,
                                   overrep_seqs1=c1, overrep_seqs2=c2)
    raise KeyError(name)


def host_overrep_candidates(lib, seq, lens, stride, seqlen):
    """Evaluator::computeOverRepSeq equivalent of the product library (host pre-scan, control plane) on rows in host memory."""
    from fastp_b200 import capi
    n_out = C.c_int32(); used = C.c_int64()
    cap = 1 << 22
    buf = C.create_string_buffer(cap)
    capi.check(lib.fp_host_overrep_candidates(seq.ctypes.data, lens.ctypes.data, seq.shape[0], stride, seqlen, buf, cap,
                                              C.byref(n_out), C.byref(used)), lib)
    return [x.decode() for x in buf.raw[:used.value].split(b"\0")[:-1]]


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def bind_to_gpu_numa(torch, dev_index):
    """Pin this process (and the threads / pinned buffers it creates from here on) to the NUMA node the GPU hangs off: host staging that
    sits on the other socket costs a third of the H2D rate.  Returns what was done (goes into the e2e object)."""
    try:
        pr = torch.cuda.get_device_properties(dev_index)
        bus = None
        if hasattr(pr, "pci_bus_id") and hasattr(pr, "pci_device_id"):
            bus = f"{getattr(pr, 'pci_domain_id', 0):04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        else:
            import pynvml
            pynvml.nvmlInit()
            hnd = pynvml.nvmlDeviceGetHandleByIndex(dev_index)
            b = pynvml.nvmlDeviceGetPciInfo(hnd).busId
            bus = (b.decode() if isinstance(b, bytes) else b).lower()[-12:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return {"pci": bus, "node": None}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"pci": bus, "node": node, "cpus_bound": len(cpus)}
    except Exception as e:      # a hint, never a reason to fail
        return {"error": repr(e)}


def cpu_resources():
    """Threads this process may use: affinity mask and the cgroup CPU quota (a 128-core box leased with a quota reports 128)."""
    aff = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        f = open("/sys/fs/cgroup/cpu.max").read().split()
        if f[0] != "max":
            quota = float(f[0]) / float(f[1])
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    usable = aff if not quota else max(1, min(aff, int(quota + 0.999)))
    return {"os_cpu_count": os.cpu_count(), "affinity": aff, "cgroup_quota_cpus": quota, "usable": usable}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# CPU legs (the ONLY places bench.py touches oracle/): cpu_baseline and --impl reference
# ------------------------------------------------------------------------------------------------
def load_cpu_checker():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import fp_testlib as T
    if T.have_ref():
        return T, "reference"
    return T, "port"


def synth_host_parallel(T, n, W, first, profile, threads):
    from fastp_b200 import capi
    b, arrs = capi.host_batch(n, W["S"], W["paired"])
    lib = T.oracle()
    bounds = [n * i // threads for i in range(threads + 1)]

    def work(i):
        lo, hi = bounds[i], bounds[i + 1]
        if hi <= lo:
            return
        sub = {k: v[lo:hi] for k, v in arrs.items()}
        sb = capi.batch_from_arrays(sub)
        lib.fp_synth_fill_host(C.byref(sb), first + lo, SEED, profile, W["L"])
    ts = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    return b, arrs


def cpu_params(T, name, W, arrs):
    """fp_params for the CPU leg (same option set; the over-representation candidates come from the same pre-scan rule, here
    through the product's host function on the host-generated rows -- the checker for it is tests/test_overrep_prescan.py)."""
    from fastp_b200 import capi
    if name == "pe250_overrep":
        lib = capi.load()
        m = min(OVERREP_PRESCAN_UNITS, arrs["seq1"].shape[0])
        c = [host_overrep_candidates(lib, np.ascontiguousarray(arrs["seq" + sd][:m]), np.ascontiguousarray(arrs["len" + sd][:m]), W["S"], W["L"]) for sd in "12"]
        return workload_params(capi, T.oracle(), name, overrep=(c[0], c[1]))
    return workload_params(capi, T.oracle(), name)


def cpu_run(T, kind, params, W, arrs, threads):
    """One pass of the reference worker body over the sample on `threads` host threads.
    Returns (seconds inside the worker bodies, merged counter block).  The input copy (base correction rewrites rows in
    place, so every pass needs pristine rows) and the allocation of the counter block are OUTSIDE the clock."""
    from fastp_b200 import capi
    paired = bool(params.paired)
    a = {k: v.copy() for k, v in arrs.items()}
    b = capi.batch_from_arrays(a)
    L = capi.make_layout(T.oracle(), paired, W["S"], params.insert_size_max, params=params)
    cnt = np.zeros(L.total, np.int64)
    if kind == "reference":
        t0 = time.perf_counter()
        rc = T.ref().fp_ref_process_mt(C.byref(params), C.byref(L), C.byref(b), None, None, None, cnt.ctypes.data, threads)
        dt = time.perf_counter() - t0
        assert rc == 0
    else:
        # the C port is single-threaded per call: shard over python threads (ctypes drops the GIL)
        n = b.n
        bounds = [n * i // threads for i in range(threads + 1)]
        outs = []

        def work(i):
            lo, hi = bounds[i], bounds[i + 1]
            if hi <= lo:
                return
            sub = {k: v[lo:hi] for k, v in a.items()}
            sb = capi.batch_from_arrays(sub)
            o1 = np.zeros(hi - lo, capi.READ_RESULT_DTYPE); o2 = np.zeros(hi - lo, capi.READ_RESULT_DTYPE)
            c = np.zeros(L.total, np.int64)
            T.oracle().fp_oracle_process(C.byref(params), C.byref(L), C.byref(sb), o1.ctypes.data, o2.ctypes.data if paired else None,
                                         None, c.ctypes.data)
            outs.append(c)
        ts = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
        t0 = time.perf_counter()
        [t.start() for t in ts]
        [t.join() for t in ts]
        dt = time.perf_counter() - t0
        for c in outs:
            cnt += c
    return dt, (L, cnt)


def cpu_baseline(name, profile=None, target_seconds=10.0, max_units=6_000_000):
    """The reference's worker body (oracle/_ref, else the C port) on a bounded sample of the workload's own stream."""
    T, kind = load_cpu_checker()
    W = WORKLOADS[name]
    profile = W["profile"] if profile is None else profile
    res = cpu_resources()
    cores = res["usable"]                        # threads actually used: the affinity mask capped by the cgroup CPU quota
    probe_n = 20000 * max(1, min(cores, 16))
    _, arrs = synth_host_parallel(T, probe_n, W, 0, profile, min(cores, 32))
    params = cpu_params(T, name, W, arrs)
    dt, blk = cpu_run(T, kind, params, W, arrs, cores)
    rate = probe_n / dt
    n = int(min(max(rate * target_seconds, probe_n), max_units))
    if n > probe_n:
        _, arrs = synth_host_parallel(T, n, W, 0, profile, min(cores, 32))
        dt, blk = cpu_run(T, kind, params, W, arrs, cores)
    else:
        n = probe_n
    unit = "pairs/s" if W["paired"] else "reads/s"
    note = ""
    if name == "pe250_overrep":
        note = "; over-representation counts of this multi-threaded run sample per worker thread (SURVEY App. C): timing only"
    return ({"value": n / dt, "unit": unit, "cores": cores, "kind": kind, "cpu": res,
             "sample": f"first {n} units of the same synthetic stream (seed {SEED}, profile {profile}), in-memory batches, "
                       f"{cores} worker threads each with private Stats/FilterResult, {dt:.2f} s inside the worker bodies{note}"},
            dict(T=T, kind=kind, params=params, arrs=arrs, n=n, block=blk, W=W))


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from fastp_b200 import capi  # noqa: F401  (ctypes structs + the host pre-scan only; no CUDA is touched on this arm)
    W = WORKLOADS[args.workload]
    base, ctx = cpu_baseline(args.workload, args.profile, target_seconds=6.0)
    T, kind, params, arrs, n = ctx["T"], ctx["kind"], ctx["params"], ctx["arrs"], ctx["n"]
    cores = base["cores"]
    for _ in range(args.warmup):
        cpu_run(T, kind, params, W, arrs, cores)
    dt = 0.0
    for _ in range(args.steps):
        dt += cpu_run(T, kind, params, W, arrs, cores)[0]      # seconds inside fp_ref_process_mt only
    value = n * args.steps / dt
    unit = "pairs/s" if W["paired"] else "reads/s"
    line = {
        "impl": "reference", "metric": metric_string(W["paired"], W["L"]),
        "value": value, "unit": unit, "reads_per_s": value * (2 if W["paired"] else 1), "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": args.workload, "baseline_config": W["cfg"], "units_per_step": n, "read_len": W["L"],
                   "profile": W["profile"] if args.profile is None else args.profile, "threads": cores,
                   "note": "reference worker body (unmodified objects, scalar simd shim) on in-memory batches; the clock covers the worker "
                           "bodies only (input copy / allocation outside)"},
        "cpu_baseline": {"value": value, "unit": unit, "cores": cores, "kind": kind, "cpu": base["cpu"],
                         "sample": f"{n} units per step x {args.steps} steps, in-memory batches, {cores} threads"},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------

def fastq_text_np(np, seq, qual, lens, tag):
    """FASTQ text of one side as a uint8 array, vectorised (names @SIM:1:<9 digits> <tag>, '+' strand lines)."""
    n, S = seq.shape
    lens = lens.astype(np.int64)
    name = np.frombuffer(("@SIM:1:000000000 " + tag + "\n").encode(), np.uint8)
    nl = name.size
    rec = nl + 2 * lens + 4                                   # name\n seq\n +\n qual\n  (name already holds its \n)
    off = np.concatenate([[0], np.cumsum(rec)[:-1]])
    out = np.zeros(int(rec.sum()), np.uint8)
    idx = np.arange(n)
    for k in range(nl):
        out[off + k] = name[k]
    for d in range(9):                                        # decimal digits of the index, most significant first
        out[off + 7 + d] = 48 + (idx // 10 ** (8 - d)) % 10
    col = np.arange(S)[None, :]
    m = col < lens[:, None]
    rows = np.nonzero(m)
    out[(off + nl)[rows[0]] + rows[1]] = seq[m]
    out[off + nl + lens] = 10
    out[off + nl + lens + 1] = 43
    out[off + nl + lens + 2] = 10
    out[(off + nl + lens + 3)[rows[0]] + rows[1]] = qual[m]
    out[off + nl + 2 * lens + 3] = 10
    return out


def fastq_path(args, torch, capi, lib, params, paired, dev, unit):
    """Text in -> text out through fp_fastq_process_host (pinned host buffers; H2D of the raw text, device parse, operator chain,
    device encode, D2H of the output text inside the timed region), the two codec kernels' own throughput on HBM-resident text,
    and the unmodified reference CLI on the same files with all host threads."""
    import numpy as np
    nf = args.fastq_units
    gen = min(nf, 250_000)                                    # the text of `gen` units is tiled up to nf
    hctx = C.c_void_p()
    capi.check(lib.fp_ctx_create(C.byref(params), torch.cuda.current_device(), nf, STRIDE, STRIDE, C.byref(hctx)), lib)
    t = {k: torch.empty(gen * (2 if k.startswith("len") else STRIDE), dtype=torch.uint8, device=dev)
         for k in (["seq1", "qual1", "len1"] + (["seq2", "qual2", "len2"] if paired else []))}
    b = capi.Batch(); b.n, b.stride = gen, STRIDE
    for k, v in t.items():
        setattr(b, k, v.data_ptr())
    capi.check(lib.fp_synth_fill(hctx, C.byref(b), 0, SEED, WORKLOADS[args.workload]["profile"] if args.profile is None else args.profile, READ_LEN, None), lib)
    torch.cuda.synchronize()
    reps = max(1, nf // gen)
    nf = gen * reps
    texts = []
    for side in ("1", "2")[: 2 if paired else 1]:
        seq = t["seq" + side].cpu().numpy().reshape(gen, STRIDE); qual = t["qual" + side].cpu().numpy().reshape(gen, STRIDE)
        lens = t["len" + side].cpu().numpy().view(np.uint16)
        one = fastq_text_np(np, seq, qual, lens, side + ":N:0")
        texts.append(np.tile(one, reps))
    del t
    pin = [torch.from_numpy(x).pin_memory() for x in texts]
    outs = [torch.empty(x.numel() + 64, dtype=torch.uint8).pin_memory() for x in pin]
    ob = [C.c_int64(), C.c_int64()]; nu = C.c_int64(); c1 = C.c_int64(); c2 = C.c_int64()
    i1, i2 = capi.FastqInfo(), capi.FastqInfo()

    def call():
        capi.check(lib.fp_fastq_process_host(hctx, pin[0].data_ptr(), pin[0].numel(), pin[1].data_ptr() if paired else None, pin[1].numel() if paired else 0, 1, 0,
                                             outs[0].data_ptr(), outs[0].numel(), C.byref(ob[0]),
                                             outs[1].data_ptr() if paired else None, outs[1].numel() if paired else 0, C.byref(ob[1]) if paired else None,
                                             C.byref(nu), C.byref(c1), C.byref(c2) if paired else None, C.byref(i1), C.byref(i2) if paired else None), lib)
    for _ in range(2):
        call()
    assert nu.value == nf, (nu.value, nf)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        call()
    dt = (time.perf_counter() - t0) / args.steps
    # two worker threads, one context each (the reference runs one ThreadConfig per worker): the H2D of one overlaps the D2H of the other
    import threading
    h2 = C.c_void_p()
    capi.check(lib.fp_ctx_create(C.byref(params), torch.cuda.current_device(), nf, STRIDE, STRIDE, C.byref(h2)), lib)
    outs2 = [torch.empty(x.numel() + 64, dtype=torch.uint8).pin_memory() for x in pin]

    def worker(hc, ob_):
        o = [C.c_int64(), C.c_int64()]; n_ = C.c_int64(); a_ = C.c_int64(); b_ = C.c_int64(); j1, j2 = capi.FastqInfo(), capi.FastqInfo()
        for _ in range(args.steps):
            capi.check(lib.fp_fastq_process_host(hc, pin[0].data_ptr(), pin[0].numel(), pin[1].data_ptr() if paired else None, pin[1].numel() if paired else 0, 1, 0,
                                                 ob_[0].data_ptr(), ob_[0].numel(), C.byref(o[0]),
                                                 ob_[1].data_ptr() if paired else None, ob_[1].numel() if paired else 0, C.byref(o[1]) if paired else None,
                                                 C.byref(n_), C.byref(a_), C.byref(b_) if paired else None, C.byref(j1), C.byref(j2) if paired else None), lib)
    worker(h2, outs2)
    th = [threading.Thread(target=worker, args=(hctx, outs), daemon=True), threading.Thread(target=worker, args=(h2, outs2), daemon=True)]
    t0 = time.perf_counter()
    for x in th:
        x.start()
    for x in th:
        x.join(timeout=120)
    if any(x.is_alive() for x in th):
        raise RuntimeError("two-worker text path did not finish within 120 s")
    dt2 = (time.perf_counter() - t0) / (2 * args.steps)
    lib.fp_ctx_destroy(h2)
    in_bytes = sum(int(x.numel()) for x in pin); out_bytes = ob[0].value + (ob[1].value if paired else 0)
    res = {"value": nf / dt, "unit": unit, "units_per_step": nf, "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": out_bytes,
           "text_GBps_in": in_bytes / dt / 1e9, "api": "fp_fastq_process_host", "two_workers": {"value": nf / dt2, "unit": unit, "text_GBps_in": in_bytes / dt2 / 1e9},
           "note": "plain FASTQ text in pinned host memory -> H2D -> device decode (FastqReader::read) -> operator chain -> device encode "
                   "(Read::appendToString) -> D2H of the output text"}
    # codec kernels alone, text and rows resident in HBM
    d_text = pin[0].to(dev)
    d_seq = torch.empty(nf * STRIDE + 64, dtype=torch.uint8, device=dev); d_qual = torch.empty_like(d_seq)
    d_len = torch.empty(nf * 2, dtype=torch.uint8, device=dev); d_recs = torch.empty(nf * 16, dtype=torch.uint8, device=dev)
    info = capi.FastqInfo()

    def dec():
        capi.check(lib.fp_fastq_decode(hctx, d_text.data_ptr(), d_text.numel(), 1, 0, d_seq.data_ptr(), d_qual.data_ptr(), d_len.data_ptr(), nf,
                                       d_recs.data_ptr(), C.byref(info)), lib)
    dec(); dec()
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(args.steps):
        dec()
    torch.cuda.synchronize(); td = (time.perf_counter() - t0) / args.steps
    d_res = torch.zeros(nf * 16, dtype=torch.uint8, device=dev)
    d_res.view(torch.int16).view(nf, 8)[:, 1] = d_len.view(torch.int16)          # front 0, len = read length, verdicts PASS
    d_out = torch.empty(d_text.numel() + 64, dtype=torch.uint8, device=dev); tot = C.c_int64()

    def enc():
        capi.check(lib.fp_fastq_encode(hctx, d_text.data_ptr(), d_recs.data_ptr(), d_res.data_ptr(), d_seq.data_ptr(), d_qual.data_ptr(), nf,
                                       d_out.data_ptr(), d_out.numel(), C.byref(tot)), lib)
    enc(); enc()
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(args.steps):
        enc()
    torch.cuda.synchronize(); te = (time.perf_counter() - t0) / args.steps
    assert tot.value == d_text.numel(), (tot.value, d_text.numel())        # untouched reads re-encode to the input text
    tb = int(d_text.numel())
    res["decode"] = {"ms": td * 1e3, "text_GBps": tb / td / 1e9, "algorithmic_bytes": tb + 2 * nf * READ_LEN,
                     "achieved_GBps": (tb + 2 * nf * READ_LEN) / td / 1e9, "note": "one side; synchronous call incl. its host round trips"}
    res["encode"] = {"ms": te * 1e3, "text_GBps": tb / te / 1e9, "achieved_GBps": (tb + 2 * nf * READ_LEN) / te / 1e9}
    lib.fp_ctx_destroy(hctx)
    # the unmodified reference CLI on the same text (plain files in a temp dir), all host threads, no output files
    cli = os.path.join(ROOT, "oracle", "_ref", "fastp_ref")
    if os.path.exists(cli) and not args.no_cpu_baseline:
        import subprocess
        import tempfile
        try:
            with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as d:
                names = []
                for k, x in enumerate(texts):
                    fn = os.path.join(d, f"r{k + 1}.fq"); x.tofile(fn); names.append(fn)
                flags = {"pe150_overlap_correction": ["-c"], "pe150_full": ["--cut_right", "-g", "-x", "-c", "-a", "AGATCGGAAGAGCACACGTCTGAACTCCAGTCA",
                                                                           "--adapter_sequence_r2", "AGATCGGAAGAGCGTCGTGTAGGGAAAGAGTGT"],
                         "se150_cut_right_polyg": ["--cut_right", "-g", "-A"]}[args.workload]
                # 16 worker threads (about a second for 1 M pairs).  The one bench run that asked for one thread per core of the 128-core
                # GPU box (-w 128) was still running when its 6-minute limit killed it, so the CLI arm stays at 16 and is capped at 90 s;
                # the in-memory reference arm (cpu_baseline / --impl reference) does use every core
                thr = min(os.cpu_count() or 1, 16)
                cmd = [cli, "-i", names[0], "-w", str(thr), "--dont_eval_duplication", "-j", os.path.join(d, "x.json"), "-h", os.path.join(d, "x.html")] + flags
                if paired:
                    cmd += ["-I", names[1]]
                t0 = time.perf_counter()
                subprocess.run(cmd, check=True, capture_output=True, cwd=d, timeout=90)
                tc = time.perf_counter() - t0
            res["cpu_cli"] = {"value": nf / tc, "unit": unit, "threads": thr, "seconds": tc,
                              "sample": f"{nf} units, unmodified reference CLI (oracle/_ref/fastp_ref, plain FASTQ in a RAM-backed dir, no output files, -w {thr}; wall clock of the whole process incl. start-up)"}
        except Exception as e:
            res["cpu_cli"] = {"value": None, "sample": repr(e)}
    return res


class _Raw:
    """Expose a raw device pointer to torch (zero-copy) through __cuda_array_interface__."""

    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 3}


DUMP_SAMPLE_UNITS = 1 << 18       # per-read records of this many units (seeded sample, sorted indices) go into the dump


def dump_outputs(path, torch, capi, n, cnt, out1, out2, ov, patches, npatch):
    """Write what the last timed pass handed back to its caller as DIR/<name>.npy (float32, float64 where an integer can pass
    2**24): the whole counter block, every field of the per-read and overlap records of a fixed sample of units, and the
    correction patches of those units sorted by (unit, read, position).  Two builds run with the same arguments see the same
    inputs, so their dumps compare array for array."""
    os.makedirs(path, exist_ok=True)
    m = min(n, DUMP_SAMPLE_UNITS)
    idx = np.sort(np.random.default_rng(SEED).choice(n, size=m, replace=False))
    it = torch.from_numpy(idx).to(out1.device)
    arrays = {"sample_index": idx.astype(np.float64), "counters": cnt.astype(np.float64)}
    for tag, buf, dt in (("out1", out1, capi.READ_RESULT_DTYPE), ("out2", out2, capi.READ_RESULT_DTYPE), ("ov", ov, capi.OV_RESULT_DTYPE)):
        if buf is None:
            continue
        rec = buf.view(n, dt.itemsize)[it].cpu().numpy().view(dt).reshape(m)
        for f in dt.names:
            if f != "reserved":
                arrays[f"{tag}_{f}"] = rec[f].astype(np.float32)
    if patches is not None:
        k = int(npatch.item())
        rows = patches[: min(k, patches.numel() // 12) * 12].view(-1, 12)
        keep = torch.zeros(n, dtype=torch.bool, device=out1.device)
        keep[it] = True
        rows = rows[keep[rows[:, :4].contiguous().view(torch.int32).view(-1).long()]]
        pt = np.sort(rows.cpu().numpy().view(capi.PATCH_DTYPE).reshape(-1), order=["pair", "which", "pos"])
        arrays["patch_count"] = np.array([k], np.float64)
        arrays["patch_unit"] = pt["pair"].astype(np.float64)
        for f in ("pos", "which", "base", "qual", "old_base", "old_qual"):
            arrays[f"patch_{f}"] = pt[f].astype(np.float32)
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64 << 20, f"dump of {total} bytes"
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def gpu_workload(name, args, env, units, steps, warmup, with_e2e=False, dump_dir=None):
    """W warm-up + K timed passes of one BASELINE config over a batch resident in HBM; returns the result dict
    (value, roofline, checks, ...).  env: torch, dist, capi, lib, world, rank, local_rank, dev, comm.
    dump_dir: write the outputs of the last timed pass there (dump_outputs)."""
    torch, dist, capi, lib = env["torch"], env["dist"], env["capi"], env["lib"]
    world, rank, local_rank, dev = env["world"], env["rank"], env["local_rank"], env["dev"]
    W = WORKLOADS[name]
    paired, L_, S = bool(W["paired"]), W["L"], W["S"]
    profile = W["profile"] if args.profile is None else args.profile
    unit = "pairs/s" if paired else "reads/s"
    sides = 2 if paired else 1
    torch.cuda.empty_cache()
    free_b, _ = torch.cuda.mem_get_info()
    per_unit = sides * (2 * S + 2 + 16) + (8 + 15 if paired else 0)
    n = int(min(units, 0.85 * free_b / per_unit))
    if dump_dir is not None and n < units:
        raise SystemExit(f"bench.py --dump-outputs: {units} units do not fit in free device memory ({free_b / 1e9:.1f} GB); "
                         "a smaller batch would change the inputs")
    first = rank * n                                   # rank r owns global indices [r*n, (r+1)*n)

    def alloc(nbytes):
        return torch.empty(int(nbytes), dtype=torch.uint8, device=dev)

    # ---- over-representation candidates: host pre-scan (Evaluator::computeOverRepSeq) of the START of the global stream ----
    overrep = None
    if name == "pe250_overrep":
        m = OVERREP_PRESCAN_UNITS
        p0 = capi.default_params(1, lib=lib)
        h0 = C.c_void_p()
        capi.check(lib.fp_ctx_create(C.byref(p0), local_rank, m, S, S, C.byref(h0)), lib)
        tt = {k: alloc(m * (2 if k.startswith("len") else S)) for k in ("seq1", "qual1", "len1", "seq2", "qual2", "len2")}
        b0 = capi.Batch(); b0.n, b0.stride = m, S
        for k, v in tt.items():
            setattr(b0, k, v.data_ptr())
        capi.check(lib.fp_synth_fill(h0, C.byref(b0), 0, SEED, profile, L_, None), lib)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        overrep = tuple(host_overrep_candidates(lib, tt["seq" + sd].cpu().numpy().reshape(m, S), tt["len" + sd].cpu().numpy().view(np.uint16), S, L_)
                        for sd in "12")
        prescan_s = time.perf_counter() - t0
        lib.fp_ctx_destroy(h0)
        del tt
    params = workload_params(capi, lib, name, overrep=overrep)
    has_ovr = bool(params.overrep_enabled)

    h = C.c_void_p()
    capi.check(lib.fp_ctx_create(C.byref(params), local_rank, min(n, 1 << 18), S, S, C.byref(h)), lib)
    Lc = capi.CounterLayout()
    capi.check(lib.fp_ctx_layout(h, C.byref(Lc)), lib)
    t = {"seq1": alloc(n * S), "qual1": alloc(n * S), "len1": alloc(n * 2)}
    if paired:
        t.update(seq2=alloc(n * S), qual2=alloc(n * S), len2=alloc(n * 2))
    out1 = alloc(n * 16)
    out2 = alloc(n * 16) if paired else None
    ov = alloc(n * 8) if paired else None
    corr = paired and bool(params.correction_enabled)
    patch_cap = int(1.25 * n) + 4096 if corr else 0      # measured: 0.67 corrected bases per pair on the enriched profile
    patches = alloc(patch_cap * 12) if corr else None
    npatch = torch.zeros(1, dtype=torch.int32, device=dev) if corr else None
    b = capi.Batch()
    b.n, b.stride = n, S
    b.flags, b.first_read_index = 1, first              # FP_B_INDEXED: pre-filter over-representation sampling by GLOBAL index
    for k, v in t.items():
        setattr(b, k, v.data_ptr())
    capi.check(lib.fp_synth_fill(h, C.byref(b), first, SEED, profile, L_, None), lib)
    torch.cuda.synchronize()
    stream = torch.cuda.Stream(device=dev)
    sp = C.c_void_p(stream.cuda_stream)
    if has_ovr and world > 1:
        capi.check(lib.fp_overrep_defer_post(h, 1), lib)
    from fastp_b200 import sharding

    def run_pass(bb, o1, o2, ovp, undo=True):
        """one pass of the hot path over batch bb (+ the cross-rank exchanges of a sharded run)"""
        capi.check(lib.fp_counters_reset(h), lib)
        if corr:
            with torch.cuda.stream(stream):
                npatch.zero_()
        if paired:
            capi.check(lib.fp_process_pe(h, C.byref(bb), o1, o2, ovp, patches.data_ptr() if corr else None, patch_cap,
                                         npatch.data_ptr() if corr else None, sp), lib)
        else:
            capi.check(lib.fp_process_se(h, C.byref(bb), o1, sp), lib)
        if has_ovr and world > 1:
            # post-filter sampling counts PASSING reads of the whole stream: exclusive scan of the shards' pass counts (8e)
            cnt = C.c_int64()
            capi.check(lib.fp_pass_count(h, o1, bb.n, C.byref(cnt), sp), lib)
            base, _ = sharding.exclusive_pass_base(cnt.value, device=dev)
            capi.check(lib.fp_overrep_post(h, C.byref(bb), o1, o2, base, sp), lib)
        if corr and undo:
            # base correction rewrites rows in place: put the old bases back so the NEXT pass corrects again (inside the timed region)
            capi.check(lib.fp_patches_undo(h, C.byref(bb), patches.data_ptr(), npatch.data_ptr(), patch_cap, sp), lib)
        if world > 1:
            capi.check(lib.fp_counters_allreduce(h, env["comm"].handle, sp), lib)     # Stats::merge / FilterResult::merge are plain sums

    def step():
        run_pass(b, out1.data_ptr(), out2.data_ptr() if paired else None, ov.data_ptr() if paired else None)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        step()
    barrier()
    ms_tmp = C.c_double(); nl = C.c_int64()
    capi.check(lib.fp_kernel_time_ms(h, C.byref(ms_tmp), C.byref(nl), 1), lib)   # reset kernel timers
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(steps):
        step()
    ev1.record(stream)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    elapsed_ms = ev0.elapsed_time(ev1)
    if world > 1:
        tt_ = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tt_, op=dist.ReduceOp.MAX)
        elapsed_ms = float(tt_.item())
    capi.check(lib.fp_kernel_time_ms(h, C.byref(ms_tmp), C.byref(nl), 1), lib)
    kernel_ms = ms_tmp.value / max(nl.value, 1)

    # ---- size-independent invariants of the last full-size pass (the block is the job's total after the all-reduce) ----
    cnt = np.zeros(Lc.total, np.int64)
    capi.check(lib.fp_counters_fetch(h, cnt.ctypes.data), lib)
    cv = capi.CounterView(Lc, cnt)
    if dump_dir is not None and rank == 0:     # before the parity pass below overwrites the records and the counter block
        dump_outputs(dump_dir, torch, capi, n, cnt, out1, out2, ov, patches, npatch)
    total_units = n * world
    checks = {
        "pre_reads_eq_units": bool(cv.stats(capi.STATS_PRE1)["reads"] == total_units),
        "verdicts_sum": bool(int(cv.filter[:32].sum()) == total_units * sides),
        "post_le_pre": bool(cv.stats(capi.STATS_POST1)["reads"] <= cv.stats(capi.STATS_PRE1)["reads"]),
        "qualhist_eq_bases": bool(int(cv.stats(capi.STATS_PRE1)["qualhist"].sum()) == cv.stats(capi.STATS_PRE1)["length_sum"]),
    }
    if corr:
        checks["corrected_reads_gt0_in_timed_steps"] = bool(int(cv.filter[106]) > 0)     # FP_FR_CORRECTED_READS
        checks["patch_list_complete"] = bool(int(npatch.item()) <= patch_cap)            # else the undo (and the next step) would be partial
    if has_ovr:
        checks["overrep_hits_gt0"] = bool(int(cv.overrep(capi.STATS_PRE1)[0].sum()) > 0)

    # ---- parity at scale: the whole counter block of the first units of the stream == the reference's (cpu leg) ----
    parity = None
    cpu = env.get("cpu", {}).get(name)
    if cpu is not None:
        # every rank takes an equal share of the CPU sample's prefix [0, m*world), at its place in the global stream
        m = min(cpu["n"] // world, n)
        bb = capi.Batch(); bb.n, bb.stride, bb.flags, bb.first_read_index = m, S, 1, rank * m
        for k, v in t.items():
            setattr(bb, k, v.data_ptr())
        if world > 1:     # ranks > 0 hold other indices: regenerate the prefix shard in place (the timed data is not needed any more)
            capi.check(lib.fp_synth_fill(h, C.byref(bb), rank * m, SEED, profile, L_, None), lib)
        torch.cuda.synchronize()
        run_pass(bb, out1.data_ptr(), out2.data_ptr() if paired else None, ov.data_ptr() if paired else None)      # (rows restored afterwards: e2e below reads them)
        got = np.zeros(Lc.total, np.int64)
        capi.check(lib.fp_counters_fetch(h, got.ctypes.data), lib)
        parity = {"units": m * world, "got": got}
    value = total_units * steps / (elapsed_ms / 1e3)
    peak, peak_src = measured_peak()
    bpu = bytes_per_unit(paired, L_)
    achieved = n * bpu / (kernel_ms / 1e3) / 1e9
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp)).get(name)
            if tj:
                traffic = tj["dram_bytes_per_unit"] * n
                traffic_src = "static: " + tj.get("source", "ncu --set full capture under profiles/") + ", scaled per launch (not measured in this run)"
        except Exception:
            pass
    res = {
        "metric": metric_string(paired, L_), "value": value, "unit": unit, "reads_per_s": value * sides,
        "ms_per_step": elapsed_ms / steps, "steps": steps, "warmup": warmup,
        "config": {"workload": name, "baseline_config": W["cfg"], "units_per_gpu": n, "read_len": L_, "stride": S,
                   "profile": {0: "ref-style", 1: "enriched", 2: "enriched+indels", 3: "enriched+planted over-represented sequences"}[profile],
                   "seed": SEED, "parallelism": f"shard{world}",
                   "l2_policy": "inputs (%.1f GB per GPU) larger than L2" % (n * sides * 2 * S / 1e9),
                   "note": ("every timed step corrects bases again: the pass's own patch list (old base / quality) is played back by "
                            "fp_patches_undo inside the timed region" if corr else "")
                           + (f"; over-representation candidates: {len(overrep[0])}+{len(overrep[1])} from the host pre-scan of the first "
                              f"{OVERREP_PRESCAN_UNITS} pairs ({prescan_s:.1f} s, outside the timed region)" if overrep else "")},
        "gpu_launches": int(nl.value),
        "checks": checks,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "kernel": "fp_chain2_kernel", "kernel_ms": kernel_ms,
                     "algorithmic_bytes_per_unit": bpu, "peak_source": peak_src},
        "clocks": clocks,
    }

    # ---- duplicate filter (SURVEY 8f rank 2) on the resident rows: Duplicate::checkRead / checkPair for every unit, in index order ----
    if with_e2e and rank == 0:
        try:
            nd = int(min(n, 20_000_000))
            bd = capi.Batch(); bd.n, bd.stride = nd, S
            for k, v in t.items():
                setattr(bd, k, v.data_ptr())
            flags_d = alloc(nd)
            capi.check(lib.fp_dup_check(h, C.byref(bd), 1, flags_d.data_ptr(), sp), lib)       # allocates the 1 GiB of bit arrays, warms up
            torch.cuda.synchronize()
            capi.check(lib.fp_dup_reset(h), lib)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(3):
                capi.check(lib.fp_dup_check(h, C.byref(bd), 1, flags_d.data_ptr(), sp), lib)
            e1.record(stream)
            torch.cuda.synchronize()
            dms = e0.elapsed_time(e1) / 3
            tot_d, dup_d = C.c_int64(), C.c_int64()
            capi.check(lib.fp_dup_totals(h, C.byref(tot_d), C.byref(dup_d)), lib)
            dbytes = sides * L_ + 1
            res["dup_filter"] = {"value": nd / (dms / 1e3), "unit": unit, "units": nd, "ms": dms, "accuracy_level": 1,
                                 "algorithmic_bytes_per_unit": dbytes, "achieved_GBps": nd * dbytes / (dms / 1e3) / 1e9,
                                 "frac_of_hbm_peak": nd * dbytes / (dms / 1e3) / 1e9 / measured_peak()[0],
                                 "duplicates_second_and_third_pass": int(dup_d.value),
                                 "note": "fp_dup_check: warp-per-unit hash + first-toucher table + commit (4 kernels); the second and third timed passes see every unit again, so all of them are duplicates"}
            del flags_d
        except Exception as e:
            res["dup_filter"] = {"value": None, "error": repr(e)}

    # ---- e2e: same metric through the host-buffer C-ABI call (H2D + kernel + D2H inside the timed region) ----
    if with_e2e:
        ne = int(min(args.e2e_units, n))
        hb = {}
        keys = ["seq1", "qual1"] + (["seq2", "qual2"] if paired else [])
        if world > 1:        # the parity pass above regenerated a prefix in place: refill this rank's own rows
            capi.check(lib.fp_synth_fill(h, C.byref(b), first, SEED, profile, L_, None), lib)
            torch.cuda.synchronize()
        HP = L_                                             # host row pitch = read length: no padding bytes over PCIe (re-pitched in HBM)
        for k in keys:
            hb[k] = torch.empty(ne * HP, dtype=torch.uint8).pin_memory()
            hb[k].view(ne, HP).copy_(t[k][: ne * S].view(ne, S)[:, :HP])
        for k in (["len1", "len2"] if paired else ["len1"]):
            hb[k] = torch.empty(ne * 2, dtype=torch.uint8).pin_memory()
            hb[k].copy_(t[k][: ne * 2])
        ho1 = torch.empty(ne * 16, dtype=torch.uint8).pin_memory()
        ho2 = torch.empty(ne * 16, dtype=torch.uint8).pin_memory() if paired else None
        hov = torch.empty(ne * 8, dtype=torch.uint8).pin_memory() if paired else None
        hp_cap = int(1.25 * ne) + 4096
        hpat = np.zeros(hp_cap, capi.PATCH_DTYPE) if corr else None
        hnp = C.c_uint64()
        hbt = capi.Batch()
        hbt.n, hbt.stride, hbt.flags, hbt.first_read_index = ne, HP, 1, first
        for k, v in hb.items():
            setattr(hbt, k, v.data_ptr())
        views = {k: hb[k].numpy().reshape(ne, HP) for k in keys}

        def e2e_step():
            capi.check(lib.fp_counters_reset(h), lib)
            if paired:
                capi.check(lib.fp_process_pe_host_patches(h, C.byref(hbt), ho1.data_ptr(), ho2.data_ptr(), hov.data_ptr(),
                                                          hpat.ctypes.data if corr else None, hp_cap if corr else 0, C.byref(hnp)), lib)
            else:
                capi.check(lib.fp_process_se_host(h, C.byref(hbt), ho1.data_ptr()), lib)

        def e2e_undo():       # harness only (outside the clock): put the corrected host bytes back so the next step corrects again
            if not corr:
                return
            k = int(min(hnp.value, hp_cap))
            pt = hpat[:k]
            for which, (sk, qk) in enumerate((("seq1", "qual1"), ("seq2", "qual2"))):
                sel = pt[pt["which"] == which]
                views[sk][sel["pair"], sel["pos"]] = sel["old_base"]
                views[qk][sel["pair"], sel["pos"]] = sel["old_qual"]
        for _ in range(max(1, min(warmup, 2))):
            e2e_step(); e2e_undo()
        barrier()
        dt = 0.0
        for _ in range(steps):
            t0 = time.perf_counter()
            e2e_step()
            torch.cuda.synchronize()
            dt += time.perf_counter() - t0
            e2e_undo()
        barrier()
        e2e_cnt = np.zeros(Lc.total, np.int64)
        capi.check(lib.fp_counters_fetch(h, e2e_cnt.ctypes.data), lib)
        if world > 1:
            tt_ = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(tt_, op=dist.ReduceOp.MAX)
            dt = float(tt_.item())
        h2d = ne * (sides * 2 * HP + sides * 2)
        d2h = ne * ((32 + 8) if paired else 16)
        e2e_val = ne * world * steps / dt
        PCIE_PEAK = 63.0
        soa = {"value": e2e_val, "unit": unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "api": "fp_process_pe_host_patches" if paired else "fp_process_se_host",
               "pcie": {"h2d_GBps": h2d * steps / dt / 1e9, "d2h_GBps": d2h * steps / dt / 1e9, "frac": h2d * steps / dt / 1e9 / PCIE_PEAK},
               "corrected_reads_last_step": int(capi.CounterView(Lc, e2e_cnt).filter[106]) if corr else None}
        # ---- the same call with FP_B_PACK2BIT: the library's host threads pack the bases to 2 bits chunk by chunk UNDER the copies
        #      (packing inside the clock, overlapped); qualities go up from the caller's rows as they are ----
        p2 = None
        try:
            nthr2 = int(os.environ.get("FP_BENCH_PACK_THREADS", "0")) or max(1, min(cpu_resources()["usable"] // max(world, 1) - 1, 32))
            capi.check(lib.fp_set_host_threads(h, nthr2), lib)
            hbt.flags = 1 | capi.FP_B_PACK2BIT
            for _ in range(2):
                e2e_step(); e2e_undo()
            barrier()
            t2 = 0.0
            for _ in range(steps):
                t0 = time.perf_counter()
                e2e_step()
                torch.cuda.synchronize()
                t2 += time.perf_counter() - t0
                e2e_undo()
            barrier()
            p2_cnt = np.zeros(Lc.total, np.int64)
            capi.check(lib.fp_counters_fetch(h, p2_cnt.ctypes.data), lib)
            if world > 1:
                tt_ = torch.tensor([t2], device=dev, dtype=torch.float64)
                dist.all_reduce(tt_, op=dist.ReduceOp.MAX)
                t2 = float(tt_.item())
            PB = (((HP + 3) // 4) + 3) & ~3
            n_N = int(sum(int((views[k] == ord("N")).sum()) for k in keys if k.startswith("seq")))
            h2d_2 = ne * sides * (PB + HP + 2) + n_N * 8
            p2 = {"value": ne * world * steps / t2, "unit": unit, "h2d_bytes_per_step": h2d_2, "d2h_bytes_per_step": d2h,
                  "api": ("fp_process_pe_host_patches" if paired else "fp_process_se_host") + " with FP_B_PACK2BIT", "pack_threads": nthr2,
                  "pcie": {"h2d_GBps": h2d_2 * steps / t2 / 1e9, "d2h_GBps": d2h * steps / t2 / 1e9, "frac": h2d_2 * steps / t2 / 1e9 / PCIE_PEAK},
                  "counters_eq_unpacked_path": bool(np.array_equal(p2_cnt, e2e_cnt))}
        except Exception as e:
            p2 = {"value": None, "error": repr(e)}
        hbt.flags = 1
        # ---- the same through the PACKED host rows (2-bit bases + N list + unpadded qualities): packing is inside the clock ----
        pk = None
        try:
            pitch_b, pitch_q = (L_ + 3) // 4, L_ + (L_ & 1)
            pbuf = {"npos": torch.empty(max(ne // 2, 4096) * 8, dtype=torch.uint8).pin_memory()}
            pb = capi.PackedBatch(); pb.pitch_b, pb.pitch_q = pitch_b, pitch_q
            for sd in ("1", "2")[:sides]:
                pbuf["bases" + sd] = torch.empty(ne * pitch_b + 64, dtype=torch.uint8).pin_memory()
                pbuf["qual" + sd] = torch.empty(ne * pitch_q + 64, dtype=torch.uint8).pin_memory()
                pbuf["len" + sd] = torch.empty(ne * 2, dtype=torch.uint8).pin_memory()
                for kk in ("bases", "qual", "len"):
                    setattr(pb, kk + sd, pbuf[kk + sd].data_ptr())
            pb.npos = pbuf["npos"].data_ptr(); pb.npos_cap = pbuf["npos"].numel() // 8
            nthr = max(1, min(cpu_resources()["usable"] // max(world, 1), 64))

            def packed_step():
                capi.check(lib.fp_counters_reset(h), lib)
                capi.check(lib.fp_host_pack_rows(C.byref(hbt), 1 if paired else 0, C.byref(pb), nthr), lib)
                if paired:
                    capi.check(lib.fp_process_pe_host_packed(h, C.byref(pb), ho1.data_ptr(), ho2.data_ptr(), hov.data_ptr(),
                                                             hpat.ctypes.data if corr else None, hp_cap if corr else 0, C.byref(hnp)), lib)
                else:
                    capi.check(lib.fp_process_se_host_packed(h, C.byref(pb), ho1.data_ptr()), lib)
            for _ in range(2):
                packed_step()
            barrier()
            tpk = 0.0; tpack = 0.0
            for _ in range(steps):
                t0 = time.perf_counter()
                packed_step()
                torch.cuda.synchronize()
                tpk += time.perf_counter() - t0
            t0 = time.perf_counter()
            capi.check(lib.fp_host_pack_rows(C.byref(hbt), 1 if paired else 0, C.byref(pb), nthr), lib)
            tpack = time.perf_counter() - t0
            barrier()
            pk_cnt = np.zeros(Lc.total, np.int64)
            capi.check(lib.fp_counters_fetch(h, pk_cnt.ctypes.data), lib)
            if world > 1:
                tt_ = torch.tensor([tpk], device=dev, dtype=torch.float64)
                dist.all_reduce(tt_, op=dist.ReduceOp.MAX)
                tpk = float(tt_.item())
            h2d_p = ne * sides * (pitch_b + pitch_q + 2) + int(pb.n_npos) * 8
            pk = {"value": ne * world * steps / tpk, "unit": unit, "h2d_bytes_per_step": h2d_p, "d2h_bytes_per_step": d2h + (int(min(hnp.value, hp_cap)) * 12 if corr else 0),
                  "api": "fp_host_pack_rows + " + ("fp_process_pe_host_packed" if paired else "fp_process_se_host_packed"),
                  "pack_threads": nthr, "pack_ms_alone": tpack * 1e3,
                  "pcie": {"h2d_GBps": h2d_p * steps / tpk / 1e9, "frac": h2d_p * steps / tpk / 1e9 / PCIE_PEAK},
                  "counters_eq_unpacked_path": bool(np.array_equal(pk_cnt, e2e_cnt))}
        except Exception as e:       # an alternative measurement: never a reason to lose the line
            pk = {"value": None, "error": repr(e)}
        best = soa
        for alt in (p2, pk):
            if alt and alt.get("value") and alt.get("counters_eq_unpacked_path") and alt["value"] > best["value"]:
                best = alt
        res["e2e"] = dict(best)
        res["e2e"].update({"units_per_step_per_gpu": ne, "numa": env.get("numa"), "pcie_peak_GBps": PCIE_PEAK, "pcie_peak_source": "PCIe Gen5 x16, 63 GB/s per direction nominal",
                           "soa_rows": soa, "pack2bit_rows": p2, "packed_rows": pk,
                           "host_row_pitch": HP, "note": "pinned host SoA rows at pitch = read length -> (FP_B_PACK2BIT: bases packed to 2 bits by the library's host threads, chunk by chunk under the copies; "
                                   "packed_rows: a separate fp_host_pack_rows pass; both inside the clock) -> chunked H2D on two streams -> kernel -> D2H of per-read records + correction "
                                   "patches; the headline value is the fastest of the host formats"})
    lib.fp_ctx_destroy(h)
    del t, out1, out2, ov, patches
    torch.cuda.empty_cache()
    return res, parity, params


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="pe150_overlap_correction", choices=sorted(WORKLOADS))
    ap.add_argument("--units", type=int, default=0, help="reads/pairs per GPU per step (default: BASELINE config size)")
    ap.add_argument("--e2e-units", type=int, default=4_000_000, help="host-buffer batch for the e2e measurement")
    ap.add_argument("--profile", type=int, default=None, help="synthetic profile (default: the workload's): 1 = enriched fragment model, 0 = ref-style, 3 = enriched + planted over-represented sequences")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-workloads", action="store_true", help="skip the other BASELINE configs (the `workloads` object)")
    ap.add_argument("--fastq-units", type=int, default=1_000_000,
                    help="units of the text-in/text-out measurement (device FASTQ decode + chain + encode); 0 = skip")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of --workload as DIR/<name>.npy (counter block, records of a seeded sample of units)")
    args = ap.parse_args()

    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    from fastp_b200 import capi, sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (fastp_b200 has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    comm = None
    if world > 1:
        # NCCL may print a version banner on stdout (NCCL_DEBUG=VERSION in the environment): keep stdout for the one JSON line
        sys.stdout.flush()
        saved_out = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
            comm = sharding.NcclComm(world, rank)   # raw ncclComm_t for the C-ABI collective fp_counters_allreduce
            tt0 = torch.zeros(1, device=f"cuda:{local_rank}")
            dist.all_reduce(tt0)                    # first collective (lazy communicator setup) while stdout is parked
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_out, 1)
            os.close(saved_out)
    dev = f"cuda:{local_rank}"
    lib = capi.load()
    env = dict(torch=torch, dist=dist, capi=capi, lib=lib, world=world, rank=rank, local_rank=local_rank, dev=dev, comm=comm, cpu={})

    names = [args.workload] + ([] if args.no_workloads else [w for w in ("se150_cut_right_polyg", "pe150_full", "pe250_overrep") if w != args.workload])
    # ---- CPU legs first (rank 0): the reference's worker body on a bounded sample of each workload's stream; the same
    #      sample's counter block is the parity target of the GPU pass below ----
    cpu_lines = {}
    if rank == 0 and not args.no_cpu_baseline:
        for nm in names:
            try:
                tsec = 10.0 if nm == args.workload else 5.0
                cpu_lines[nm], ctx = cpu_baseline(nm, args.profile if nm == args.workload else None, target_seconds=tsec,
                                                  max_units=6_000_000 if nm == args.workload else 2_000_000)
                if nm == "pe250_overrep":
                    # over-representation counts depend on the worker-thread split: the parity target is ONE worker over a shorter prefix
                    T = ctx["T"]; m = min(ctx["n"], 60_000)
                    sub = {k: v[:m] for k, v in ctx["arrs"].items()}
                    _, blk = cpu_run(T, ctx["kind"], ctx["params"], ctx["W"], sub, 1)
                    ctx = dict(ctx, n=m, block=blk)
                env["cpu"][nm] = ctx
            except Exception as e:  # the baseline is a reported number, never a reason to lose the GPU line
                cpu_lines[nm] = {"value": None, "cores": os.cpu_count(), "kind": "unavailable", "sample": repr(e)}
    if world > 1:
        # every rank must take the parity pass with the same sample size
        nn = torch.tensor([env["cpu"].get(nm, {}).get("n", 0) for nm in names], device=dev, dtype=torch.int64)
        dist.broadcast(nn, src=0)
        if rank != 0:
            for nm, v in zip(names, nn.tolist()):
                if v:
                    env["cpu"][nm] = {"n": int(v)}

    results = {}
    env["numa"] = bind_to_gpu_numa(torch, local_rank)       # after the CPU legs (they use every CPU the process may use)
    for nm in names:
        main_wl = nm == args.workload
        units = (args.units or WORKLOADS[nm]["units"]) if main_wl else min(args.units or WORKLOADS[nm]["units"], WORKLOADS[nm]["units"])
        try:
            res, parity, _ = gpu_workload(nm, args, env, units, args.steps if main_wl else max(2, min(args.steps, 3)),
                                          args.warmup if main_wl else 3, with_e2e=main_wl and not args.no_e2e,
                                          dump_dir=args.dump_outputs if main_wl else None)
        except Exception as e:
            if main_wl:
                raise
            results[nm] = {"value": None, "error": repr(e)}
            continue
        if rank == 0 and parity is not None and "block" in env["cpu"].get(nm, {}):
            Lc_, want = env["cpu"][nm]["block"]
            m = parity["units"]
            key = f"counters_eq_reference_{m}_units"
            if m == env["cpu"][nm]["n"]:
                res["checks"][key] = bool(np.array_equal(parity["got"], want))
            else:   # the sample did not divide evenly over the ranks: compare against a fresh CPU pass over exactly m units
                ctx = env["cpu"][nm]
                sub = {k: v[:m] for k, v in ctx["arrs"].items()}
                _, blk = cpu_run(ctx["T"], ctx["kind"], ctx["params"], ctx["W"], sub, 1 if nm == "pe250_overrep" else cpu_resources()["usable"])
                res["checks"][key] = bool(np.array_equal(parity["got"], blk[1]))
        if nm in cpu_lines:
            res["cpu_baseline"] = cpu_lines[nm]
        results[nm] = res

    line = dict(results[args.workload])
    line.update({"n_gpus": world, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic"})
    if rank != 0:
        line.pop("clocks", None)
    others = {k: v for k, v in results.items() if k != args.workload}
    if others:
        line["workloads"] = {k: ({kk: vv for kk, vv in v.items() if kk not in ("metric",)} if isinstance(v, dict) else v) for k, v in others.items()}
    if rank == 0 and world == 1 and args.fastq_units > 0:
        try:
            params = workload_params(capi, lib, args.workload) if args.workload != "pe250_overrep" else None
            if params is not None and WORKLOADS[args.workload]["S"] == STRIDE:
                paired = bool(params.paired)
                line["fastq_path"] = fastq_path(args, torch, capi, lib, params, paired, dev, "pairs/s" if paired else "reads/s")
        except Exception as e:   # an extra object: never a reason to lose the main line
            line["fastq_path"] = {"value": None, "error": repr(e)}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        comm.destroy()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
