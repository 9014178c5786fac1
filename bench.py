#!/usr/bin/env python
"""bench.py -- k-mers counted/sec at k=21 on N B200s (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            our engine (CUDA, via the C ABI)
  python bench.py --impl reference --gpus N ...            the reference's own CPU path

A "step" = one pass of the hot path (FASTA text -> canonical 21-mers -> GF(2) hash ->
insert/increment) over the whole synthetic input, into a zeroed table.

  value  device-resident input (HBM), timed with CUDA events            [k-mers/s, whole job]
  e2e    the same through the public host API (jfgpu_feed) from pinned HOST memory:
         host->device copies and the device->host read of the result inside the timed region
  roofline      for the fused count kernel, against MEASURED_PEAKS.json's HBM figure
  cpu_baseline  the reference binary (oracle/_ref/jellyfish, all host threads) on a bounded
                sample of the same workload

--dump-outputs DIR writes what the last timed step computed (see dump_outputs) as DIR/<name>.npy; the
inputs are generated from fixed seeds, so two builds given the same arguments can be compared file by file.

Workload (N=1, default --config k21): BASELINE configs[1], k=21 canonical, 10 Gbp synthetic FASTA.
configs[1] names a "4 G-entry hash", which cannot hold the ~9.98e9 distinct 21-mers of 10 Gbp iid
sequence: the reference doubles it twice to 2^34 slots.  The bench therefore sizes the table at
its final size, -s 16G (2^34 slots), for both arms; set --size 4G to time the doubling too.
Input is larger than L2 (10 GB text, 68 GB table), so no L2 flush is needed between steps.

The other BASELINE configs are bench lines of their own (`--config`, results under profiles/):
  k31   configs[2]  k=31 canonical, 10 Gbp over 8 GPUs = 1.25 Gbp and 2^31 slots (64-bit) per GPU
  k63   configs[4]  k=63 canonical, 2 Gbp, 2^32 slots of 128 bits
  bf    configs[3]  k=21 with the --bf-size 10G Bloom prefilter in front of the table
"""
import argparse
import ctypes as C
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "k-mers counted/sec at k=21"
UNIT = "k-mers/s"

# per-GPU workloads of the BASELINE configs: k, bases, -s (table share of one GPU), Bloom prefilter size
CONFIGS = {
    "k21": {"k": 21, "bases": 10_000_000_000, "size": "16G", "bf": 0},
    "k31": {"k": 31, "bases": 1_250_000_000, "size": "2G", "bf": 0},
    "k63": {"k": 63, "bases": 2_000_000_000, "size": "4G", "bf": 0},
    "bf":  {"k": 21, "bases": 10_000_000_000, "size": "16G", "bf": 10_000_000_000},
}


def workload_config(args, world):
    """The `config` object of the JSON line: identical in both arms (it names the workload, not the engine)."""
    bf = (", --bf-size %d Bloom prefilter" % args.bf_size) if args.bf_size else ""
    return {"workload": "k=%d canonical, %d bp synthetic FASTA per GPU (one record, 70-column lines: the shape generate_sequence writes), "
                        "-s %s per GPU%s" % (args.k, args.bases, args.size, bf),
            "l2": "text and table are far larger than L2 (126 MB): no flush between steps",
            "parallelism": "1 GPU" if world == 1 else "table sharded by the top hash bits over %d GPUs" % world}


def parse_size(s):
    mult = {"k": 10**3, "M": 10**6, "G": 10**9, "T": 10**12}
    return int(s[:-1]) * mult[s[-1]] if s[-1] in mult else int(s)


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        self.index = index
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for line in self.lines:
            p = [x.strip() for x in line.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v == "Active":
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# the reference's own CPU path on a bounded sample
# ------------------------------------------------------------------------------------------------
def write_sample_fasta(path, n_bases, seed=3141592653):
    """The sample input: the reference's own generator (jellyfish/generate_sequence.cc, the seed of its test-suite) when
    oracle/_ref was built; otherwise numpy iid ACGT in the same shape ('>read1', 70 bases per line)."""
    import jfutil
    if os.path.exists(jfutil.REF_GEN):
        prefix = path[:-3] if path.endswith(".fa") else path
        jfutil.run([jfutil.REF_GEN, "-o", prefix, "-s", str(seed), str(n_bases)])
        if prefix + ".fa" != path:
            os.rename(prefix + ".fa", path)
        return "generate_sequence -s %d %d" % (seed, n_bases)
    import numpy as np
    rng = np.random.default_rng(seed)
    with open(path, "wb") as f:
        f.write(b">read1\n")
        left = n_bases
        lut = np.frombuffer(b"ACGT", dtype=np.uint8)
        while left > 0:
            n = min(left, 70 * 400000)
            seq = lut[rng.integers(0, 4, size=n, dtype=np.uint8)]
            full = (n // 70) * 70
            body = np.empty((n // 70, 71), dtype=np.uint8)
            body[:, :70] = seq[:full].reshape(-1, 70)
            body[:, 70] = 10
            f.write(body.tobytes())
            if n > full:
                f.write(seq[full:].tobytes() + b"\n")
            left -= n
    return "numpy iid ACGT, %d bases" % n_bases


def cpu_reference_run(sample_fa, n_bases, k, size, threads, workdir, bf_size=0):
    """One timed run of the reference binary (or the C restatement) -> k-mers/s of its Counting phase."""
    import jfutil
    timing = os.path.join(workdir, "timing.txt")
    out = os.path.join(workdir, "ref.jf")
    bf = ["--bf-size", str(bf_size)] if bf_size else []
    if os.path.exists(jfutil.REF_JF):
        kind = "reference"
        cmd = [jfutil.REF_JF, "count", "-m", str(k), "-s", str(size), "-t", str(threads), "-C", "--no-write",
               "--timing", timing, "-o", out] + bf + [sample_fa]
        t0 = time.perf_counter()
        subprocess.check_call(cmd, env=dict(os.environ, SOURCE_DATE_EPOCH="0"))
        wall = time.perf_counter() - t0
        secs = None
        for line in open(timing):
            if line.startswith("Counting"):
                secs = float(line.split()[1])
        secs = secs or wall
    else:
        kind = "port"
        threads = 1
        cmd = [jfutil.ORACLE_C, "count", "-m", str(k), "-s", str(size), "-C", "-o", out] + bf + [sample_fa]
        t0 = time.perf_counter()
        subprocess.check_call(cmd, stderr=subprocess.DEVNULL)
        secs = time.perf_counter() - t0
    return (n_bases - k + 1) / secs, kind, threads, secs


def cpu_sample_plan(args):
    """Bounded sample of the workload for the CPU arm: bases and table size (final load ~0.37, no doubling)."""
    import jfutil
    sample = min(args.cpu_sample_bases, args.bases)
    if not os.path.exists(jfutil.REF_JF):
        sample = min(sample, 5_000_000)
    size = 1 << max(10, (int(sample / 0.6) - 1).bit_length())
    bf = int(args.bf_size * (sample / float(args.bases))) if args.bf_size else 0
    return sample, size, bf


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    k = args.k
    threads = os.cpu_count() or 1
    sample, size, bf = cpu_sample_plan(args)
    with tempfile.TemporaryDirectory() as d:
        fa = os.path.join(d, "sample.fa")
        how = write_sample_fasta(fa, sample)
        with open(fa, "rb") as f:          # warm the page cache
            while f.read(1 << 24):
                pass
        vals = []
        for i in range(args.warmup + args.steps):
            v, kind, cores, secs = cpu_reference_run(fa, sample, k, size, threads, d, bf)
            if i >= args.warmup:
                vals.append((v, secs))
    rates = sorted(v for v, _ in vals)
    value = sum(rates) / len(rates)
    ms = 1e3 * sum(s for _, s in vals) / len(vals)
    sample_desc = ("each step = %s (%d bp of the %d bp workload), jellyfish count -m %d -s %d%s -t %d -C --no-write, Counting phase of "
                   "--timing; the table is sized for the sample (the workload's -s %s would be %d GB of host memory per step)"
                   % (how, sample, args.bases, k, size, (" --bf-size %d" % bf) if bf else "", cores, args.size,
                      parse_size(args.size) * 26 // 8 // 10**9))
    line = {
        "impl": "reference", "metric": METRIC if k == 21 else "k-mers counted/sec at k=%d" % k, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic", "config": workload_config(args, args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample_desc,
                         "min": rates[0], "median": statistics.median(rates), "max": rates[-1]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="k21", choices=sorted(CONFIGS), help="BASELINE config (see the module docstring)")
    ap.add_argument("--bases", type=int, default=None, help="bases of synthetic sequence per GPU")
    ap.add_argument("--size", default=None, help="-s of the per-GPU table share (global table = N x this)")
    ap.add_argument("--k", type=int, default=None)
    ap.add_argument("--bf-size", type=int, default=None)
    ap.add_argument("--cpu-sample-bases", type=int, default=400_000_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump", action="store_true", help="also time one full sorted dump (Writing phase) to /dev/null-like sink")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    cfg = CONFIGS[args.config]
    args.k = args.k or cfg["k"]
    args.bases = args.bases or cfg["bases"]
    args.size = args.size or cfg["size"]
    args.bf_size = cfg["bf"] if args.bf_size is None else args.bf_size

    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    from jellyfish_b200 import HashCounter, _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_MAX_CTAS", "16")      # K1 leaves 16 SMs to the exchange that runs beside it
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if world != args.gpus:
        if rank == 0:
            sys.stderr.write("bench.py: --gpus %d but WORLD_SIZE=%d; launch with torchrun for N>1\n" % (args.gpus, world))
        args.gpus = world
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    lib = _lib.load()

    k = args.k
    n_bases = args.bases
    nbytes = lib.jfgpu_synth_fasta_bytes(n_bases)
    text = torch.empty(nbytes + 256, dtype=torch.uint8, device=dev)
    got = C.c_uint64(0)
    rc = lib.jfgpu_synth_fasta_device(local_rank, C.c_void_p(text.data_ptr()), nbytes + 256, n_bases, (0x9E3779B97F4A7C15 * (rank + 1)) & ((1 << 64) - 1), C.byref(got), None)      # (the seed is an OFFSET into one stream:
    # ranks far apart, or they would count nearly the same k-mers and halve the load of the shared table)
    assert rc == 0, "synthetic FASTA generation failed"
    torch.cuda.synchronize()
    n_text = got.value
    kmers_per_step = n_bases - k + 1

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    size = parse_size(args.size)
    t_init = time.perf_counter()
    if world > 1:
        from jellyfish_b200.distributed import ShardedCounter
        counter = ShardedCounter(size * world, 7, k=k, canonical=True, rank=rank, world=world, device=local_rank)
        hc = counter.hc
    else:
        counter = None
        hc = HashCounter(size, 7, k=k, canonical=True, device=local_rank, bf_size=args.bf_size)
    torch.cuda.synchronize()
    init_s = time.perf_counter() - t_init
    info = hc.info()

    def one_step_device():
        hc.clear()
        if counter is not None:
            counter.add_device_text(text.data_ptr(), n_text)
        else:
            hc.add_device_text(text.data_ptr(), n_text)
        return hc.done()

    # ---- value: device-resident input; whole steps between synchronised barriers, max over ranks ----
    for _ in range(args.warmup):
        st = one_step_device()
    launches0 = lib.jfgpu_kernel_launches()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    t0 = time.perf_counter()
    acc = {"seconds_count": 0.0, "seconds_count_kernel": 0.0, "count_kernel_launches": 0, "seconds_drain": 0.0,
           "seconds_win_hist": 0.0, "seconds_win_scatter": 0.0, "seconds_win_insert": 0.0}
    step_secs = []
    for _ in range(args.steps):
        ts = time.perf_counter()
        st = one_step_device()
        torch.cuda.synchronize()
        step_secs.append(time.perf_counter() - ts)
        for key in acc:
            acc[key] += st[key]
    barrier()
    wall = time.perf_counter() - t0
    xtrace = counter.records.trace if counter is not None and counter.records is not None else None     # (stages of the last step)
    clocks = sampler.stop()
    launches = lib.jfgpu_kernel_launches() - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, hc, st, text, n_bases, k, rank if world > 1 else None)
    tot = torch.tensor([st["kmers"], st["inserted"], st["distinct"]], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(tot)          # keys are inserted by their owner: only the sums must agree
    assert st["kmers"] == kmers_per_step and tot[0].item() == kmers_per_step * world, (st, tot.tolist())
    if not args.bf_size:
        assert tot[0].item() == tot[1].item(), (st, tot.tolist())
    distinct_total = int(tot[2].item())
    t = torch.tensor([acc["seconds_count"], wall], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_secs, wall = t.tolist()
    ms_per_step = 1e3 * wall / args.steps
    value = kmers_per_step * world * args.steps / wall

    # ---- roofline: every kernel class of a step against the measured HBM peak, the dominant one on top ----
    # algorithmic bytes per k-mer (DESIGN.md section 4):
    #   K1  extract: 71/70 text + rec written
    #   K2  window form: win_hist reads rec; win_scatter reads + writes rec; win_insert reads rec and sweeps the table
    #       once (read + write every slot); L2 form (insert_chunks): rec + table sweep
    #   direct insertion (small tables / Bloom counter): the north star's 71/70 + 32 p + 32
    p_mean = 1.0 + st["reprobes"] / max(1, st["inserted"])
    peak, peak_src = measured_peak()
    tinfo = {}
    tfile = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tfile):
        try:
            tinfo = json.load(open(tfile))
        except Exception:
            tinfo = {}
    nk = float(kmers_per_step * args.steps)
    kernels = []

    def add_kernel(name, secs, bpk, launches_=None, traffic_key=None):
        if secs <= 0:
            return
        ach = nk * bpk / secs / 1e9
        tr = tinfo.get(traffic_key) if traffic_key else None
        kernels.append({"kernel": name, "seconds_per_step": secs / args.steps, "alg_bytes_per_kmer": bpk, "achieved": ach, "frac": ach / peak,
                        "launches_per_step": (launches_ / args.steps) if launches_ else None,
                        "traffic": (tr or {}).get("dram_bytes_per_launch"), "traffic_note": (tr or {}).get("note")})

    sweep = 2.0 * info["table_bytes"] / kmers_per_step
    if info["part_regions"]:
        rec = info["part_rec_bytes"]
        add_kernel("extract_kernel (K1: parse, canonical k-mers, GF(2) hash, region records)", acc["seconds_count_kernel"], 71.0 / 70.0 + rec,
                   acc["count_kernel_launches"], "extract_kernel")
        if acc["seconds_win_insert"] > 0:
            add_kernel("win_hist_kernel (K2a: records per window)", acc["seconds_win_hist"], rec, None, "win_hist_kernel")
            add_kernel("win_scatter_kernel (K2b: records grouped by window)", acc["seconds_win_scatter"], 2.0 * rec, None, "win_scatter_kernel")
            add_kernel("win_insert2_kernel (K2c: shared-memory window insert, table swept once)", acc["seconds_win_insert"], rec + sweep, None, "win_insert2_kernel")
        else:
            add_kernel("insert_chunks_kernel (K2, L2 form: region-by-region insert)", acc["seconds_drain"], rec + sweep, None, "insert_chunks_kernel")
    else:
        add_kernel("extract_kernel (direct insert)", acc["seconds_count_kernel"], 71.0 / 70.0 + 32.0 * p_mean + 32.0, acc["count_kernel_launches"], "extract_kernel_direct")
    dom = max(kernels, key=lambda x: x["seconds_per_step"])
    step_bytes = sum(x["alg_bytes_per_kmer"] for x in kernels)
    roofline = {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved"], "peak": peak, "unit": "GB/s", "frac": dom["frac"],
                "traffic": dom["traffic"], "peak_source": peak_src, "alg_bytes_per_kmer": dom["alg_bytes_per_kmer"], "mean_probes": p_mean,
                "avg_seconds_per_step": dom["seconds_per_step"], "kernels": kernels,
                "whole_step": {"alg_bytes_per_kmer": step_bytes, "achieved": value / world * step_bytes / 1e9,
                               "frac": value / world * step_bytes / 1e9 / peak,
                               "note": "all kernels of the step (table clear excluded from the bytes, included in the time)"}}
    # the north star's own yardstick: k-mers/s x (71/70 + 32 p + 32) bytes against the HBM peak, i.e. what a table filled by
    # random HBM accesses would have to move
    b_rand = 71.0 / 70.0 + 32.0 * p_mean + 32.0
    roofline["random_access_model"] = {"alg_bytes_per_kmer": b_rand, "achieved": value / world * b_rand / 1e9, "unit": "GB/s",
                                       "frac_of_hbm_peak": value / world * b_rand / 1e9 / peak}

    # ---- e2e: the public host API with pinned HOST buffers, copies inside the timed region ----
    e2e = None
    if not args.no_e2e:
        hptr = lib.jfgpu_host_alloc(n_text)
        assert hptr, "pinned host allocation failed"
        torch.cuda.synchronize()
        # fill the host buffer once (untimed set-up): device -> pinned host
        host = torch.frombuffer((C.c_uint8 * n_text).from_address(hptr), dtype=torch.uint8)
        host.copy_(text[:n_text])
        torch.cuda.synchronize()

        def one_step_host():
            hc.clear()
            if counter is not None:
                counter.add_host_text(hptr, n_text)
            else:
                hc.add_text((C.c_void_p(hptr), n_text))
            return hc.done()          # reads the statistics block back to the host

        for _ in range(min(args.warmup, 1)):
            one_step_host()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            st2 = one_step_host()
        barrier()
        wall2 = time.perf_counter() - t0
        assert st2["kmers"] == kmers_per_step and (world > 1 or st2["distinct"] == st["distinct"]), "the host feed counted something else"
        t = torch.tensor([wall2], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        wall2 = t.item()
        e2e = {"value": kmers_per_step * world * args.steps / wall2, "unit": UNIT, "h2d_bytes_per_step": n_text * world,
               "d2h_bytes_per_step": 104 * world, "ms_per_step": 1e3 * wall2 / args.steps}
        lib.jfgpu_host_free(hptr)

    # ---- Writing phase: one full sorted dump of the resident table through the C ABI (bytes discarded by the sink) ----
    writing = None
    if args.dump and world == 1:
        torch.cuda.synchronize()
        tw = time.perf_counter()
        nrec = hc.dump_records(sink="discard")
        writing_s = time.perf_counter() - tw
        out_bytes = nrec * ((2 * k + 7) // 8 + 4)
        writing = {"seconds": writing_s, "records": nrec, "bytes": out_bytes, "GB_per_s": out_bytes / writing_s / 1e9,
                   "note": "jfgpu_dump: records ordered tile by tile on the device, device->pinned host copies overlapped with the next "
                           "segment; the sink discards the bytes (no file system in the timed region)"}

    # ---- multi-GPU parity inside the bench: a committed golden case through the sharded path ----
    parity_n = None
    if world > 1:
        parity_n = sharded_parity_check(world, rank, local_rank)

    # ---- CPU baseline (rank 0, N=1 only): bounded sample of the same workload ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sample, csize, cbf = cpu_sample_plan(args)
        with tempfile.TemporaryDirectory() as d:
            fa = os.path.join(d, "sample.fa")
            how = write_sample_fasta(fa, sample)
            v, kind, cores, secs = cpu_reference_run(fa, sample, k, csize, os.cpu_count() or 1, d, cbf)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
               "sample": "%s; jellyfish count -m %d -s %d -t %d -C (Counting phase, %.1f s); table sized for the sample" % (how, k, csize, cores, secs)}

    if rank == 0:
        line = {
            "metric": METRIC if k == 21 else "k-mers counted/sec at k=%d" % k, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic", "config": workload_config(args, world),
            "engine": {"global_lsize": info["lsize"], "slot_bits": info["slot_bits"], "table_bytes_per_gpu": info["table_bytes"],
                       "regions": info["part_regions"], "record_bytes": info["part_rec_bytes"], "text_bytes_per_gpu": n_text,
                       "timed_region": "table clear + all kernels of a step; inputs resident in HBM; wall clock between synchronised barriers",
                       "input": "device-generated iid ACGT (counter-based RNG), one '>read1' record, 70-column lines"},
            "device_seconds_per_step": dev_secs / args.steps, "step_ms": {"min": 1e3 * min(step_secs), "median": 1e3 * statistics.median(step_secs), "max": 1e3 * max(step_secs)},
            "init_s": init_s, "writing": writing,
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "distinct": distinct_total, "load_factor": distinct_total / float(info["size"]), "parity_n": parity_n,
            "exchange": dict(xtrace, form="records") if xtrace else ({"form": "keys"} if counter is not None else None),
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


OUTPUT_SAMPLE = 1 << 16          # k-mers of the input whose counts --dump-outputs writes
OUTPUT_SEED = 0x5EED0F0B


def dump_outputs(out_dir, hc, st, text, n_bases, k, rank):
    """What a caller of the timed path receives from its last step, as float64 arrays (every value is an integer below 2^53):
      stats             kmers, inserted, distinct of the statistics done() returns
      histogram         distinct k-mers by count, counts of 1023 and more in the last bin (`jellyfish histo`)
      sample_positions  OUTPUT_SAMPLE positions in the sequence, drawn with OUTPUT_SEED
      sample_counts     the table's count of the k-mer starting at each of them
    Written as DIR/<name>.npy, DIR/<name>_rank<r>.npy for the shard of rank r of a sharded run (keys of other shards count 0)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    # the text is one record, 70-column lines: base q sits at offset (header line) + q + q // 70
    head = text[:4096].cpu().numpy().tobytes()
    first = head.index(b"\n") + 1
    pos = np.sort(np.random.default_rng(OUTPUT_SEED).integers(0, n_bases - k + 1, size=OUTPUT_SAMPLE))
    q = pos[:, None] + np.arange(k)
    idx = torch.from_numpy((first + q + q // 70).reshape(-1)).to(text.device)
    bases = text[idx].cpu().numpy().reshape(OUTPUT_SAMPLE, k)
    assert np.isin(bases, np.frombuffer(b"ACGT", dtype=np.uint8)).all(), "sampled k-mers are not all ACGT: text layout changed"
    counts = hc.get_many([row.tobytes().decode() for row in bases])
    suffix = "" if rank is None else "_rank%d" % rank
    arrays = {"stats": [st["kmers"], st["inserted"], st["distinct"]], "histogram": hc.histogram(1024),
              "sample_positions": pos, "sample_counts": counts}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), np.asarray(a, dtype=np.float64))


def sharded_parity_check(world, rank, local_rank):
    """After the timed steps: the golden case `multi_files` counted through the sharded (NCCL) path, the rank-ordered
    concatenation of the shard dumps compared with the reference's golden md5.  Returns the parity_n object (rank 0)."""
    import torch
    import torch.distributed as dist
    import gen
    import jfutil
    from cases import CASES
    from jellyfish_b200.distributed import ShardedCounter, concat_shards
    name = "multi_files"
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "golden.json")))[name]
    args, ins = CASES[name]
    k = int(args[args.index("-m") + 1])
    v = args[args.index("-s") + 1]
    size = int(v[:-1]) * {"k": 10**3, "M": 10**6, "G": 10**9}[v[-1]] if v[-1] in "kMG" else int(v)
    tmp = os.path.join(tempfile.gettempdir(), "jf_parity_n")
    if rank == 0:
        os.makedirs(tmp, exist_ok=True)
        gen.make_all(tmp)
    dist.barrier()
    inputs = {n: os.path.join(tmp, n) for n in os.listdir(tmp)}
    os.environ["SOURCE_DATE_EPOCH"] = "0"
    sc = ShardedCounter(size, 7, k=k, canonical="-C" in args, rank=rank, world=world, device=local_rank, batch_bytes=300000)
    for j, nm in enumerate(ins):
        data = open(inputs[nm], "rb").read() if (j % world) == rank else b""
        buf = torch.frombuffer(bytearray(data + b"\0" * 16), dtype=torch.uint8).to(torch.device("cuda", local_rank))
        sc.add_device_text(buf.data_ptr(), len(data))
    sc.done()
    out = os.path.join(tmp, "parity")
    sc.dump_shard(out)
    dist.barrier()
    res = None
    if rank == 0:
        db = concat_shards(out, world, out + ".jf")
        h, b = jfutil.split_db(db)
        res = {"case": name, "world": world, "md5_ok": jfutil.md5(b) == golden["body_md5"], "header_ok": jfutil.semantic(h) == golden["header"]}
    sc.hc.close()
    return res


if __name__ == "__main__":
    main()
