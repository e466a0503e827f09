#!/usr/bin/env python
"""bench.py — headline benchmark of the sylph_b200 hot paths (contract: see DESIGN.md §Measurement).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload sketch|profile]
                  [--dump-outputs DIR]

Primary line (default --workload sketch) = BASELINE.json configs[1]:
  sketch 1 Gbp of synthetic 150 bp single-end reads, k=31 c=200, per GPU (weak scaling: every
  rank sketches its own 1 Gbp sample; no data-path collective).
  step   = bases resident in HBM -> sample sketch (sorted hash/count table) resident in HBM
  value  = whole-job bases/s, CUDA events, max over ranks
  e2e    = same through the C ABI with PINNED HOST buffers: H2D of bases+offsets and D2H of the
           sketch inside the timed region
  roofline = the seeding kernel (dominant), algorithmic bytes (1 B/base + 16 B/survivor) over its
           CUDA-event time measured inside the library on the launching stream
The same JSON line carries "pairs": the containment metric (BASELINE.json configs[2]:
1 sample vs 10k synthetic 4 Mbp genome sketches) measured the same way.
--impl reference times the CPU restatement of the reference (oracle/, AVX2 intrinsics + OpenMP)
on a bounded sample of the same workload on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

READ_LEN = 150
K, C = 31, 200
GENOME_LEN = 4_000_000


def usable_cores():
    """Host cores this process may really use: the container's CPU quota (cgroup cpu.max) caps os.cpu_count();
    running the CPU arm with more threads than the quota only gets it throttled."""
    n = os.cpu_count() or 1
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = max(1, min(n, int(int(q) / int(per))))
    except Exception:
        pass
    return n


def sketch_config(args):
    """The `config` object of the sketch workload: identical in our arm and in the reference arm."""
    n_bases = args.reads * READ_LEN
    return {"workload": "sketch 1 Gbp synthetic 150 bp SE reads k=31 c=200 (BASELINE.json configs[1])",
            "reads_per_gpu": args.reads, "read_len": READ_LEN, "k": K, "c": C, "sem": "avx2-lane",
            "l2": "inputs (%.2f GB per step) are larger than L2; no flush needed" % (n_bases / 1e9)}


def profile_config(args, world):
    n_samples = args.samples or (1 if world == 1 else 16)
    return {"workload": "profile %d sample sketch(es) vs %d synthetic 4 Mbp genome sketches per GPU (BASELINE.json configs[%d])"
                        % (n_samples, args.genomes, 2 if n_samples == 1 else 3),
            "genomes_per_gpu": args.genomes, "samples": n_samples, "reads_per_sample": args.reads, "k": K, "c": C}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="sketch", choices=["sketch", "profile", "genomes"])
    ap.add_argument("--batch-genomes", type=int, default=250, help="genomes (4 Mbp each) per syl_sketch_genomes call of --workload genomes")
    ap.add_argument("--reads", type=int, default=6_666_667, help="reads per GPU (150 bp each)")
    ap.add_argument("--genomes", type=int, default=None,
                    help="genomes per GPU for the containment metric (default 10000; 12500 for the 16-sample config-4 shape)")
    ap.add_argument("--samples", type=int, default=None, help="samples for the containment metric (1; 16 when N>1)")
    ap.add_argument("--no-pairs", action="store_true", help="skip the secondary containment measurement")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--fixed-warmup", action="store_true",
                    help="exactly --warmup untimed steps (no settle loop): for runs under ncu, whose numbers are never bench values")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what each timed path returned in its last step as DIR/<name>.npy "
                         "(float64, at most 64 MiB in all), to compare two builds output for output")
    return ap.parse_args()


# --dump-outputs: rows kept per table (a longer table is cut to a fixed, seeded sample of its rows).  In float64
# columns that is at most 3 x 8 B x 2^20 (sketch) + 2 x 8 B x 2^20 (genome k-mers) + 2 x 8 B x 2^19 (tracked)
# + 6 x 8 B x 2^16 (per genome) + 21 x 8 B x 2^14 (profile rows) = 53.6 MiB
DUMP_ROWS = {"sketch": 1 << 20, "sketch_stats": 1, "genome_kmers": 1 << 20, "genome_tracked": 1 << 19, "genomes": 1 << 16,
             "profile": 1 << 14}
DUMP_MAX_BYTES = 64 << 20
_dumped = [0]


def dump_table(out_dir, name, cols):
    """Write the equal-length columns `cols` (field -> array) of one output table as DIR/<name>_<field>.npy in float64,
    and its row count as DIR/<name>_rows.npy.  uint64 fields are split into exact 32-bit halves <field>_hi / <field>_lo
    (float64 holds 53 bits).  A table longer than DUMP_ROWS[name] keeps a seeded sample of rows: the same rows in
    every run that produced as many."""
    import numpy as np
    n = len(next(iter(cols.values())))
    idx = np.arange(n)
    if n > DUMP_ROWS[name]:
        idx = np.sort(np.random.default_rng(0x5EED).choice(n, DUMP_ROWS[name], replace=False))
    out = {"rows": np.array([n], dtype=np.float64)}
    for field, a in cols.items():
        a = np.asarray(a)[idx]
        if a.dtype == np.uint64:
            out[field + "_hi"], out[field + "_lo"] = a >> np.uint64(32), a & np.uint64(0xFFFFFFFF)
        else:
            out[field] = a
    os.makedirs(out_dir, exist_ok=True)
    for field, a in out.items():
        a = a.astype(np.float64)
        _dumped[0] += a.nbytes
        assert _dumped[0] <= DUMP_MAX_BYTES, "--dump-outputs exceeds 64 MiB"
        np.save(os.path.join(out_dir, "%s_%s.npy" % (name, field)), a)


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons of THIS rank's GPU during the timed region (B200_PROFILING.md's clocks line).
    In-process NVML from a background thread (20 samples/s: two driver calls of a few microseconds each) — a polling
    `nvidia-smi -lms` process that watches all N GPUs takes driver locks on every one of them per sample, and a
    sample that lands inside a 40 ms timed region costs the slowest rank milliseconds (seen as 1.9 vs 2.4 ms per
    step at N = 8).  Falls back to nvidia-smi when NVML cannot be loaded."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index):
        """index: the GPU index of this process (None = no sampling)."""
        self.index, self.rows, self.proc, self.nvml, self.stop_flag, self.how = index, [], None, None, False, None

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:  # CUDA_VISIBLE_DEVICES may renumber: resolve through the PCI bus id torch reports
            import torch
            bus = torch.cuda.get_device_properties(self.index).pci_bus_id
            dom = getattr(torch.cuda.get_device_properties(self.index), "pci_domain_id", 0)
            dev = torch.cuda.get_device_properties(self.index).pci_device_id
            h = pynvml.nvmlDeviceGetHandleByPciBusId(("%08x:%02x:%02x.0" % (dom, bus, dev)).encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(int(self.index))
        return pynvml, h

    def start(self):
        if self.index is None:
            return
        try:
            self.nvml, self.h = self._nvml_handle()
            self.mx = float(self.nvml.nvmlDeviceGetMaxClockInfo(self.h, self.nvml.NVML_CLOCK_SM))
            self.how = "nvml"
            self.t = threading.Thread(target=self._poll_nvml, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.how = "nvidia-smi -lms 100"
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        n = self.nvml
        reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag:
            try:
                self.rows.append((float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)), int(reasons(self.h))))
            except Exception:
                pass
            time.sleep(0.05)

    def _read(self):
        for line in self.proc.stdout:
            r = [x.strip() for x in line.split(",")]
            try:
                mask = sum(bit for (name, bit), v in zip(self.BITS, r[2:6]) if v.lower().startswith("active"))
                self.rows.append((float(r[0]), mask))
                self.mx = float(r[1])
            except Exception:
                pass

    def stop(self):
        if self.index is None:
            return {}
        if self.nvml is not None:
            self.stop_flag = True
            self.t.join(timeout=1)
        elif self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML and nvidia-smi unavailable"]}
        sm = sorted(r[0] for r in self.rows)
        mask = 0
        for r in self.rows:
            mask |= r[1]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": getattr(self, "mx", None),
                "reasons": sorted(name for name, bit in self.BITS if mask & bit), "samples": len(sm), "sampler": self.how}


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def dist_setup(n):
    import torch
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
    return rank, world, local


def max_over_ranks(x, world):
    if world == 1:
        return x
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(x, world):
    if world == 1:
        return x
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


def barrier(world):
    import torch
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def timed(fn, steps, world):
    """barrier+sync, K steps between CUDA events on the current stream, sync+barrier; -> ms (max over ranks)"""
    import torch
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3
    barrier(world)
    return max_over_ranks(e0.elapsed_time(e1), world), max_over_ranks(wall_ms, world)


# ------------------------------------------------------------------------------------------------
def cpu_sketch_baseline(host_bases, host_off, n_reads_sample, repeats=1):
    """Oracle (AVX2-intrinsic seeding + OpenMP, dedup sequential like the reference) on a bounded sample."""
    import numpy as np
    from oracle import oracle as O
    cores = usable_cores()
    nb = int(host_off[n_reads_sample])
    b = host_bases[:nb]
    o = host_off[:n_reads_sample + 1].astype(np.uint64)
    O.sketch_reads(b[: nb // 50], o[: n_reads_sample // 50 + 1], k=K, c=C, sem=O.SEM_AVX2_INTRIN, nthreads=cores)
    best = None
    for _ in range(repeats):
        t = time.perf_counter()
        O.sketch_reads(b, o, k=K, c=C, sem=O.SEM_AVX2_INTRIN, nthreads=cores)
        dt = time.perf_counter() - t
        best = dt if best is None else min(best, dt)
    t = time.perf_counter()
    O.sketch_reads(b[: nb // 4], o[: n_reads_sample // 4 + 1], k=K, c=C, sem=O.SEM_AVX2_INTRIN, nthreads=1)
    dt1 = time.perf_counter() - t
    return {"value": nb / best, "unit": "bases/s", "cores": cores, "kind": "port",
            "sample": "%d reads (%d bases) of the same synthetic sample; AVX2-intrinsic seeding over %d OpenMP "
                      "threads + sequential dedup (reference decomposition: 1 thread per file)" % (n_reads_sample, nb, cores),
            "single_thread_value": (nb // 4) / dt1}


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port: no Rust toolchain in the image) on the host
    cores, same config / metric / unit as our arm.  sketch: every step sketches ALL reads of the workload
    (AVX2-intrinsic seeding over all cores + the sequential dedup).  profile: every step is the oracle's
    `profile` of the sample against all genomes over all cores (the db is sketched on the GPU when there
    is one — database construction is not part of the timed path in either arm)."""
    import numpy as np
    import torch
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    from sylph_b200 import synth
    from oracle import oracle as O
    cores = usable_cores()
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    b, o = synth.reads(args.reads, READ_LEN, device=dev)
    b, o = b.cpu().numpy(), o.cpu().numpy().astype(np.uint64)
    if args.workload == "sketch":
        fn = lambda: O.sketch_reads(b, o, k=K, c=C, sem=O.SEM_AVX2_INTRIN, nthreads=cores)
        units, unit, metric = len(b), "bases/s", "bases/s sketched"
        sample = "all %d reads per step (%d bases), %d OpenMP threads" % (args.reads, len(b), cores)
        cfg = sketch_config(args)
    else:
        cfg = profile_config(args, 1)
        G = args.genomes
        h, c, _, _ = O.sketch_reads(b, o, k=K, c=C, sem=O.SEM_AVX2_INTRIN, nthreads=cores)
        if dev == "cuda":
            import sylph_b200
            ctx = sylph_b200.Context(0)
            g = synth.sketch_db_range(ctx, 0, G)
            d = g.download()
            g.free()
            ctx.close()
        else:  # no GPU (CPU test of this arm): the oracle sketches the genomes itself
            km, tr, gs, ko, to = [], [], [], [0], [0]
            for i in range(G):
                gb, _ = synth.db_chunk(i, i + 1, GENOME_LEN)
                a, t, n = O.sketch_genome(gb.numpy(), np.array([0, GENOME_LEN], np.uint64), k=K, c=C)
                km.append(a); tr.append(t); gs.append(n); ko.append(ko[-1] + len(a)); to.append(to[-1] + len(t))
            d = dict(kmers=np.concatenate(km), kmer_off=np.array(ko, np.uint64), tracked=np.concatenate(tr),
                     tracked_off=np.array(to, np.uint64), gn_size=np.array(gs, np.uint64))
        smp = O.Sample(h, c)
        p = O.default_params(pseudotax=True)
        fn = lambda: O.contain_sample(p, d["kmers"], d["kmer_off"], d["tracked"], d["tracked_off"], d["gn_size"], smp, nthreads=cores)
        units, unit, metric = float(G), "pairs/s", "(sample x genome) containment pairs/s"
        sample = "all %d pairs per step: oracle profile (2 x get_stats + winner table), %d OpenMP threads" % (G, cores)
    for _ in range(args.warmup):
        fn()
    t = time.perf_counter()
    for _ in range(args.steps):
        fn()
    dt = time.perf_counter() - t
    v = units * args.steps / dt
    line = {"impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": v, "unit": unit, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
def bench_sketch(args, ctx, rank, world, local):
    import numpy as np
    import torch
    from sylph_b200 import synth
    n_reads = args.reads
    bases, off = synth.reads(n_reads, READ_LEN, seed=synth.SEED_READS + 0x10 * rank, device="cuda")
    n_bases = bases.numel()
    torch.cuda.synchronize()
    state = {}

    def step_resident():
        # frees the previous step's sketch: every step frees one and makes one, and the last timed one stays readable
        if "s" in state:
            state["s"].free()
        s = ctx.sketch_sequences(bases, off, k=K, c=C)
        state["n"] = len(s)
        state["s"] = s

    # clocks are sampled from before the warm-up to the end of the timed region: nvidia-smi needs ~100 ms to
    # start and its first query can stall the GPU, so neither may fall inside the (tens of ms) timed region;
    # the warm-up keeps the same load running for >= 0.5 s so that the samples are taken under load
    # every rank samples its own GPU (in-process NVML); rank 0 reports the slowest GPU and the union of the reasons
    clocks = ClockSampler(local)
    clocks.start()
    # ... and until the device has settled: a freshly started process on an idle GPU shows sporadic
    # 30-500 ms stalls in its first seconds (clock ramp / driver housekeeping, also seen with no sampler);
    # the untimed warm-up therefore runs until 40 consecutive steps stay within 1.5x of the fastest step
    # (bounded by 8 s), always at least W steps and 0.5 s
    t_w = time.perf_counter()
    n_w, calm, best = 0, 0, float("inf")
    while True:
        a = time.perf_counter()
        step_resident()
        torch.cuda.synchronize()
        dt = time.perf_counter() - a
        n_w += 1
        best = min(best, dt)
        calm = calm + 1 if dt < 1.5 * best else 0
        el = time.perf_counter() - t_w
        if n_w >= args.warmup and (args.fixed_warmup or (el >= 0.5 and (calm >= 40 or el > 8.0))):
            break
    ctx.enable_timing(True)
    ctx.seed_kernel_time(reset=True)
    l0 = ctx.launches
    ms, _ = timed(step_resident, args.steps, world)
    clk = clocks.stop()
    if world > 1:
        import torch.distributed as dist
        allc = [None] * world
        dist.all_gather_object(allc, clk)
        ok = [c for c in allc if c and c.get("sm_mhz") is not None]
        if ok:
            clk = {"sm_mhz": min(c["sm_mhz"] for c in ok), "sm_max_mhz": max(c["sm_max_mhz"] or 0 for c in ok),
                   "reasons": sorted(set(sum((c["reasons"] for c in ok), []))), "samples": sum(c["samples"] for c in ok),
                   "sampler": ok[0].get("sampler"), "gpus_sampled": len(ok)}
    clk["warmup_steps_run"] = n_w
    launches = ctx.launches - l0
    kms, klaunch, kbases = ctx.seed_kernel_time(reset=True)
    ctx.enable_timing(False)
    total_bases = sum_over_ranks(float(n_bases), world)
    value = total_bases * args.steps / (ms * 1e-3)
    s = state.pop("s")
    if args.dump_outputs and rank == 0:
        h, c = s.download()
        dump_table(args.dump_outputs, "sketch", {"hash": h, "count": c})
        dump_table(args.dump_outputs, "sketch_stats", {"num_dup_removed": [s.num_dup_removed],
                                                       "mean_read_length": [s.mean_read_length]})
    s.free()

    # one extra call for the survivor count (algorithmic output bytes of the seeding kernel)
    surv_buf = torch.empty(int(n_bases / C * 1.3 + 65536) * 2, dtype=torch.int64, device="cuda")
    n_surv = ctx.extract_markers_batch(bases, off, k=K, c=C, out=surv_buf)
    del surv_buf
    alg_bytes = n_bases + 8 * n_surv   # SURVEY §8(d): 1 B per base read + 8 B per survivor written
    model_bytes = n_bases + 32 * n_surv  # what this kernel really writes: one 32-byte event (hash, read, pair keys) per survivor
    peak, peak_src = measured_peak_hbm()
    k_ms = kms / max(klaunch, 1)
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r01_k_seed_traffic.json")
    if os.path.exists(tpath):  # dram__bytes_read+write of one ncu --set full capture, scaled by bases per launch
        traffic = json.load(open(tpath))["dram_bytes_per_base"] * n_bases
    roofline = {"kernel": "k_seed<31, events, W=30>", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "kernel_ms": k_ms, "kernel_share_of_step": kms / ms if ms else None,
                "algorithmic_bytes_per_launch": alg_bytes, "traffic_model_bytes_per_launch": model_bytes,
                "note": "integer-issue bound: ~33 SASS instructions per window, 18.4 of them on the ALU pipe (1 warp "
                        "instruction / 2 cycles) and 12.4 IMADs on the FMA pipe; ncu: ALU pipe 75 % active, fmaheavy 59 %, "
                        "DRAM 9 %; see DESIGN.md 4.1 and profiles/"}

    # ---- e2e: pinned host buffers through the C ABI, H2D + D2H inside the timed region
    hb = torch.empty(n_bases, dtype=torch.uint8, pin_memory=True)
    ho = torch.empty(n_reads + 1, dtype=torch.int64, pin_memory=True)
    hb.copy_(bases)
    ho.copy_(off)
    torch.cuda.synchronize()
    hb_np, ho_np = hb.numpy(), ho.numpy().view(np.uint64)
    # result buffers: pinned and reused across steps, as a caller that sketches file after file would
    out_cap = int(n_bases // C * 2 + 65536)
    oh = torch.empty(out_cap, dtype=torch.int64, pin_memory=True).numpy().view(np.uint64)
    oc = torch.empty(out_cap, dtype=torch.int32, pin_memory=True).numpy().view(np.uint32)
    e2e_state = {}

    e2e_state["t"] = []

    def step_e2e():
        t_s = time.perf_counter()
        s = ctx.sketch_sequences(hb_np, ho_np, k=K, c=C)
        h, c = s.download(oh, oc)
        e2e_state["n"] = len(h)
        s.free()
        e2e_state["t"].append(round((time.perf_counter() - t_s) * 1e3, 3))

    for _ in range(max(1, args.warmup // 2)):
        step_e2e()
    e2e_steps = args.steps
    e2e_state["t"] = []
    ctx.enable_timing(True)
    ctx.seed_kernel_time(reset=True)
    _, wall_ms = timed(step_e2e, e2e_steps, world)
    e2e_seed_ms = ctx.seed_kernel_time(reset=True)[0] / e2e_steps
    ctx.enable_timing(False)
    e2e_value = total_bases * e2e_steps / (wall_ms * 1e-3)
    from sylph_b200 import _lib
    # bytes as the library copied them in the last timed step (rank 0), and how the chunks crossed the link
    h2d, ch_packed, ch_ascii = ctx.ingest_stats()
    if ch_packed == 0:
        what = "ASCII bases + u64 record offsets copied as they are (%d chunks)" % ch_ascii
        if int(os.environ.get("LOCAL_WORLD_SIZE", "1")) > 4 and "SYL_HOST_INGEST" not in os.environ:
            what += "; the library does not pack when more than 4 ranks share a host (its memory system, not PCIe, is then the narrow resource)"
    else:
        what = ("host ASCII -> 2-bit words by %d packer threads into pinned staging (inside the timed region), u32 chunk-relative "
                "record offsets: %d chunks packed; %d chunks shipped as ASCII because the link was idle while the packers lagged"
                % (_lib.lib().syl_pack_threads(), ch_packed, ch_ascii))
    e2e = {"value": e2e_value, "unit": "bases/s", "h2d_bytes_per_step": int(h2d),
           "d2h_bytes_per_step": int(12 * e2e_state["n"]), "steps": e2e_steps, "ms_per_step": wall_ms / e2e_steps,
           "timing": "wall clock bracketed by device syncs, max over ranks", "per_step_ms": e2e_state["t"],
           "seed_kernel_ms_per_step": e2e_seed_ms, "ingest": what,
           "call": "syl_sketch_reads(SYL_MEM_HOST, ASCII bases, u64 offsets) + syl_sample_download into pinned result buffers"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_sketch_baseline(hb_np, ho_np, min(n_reads, 2_000_000))
    line = {"metric": "bases/s sketched", "value": value, "unit": "bases/s", "n_gpus": world, "steps": args.steps,
            "warmup": n_w, "warmup_requested": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": sketch_config(args), "workload_stats": {"sketch_entries": state["n"], "survivors": int(n_surv)},
            "clocks": clk, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline}
    if cpu:
        line["cpu_baseline"] = cpu
    return line, (bases, off)


def genomes_config(args):
    return {"workload": "sketch %d synthetic 4 Mbp genomes per step (one syl_sketch_genomes call; the unit of BASELINE.json "
                        "configs[4]: 113k x 4 Mbp, GTDB-R220-scale db build)" % args.batch_genomes,
            "genomes_per_step": args.batch_genomes, "genome_len": GENOME_LEN, "k": K, "c": C, "min_spacing": 30,
            "l2": "inputs (%.2f GB per step) are larger than L2; no flush needed" % (args.batch_genomes * GENOME_LEN / 1e9)}


def bench_genomes(args, ctx, rank, world, local):
    """Genome (database) sketching, device-resident synthetic genomes generated on the device (config 5: 452 GB of bases
    cannot cross PCIe in useful time).  step = one batch of genomes -> CSR genome_kmers + tracked, resident."""
    import numpy as np
    import torch
    from sylph_b200 import synth
    nG = args.batch_genomes
    bases, off = synth.db_chunk(rank * nG, (rank + 1) * nG, GENOME_LEN, device="cuda")
    goff = torch.arange(nG + 1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    st = {}

    def step():
        # frees the previous step's sketches: every step frees one batch and makes one, and the last timed one stays
        if "g" in st:
            st["g"].free()
        st["g"] = ctx.sketch_genomes(bases, off, goff, k=K, c=C)

    for _ in range(max(args.warmup, 3)):
        step()
    ctx.enable_timing(True)
    ctx.seed_kernel_time(reset=True)
    ctx.kernel_time("genome_post", reset=True)
    l0 = ctx.launches
    ms, _ = timed(step, args.steps, world)
    launches = ctx.launches - l0
    kms = ctx.seed_kernel_time(reset=True)[0] / args.steps
    pms = ctx.kernel_time("genome_post", reset=True)[0] / args.steps
    ctx.enable_timing(False)
    n_bases = float(bases.numel())
    value = sum_over_ranks(n_bases, world) * args.steps / (ms * 1e-3)
    g = st["g"]
    d = g.download()
    if args.dump_outputs and rank == 0:
        dump_table(args.dump_outputs, "genome_kmers", {"hash": d["kmers"]})
        dump_table(args.dump_outputs, "genome_tracked", {"hash": d["tracked"]})
        dump_table(args.dump_outputs, "genomes", {"kmer_end": d["kmer_off"][1:], "tracked_end": d["tracked_off"][1:],
                                                  "gn_size": d["gn_size"]})
    peak, peak_src = measured_peak_hbm()
    n_surv_est = int(d["kmer_off"][-1] + d["tracked_off"][-1])
    alg = n_bases + 16.0 * n_surv_est   # SURVEY §8(d), positions variant: 1 B/base + 16 B per survivor
    out = {"metric": "bases/s sketched (genomes)", "value": value, "unit": "bases/s", "n_gpus": world, "steps": args.steps,
           "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": genomes_config(args), "gpu_launches": int(launches),
           "workload_stats": {"genome_kmers": int(d["kmer_off"][-1]), "tracked": int(d["tracked_off"][-1])},
           "kernels_ms_per_step": {"k_seed": kms, "post_pass": pms},
           "roofline": {"kernel": "k_seed<31, survivors, W=32>", "bound": "hbm", "achieved": alg / (kms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": alg / (kms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src, "kernel_ms": kms,
                        "kernel_share_of_step": kms / (ms / args.steps), "algorithmic_bytes_per_launch": alg,
                        "note": "integer-issue bound like the read-sketch kernel (same hot loop)"}}
    if rank == 0 and not args.no_cpu:   # parity + CPU arm on a few genomes of the batch
        from oracle import oracle as O
        from concurrent.futures import ThreadPoolExecutor
        cores = usable_cores()
        hb = bases.cpu().numpy()
        idx = list(range(0, nG, max(1, nG // 16)))

        def one(i):
            return O.sketch_genome(hb[i * GENOME_LEN:(i + 1) * GENOME_LEN], np.array([0, GENOME_LEN], np.uint64), k=K, c=C)

        t = time.perf_counter()
        with ThreadPoolExecutor(max_workers=min(len(idx), cores)) as ex:
            exp = list(ex.map(one, idx))
        dt = time.perf_counter() - t
        ok = all(np.array_equal(km, d["kmers"][int(d["kmer_off"][i]):int(d["kmer_off"][i + 1])]) and
                 np.array_equal(tr, d["tracked"][int(d["tracked_off"][i]):int(d["tracked_off"][i + 1])]) for i, (km, tr, _) in zip(idx, exp))
        out["parity_checked"] = bool(ok)
        out["cpu_baseline"] = {"value": len(idx) * GENOME_LEN / dt, "unit": "bases/s", "cores": min(len(idx), cores), "kind": "port",
                               "sample": "%d of the batch's genomes, one oracle thread per genome (reference decomposition: 1 thread per file)" % len(idx)}
        if not ok:
            raise SystemExit("bench: genome sketches differ from the oracle")
    g.free()
    return out


def rows_equal_oracle(rows, exp, tol=1e-6):
    """Field-by-field comparison of syl_profile rows with the oracle's rows (same order): integers exact,
    floats within `tol` relative — the same bar as tests/test_contain_gpu.py::compare. -> (ok, first difference)"""
    if len(rows) != len(exp):
        return False, "row count %d != %d" % (len(rows), len(exp))
    for i, (r, e) in enumerate(zip(rows, exp)):
        for f in ("genome", "contain", "glen", "lambda_status", "kmers_lost", "ci_valid"):
            if int(r[f]) != int(getattr(e, f)):
                return False, "row %d %s: %s != %s" % (i, f, r[f], getattr(e, f))
        for f in ("naive_ani", "final_est_ani", "final_est_cov", "mean_cov", "median_cov", "rel_abund", "seq_abund"):
            x, y = float(r[f]), float(getattr(e, f))
            if abs(x - y) > tol * max(1.0, abs(y)):
                return False, "row %d %s: %r != %r" % (i, f, x, y)
        if e.ci_valid:
            for j in range(4):
                if abs(float(r["ci"][j]) - e.ci[j]) > tol * max(1.0, abs(e.ci[j])):
                    return False, "row %d ci[%d]" % (i, j)
    return True, None


PAIR_KERNELS = {"join": "k_join_hist<pass 1> (+ k_range_bounds)", "join2": "k_join2_order (+ k_local_best)", "stats": "k_stats_hist", "boot": "k_boot_iter_p"}
PAIR_LIMITER = {"join": "DRAM: random sectors of the db index (ncu: 0.32 GB per sample at 4.9 TB/s)",
                "join2": "DRAM / latency: genome ids of the recorded equal ranges",
                "stats": "latency (one warp per touched pair)",
                "boot": "integer issue: 39 instructions per 32 bootstrap draws on the main path (11 of them the 128-bit multiply), ~50 all-in; issue slots ~70 % busy, no DRAM traffic"}


def bench_pairs(args, ctx, rank, world, local, reads):
    """BASELINE.json configs[2] (1 sample x G genomes, 1 GPU) and configs[3] (16 samples x G genomes PER GPU, db sharded
    by genome, weak scaling: --samples 16 runs the same 16-sample workload on 1 GPU).  Multi-sample runs draw a
    different community for every sample (seeds 0x5EED0010 + s) from the WHOLE genome range, so pass-1 survivors,
    winners and lost k-mers come from every shard."""
    import numpy as np
    import torch
    from sylph_b200 import _lib, synth
    from sylph_b200 import dist as D
    from sylph_b200.api import contain_params
    n_samples = args.samples or (1 if world == 1 else 16)
    G = args.genomes
    G_total = G * world
    t0 = time.perf_counter()
    genomes = synth.sketch_db_range(ctx, rank * G, (rank + 1) * G, GENOME_LEN, k=K, c=C)
    db = ctx.build_db(genomes, genome_base=rank * G)
    torch.cuda.synchronize()
    t_db = time.perf_counter() - t0
    db_keys = int(_lib.lib().syl_genomes_total_kmers(genomes._h))
    samples = []
    bases, off = reads
    t0 = time.perf_counter()
    for si in range(n_samples):
        if n_samples == 1:
            samples.append(ctx.sketch_sequences(bases, off, k=K, c=C))     # the config-2 sample (community = genomes 0..63)
        else:  # replicated on every rank: full-depth samples, community of 64 genomes spread over all shards
            seed = synth.SEED_READS + 0x10 + si
            comm = synth.community_ids(64, G_total, seed=seed)
            b, o = synth.reads(args.reads, READ_LEN, seed=seed, device="cuda", comm=comm)
            samples.append(ctx.sketch_sequences(b, o, k=K, c=C))
            del b, o
    torch.cuda.synchronize()
    t_samples = time.perf_counter() - t0
    P = contain_params(k=K, pseudotax=True)
    st = {}

    def step():
        # `sylph profile`: pass 1, winner table, pass 2, derep, abundances.  N>1: three fixed-size collectives
        # between the library's stages (sylph_b200/dist.py profile_sharded)
        if world == 1:
            st["rows"] = ctx.profile(db, samples, P)
        else:
            st["rows"] = D.profile_sharded(ctx, genomes, db, samples, rank * G, P)

    for _ in range(args.warmup):
        step()
    ctx.enable_timing(True)
    for kname in PAIR_KERNELS:
        ctx.kernel_time(kname, reset=True)
    l0 = ctx.launches
    ms, wall = timed(step, args.steps, world)
    launches = ctx.launches - l0
    per_step = {kname: ctx.kernel_time(kname, reset=True)[0] / args.steps for kname in PAIR_KERNELS}
    ctx.enable_timing(False)
    pairs = float(n_samples) * G_total
    value = pairs * args.steps / (ms * 1e-3)
    rows = st["rows"]
    if args.dump_outputs and rank == 0:
        dump_table(args.dump_outputs, "profile", {f: rows[f] for f in rows.dtype.names if f != "reserved"})
    out = {"metric": "(sample x genome) containment pairs/s", "value": value, "unit": "pairs/s", "ms_per_step": ms / args.steps,
           "wall_ms_per_step": wall / args.steps, "steps": args.steps, "gpu_launches": int(launches),
           "config": profile_config(args, world),
           "workload_stats": {"sample_keys": int(np.sum([len(s) for s in samples])), "rows_per_step": int(len(rows)),
                              "db_build_s": t_db, "samples_build_s": t_samples, "db_keys_per_gpu": db_keys,
                              "shards_with_result_rows": int(len(set((rows["genome"] // G).tolist()))) if len(rows) else 0,
                              "collectives": ("all_gather(pass-1 row tables) + all_reduce MIN(winner order per sample key) + "
                                              "all_gather(pass-2 row tables), NCCL, no host sync in between") if world > 1 else "none"},
           "e2e_note": "syl_profile returns rows in host memory: the D2H of the result rows is inside the timed region"}
    # live roofline: CUDA events recorded inside the library around every launch.  SURVEY §8(d)'s byte model (8 B x |G| per
    # pair: the reference streams every genome sketch past every sample) describes the STEP, not one kernel — the largest
    # kernel at one sample is the bootstrap, which touches 17 counters per row — so the bytes are taken over the device
    # time of all the step's kernels; the dominant kernel and its share are named next to it.
    peak, peak_src = measured_peak_hbm()
    dom = max(per_step, key=lambda kname: per_step[kname])
    alg_bytes = 8.0 * db_keys + 64.0 * G * n_samples  # 8 B x |G| per pair (db streamed once for all samples) + 64 B per row
    kern_ms = sum(per_step.values())
    ach = alg_bytes / (kern_ms * 1e-3) / 1e9 if kern_ms else None
    out["kernels_ms_per_step"] = per_step
    out["roofline"] = {"kernel": "profile step kernels (%s); largest: %s" % (" + ".join(PAIR_KERNELS[k_] for k_ in per_step), PAIR_KERNELS[dom]),
                       "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                       "frac": ach / peak if ach else None, "traffic": None, "peak_source": peak_src,
                       "kernel_ms": kern_ms, "kernel_share_of_step": kern_ms / (ms / args.steps),
                       "dominant_kernel": {"name": PAIR_KERNELS[dom], "ms": per_step[dom], "share_of_step": per_step[dom] / (ms / args.steps),
                                           "limiter": PAIR_LIMITER.get(dom)},
                       "algorithmic_bytes_per_launch": alg_bytes,
                       "note": "SURVEY §8(d) byte model of a genome-streaming probe loop; this implementation probes a sorted db "
                               "index with the sample keys and never streams the db, so this is an EQUIVALENT bandwidth (DESIGN.md "
                               "4.4); ncu --set full of the kernels: profiles/r02_contain_kernels_ncu_full_selected.csv"}
    # ---- parity: sample 0's rows against the CPU oracle on the WHOLE db (N>1: shards gathered on every rank)
    if not args.no_cpu:
        if world > 1:
            gsub = genomes.device_tensors()
            merged, _ = D.gather_survivor_genomes(gsub, np.arange(rank * G, (rank + 1) * G, dtype=np.uint64))
            d = {k_: v.cpu().numpy().view(np.uint64) for k_, v in merged.items()} if rank == 0 else None
            del merged
        else:
            d = genomes.download()
        if rank == 0:
            from oracle import oracle as O
            cores = usable_cores()
            h, c = samples[0].download()
            smp = O.Sample(h, c)
            p = O.default_params(pseudotax=True)
            t = time.perf_counter()
            res = O.contain_sample(p, d["kmers"], d["kmer_off"], d["tracked"], d["tracked_off"], d["gn_size"], smp, nthreads=cores)
            dt = time.perf_counter() - t
            out["cpu_baseline"] = {"value": G_total / dt, "unit": "pairs/s", "cores": cores, "kind": "port",
                                   "sample": "all %d pairs of sample 0 against the whole db, oracle profile (2 x get_stats + winner table) "
                                             "over %d OpenMP threads" % (G_total, cores), "rows": len(res)}
            mine = rows[rows["sample"] == 0]
            ok, why = rows_equal_oracle(mine, res)
            out["parity_checked"] = bool(ok)
            out["parity_detail"] = ("all %d profile rows of sample 0 (genomes from %d of %d shards) equal the oracle's rows on the "
                                    "whole %d-genome db field by field (ints exact, floats 1e-6)"
                                    % (len(res), len(set(int(r.genome) // G for r in res)), world, G_total)) if ok else why
            if not ok:
                raise SystemExit("bench: profile rows differ from the oracle: " + str(why))
    for s in samples:
        s.free()
    db.free()
    genomes.free()
    return out


def main():
    args = parse()
    if args.genomes is None:
        world_env = int(os.environ.get("WORLD_SIZE", 1))
        args.genomes = 12_500 if ((args.samples or (1 if world_env == 1 else 16)) > 1) else 10_000
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    rank, world, local = dist_setup(args.gpus)
    import sylph_b200
    ctx = sylph_b200.Context(local, stream=torch.cuda.current_stream().cuda_stream)
    if args.workload == "sketch":
        line, reads = bench_sketch(args, ctx, rank, world, local)
        if not args.no_pairs:
            line["pairs"] = bench_pairs(args, ctx, rank, world, local, reads)
            del reads
            line["genomes"] = bench_genomes(args, ctx, rank, world, local)
    elif args.workload == "genomes":
        line = bench_genomes(args, ctx, rank, world, local)
    else:
        from sylph_b200 import synth
        reads = synth.reads(args.reads, READ_LEN, seed=synth.SEED_READS + 0x10 * rank, device="cuda")
        p = bench_pairs(args, ctx, rank, world, local, reads)
        line = {"metric": p["metric"], "value": p["value"], "unit": p["unit"], "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": p["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": p["config"],
                "gpu_launches": p["gpu_launches"], "pairs": p}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
