#!/usr/bin/env python
"""bench.py — reads/sec of the `coverm contig|genome --bam-files` coverage hot path (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|ns|3] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workloads (`--config`, all synthetic, SURVEY.md §8d; the default is BASELINE.json configs[1]):
  2    coverm contig -m mean trimmed_mean covered_fraction, 500 000 contigs / ~2.8 Gbp / ~10.5 M records
  ns   the north-star target: the same command on a ~5 Gbp / ~52 M-record BAM (906 000 contigs)
  3    coverm genome -s '~' -m mean trimmed_mean covered_fraction --min-read-percent-identity 95,
       1000 MAGs / 200 000 contigs / ~52 M records

One "step" = one pass of the hot path over one sample.
  value     whole-job reads/s with the per-read tuples already resident in HBM: K1 filter + delta accumulation, K1b chunk
            carries, K2 TMA-staged segmented scan + reductions, K3 per-contig finalise (N > 1: plus the collective of the
            path), timed with CUDA events on the library's stream.  It explains the kernels; it is NOT the speed-up.
  e2e       the same metric through the public C ABI call a user makes (cmbh_run == `coverm ...  -b sample.bam`): BAM
            bytes in pinned HOST memory -> H2D of the compressed file -> device inflate + record decode -> kernels -> D2H of the
            per-contig table -> printed TSV in a host buffer.  Wall clock, everything inside, every step.  `cold_cli` is
            one fresh `bin/coverm` process on the same file (CUDA context, allocations, header parse, file read included).
  parity    the e2e output of the FULL file compared as text with the CPU oracle's output of the same file.
  roofline / cpu_baseline as described in DESIGN.md (Measurement).
`--impl reference` times the CPU restatement of the reference (oracle/, all host threads for BGZF inflate, the record loop
single-threaded exactly as the reference's) on the SAME file and command; one step = one full run.

`--dump-outputs DIR` writes what the last timed step returned, as float64 .npy files (at most 64 MB), so that two builds can be
compared output for output; the workload's records depend only on the arguments (`--seed` included):
  contig_stats.npy    the device step's per-contig table (cmb_contig_stats in declaration order, without `hist_offset` and
                      `reserved`), one row per contig of contig_stats_rows.npy (all contigs, or a fixed sample seeded by --seed);
                      sum_identity_primary / sum_identity_nonsupp are f64 sums of atomic adds: their last bits vary run to run
  table.npy           the numbers of the last e2e step's printed table (header and name column dropped), one row per table row
                      of table_rows.npy (same sampling); with --impl reference the oracle's table of its last run
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

GEN_CONTIG = ["--median-len", "4000", "--sigma", "0.8", "--min-len", "1000", "--max-len", "2000000"]
CONFIGS = {
    "2": {"label": "configs[1]", "sub": "contig", "contigs": 500000, "reads": 10000000, "gen": GEN_CONTIG,
          "methods": ["mean", "trimmed_mean", "covered_fraction"], "extra": []},
    "ns": {"label": "north_star target (5 Gbp / 50 M reads)", "sub": "contig", "contigs": 906000, "reads": 50000000,
           "gen": GEN_CONTIG, "methods": ["mean", "trimmed_mean", "covered_fraction"], "extra": []},
    "3": {"label": "configs[2]", "sub": "genome", "contigs": 200000, "reads": 50000000,
          "gen": ["--genomes", "1000", "--median-len", "15000", "--sigma", "0.8", "--min-len", "1000", "--max-len", "2000000"],
          "methods": ["mean", "trimmed_mean", "covered_fraction"], "extra": ["-s", "~", "--min-read-percent-identity", "95"]},
}


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


def effective_cpus():
    """CPUs this process may actually use: the smaller of the visible CPUs and the cgroup CPU quota
    (the GPU boxes expose 128 logical CPUs but cap the container via cpu.max; more threads only get throttled)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst: K2 is timed as a single launch)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """nvidia-smi SM clock / throttle-reason sampling during the timed regions."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                o = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                   capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(o[0]))
                self.max_mhz = float(o[1])
                for n, v in zip(names, o[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def gen_bam(path, cfg, contigs, reads, seed, threads):
    import coverm_b200
    t = time.time()
    meta = path + ".json"
    key = [contigs, reads, seed] + cfg["gen"]
    if os.path.exists(path) and os.path.exists(meta):  # same workload already generated in this workdir
        info = json.load(open(meta))
        if info.get("key") == key:
            info["gen_s"] = 0.0
            return info
    out = subprocess.run([coverm_b200.BAMGEN_BIN, "--out", path, "--contigs", str(contigs), "--reads", str(reads), "--seed",
                          str(seed), "--threads", str(threads)] + cfg["gen"], capture_output=True, text=True, check=True).stdout
    info = json.loads(out)
    info["gen_s"] = round(time.time() - t, 2)
    info["bam_bytes"] = os.path.getsize(path)
    info["key"] = key
    json.dump(info, open(meta, "w"))
    return info


def coverm_argv(cfg, bam, threads):
    return [cfg["sub"], "-m"] + cfg["methods"] + cfg["extra"] + ["-b", bam, "-t", str(threads)]


def workload_config(cfg, args, info, world, scaling):
    """The `config` object: a description of the WORKLOAD, identical for our arm and the reference arm (same file, same
    command, same N)."""
    if world == 1:
        par = "1 sample on 1 GPU"
    elif scaling == "weak":
        par = f"{world} samples, one per GPU; all-gather of the per-contig table"
    else:
        par = f"1 sample, contigs range-partitioned over {world} GPUs (each rank decodes its own BGZF block range); all-gather of the per-contig table"
    return {"workload": f"{cfg['label']}: coverm {cfg['sub']} -m {' '.join(cfg['methods'])} {' '.join(cfg['extra'])}".rstrip() +
                        f" on a synthetic reference-sorted BAM, {args.contigs} contigs / {info['bases']} bp / {info['records']} records",
            "config_id": args.config, "contigs": args.contigs, "reads": int(info["records"]), "bases": int(info["bases"]),
            "bam_bytes": int(info["bam_bytes"]), "seed": args.seed, "parallelism": par,
            "l2": f"inputs larger than L2 (126 MB), no flush needed: {4 * info['bases'] / 1e9:.1f} GB delta arena (4 B per reference base) + "
                  f"{48.5 * info['records'] / 1e6:.0f} MB tuples per step; e2e additionally streams the {info['bam_bytes'] / 1e9:.2f} GB file"}


def run_oracle(cfg, bam, threads, runs, warmup):
    """oracle/coverm_oracle (the CPU restatement of the reference) on `bam`: (mean seconds per run, stdout of the last run)."""
    oracle = os.path.join(ROOT, "oracle", "coverm_oracle")
    argv = [oracle] + coverm_argv(cfg, bam, threads)
    times, out = [], None
    for i in range(warmup + runs):
        t = time.perf_counter()
        p = subprocess.run(argv, capture_output=True, text=True, check=True)
        dt = time.perf_counter() - t
        if i >= warmup:
            times.append(dt)
        out = p.stdout
        log(f"oracle run {i + 1}/{warmup + runs}: {dt:.2f} s")
    return sum(times) / len(times), out


DUMP_BYTES = 64 << 20  # everything --dump-outputs writes, row indices included


def sample_rows(n, row_bytes, budget, seed):
    """Indices of the rows of an n-row output that fit in `budget` bytes: all of them, or a sorted sample fixed by `seed`."""
    import numpy as np
    cap = max(1, budget // row_bytes)
    if n <= cap:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, cap, replace=False))


def device_table(ptr, n_rows):
    """The n_rows cmb_contig_stats rows at device address `ptr` (cmb_end_sample_device), copied into a host array."""
    import numpy as np
    import torch
    from coverm_b200 import ContigStats
    cai = {"shape": (n_rows * C_sizeof(ContigStats),), "typestr": "|u1", "data": (ptr, False), "version": 2}
    rows = torch.as_tensor(type("DeviceRows", (), {"__cuda_array_interface__": cai})(), device="cuda")
    return rows.cpu().numpy().view(np.dtype(ContigStats))


def dump_outputs(out_dir, seed, table_text, stats=None):
    """--dump-outputs: the printed table's numbers and, for our arm, the device step's per-contig table (module docstring)."""
    import numpy as np
    from coverm_b200 import ContigStats
    arrays = {}
    if stats is not None:
        # hist_offset is where K3's atomic counter placed the row's histogram pairs: it follows the order the rows finished in
        fields = [f for f, _ in ContigStats._fields_ if f not in ("hist_offset", "reserved")]
        rows = sample_rows(len(stats), 8 * (len(fields) + 1), DUMP_BYTES // 3, seed)
        arrays["contig_stats"] = np.stack([stats[f][rows].astype(np.float64) for f in fields], axis=1)
        arrays["contig_stats_rows"] = rows.astype(np.float64)
    lines = table_text.splitlines()[1:]
    table = np.array([[float(x) for x in l.split("\t")[1:]] for l in lines], dtype=np.float64).reshape(len(lines), -1)
    rows = sample_rows(len(table), 8 * (table.shape[1] + 1), DUMP_BYTES // 2, seed)
    arrays["table"] = table[rows]
    arrays["table_rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log(f"wrote {', '.join(f'{n}.npy {a.shape}' for n, a in arrays.items())} to {out_dir}")


def cpu_baseline_entry(records, sec, threads, runs, what):
    return {"value": records / sec, "unit": "reads/s", "cores": threads, "kind": "port",
            "sample": f"{what}; oracle/coverm_oracle -t {threads}: {threads} BGZF inflate threads, single-threaded record loop + one "
                      f"O(L) pass per estimator as in the reference; mean of {runs} run(s)",
            "seconds_per_run": sec}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="2", choices=sorted(CONFIGS))
    ap.add_argument("--lib", default=None, help="bind another build of libcoverm_b200.so (kernel A/B experiments)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--contigs", type=int, default=0, help="override the workload's contig count")
    ap.add_argument("--reads", type=int, default=0, help="override the workload's read count")
    ap.add_argument("--seed", type=int, default=20260925)
    ap.add_argument("--e2e-steps", type=int, default=0, help="timed e2e steps (default: --steps)")
    ap.add_argument("--skip-cpu-baseline", action="store_true", help="no oracle run (then no parity check and no cpu_baseline)")
    ap.add_argument("--skip-cold-cli", action="store_true")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="N > 1: strong = one sample range-partitioned by contig over the N GPUs (default); weak = N samples, one per GPU")
    ap.add_argument("--workdir", default=os.environ.get("CMB_BENCH_DIR", "/tmp/coverm_b200_bench"))
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = CONFIGS[args.config]
    args.contigs = args.contigs or cfg["contigs"]
    args.reads = args.reads or cfg["reads"]
    metric = f"reads/sec `coverm {cfg['sub']}` ({'+'.join(cfg['methods'])})"
    if args.lib:
        import coverm_b200 as _cb
        _cb.LIB_PATH = os.path.abspath(args.lib)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    ncpu = effective_cpus()
    threads = max(1, ncpu // world)
    # stdout carries exactly one JSON line: everything else (NCCL banners, library chatter) goes to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    os.makedirs(args.workdir, exist_ok=True)

    if args.impl == "reference":
        # The reference's CPU path on the SAME file and command as our arm (rank 0's sample), every run a full pass.
        if rank != 0:
            return
        bam = os.path.join(args.workdir, f"sample_c{args.config}_r0_{args.contigs}_{args.reads}.bam")
        info = gen_bam(bam, cfg, args.contigs, args.reads, args.seed, ncpu)
        warm = 0
        if args.warmup > 0:  # one untimed warm-up run (page cache, CPU clocks); more would only repeat it
            run_oracle(cfg, bam, ncpu, 1, 0)
            warm = 1
        times = []
        for _ in range(args.steps):
            sec, out = run_oracle(cfg, bam, ncpu, 1, 0)
            times.append(sec)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, args.seed, out)
        steps = len(times)
        sec = sum(times) / steps
        cpu = cpu_baseline_entry(info["records"], sec, ncpu, steps, "the full workload file")
        line = {"impl": "reference", "metric": metric, "value": cpu["value"], "unit": "reads/s", "n_gpus": args.gpus,
                "steps": steps, "warmup": warm, "steps_requested": args.steps, "warmup_requested": args.warmup,
                "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": args.scaling if args.gpus > 1 else "weak",
                "vs_baseline": None, "dtype": "i32", "data": "synthetic",
                "config": workload_config(cfg, args, info, args.gpus, args.scaling),
                "cpu_baseline": cpu,
                "e2e": {"value": cpu["value"], "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "note": f"each step is one full `coverm` run on the whole file ({sec:.1f} s); at most one warm-up run"}
        emit(line)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import coverm_b200
    from coverm_b200 import ContigStats

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---------------------------------------------------------------- workload
    # N == 1: one sample on one GPU.  N > 1, --scaling strong (default): the SAME sample, contigs range-partitioned over the N GPUs
    # (every rank decodes only its BGZF block range; one NCCL gather of the per-contig table inside the library).
    # --scaling weak: N different samples, one per GPU, no exchange at all (replicas).
    strong = world > 1 and args.scaling == "strong"
    if strong:
        threads = ncpu  # after the gather only rank 0 works on the host (estimator replay + printing): it gets every core
    file_rank = 0 if strong else rank
    bam = os.path.join(args.workdir, f"sample_c{args.config}_r{file_rank}_{args.contigs}_{args.reads}.bam")
    if not strong or rank == 0:
        info = gen_bam(bam, cfg, args.contigs, args.reads, args.seed + file_rank, ncpu if strong else threads)
        log(f"rank {rank}: generated {bam}: {info}")
    barrier()
    if strong and rank != 0:
        info = json.load(open(bam + ".json"))
    # HOST buffer handed to the C ABI: the BAM file's bytes in pinned host memory (the contract's "inputs in pinned host
    # memory"); every e2e step copies this rank's share of them host->device again inside the timed region.
    bam_size = os.path.getsize(bam)
    bam_pinned = torch.empty(bam_size, dtype=torch.uint8, pin_memory=True)
    bam_bytes = bam_pinned.numpy()
    with open(bam, "rb") as f:
        f.readinto(memoryview(bam_bytes))
    argv = coverm_argv(cfg, bam, threads)
    file_records = int(info["records"])

    sess = coverm_b200.Session(device=local_rank, threads=threads)
    single_out = None
    if strong:
        if rank == 0:  # the single-GPU answer for the same file, before the group forms: the sharded run must print the same text
            r1 = sess.run(argv, memory_inputs={bam: bam_bytes})
            if r1.status != 0:
                raise SystemExit(f"coverm_b200 failed: {r1.err}")
            single_out = r1.out
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(coverm_b200.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        sess.set_group(rank, world, nccl_id=bytes(idt.cpu().numpy()))

    # ---------------------------------------------------------------- one e2e pass: warms the session and leaves this rank's
    # tuples in HBM (cmb_last_bgzf_batch) for the device-resident arm
    res = sess.run(argv, memory_inputs={bam: bam_bytes})
    if res.status != 0:
        raise SystemExit(f"coverm_b200 failed: {res.err}")
    s_first = res.samples[0]
    if not s_first["device_decode"]:
        raise SystemExit("the device-side decoder declined the bench file; the device-resident arm needs its tuples in HBM")
    n_contigs = args.contigs
    ctx = sess.device_context()
    ctx.n_contigs = n_contigs
    batch, n_rec, n_iv = ctx.last_bgzf_batch()
    log(f"rank {rank}: {n_rec} records, {n_iv} interval slots resident in HBM; contigs [{s_first['tid_begin']}, {s_first['tid_end']}), "
        f"{s_first['shard_blocks']} of {s_first['total_blocks']} BGZF blocks")
    cuts = None
    if strong:
        t = torch.tensor([s_first["tid_begin"]], dtype=torch.int64, device="cuda")
        allb = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allb, t)
        cuts = [int(x.item()) for x in allb] + [n_contigs]

    # ---------------------------------------------------------------- device arm: tuples resident in HBM
    stream = torch.cuda.ExternalStream(ctx.stream())
    row_bytes = n_contigs * C_sizeof(ContigStats)

    def device_step():
        ctx.begin_sample()
        ctx.submit_device_batch(batch, n_rec, n_iv)
        rows = ctx.end_sample_device()  # K1c/K1b/K2/K3 + error check (stream-synchronous); the table stays in HBM
        if strong:
            ctx.allgather_stats(cuts)  # the collective of the path, on the same stream (NCCL broadcasts of each rank's row range)
        return rows

    sampler = ClockSampler(local_rank)
    n_warm = max(3, args.warmup)
    for _ in range(n_warm):
        device_step()
    torch.cuda.synchronize()
    barrier()
    sampler.start()
    k2_ms, k1_ms, k3_ms, k0_ms, dev_ms = [], [], [], [], []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t_wall = time.perf_counter()
    with torch.cuda.stream(stream):
        ev0.record()
    launches = 0
    for _ in range(args.steps):
        dev_rows = device_step()
        tm = ctx.timing()
        k0_ms.append(tm["ms_zero"]); k1_ms.append(tm["ms_accumulate"]); k2_ms.append(tm["ms_scan"]); k3_ms.append(tm["ms_finalize"])
        dev_ms.append(tm["ms_total"])
        launches += tm["k1_launches"] + 3 + tm["k2_launches"] + tm["k3_launches"]  # K1 per batch, K1c, K1b x2, K2, K3
    with torch.cuda.stream(stream):
        ev1.record()
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t_wall) * 1e3
    barrier()
    event_ms = ev0.elapsed_time(ev1)  # the gather is enqueued on the same stream: the events bracket it too
    # the last step's table, before the e2e arm's next sample overwrites it
    dumped_stats = device_table(dev_rows, n_contigs) if args.dump_outputs and rank == 0 else None
    step_ms = max_over_ranks(event_ms / args.steps)
    total_reads = float(file_records) if strong else sum_over_ranks(float(n_rec))
    value = total_reads / (step_ms * 1e-3)
    arena_elems = ctx.timing()["arena_elems"]
    mean = lambda v: sum(v) / len(v)
    peak, peak_src = measured_peaks()
    k2_mean = mean(k2_ms)
    algo_bytes = 4.0 * arena_elems
    achieved = algo_bytes / (k2_mean * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "k2_traffic.json")
    if os.path.exists(tpath) and args.config == "2" and world == 1:
        tj = json.load(open(tpath))
        traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source", "profiles/k2_traffic.json (ncu --set full capture of this workload)")

    # ---------------------------------------------------------------- e2e arm: BAM bytes in host memory -> TSV
    e2e_steps = args.e2e_steps or args.steps
    for _ in range(max(1, min(2, args.warmup))):
        res = sess.run(argv, memory_inputs={bam: bam_bytes})
    torch.cuda.synchronize()
    barrier()
    t_e = time.perf_counter()
    breakdown = []
    step_walls = []
    for _ in range(e2e_steps):
        t_s = time.perf_counter()
        res = sess.run(argv + ["--timing"], memory_inputs={bam: bam_bytes})
        step_walls.append(time.perf_counter() - t_s)
        breakdown.append(res.samples[0])
    log("e2e step walls (s): " + " ".join(f"{w:.4f}" for w in step_walls))
    log("e2e per step: copy+inflate ms " + " ".join(f"{b['decode_copy_inflate_ms']:.1f}" for b in breakdown) + " | second-pass blocks " +
        " ".join(str(b["decode_second_pass_blocks"]) for b in breakdown) + " | host blocks " + " ".join(str(b["decode_host_blocks"]) for b in breakdown) + " | copy-enqueue wall ms " +
        " ".join(f"{b['decode_copy_enqueue_wall_ms']:.0f}" for b in breakdown) + " | submit_bgzf host wall ms " + " ".join(f"{b['decode_host_wall_ms']:.0f}" for b in breakdown))
    log("e2e last step host timing: " + " | ".join(l for l in res.err.splitlines() if l.startswith("#timing")))
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t_e) / e2e_steps
    barrier()
    e2e_s = max_over_ranks(e2e_s)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    s0 = breakdown[-1]
    e2e_value = total_reads / e2e_s
    # device decode: the BGZF bytes of the rank's block range + block table; host decode: 40 B/record + 8 B/interval tuples
    h2d = sum_over_ranks(float(s0["h2d_bytes"]))
    d2h = row_bytes * world
    e2e_launches = s0["decode_launches"] + s0["k1_launches"] + 3 + s0["k2_launches"] + s0["k3_launches"]
    e2e_out = res.out  # the table of the last timed step (full file)
    same_as_single = None
    if strong and rank == 0:
        same_as_single = e2e_out == single_out
        if not same_as_single:
            log("MISMATCH: the sharded run's table differs from the single-GPU run of the same file")

    # ---------------------------------------------------------------- cold CLI: one fresh process on the same file
    cold = None
    if rank == 0 and not args.skip_cold_cli:
        out_path = os.path.join(args.workdir, "cold_cli.tsv")
        extra = ["--gpus", str(world)] if strong else []
        t_c = time.perf_counter()
        p = subprocess.run([coverm_b200.COVERM_BIN] + coverm_argv(cfg, bam, ncpu if strong else threads) + extra + ["-o", out_path],
                           capture_output=True, text=True) if (world == 1 or strong) else None
        cold_s = time.perf_counter() - t_c
        if p is not None:
            same = p.returncode == 0 and open(out_path).read() == e2e_out
            cold = {"seconds": cold_s, "reads_per_s": file_records / cold_s, "output_identical_to_session_run": same,
                    "what": "one fresh `bin/coverm" + (f" --gpus {world}" if strong else "") + "` process, file read from the page cache: CUDA "
                            "context(s) + arena cudaMalloc + tensor-map encode + header parse + decode + kernels + printing to a file"}
            if not same:
                log(f"cold CLI run differs or failed (rc {p.returncode}): {p.stderr[-400:]}")
    barrier()

    # ---------------------------------------------------------------- CPU baseline + parity on the FULL file (N = 1 only)
    cpu = None
    parity = None
    if rank == 0 and world == 1 and not args.skip_cpu_baseline:
        sec, oracle_out = run_oracle(cfg, bam, ncpu, 1, 0)
        cpu = cpu_baseline_entry(n_rec, sec, ncpu, 1, "the full workload file (the same file the GPU arm ran)")
        parity = e2e_out == oracle_out
        if not parity:
            gl, ol = e2e_out.splitlines(), oracle_out.splitlines()
            diff = [(i, a, b) for i, (a, b) in enumerate(zip(gl, ol)) if a != b][:5]
            log(f"PARITY FAILURE on the full file: {len(gl)} vs {len(ol)} lines; first differences {diff}")
    sess.close()

    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, args.seed, e2e_out, dumped_stats)
    if rank == 0:
        scaling = "strong" if strong else "weak"
        config = workload_config(cfg, args, info, world, scaling)
        host = {"host_threads_per_rank": threads, "host_cpus_effective": ncpu, "host_cpus_visible": os.cpu_count(), "records_rank0": n_rec}
        line = {
            "metric": metric, "value": value, "unit": "reads/s", "n_gpus": world, "steps": args.steps, "warmup": n_warm,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "i32",
            "data": "synthetic", "config": config, "host": host, "clocks": sampler.summary(),
            "e2e": {"value": e2e_value, "unit": "reads/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "seconds_per_step": e2e_s, "steps": e2e_steps,
                    "breakdown_last_step_rank0": {k: s0[k] for k in ["total_s", "decode_s", "submit_wait_s", "end_sample_s", "gather_s", "k0_ms", "k1_ms",
                                                                     "k2_ms", "k3_ms", "device_total_ms", "device_decode",
                                                                     "decode_host_blocks", "decode_copy_inflate_ms", "decode_chain_ms",
                                                                     "decode_extract_ms", "shard_blocks", "total_blocks", "range_probes",
                                                                     "tid_begin", "tid_end", "group_ranks"]},
                    "step_walls_s": step_walls, "gpu_launches_per_step": int(e2e_launches),
                    "decode": "device (kd_inflate_t1 or kd_inflate_g8 by block count, kd_guess/kd_walk/kd_extract: compressed BGZF bytes cross PCIe)" if s0["device_decode"] else "host pipeline (tuples cross PCIe)",
                    "input": f"BAM bytes ({len(bam_bytes)} B) in pinned host memory, cmbh_run (== `coverm {cfg['sub']}`), TSV text out; "
                             "warm session (context, arena, decode buffers and the parsed header are reused across steps)" +
                             ("; collective: every rank calls cmbh_run, the in-library NCCL gather is inside the timed region" if strong else ""),
                    "output_identical_to_single_gpu_run": same_as_single,
                    "cold_cli": cold},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "k2_scan_reduce<HIST,CLEAN>", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": algo_bytes, "avg_launch_ms": k2_mean,
                         "note": "rank 0's launch" + (" (1/N of the arena)" if strong else "")},
            "device_breakdown_ms_rank0": {"k0_zero": mean(k0_ms), "k1_filter_delta+carry": mean(k1_ms), "k2_scan_reduce": k2_mean,
                                          "k3_finalize": mean(k3_ms), "kernels_stream_total": mean(dev_ms), "step_incl_gather": event_ms / args.steps,
                                          "wall_per_step": wall_ms / args.steps},
            "cpu_baseline": cpu, "parity": parity,
            "parity_what": "text of the e2e table of the full file == oracle/coverm_oracle's output of the same file" if parity is not None else None,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def C_sizeof(t):
    import ctypes
    return ctypes.sizeof(t)


if __name__ == "__main__":
    main()
