#!/usr/bin/env python
"""bench.py — throughput of the B200 seed-and-extend hot path (BASELINE.json metric: paired 151 bp
reads/s) with roofline and the reference CPU path beside it.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload bsw|pipeline] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic reads.  See DESIGN.md §Measurement.
--dump-outputs DIR (default workload) writes the alignment regions of the timed path as DIR/*.npy, so that two builds
can be compared output for output on the same seeded inputs (see dump_pipeline_outputs).
"""
from __future__ import annotations
import argparse, json, os, subprocess, sys, tempfile, threading, time
import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from __graft_entry__ import load_package  # noqa: E402


def _smem_traffic(args):
    """DRAM bytes per step of the SMEM-stage kernels from the committed ncu capture, when it was taken on this workload."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "smem_traffic.json")))
        if t["ref_mbp"] == args.ref_mbp and t["pairs"] == args.pairs:
            return t["dram_bytes_per_step"]
    except Exception:
        pass
    return None


def _isa():
    flags = open("/proc/cpuinfo").read()
    return "avx512bw" if "avx512bw" in flags else "avx2"


def _refbin(name):
    p = os.path.join(ROOT, "oracle", "_ref", _isa(), name)
    if not os.path.exists(p):
        raise RuntimeError(f"{p} missing: run __graft_entry__.build() where /root/reference exists")
    return p


def _cgroup_cpu_limit():
    """CPU quota of this process's cgroup in cores (None = unlimited / unknown); v2 cpu.max, v1 cfs_quota/period."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        return None if q == "max" else float(q) / float(per)
    except Exception:
        pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return None if q <= 0 else q / per
    except Exception:
        return None


def host_threads():
    """Threads for the reference arm: the cores this process may really use (affinity, cgroup quota), at most 128
    (the reference's tprof[][] is 128 columns wide, src/macro.h LIM_C)."""
    n = len(os.sched_getaffinity(0))
    q = _cgroup_cpu_limit()
    if q is not None:
        n = min(n, max(1, int(q + 0.5)))
    return max(1, min(n, 128))


def host_info(probe=True):
    """What the CPU arm ran on: model, logical CPUs, affinity, cgroup quota, load, and the MEASURED parallel capacity
    (oracle/libbm2oracle.so:bm2o_cpu_probe - rate of a fixed integer loop on n threads / rate on 1 thread)."""
    info = {"cpu_model": None, "logical_cpus": os.cpu_count(), "affinity": len(os.sched_getaffinity(0)),
            "cgroup_cpu_max": _cgroup_cpu_limit(), "threads_used": host_threads(), "isa": _isa()}
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                info["cpu_model"] = ln.split(":", 1)[1].strip(); break
        info["loadavg_1min"] = float(open("/proc/loadavg").read().split()[0])
    except Exception:
        pass
    if probe:
        try:
            import ctypes as C
            L = C.CDLL(os.path.join(ROOT, "oracle", "libbm2oracle.so")); L.bm2o_cpu_probe.restype = C.c_double
            r1 = L.bm2o_cpu_probe(1, C.c_double(0.25)); rn = L.bm2o_cpu_probe(info["threads_used"], C.c_double(0.5))
            info["effective_cores"] = round(rn / r1, 1) if r1 > 0 else None
            info["effective_cores_how"] = f"integer-loop rate on {info['threads_used']} threads / rate on 1 thread (0.5 s)"
        except Exception as e:
            info["effective_cores"] = None; info["effective_cores_how"] = f"probe failed: {e!r}"
    return info


METRIC_BSW = "paired 151bp reads/s (BSW extension only, seeds from the reference CPU path)"
METRIC = "paired 151bp reads/s (seed+chain+extend hot path)"      # the SAME string in both arms: the driver compares them


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, gpu=0):
        self.gpu = gpu; self.rows = []; self._stop = False; self.t = None

    def start(self):
        def run():
            q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
            while not self._stop:
                try:
                    o = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                       capture_output=True, text=True, timeout=5).stdout.strip()
                    if o:
                        self.rows.append([x.strip() for x in o.split(",")])
                except Exception:
                    pass
                time.sleep(0.2)
        self.t = threading.Thread(target=run, daemon=True); self.t.start()

    def stop(self):
        self._stop = True
        if self.t:
            self.t.join(timeout=6)
        sm = [int(r[0]) for r in self.rows if r and r[0].isdigit()]
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) > 2 + i and r[2 + i] == "Active"})
        return {"sm_mhz": int(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# workload preparation (untimed): synthetic genome + reads, reference-built index, and for the
# BSW-only configuration the extension jobs as the reference's CPU seeding/chaining produces them
# ------------------------------------------------------------------------------------------------
def prepare_inputs(work, ref_bp, n_pairs, seed):
    pkg = load_package()
    from bwa_mem2_b200 import synth
    os.makedirs(work, exist_ok=True)
    fa = os.path.join(work, "ref.fa")
    if not os.path.exists(fa + ".bwt.2bit.64"):
        ctg = synth.make_reference(ref_bp, seed=seed, n_contigs=4)
        synth.write_fasta(fa, ctg)
        subprocess.check_call([_refbin("bwa-mem2"), "index", fa], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        r1, r2 = synth.make_pairs(ctg, n_pairs, seed=seed + 1)
        synth.write_fastq(os.path.join(work, "r1.fq"), r1, "p"); synth.write_fastq(os.path.join(work, "r2.fq"), r2, "p")
        np.save(os.path.join(work, "reads.npy"), np.stack([r1, r2], 1).reshape(-1, r1.shape[1]))
    return fa


def reference_bsw_jobs(work, fa):
    """Extension jobs exactly as the reference builds them (seeds from the CPU path), via ref_driver."""
    import refdump
    dump = os.path.join(work, "dump")
    stats = os.path.join(work, "stats.json")
    if not os.path.exists(dump + ".bsw.bin"):
        env = dict(os.environ, BM2_DUMP_PREFIX=dump, BM2_STATS=stats)
        with open(os.path.join(work, "ref.sam"), "w") as f:
            subprocess.check_call([_refbin("ref_driver"), "mem", "-t", "1", "-K", "100000000", fa, os.path.join(work, "r1.fq"),
                                   os.path.join(work, "r2.fq")], stdout=f, stderr=subprocess.DEVNULL, env=env)
    g = refdump.merge_bsw(refdump.read_bsw(dump + ".bsw.bin"))
    g = [x for x in g if x["w"] == 100][0]
    st = json.load(open(stats))
    return g, st


def bsw_check(got, ref_out):
    """score/qle/tle/max_off exact; gscore/gtle exact where the reference's gscore > 0.  With gscore <= 0 the
    reference's SIMD kernels return 0 or -1 depending on the lane neighbours (3 of 906 530 jobs here) and its
    only consumer tests `gscore <= 0` (src/bwamem.cpp:2498, :2715)."""
    for k, f in ((0, "score"), (1, "tle"), (3, "qle"), (5, "max_off")):
        assert np.array_equal(got[f], ref_out[:, k]), f"bench workload: {f} differs from the reference"
    pos = ref_out[:, 4] > 0
    assert np.array_equal(got["gscore"][pos], ref_out[pos, 4]) and np.array_equal(got["gtle"][pos], ref_out[pos, 2])
    assert np.all(got["gscore"][~pos] <= 0)


def run_bsw(args, rank, world):
    import torch
    pkg = load_package()
    capi = pkg.capi
    import oracle_lib as ol
    dev = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(dev)
    work = os.path.join(tempfile.gettempdir(), f"bm2_bench_bsw_{args.ref_mbp}_{args.pairs}")
    if rank == 0:
        fa = prepare_inputs(work, args.ref_mbp * 1_000_000, args.pairs, seed=11)
        reference_bsw_jobs(work, fa)
    if world > 1:
        torch.distributed.barrier()
    g, st = reference_bsw_jobs(work, os.path.join(work, "ref.fa"))
    n0 = len(g["h0"])
    reads_per_rep = st["reads"]
    # replicate the job list so that one step is well above L2 (126 MB) in sequence bytes
    rep = max(1, int(np.ceil(args.bsw_jobs / n0)))
    n = n0 * rep
    pairs = np.zeros(n, capi.PAIR_DT)
    ref_len = len(g["ref"]); qer_len = len(g["qer"])
    for r in range(rep):
        s = slice(r * n0, (r + 1) * n0)
        pairs["len1"][s] = g["len1"]; pairs["len2"][s] = g["len2"]; pairs["h0"][s] = g["h0"]
        pairs["idr"][s] = g["idr"] + r * ref_len; pairs["idq"][s] = g["idq"] + r * qer_len
    ref = np.tile(g["ref"], rep); qer = np.tile(g["qer"], rep)
    assert int(pairs["idr"].astype(np.int64).max()) < 2 ** 31 - 70000
    ctx = capi.Context(dev)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    ctx.set_sub_batches(args.sub_batches)
    int_gops = ctx.int_pipe_gops()
    d_pairs = torch.from_numpy(pairs.view(np.uint8).reshape(-1)).cuda()
    d_ref = torch.from_numpy(ref).cuda(); d_qer = torch.from_numpy(qer).cuda()
    d_cells = torch.zeros(1, dtype=torch.int64, device="cuda")
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")

    def step():
        ctx.extend_pairs_device(d_pairs.data_ptr(), d_ref.data_ptr(), d_qer.data_ptr(), n, 100, 5, d_cells.data_ptr())

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    # parity spot check of the bench workload itself (first replica) against the reference outputs
    got = d_pairs.cpu().numpy().view(capi.PAIR_DT)[:n0]
    bsw_check(got, g["out"])
    d_cells.zero_()
    sampler = ClockSampler(dev); sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for a, b in evs:
        flush.fill_(1)                      # L2 flush between timed iterations
        a.record(stream); step(); b.record(stream)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    ms = [a.elapsed_time(b) for a, b in evs]
    ms_step = float(np.mean(ms))
    cells = int(d_cells.item()) / args.steps
    if world > 1:
        t = torch.tensor([ms_step], device="cuda"); torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms_step = float(t.item())
    reads_per_step = reads_per_rep * rep
    value = world * reads_per_step / (ms_step * 1e-3)
    # e2e through the host C ABI: pinned host buffers, H2D + D2H inside the timed region
    h_pairs = torch.from_numpy(pairs.view(np.uint8).reshape(-1).copy()).pin_memory()
    h_ref = torch.from_numpy(ref).pin_memory(); h_qer = torch.from_numpy(qer).pin_memory()
    ctx.set_stream(None)
    hp = h_pairs.numpy().view(capi.PAIR_DT)
    ctx.extend_pairs(hp, h_ref.numpy(), h_qer.numpy(), 100, 5)
    t0 = time.perf_counter()
    e2e_steps = max(1, min(args.steps, 3))
    for _ in range(e2e_steps):
        ctx.extend_pairs(hp, h_ref.numpy(), h_qer.numpy(), 100, 5)
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    if world > 1:
        t = torch.tensor([e2e_s], device="cuda"); torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        e2e_s = float(t.item())
    out = None
    if rank == 0:
        gcups = cells / (ms_step * 1e-3) / 1e9
        peak_cells = int_gops / 14.0          # 14 two-input ops per cell update (SURVEY.md 8d)
        # CPU baseline: the reference's own AVX-512 BSW calls timed by ref_driver on this host (1 thread)
        cpu = {"value": st["reads"] / st["t_bsw"], "unit": "reads/s", "cores": 1, "kind": "reference",
               "sample": f"{st['bsw_pairs']} extension jobs of {st['reads']} reads, reference getScores8/16 ({_isa()}), 1 thread"}
        out = {"metric": METRIC_BSW, "value": value,
               "unit": "reads/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16", "data": "synthetic",
               "config": {"workload": f"config[1]-like: BSW kernel only; {reads_per_step} reads/step/GPU = {n} extension jobs "
                                      f"(jobs of {st['reads']} synthetic 2x151 reads vs {args.ref_mbp} Mbp synthetic reference, x{rep})",
                          "l2": "256 MB flush between steps", "band": 100},
               "e2e": {"value": world * reads_per_step / e2e_s, "unit": "reads/s", "h2d_bytes_per_step": int(pairs.nbytes + ref.nbytes + qer.nbytes),
                       "d2h_bytes_per_step": int(pairs.nbytes)},
               "gpu_launches": 14 * args.steps,
               "roofline": {"bound": "int_alu", "achieved": gcups, "peak": peak_cells, "unit": "Gcell/s", "frac": gcups / peak_cells,
                            "traffic": None, "note": f"cells = banded DP cells actually computed; peak = measured int pipe {int_gops:.0f} Gop/s / 14 ops per cell"},
               "cpu_baseline": cpu, "clocks": clocks, "wall_s": wall}
    ctx.close()
    return out


def prepare_pipeline_inputs(work, ref_bp, n_pairs, seed):
    """Synthetic genome + index + vectorised 2x151 read pairs (cached in `work`).  Genomes up to 400 Mbp are indexed by
    the reference binary itself; larger ones (the ~3 Gbp configurations) by bwa_mem2_b200.index_build on the GPU, which
    writes the same files byte for byte (tests/test_index_build.py) - the reference's builder needs 1-2 h for 3 Gbp."""
    load_package()
    from bwa_mem2_b200 import synth
    os.makedirs(work, exist_ok=True)
    fa = os.path.join(work, "ref.fa")
    if os.path.exists(os.path.join(work, "reads.npy")):
        return fa
    t0 = time.time()
    if ref_bp <= 400_000_000:
        ctg = synth.make_reference(ref_bp, seed=seed, n_contigs=max(4, min(24, ref_bp // 25_000_000)))
        synth.write_fasta(fa, ctg)
        subprocess.check_call([_refbin("bwa-mem2"), "index", fa], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        sys.stderr.write(f"[bench] reference binary indexed {ref_bp} bp in {time.time() - t0:.1f}s\n")
        r1, r2 = synth.make_pairs_fast(ctg, n_pairs, seed=seed + 1)
    else:
        import torch
        from bwa_mem2_b200 import index_build
        ctg = index_build.make_big_reference(ref_bp, seed=seed, n_contigs=24, device="cuda")
        sys.stderr.write(f"[bench] synthetic genome of {ref_bp} bp generated in {time.time() - t0:.1f}s\n")
        genome = torch.cat([c for _, c in ctg])
        r1, r2 = synth.make_pairs_torch(genome, [len(c) for _, c in ctg], n_pairs, seed=seed + 1)
        del genome
        t1 = time.time()
        fm = index_build.write_index(fa, ctg, device="cuda", log=lambda m: sys.stderr.write(f"[bench] index_build: {m}\n"))
        del fm, ctg
        torch.cuda.empty_cache()
        sys.stderr.write(f"[bench] GPU index build + write of {ref_bp} bp took {time.time() - t1:.1f}s\n")
    reads = np.empty((2 * n_pairs, r1.shape[1]), np.uint8); reads[0::2] = r1; reads[1::2] = r2
    synth.write_fastq_fast(os.path.join(work, "r1.fq"), r1); synth.write_fastq_fast(os.path.join(work, "r2.fq"), r2)
    np.save(os.path.join(work, "reads.npy"), reads)
    return fa


def reference_hotpath(work, fa, n_pairs_sample, threads, steps=1, warmup=0, dump_regs=None):
    """reads/s of the unmodified reference's worker_bwt + worker_aln (ref_driver BM2_MODE=hotpath) on the first
    n_pairs_sample pairs: ONE process (one index load), warmup + steps repetitions of the two kt_for phases inside it
    (BM2_REPEAT), each timed alone.  dump_regs: file that receives the reference's regs of those reads (parity of the
    bench workload against the reference itself).  -> (mean reads/s over the timed repetitions, per-repetition list, stats)."""
    r1 = os.path.join(work, "r1.fq"); r2 = os.path.join(work, "r2.fq")
    s1 = os.path.join(work, f"s1_{n_pairs_sample}.fq"); s2 = os.path.join(work, f"s2_{n_pairs_sample}.fq")
    if not os.path.exists(s1):
        rec = os.path.getsize(r1) // (np.load(os.path.join(work, "reads.npy"), mmap_mode="r").shape[0] // 2)
        for src, dst in ((r1, s1), (r2, s2)):
            with open(src, "rb") as f, open(dst, "wb") as o:
                o.write(f.read(rec * n_pairs_sample))
    stats = os.path.join(work, "stats_ref.json")
    env = dict(os.environ, BM2_MODE="hotpath", BM2_STATS=stats, BM2_REPEAT=str(warmup + steps))
    if dump_regs:
        env["BM2_DUMP_REGS"] = dump_regs
    subprocess.check_call([_refbin("ref_driver"), "mem", "-t", str(threads), "-K", "1000000000", fa, s1, s2],
                          stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, env=env)
    st = json.load(open(stats))
    reps = st.get("rep_s") or [st["t_bwt"] + st["t_aln"]]
    vals = [st["reads"] / t for t in reps[warmup:]]
    return float(np.mean(vals)), vals, st


def check_against_reference_dump(regs, ro, dump_path, n_reads):
    """Every field of every alignment region of the first n_reads reads == the unmodified reference's own regs
    (ref_driver BM2_DUMP_REGS).  Raises on a difference."""
    import refdump, oracle_lib as ol
    d_regs, d_off = refdump.read_regs(dump_path)
    assert len(d_off) == n_reads + 1, f"reference dump holds {len(d_off) - 1} reads, expected {n_reads}"
    bad = ol.regs_equal_to_dump(regs[:ro[n_reads]], ro[:n_reads + 1], d_regs, d_off)
    if bad or len(d_regs) != ro[n_reads]:
        raise AssertionError(f"bench workload: GPU regs differ from the unmodified reference on reads {bad[:10]} "
                             f"({ro[n_reads]} vs {len(d_regs)} regs)")
    return int(len(d_regs))


DUMP_SAMPLE_READS = 16384
DUMP_U64_FIELDS = ("c", "hash")


def dump_pipeline_outputs(out_dir, regs, ro, seed=1234):
    """The regions a caller of the timed path receives, as float64 / float32 .npy files (well under 64 MB):
    regs_per_read.npy (every read), sample_reads.npy (a fixed, seeded sample of DUMP_SAMPLE_READS reads, ascending) and
    reg_<field>.npy for every field of every region of the sampled reads, in output order.  64-bit unsigned fields are
    split into <field>_lo / <field>_hi 32-bit halves so that float64 holds them exactly; padding is left out."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(ro) - 1
    per_read = np.diff(ro)
    assert per_read.max(initial=0) < 1 << 24
    np.save(os.path.join(out_dir, "regs_per_read.npy"), per_read.astype(np.float32))
    sample = np.sort(np.random.default_rng(seed).choice(n, min(n, DUMP_SAMPLE_READS), replace=False))
    np.save(os.path.join(out_dir, "sample_reads.npy"), sample.astype(np.float64))
    idx = np.concatenate([np.arange(ro[r], ro[r + 1]) for r in sample]) if len(sample) else np.zeros(0, np.int64)
    sel = regs[idx]
    for f in regs.dtype.names:
        if f.startswith("_"):
            continue
        v = sel[f]
        if f in DUMP_U64_FIELDS:
            v = v.astype(np.uint64)
            np.save(os.path.join(out_dir, f"reg_{f}_lo.npy"), (v & np.uint64(0xFFFFFFFF)).astype(np.float64))
            np.save(os.path.join(out_dir, f"reg_{f}_hi.npy"), (v >> np.uint64(32)).astype(np.float64))
        else:
            assert v.dtype.kind == "f" or np.abs(v.astype(np.int64)).max(initial=0) < 1 << 53, f
            np.save(os.path.join(out_dir, f"reg_{f}.npy"), v.astype(np.float64))


def run_pipeline(args, rank, world):
    import torch
    pkg = load_package()
    capi = pkg.capi
    import oracle_lib as ol
    dev = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(dev)
    work = os.path.join(tempfile.gettempdir(), f"bm2_bench_pipe_{args.ref_mbp}_{args.pairs}")
    if rank == 0:
        prepare_pipeline_inputs(work, args.ref_mbp * 1_000_000, args.pairs, seed=21)     # a failure here fails the bench (no smaller stand-in)
    if world > 1:
        torch.distributed.barrier()
    fa = os.path.join(work, "ref.fa")
    sa = None
    startup = {}
    if world > 1:
        # the product's multi-GPU start-up (bwa_mem2_b200.shard): rank 0 reads the index files, the other ranks receive the four big
        # arrays by ONE NCCL broadcast over NVLink and adopt them in place (bm2_create_resident); chunk c of the stream goes to rank c % N
        import importlib
        shard = importlib.import_module("bwa_mem2_b200.shard")
        sa = shard.ShardedAligner(capi, fa, device=dev, keep_host_index=(rank == 0))
        ctx = sa.ctx; index = sa.index
        startup = {k: round(v, 3) for k, v in sa.startup.items()}
        if rank == 0:
            reads = np.load(os.path.join(work, "reads.npy"))
        else:       # weak scaling over ONE stream of N x 1 M reads: this rank's chunk is its own reads, drawn from the resident reference
            from bwa_mem2_b200 import synth
            m = sa.meta
            r1, r2 = synth.make_pairs_torch(sa.big[3][:m["l_pac"]], m["ann_len"], args.pairs, seed=22 + rank)
            reads = np.empty((2 * args.pairs, r1.shape[1]), np.uint8); reads[0::2] = r1; reads[1::2] = r2
            del r1, r2
    else:
        reads = np.load(os.path.join(work, "reads.npy"))
        index = capi.Index(fa)
        ctx = capi.Context(dev, index=index)
    n = reads.shape[0]
    codes = reads.reshape(-1); offs = (np.arange(n + 1, dtype=np.int64) * reads.shape[1])
    # parity of the bench workload itself: a slice against the oracle, every field of every reg
    ns = 4000
    if index is not None:
        got, go = ctx.seed_chain_extend(codes[:ns * reads.shape[1]], offs[:ns + 1])
        want, wo, _, rc = ol.seed_chain_extend(index, ctx.opt, codes[:ns * reads.shape[1]], offs[:ns + 1])
        assert rc == 0 and np.array_equal(go, wo) and got.tobytes() == want.tobytes(), "bench workload differs from the oracle"
    # ... and of the sub-batch path the timed steps use: the same reads split into sub-batches in flight give the same bytes
    nsb = min(n, 65536)
    if args.sub_batches > 1 and nsb >= 2 * 16384:
        ctx.set_sub_batches(1)
        r_one, o_one = ctx.seed_chain_extend(codes[:nsb * reads.shape[1]], offs[:nsb + 1])
        ctx.set_sub_batches(args.sub_batches)
        r_sub, o_sub = ctx.seed_chain_extend(codes[:nsb * reads.shape[1]], offs[:nsb + 1])
        assert np.array_equal(o_one, o_sub) and r_one.tobytes() == r_sub.tobytes(), "sub-batches in flight differ from the unsplit batch"
        del r_one, r_sub
    int_gops = ctx.int_pipe_gops()
    # random-gather probes over the Occ table: request shape (64 B as 4 x 16 B loads / 32 B as one 256-bit load / 64 B as two) x
    # requests in flight per thread, inside L2 (32 MB span) and over 4 GB: separates DRAM, request-rate and latency limits; the last shape is
    # the bulk-async (TMA) path: cp.async.bulk of 32 B into shared memory behind a per-thread mbarrier
    gather_by_span = {f"{mb}MB_{nm}_mlp{k}": round(ctx.gather_probe(mb << 20, k, sh), 1)
                      for mb in (32, 4096) for sh, nm in ((0, "64B_4x16"), (1, "32B_1x256"), (2, "64B_2x256"), (3, "32B_bulk_async_tma"), (4, "32B_tma_plus_loads")) for k in (1, 4, 8)
                      if not (sh >= 3 and k == 8)}
    index_how = "built by the reference binary" if args.ref_mbp <= 400 else "built on the GPU by bwa_mem2_b200.index_build, byte-identical format"
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    d_codes = torch.from_numpy(codes).cuda(); d_offs = torch.from_numpy(offs).cuda()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    for _ in range(args.warmup):
        ctx.seed_chain_extend_resident(codes, offs, d_codes.data_ptr(), d_offs.data_ptr(), False)
    torch.cuda.synchronize()
    sampler = ClockSampler(dev); sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    stage_acc = {}; cnt = None
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for a, b in evs:
        flush.fill_(1)
        a.record(stream)
        n_regs = ctx.seed_chain_extend_resident(codes, offs, d_codes.data_ptr(), d_offs.data_ptr(), False)
        b.record(stream)
        for k, v in ctx.stage_ms().items():
            stage_acc[k] = stage_acc.get(k, 0.0) + v / args.steps
        cnt = ctx.counters()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    ms_step = float(np.mean([a.elapsed_time(b) for a, b in evs]))
    if world > 1:
        t = torch.tensor([ms_step], device="cuda"); torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms_step = float(t.item())
    value = world * n / (ms_step * 1e-3)
    if args.dump_outputs and rank == 0:
        # the timed calls leave their regions on the device (copy_out=False); one more call, same batch and sub-batches, copies them out
        d_regs, d_ro = ctx.seed_chain_extend_resident(codes, offs, d_codes.data_ptr(), d_offs.data_ptr(), True, return_arrays=True)
        assert len(d_regs) == n_regs, f"regions of the dumped step ({len(d_regs)}) differ from the last timed step ({n_regs})"
        dump_pipeline_outputs(args.dump_outputs, d_regs, d_ro)
        del d_regs, d_ro
    # the stages alone: one more pass of the same batch UNSPLIT, so that every kernel is timed without another sub-batch's
    # kernels beside it (the roofline figures below; the timed steps above run args.sub_batches sub-batches in flight,
    # whose per-stage times are sums over sub-batches and overlap each other)
    stage_split = dict(stage_acc)
    if args.sub_batches > 1:
        ctx.set_sub_batches(1)
        flush.fill_(1)
        ctx.seed_chain_extend_resident(codes, offs, d_codes.data_ptr(), d_offs.data_ptr(), False)     # buffers of the unsplit path
        flush.fill_(1)
        ctx.seed_chain_extend_resident(codes, offs, d_codes.data_ptr(), d_offs.data_ptr(), False)
        torch.cuda.synchronize()
        stage_acc = dict(ctx.stage_ms()); cnt = ctx.counters()
        ctx.set_sub_batches(args.sub_batches)
    # e2e through the host C ABI (pinned host reads in, regs out to pinned host memory)
    ctx.set_stream(None)
    h_codes = torch.from_numpy(codes.copy()).pin_memory(); h_offs = torch.from_numpy(offs.copy()).pin_memory()
    regs, ro = ctx.seed_chain_extend(h_codes.numpy(), h_offs.numpy(), copy=False)
    n_out = len(regs)
    e2e_steps = max(1, min(args.steps, 3))
    tab = torch.zeros((world, 4), dtype=torch.int64, device="cuda") if world > 1 else None
    if world > 1:
        torch.distributed.barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    for step_i in range(e2e_steps):
        regs, ro = ctx.seed_chain_extend(h_codes.numpy(), h_offs.numpy(), copy=False)
        if world > 1:    # the ordering step of the sharded run: every rank learns (chunk id, owner, reads, regs) of the step's N chunks
            mine = torch.tensor([step_i * world + rank, rank, n, len(regs)], dtype=torch.int64, device="cuda")
            torch.distributed.all_gather_into_tensor(tab, mine)
    if world > 1:
        torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    if world > 1:
        assert tab[:, 1].tolist() == list(range(world)) and int(tab[:, 2].sum()) == world * n
        t = torch.tensor([e2e_s], device="cuda"); torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        e2e_s = float(t.item())
    out = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        smem_ms = stage_acc.get("smem", 0.0)
        alg_bytes = cnt["n_ext"] * 128.0
        achieved = alg_bytes / (smem_ms * 1e-3) / 1e9 if smem_ms > 0 else 0.0
        bsw_ms = stage_acc.get("bsw_left", 0.0) + stage_acc.get("bsw_right", 0.0)
        # CPU arm + parity against the reference ITSELF: the unmodified reference's worker_bwt + worker_aln on the first
        # sample of the same reads (all usable host threads, one process), its regs dumped and compared field by field
        hi = host_info()
        nt = hi["threads_used"]
        sample_pairs = min(args.pairs, 100_000)
        dump = os.path.join(work, "ref_regs.bin")
        cpu_v, cpu_vals, cpu_st = reference_hotpath(work, fa, sample_pairs, nt, steps=3, warmup=1, dump_regs=dump)
        n_ref_regs = check_against_reference_dump(regs, ro, dump, 2 * sample_pairs)
        os.remove(dump)
        # roofline objects of the two big stages; `roofline` is the one that dominates the unsplit stage times
        gcells = cnt["cells"] / (bsw_ms * 1e-3) / 1e9 if bsw_ms > 0 else 0.0
        ceil = {"pack1_s32": int_gops / 14.0, "pack2_s16x2": 2 * int_gops / 14.0, "pack4_s8x4": 4 * int_gops / 14.0}
        roof_bsw = {"bound": "int_alu", "achieved": gcells, "peak": ceil["pack2_s16x2"], "unit": "Gcell/s",
                    "frac": gcells / ceil["pack2_s16x2"] if int_gops > 0 else None, "traffic": None,
                    "kernel": "extension stage: bsw_col2_kernel launches of bsw_left + bsw_right (incl. job bucketing, fold, doubled-band retry)",
                    "kernel_ms": bsw_ms, "ceilings_gcell_s": {k: round(v, 1) for k, v in ceil.items()},
                    "frac_by_ceiling": {k: (gcells / v if v > 0 else None) for k, v in ceil.items()},
                    "note": f"cells = banded DP cells counted by the kernels; ceilings = {int_gops:.0f} G two-input int32 op/s measured in-library "
                            "(bm2_int_pipe_gops: dependent VIADDMNMX chains on all SMs) x pack / 14 ops per cell (SURVEY 8d).  peak/frac use pack 2: the "
                            "kernel issues s16x2 DPX instructions; pack 4 (byte SIMD) is emulated on sm_100a (profiles/r1_study_packed_simd_sass.md) "
                            "and is listed because north_star names it"}
        roof_smem = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                     "traffic": _smem_traffic(args),
                     "kernel": "SMEM stage: smem_fwd1_kernel + smem_bwd_kernel + smem_fwd2_kernel + smem_bwd_kernel (+ smem_pass3_kernel on a side stream)",
                     "note": "algorithmic bytes = 128 B (two 64-B Occ checkpoints) x interval extensions counted by the kernels; peak = "
                             + ("MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback of B200_PROFILING.md")
                             + "; traffic = DRAM read+write bytes of those kernels per step from profiles/ (ncu), null when the workload differs",
                     "extensions_per_read": cnt["n_ext"] / n, "kernel_ms": smem_ms,
                     "random_64B_gather_gbs_by_span_and_mlp": gather_by_span}
        timed_how = ("one extra pass of the same batch, unsplit (stage timed alone, CUDA events inside the library)" if args.sub_batches > 1
                     else "timed steps")
        roof_bsw["timed"] = roof_smem["timed"] = timed_how
        dominant = "bsw" if bsw_ms >= smem_ms else "smem"
        out = {"metric": METRIC, "value": value,
               "unit": "reads/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64/int16", "data": "synthetic",
               "config": pipeline_config(args),          # the same object in the reference arm's line
               "config_detail": {"index_files": index_how, "l2": "256 MB flush between steps; FM-index %d MB" % (index.desc.reference_seq_len // 64 * 64 // 1_000_000),
                                 "sub_batches_in_flight": args.sub_batches, "regs_per_step": int(n_regs)},
               "e2e": {"value": world * n / e2e_s, "unit": "reads/s", "h2d_bytes_per_step": int(codes.nbytes + offs.nbytes),
                       "d2h_bytes_per_step": int(n_out * capi.REG_DT.itemsize + offs.nbytes)},
               # our own kernels per step and sub-batch (profiles/r1n_kernel_traffic_3gbp.md: 115 launches, 48 of them cub sort/scan)
               "gpu_launches": 67 * args.steps * max(1, args.sub_batches),
               "roofline": dict(roof_bsw if dominant == "bsw" else roof_smem, dominant_stage=dominant),
               "roofline_bsw": roof_bsw, "roofline_smem": roof_smem,
               "stages_ms": {k: round(v, 3) for k, v in stage_acc.items()},
               "stages_ms_sum_over_sub_batches_in_timed_steps": {k: round(v, 3) for k, v in stage_split.items()},
               "bsw": {"gcups": gcells, "cells_per_step": int(cnt["cells"]),
                       "retry_left": int(cnt["retry_left"]), "retry_right": int(cnt["retry_right"])},
               "parity": {"vs": "unmodified reference (ref_driver regs dump of the CPU arm's run), every field of every alignment region",
                          "reads": 2 * sample_pairs, "regs": n_ref_regs, "identical": True,
                          "also": f"first {ns} reads against the oracle; sub-batch path == unsplit path on {nsb} reads"},
               "cpu_baseline": {"value": cpu_v, "unit": "reads/s", "cores": nt, "kind": "reference",
                                "sample": f"first {2 * sample_pairs} reads of the same workload, worker_bwt+worker_aln of the unmodified reference "
                                          f"({_isa()}), {nt} threads, one process, mean of {len(cpu_vals)} repetitions after 1 warm-up",
                                "per_repetition": [round(v, 1) for v in cpu_vals], "host": hi},
               "clocks": clocks, "wall_s": wall}
        if world > 1:
            out["sharding"] = {"how": "bwa_mem2_b200.shard.ShardedAligner: one stream of N x %d reads, chunk c (= %d reads, -K %d) to rank c %% N; "
                                      "different reads per rank; index read once on rank 0 and broadcast over NCCL (bm2_create_resident); results stay in "
                                      "each rank's pinned buffers, the e2e region includes the chunk-table all_gather" % (n, n, n * reads.shape[1]),
                               "startup_s_rank0": startup}
    if sa is not None:
        sa.close()
    else:
        ctx.close(); index.close()
    return out


def run_cigar(args, rank, world):
    """Seam 3 (SURVEY 8f item 2, the first widening step): CIGAR / NM / MD of the final alignment regions of a slice of the
    default workload through bm2_gen_cigar (host requests in, host results out), next to the reference's own bwa_gen_cigar2
    (ref_driver cigar, one host thread) on a sample of the same requests.  Not the headline line: `--workload cigar`."""
    import torch
    pkg = load_package(); capi = pkg.capi
    import oracle_lib as ol, cigar_util as cu
    dev = int(os.environ.get("LOCAL_RANK", 0)); torch.cuda.set_device(dev)
    work = os.path.join(tempfile.gettempdir(), f"bm2_bench_pipe_{args.ref_mbp}_{args.pairs}")
    fa = prepare_pipeline_inputs(work, args.ref_mbp * 1_000_000, args.pairs, seed=21)
    reads = np.load(os.path.join(work, "reads.npy"))[:min(2 * args.pairs, 200_000)]
    n, L = reads.shape
    codes = np.ascontiguousarray(reads.reshape(-1)); offs = np.arange(n + 1, dtype=np.int64) * L
    index = capi.Index(fa); ctx = capi.Context(dev, index=index)
    regs, ro = ctx.seed_chain_extend(codes, offs)
    rd = np.searchsorted(ro, np.arange(len(regs)), side="right") - 1
    reqs = np.zeros(len(regs), capi.CIGAR_REQ_DT)
    reqs["rb"] = regs["rb"]; reqs["re"] = regs["re"]; reqs["read"] = rd; reqs["qb"] = regs["qb"]; reqs["qe"] = regs["qe"]
    reqs["w"] = np.minimum(np.maximum(regs["w"], 1), 4 * ctx.opt.w)
    ns = min(len(reqs), 20_000)
    got = ctx.gen_cigar(codes, offs, reqs[:ns]); want = ol.gen_cigar(index, ctx.opt, codes, offs, reqs[:ns])
    assert want[3] == 0 and cu.same(got, want[:3]) == [], "bm2_gen_cigar differs from the oracle on the bench workload"
    for _ in range(max(1, args.warmup)):
        ctx.gen_cigar(codes, offs, reqs)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        recs, ops, md = ctx.gen_cigar(codes, offs, reqs)
    dt = (time.perf_counter() - t0) / args.steps
    sample = reqs[:min(len(reqs), 100_000)]
    t0 = time.perf_counter(); cu.reference_gen_cigar(capi, fa, codes, offs, sample[:1]); t_load = time.perf_counter() - t0     # index load + process start
    t0 = time.perf_counter(); cu.reference_gen_cigar(capi, fa, codes, offs, sample); t_ref = max(time.perf_counter() - t0 - t_load, 1e-6)
    out = {"metric": "alignments/s through bwa_gen_cigar2's replacement (CIGAR + NM + MD, seam 3)", "value": len(reqs) / dt, "unit": "alignments/s",
           "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "int32", "data": "synthetic",
           "config": {"workload": f"final alignment regions of {n} reads of the default workload ({len(reqs)} requests per step, {args.ref_mbp} Mbp reference), "
                                  "host requests in / host CIGAR, NM, MD out (timed end to end, wall clock)",
                      "mean_ops": float(recs["n_cigar"].mean()), "with_indels": int((recs["n_cigar"] > 1).sum())},
           "e2e": {"value": len(reqs) / dt, "unit": "alignments/s", "h2d_bytes_per_step": int(codes.nbytes + offs.nbytes + reqs.nbytes),
                   "d2h_bytes_per_step": int(recs.nbytes + ops.nbytes + md.nbytes)},
           "gpu_launches": 4 * args.steps,            # cigar_kernel + two scans + gather per call
           "cpu_baseline": {"value": len(sample) / t_ref, "unit": "alignments/s", "cores": 1, "kind": "reference",
                            "sample": f"the reference's bwa_gen_cigar2 (ref_driver cigar) on the first {len(sample)} requests, one host thread, index load subtracted"}}
    ctx.close(); index.close()
    return out


def run_sam(args, rank, world):
    """Seam 4 (SURVEY 8f items 1-3): mate rescue, pairing, MAPQ, CIGAR / NM / MD and the SAM records of a slice of the default workload
    through bm2_sam_pe (host regs in, host records out), checked against the oracle on its first pairs; the oracle's restatement of
    mem_sam_pe timed beside it on one host thread.  Not the headline line: `--workload sam`.  (Added at the end of round 1: first
    timing is round 2's.)"""
    import torch
    pkg = load_package(); capi = pkg.capi
    import oracle_lib as ol, test_oracle_sam_pe as tp
    dev = int(os.environ.get("LOCAL_RANK", 0)); torch.cuda.set_device(dev)
    work = os.path.join(tempfile.gettempdir(), f"bm2_bench_pipe_{args.ref_mbp}_{args.pairs}")
    fa = prepare_pipeline_inputs(work, args.ref_mbp * 1_000_000, args.pairs, seed=21)
    reads = np.load(os.path.join(work, "reads.npy"))[:min(2 * args.pairs, 200_000)]
    n, L = reads.shape
    codes = np.ascontiguousarray(reads.reshape(-1)); offs = np.arange(n + 1, dtype=np.int64) * L
    index = capi.Index(fa)
    opt = capi.default_opt(); opt.flag |= 0x2
    ctx = capi.Context(dev, index=index, opt=opt)
    regs, ro = ctx.seed_chain_extend(codes, offs)
    pes = capi.pestat(opt, index.desc.l_pac, regs, ro)
    lh = np.array([v for d in range(4) for v in (pes[d]["low"], pes[d]["high"], pes[d]["failed"])], np.int32)
    as_ = np.array([v for d in range(4) for v in (pes[d]["avg"], pes[d]["std"])], np.float64)
    ns = min(n, 8000)                                             # parity on the first pairs (same statistics)
    names = [l.split()[1] for i, l in enumerate(open(fa + ".ann")) if i % 2 == 1]
    got = ctx.sam_pe(codes[:offs[ns]], offs[:ns + 1], regs[:ro[ns]], ro[:ns + 1], pes)
    t0 = time.perf_counter()
    want = tp.oracle_sam_pe(capi, index, opt, codes[:offs[ns]], offs[:ns + 1], regs[:ro[ns]], ro[:ns + 1], lh, as_)
    t_cpu = time.perf_counter() - t0
    assert tp.fields(got[0], got[2], got[3], names) == tp.fields(*want, names), "bm2_sam_pe differs from the oracle on the bench workload"
    def timed(staged):
        ctx.set_sam_staged(staged)
        for _ in range(max(1, args.warmup)):
            ctx.sam_pe(codes, offs, regs, ro, pes)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            res = ctx.sam_pe(codes, offs, regs, ro, pes)
        return (time.perf_counter() - t0) / args.steps, res, ctx.last_sam_stats()
    dt, (recs, xa, ops, md), st_default = timed(0)
    # the staged rescue (the windows of all pairs aligned as one batch; mode 1: one window per warp, mode 2: one window per thread): same bytes,
    # its own time and stage split
    staged = {}
    for mode, name in ((1, "warp_per_window"), (2, "thread_per_window")):
        try:
            dt_s, res_s, st_staged = timed(mode)
            same = all(x.tobytes() == y.tobytes() for x, y in zip((recs, xa, ops, md), res_s))
            staged[name] = {"ms_per_step": dt_s * 1e3, "reads_per_s": n / dt_s, "identical_to_default": bool(same), "stats_last_step": st_staged}     # parity gate: tests/test_zzz_sam_staged_gpu.py
        except Exception as e:                               # the staged kernels are new: report, keep the default mode's line
            staged[name] = {"error": str(e)[:300]}
            break                                            # a device fault is sticky: no further launches in this process
    ctx.set_sam_staged(0)
    out = {"metric": "paired 151bp reads/s through mem_sam_pe's replacement (mate rescue, pairing, MAPQ, CIGAR, SAM records; seam 4)", "value": n / dt,
           "unit": "reads/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "int32/f64", "data": "synthetic",
           "config": {"workload": f"{n} reads ({n // 2} pairs) of the default workload with their {len(regs)} alignment regions, {args.ref_mbp} Mbp reference; "
                                  "host regs in / host records, XA entries, CIGAR, MD out (timed end to end, wall clock)",
                      "records": int(len(recs)), "xa_entries": int(len(xa))},
           "stats_last_step": st_default, "staged_rescue": staged,
           "e2e": {"value": n / dt, "unit": "reads/s", "h2d_bytes_per_step": int(codes.nbytes + offs.nbytes + regs.nbytes + ro.nbytes),
                   "d2h_bytes_per_step": int(recs.nbytes + xa.nbytes + ops.nbytes + md.nbytes)},
           "gpu_launches": 2 * st_default["waves"] * args.steps,
           "cpu_baseline": {"value": ns / t_cpu, "unit": "reads/s", "cores": 1, "kind": "port",
                            "sample": f"the oracle's mem_sam_pe restatement on the first {ns} reads, one host thread"}}
    ctx.close(); index.close()
    return out


def prepare_longread_inputs(work, index, n_reads, read_len, seed=31):
    """config 5 reads (10 kbp, 4 % substitutions, 3 % insertions, 3 % deletions) drawn from the bench genome on the GPU; cached in `work`."""
    import ctypes as C
    f = os.path.join(work, f"long_{n_reads}_{read_len}.npy")
    if not os.path.exists(f):
        import torch
        load_package()
        from bwa_mem2_b200 import synth
        l_pac = int(index.desc.l_pac); ns = int(index.desc.n_seqs)
        ref = np.ctypeslib.as_array(C.cast(index.desc.ref_string, C.POINTER(C.c_uint8)), shape=(l_pac,))
        lens = np.ctypeslib.as_array(C.cast(index.desc.ann_len, C.POINTER(C.c_int32)), shape=(ns,)).astype(np.int64)
        genome = torch.from_numpy(ref.copy())
        if torch.cuda.is_available():
            genome = genome.cuda()
        reads = synth.make_long_reads_torch(genome, lens, n_reads, read_len, seed=seed)
        del genome
        if torch.cuda.is_available():
            torch.cuda.empty_cache()
        synth.write_fastq_fast(os.path.join(work, f"long_{n_reads}_{read_len}.fq"), reads, prefix=b"l")
        np.save(f, reads)
    return np.load(f)


ONT2D_ARGS = ["-x", "ont2d"]


def reference_longread(work, fa, n_reads, read_len, n_sample, threads, steps=1, warmup=0, dump_regs=None):
    """reads/s of the unmodified reference's worker_bwt + worker_aln with -x ont2d on the first n_sample long reads (one process)."""
    src = os.path.join(work, f"long_{n_reads}_{read_len}.fq"); dst = os.path.join(work, f"long_{n_reads}_{read_len}_s{n_sample}.fq")
    if not os.path.exists(dst):
        rec = os.path.getsize(src) // n_reads
        with open(src, "rb") as f, open(dst, "wb") as o:
            o.write(f.read(rec * n_sample))
    stats = os.path.join(work, "stats_ref_long.json")
    env = dict(os.environ, BM2_MODE="hotpath", BM2_STATS=stats, BM2_REPEAT=str(warmup + steps))
    if dump_regs:
        env["BM2_DUMP_REGS"] = dump_regs
    subprocess.check_call([_refbin("ref_driver"), "mem"] + ONT2D_ARGS + ["-t", str(threads), "-K", "2000000000", fa, dst],
                          stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, env=env)
    st = json.load(open(stats))
    reps = st.get("rep_s") or [st["t_bwt"] + st["t_aln"]]
    vals = [st["reads"] / t for t in reps[warmup:]]
    return float(np.mean(vals)), vals, st


METRIC_LONG = "10 kbp reads/s (seed+chain+extend hot path, -x ont2d; config 5)"


def run_longread(args, rank, world):
    """BASELINE.json config 5: single-end 10 kbp reads with the ont2d preset (k14 W20 r10 A1 B1 O1 E1 L0, src/fastmap.cpp:812-826)
    against the ~3 Gbp bench genome: mem_flt_chained_seeds (seed SW), wide-band extensions (bsw_warp_kernel), doubled-band retries.
    reads/s device-timed and end to end, GCUPS of the extension stage, the reference beside it, parity against the reference's regs."""
    import torch
    pkg = load_package(); capi = pkg.capi
    import longread_util as lu
    dev = int(os.environ.get("LOCAL_RANK", 0)); torch.cuda.set_device(dev)
    work = os.path.join(tempfile.gettempdir(), f"bm2_bench_pipe_{args.ref_mbp}_{args.pairs}")
    fa = prepare_pipeline_inputs(work, args.ref_mbp * 1_000_000, args.pairs, seed=21)
    index = capi.Index(fa)
    n, L = args.long_reads, args.long_len
    reads = prepare_longread_inputs(work, index, n, L)
    codes = np.ascontiguousarray(reads.reshape(-1)); offs = np.arange(n + 1, dtype=np.int64) * L
    opt = lu.ont2d_opt(capi)
    ctx = capi.Context(dev, index=index, opt=opt)
    int_gops = ctx.int_pipe_gops()
    stream = torch.cuda.current_stream(); ctx.set_stream(stream.cuda_stream)
    d_codes = torch.from_numpy(codes).cuda(); d_offs = torch.from_numpy(offs).cuda()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    for _ in range(max(1, args.warmup)):
        ctx.seed_chain_extend_resident(codes, offs, d_codes.data_ptr(), d_offs.data_ptr(), False)
    torch.cuda.synchronize()
    sampler = ClockSampler(dev); sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    stage_acc = {}
    t0 = time.perf_counter()
    for a, b in evs:
        flush.fill_(1)
        a.record(stream)
        n_regs = ctx.seed_chain_extend_resident(codes, offs, d_codes.data_ptr(), d_offs.data_ptr(), False)
        b.record(stream)
        for k, v in ctx.stage_ms().items():
            stage_acc[k] = stage_acc.get(k, 0.0) + v / args.steps
        cnt = ctx.counters()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    ms_step = float(np.mean([a.elapsed_time(b) for a, b in evs]))
    ctx.set_stream(None)
    h_codes = torch.from_numpy(codes.copy()).pin_memory(); h_offs = torch.from_numpy(offs.copy()).pin_memory()
    regs, ro = ctx.seed_chain_extend(h_codes.numpy(), h_offs.numpy(), copy=False)
    t0 = time.perf_counter()
    e2e_steps = max(1, min(args.steps, 2))
    for _ in range(e2e_steps):
        regs, ro = ctx.seed_chain_extend(h_codes.numpy(), h_offs.numpy(), copy=False)
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    hi = host_info(); nt = hi["threads_used"]
    ns = min(n, args.long_sample)
    busy = min(nt, (ns + 511) // 512)        # kt_for hands out blocks of 512 reads (BATCH_SIZE, src/macro.h:48): threads that get work
    dump = os.path.join(work, "ref_regs_long.bin")
    cpu_v, cpu_vals, _ = reference_longread(work, fa, n, L, ns, nt, steps=1, warmup=0, dump_regs=dump)
    n_ref_regs = check_against_reference_dump(regs, ro, dump, ns)
    os.remove(dump)
    bsw_ms = stage_acc.get("bsw_left", 0.0) + stage_acc.get("bsw_right", 0.0)
    gcells = cnt["cells"] / (bsw_ms * 1e-3) / 1e9 if bsw_ms > 0 else 0.0
    ceil = {"pack1_s32": int_gops / 14.0, "pack2_s16x2": 2 * int_gops / 14.0}
    out = {"metric": METRIC_LONG, "value": n / (ms_step * 1e-3), "unit": "reads/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64/int32", "data": "synthetic",
           "config": {"workload": f"config[4]: {n} single-end reads of {L} bp per step (4% subs, 3% ins, 3% del), -x ont2d, vs {args.ref_mbp} Mbp synthetic reference",
                      "l2": "256 MB flush between steps", "regs_per_step": int(n_regs)},
           "e2e": {"value": n / e2e_s, "unit": "reads/s", "h2d_bytes_per_step": int(codes.nbytes + offs.nbytes),
                   "d2h_bytes_per_step": int(len(regs) * capi.REG_DT.itemsize + offs.nbytes)},
           "gpu_launches": 80 * args.steps,
           "roofline": {"bound": "int_alu", "achieved": gcells, "peak": ceil["pack1_s32"], "unit": "Gcell/s", "frac": gcells / ceil["pack1_s32"] if int_gops else None,
                        "traffic": None, "kernel": "extension stage (bsw_warp_kernel: one job per warp, 32-bit cells)", "kernel_ms": bsw_ms,
                        "ceilings_gcell_s": {k: round(v, 1) for k, v in ceil.items()}},
           "stages_ms": {k: round(v, 3) for k, v in stage_acc.items()},
           "bsw": {"gcups": gcells, "cells_per_step": int(cnt["cells"]), "retry_left": int(cnt["retry_left"]), "retry_right": int(cnt["retry_right"])},
           "parity": {"vs": "unmodified reference (ref_driver regs dump, -x ont2d), every field of every alignment region", "reads": ns, "regs": n_ref_regs,
                      "identical": True},
           "cpu_baseline": {"value": cpu_v, "unit": "reads/s", "cores": nt, "kind": "reference",
                            "sample": f"first {ns} reads, worker_bwt+worker_aln of the unmodified reference ({_isa()}, -x ont2d), {nt} threads of which "
                                      f"{busy} get work (kt_for deals blocks of 512 reads), one repetition",
                            "threads_with_work": busy, "host": hi},
           "clocks": clocks, "wall_s": wall}
    ctx.close(); index.close()
    return out


def run_reference_longread(args, rank, world):
    if rank != 0:
        return None
    pkg = load_package(); capi = pkg.capi
    work = os.path.join(tempfile.gettempdir(), f"bm2_bench_pipe_{args.ref_mbp}_{args.pairs}")
    fa = prepare_pipeline_inputs(work, args.ref_mbp * 1_000_000, args.pairs, seed=21)
    index = capi.Index(fa)
    prepare_longread_inputs(work, index, args.long_reads, args.long_len)
    index.close()
    hi = host_info(); nt = hi["threads_used"]
    ns = min(args.long_reads, args.long_sample)
    v, vals, st = reference_longread(work, fa, args.long_reads, args.long_len, ns, nt, steps=args.steps, warmup=args.warmup)
    return {"impl": "reference", "metric": METRIC_LONG, "value": v, "unit": "reads/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * ns / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64/int32", "data": "synthetic",
            "config": {"workload": f"config[4]: first {ns} of {args.long_reads} single-end reads of {args.long_len} bp per step, -x ont2d, unmodified reference ({_isa()}), {nt} threads"},
            "cpu_baseline": {"value": v, "unit": "reads/s", "cores": nt, "kind": "reference", "sample": f"{ns} reads per step", "host": hi,
                             "per_repetition": [round(x, 2) for x in vals]},
            "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


METRIC_SAM = "paired 151bp reads/s, FASTQ bytes in -> SAM text out (parse+encode, seed+chain+extend, pestat, SAM stage, formatting)"


def reference_mem_full(work, fa, n_pairs_sample, threads, sam_out):
    """The unmodified reference's whole mem path on the first pairs of the bench reads (ref_driver BM2_MODE=ref = bwa-mem2 mem with the phase
    timers): reads/s over worker_bwt + worker_aln + worker_sam (FASTQ parsing, mem_pestat and the SAM write are NOT in its time)."""
    r1 = os.path.join(work, "r1.fq"); r2 = os.path.join(work, "r2.fq")
    s1 = os.path.join(work, f"s1_{n_pairs_sample}.fq"); s2 = os.path.join(work, f"s2_{n_pairs_sample}.fq")
    if not os.path.exists(s1):
        rec = os.path.getsize(r1) // (np.load(os.path.join(work, "reads.npy"), mmap_mode="r").shape[0] // 2)
        for src, dst in ((r1, s1), (r2, s2)):
            with open(src, "rb") as f, open(dst, "wb") as o:
                o.write(f.read(rec * n_pairs_sample))
    stats = os.path.join(work, "stats_ref_full.json")
    env = dict(os.environ, BM2_MODE="ref", BM2_STATS=stats)
    with open(sam_out, "w") as f:
        subprocess.check_call([_refbin("ref_driver"), "mem", "-t", str(threads), "-K", "1000000000", fa, s1, s2], stdout=f, stderr=subprocess.DEVNULL, env=env)
    st = json.load(open(stats))
    return st["reads"] / (st["t_bwt"] + st["t_aln"] + st["t_sam"]), st, s1, s2


def run_fastq2sam(args, rank, world):
    """SURVEY 8f item 3 end to end: the raw bytes of two FASTQ files in host memory -> SAM text in host memory, through the C ABI:
    bm2_fastq_encode (parse + encode on the GPU), bm2_seed_chain_extend_resident, bm2_pestat, bm2_sam_pe (staged rescue), bm2_sam_format
    (host threads).  One chunk per step (the sample), wall clock.  Beside it the unmodified reference's mem on the same files and threads;
    the two SAM texts must be byte-identical (header lines aside)."""
    import torch
    pkg = load_package(); capi = pkg.capi
    dev = int(os.environ.get("LOCAL_RANK", 0)); torch.cuda.set_device(dev)
    work = os.path.join(tempfile.gettempdir(), f"bm2_bench_pipe_{args.ref_mbp}_{args.pairs}")
    fa = prepare_pipeline_inputs(work, args.ref_mbp * 1_000_000, args.pairs, seed=21)
    hi = host_info(); nt = hi["threads_used"]
    sample_pairs = min(args.pairs, args.sam_pairs)
    ref_sam = os.path.join(work, "ref_full.sam")
    cpu_v, cpu_st, s1, s2 = reference_mem_full(work, fa, sample_pairs, nt, ref_sam)
    b1 = open(s1, "rb").read(); b2 = open(s2, "rb").read()
    index = capi.Index(fa)
    contigs = [l.split()[1] for i, l in enumerate(open(fa + ".ann")) if i % 2 == 1]
    opt = capi.default_opt(); opt.flag |= 0x2
    ctx = capi.Context(dev, index=index, opt=opt)
    ctx.set_sam_staged(1)

    def step():
        t = [time.perf_counter()]
        fq = ctx.fastq_encode(b1, b2); t.append(time.perf_counter())
        regs, ro = ctx.seed_chain_extend_resident(fq["codes"], fq["offsets"], fq["d_codes"], fq["d_offsets"], True, return_arrays=True); t.append(time.perf_counter())
        pes = capi.pestat(opt, index.desc.l_pac, regs, ro); t.append(time.perf_counter())
        recs, xa, cig, md = ctx.sam_pe(fq["codes"], fq["offsets"], regs, ro, pes); t.append(time.perf_counter())
        text = capi.sam_format(recs, xa, cig, md, fq["codes"], fq["offsets"], contigs, read_names=fq["names"], quals=fq["quals"], n_threads=nt); t.append(time.perf_counter())
        return text, np.diff(t), fq["n_reads"]

    for _ in range(max(1, args.warmup)):
        text, _, n = step()
    want = b"".join(ln for ln in open(ref_sam, "rb") if not ln.startswith(b"@"))
    if text != want:
        a_ = text.split(b"\n"); b_ = want.split(b"\n")
        bad = [i for i in range(min(len(a_), len(b_))) if a_[i] != b_[i]][:3]
        raise AssertionError(f"FASTQ -> SAM text differs from the unmodified reference: {len(a_)} vs {len(b_)} lines, first differing {[(a_[i][:200], b_[i][:200]) for i in bad]}")
    # ... and the same through the C++ host program over the C ABI (bwa-mem2_b200/bm2_mem: no python in the loop) on the WHOLE read files,
    # cut by -K into chunks of the sample's size: the first chunk pays the process's allocations, the later ones are the steady state
    tool = os.path.join(ROOT, "bwa-mem2_b200", "bm2_mem")
    tool_out = os.path.join(work, "bm2_mem.sam")
    ctx.close(); ctx = None                       # (one context at a time on the GPU: the program uploads the index itself)
    reads_all = np.load(os.path.join(work, "reads.npy"), mmap_mode="r")
    L_read = int(reads_all.shape[1])
    k_bases = 2 * sample_pairs * L_read
    r1_all = os.path.join(work, "r1.fq"); r2_all = os.path.join(work, "r2.fq")
    import hashlib
    tool_stats = []; digests = []
    for workers in (1, 2):                        # one chunk at a time / two chunks in flight (two contexts, one index: bm2_create_sibling)
        pr = subprocess.run([tool, "-t", str(nt), "-K", str(k_bases), "-p", str(workers), "-o", tool_out, fa, r1_all, r2_all], capture_output=True, text=True, check=True)
        tool_stats.append(json.loads(pr.stderr.strip().splitlines()[-1]))
        h = hashlib.sha256()
        with open(tool_out, "rb") as f:
            got_tool = b"".join(ln for _, ln in zip(range(len(want.splitlines()) + 64), f) if not ln.startswith(b"@"))
        with open(tool_out, "rb") as f:
            for ln in f:
                if not ln.startswith(b"@PG"):
                    h.update(ln)
        digests.append(h.hexdigest())
        assert got_tool[:len(want)] == want, "bm2_mem's SAM (first chunk) differs from the unmodified reference"
        os.remove(tool_out)
    assert digests[0] == digests[1], "bm2_mem -p 2 wrote a different SAM file than -p 1"
    os.remove(ref_sam)
    ts = tool_stats[-1]
    ctx = capi.Context(dev, index=index, opt=opt); ctx.set_sam_staged(1)
    step()
    torch.cuda.synchronize()
    acc = np.zeros(5); t0 = time.perf_counter()
    for _ in range(args.steps):
        text, dt, n = step(); acc += dt
    wall = (time.perf_counter() - t0) / args.steps
    acc /= args.steps
    wall_py = wall; n_py = n
    ts1 = tool_stats[0]
    serial_rps = (ts1["reads"] - ts1["chunk_reads"][0]) / (ts1["loop_s"] - ts1["chunk_s"][0])      # one chunk at a time: the loop after its first chunk
    # two chunks in flight: completions in the steady state = from the moment the 2nd chunk is written (both workers past their first,
    # allocating, chunk) to the end of the loop
    assert ts["chunks"] >= 4, "the read files give fewer than 4 chunks"
    steady_reads = sum(ts["chunk_reads"][2:]); steady_s = ts["chunk_done_s"][-1] - ts["chunk_done_s"][1]
    n = steady_reads; wall = steady_s            # the headline of this workload: the C++ program's chunk loop in its steady state
    out = {"metric": METRIC_SAM, "value": n / wall, "unit": "reads/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall * 1e3,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64/int16/f64", "data": "synthetic",
           "config": {"workload": f"chunks of {2 * sample_pairs} reads ({sample_pairs} pairs) of the default workload as FASTQ bytes ({len(b1) + len(b2)} B per chunk) -> {len(text)} B of SAM text per chunk, "
                                  f"{args.ref_mbp} Mbp reference; one chunk per step, wall clock; python binding overheads (array copies, name list) included"},
           "how": "bwa-mem2_b200/bm2_mem (C++ over the C ABI) on the whole read files (%d reads, %d chunks of -K %d bases): FASTQ files already read into "
                  "host memory -> SAM bytes written to a file; two chunks in flight (-p 2: two contexts on one index, output in chunk order); the clock runs from "
                  "the completion of the 2nd chunk to the end (parse+encode, align, pestat, SAM stage, format, fwrite of the chunks after it); whole loop %.3f s; "
                  "the same files with one chunk at a time (-p 1) and the identical SAM file: see one_chunk_at_a_time" % (ts["reads"], ts["chunks"], k_bases, ts["loop_s"]),
           "chunk_s": ts["chunk_s"], "chunk_done_s": ts["chunk_done_s"],
           "one_chunk_at_a_time": {"reads_per_s": serial_rps, "loop_s": ts1["loop_s"], "chunk_s": ts1["chunk_s"],
                                   "stage_s": {k: ts1[k] for k in ("fastq_encode_s", "seed_chain_extend_s", "pestat_s", "sam_stage_s", "sam_format_s", "write_s")}},
           "stage_s": {k: ts[k] for k in ("fastq_encode_s", "seed_chain_extend_s", "pestat_s", "sam_stage_s", "sam_format_s", "wait_for_turn_s", "write_s")},
           "through_the_python_binding": {"reads_per_s": n_py / wall_py, "stage_s": dict(zip(["fastq_encode", "seed_chain_extend", "pestat", "sam_pe_staged", "sam_format"],
                                                                                      [round(float(x), 4) for x in acc]))},
           "e2e": {"value": n / wall, "unit": "reads/s", "h2d_bytes_per_step": int(len(b1) + len(b2)), "d2h_bytes_per_step": int(len(text))},
           "gpu_launches": 80 * args.steps,
           "parity": {"vs": "SAM text of the unmodified reference (bwa-mem2 mem through ref_driver) on the same FASTQ files", "lines": int(text.count(b"\n")),
                      "identical": True},
           "cpu_baseline": {"value": cpu_v, "unit": "reads/s", "cores": nt, "kind": "reference",
                            "sample": f"the same {n} reads, worker_bwt + worker_aln + worker_sam of the unmodified reference ({_isa()}), {nt} threads "
                                      "(its FASTQ parsing, mem_pestat and SAM write are not in its time)", "host": hi}}
    ctx.close(); index.close()
    return out


def pipeline_config(args):
    """`config` of the default workload, identical in both arms' lines (the driver compares them)."""
    return {"workload": f"config[2]-like: seed+chain+extend hot path (SMEM, SA lookup, chaining, BSW, post-filter), {2 * args.pairs} reads/step/GPU "
                        f"(2x151 bp pairs, 1% subs, 25% reads with an indel, 1% garbage) vs {args.ref_mbp} Mbp synthetic reference (planted repeat families), "
                        "L2 flushed between steps (256 MB)"}


def run_reference_pipeline(args, rank, world):
    """--impl reference: the unmodified reference's worker_bwt + worker_aln on the host cores, same metric / config as our arm.
    Each step = the first `sample` pairs of the same 1 M-read workload (bounded: the whole run ends within minutes); one process,
    one index load, warmup + steps repetitions timed one by one inside it."""
    if rank != 0:
        return None
    work = os.path.join(tempfile.gettempdir(), f"bm2_bench_pipe_{args.ref_mbp}_{args.pairs}")
    fa = prepare_pipeline_inputs(work, args.ref_mbp * 1_000_000, args.pairs, seed=21)
    hi = host_info()
    nt = hi["threads_used"]
    sample_pairs = min(args.pairs, 100_000)
    v, vals, st = reference_hotpath(work, fa, sample_pairs, nt, steps=args.steps, warmup=args.warmup)
    n = 2 * sample_pairs
    return {"impl": "reference", "metric": METRIC, "value": v, "unit": "reads/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * n / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int64/int16", "data": "synthetic",
            "config": pipeline_config(args),            # the GPU arm's config; what this arm ran of it: config_detail / cpu_baseline.sample
            "config_detail": {"how": f"worker_bwt + worker_aln of the unmodified reference ({_isa()}) on the first {n} reads per step of that workload "
                                     f"(bounded sample), {nt} threads, same index files"},
            "cpu_baseline": {"value": v, "unit": "reads/s", "cores": nt, "kind": "reference",
                             "sample": f"{n} reads per step, kt_for over {nt} threads, one process, {len(vals)} timed repetitions",
                             "per_repetition": [round(x, 1) for x in vals], "host": hi},
            "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def run_reference(args, rank, world):
    """The reference's own CPU implementation of the path, all host threads, bounded sample."""
    if rank != 0:
        return None
    work = os.path.join(tempfile.gettempdir(), f"bm2_bench_ref_{args.ref_mbp}_{args.pairs}")
    fa = prepare_inputs(work, args.ref_mbp * 1_000_000, args.pairs, seed=11)
    nt = host_threads()
    vals = []
    for i in range(args.warmup + args.steps):
        stats = os.path.join(work, f"stats_ref.json")
        env = dict(os.environ, BM2_MODE="hotpath", BM2_STATS=stats)
        subprocess.check_call([_refbin("ref_driver"), "mem", "-t", str(nt), "-K", "100000000", fa, os.path.join(work, "r1.fq"),
                               os.path.join(work, "r2.fq")], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, env=env)
        st = json.load(open(stats))
        if i >= args.warmup:
            vals.append(st["reads"] / (st["t_bwt"] + st["t_aln"]))
    v = float(np.mean(vals))
    return {"impl": "reference", "metric": METRIC_BSW, "value": v, "unit": "reads/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * 2 * args.pairs / v, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int16", "data": "synthetic",
            "config": {"workload": f"worker_bwt + worker_aln of the unmodified reference ({_isa()}) on {2 * args.pairs} synthetic 2x151 reads "
                                   f"vs {args.ref_mbp} Mbp synthetic reference"},
            "cpu_baseline": {"value": v, "unit": "reads/s", "cores": nt, "kind": "reference",
                             "sample": f"{2 * args.pairs} reads per step, kt_for over {nt} threads"},
            "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="pipeline", choices=["bsw", "pipeline", "cigar", "sam", "longread", "fastq2sam"])
    ap.add_argument("--sam-pairs", type=int, default=100_000, help="--workload fastq2sam: pairs per chunk")
    ap.add_argument("--long-reads", type=int, default=2048, help="--workload longread: reads per step")
    ap.add_argument("--long-len", type=int, default=10000)
    ap.add_argument("--long-sample", type=int, default=2048, help="--workload longread: reads of the CPU arm / parity check (512 per busy thread)")
    ap.add_argument("--ref-mbp", type=int, default=3000)
    ap.add_argument("--pairs", type=int, default=500_000)
    ap.add_argument("--bsw-jobs", type=int, default=4_000_000)
    ap.add_argument("--sub-batches", type=int, default=4, help="sub-batches in flight per GPU (bm2_set_sub_batches); 1 = unsplit")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the regions of the timed path (default workload) as DIR/*.npy; see dump_pipeline_outputs")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.workload != "pipeline" or args.impl != "ours"):
        ap.error("--dump-outputs is implemented for --workload pipeline --impl ours")
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        out = (run_reference_pipeline(args, rank, world) if args.workload == "pipeline" else
               run_reference_longread(args, rank, world) if args.workload == "longread" else run_reference(args, rank, world))
        if rank == 0:
            print(json.dumps(out))
        return
    if world > 1:
        import torch, torch.distributed as dist
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
        dist.init_process_group("nccl")
    runner = {"pipeline": run_pipeline, "cigar": run_cigar, "sam": run_sam, "bsw": run_bsw, "longread": run_longread, "fastq2sam": run_fastq2sam}[args.workload]
    out = runner(args, rank, world)
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        import torch.distributed as dist
        dist.barrier(); dist.destroy_process_group()


if __name__ == "__main__":
    main()
