#!/usr/bin/env python
"""bench.py — mapped reads/s of the `pandora map` hot path (BASELINE.json metric) on N B200s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--reads R] [--impl ours|reference] [--no-extras] [--dump-outputs DIR]

Workload = BASELINE config 3, the configuration the metric ("mapped reads/sec at 1/2/4/8 B200") is quoted on: the
config-2 panel and genome with 30 M simulated 150 bp reads (~1000x panel depth), STRONG-scaled: the same 30 M reads are
read-sharded over the N GPUs (rank r owns sub-shards [240 r/N, 240 (r+1)/N)), the index is replicated.  A step = one pass
of the whole hot path over the sample: sketch -> index lookup -> grouping -> cluster/filter -> k-mer coverage (S1-S5) on
every rank's shard, the coverage of the non-root ranks added straight into the root rank's accumulator over NVLink by the
coverage kernel itself (no collective call; DRPRG_REDUCE=nccl switches to one NCCL allreduce for comparison), then
parameter estimation, ML path, genotyping and the VCF text (S6-S8) on the root rank.
`value` times that with the packed reads already resident in HBM; `e2e` times the same call sequence from pinned HOST
buffers (H2D inside the timed region) down to the VCF text in host memory.  Extra keys (N = 1): `e2e_file` = the
reference-facing plugin call drprg_cuda_map_genotype(reads_path, ...) on a 1 M-read FASTQ (plain and gzip), `config2`,
`config4`, `config5` = the other BASELINE configurations.
`--impl reference` times the CPU oracle (restated pandora algorithm; the reference's pandora binary is not in the
reference tree) on the box's host cores on a bounded sample of the same workload.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np

METRIC = "mapped reads/sec (pandora-map hot path: sketch+lookup+cluster+coverage+ML path+genotype)"
UNIT = "reads/s"
CPU_SAMPLE_SUBSHARDS = 8  # 1 M reads: the bounded sample the CPU arms map


def screen_profile():
    """ncu-derived constants of the sketch+lookup kernels (per million reads), kept with the profile they come from"""
    for name in ("r2_screen4m.json", "r2_screen.json", "r1_screen.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            d = json.load(open(p))
            d["source"] = "profiles/" + name
            return d
    return None


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def workload_config(wl, total_reads):
    """identical in both arms (the driver compares the dicts)"""
    from drprg_b200 import workload
    return {"workload": wl.name, "reads_total": int(total_reads), "read_len": workload.READ_LEN,
            "sharding": "contiguous shards of the reads, one per GPU (strong scaling; even for `value`, sized by each rank's measured upload "
                        "bandwidth for `e2e`), index replicated, genotype step on the root"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, dev):
        self.dev, self.proc, self.lines = dev, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.dev), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
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
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
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
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_sample(wl, device):
    """the bounded CPU sample: the first 1 M reads of the workload (sub-shards 0..7), ASCII on the host"""
    parts = [wl.subshard_ascii(i, device)[0] for i in range(min(CPU_SAMPLE_SUBSHARDS, wl.n_subshards))]
    data = np.concatenate(parts)
    n = len(data) // 150
    return data, np.arange(n + 1, dtype=np.uint64) * np.uint64(150), n


def oracle_step(O, ox, data, off, oo, refs):
    mr = O.MapRun(ox, data, off, oo)
    return O.Genotype(ox, mr, oo, refs).vcf()


def run_reference(args, rank, world):
    """CPU arm: the oracle (restated pandora map) with all host threads on a bounded sample of the same workload."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py as O
    from drprg_b200 import workload
    try:
        import torch
        device = "cuda" if torch.cuda.is_available() else "cpu"  # read generation only: same sub-shards as the GPU arm
    except Exception:
        device = "cpu"
    cores = os.cpu_count() or 1
    wl = workload.Config3(total_reads=args.reads)
    data, off, n = cpu_sample(wl, device)
    ox = O.Index(wl.prg_path, wl.w, wl.k)
    opts = O.make_opts(threads=cores, illumina=True, genome_size=workload.GENOME_SIZE)
    for _ in range(args.warmup):
        oracle_step(O, ox, data, off, opts, wl.refs_path)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        oracle_step(O, ox, data, off, opts, wl.refs_path)
    dt = (time.perf_counter() - t0) / args.steps
    v = n / dt
    sample = (f"each step maps the first {n} reads of the workload (sub-shards 0-{CPU_SAMPLE_SUBSHARDS - 1}) and genotypes them: restated CPU "
              f"oracle on {cores} threads, not the pandora binary (absent from the reference tree)")
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u32 (hash/cluster/coverage), f64 (likelihoods)", "data": f"synthetic (reads generated on {device})",
        "config": workload_config(wl, args.reads),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def strip_file_date(vcf_text):
    """the VCF text without its ##fileDate line, the one line that differs between two runs on the same reads"""
    return b"\n".join(l for l in vcf_text.splitlines() if not l.startswith(b"##fileDate"))


def dump_outputs(out_dir, ix, vcf_text, st):
    """Writes what the last timed step computed as DIR/<name>.npy, so that two builds can be compared output for output:
    the VCF text (byte codes as float32, without ##fileDate: its SHA-1 is the run's `vcf_sha1`), the hit counts of the map
    step (hits, kept hits, bases, reads), the k-mer coverage the genotype step started from, the fitted parameters (in the
    order of lib.Index.params()) and every per-record and per-allele array behind the VCF (float64).  All arrays are sized
    by the panel, not by the reads (~38 k k-mer nodes, ~4.5 k sites, ~5 MB in all), so they are written whole."""
    os.makedirs(out_dir, exist_ok=True)
    cov = ix.coverage()
    out = {"vcf_text": np.frombuffer(strip_file_date(vcf_text), np.uint8).astype(np.float32),
           "map_totals": np.array([st["hits"][-1], st["kept"][-1], cov["total_bases"], cov["n_reads"]], np.float64),
           "coverage_fwd": cov["fwd"], "coverage_rev": cov["rev"], "locus_reads": cov["locus_reads"],
           "gt_params": np.array(list(ix.params().values()), np.float64)}
    out.update({"gt_" + k: v for k, v in ix.gt_records().items()})
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def extras_single_gpu(lib, workload, sim, wl, ix, opts, torch, flush):
    """the other BASELINE configurations and the file-level plugin call, measured on one GPU (bounded: a few seconds)"""
    out = {}

    def timed_steps(fn, steps=8, warmup=2):
        for _ in range(warmup):
            fn()
        ms = []
        for _ in range(steps):
            flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ms.append((time.perf_counter() - t0) * 1e3)
        return float(np.median(ms))

    # ---- config 2: 1 M reads per step, resident
    codes = torch.cat([wl.subshard_codes(i) for i in range(8)])
    n = codes.shape[0]
    words, lens = wl.pack_codes(codes), torch.full((n,), workload.READ_LEN, dtype=torch.int32, device="cuda")
    b = ix.wrap_device(words.data_ptr(), lens.data_ptr(), n, workload.STRIDE_WORDS, n * workload.READ_LEN, keep=(words, lens))

    def step2():
        ix.sample_begin(opts, workload.READ_LEN)
        ix.map_batch(b)
        ix.genotype(wl.refs_path)

    ms = timed_steps(step2)
    out["config2"] = {"workload": "config2: 1 M x 150 bp reads per step, resident in HBM", "ms_per_step": ms, "reads_per_s": n / (ms * 1e-3),
                      "stage_ms": ix.last_timings()}
    # ---- the plugin call on files: drprg_cuda_map_genotype(reads_path, vcf_refs, outdir) = Pandora::genotype_with
    tmp = tempfile.mkdtemp(prefix="drprg_bench_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    data = sim.BASES[codes.cpu().numpy()].reshape(-1)
    off = np.arange(n + 1, dtype=np.uint64) * np.uint64(workload.READ_LEN)
    fo = lib.make_opts(illumina=True, genome_size=workload.GENOME_SIZE, threads=os.cpu_count() or 1)
    e2e_file = {}
    for label, gz in (("plain", False), ("gzip", True)):
        path = os.path.join(tmp, "reads.fq" + (".gz" if gz else ""))
        sim.write_fastq_fast(path, data, off, gz=gz)
        ms = timed_steps(lambda: ix.map_genotype(path, wl.refs_path, tmp, fo), steps=5 if not gz else 3, warmup=1)
        e2e_file[label] = {"ms_per_sample": ms, "reads_per_s": n / (ms * 1e-3), "file_bytes": os.path.getsize(path),
                           "samples_per_hour_per_gpu": 3.6e6 / ms}
    out["e2e_file"] = {"call": "drprg_cuda_map_genotype(reads.fq[.gz], genes.fa, outdir): 1 M reads in, pandora_genotyped.vcf out "
                               "(file read, parse, H2D, S1-S8, VCF write; page cache warm)", **e2e_file}
    # ---- config 3 from a file: the first 10 M reads of the workload as one 3.15 GB FASTQ through the same plugin call (read
    # wave by wave, 1 GiB of text per wave); its VCF must be the one the staged calls give for the same reads in HBM
    try:
        big = os.path.join(tmp, "config3_10M.fq")
        nb = wl.write_fastq(big, n_subshards=80)
        msb = timed_steps(lambda: ix.map_genotype(big, wl.refs_path, tmp, fo), steps=3, warmup=1)
        strip = lambda t: b"\n".join(l for l in t.splitlines() if not l.startswith(b"##fileDate"))
        sha_file = hashlib.sha1(strip(open(os.path.join(tmp, "pandora_genotyped.vcf"), "rb").read())).hexdigest()
        ix.sample_begin(opts, workload.READ_LEN)
        for g0 in range(0, 80, 16):
            w = torch.cat([wl.pack_codes(wl.subshard_codes(i)) for i in range(g0, g0 + 16)])
            l = torch.full((w.shape[0],), workload.READ_LEN, dtype=torch.int32, device="cuda")
            ix.map_batch(ix.wrap_device(w.data_ptr(), l.data_ptr(), w.shape[0], workload.STRIDE_WORDS, w.shape[0] * workload.READ_LEN,
                                        read_id_base=g0 * wl.SUBSHARD, keep=(w, l)))
        ix.genotype(wl.refs_path)
        out["config3_file"] = {"workload": f"the first {nb} reads of config 3 as one plain FASTQ ({os.path.getsize(big) / 1e9:.2f} GB, page cache warm) through "
                                           "drprg_cuda_map_genotype: host-framed ingest wave by wave, S1-S8, VCF written",
                               "ms_per_call": msb, "reads_per_s": nb / (msb * 1e-3), "host_cores": os.cpu_count(),
                               "vcf_equals_resident_run": hashlib.sha1(strip(bytes(ix.vcf_view()))).hexdigest() == sha_file}
        os.remove(big)
    except Exception as e:  # e.g. no room for the 3 GB file: the other extras still count
        out["config3_file"] = {"error": repr(e)}
    # ---- config 5: a batch of samples through drprg_cuda_map_genotype_batch (index resident)
    import ctypes as C
    k = 6
    outs = []
    for s in range(k):
        od = os.path.join(tmp, f"out{s}")
        os.makedirs(od, exist_ok=True)
        outs.append(od.encode())
    arr_r = (C.c_char_p * k)(*[os.path.join(tmp, "reads.fq").encode()] * k)
    arr_o = (C.c_char_p * k)(*outs)
    t0 = time.perf_counter()
    rc = lib.lib().drprg_cuda_map_genotype_batch(ix.h, C.c_size_t(k), arr_r, wl.refs_path.encode(), arr_o, C.byref(fo), None)
    dt = time.perf_counter() - t0
    if rc == 0:
        out["config5"] = {"workload": f"batch of {k} samples x 1 M reads (plain FASTQ files in, VCF files out) on one GPU; sample-sharding over GPUs is replicas only",
                          "ms_per_sample": dt / k * 1e3, "samples_per_hour_per_gpu": 3600.0 * k / dt}
    # ---- config 4: nanopore mode (no -I), ~10 kb reads at 5 % error
    d4, o4 = sim.simulate_long_reads(wl.genome, 3000, mean_len=10_000, sigma=0.3, seed=workload.PANEL_SEED + 3, err=0.05)
    w4, wo4, l4 = lib.pack_reads(d4, o4)
    o4opts = lib.make_opts(illumina=False, genome_size=workload.GENOME_SIZE)
    b4 = ix.upload(w4, wo4, l4, total_bases=int(o4[-1]))

    def step4():
        ix.sample_begin(o4opts, int(o4[1] - o4[0]))
        ix.map_batch(b4)
        ix.genotype(wl.refs_path)

    ms = timed_steps(step4, steps=5, warmup=2)
    out["config4"] = {"workload": "config4: 3 000 simulated nanopore reads (~10 kb, 5 % error, no -I) per step, resident in HBM "
                                  "(the full 15 000-read shape is a -m gpu parity test)",
                      "ms_per_step": ms, "reads_per_s": (len(o4) - 1) / (ms * 1e-3), "bases_per_s": float(o4[-1]) / (ms * 1e-3),
                      "stage_ms": ix.last_timings()}
    try:
        import shutil
        shutil.rmtree(tmp, ignore_errors=True)
    except Exception:
        pass
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reads", type=int, default=30_000_000, help="reads of the whole sample (all GPUs together)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from drprg_b200 import lib, sharded, sim, workload

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the map path has no CPU fallback")
    # the root rank runs the genotype step (VCF text, ML-path verification on the host): it gets the host cores its
    # sibling ranks do not need; must be set before the library creates its worker pool
    os.environ.setdefault("DRPRG_THREADS", str(sharded.host_threads_for_rank(rank, world)))
    torch.cuda.set_device(local_rank)
    sharded.bind_to_gpu_numa_node(local_rank)  # pinned buffers and host threads next to the GPU's PCIe root
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    reduce_mode = os.environ.get("DRPRG_REDUCE", "fused")

    wl = workload.Config3(total_reads=args.reads)
    mine = wl.rank_subshards(rank, world)
    n = len(mine) * wl.SUBSHARD
    id_base = mine.start * wl.SUBSHARD
    total_bases = n * workload.READ_LEN
    # device-resident inputs (value) and pinned host inputs (e2e): this rank's contiguous part of the 30 M reads
    d_words = torch.empty((n, workload.STRIDE_WORDS), dtype=torch.int32, device="cuda")
    for j, i in enumerate(mine):
        d_words[j * wl.SUBSHARD:(j + 1) * wl.SUBSHARD] = wl.pack_codes(wl.subshard_codes(i))
    d_lens = torch.full((n,), workload.READ_LEN, dtype=torch.int32, device="cuda")
    # The host-buffer (e2e) loop shards by measured upload bandwidth: on the 8-GPU boxes of this pool the eight concurrent
    # H2D streams do not get equal shares of the host's memory / PCIe paths (tools/h2d_concurrency.py: 21.7 GB/s each for
    # GPUs 0-3, 33.3 GB/s each for GPUs 4-7, 51.6 GB/s alone), and a step ends when the slowest upload does.  Every rank
    # still maps a contiguous range of the same 240 sub-shards; the sum over ranks is the same 30 M reads.
    mine_e2e, h2d_gbps = mine, None
    if world > 1 and os.environ.get("DRPRG_E2E_SHARDS", "bandwidth") == "bandwidth":
        h2d_gbps = sharded.concurrent_h2d_gbps(torch, dist)
        mine_e2e = sharded.proportional_subshards(wl.n_subshards, h2d_gbps, rank)
    n_e = len(mine_e2e) * wl.SUBSHARD
    id_base_e = mine_e2e.start * wl.SUBSHARD
    h_words = torch.empty((n_e, workload.STRIDE_WORDS), dtype=torch.int32).pin_memory()
    if mine_e2e == mine:
        h_words.copy_(d_words)
    else:
        for j, i in enumerate(mine_e2e):
            h_words[j * wl.SUBSHARD:(j + 1) * wl.SUBSHARD].copy_(wl.pack_codes(wl.subshard_codes(i)))
    h_lens = torch.full((n_e,), workload.READ_LEN, dtype=torch.int32).pin_memory()
    torch.cuda.synchronize()

    ix = lib.Index(wl.prg_path, wl.w, wl.k, device=local_rank)
    opts = lib.make_opts(illumina=True, genome_size=workload.GENOME_SIZE, min_cluster_size=10)
    if world > 1 and reduce_mode == "fused":
        sharded.setup_fused_reduce(ix, rank, world)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    resident = ix.wrap_device(d_words.data_ptr(), d_lens.data_ptr(), n, workload.STRIDE_WORDS, total_bases,
                              read_id_base=id_base, keep=(d_words, d_lens))
    stats = {}

    def hot_path(batch):
        ix.sample_begin(opts, workload.READ_LEN)
        nh, nk = ix.map_batch(batch)
        t = ix.last_timings()
        for k_, v_ in t.items():
            stats.setdefault(k_, []).append(v_)
        stats.setdefault("hits", []).append(nh)
        stats.setdefault("kept", []).append(nk)
        if world > 1:
            if reduce_mode == "fused":
                if rank != 0:          # this rank's coverage is already in the root's accumulator: report the arrival
                    ix.shard_done()
                    return None
            else:
                sharded.allreduce_accum(ix)
                if rank != 0:
                    torch.cuda.current_stream().synchronize()
                    return None
        ix.genotype(wl.refs_path)      # root: waits on the device for the other ranks' arrivals (fused mode)
        for k_, v_ in ix.last_genotype_timings().items():
            stats.setdefault("gt_" + k_, []).append(v_)
        return ix.vcf_view()  # the step's result: the VCF text in host memory (zero-copy view of the library's buffer)

    def step_resident():
        return hot_path(resident)

    def step_e2e():
        b = ix.upload_ptrs(h_words.data_ptr(), h_lens.data_ptr(), n_e, workload.STRIDE_WORDS, n_e * workload.READ_LEN, read_id_base=id_base_e)
        try:
            return hot_path(b)
        finally:
            b.free()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            flush.zero_()
            if world > 1:
                dist.barrier()
            fn()
        stats.clear()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        l0 = lib.launch_count()
        out = None
        for i in range(steps):
            flush.zero_()                      # L2 flush between timed iterations (outside the events)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            starts[i].record()
            out = fn()
            ends[i].record()
            ends[i].synchronize()
        torch.cuda.synchronize()
        ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends))
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)   # max over ranks
        return float(t.item()) / steps, lib.launch_count() - l0, out, {k_: list(v_) for k_, v_ in stats.items()}

    sampler = ClockSampler(local_rank)
    if not os.environ.get("DRPRG_BENCH_NO_SAMPLER"):
        sampler.start()
    ms_step, launches, vcf_text, st = timed(step_resident, args.steps, args.warmup)
    clocks = sampler.stop()
    vcf_text = bytes(vcf_text) if vcf_text is not None else b""  # a copy: the next genotype call reuses the library's buffer
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ix, vcf_text, st)
    ms_e2e, _, _, _ = timed(step_e2e, max(3, args.steps // 2), args.warmup)

    total_reads = wl.total_reads
    value = total_reads / (ms_step * 1e-3)
    e2e_value = total_reads / (ms_e2e * 1e-3)
    # roofline of the dominant kernel pair (sketch+lookup) on this rank's shard: algorithmic bytes = packed bases +
    # length word per read + 16 B per emitted hit (SURVEY §8d), over the pair's CUDA-event duration measured inside the library
    k_ms = float(np.mean(st["sketch_lookup"]))
    hits = float(np.mean(st["hits"]))
    alg_bytes = n * (workload.STRIDE_WORDS * 4 + 4) + 16.0 * hits
    peak, peak_src = measured_peak()
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9
    prof = screen_profile()
    issue_peak = ix.issue_peak() if rank == 0 else 0.0
    n_records = sum(1 for l in vcf_text.splitlines() if not l.startswith(b"#"))
    h2d = int(total_reads * (workload.STRIDE_WORDS * 4 + 4))  # all ranks together: words + lengths of the 30 M reads
    d2h = int(len(vcf_text) + 4096)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u32 (hash/cluster/coverage), f64 (likelihoods)", "data": "synthetic (reads generated on cuda)",
        "config": workload_config(wl, total_reads),
        "run": {"reads_per_gpu_per_step": n, "l2": "inputs larger than L2 from 3 M reads per GPU; also flushed with a 512 MiB memset between timed iterations",
                "reduce": ("none (one GPU)" if world == 1 else
                           "fused: coverage kernel adds into the root accumulator over NVLink (CUDA IPC mapping), device-side arrival flags"
                           if reduce_mode == "fused" else "NCCL allreduce of the accumulator (torch.distributed)"),
                "vcf_records": n_records, "vcf_sha1": hashlib.sha1(strip_file_date(vcf_text)).hexdigest()},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e,
                "what": "same steps from pinned host buffers: H2D of every rank's packed shard inside the timed region, VCF text read on the host",
                "reads_per_rank": "even" if mine_e2e == mine or h2d_gbps is None else
                                  "proportional to each rank's measured concurrent H2D bandwidth: " + ", ".join(f"{g:.0f}" for g in h2d_gbps) + " GB/s"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "stage_ms": {k_: float(np.mean(v_)) for k_, v_ in st.items() if k_ not in ("hits", "kept")},
    }
    roof = {"bound": "hbm", "kernel": "screen_kernel<15,10> + resolve_kernel<11,15> (S1+S2: k-mer screen of every read, then hash/probe/minimizer test of the flagged positions)",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
            "kernel_ms": k_ms, "algorithmic_bytes_per_launch": alg_bytes, "reads_per_launch": n}
    if prof:
        scale = n / 1e6
        roof["traffic"] = prof.get("dram_bytes_per_million_reads", 0) * scale or None
        roof["traffic_source"] = prof["source"]
        wi = prof.get("warp_instr_per_read_screen", 0) + prof.get("warp_instr_per_read_resolve", 0)
        if issue_peak > 0 and wi:
            roof["issue"] = {"warp_instr_per_read": wi, "achieved_warp_instr_per_s": wi * n / (k_ms * 1e-3),
                             "measured_int_issue_peak_warp_instr_per_s": issue_peak,
                             "issue_frac": wi * n / (k_ms * 1e-3) / issue_peak,
                             "note": "the pair is bound by instruction issue (32-bit multiply-add / shift / logic + one shared-memory probe per "
                                     "k-mer position), not by HBM: issue_frac is its warp-instruction rate over the rate a pure INT32 "
                                     "mad/shf/lop3 loop reaches on this GPU (measured in this run)"}
    line["roofline"] = roof

    if world > 1:
        # sharded parity, outside the timed region: the root maps ALL 30 M reads alone (regenerated sub-shard by sub-shard)
        # into one accumulator and must reproduce the sharded run's accumulator and VCF bit for bit
        acc_sharded = ix.accum_download() if rank == 0 else None
        dist.barrier()
        if rank == 0:
            sx = lib.Index(wl.prg_path, wl.w, wl.k, device=local_rank)
            sx.sample_begin(opts, workload.READ_LEN)
            group = 16  # 2 M reads per batch
            for g0 in range(0, wl.n_subshards, group):
                ids = range(g0, min(g0 + group, wl.n_subshards))
                w = torch.cat([wl.pack_codes(wl.subshard_codes(i)) for i in ids])
                l = torch.full((w.shape[0],), workload.READ_LEN, dtype=torch.int32, device="cuda")
                sx.map_batch(sx.wrap_device(w.data_ptr(), l.data_ptr(), w.shape[0], workload.STRIDE_WORDS, w.shape[0] * workload.READ_LEN,
                                            read_id_base=g0 * wl.SUBSHARD, keep=(w, l)))
            sx.genotype(wl.refs_path)
            whole = sx.accum_download()
            vcf_whole = b"\n".join(l for l in bytes(sx.vcf_view()).splitlines() if not l.startswith(b"##fileDate"))
            acc_ok = bool((acc_sharded[:-4] == whole[:-4]).all()) and sharded.decode_scalars(acc_sharded[-4:]) == sharded.decode_scalars(whole[-4:])
            line["sharded_parity"] = bool(acc_ok and hashlib.sha1(vcf_whole).hexdigest() == line["run"]["vcf_sha1"])
            line["sharded_parity_detail"] = {"accumulators_equal": acc_ok, "vcf_sha1_single_gpu": hashlib.sha1(vcf_whole).hexdigest()}
            sx.close()
        dist.barrier()
    else:
        line["sharded_parity"] = None

    if rank == 0 and world == 1 and not args.no_extras:
        try:
            line["extras"] = extras_single_gpu(lib, workload, sim, wl, ix, opts, torch, flush)
        except Exception as e:  # the headline must survive a failing side measurement
            line["extras"] = {"error": repr(e)}
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle_py as O
        ox = O.Index(wl.prg_path, wl.w, wl.k)
        cores = os.cpu_count() or 1
        oo = O.make_opts(threads=cores, illumina=True, genome_size=workload.GENOME_SIZE)
        data, off, ns = cpu_sample(wl, "cuda")
        oracle_step(O, ox, data, off, oo, wl.refs_path)
        t0 = time.perf_counter()
        reps = 3
        for _ in range(reps):
            oracle_step(O, ox, data, off, oo, wl.refs_path)
        dt = (time.perf_counter() - t0) / reps
        line["cpu_baseline"] = {"value": ns / dt, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"the first {ns} reads of the workload (sub-shards 0-{CPU_SAMPLE_SUBSHARDS - 1}) mapped and genotyped {reps} times, "
                                          f"restated CPU oracle on {cores} threads (not the pandora binary)"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
