"""BASELINE config 5: a batch of simulated Illumina samples, SAMPLE-sharded over the GPUs of the box (replicas only: no
collective on the data path).  Rank r of N keeps the index resident on its GPU and runs samples r, r + N, ... through the
drop-in batch call drprg_cuda_map_genotype_batch (FASTQ files in, pandora_genotyped.vcf files out).  Reports samples/hour
end to end and checks every VCF against the VCF the same reads give on rank 0 alone.
With `discover`, each rank first runs its samples through drprg_cuda_discover_batch (denovo_paths.txt out) and then through
drprg_cuda_map_genotype_batch on the same files: the two pandora steps drprg predict asks for per sample.  Reports
samples/hour for discover, for map and for the two together, and also checks every denovo_paths.txt against the file a
single drprg_cuda_discover call on rank 0 writes for the same reads.
   python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/batch_bench.py [n_samples] [gz] [discover]"""
import ctypes as C
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

from drprg_b200 import lib, sharded, sim, workload

rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
n_samples = int(sys.argv[1]) if len(sys.argv) > 1 else 96
gz = "gz" in sys.argv[2:]
discover = "discover" in sys.argv[2:]
cores = os.cpu_count() or 1
os.environ.setdefault("DRPRG_THREADS", str(max(2, cores // world)))
torch.cuda.set_device(local)
if world > 1:
    dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
wl = workload.Config3()
DISTINCT = 4  # distinct read sets (different sub-shards of the workload = different read seeds); samples cycle through them
root = "/dev/shm" if os.path.isdir("/dev/shm") else None
tmp = os.path.join(root or tempfile.gettempdir(), "drprg_batch_bench")
sample_path = lambda s: os.path.join(tmp, f"sample{s}.fq" + (".gz" if gz else ""))
if rank == 0:
    shutil.rmtree(tmp, ignore_errors=True)
    os.makedirs(tmp)
    for s in range(DISTINCT):
        codes = torch.cat([wl.subshard_codes(8 * s + i) for i in range(8)])  # 1 M reads
        data = sim.BASES[codes.cpu().numpy()].reshape(-1)
        off = np.arange(codes.shape[0] + 1, dtype=np.uint64) * np.uint64(workload.READ_LEN)
        sim.write_fastq_fast(sample_path(s), data, off, gz=gz, seed=s)
if world > 1:
    dist.barrier()
ix = lib.Index(wl.prg_path, wl.w, wl.k, device=local)
opts = lib.make_opts(illumina=True, genome_size=workload.GENOME_SIZE, threads=max(2, cores // world))
mine = list(range(n_samples))[rank::world]
reads = [sample_path(s % DISTINCT).encode() for s in mine]


def dirs(tag):
    out = []
    for s in mine:
        od = os.path.join(tmp, f"{tag}{s}")
        os.makedirs(od, exist_ok=True)
        out.append(od.encode())
    return out


outs = dirs("out")
disc = dirs("disc") if discover else []
# warm-up: one sample (buffers, site tables)
ix.map_genotype(reads[0].decode(), wl.refs_path, outs[0].decode(), opts)
if discover:
    ix.discover(reads[0].decode(), disc[0].decode(), opts)
torch.cuda.synchronize()
if world > 1:
    dist.barrier()


def timed(call):
    t0 = time.perf_counter()
    call()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    return time.perf_counter() - t0


arr_r, arr_o = (C.c_char_p * len(mine))(*reads), (C.c_char_p * len(mine))(*outs)


def map_batch():
    rc = lib.lib().drprg_cuda_map_genotype_batch(ix.h, C.c_size_t(len(mine)), arr_r, wl.refs_path.encode(), arr_o, C.byref(opts), None)
    assert rc == 0, lib.lib().drprg_cuda_last_error()


dt_d = timed(lambda: ix.discover_batch(None, [r.decode() for r in reads], [d.decode() for d in disc], opts)) if discover else 0.0
dt = timed(map_batch)


def sha(path):
    return hashlib.sha1(b"\n".join(l for l in open(path, "rb").read().splitlines() if not l.startswith(b"##fileDate"))).hexdigest()


def rate(seconds):
    return {"seconds": seconds, "samples_per_hour": 3600.0 * n_samples / seconds, "ms_per_sample_per_gpu": seconds / max(1, len(mine)) * 1e3}


ok = ok_d = True
if rank == 0:
    want, want_d = {}, {}
    for s in range(min(DISTINCT, n_samples)):
        od = os.path.join(tmp, f"ref{s}")
        os.makedirs(od, exist_ok=True)
        ix.map_genotype(sample_path(s), wl.refs_path, od, opts)
        want[s] = sha(os.path.join(od, "pandora_genotyped.vcf"))
        if discover:
            ix.discover(sample_path(s), od, opts)
            want_d[s] = open(os.path.join(od, "denovo_paths.txt"), "rb").read()
    for s in range(n_samples):
        ok = ok and sha(os.path.join(tmp, f"out{s}", "pandora_genotyped.vcf")) == want[s % DISTINCT]
        if discover:
            ok_d = ok_d and open(os.path.join(tmp, f"disc{s}", "denovo_paths.txt"), "rb").read() == want_d[s % DISTINCT]
    if not discover:
        print(json.dumps({"config": "config5: batch of simulated Illumina samples (1 M x 150 bp reads each), sample-sharded, replicas only",
                          "n_gpus": world, "samples": n_samples, "input": "gzip FASTQ" if gz else "plain FASTQ", "seconds": dt,
                          "samples_per_hour": 3600.0 * n_samples / dt, "ms_per_sample_per_gpu": dt / max(1, len(mine)) * 1e3,
                          "every_vcf_equals_single_gpu_run": bool(ok), "host_cores": cores}))
    else:
        card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)],
                              capture_output=True, text=True).stdout.strip()
        print(json.dumps({"config": "config5, both pandora steps: discover batch, then map batch on the same files "
                                    "(1 M x 150 bp simulated Illumina reads each), sample-sharded, replicas only",
                          "n_gpus": world, "samples": n_samples, "input": "gzip FASTQ" if gz else "plain FASTQ",
                          "discover": rate(dt_d), "map": rate(dt), "discover_and_map": rate(dt_d + dt),
                          "every_denovo_paths_equals_single_call": bool(ok_d), "every_vcf_equals_single_gpu_run": bool(ok),
                          "host_cores": cores, "card": card}))
    shutil.rmtree(tmp, ignore_errors=True)
if world > 1:
    dist.barrier()
    dist.destroy_process_group()
sys.exit(0 if ok and ok_d else 1)
