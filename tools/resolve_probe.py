"""Split of the sketch+lookup stage (S1+S2) at config-3 size: `screen_kernel` and `resolve_kernel` times from torch.profiler
(CUDA activities), the stage's CUDA-event time, and queue entries, probe survivors and hits per read.  Inputs are larger
than L2 and a 512 MiB memset runs between iterations, as in bench.py.
   python tools/resolve_probe.py [--reads N] [--iters I] [LIB.so ...]
Every library (default: the in-tree build) is loaded in a subprocess of its own through DRPRG_CUDA_LIB, so builds can be
compared in one call; one JSON line per library.  The counts come from the library's DRPRG_TIMING report of the batch
(builds without that report give null).  That report gives the largest chunk's queue; the batch here is device-resident,
i.e. one chunk, so it is the whole queue (a batch of several chunks would report no queue_per_read)."""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REPORT = re.compile(r"\[drprg-cuda\] map batch: (\d+) reads, (\d+) chunks, screen queue (\d+) \(largest chunk\), probe survivors (\d+), hits (\d+)")


def run(n_reads, iters):
    import torch
    from torch.profiler import ProfilerActivity, profile
    from torch.autograd import DeviceType
    from drprg_b200 import lib, workload

    wl = workload.Config3(total_reads=n_reads)
    d_words = torch.empty((n_reads, workload.STRIDE_WORDS), dtype=torch.int32, device="cuda")
    for i in range(wl.n_subshards):
        d_words[i * wl.SUBSHARD:(i + 1) * wl.SUBSHARD] = wl.pack_codes(wl.subshard_codes(i))
    d_lens = torch.full((n_reads,), workload.READ_LEN, dtype=torch.int32, device="cuda")
    ix = lib.Index(wl.prg_path, wl.w, wl.k)
    opts = lib.make_opts(illumina=True, genome_size=workload.GENOME_SIZE, min_cluster_size=10)
    batch = ix.wrap_device(d_words.data_ptr(), d_lens.data_ptr(), n_reads, workload.STRIDE_WORDS, n_reads * workload.READ_LEN,
                           keep=(d_words, d_lens))
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")

    def step():
        flush.zero_()
        torch.cuda.synchronize()
        ix.sample_begin(opts, workload.READ_LEN)
        nh, _ = ix.map_batch(batch)
        return nh, ix.last_timings()["sketch_lookup"]

    for _ in range(3):
        step()
    stage = [step()[1] for _ in range(iters)]
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            nh, _ = step()
    kern = {}
    for e in prof.events():
        if e.device_type != DeviceType.CUDA:
            continue
        for tag in ("screen_kernel", "resolve_kernel"):
            if tag in e.name:
                kern.setdefault(tag, []).append(e.time_range.end - e.time_range.start)
    return {"reads": n_reads, "iters": iters, "gpu": torch.cuda.get_device_name(),
            "sketch_lookup_ms_median": round(statistics.median(stage), 4),
            "sketch_lookup_ms_spread": round(max(stage) - min(stage), 4),
            **{f"{t}_us_median": round(statistics.median(v), 1) for t, v in kern.items()},
            **{f"{t}_launches": len(v) for t, v in kern.items()},
            "hits": nh}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=30_000_000)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--run", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("libs", nargs="*")
    args = ap.parse_args()
    if args.run:
        print(json.dumps(run(args.reads, args.iters)), flush=True)
        return
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                               text=True).stdout.strip().splitlines()
    except OSError:
        power = []
    print(json.dumps({"nvidia_smi_name_power_limit": power}), flush=True)
    for so in args.libs or [None]:
        env = dict(os.environ, DRPRG_TIMING="1")
        if so:
            env["DRPRG_CUDA_LIB"] = os.path.abspath(so)
        p = subprocess.run([sys.executable, os.path.abspath(__file__), "--run", "--reads", str(args.reads), "--iters", str(args.iters)],
                           env=env, capture_output=True, text=True)
        if p.returncode != 0:
            sys.stderr.write(p.stderr[-4000:])
            print(json.dumps({"lib": so or "in-tree", "error": f"exit {p.returncode}"}), flush=True)
            continue
        line = json.loads(p.stdout.strip().splitlines()[-1])
        m = REPORT.findall(p.stderr)
        n = args.reads
        if m:
            reads, chunks, queue, surv, hits = map(int, m[-1])
            line.update(queue_per_read=round(queue / reads, 4) if chunks == 1 else None, survivors_per_read=round(surv / reads, 4), hits_per_read=round(hits / reads, 4))
        else:
            line.update(queue_per_read=None, survivors_per_read=None, hits_per_read=round(line["hits"] / n, 4))
        line["lib"] = so or "in-tree"
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
