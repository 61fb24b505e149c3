"""Host wall-clock of every call of one bench step (resident batch): where the step's time goes outside the kernels."""
import sys, os, time, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from drprg_b200 import lib, workload
import numpy as np, torch
n = int(sys.argv[1]) if len(sys.argv) > 1 else 1000000
wl = workload.Config2(); d, o = wl.reads(n, 0); words, _, lens = lib.pack_reads(d, o, 10)
ix = lib.Index(wl.prg_path, 11, 15); opts = lib.make_opts(illumina=True)
dw = torch.from_numpy(words.view(np.int32)).cuda(); dl = torch.from_numpy(lens.view(np.int32)).cuda()
b = ix.wrap_device(dw.data_ptr(), dl.data_ptr(), n, 10, int(o[-1]), keep=(dw, dl))
flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
acc = {}
def lap(name, t0):
    t = time.perf_counter(); acc.setdefault(name, []).append((t - t0) * 1e3); return t
for i in range(25):
    flush.zero_(); torch.cuda.synchronize()
    t = t00 = time.perf_counter()
    ix.sample_begin(opts, 150); t = lap("sample_begin", t)
    nh, nk = ix.map_batch(b); t = lap("map_batch", t)
    tm = ix.last_timings(); t = lap("last_timings", t)
    ix.genotype(wl.refs_path); t = lap("genotype", t)
    gt = ix.last_genotype_timings(); t = lap("last_gt_timings", t)
    v = ix.vcf_bytes(); t = lap("vcf_bytes", t)
    lap("total", t00)
    acc.setdefault("map_kernels_sum", []).append(sum(tm.values()))
    acc.setdefault("gt_stages_sum", []).append(sum(v_ for k_, v_ in gt.items() if k_ != "mlpath_kernel"))
print(json.dumps({k: round(float(np.median(v[5:])), 4) for k, v in acc.items()}))
print(json.dumps({k: round(v, 4) for k, v in tm.items()}), json.dumps({k: round(v, 4) for k, v in gt.items()}))
