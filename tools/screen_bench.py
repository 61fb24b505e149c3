"""A/B of the k-mer screen inside one gpurun call: sketch+lookup stage time (device-resident batch, one launch per
kernel) with the screen off and on; the hit set must be identical.
   python tools/screen_bench.py [n_reads]"""
import sys, os, subprocess, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if len(sys.argv) > 1 and sys.argv[1] == "run":
    from drprg_b200 import lib, workload
    import numpy as np, torch, hashlib
    n = int(sys.argv[2])
    wl = workload.Config2(); d, o = wl.reads(n, 0); words, _, lens = lib.pack_reads(d, o, 10)
    ix = lib.Index(wl.prg_path, 11, 15); opts = lib.make_opts(illumina=True)
    dw = torch.from_numpy(words.view(np.int32)).cuda(); dl = torch.from_numpy(lens.view(np.int32)).cuda()
    b = ix.wrap_device(dw.data_ptr(), dl.data_ptr(), n, 10, int(o[-1]), keep=(dw, dl))
    ts = []
    for i in range(12):
        ix.sample_begin(opts, 150); nh, nk = ix.map_batch(b); ts.append(ix.last_timings()["sketch_lookup"])
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda"); cold = []
    for i in range(8):
        flush.zero_(); torch.cuda.synchronize()
        ix.sample_begin(opts, 150); nh, nk = ix.map_batch(b); cold.append(ix.last_timings()["sketch_lookup"])
    h = ix.last_hits(nh)
    dig = hashlib.sha1(b"".join(np.ascontiguousarray(h[k]).tobytes() for k in ("read", "prg", "fwd", "start", "knode", "kept"))).hexdigest()
    print(json.dumps({"screen": os.environ.get("DRPRG_SCREEN"), "reads": n,
                      "sketch_ms_min": round(min(ts[2:]), 4), "sketch_ms_med": round(sorted(ts[2:])[len(ts[2:]) // 2], 4), "cold_ms_min": round(min(cold[1:]), 4), "cold_ms_med": round(sorted(cold[1:])[len(cold[1:]) // 2], 4),
                      "hits": nh, "kept": nk, "sha1": dig[:12]}))
else:
    n = sys.argv[1] if len(sys.argv) > 1 else "1000000"
    for s in ("0", "1"):
        subprocess.run([sys.executable, __file__, "run", n], env=dict(os.environ, DRPRG_SCREEN=s))
