"""Drop-in call from a FASTQ file (drprg_cuda_map_genotype): wall time with the host-framed ingest (default) and the host
parser (DRPRG_HOST_INGEST=1).
   python tools/e2e_probe.py [n_reads]"""
import sys, os, subprocess, json, tempfile, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if len(sys.argv) > 1 and sys.argv[1] == "run":
    from drprg_b200 import lib, workload, sim
    fq, gz, prg, refs = sys.argv[2:6]
    ix = lib.Index(prg, 11, 15); opts = lib.make_opts(illumina=True, threads=os.cpu_count() or 1)
    out = tempfile.mkdtemp()
    res = {}
    for name, path in (("plain", fq), ("gzip", gz)):
        ts = []
        for i in range(6):
            t0 = time.perf_counter(); st = ix.map_genotype(path, refs, out, opts); ts.append((time.perf_counter() - t0) * 1e3)
        res[name] = dict(wall_ms_min=round(min(ts[1:]), 2), ingest_ms=round(st["ms_ingest"], 2), map_ms=round(st["ms_map"], 2),
                         genotype_ms=round(st["ms_genotype"], 2), n_reads=st["n_reads"], records=st["n_records"])
    import hashlib
    res["vcf_sha1"] = hashlib.sha1(b"".join(l for l in open(os.path.join(out, "pandora_genotyped.vcf"), "rb") if not l.startswith(b"##fileDate"))).hexdigest()[:12]
    print(json.dumps({"host_ingest": os.environ.get("DRPRG_HOST_INGEST", "0"), **res}))
else:
    from drprg_b200 import workload, sim
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 1000000
    wl = workload.Config2(); d, o = wl.reads(n, 0)
    tmp = tempfile.mkdtemp()
    fq, gz = os.path.join(tmp, "r.fq"), os.path.join(tmp, "r.fq.gz")
    import numpy as np
    # fast FASTQ writer (1 M reads)
    L = 150
    reads = d.reshape(n, L)
    rec = np.empty((n, 8 + 1 + L + 3 + L + 1), np.uint8)
    ids = np.char.zfill(np.arange(n).astype(str), 7).astype("S7")
    rec[:, 0] = ord("@"); rec[:, 1:8] = np.frombuffer(ids.tobytes(), np.uint8).reshape(n, 7); rec[:, 8] = 10
    rec[:, 9:9 + L] = reads; rec[:, 9 + L] = 10; rec[:, 10 + L] = ord("+"); rec[:, 11 + L] = 10
    rec[:, 12 + L:12 + 2 * L] = ord("I"); rec[:, 12 + 2 * L] = 10
    rec.tofile(fq)
    subprocess.run(f"gzip -1 -c {fq} > {gz}", shell=True, check=True)
    for extra in ({}, {"DRPRG_HOST_INGEST": "1"}):
        subprocess.run([sys.executable, __file__, "run", fq, gz, wl.prg_path, wl.refs_path], env=dict(os.environ, **extra))
