"""Host-side mirror of the reference's adapter for this path: `Pandora::genotype_with`
(/root/reference/src/lib.rs:580-642), `Pandora::vcf_filename` (:644-646) and `Pandora::index_with` (:479-510), same
names, argument meaning and error behaviour, but backed by the CUDA library instead of a pandora subprocess.
`discover_with` is `Pandora::discover_with` (:513-578): one map pass, the local assembly on the GPU and
discover/denovo_paths.txt.  `discover_candidates` and `discover_paths` return its intermediate results after a
`genotype_with(..., retain_hits=True)`.

The reference builds the argv  -t T -w W -k K -c C [-I] [-K]  (src/predict.rs:288-294) after the fixed
`map --genotype --local --gt-conf 0 -v -o OUT -g 4411532 --max-covg 4294967295 --vcf-refs REF`
(src/lib.rs:594-609); `genotype_with` here accepts that same `args` list.
"""
from __future__ import annotations

import os

from . import lib

MTB_GENOME_SIZE = 4411532  # src/lib.rs:36


class DependencyError(RuntimeError):
    """Mirror of DependencyError::ProcessError (src/lib.rs:65-90): raised where the reference returns Err."""


class Pandora:
    def __init__(self, device: int = 0):
        self.device = device
        self._index = None
        self._key = None

    @classmethod
    def from_path(cls, path=None, device: int = 0):
        """The reference locates an executable (src/lib.rs:464-476); here the 'executable' is the in-tree
        CUDA library, and a missing library is the same error class."""
        try:
            lib.lib()
        except lib.DrprgCudaError as e:
            raise DependencyError(str(e)) from e
        return cls(device)

    @staticmethod
    def vcf_filename() -> str:
        return "pandora_genotyped.vcf"

    @staticmethod
    def _parse_args(args):
        o = dict(threads=1, w=14, k=15, c=10, illumina=False, debug=False)
        it = iter([str(a) for a in args])
        for a in it:
            if a == "-t":
                o["threads"] = int(next(it))
            elif a == "-w":
                o["w"] = int(next(it))
            elif a == "-k":
                o["k"] = int(next(it))
            elif a == "-c":
                o["c"] = int(next(it))
            elif a == "-I":
                o["illumina"] = True
            elif a == "-K":
                o["debug"] = True
            else:
                raise DependencyError(f"unsupported pandora map argument: {a}")
        return o

    def load_index(self, prg, w, k):
        key = (os.path.abspath(str(prg)), os.path.getmtime(str(prg)), w, k)
        if key != self._key:
            if self._index is not None:
                self._index.close()
            self._index = lib.Index(prg, w, k, device=self.device)
            self._key = key
        return self._index

    def index_with(self, input, args=()):
        """`pandora index -t T -w W -k K <prg>` (src/predict.rs:283, src/builder.rs:644-657): writes <prg>.kK.wW.idx and
        kmer_prgs/ next to the PRG (host work, no GPU)."""
        o = dict(w=14, k=15)
        it = iter([str(a) for a in args])
        for a in it:
            if a == "-t":
                next(it)
            elif a == "-w":
                o["w"] = int(next(it))
            elif a == "-k":
                o["k"] = int(next(it))
            else:
                raise DependencyError(f"unsupported pandora index argument: {a}")
        try:
            ix = lib.Index(input, o["w"], o["k"], device=-1)
            try:
                ix.write_pandora_index(input)
            finally:
                ix.close()
        except lib.DrprgCudaError as e:
            raise DependencyError(str(e)) from e

    def genotype_with(self, prg, vcf_ref, reads, outdir, args=(), retain_hits=False):
        """Blocking; writes <outdir>/pandora.log and <outdir>/pandora_genotyped.vcf; raises DependencyError
        where the reference returns Err(DependencyError::ProcessError)."""
        o = self._parse_args(args)
        try:
            ix = self.load_index(prg, o["w"], o["k"])
            ix.retain_hits(retain_hits)  # True: discover_candidates() may be asked afterwards (one pass for discover + map)
            opts = lib.make_opts(threads=o["threads"], min_cluster_size=o["c"], illumina=o["illumina"],
                                 genome_size=MTB_GENOME_SIZE, gt_conf=0.0, debug=o["debug"])
            return ix.map_genotype(reads, vcf_ref, outdir, opts)
        except lib.DrprgCudaError as e:
            raise DependencyError(str(e)) from e

    def discover_with(self, prg, query_idx, outdir, args=()):
        """`pandora discover -g 4411532 --max-covg 4294967295 -v -o OUT -t T -w W -k K -c C [-I] [-K] <prg> <query.tsv>`
        (src/lib.rs:513-578): query_idx holds one `sample<TAB>reads` line (a relative reads path is taken from the query
        file's directory); writes OUT/denovo_paths.txt and returns its path; raises DependencyError where the reference
        returns Err."""
        o = self._parse_args(args)
        try:
            lines = [l for l in open(query_idx).read().splitlines() if l.strip()]
        except OSError as e:
            raise DependencyError(f"cannot read {query_idx}: {e}") from e
        if len(lines) != 1:
            raise DependencyError(f"{query_idx}: {len(lines)} samples; discover takes a query file with exactly one")
        fields = lines[0].split("\t")
        if len(fields) != 2:
            raise DependencyError(f"{query_idx}: expected `sample<TAB>reads`")
        sample, reads = fields
        reads = os.path.join(os.path.dirname(os.path.abspath(str(query_idx))), reads)
        os.makedirs(outdir, exist_ok=True)
        try:
            ix = self.load_index(prg, o["w"], o["k"])
            opts = lib.make_opts(threads=o["threads"], min_cluster_size=o["c"], illumina=o["illumina"],
                                 genome_size=MTB_GENOME_SIZE, gt_conf=0.0, debug=o["debug"])
            ix.discover(reads, outdir, opts, sample=sample)
        except lib.DrprgCudaError as e:
            raise DependencyError(str(e)) from e
        return os.path.join(str(outdir), "denovo_paths.txt")

    def discover_candidates(self, **opts):
        """After genotype_with(..., retain_hits=True): the inputs of pandora discover's local assembler (ML consensus and
        per-base coverage per locus, low-coverage candidate regions, the reads over them) without mapping the reads again."""
        if self._index is None:
            raise DependencyError("genotype_with(..., retain_hits=True) has not been run")
        try:
            return self._index.discover_candidates(**opts)
        except lib.DrprgCudaError as e:
            raise DependencyError(str(e)) from e

    def discover_paths(self, **opts):
        """After genotype_with(..., retain_hits=True): pandora discover's de-novo alleles from the same pass, with pandora's
        defaults for the candidate regions -> {locus name: [(a, b, sequence), ...]}, each replacing [a, b) of the locus's
        maximum-likelihood sequence; opts go to lib.Index.discover_assemble."""
        if self._index is None:
            raise DependencyError("genotype_with(..., retain_hits=True) has not been run")
        try:
            ix = self._index
            _, regions = ix.discover_candidates()
            _, paths = ix.discover_assemble(**opts)
        except lib.DrprgCudaError as e:
            raise DependencyError(str(e)) from e
        out = {}
        for r, a, b, seq in paths:
            out.setdefault(ix.names[regions[r][0]], []).append((a, b, seq))
        return out
