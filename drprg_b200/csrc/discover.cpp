// One mapping pass for `pandora discover` AND `pandora map` (SURVEY.md §8f rank 1).  drprg runs pandora twice per sample:
// discover (/root/reference/src/predict.rs:247-256 -> src/lib.rs:513-578) maps every read to find the regions of each
// locus's maximum-likelihood sequence that the reads do not support and hands the reads over those regions to its local
// assembler; map (src/predict.rs:296-302) then maps the same reads again.  The first half of discover is exactly S1-S7
// of the hot path, so its results are taken from the pass that is run anyway:
//   per-base coverage   along the ML local path: the largest (fwd + rev) coverage among the ML k-mers covering a base
//                       (pandora get_covgs_along_localnode_path)
//   candidate regions   maximal runs of positions with coverage below --covg-threshold (3) whose length lies in [-l, -L]
//                       = [1, 30] (identify_low_coverage_intervals), padded by -P 22 either side
//   region reads        for every read with kept hits on the locus: its hits whose k-mer lies on the ML path inside the
//                       padded region; reads with at least two such hits contribute the span [min start, max start + k) and
//                       the strand of the first hit (get_read_overlap_coordinates / find_hits_inside_path).  These are
//                       found on the GPU from the retained hits (assemble.cu, region_reads_kernel) with the tables made here.
// The de-novo assembly itself (pandora's de Bruijn graph walk) runs on the GPU (assemble.cu); this file produces its inputs
// and writes its result, discover/denovo_paths.txt.
// Option names and defaults are upstream pandora's `discover` (drprg passes none of them, src/predict.rs:236-245).
#include <algorithm>
#include <stdexcept>

#include "genotype_host.hpp"

namespace drprg {

static inline uint32_t sat16u(int32_t c) { return c > 65535 ? 65535u : (c < 0 ? 0u : (uint32_t)c); }

std::vector<uint32_t> ml_path_base_coverage(const HostIndex& H, uint32_t locus, const std::vector<uint32_t>& kpath,
                                            const std::vector<uint32_t>& lpath, const int32_t* cov) {
    const Locus& L = H.loci[locus];
    const uint32_t base = H.knode_base[locus];
    std::vector<int64_t> node_off(L.nodes.size(), -1);
    size_t nbases = 0;
    for (uint32_t n : lpath) {
        node_off[n] = (int64_t)nbases;
        nbases += L.node_len(n);
    }
    std::vector<uint32_t> per_base(nbases, 0);
    for (uint32_t r : kpath) {
        const uint32_t g = base + r;
        const uint32_t c = sat16u(cov[2 * g]) + sat16u(cov[2 * g + 1]);
        for (auto& sg : L.kpath[r]) {
            if (sg.s == sg.e || node_off[sg.node] < 0) continue;
            uint32_t* v = per_base.data() + node_off[sg.node];
            for (uint32_t x = sg.s - L.nodes[sg.node].s; x < sg.e - L.nodes[sg.node].s; ++x) v[x] = std::max(v[x], c);
        }
    }
    return per_base;
}

std::string spell_local_path(const Locus& L, const std::vector<uint32_t>& lpath) {
    std::string s;
    for (uint32_t n : lpath) s += L.node_seq(n);
    return s;
}

void low_coverage_intervals(const std::vector<uint32_t>& covg, uint32_t threshold, uint32_t min_len, uint32_t max_len,
                            std::vector<std::pair<uint32_t, uint32_t>>& out) {
    const size_t n = covg.size();
    size_t cur = 0;
    while (cur < n) {
        const size_t prev = cur;
        while (cur < n && covg[cur] < threshold) ++cur;  // find_if_not(below threshold)
        if (cur - prev >= min_len && cur - prev <= max_len && cur > prev) out.emplace_back((uint32_t)prev, (uint32_t)cur);
        if (cur == n) break;
        ++cur;
    }
}

// consensus interval [start, start + k) of every k-mer node of the locus that lies on the local path; UINT32_MAX otherwise
std::vector<uint32_t> knode_consensus_start(const Locus& L, const std::vector<uint32_t>& lpath) {
    std::vector<int64_t> node_off(L.nodes.size(), -1);
    std::vector<int32_t> node_idx(L.nodes.size(), -1);
    size_t nb = 0;
    for (size_t i = 0; i < lpath.size(); ++i) {
        node_off[lpath[i]] = (int64_t)nb;
        node_idx[lpath[i]] = (int32_t)i;
        nb += L.node_len(lpath[i]);
    }
    std::vector<uint32_t> out(L.kpath.size(), UINT32_MAX);
    for (size_t r = 0; r < L.kpath.size(); ++r) {
        const KPath& kp = L.kpath[r];
        if (kp.empty()) continue;
        bool on = true;
        uint32_t len = 0;
        for (size_t i = 0; i < kp.size() && on; ++i) {
            if (node_idx[kp[i].node] < 0) on = false;
            else if (i && node_idx[kp[i].node] != node_idx[kp[i - 1].node] + 1) on = false;
            len += kp[i].e - kp[i].s;
        }
        if (!on || len == 0) continue;  // null start / end nodes carry no bases
        out[r] = (uint32_t)(node_off[kp[0].node] + (kp[0].s - L.nodes[kp[0].node].s));
    }
    return out;
}

void discover_regions(const HostIndex& H, const std::vector<char>& present, const std::vector<std::vector<uint32_t>>& mlpaths,
                      const int32_t* cov, const DiscoverOpts& o, DiscoverResult& R, std::vector<uint32_t>& cons_start) {
    R = DiscoverResult();
    const uint32_t P = (uint32_t)H.loci.size();
    R.consensus.assign(P, std::string());
    R.coverage.assign(P, {});
    R.local_path.assign(P, {});
    cons_start.assign(H.total_knodes(), UINT32_MAX);
    for (uint32_t l = 0; l < P; ++l) {
        if (l >= present.size() || !present[l]) continue;
        const Locus& L = H.loci[l];
        const std::vector<uint32_t>& lp = R.local_path[l] = local_path_of(L, mlpaths[l]);
        R.consensus[l] = spell_local_path(L, lp);
        R.coverage[l] = ml_path_base_coverage(H, l, mlpaths[l], lp, cov);
        std::vector<std::pair<uint32_t, uint32_t>> iv;
        low_coverage_intervals(R.coverage[l], o.covg_threshold, o.min_len, o.max_len, iv);
        if (iv.empty()) continue;
        const std::vector<uint32_t> cs = knode_consensus_start(L, lp);
        std::copy(cs.begin(), cs.end(), cons_start.begin() + H.knode_base[l]);
        const uint32_t n = (uint32_t)R.coverage[l].size();
        for (auto& p : iv) {
            CandidateRegion c;
            c.locus = l;
            c.start = p.first;
            c.end = p.second;
            c.pad_start = p.first > o.padding ? p.first - o.padding : 0u;
            c.pad_end = std::min(n, p.second + o.padding);
            R.regions.push_back(c);
        }
    }
}

// R = cons[a, b) against the allele by global unit-cost edit distance; the traceback from the end extends an open gap while
// that stays optimal (one indel stays one run), and otherwise prefers the diagonal, then a deletion (a base of R), then an
// insertion.  Every maximal run of non-match columns is one variant.  A run with an empty side is anchored VCF-style by
// the consensus base before it, or by the base after it when it starts at R[0].
void allele_variants(const std::string& cons, uint32_t a, uint32_t b, const std::string& allele, std::vector<DenovoVariant>& out) {
    const std::string R = cons.substr(a, b - a);
    const std::string& A = allele;
    const size_t n = R.size(), m = A.size(), W = m + 1;
    std::vector<uint32_t> D((n + 1) * W);
    for (size_t i = 0; i <= n; ++i) D[i * W] = (uint32_t)i;
    for (size_t j = 0; j <= m; ++j) D[j] = (uint32_t)j;
    for (size_t i = 1; i <= n; ++i)
        for (size_t j = 1; j <= m; ++j)
            D[i * W + j] = std::min({D[(i - 1) * W + j - 1] + (R[i - 1] != A[j - 1]), D[(i - 1) * W + j] + 1, D[i * W + j - 1] + 1});
    struct Col {
        int32_t i, j;  // the base of R / of the allele the column holds, -1 for a gap
    };
    std::vector<Col> cols;
    char op = 0;  // the last column's kind: M(atch or substitution), D(eletion), I(nsertion)
    for (size_t i = n, j = m; i || j;) {
        const bool diag = i && j && D[i * W + j] == D[(i - 1) * W + j - 1] + (R[i - 1] != A[j - 1]);
        const bool del = i && D[i * W + j] == D[(i - 1) * W + j] + 1;
        const bool ins = j && D[i * W + j] == D[i * W + j - 1] + 1;
        if (!((op == 'D' && del) || (op == 'I' && ins))) op = diag ? 'M' : del ? 'D' : 'I';  // else an open gap is extended
        if (op != 'I') --i;
        if (op != 'D') --j;
        cols.push_back({op != 'I' ? (int32_t)i : -1, op != 'D' ? (int32_t)j : -1});
    }
    std::reverse(cols.begin(), cols.end());
    auto match = [&](const Col& c) { return c.i >= 0 && c.j >= 0 && R[c.i] == A[c.j]; };
    uint32_t ri = 0;  // bases of R before the column
    for (size_t c = 0; c < cols.size();) {
        if (match(cols[c])) {
            ++ri;
            ++c;
            continue;
        }
        const uint32_t i0 = ri;
        DenovoVariant v{a + i0 + 1, "", ""};
        for (; c < cols.size() && !match(cols[c]); ++c) {
            if (cols[c].i >= 0) {
                v.ref += R[cols[c].i];
                ++ri;
            }
            if (cols[c].j >= 0) v.alt += A[cols[c].j];
        }
        if (v.ref.empty() || v.alt.empty()) {
            if (i0 == 0 && a + ri < cons.size()) {
                v.ref += cons[a + ri];
                v.alt += cons[a + ri];
            } else if (a + i0 > 0) {
                v.ref.insert(v.ref.begin(), cons[a + i0 - 1]);
                v.alt.insert(v.alt.begin(), cons[a + i0 - 1]);
                --v.pos;
            }
        }
        out.push_back(std::move(v));
    }
}

// pandora 0.10's discover/denovo_paths.txt [P]: the header, then per locus with variants its name, its ML local path (node
// id, PRG-string interval, sequence) and its variants
std::string denovo_paths_text(const HostIndex& H, const std::string& sample, const DiscoverResult& D,
                              const std::vector<std::vector<DenovoVariant>>& variants) {
    size_t n_loci = 0;
    for (const auto& v : variants) n_loci += !v.empty();
    std::string s = "1 samples\nSample " + sample + "\n" + std::to_string(n_loci) + " loci with denovo variants\n";
    for (size_t l = 0; l < variants.size(); ++l) {
        if (variants[l].empty()) continue;
        const Locus& L = H.loci[l];
        s += L.name + "\n" + std::to_string(D.local_path[l].size()) + " nodes\n";
        for (uint32_t n : D.local_path[l])
            s += "(" + std::to_string(n) + " [" + std::to_string(L.nodes[n].s) + ", " + std::to_string(L.nodes[n].e) + ") " + L.node_seq(n) + ")\n";
        s += std::to_string(variants[l].size()) + " variants found\n";
        for (const DenovoVariant& v : variants[l]) s += std::to_string(v.pos) + "\t" + v.ref + "\t" + v.alt + "\n";
    }
    return s;
}

// ============================================================================================
// `pandora index` replacement (SURVEY.md §8f rank 3): drprg runs `pandora index -t T -w W -k K <prg>` when an index is
// built (/root/reference/src/builder.rs:644-659 -> src/lib.rs:479-510) and again per sample when discover changed the PRG
// (src/predict.rs:281-284), and later only checks that the files exist (validate_index, src/predict.rs:400-418:
// `<prg>.k{K}.w{W}.idx` found by find_prg_index_in, src/lib.rs:1222-1231, and the `kmer_prgs/` directory,
// src/builder.rs:257-269).  The loader of this library already computes what those files hold; this writes them in
// pandora's text layout [P, from upstream Index::save / KmerGraph::save; no pandora binary here to read them back]:
//   <prg>.k{K}.w{W}.idx            first line: number of distinct minimizer hashes; then one line per hash:
//                                  hash \t n \t (prg_id, <path>, knode_id, strand) ...   with <path> = n{[s, e)[s, e)...}
//   kmer_prgs/NN/<locus>.k{K}.w{W}.gfa   H line, then per k-mer node "S id path FC:i:0 RC:i:0" followed by its "L" edges
// K-mer node ids are the ranks of this library's graphs (start node 0, terminus last): consistent between the two files.
// ============================================================================================
}  // namespace drprg

#include <sys/stat.h>

#include <cstdio>
#include <fstream>

namespace drprg {

static void append_path(std::string& s, const KPath& kp, uint32_t term_coord, bool is_start, bool is_end) {
    if (kp.empty()) {  // null start [0, 0) / null end [L, L)
        const uint32_t c = is_start ? 0u : term_coord;
        (void)is_end;
        s += "1{[" + std::to_string(c) + ", " + std::to_string(c) + ")}";
        return;
    }
    s += std::to_string(kp.size()) + "{";
    for (auto& sg : kp) s += "[" + std::to_string(sg.s) + ", " + std::to_string(sg.e) + ")";
    s += "}";
}

void write_pandora_index(const HostIndex& H, const std::string& prg_path) {
    const std::string suffix = ".k" + std::to_string(H.k) + ".w" + std::to_string(H.w);
    // ---- the minimizer index
    {
        const std::string path = prg_path + suffix + ".idx";
        std::ofstream f(path);
        if (!f) throw std::runtime_error("cannot write " + path);
        size_t distinct = 0;
        for (size_t i = 0; i < H.records.size(); ++i)
            if (i == 0 || H.records[i - 1].hash != H.records[i].hash) ++distinct;
        std::string out = std::to_string(distinct) + "\n";
        for (size_t i = 0; i < H.records.size();) {
            size_t j = i;
            while (j < H.records.size() && H.records[j].hash == H.records[i].hash) ++j;
            out += std::to_string(H.records[i].hash) + "\t" + std::to_string(j - i);
            for (size_t q = i; q < j; ++q) {
                const Record& r = H.records[q];
                const Locus& L = H.loci[r.prg];
                out += "\t(" + std::to_string(r.prg) + ", ";
                append_path(out, L.kpath[r.knode], L.end_coord(), false, false);
                out += ", " + std::to_string(r.knode) + ", " + std::to_string((int)r.strand) + ")";
            }
            out += "\n";
            if (out.size() > (1u << 20)) {
                f << out;
                out.clear();
            }
            i = j;
        }
        f << out;
        if (!f) throw std::runtime_error("write error on " + path);
    }
    // ---- the k-mer graphs
    const size_t slash = prg_path.find_last_of('/');
    const std::string dir = (slash == std::string::npos ? std::string(".") : prg_path.substr(0, slash)) + "/kmer_prgs";
    mkdir(dir.c_str(), 0755);
    for (size_t l = 0; l < H.loci.size(); ++l) {
        const Locus& L = H.loci[l];
        char sub[16];
        snprintf(sub, sizeof sub, "%02d", (int)(l / 4000) + 1);
        const std::string d = dir + "/" + sub;
        mkdir(d.c_str(), 0755);
        const std::string path = d + "/" + L.name + suffix + ".gfa";
        std::ofstream f(path);
        if (!f) throw std::runtime_error("cannot write " + path);
        std::string out = "H\tVN:Z:1.0\tbn:Z:--linear --singlearr\n";
        const size_t n = L.kpath.size();
        for (size_t r = 0; r < n; ++r) {
            out += "S\t" + std::to_string(r) + "\t";
            append_path(out, L.kpath[r], L.end_coord(), r == 0, r + 1 == n);
            out += "\tFC:i:0\t\tRC:i:0\n";
            for (uint32_t o : L.kout[r]) out += "L\t" + std::to_string(r) + "\t+\t" + std::to_string(o) + "\t+\t0M\n";
        }
        f << out;
        if (!f) throw std::runtime_error("write error on " + path);
    }
}

}  // namespace drprg
