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
//                       the strand of the first hit (get_read_overlap_coordinates / find_hits_inside_path)
// The de-novo assembly itself (pandora's de Bruijn graph walk) runs on the GPU (assemble.cu); this file produces its inputs.
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

void discover_candidates(const HostIndex& H, const std::vector<char>& present, const std::vector<std::vector<uint32_t>>& mlpaths,
                         const int32_t* cov, const std::vector<RetainedHit>& hits, const DiscoverOpts& o, DiscoverResult& R) {
    R = DiscoverResult();
    const uint32_t P = (uint32_t)H.loci.size();
    R.consensus.assign(P, std::string());
    R.coverage.assign(P, {});
    std::vector<std::vector<uint32_t>> cons_start(P);
    std::vector<std::pair<size_t, size_t>> locus_regions(P, {0, 0});
    for (uint32_t l = 0; l < P; ++l) {
        if (l >= present.size() || !present[l]) continue;
        const Locus& L = H.loci[l];
        const std::vector<uint32_t> lp = local_path_of(L, mlpaths[l]);
        R.consensus[l] = spell_local_path(L, lp);
        R.coverage[l] = ml_path_base_coverage(H, l, mlpaths[l], lp, cov);
        cons_start[l] = knode_consensus_start(L, lp);
        std::vector<std::pair<uint32_t, uint32_t>> iv;
        low_coverage_intervals(R.coverage[l], o.covg_threshold, o.min_len, o.max_len, iv);
        locus_regions[l].first = R.regions.size();
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
        locus_regions[l].second = R.regions.size();
    }
    // reads over the regions: hits arrive grouped by read (any read order), sorted (prg, strand, start, k-mer node) within
    struct Acc { uint32_t n = 0, lo = 0, hi = 0; uint8_t fwd = 0; };
    std::vector<std::vector<ReadCoordinate>> per_region(R.regions.size());
    std::vector<Acc> acc;
    size_t i = 0;
    while (i < hits.size()) {
        size_t j = i;
        while (j < hits.size() && hits[j].read == hits[i].read && hits[j].prg == hits[i].prg) ++j;
        const uint32_t l = hits[i].prg;
        const size_t r0 = l < P ? locus_regions[l].first : 0, r1 = l < P ? locus_regions[l].second : 0;
        if (r1 > r0) {
            acc.assign(r1 - r0, Acc());
            for (size_t q = i; q < j; ++q) {
                const uint32_t cs = hits[q].knode < cons_start[l].size() ? cons_start[l][hits[q].knode] : UINT32_MAX;
                if (cs == UINT32_MAX) continue;
                for (size_t rg = r0; rg < r1; ++rg) {
                    const CandidateRegion& c = R.regions[rg];
                    if (cs < c.pad_start || cs + H.k > c.pad_end) continue;
                    Acc& a = acc[rg - r0];
                    if (a.n == 0) {
                        a.lo = hits[q].start;
                        a.fwd = hits[q].fwd;
                    }
                    a.lo = std::min(a.lo, hits[q].start);
                    a.hi = std::max(a.hi, hits[q].start + H.k);
                    ++a.n;
                }
            }
            for (size_t rg = r0; rg < r1; ++rg)
                if (acc[rg - r0].n >= o.min_hits) per_region[rg].push_back(ReadCoordinate{hits[i].read, acc[rg - r0].lo, acc[rg - r0].hi, acc[rg - r0].fwd});
        }
        i = j;
    }
    for (size_t rg = 0; rg < R.regions.size(); ++rg) {
        auto& v = per_region[rg];
        std::sort(v.begin(), v.end(), [](const ReadCoordinate& a, const ReadCoordinate& b) { return a.read < b.read; });
        R.regions[rg].read_off = R.reads.size();
        R.regions[rg].n_reads = (uint32_t)v.size();
        R.reads.insert(R.reads.end(), v.begin(), v.end());
    }
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
