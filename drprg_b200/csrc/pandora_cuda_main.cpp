// `pandora`-argv-compatible front end of libdrprg_cuda: lets an unmodified drprg use the GPU path through its
// own -p/--pandora option (/root/reference/src/predict.rs:137-144).  `map` (the argv built at
// /root/reference/src/lib.rs:594-617 + src/predict.rs:288-294) runs on the GPU; `index` (argv of src/lib.rs:479-510,
// `-t N -w W -k K <prg>` at src/predict.rs:283 and src/builder.rs:644-657) is served by the library's own index builder,
// which writes <prg>.kK.wW.idx and kmer_prgs/ in pandora's layout (no GPU needed); `discover` (argv of src/lib.rs:513-578)
// maps the one sample of its query file on the GPU, assembles its candidate regions there and writes
// OUT/denovo_paths.txt; every other sub-command is handed to the real pandora named by $DRPRG_REAL_PANDORA.
#include <unistd.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <filesystem>
#include <fstream>
#include <string>
#include <system_error>
#include <vector>

#include "../../include/drprg_cuda.h"

static bool mkdirs(const std::string& dir) {  // pandora creates its output directory; no shell (the path is user input)
    std::error_code ec;
    std::filesystem::create_directories(dir, ec);
    if (ec) fprintf(stderr, "pandora_cuda: cannot create %s: %s\n", dir.c_str(), ec.message().c_str());
    return !ec;
}

// drprg's argv: discover -g G --max-covg M -v -o OUT -t T -w W -k K -c C [-I] [-K] <prg> <query.tsv>.  The query file holds
// one `sample<TAB>reads` line (drprg writes one); a relative reads path is taken from the query file's directory [P].
static int discover_main(int argc, char** argv) {
    drprg_map_opts o{};
    o.threads = 1;
    o.min_cluster_size = 10;
    o.genome_size = 5000000;  // pandora defaults; drprg always passes -g, -c
    o.max_covg = 300;
    o.genotyping_error_rate = 0.01;
    uint32_t w = 14, k = 15;
    std::string outdir = "pandora";
    std::vector<std::string> pos;
    for (int i = 2; i < argc; ++i) {
        std::string a = argv[i];
        auto val = [&]() -> const char* { return (i + 1 < argc) ? argv[++i] : ""; };
        if (a == "-v" || a == "-vv") continue;
        else if (a == "-o" || a == "--outdir") outdir = val();
        else if (a == "-g" || a == "--genome-size") o.genome_size = (uint32_t)strtoul(val(), nullptr, 10);
        else if (a == "--max-covg") o.max_covg = (uint32_t)strtoul(val(), nullptr, 10);
        else if (a == "-t" || a == "--threads") o.threads = (uint32_t)atoi(val());
        else if (a == "-w") w = (uint32_t)atoi(val());
        else if (a == "-k") k = (uint32_t)atoi(val());
        else if (a == "-c" || a == "--min-cluster-size") o.min_cluster_size = (uint32_t)atoi(val());
        else if (a == "-I" || a == "--illumina") o.illumina = 1;
        else if (a == "-K" || a == "--debugging-files") o.debug = 1;  // accepted; no extra files are written
        else if (!a.empty() && a[0] == '-') {
            fprintf(stderr, "pandora_cuda discover: unsupported option %s\n", a.c_str());
            return 2;
        } else pos.push_back(a);
    }
    if (pos.size() != 2) {
        fprintf(stderr, "pandora_cuda discover: need <prg> <query.tsv>\n");
        return 2;
    }
    std::ifstream q(pos[1]);
    if (!q) {
        fprintf(stderr, "pandora_cuda discover: cannot read %s\n", pos[1].c_str());
        return 1;
    }
    std::vector<std::string> lines;
    for (std::string l; std::getline(q, l);)
        if (l.find_first_not_of(" \t\r") != std::string::npos) lines.push_back(l);
    if (lines.size() != 1) {
        fprintf(stderr, "pandora_cuda discover: %s lists %zu samples; exactly one is supported\n", pos[1].c_str(), lines.size());
        return 2;
    }
    std::string line = lines[0];
    if (!line.empty() && line.back() == '\r') line.pop_back();
    const size_t tab = line.find('\t');
    if (tab == std::string::npos || line.find('\t', tab + 1) != std::string::npos) {
        fprintf(stderr, "pandora_cuda discover: %s: expected `sample<TAB>reads`\n", pos[1].c_str());
        return 2;
    }
    const std::string sample = line.substr(0, tab);
    const std::filesystem::path reads = std::filesystem::path(pos[1]).parent_path() / line.substr(tab + 1);
    if (!mkdirs(outdir)) return 1;
    const int device = getenv("DRPRG_CUDA_DEVICE") ? atoi(getenv("DRPRG_CUDA_DEVICE")) : 0;
    drprg_index* idx = nullptr;
    if (drprg_cuda_index_load(pos[0].c_str(), w, k, device, &idx) != 0) {
        fprintf(stderr, "pandora_cuda: %s\n", drprg_cuda_last_error());
        return 1;
    }
    drprg_discover_stats st{};
    const int rc = drprg_cuda_discover(idx, sample.c_str(), reads.c_str(), outdir.c_str(), &o, nullptr, nullptr, &st);
    if (rc != 0) fprintf(stderr, "pandora_cuda discover: %s\n", drprg_cuda_last_error());
    else printf("pandora_cuda discover: %llu reads, %u regions, %u loci with %u variants, %.1f ms\n", (unsigned long long)st.n_reads,
                st.n_regions, st.n_loci_with_variants, st.n_variants, st.ms_total);
    drprg_cuda_index_free(idx);
    return rc ? 1 : 0;
}

int main(int argc, char** argv) {
    if (argc < 2) {
        fprintf(stderr, "usage: pandora_cuda map [pandora map options] <prg> <reads> | pandora_cuda index [-t N] [-w W] [-k K] <prg> | "
                        "pandora_cuda discover [-g G] [--max-covg M] [-o OUT] [-t N] [-w W] [-k K] [-c C] [-I] [-K] <prg> <query.tsv>\n");
        return 2;
    }
    if (strcmp(argv[1], "index") == 0) {
        uint32_t w = 14, k = 15;  // pandora's defaults; drprg always passes -w and -k
        std::string prg;
        for (int i = 2; i < argc; ++i) {
            std::string a = argv[i];
            auto val = [&]() -> const char* { return (i + 1 < argc) ? argv[++i] : ""; };
            if (a == "-w") w = (uint32_t)atoi(val());
            else if (a == "-k") k = (uint32_t)atoi(val());
            else if (a == "-t" || a == "--threads") val();
            else if (a == "-v" || a == "-vv") continue;
            else if (!a.empty() && a[0] == '-') {
                fprintf(stderr, "pandora_cuda index: unsupported option %s\n", a.c_str());
                return 2;
            } else prg = a;
        }
        if (prg.empty()) {
            fprintf(stderr, "usage: pandora_cuda index [-t N] [-w W] [-k K] <prg>\n");
            return 2;
        }
        drprg_index* idx = nullptr;
        if (drprg_cuda_index_load(prg.c_str(), w, k, -1 /* host-only handle */, &idx) != 0 || drprg_cuda_index_write(idx, prg.c_str()) != 0) {
            fprintf(stderr, "pandora_cuda index: %s\n", drprg_cuda_last_error());
            if (idx) drprg_cuda_index_free(idx);
            return 1;
        }
        drprg_cuda_index_free(idx);
        return 0;
    }
    if (strcmp(argv[1], "discover") == 0) return discover_main(argc, argv);
    if (strcmp(argv[1], "map") != 0) {
        const char* real = getenv("DRPRG_REAL_PANDORA");
        if (!real) {
            fprintf(stderr, "pandora_cuda: `map`, `index` and `discover` are served here; set DRPRG_REAL_PANDORA for `%s`\n", argv[1]);
            return 2;
        }
        argv[0] = const_cast<char*>(real);
        execv(real, argv);
        perror("pandora_cuda: exec of DRPRG_REAL_PANDORA failed");
        return 127;
    }
    drprg_map_opts o{};
    o.threads = 1;
    o.min_cluster_size = 10;
    o.genome_size = 5000000;  // pandora defaults; drprg always passes -g, -c, --gt-conf
    o.max_covg = 300;
    o.gt_conf = 1;
    o.genotyping_error_rate = 0.01;
    uint32_t w = 14, k = 15;
    std::string outdir = "pandora", vcf_refs;
    std::vector<std::string> pos;
    for (int i = 2; i < argc; ++i) {
        std::string a = argv[i];
        auto val = [&]() -> const char* { return (i + 1 < argc) ? argv[++i] : ""; };
        if (a == "--genotype" || a == "--local" || a == "-v" || a == "-vv") continue;
        else if (a == "--gt-conf" || a == "-G") o.gt_conf = atof(val());
        else if (a == "-o" || a == "--outdir") outdir = val();
        else if (a == "-g" || a == "--genome-size") o.genome_size = (uint32_t)strtoul(val(), nullptr, 10);
        else if (a == "--max-covg") o.max_covg = (uint32_t)strtoul(val(), nullptr, 10);
        else if (a == "--vcf-refs") vcf_refs = val();
        else if (a == "-t" || a == "--threads") o.threads = (uint32_t)atoi(val());
        else if (a == "-w") w = (uint32_t)atoi(val());
        else if (a == "-k") k = (uint32_t)atoi(val());
        else if (a == "-c" || a == "--min-cluster-size") o.min_cluster_size = (uint32_t)atoi(val());
        else if (a == "-m" || a == "--max-diff") o.max_diff = (uint32_t)atoi(val());
        else if (a == "-e" || a == "--error-rate") o.error_rate = atof(val());
        else if (a == "-E" || a == "--gt-error-rate") o.genotyping_error_rate = atof(val());
        else if (a == "-I" || a == "--illumina") o.illumina = 1;
        else if (a == "-K" || a == "--debugging-files") o.debug = 1;
        else if (!a.empty() && a[0] == '-') {
            fprintf(stderr, "pandora_cuda: unsupported option %s\n", a.c_str());
            return 2;
        } else pos.push_back(a);
    }
    if (pos.size() != 2) {
        fprintf(stderr, "pandora_cuda: need <prg> <reads>\n");
        return 2;
    }
    if (!mkdirs(outdir)) return 1;
    const int device = getenv("DRPRG_CUDA_DEVICE") ? atoi(getenv("DRPRG_CUDA_DEVICE")) : 0;
    drprg_index* idx = nullptr;
    if (drprg_cuda_index_load(pos[0].c_str(), w, k, device, &idx) != 0) {
        fprintf(stderr, "pandora_cuda: %s\n", drprg_cuda_last_error());
        return 1;
    }
    drprg_map_stats st{};
    int rc = drprg_cuda_map_genotype(idx, pos[1].c_str(), vcf_refs.empty() ? nullptr : vcf_refs.c_str(), outdir.c_str(), &o, &st);
    if (rc != 0) fprintf(stderr, "pandora_cuda: %s\n", drprg_cuda_last_error());
    else printf("pandora_cuda map: %llu reads, %u records, %.1f ms (ingest %.1f, map %.1f, genotype %.1f)\n",
                (unsigned long long)st.n_reads, st.n_records, st.ms_total, st.ms_ingest, st.ms_map, st.ms_genotype);
    drprg_cuda_index_free(idx);
    return rc ? 1 : 0;
}
