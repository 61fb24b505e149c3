// Ingest of 4-line FASTQ (plain, or gzip inflated into host memory), SURVEY.md §8f rank 2: the reads file that `drprg
// predict` hands to the map step (/root/reference/src/predict.rs:166-170, 288-294) becomes a 2-bit packed batch in HBM.
// The record structure is found on the HOST (fastq_frame.cpp), only the sequence lines and a (start, length) table cross
// PCIe, and the device packs:
//   pack_stride/ragged  ASCII -> 2-bit words (first base in the top bits), non-ACGT reads flagged
//   finish_lens         lens[r] = 0 for a flagged read (pandora drops it), dropped-read count
// Anything that is not strict 4-line FASTQ (FASTA, wrapped records, blank lines, damaged records) is left to the general
// host parser (load_reads_packed), which produces the same packed layout.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

#include "fastq_frame.hpp"
#include "genotype_host.hpp"
#include "ingest.hpp"
#include "kernels.cuh"

namespace drprg {
namespace {

struct Staging {  // process-wide grow-only pinned and device buffers (one ingest at a time)
    std::mutex m;
    int device = -1;
    DBuf<char> d_text;      // the sequence lines
    DBuf<uint32_t> d_rec;   // per record: sequence start | raw length | bad flag (3 columns of d_rec.cap / 3)
    DBuf<unsigned long long> d_scalars;  // [4] dropped reads (finish_lens_kernel)
    PinnedBuf<unsigned long long> h_scalars;
    PinnedBuf<char> pinned_seq;  // the sequence lines, framed on the host
    PinnedBuf<uint32_t> h_rec;   // sequence start | length per read (2 columns of h_rec.cap / 2)
};
// never destroyed: static teardown may run after the CUDA runtime has been unloaded
Staging& g_stage = *new Staging;

__device__ __forceinline__ uint32_t code4_dev(uint32_t c) {
    c &= 0xdfu;  // fold case (only letters matter)
    return c == 'A' ? 0u : c == 'C' ? 1u : c == 'G' ? 2u : c == 'T' ? 3u : 4u;
}

__device__ __forceinline__ uint32_t pack_word(const char* __restrict__ s, uint32_t n, uint32_t& bad) {
    uint32_t word = 0;
#pragma unroll 4
    for (uint32_t i = 0; i < n; ++i) {
        const uint32_t c = code4_dev((uint8_t)s[i]);
        bad |= c >> 2;
        word |= (c & 3u) << (30 - 2 * i);
    }
    return word;
}

// fixed stride: one thread per (read, word)
__global__ void pack_stride_kernel(const char* __restrict__ text, const uint32_t* __restrict__ seq_start,
                                   const uint32_t* __restrict__ raw_len, uint64_t n_records, uint32_t stride,
                                   uint32_t* __restrict__ words, uint32_t* __restrict__ bad_flag) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_records * stride) return;
    const uint64_t r = i / stride;
    const uint32_t j = (uint32_t)(i - r * stride);
    const uint32_t len = raw_len[r];
    uint32_t word = 0, bad = 0;
    if (j * 16 < len) word = pack_word(text + seq_start[r] + j * 16, min(16u, len - j * 16), bad);
    words[i] = word;
    if (bad) bad_flag[r] = 1u;  // every writer stores the same value
}

// ragged layout (long reads): one warp per read
__global__ void pack_ragged_kernel(const char* __restrict__ text, const uint32_t* __restrict__ seq_start,
                                   const uint32_t* __restrict__ raw_len, uint64_t n_records,
                                   const unsigned long long* __restrict__ word_off, uint32_t* __restrict__ words,
                                   uint32_t* __restrict__ bad_flag) {
    const uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= n_records) return;
    const uint32_t lane = threadIdx.x & 31, len = raw_len[r], nw = (len + 15) >> 4;
    const char* s = text + seq_start[r];
    uint32_t* w = words + word_off[r];
    uint32_t bad = 0;
    for (uint32_t j = lane; j < nw; j += 32) w[j] = pack_word(s + j * 16, min(16u, len - j * 16), bad);
    if (__any_sync(0xffffffffu, bad != 0) && lane == 0) bad_flag[r] = 1u;
}

__global__ void finish_lens_kernel(const uint32_t* __restrict__ raw_len, const uint32_t* __restrict__ bad_flag, uint64_t n,
                                   uint32_t* __restrict__ lens, unsigned long long* __restrict__ scalars) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool dropped = false;
    if (r < n) {
        const uint32_t len = raw_len[r];
        dropped = bad_flag[r] != 0u && len > 0;
        lens[r] = bad_flag[r] ? 0u : len;
    }
    const uint32_t b = __ballot_sync(0xffffffffu, dropped);
    if ((threadIdx.x & 31) == 0 && b) atomicAdd(scalars + 4, (unsigned long long)__popc(b));
}

// records (sequence start, raw length in g_stage.d_rec) -> 2-bit words, lengths (0 = dropped), dropped-read count
// h_lens: the same raw lengths on the host, from which the ragged layout's word offsets are summed
void pack_records(const char* text, uint64_t n, uint32_t max_len, uint64_t total_bases, uint32_t first_len, IngestResult& out,
                  cudaStream_t st, int device, const uint32_t* h_lens) {
    const size_t rec_cap = g_stage.d_rec.cap / 3;
    uint32_t *d_start = g_stage.d_rec.p, *d_rawlen = d_start + rec_cap, *d_bad = d_start + 2 * rec_cap;
    const unsigned rb = (unsigned)((n + 255) / 256);
    CK(cudaMemsetAsync(d_bad, 0, n * 4, st));
    CK(cudaMemsetAsync(g_stage.d_scalars.p + 4, 0, sizeof(unsigned long long), st));
    out.max_len = max_len;
    out.total_bases = total_bases;
    out.first_read_len = first_len;
    out.n_reads = n;
    out.lens = pool_get<uint32_t>(std::max<uint64_t>(1, n) * 4, device);
    if (out.max_len <= SHORT_READ_MAX) {
        uint32_t stride = std::max(1u, (out.max_len + 15) / 16);
        stride += stride & 1u;  // even: every read starts 8-byte aligned (wide loads in the screen kernel)
        out.stride_words = stride;
        out.words = pool_get<uint32_t>((n * (uint64_t)stride + 2) * 4, device);
        const uint64_t items = n * (uint64_t)stride;
        pack_stride_kernel<<<(unsigned)((items + 255) / 256), 256, 0, st>>>(text, d_start, d_rawlen, n, stride, out.words.get(), d_bad);
    } else {
        out.word_off = pool_get<uint64_t>((n + 1) * 8, device);
        unsigned long long total_words = 0;
        std::vector<uint64_t> off(n + 1);
        for (uint64_t r = 0; r < n; ++r) {
            off[r] = total_words;
            total_words += (h_lens[r] + 15u) >> 4;
        }
        off[n] = total_words;
        CK(cudaMemcpyAsync(out.word_off.get(), off.data(), (n + 1) * 8, cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st));  // `off` dies with this scope
        out.words = pool_get<uint32_t>((total_words + 2) * 4, device);
        pack_ragged_kernel<<<(unsigned)((n * 32 + 255) / 256), 256, 0, st>>>(text, d_start, d_rawlen, n,
                                                                            (const unsigned long long*)out.word_off.get(), out.words.get(), d_bad);
    }
    finish_lens_kernel<<<rb, 256, 0, st>>>(d_rawlen, d_bad, n, out.lens.get(), g_stage.d_scalars.p);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(g_stage.h_scalars.p, g_stage.d_scalars.p, 5 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    out.n_dropped = g_stage.h_scalars.p[4];
}

}  // namespace

// The text (a plain file read in pieces by the pool threads, or a gzip file already inflated into host memory) is cut into
// slices at record starts; every slice is framed by one thread (fastq_frame.cpp) straight into its own part of a pinned
// buffer — the sequence lines of the slice [lo, hi) go to offset lo / 2, which cannot collide with the next slice because
// a record's sequence is less than half of its bytes — and the thread that framed a slice also queues its H2D copy, so
// the copies overlap the framing of the other slices.  Then (start, length) of every read is uploaded and the pack
// kernels run.  false = not strict 4-line FASTQ (nothing is left behind; the caller goes on with the host parser).
bool ingest_fastq_text(const TextSource& src, int device, uint32_t threads, IngestResult& out, cudaStream_t st) {
    out = IngestResult();
    std::lock_guard<std::mutex> lock(g_stage.m);
    static const bool timing = getenv("DRPRG_TIMING") != nullptr;
    const double t0 = now_ms();
    if (src.size < 8 || src.size / 2 + 64 >= 0xfff00000ull) return false;  // 32-bit sequence offsets
    CK(cudaSetDevice(device));
    const size_t seq_bytes = src.size / 2 + 64;
    g_stage.pinned_seq.reserve(seq_bytes, seq_bytes + seq_bytes / 8 + (1u << 20));
    if (device != g_stage.device) {  // device buffers belong to one device; switching devices starts over
        g_stage.d_text.release();
        g_stage.d_scalars.release();
        g_stage.d_rec.release();
        g_stage.device = device;
    }
    g_stage.d_scalars.reserve(8, 8);
    g_stage.h_scalars.reserve(8, 8);
    // every ingest writes the text buffer afresh: nothing to carry over
    g_stage.d_text.reserve(seq_bytes, seq_bytes + seq_bytes / 8 + (1u << 20));
    char* const pinned = g_stage.pinned_seq.p;
    char* const d_text = g_stage.d_text.p;
    std::vector<FramedSlice> sl;
    std::atomic<bool> cuda_failed{false};
    bool is_fastq = false;
    try {
        is_fastq = fastq_frame_text(src, threads, pinned, sl, [&](size_t at, size_t bytes) {
            if (cudaSetDevice(device) != cudaSuccess ||
                cudaMemcpyAsync(d_text + at, pinned + at, bytes, cudaMemcpyHostToDevice, st) != cudaSuccess) {
                cuda_failed = true;
                return false;
            }
            return true;
        });
    } catch (...) {
        cudaStreamSynchronize(st);  // copies of the slices framed so far still read the pinned buffer
        throw;
    }
    if (!is_fastq || cuda_failed) {
        cudaStreamSynchronize(st);  // the queued copies read the pinned buffer
        cudaGetLastError();
        if (cuda_failed) throw std::runtime_error("reads file: upload error");
        return false;
    }
    const size_t S = sl.size();
    const double t1 = now_ms();
    // ---- totals, then (start, length) of every read to the device
    FrameStats T;
    std::vector<size_t> first(S + 1, 0);
    bool have_first = false;
    for (size_t s = 0; s < S; ++s) {
        const FrameStats& z = sl[s].st;
        first[s + 1] = first[s] + z.n_reads;
        if (z.n_reads && !have_first) {
            T.first_len = z.first_len;
            have_first = true;
        }
        T.max_len = std::max(T.max_len, z.max_len);
        T.total_bases += z.total_bases;
    }
    const uint64_t n = first[S];
    if (n == 0) {
        cudaStreamSynchronize(st);
        return false;
    }
    if (n > 0xfffffff0ull) throw std::runtime_error("more than 2^32 reads in one sample");
    // grow-only record tables: cudaMalloc / cudaFree per sample cost more than the kernels
    g_stage.h_rec.reserve(2 * n, 2 * (n + n / 8 + 1024));
    g_stage.d_rec.reserve(3 * n, 3 * (n + n / 8 + 1024));
    uint32_t* h_start = g_stage.h_rec.p;
    uint32_t* h_len = h_start + g_stage.h_rec.cap / 2;
    parallel_for(S, [&](size_t s) {
        const size_t k = sl[s].lens.size();
        if (!k) return;
        memcpy(h_start + first[s], sl[s].starts.data(), k * 4);
        memcpy(h_len + first[s], sl[s].lens.data(), k * 4);
    }, std::max<size_t>(1, std::min<size_t>(threads, 8)));
    CK(cudaMemcpyAsync(g_stage.d_rec.p, h_start, n * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(g_stage.d_rec.p + g_stage.d_rec.cap / 3, h_len, n * 4, cudaMemcpyHostToDevice, st));
    const double t2 = now_ms();
    pack_records(d_text, n, T.max_len, T.total_bases, T.first_len, out, st, device, h_len);
    if (timing)
        fprintf(stderr, "[drprg-cuda] ingest (host-framed): %.1f MB text in %zu slices, frame + queue H2D %.2f ms, record table %.2f ms, "
                        "upload tail + pack %.2f ms\n", src.size / 1e6, S, t1 - t0, t2 - t1, now_ms() - t2);
    return true;
}

}  // namespace drprg
