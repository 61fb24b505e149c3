// FASTQ ingest (SURVEY.md §8f rank 2): framed on the host, sequence lines to the GPU, 2-bit packed there (ingest.cu).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <functional>

namespace drprg {

struct IngestResult {  // device buffers from cudaMalloc, owned by the caller
    uint32_t* d_words = nullptr;
    uint64_t* d_word_off = nullptr;  // nullptr with a fixed stride
    uint32_t* d_lens = nullptr;
    size_t b_words = 0, b_off = 0, b_lens = 0;
    uint32_t stride_words = 0, max_len = 0, first_read_len = 0;
    uint64_t n_reads = 0, total_bases = 0, n_dropped = 0;
};

struct TextSource;
// Host-framed ingest of one piece of FASTQ text (a whole file, or a wave of a large one that starts and ends at record
// starts): only the sequence lines are uploaded (fastq_frame.cpp), then packed on the device.  false = not strict 4-line
// FASTQ (the caller uses the host parser); throws on IO errors.  The text must be smaller than 8 GB (32-bit offsets into
// the sequence buffer).  `alloc` supplies the output buffers (e.g. from the caller's buffer pool); default: cudaMalloc.
bool ingest_fastq_text(const TextSource& src, int device, uint32_t threads, IngestResult& out, cudaStream_t st,
                       const std::function<void*(size_t)>& alloc = nullptr);

}  // namespace drprg
