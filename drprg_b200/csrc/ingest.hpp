// FASTQ ingest (SURVEY.md §8f rank 2): framed on the host, sequence lines to the GPU, 2-bit packed there (ingest.cu).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "cuda_owned.hpp"

namespace drprg {

// device buffers from g_pool; hidden like the owner types it holds (library internal)
struct __attribute__((visibility("hidden"))) IngestResult {
    PoolBuf<uint32_t> words;
    PoolBuf<uint64_t> word_off;  // empty with a fixed stride
    PoolBuf<uint32_t> lens;
    uint32_t stride_words = 0, max_len = 0, first_read_len = 0;
    uint64_t n_reads = 0, total_bases = 0, n_dropped = 0;
};

struct TextSource;
// Host-framed ingest of one piece of FASTQ text (a whole file, or a wave of a large one that starts and ends at record
// starts): only the sequence lines are uploaded (fastq_frame.cpp), then packed on the device.  false = not strict 4-line
// FASTQ (the caller uses the host parser); throws on IO errors.  The text must be smaller than 8 GB (32-bit offsets into
// the sequence buffer).
bool ingest_fastq_text(const TextSource& src, int device, uint32_t threads, IngestResult& out, cudaStream_t st);

}  // namespace drprg
