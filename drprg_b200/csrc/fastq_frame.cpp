// Host-side FASTQ framing for the ingest pipeline (SURVEY.md §8f rank 2; the reads file of
// /root/reference/src/predict.rs:166-170, 288-294).  A 150 bp FASTQ record is ~315 bytes of which only the 150 sequence
// bytes matter to the map step; sending the whole text over PCIe made the drop-in call transfer-bound.  The host threads
// therefore find the record structure (newline bitmasks, 32 bytes per AVX2 step) and copy ONLY the sequence lines into
// the pinned staging buffer; packing to 2 bits, the non-ACGT check and everything else stay on the device.
#include "fastq_frame.hpp"

#include <immintrin.h>

#include <unistd.h>

#include <atomic>
#include <cstring>
#include <stdexcept>

#include "genotype_host.hpp"  // parallel_for_io

namespace drprg {
namespace {

}  // namespace

size_t fastq_next_record(const char* t, size_t n, size_t p) {
    if (p == 0) return 0;
    if (p >= n) return n;
    // start of the line after the one containing p - 1
    const char* h = (const char*)memchr(t + p - 1, '\n', n - (p - 1));
    if (!h) return n;
    size_t q = (size_t)(h - t) + 1;
    while (q < n) {
        const char* e1 = (const char*)memchr(t + q, '\n', n - q);
        if (!e1) return n;
        if (t[q] == '@') {  // a header line is followed, two lines later, by a '+' line
            const size_t l2 = (size_t)(e1 - t) + 1;
            const char* e2 = l2 < n ? (const char*)memchr(t + l2, '\n', n - l2) : nullptr;
            if (e2 && (size_t)(e2 - t) + 1 < n && e2[1] == '+') return q;
        }
        q = (size_t)(e1 - t) + 1;
    }
    return n;
}

__attribute__((target("avx2"))) static void stream_lines_avx2(char* dst, const char* src, size_t n_lines) {
    for (size_t i = 0; i < n_lines; ++i) {
        const __m256i a = _mm256_load_si256((const __m256i*)(src + 64 * i));
        const __m256i b = _mm256_load_si256((const __m256i*)(src + 64 * i + 32));
        _mm256_stream_si256((__m256i*)(dst + 64 * i), a);
        _mm256_stream_si256((__m256i*)(dst + 64 * i + 32), b);
    }
}

// stage_ mirrors the destination's position inside a 64-byte line: byte k of the pending output sits at
// stage_[phase_off_ + k], so whole destination lines are whole (aligned) staging lines
void FastqFramer::flush(bool all) {
    static const bool avx2 = __builtin_cpu_supports("avx2");
    char* dst = out_ + flushed_;
    const char* src = stage_ + phase_off_;
    size_t n = staged_;
    if (!n) return;
    size_t done = 0;
    if (avx2 && n >= 128) {
        const size_t head = phase_off_ ? 64 - phase_off_ : 0;  // up to the first line boundary: ordinary stores
        if (head) memcpy(dst, src, head);
        const size_t lines = (n - head) / 64;
        stream_lines_avx2(dst + head, src + head, lines);
        done = head + lines * 64;
    }
    if (all) {
        memcpy(dst + done, src + done, n - done);
        done = n;
        _mm_sfence();  // the streamed lines are globally visible before the slice's H2D copy is queued
    }
    // keep the unflushed tail at its line phase
    const size_t left = n - done;
    flushed_ += done;
    const size_t new_phase = (size_t)((uintptr_t)(out_ + flushed_) & 63u);
    if (left) memmove(stage_ + new_phase, src + done, left);
    phase_off_ = new_phase;
    staged_ = left;
}

inline void FastqFramer::put(const char* p, size_t len) {
    if (flushed_ == 0 && staged_ == 0) phase_off_ = (size_t)((uintptr_t)out_ & 63u);
    while (len) {
        const size_t room = STAGE - staged_;
        const size_t take = len < room ? len : room;
        memcpy(stage_ + phase_off_ + staged_, p, take);
        staged_ += take;
        p += take;
        len -= take;
        if (staged_ == STAGE) flush(false);
    }
}

inline bool FastqFramer::line(const char* ls, const char* le) {
    switch (phase_) {
        case 0:
            if (le == ls || *ls != '@') return false;  // blank line or broken framing
            break;
        case 1: {
            size_t len = (size_t)(le - ls);
            if (len && le[-1] == '\r') --len;
            if (fill_ + len > cap_ || base_ + fill_ + len > 0xfffffff0ull) return false;
            put(ls, len);
            starts_.push_back(base_ + (uint32_t)fill_);
            fill_ += len;
            seq_len_ = len;
            break;
        }
        case 2:
            if (le == ls || *ls != '+') return false;
            plus_plain_ = (le - ls == 1);
            break;
        default: {
            size_t len = (size_t)(le - ls);
            if (len && le[-1] == '\r') --len;
            if (len != seq_len_) return false;  // wrapped or damaged record
            lens_.push_back((uint32_t)seq_len_);
            if (S_.n_reads == 0) S_.first_len = (uint32_t)seq_len_;
            ++S_.n_reads;
            S_.max_len = std::max<uint32_t>(S_.max_len, (uint32_t)seq_len_);
            S_.min_len = std::min<uint32_t>(S_.min_len, (uint32_t)seq_len_);
            S_.total_bases += seq_len_;
            S_.seq_bytes = fill_;
            plain_prev_ = plus_plain_;
            break;
        }
    }
    phase_ = (phase_ + 1) & 3u;
    return true;
}

// number of '\n' in p[0..n); reads up to 31 bytes past p + n (the callers leave that much readable text behind the span)
__attribute__((target("avx2,popcnt"))) static inline uint32_t count_newlines_avx2(const char* p, size_t n) {
    const __m256i needle = _mm256_set1_epi8('\n');
    uint32_t c = 0;
    size_t i = 0;
    for (; i + 32 <= n; i += 32)
        c += (uint32_t)__builtin_popcount((uint32_t)_mm256_movemask_epi8(_mm256_cmpeq_epi8(_mm256_loadu_si256((const __m256i*)(p + i)), needle)));
    if (i < n) {
        const uint32_t m = (uint32_t)_mm256_movemask_epi8(_mm256_cmpeq_epi8(_mm256_loadu_si256((const __m256i*)(p + i)), needle));
        c += (uint32_t)__builtin_popcount(m & (uint32_t)((1ull << (n - i)) - 1ull));
    }
    return c;
}

bool FastqFramer::feed(const char* p, size_t n, size_t& used) {
    static const bool avx2 = __builtin_cpu_supports("avx2") && __builtin_cpu_supports("popcnt");
    size_t at = 0;  // always a line start
    for (;;) {
        // A record whose sequence is as long as the previous one's (every Illumina file): after the header line the
        // other three line ends are where they were last time; one vector pass confirms that the span holds exactly those
        // three newlines, so the record is framed without looking for its lines one by one.
        if (avx2 && phase_ == 0 && plain_prev_ && at < n) {
            const char* r = p + at;
            const char* he = (const char*)memchr(r, '\n', n - at);
            if (!he) break;
            const size_t L = seq_len_, h = (size_t)(he - r);  // r[h] = end of the header line
            const size_t n2 = h + 1 + L, n3 = n2 + 2, n4 = n3 + 1 + L;
            if (at + n4 + 33 <= n && h >= 1 && r[0] == '@' && r[n2] == '\n' && r[n2 + 1] == '+' && r[n3] == '\n' && r[n4] == '\n' &&
                r[h - 1] != '\r' && (L == 0 || (r[n2 - 1] != '\r' && r[n4 - 1] != '\r')) && count_newlines_avx2(r + h + 1, n4 - h) == 3 &&
                fill_ + L <= cap_ && base_ + fill_ + L <= 0xfffffff0ull) {
                put(r + h + 1, L);
                starts_.push_back(base_ + (uint32_t)fill_);
                lens_.push_back((uint32_t)L);
                fill_ += L;
                ++S_.n_reads;
                S_.total_bases += L;
                S_.seq_bytes = fill_;
                at += n4 + 1;
                continue;
            }
        }
        if (at >= n) break;
        const char* le = (const char*)memchr(p + at, '\n', n - at);
        if (!le) break;
        if (!line(p + at, le)) return false;
        at = (size_t)(le - p) + 1;
    }
    used = at;
    return true;
}

bool FastqFramer::finish(const char* p, size_t n, bool end_of_file) {
    if (n) {  // text after the last newline: the final line of a file without a trailing newline
        if (!end_of_file) return false;
        if (!line(p, p + n)) return false;
    }
    flush(true);
    return phase_ == 0;  // the slice must end on a record boundary
}

size_t TextSource::read(char* buf, size_t at, size_t n) const {
    n = at < size ? std::min(n, size - at) : 0;
    if (mem) {
        memcpy(buf, mem + at, n);
        return n;
    }
    size_t done = 0;
    while (done < n) {
        const ssize_t r = pread(fd, buf + done, n - done, (off_t)(origin + at + done));
        if (r <= 0) break;
        done += (size_t)r;
    }
    return done;
}

size_t TextSource::boundary(size_t b, std::vector<char>& scratch) const {
    if (b == 0) return 0;
    if (b >= size) return size;
    if (mem) return fastq_next_record(mem, size, b);
    for (size_t window = 64u << 10;; window *= 4) {
        const size_t want = std::min(window, size - (b - 1));
        if (scratch.size() < want) scratch.resize(want);
        if (read(scratch.data(), b - 1, want) != want) return SIZE_MAX;
        const size_t q = fastq_next_record(scratch.data(), want, 1);
        if (q < want) return b - 1 + q;
        if (b - 1 + want >= size) return size;
        if (window > (512u << 20)) return SIZE_MAX;
    }
}

bool fastq_frame_text(const TextSource& src, uint32_t threads, char* seq_buf, std::vector<FramedSlice>& sl,
                      const std::function<bool(size_t, size_t)>& on_slice) {
    static const size_t slice_bytes = [] {  // tests lower it to cut small files into many slices
        const char* e = getenv("DRPRG_FRAME_SLICE");
        return e && atol(e) > 0 ? (size_t)atol(e) : (size_t)(1u << 20);
    }();
    const size_t S = std::max<size_t>(1, std::min<size_t>(src.size / slice_bytes, 8192));
    sl.clear();
    sl.resize(S);
    std::atomic<bool> failed{false};
    parallel_for_io(S, [&](size_t s) {
        FramedSlice& Z = sl[s];
        if (failed.load(std::memory_order_relaxed)) return;
        thread_local std::vector<char> buf;
        const size_t lo = src.boundary(src.size / S * s + std::min(s, src.size % S), buf);
        const size_t hi = s + 1 == S ? src.size : src.boundary(src.size / S * (s + 1) + std::min(s + 1, src.size % S), buf);
        if (lo == SIZE_MAX || hi == SIZE_MAX) {
            Z.state = -2;
            failed = true;
            return;
        }
        Z.lo = lo;
        Z.state = 1;
        if (lo >= hi) return;
        Z.starts.reserve((hi - lo) / 256 + 16);
        Z.lens.reserve((hi - lo) / 256 + 16);
        FastqFramer F(seq_buf + lo / 2, (hi - lo) / 2, (uint32_t)(lo / 2), Z.starts, Z.lens);
        bool ok = true;
        if (src.mem) {
            size_t used = 0;
            ok = F.feed(src.mem + lo, hi - lo, used) && F.finish(src.mem + lo + used, hi - lo - used, hi == src.size);
        } else {
            // pread into an L2-resident bounce buffer: mapping the slices instead saves the copy but was measured 2-3x
            // slower from 16 threads (10 M reads from a 3.15 GB file: 64 ms with pread, 134-191 ms mapped with 1-16 MB slices)
            constexpr size_t CH = 512u << 10;  // stays in the core's L2
            if (buf.size() < 2 * CH) buf.resize(2 * CH);
            size_t at = lo, carry = 0;
            while (ok && at < hi) {
                const size_t want = std::min(CH, hi - at);
                if (buf.size() < carry + want) buf.resize(std::max(buf.size() * 2, carry + want));
                if (src.read(buf.data() + carry, at, want) != want) {
                    Z.state = -2;
                    failed = true;
                    return;
                }
                at += want;
                size_t used = 0;
                ok = F.feed(buf.data(), carry + want, used);
                carry = carry + want - used;
                if (ok && carry) memmove(buf.data(), buf.data() + used, carry);
            }
            ok = ok && F.finish(buf.data(), carry, hi == src.size);
        }
        if (!ok) {
            Z.state = -1;
            failed = true;
            return;
        }
        Z.st = F.stats();
        if (Z.st.seq_bytes && on_slice && !on_slice(lo / 2, Z.st.seq_bytes)) failed = true;
    }, std::max<size_t>(1, threads));
    for (const FramedSlice& Z : sl)
        if (Z.state == -2) throw std::runtime_error("reads file: read error");
    return !failed;
}

}  // namespace drprg
