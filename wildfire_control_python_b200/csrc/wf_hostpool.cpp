// wf_hostpool.cpp -- host half of wf_step_host's packed-observation path (plain C++, no CUDA).
//
// World.get_state (environment.py:399-402) is three 0/1 planes: over PCIe the step kernel sends the
// bit stream itself (1 bit per element, 8x fewer bytes than the uint8 array) and the host expands it
// into the caller's [N][W][H][3] uint8 buffer: output bytes 8i..8i+7 = the 8 bits of input byte i
// (AVX2: 32 output bytes per iteration; else one PDEP per 8 output bytes, or a 256-entry table).  A small persistent thread pool
// splits the records; workers spin briefly for the next step and then sleep on a condition variable.
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>

#if defined(__x86_64__)
#include <immintrin.h>
#endif

namespace wf {

struct ExpandJob {
    const uint32_t* packed;  // [records][rec_stride]: rec_words of observation bits (+ one status word in session mode)
    uint8_t* out;            // [n_envs][env_bits] bytes
    int64_t records, rec_words, env_bits, envs_per_record, n_envs;
    int64_t rec_stride;      // words between records (rec_words, or rec_words + 1 with a status word)
    int64_t recs_per_block, block_stride;  // session: records come in blocks of recs_per_block (one CTA's), block_stride words
                                           // apart (whole 128-byte lines); otherwise 1 and rec_stride
    // step-server session (wf_host_session): the records of slice t are complete once flags[16 * t] == seq
    const volatile uint32_t* flags;
    uint32_t seq;
    int64_t records_per_slice;  // session: flag s covers records [s * records_per_slice, (s + 1) * records_per_slice)
    double* reward;             // session: decoded from the status word (may be null)
    uint8_t* done;
    double default_reward, death_penalty, contained_bonus, cells;
    int64_t timeout_ns;         // session: give up waiting for a flag after this long (the caller then checks the kernel)
    const uint32_t* full_area;  // session with a persistent observation array (wf_host_session mode 2), != nullptr: `packed` holds
    int64_t full_stride;        // change-list blocks (32 words per 4 records, wf_common.cuh); a record flagged in its block's header
                                // is complete in full_area[record * full_stride] instead
    int64_t sectors;            // session, != 0: each record is `sectors` self-validating 32-byte sectors (7 payload words + tag =
                                // seq ^ hash), no flags: a record is taken as soon as all its sectors validate
    bool out_bits;              // session: `out` is WF_OBS_BITS, uint32 [n_envs][ceil(env_bits / 32)], instead of bytes
};

static inline uint32_t sector_hash(const uint32_t* w) {  // == wf_common.cuh
    uint32_t h = 0x9E3779B9u;
    for (int i = 0; i < 7; ++i) h = (h + w[i]) * 0x9E3779B1u;
    return h ^ (h >> 15);
}

static uint64_t g_tab[256];
static std::once_flag g_tab_once;
static void init_tab() {
    for (int v = 0; v < 256; ++v) {
        uint64_t o = 0;
        for (int i = 0; i < 8; ++i) o |= (uint64_t)((v >> i) & 1) << (8 * i);
        g_tab[v] = o;
    }
}

static void expand_table(const uint8_t* in, uint8_t* out, int64_t nbytes) {
    for (int64_t i = 0; i < nbytes; ++i) std::memcpy(out + 8 * i, &g_tab[in[i]], 8);
}
#if defined(__x86_64__)
__attribute__((target("bmi2"))) static void expand_pdep(const uint8_t* in, uint8_t* out, int64_t nbytes) {
    for (int64_t i = 0; i < nbytes; ++i) {
        const uint64_t v = _pdep_u64((uint64_t)in[i], 0x0101010101010101ull);
        std::memcpy(out + 8 * i, &v, 8);
    }
}
#endif

#if defined(__x86_64__)
// 4 input bytes -> 32 output bytes per iteration: broadcast, route byte k/8 to lane k, test bit k%8.  The destination of a
// record is only 8-byte aligned (W*H*3 bytes per env), and vector stores that straddle cache lines cost about twice as much:
// 8-byte pieces (one PDEP each) until the destination is aligned, aligned vector stores, 8-byte pieces for the rest.
__attribute__((target("avx2,bmi2"))) static void expand_avx2(const uint8_t* in, uint8_t* out, int64_t nbytes) {
    const __m256i route = _mm256_setr_epi8(0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 1, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 3, 3, 3, 3, 3, 3, 3, 3);
    const __m256i bit = _mm256_set1_epi64x((long long)0x8040201008040201ull);
    const __m256i one = _mm256_set1_epi8(1);
    int64_t i = 0;
    const bool can_align = (reinterpret_cast<uintptr_t>(out) & 7u) == 0;  // (odd-sized grids: plain unaligned stores)
    for (; can_align && i < nbytes && (reinterpret_cast<uintptr_t>(out + 8 * i) & 31u); ++i) {
        const uint64_t v = _pdep_u64((uint64_t)in[i], 0x0101010101010101ull);
        std::memcpy(out + 8 * i, &v, 8);
    }
    for (; i + 4 <= nbytes; i += 4) {
        uint32_t v;
        std::memcpy(&v, in + i, 4);
        const __m256i b = _mm256_shuffle_epi8(_mm256_set1_epi32((int)v), route);
        const __m256i r = _mm256_and_si256(_mm256_cmpeq_epi8(_mm256_and_si256(b, bit), bit), one);
        if (can_align) _mm256_store_si256(reinterpret_cast<__m256i*>(out + 8 * i), r);
        else _mm256_storeu_si256(reinterpret_cast<__m256i*>(out + 8 * i), r);
    }
    for (; i < nbytes; ++i) {
        const uint64_t v = _pdep_u64((uint64_t)in[i], 0x0101010101010101ull);
        std::memcpy(out + 8 * i, &v, 8);
    }
}
#endif

#if defined(__x86_64__)
// 8 input bytes -> 64 output bytes per iteration: the input IS the byte mask of a masked move of 1s.  Same alignment scheme
// as expand_avx2; no masked stores (a masked 64-byte store of the 3-byte tail cost as much as the 18 full ones together).
__attribute__((target("avx512f,avx512bw,bmi2"))) static void expand_avx512(const uint8_t* in, uint8_t* out, int64_t nbytes) {
    const __m512i one = _mm512_set1_epi8(1);
    int64_t i = 0;
    const bool aligned = (reinterpret_cast<uintptr_t>(out) & 7u) == 0;  // (odd-sized grids: plain unaligned stores)
    for (; aligned && i < nbytes && (reinterpret_cast<uintptr_t>(out + 8 * i) & 63u); ++i) {
        const uint64_t v = _pdep_u64((uint64_t)in[i], 0x0101010101010101ull);
        std::memcpy(out + 8 * i, &v, 8);
    }
    for (; i + 8 <= nbytes; i += 8) {
        uint64_t v;
        std::memcpy(&v, in + i, 8);
        const __m512i r = _mm512_maskz_mov_epi8(_cvtu64_mask64(v), one);
        if (aligned) _mm512_store_si512(reinterpret_cast<void*>(out + 8 * i), r);
        else _mm512_storeu_si512(reinterpret_cast<void*>(out + 8 * i), r);
    }
    for (; i < nbytes; ++i) {
        const uint64_t v = _pdep_u64((uint64_t)in[i], 0x0101010101010101ull);
        std::memcpy(out + 8 * i, &v, 8);
    }
}
#endif

// Reward of one env from its status bits: the expressions of World.get_reward (environment.py:379-390) in the
// reference's operation order; the burn-out fraction is the same IEEE division and multiplication the kernel does.
static inline double decode_reward(const ExpandJob& j, uint32_t st) {
    switch (st & 7u) {
        case 1: return j.default_reward;
        case 2: return j.death_penalty;
        case 3: return j.contained_bonus;
        case 4: return j.contained_bonus * ((double)((st >> 4) & 0x7ffu) / j.cells);
        default: return 0.0;
    }
}

static inline void cpu_pause() {
#if defined(__x86_64__)
    _mm_pause();
#endif
}

// Sector transport: copy record r's payload into `tmp` once every sector's tag fits its contents.  false: timed out.
static bool fetch_record(const ExpandJob& j, int64_t r, uint32_t* tmp, const std::chrono::steady_clock::time_point& t0) {
    const volatile uint32_t* base = j.packed + (r / j.recs_per_block) * j.block_stride + (r % j.recs_per_block) * j.sectors * 8;
    int spins = 0;
    for (int64_t sec = 0; sec < j.sectors; ++sec) {
        uint32_t* out = tmp + 7 * sec;
        for (;;) {
            uint32_t w[8];
            for (int i = 0; i < 8; ++i) w[i] = base[8 * sec + i];
            if (w[7] == (j.seq ^ sector_hash(w))) {
                for (int i = 0; i < 7; ++i) out[i] = w[i];
                break;
            }
            cpu_pause();
            if ((++spins & 255) == 0 && std::chrono::steady_clock::now() - t0 > std::chrono::nanoseconds(j.timeout_ns)) return false;
        }
    }
    return true;
}

// Change-list blocks (wf_common.cuh): per CTA block the status words of its 4 records, the records sent in full (expanded
// from the full area) and ONE list of the elements that changed in the others.
static void expand_one(const ExpandJob& j, const uint32_t* rec, int64_t env0, int64_t nenv);
static void apply_delta_records(const ExpandJob& j, int64_t r0, int64_t r1) {
    constexpr int kBlockWords = 32, kFirstEntry = 10;
    const int64_t b0 = (r0 + 3) >> 2, b1 = (r1 + 3) >> 2;  // whole blocks; consecutive record ranges give consecutive block ranges
#if defined(__x86_64__)
    // The GPU has just written these lines: none is in a cache of this core, and a range of a few KB is over before the
    // hardware prefetcher has caught on.  Ask for the first ones at once, the rest a little ahead.
    for (int64_t b = b0; b < b1 && b < b0 + 16; ++b) {
        _mm_prefetch(reinterpret_cast<const char*>(j.packed + b * kBlockWords), _MM_HINT_T0);
        _mm_prefetch(reinterpret_cast<const char*>(j.packed + b * kBlockWords) + 64, _MM_HINT_T0);
    }
#endif
    const int64_t rec_elems = j.envs_per_record * j.env_bits;
    for (int64_t b = b0; b < b1; ++b) {
        const uint32_t* blk = j.packed + b * kBlockWords;
#if defined(__x86_64__)
        if (b + 16 < b1) {
            _mm_prefetch(reinterpret_cast<const char*>(blk + 16 * kBlockWords), _MM_HINT_T0);
            _mm_prefetch(reinterpret_cast<const char*>(blk + 16 * kBlockWords) + 64, _MM_HINT_T0);
        }
#endif
        const uint32_t hdr = blk[0];
        const int count = (int)(hdr & 0xffu);
        const uint16_t* e = reinterpret_cast<const uint16_t*>(blk) + kFirstEntry;
        if (j.out_bits) {  // the block's envs are whole envs of this thread: no other thread writes their words
            const int64_t wpe = (j.env_bits + 31) / 32;
            uint32_t* out = reinterpret_cast<uint32_t*>(j.out);
            for (int k = 0; k < count; ++k) {
                const int64_t g = 4 * b * rec_elems + (e[k] >> 1), env = g / j.env_bits, bit = g - env * j.env_bits;
                uint32_t& w = out[env * wpe + (bit >> 5)];
                w = (w & ~(1u << (bit & 31))) | ((uint32_t)(e[k] & 1u) << (bit & 31));
            }
        } else {
            uint8_t* out = j.out + 4 * b * rec_elems;
            for (int k = 0; k < count; ++k) out[e[k] >> 1] = (uint8_t)(e[k] & 1u);
        }
        for (int w = 0; w < 4; ++w) {
            const int64_t r = 4 * b + w;
            if (r >= j.records) break;
            const int64_t env0 = r * j.envs_per_record;
            const int64_t nenv = (j.n_envs - env0 < j.envs_per_record) ? (j.n_envs - env0) : j.envs_per_record;
            const uint32_t st = blk[1 + w];
            if ((hdr >> (8 + w)) & 1u) expand_one(j, j.full_area + r * j.full_stride, env0, nenv);
            for (int64_t k = 0; k < nenv; ++k) {
                const uint32_t sk = (st >> (16 * k)) & 0x7fffu;
                if (j.reward) j.reward[env0 + k] = decode_reward(j, sk);
                if (j.done) j.done[env0 + k] = (uint8_t)((sk >> 3) & 1u);
            }
        }
    }
}

// WF_OBS_BITS: the envs of one record -> their own words (env k's stream starts at record bit k * env_bits: re-aligned to a
// word boundary, padding bits cleared).
static void copy_bits_one(const ExpandJob& j, const uint32_t* rec, int64_t env0, int64_t nenv) {
    const int64_t wpe = (j.env_bits + 31) / 32;
    const int tail = (int)(j.env_bits & 31);
    uint32_t* out = reinterpret_cast<uint32_t*>(j.out) + env0 * wpe;
    for (int64_t k = 0; k < nenv; ++k, out += wpe) {
        const int64_t w0 = (k * j.env_bits) >> 5;
        const int sh = (int)((k * j.env_bits) & 31);
        for (int64_t q = 0; q < wpe; ++q) {
            const uint32_t lo = rec[w0 + q], hi = w0 + q + 1 < j.rec_words ? rec[w0 + q + 1] : 0u;
            uint32_t v = sh ? (lo >> sh) | (hi << (32 - sh)) : lo;
            if (q == wpe - 1 && tail) v &= (1u << tail) - 1u;
            out[q] = v;
        }
    }
}

// The observation bits of one record -> the bytes of its envs.
static void expand_one(const ExpandJob& j, const uint32_t* rec, int64_t env0, int64_t nenv) {
    if (j.out_bits) {
        copy_bits_one(j, rec, env0, nenv);
        return;
    }
#if defined(__x86_64__)
    static const bool bmi2 = __builtin_cpu_supports("bmi2");
    static const bool avx2 = bmi2 && __builtin_cpu_supports("avx2") && !getenv("WF_HOST_NO_AVX2");
    static const bool avx512 = avx2 && __builtin_cpu_supports("avx512bw") && !getenv("WF_HOST_NO_AVX512");
#endif
    const int64_t bits = nenv * j.env_bits;
    const uint8_t* in = reinterpret_cast<const uint8_t*>(rec);
    uint8_t* out = j.out + env0 * j.env_bits;
#if defined(__x86_64__)
    if (avx512) expand_avx512(in, out, bits >> 3);
    else if (avx2) expand_avx2(in, out, bits >> 3);
    else if (bmi2) expand_pdep(in, out, bits >> 3);
    else
#endif
        expand_table(in, out, bits >> 3);
    for (int64_t b = bits & ~(int64_t)7; b < bits; ++b) out[b] = (in[b >> 3] >> (b & 7)) & 1;  // ragged tail
}

static bool expand_records(const ExpandJob& j, int64_t r0, int64_t r1) {
    if (j.full_area) {
        apply_delta_records(j, r0, r1);
        return true;
    }
    const auto t_begin = std::chrono::steady_clock::now();
    int64_t blk = r0 / j.recs_per_block, in_blk = r0 % j.recs_per_block;  // (no division per record)
    for (int64_t r = r0; r < r1; ++r, ++in_blk) {
        if (in_blk == j.recs_per_block) { in_blk = 0; ++blk; }
        const int64_t env0 = r * j.envs_per_record;
        const int64_t nenv = (j.n_envs - env0 < j.envs_per_record) ? (j.n_envs - env0) : j.envs_per_record;
        const uint32_t* rec = j.packed + blk * j.block_stride + in_blk * j.rec_stride;
        uint32_t tmp[7 * 16];  // sector transport: the record's payload, validated (<= 97 words)
        if (j.sectors) {
            if (!fetch_record(j, r, tmp, t_begin)) return false;
            rec = tmp;
        }
        expand_one(j, rec, env0, nenv);
        if (j.rec_stride > j.rec_words) {  // session records: reward / done of the record's envs
            const uint32_t st = rec[j.rec_words];
            for (int64_t k = 0; k < nenv; ++k) {
                const uint32_t sk = (st >> (16 * k)) & 0xffffu;
                if (j.reward) j.reward[env0 + k] = decode_reward(j, sk);
                if (j.done) j.done[env0 + k] = (uint8_t)((sk >> 3) & 1u);
            }
        }
    }
    return true;
}

class HostPool {
public:
    explicit HostPool(int n) : n_(n < 1 ? 1 : n) {
        std::call_once(g_tab_once, init_tab);
        for (int t = 1; t < n_; ++t) workers_.emplace_back([this, t] { loop(t); });
    }
    ~HostPool() {
        {
            std::lock_guard<std::mutex> lk(m_);
            stop_ = true;
            seq_.fetch_add(1, std::memory_order_release);
        }
        cv_.notify_all();
        for (auto& th : workers_) th.join();
        if (jobs_timed_ && getenv("WF_HOST_TIMING")) {  // per thread: when its flag was seen (from the job's start) and its own work
            fprintf(stderr, "wf_hostpool: %lld session jobs; thread: flag seen after / work (us):", (long long)jobs_timed_);
            for (int t = 0; t < n_; ++t) fprintf(stderr, " %d: %.2f / %.2f;", t, 1e6 * t_flag_[t] / jobs_timed_, 1e6 * t_work_[t] / jobs_timed_);
            fprintf(stderr, "\n");
        }
    }
    int threads() const { return n_; }
    double first_flag_seconds() const { return first_flag_s_; }  // session jobs: thread 0's accumulated wait for its flag(s)
    // Returns false if a session slice timed out waiting for its completion flag (nothing of that slice was expanded).
    bool run(const ExpandJob& job) {
        job_ = job;
        job_t0_ = std::chrono::steady_clock::now();
        if (job.flags) jobs_timed_ += 1;
        failed_.store(0, std::memory_order_relaxed);
        pending_.store(n_ - 1, std::memory_order_relaxed);
        {
            std::lock_guard<std::mutex> lk(m_);  // pairs with the sleepers' predicate check
            seq_.fetch_add(1, std::memory_order_release);
        }
        if (sleepers_.load(std::memory_order_acquire) > 0) cv_.notify_all();
        slice(0);
        while (pending_.load(std::memory_order_acquire) != 0) cpu_relax();
        return failed_.load(std::memory_order_acquire) == 0;
    }

private:
    static void cpu_relax() {
#if defined(__x86_64__)
        _mm_pause();
#else
        std::this_thread::yield();
#endif
    }
    void slice(int t) {
        const int64_t per = (job_.records + n_ - 1) / n_;
        const int64_t r0 = per * t, r1 = (r0 + per < job_.records) ? r0 + per : job_.records;
        if (r0 >= r1) return;
        if (job_.flags && !job_.sectors) {
            // session: the GPU raises a slice's flag once all of the slice's records are in host memory; this thread's
            // records may lie in more than one slice
            const auto t0 = std::chrono::steady_clock::now();
            int spins = 0;
            for (int64_t sl = r0 / job_.records_per_slice; sl <= (r1 - 1) / job_.records_per_slice; ++sl) {
                const volatile uint32_t* f = job_.flags + 16 * sl;
                while (*f != job_.seq) {
                    cpu_relax();
                    if ((++spins & 255) == 0 &&
                        std::chrono::steady_clock::now() - t0 > std::chrono::nanoseconds(job_.timeout_ns)) {
                        failed_.store(1, std::memory_order_release);
                        return;
                    }
                }
            }
            std::atomic_thread_fence(std::memory_order_acquire);
            if (t == 0) first_flag_s_ += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        }
        const auto t_seen = std::chrono::steady_clock::now();
        if (!expand_records(job_, r0, r1)) failed_.store(1, std::memory_order_release);
        if (job_.flags && t < 64) {
            t_flag_[t] += std::chrono::duration<double>(t_seen - job_t0_).count();
            t_work_[t] += std::chrono::duration<double>(std::chrono::steady_clock::now() - t_seen).count();
        }
    }
    void loop(int t) {
        uint64_t seen = 0;
        for (;;) {
            const auto t_idle = std::chrono::steady_clock::now();
            int spins = 0;
            while (seq_.load(std::memory_order_acquire) == seen) {
                // ~150 us of spinning covers the gap between two steps of a tight loop; then sleep, so that an
                // idle handle (or a caller that computes for long between steps) gets its cores back
                if ((++spins & 63) != 0 || std::chrono::steady_clock::now() - t_idle < std::chrono::microseconds(150)) {
                    cpu_relax();
                    continue;
                }
                std::unique_lock<std::mutex> lk(m_);
                sleepers_.fetch_add(1, std::memory_order_acq_rel);
                cv_.wait(lk, [&] { return seq_.load(std::memory_order_acquire) != seen; });
                sleepers_.fetch_sub(1, std::memory_order_acq_rel);
            }
            seen = seq_.load(std::memory_order_acquire);
            if (stop_) return;
            slice(t);
            pending_.fetch_sub(1, std::memory_order_acq_rel);
        }
    }
    int n_;
    std::vector<std::thread> workers_;
    ExpandJob job_{};
    std::atomic<uint64_t> seq_{0};
    std::atomic<int> pending_{0}, sleepers_{0}, failed_{0};
    std::mutex m_;
    std::condition_variable cv_;
    bool stop_ = false;
    double first_flag_s_ = 0.0;
    std::chrono::steady_clock::time_point job_t0_{};
    double t_flag_[64] = {0}, t_work_[64] = {0};
    int64_t jobs_timed_ = 0;
};

// C-level hooks used by wf_api.cu
HostPool* hostpool_create(int threads) { return new HostPool(threads); }
void hostpool_destroy(HostPool* p) { delete p; }
int hostpool_threads(const HostPool* p) { return p ? p->threads() : 0; }
void hostpool_expand(HostPool* p, const uint32_t* packed, uint8_t* out, int64_t records, int64_t rec_words, int64_t env_bits,
                     int64_t envs_per_record, int64_t n_envs) {
    ExpandJob j{};
    j.packed = packed; j.out = out; j.records = records; j.rec_words = rec_words; j.env_bits = env_bits;
    j.envs_per_record = envs_per_record; j.n_envs = n_envs; j.rec_stride = rec_words;
    j.recs_per_block = 1; j.block_stride = rec_words;
    p->run(j);
}
// Session step: thread t waits for flags[16 * t] == seq, then expands records [t * records_per_slice, ...) -- or, out_bits,
// copies them into WF_OBS_BITS rows -- and decodes their status words into reward / done.  false: a flag did not come within
// timeout_ns.
bool hostpool_expand_session(HostPool* p, const uint32_t* packed, uint8_t* out, int64_t records, int64_t rec_words,
                             int64_t env_bits, int64_t envs_per_record, int64_t n_envs, const volatile uint32_t* flags,
                             uint32_t seq, int64_t records_per_slice, double* reward, uint8_t* done, double default_reward,
                             double death_penalty, double contained_bonus, double cells, int64_t timeout_ns, int64_t sectors,
                             const uint32_t* full_area, int64_t full_stride, bool out_bits) {
    ExpandJob j{};
    j.packed = packed; j.out = out; j.records = records; j.rec_words = rec_words; j.env_bits = env_bits;
    j.envs_per_record = envs_per_record; j.n_envs = n_envs; j.rec_stride = rec_words + 1;
    j.recs_per_block = 4;  // wf_warp.cu: one CTA = 4 warps = 4 records
    j.sectors = sectors;
    j.block_stride = sectors ? 4 * sectors * 8 : (4 * (rec_words + 1) + 31) / 32 * 32;
    j.flags = flags; j.seq = seq; j.records_per_slice = records_per_slice; j.reward = reward; j.done = done;
    j.default_reward = default_reward; j.death_penalty = death_penalty; j.contained_bonus = contained_bonus; j.cells = cells;
    j.timeout_ns = timeout_ns;
    j.full_area = full_area; j.full_stride = full_stride;
    j.out_bits = out_bits;
    return p->run(j);
}
double hostpool_first_flag_seconds(const HostPool* p) { return p ? p->first_flag_seconds() : 0.0; }
int hostpool_default_threads() {
    if (const char* v = getenv("WF_HOST_THREADS")) {
        const int n = atoi(v);
        if (n >= 1) return n > 64 ? 64 : n;
    }
    unsigned hc = std::thread::hardware_concurrency();
    int local = 1;  // ranks sharing this host (torchrun sets LOCAL_WORLD_SIZE)
    if (const char* v = getenv("LOCAL_WORLD_SIZE")) local = atoi(v) > 0 ? atoi(v) : 1;
    // This rank's share of the cores, at most 12 (a lone rank on a 16-core host keeps 4 cores free; 8 ranks on a 32-core host
    // get 4 threads each, the caller's own thread included: the expansion is bound by each core's ~34 GB/s of store misses, so
    // every core counts -- r02, 8 GPUs: 47 us per C2 step with 3 threads per rank).
    int n = (int)(hc ? hc : 4) / local;
    return n < 1 ? 1 : (n > 12 ? 12 : n);
}

}  // namespace wf
