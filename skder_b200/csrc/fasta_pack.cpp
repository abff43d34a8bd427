// Host-side FASTA ingest and 2-bit packing for the B200 ANI/AF engine.
//
// Stands in for skani's file reader on every path named in skDER's `-l` / `--rl` / `--ql` list
// files (reference src/skDER/skder.py:16, :58, :103) and for the positional FASTA of
// `skani search` (skder.py:119).  Also computes the assembly N50 exactly as the reference's
// util.n50_calc (src/skDER/util.py:686-724), since the packer sees every record length anyway.
#include <fcntl.h>
#include <immintrin.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cerrno>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/skani_b200.h"

namespace {

constexpr uint8_t SKIP = 4;  // blanks inside a sequence line are dropped, not packed
struct CodeTable {
    uint8_t t[256];
    CodeTable() {
        std::memset(t, 0, sizeof t);  // anything that is not C/G/T (either case) packs as A
        t[(int)'C'] = t[(int)'c'] = 1;
        t[(int)'G'] = t[(int)'g'] = 2;
        t[(int)'T'] = t[(int)'t'] = 3;
        t[(int)'\r'] = t[(int)' '] = t[(int)'\t'] = SKIP;
    }
};
const CodeTable kCode;

struct Packer {
    std::vector<uint64_t> words;
    uint64_t cur = 0;
    int64_t n_bases = 0;
    inline void put(uint8_t code) {
        cur |= (uint64_t)code << (2 * (n_bases & 31));
        if ((++n_bases & 31) == 0) {
            words.push_back(cur);
            cur = 0;
        }
    }
    // n bytes of one sequence line.  Returns the number of bases packed (blanks are dropped).  The common case -- no
    // blank in the piece -- goes 32 bytes -> one word without a branch per base (32 bytes per step with AVX2 where the
    // CPU has it, a table look-up per byte otherwise); a piece with blanks is redone base by base.
    // `limit`: end of the readable buffer the line sits in (the AVX2 path may load up to 31 bytes past the line, never
    // past `limit`)
    int64_t put_line(const uint8_t *s, int64_t n, const uint8_t *limit) {
        const size_t w0 = words.size();
        const uint64_t cur0 = cur;
        const int64_t nb0 = n_bases;
        static const bool avx2 = __builtin_cpu_supports("avx2") && !std::getenv("SKB_NO_AVX2");  // SKB_NO_AVX2: tests run both
        const bool blanks = avx2 ? pack_avx2(s, n, limit) : pack_scalar(s, n);
        if (!blanks) return n;
        words.resize(w0);  // rare: blanks inside the line
        cur = cur0;
        n_bases = nb0;
        int64_t kept = 0;
        for (int64_t k = 0; k < n; k++) {
            const uint8_t c = kCode.t[s[k]];
            if (c & SKIP) continue;
            put(c);
            kept++;
        }
        return kept;
    }
    // r <= 32 codes in w (2 bits each, zero above): append
    inline void append_word(uint64_t w, int r) {
        const int sh = 2 * (int)(n_bases & 31);
        cur |= w << sh;
        if (sh + 2 * r >= 64) {
            words.push_back(cur);
            cur = sh ? w >> (64 - sh) : 0;
        }
        n_bases += r;
    }
    // both return true if the piece holds a blank (the caller then redoes it base by base)
    bool pack_scalar(const uint8_t *s, int64_t n) {
        uint8_t flags = 0;
        for (int64_t k = 0; k < n; k += 32) {
            const int r = (int)std::min<int64_t>(32, n - k);
            uint64_t w = 0;
            if (r == 32) {
#pragma GCC unroll 32
                for (int x = 0; x < 32; x++) {
                    const uint8_t c = kCode.t[s[k + x]];
                    flags |= c;
                    w |= (uint64_t)(c & 3) << (2 * x);
                }
            } else {
                for (int x = 0; x < r; x++) {
                    const uint8_t c = kCode.t[s[k + x]];
                    flags |= c;
                    w |= (uint64_t)(c & 3) << (2 * x);
                }
            }
            append_word(w, r);
        }
        return (flags & SKIP) != 0;
    }
    // 32 bytes per step: C/G/T of either case found by three compares on (byte | 0x20), everything else is 0 ('A');
    // four 2-bit codes are folded into a byte by two multiply-adds, the eight bytes gathered by one shuffle
    __attribute__((target("avx2"))) bool pack_avx2(const uint8_t *s, int64_t n, const uint8_t *limit) {
        const __m256i lc = _mm256_set1_epi8(0x20), one = _mm256_set1_epi8(1), two = _mm256_set1_epi8(2), three = _mm256_set1_epi8(3);
        const __m256i gather = _mm256_setr_epi8(0, 4, 8, 12, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1,
                                                0, 4, 8, 12, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1);
        uint32_t blank = 0;
        for (int64_t k = 0; k < n; k += 32) {
            const int r = (int)std::min<int64_t>(32, n - k);
            __m256i v;
            if (s + k + 32 <= limit)  // the bytes after a short last piece (the next lines) are masked off below
                v = _mm256_loadu_si256(reinterpret_cast<const __m256i *>(s + k));
            else {  // the end of the buffer: never read past it
                alignas(32) uint8_t tail[32] = {0};
                std::memcpy(tail, s + k, (size_t)r);
                v = _mm256_load_si256(reinterpret_cast<const __m256i *>(tail));
            }
            const __m256i low = _mm256_or_si256(v, lc);
            const __m256i code = _mm256_or_si256(
                _mm256_or_si256(_mm256_and_si256(_mm256_cmpeq_epi8(low, _mm256_set1_epi8('c')), one),
                                _mm256_and_si256(_mm256_cmpeq_epi8(low, _mm256_set1_epi8('g')), two)),
                _mm256_and_si256(_mm256_cmpeq_epi8(low, _mm256_set1_epi8('t')), three));
            const __m256i bl = _mm256_or_si256(_mm256_or_si256(_mm256_cmpeq_epi8(v, _mm256_set1_epi8(' ')),
                                                               _mm256_cmpeq_epi8(v, _mm256_set1_epi8('\t'))),
                                               _mm256_cmpeq_epi8(v, _mm256_set1_epi8('\r')));
            uint32_t bm = (uint32_t)_mm256_movemask_epi8(bl);
            if (r < 32) bm &= (1u << r) - 1u;  // a '\r' or blank behind the piece belongs to another line
            blank |= bm;
            const __m256i n4 = _mm256_maddubs_epi16(code, _mm256_set1_epi16(0x0401));   // c0 + 4 c1 per 16 bits
            const __m256i n8 = _mm256_madd_epi16(n4, _mm256_set1_epi32(0x00100001));    // + 16 (c2 + 4 c3) per 32 bits
            const __m256i by = _mm256_shuffle_epi8(n8, gather);                         // 4 bytes per 128-bit half
            uint64_t w = (uint64_t)(uint32_t)_mm256_extract_epi32(by, 0) | ((uint64_t)(uint32_t)_mm256_extract_epi32(by, 4) << 32);
            if (r < 32) w &= (1ull << (2 * r)) - 1ull;  // codes of the bytes behind the piece
            append_word(w, r);
        }
        return blank != 0;
    }
    void finish() {
        if (n_bases & 31) words.push_back(cur);
        cur = 0;
        if (words.size() & 1) words.push_back(0);  // 16-byte multiple for 128-bit device loads
        if (words.empty()) {
            words.push_back(0);
            words.push_back(0);
        }
    }
};

// N50 as reference util.n50_calc: records with empty sequence are skipped, n2 = floor(total/2),
// first cumulative sum >= n2 over lengths sorted descending.
int64_t n50_of(std::vector<int64_t> lens) {
    lens.erase(std::remove(lens.begin(), lens.end(), (int64_t)0), lens.end());
    if (lens.empty()) return 0;
    std::sort(lens.begin(), lens.end(), std::greater<int64_t>());
    int64_t total = 0;
    for (int64_t l : lens) total += l;
    int64_t n2 = total / 2, c = 0;
    for (int64_t l : lens) {
        c += l;
        if (c >= n2) return l;
    }
    return lens.back();
}

// names: the kept records' header lines ([kept.size()]), or nullptr for contigs without headers (skb_pack_contigs)
skb_packed *make_packed(Packer &pk, std::vector<int64_t> &kept, const std::string &name,
                        const std::vector<int64_t> &all_lens, const std::vector<std::string> *names) {
    pk.finish();
    skb_packed *p = (skb_packed *)std::calloc(1, sizeof(skb_packed));
    if (!p) return nullptr;
    p->n_words = (int64_t)pk.words.size();
    p->words = (uint64_t *)std::malloc(sizeof(uint64_t) * pk.words.size());
    std::memcpy(p->words, pk.words.data(), sizeof(uint64_t) * pk.words.size());
    p->n_bases = pk.n_bases;
    p->n_contigs = (int32_t)kept.size();
    p->contig_lens = (int64_t *)std::malloc(sizeof(int64_t) * std::max<size_t>(kept.size(), 1));
    if (!kept.empty()) std::memcpy(p->contig_lens, kept.data(), sizeof(int64_t) * kept.size());
    p->first_name = strdup(name.c_str());
    p->n50 = n50_of(all_lens);
    int64_t t = 0;
    for (int64_t l : all_lens) t += l;
    p->total_bases_all = t;
    if (names) {
        p->contig_names = (char **)std::calloc(std::max<size_t>(names->size(), 1), sizeof(char *));
        for (size_t k = 0; k < names->size(); k++) p->contig_names[k] = strdup((*names)[k].c_str());
    }
    return p;
}

}  // namespace

extern "C" {

int skb_pack_fasta(const char *path, int32_t min_contig_len, skb_packed **out) {
    if (!path || !out) return SKB_EINVAL;
    *out = nullptr;
    // gzip members go through zlib; anything else is read straight from the descriptor (zlib's transparent mode
    // copies every byte twice, which showed once the packing itself ran at memory speed)
    const int fd = open(path, O_RDONLY | O_CLOEXEC);
    if (fd < 0) return SKB_EIO;
    unsigned char magic[2] = {0, 0};
    const bool is_gz = pread(fd, magic, 2, 0) == 2 && magic[0] == 0x1f && magic[1] == 0x8b;
    gzFile g = nullptr;
    if (is_gz) {
        g = gzdopen(fd, "rb");
        if (!g) {
            close(fd);
            return SKB_EIO;
        }
        gzbuffer(g, 1 << 20);
    }
    auto close_input = [&]() {
        if (g)
            gzclose(g);  // closes fd
        else
            close(fd);
    };
    // per-thread scratch, kept across files: a fresh 4 MB buffer and a fresh word vector per genome cost more in page
    // faults than the packing itself once that ran at memory speed
    thread_local std::vector<char> buf;
    thread_local std::vector<uint64_t> scratch_words;
    if (buf.empty()) buf.resize(1 << 22);
    // Records are packed straight into the output; a record that turns out shorter than
    // min_contig_len is rolled back.
    Packer pk;
    pk.words.swap(scratch_words);
    pk.words.clear();
    if (pk.words.capacity() < (1u << 18)) pk.words.reserve(1 << 18);
    struct GiveBack {  // the vector (and its capacity) returns to the thread on every exit path
        Packer &pk;
        std::vector<uint64_t> &home;
        ~GiveBack() { pk.words.swap(home); }
    } give_back{pk, scratch_words};
    std::vector<int64_t> kept, all_lens;
    std::vector<std::string> kept_names;
    std::string cur_name;
    bool in_header = false, in_record = false;
    int64_t rec_len = 0, rec_start_bases = 0;
    size_t rec_start_words = 0;
    uint64_t rec_start_cur = 0;
    auto close_record = [&]() {
        if (!in_record) return;
        all_lens.push_back(rec_len);
        if (rec_len >= min_contig_len && rec_len > 0) {
            kept.push_back(rec_len);
            kept_names.push_back(cur_name);
        } else {  // roll back
            pk.words.resize(rec_start_words);
            pk.cur = rec_start_cur;
            pk.n_bases = rec_start_bases;
        }
    };
    bool at_line_start = true;
    for (;;) {
        long got;
        if (g)
            got = gzread(g, buf.data(), (unsigned)buf.size());
        else
            do got = (long)read(fd, buf.data(), buf.size());
            while (got < 0 && errno == EINTR);
        if (got < 0) {
            close_input();
            return SKB_EIO;
        }
        if (got == 0) break;
        const char *p = buf.data(), *const end = p + got;
        while (p < end) {
            if (in_header) {  // the rest of the header line
                const char *nl = (const char *)std::memchr(p, '\n', (size_t)(end - p));
                cur_name.append(p, nl ? nl : end);
                if (!nl) break;
                in_header = false;
                at_line_start = true;
                while (!cur_name.empty() && cur_name.back() == '\r') cur_name.pop_back();
                p = nl + 1;
                continue;
            }
            if (at_line_start && *p == '>') {
                close_record();
                in_record = true;
                in_header = true;
                cur_name.clear();
                rec_len = 0;
                rec_start_bases = pk.n_bases;
                rec_start_words = pk.words.size();
                rec_start_cur = pk.cur;
                p++;
                continue;
            }
            // (the rest of) a sequence line; a '>' that is not first on its line is an ordinary non-ACGT byte
            const char *nl = (const char *)std::memchr(p, '\n', (size_t)(end - p));
            const char *e = nl ? nl : end;
            if (in_record && e > p)  // else: text before the first header
                rec_len += pk.put_line((const uint8_t *)p, (int64_t)(e - p), (const uint8_t *)end);
            at_line_start = nl != nullptr;
            p = nl ? nl + 1 : end;
        }
    }
    close_input();
    close_record();
    *out = make_packed(pk, kept, kept_names.empty() ? std::string() : kept_names[0], all_lens, &kept_names);
    return *out ? SKB_OK : SKB_ENOMEM;
}

int skb_pack_contigs(const char *const *seqs, const int64_t *lens, int32_t n, int32_t min_contig_len,
                     skb_packed **out) {
    if (!out || n < 0) return SKB_EINVAL;
    Packer pk;
    std::vector<int64_t> kept, all_lens;
    for (int32_t i = 0; i < n; i++) {
        all_lens.push_back(lens[i]);
        if (lens[i] < min_contig_len || lens[i] <= 0) continue;
        const uint8_t *s = (const uint8_t *)seqs[i];
        kept.push_back(pk.put_line(s, lens[i], s + lens[i]));  // the whole contig as one line (blanks, if any, are dropped)
    }
    *out = make_packed(pk, kept, "", all_lens, nullptr);
    return *out ? SKB_OK : SKB_ENOMEM;
}

int skb_pack_fasta_many(const char *const *paths, int32_t n, int32_t min_contig_len, int32_t n_threads,
                        skb_packed **out) {
    if (!paths || !out || n < 0) return SKB_EINVAL;
    if (n_threads < 1) n_threads = 1;
    std::atomic<int32_t> next(0), failures(0);
    auto work = [&]() {
        for (;;) {
            int32_t i = next.fetch_add(1);
            if (i >= n) break;
            out[i] = nullptr;
            if (skb_pack_fasta(paths[i], min_contig_len, &out[i]) != SKB_OK) failures.fetch_add(1);
        }
    };
    std::vector<std::thread> th;
    for (int32_t t = 1; t < std::min(n_threads, std::max(n, 1)); t++) th.emplace_back(work);
    work();
    for (auto &t : th) t.join();
    return failures.load();
}

void skb_packed_free(skb_packed *p) {
    if (!p) return;
    std::free(p->words);
    std::free(p->contig_lens);
    std::free(p->first_name);
    if (p->contig_names)
        for (int32_t k = 0; k < p->n_contigs; k++) std::free(p->contig_names[k]);
    std::free(p->contig_names);
    std::free(p);
}

}  // extern "C"
