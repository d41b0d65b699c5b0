// maf.hpp — MAF alignment reader with the reference's block-concatenation semantics.
//
// Mirrors parallel_maf_reader::get_next_alignment (reference src/parallel_file_reader.hpp:430-700):
//   * `s` lines: `s <species>.<chrom> <start0> <size> <strand> <srcSize> <text>` (space separated, :180-245);
//     species = text before the first '.', lower-cased (:489-507); species unknown to the model are skipped with a
//     one-time warning (:509-524); `i`/`e`/`q` lines are ignored (:597-600);
//   * the first matched row of a chain's first block is the reference: start_pos = start0 + 1 (:528-554);
//   * build-tracks (concatenate): the next block is appended iff same chrom and start0 == (start_pos-1) + cumulative
//     reference length (:494-505); absent species are padded with 'N' (:603-611); a chain that crosses a multiple of
//     BREAKPOINT_POS keeps reading until >= 2 more reference bases are in, is truncated to exactly +2 and the cursor is
//     rewound to the first block after the crossing block (:456-473, :547-569, :616-629, :671-679);
//   * columns where the reference row has '-' are deleted from every row (:631-669);
//   * score-msa (no concatenation): one block = one alignment, any reference strand.
// Parallelism differs from the reference on purpose: instead of page-aligned byte ranges whose owners re-read a
// neighbour's block (:254-357, :396-425), a parallel pre-scan records per block what the chain logic needs (the `s` lines up
// to the first matched species), a serial pass over that metadata cuts the chains exactly as a single reader would,
// and worker threads parse whole chains.  The output is that of the reference with jobs = 1 for any thread count.
#pragma once

#include <fcntl.h>
#include <sys/mman.h>
#include <unistd.h>

#include <atomic>
#include <mutex>
#include <thread>

#include "model.hpp"

namespace host {

constexpr int64_t BREAKPOINT_POS = 1000000;

struct SLine {
    const char *ident = nullptr; int ident_len = 0;       // species.chrom
    int64_t start0 = 0, size = 0, src_size = 0;
    char strand = '+';
    const char *seq = nullptr; size_t seq_len = 0;
};

// strtok_r(" ") semantics on one line [p, e): runs of spaces collapse.  Numbers via atoi (32 bit, as the reference).
inline bool parse_s_line(const char *p, const char *e, SLine &s) {
    const char *tok[7]; int len[7]; int n = 0;
    while (p < e && n < 7) {
        while (p < e && *p == ' ') ++p;
        if (p >= e) break;
        const char *q = p;
        if (n == 6) {          // the sequence text: nearly the whole line, so let memchr find its end
            const char *sp = (const char *)memchr(p, ' ', (size_t)(e - p));
            q = sp ? sp : e;
        } else {
            while (q < e && *q != ' ') ++q;
        }
        tok[n] = p; len[n] = (int)(q - p); ++n;
        p = q;
    }
    if (n < 7) return false;
    auto num = [](const char *t, int l) {
        int64_t v = 0;
        int i = 0;
        const bool neg = l > 0 && t[0] == '-';
        if (neg) i = 1;
        for (; i < l && t[i] >= '0' && t[i] <= '9'; ++i) v = v * 10 + (t[i] - '0');
        return (int64_t)(int32_t)(neg ? -v : v);      // atoi
    };
    s.ident = tok[1]; s.ident_len = len[1];
    s.start0 = num(tok[2], len[2]); s.size = num(tok[3], len[3]);
    s.strand = tok[4][0];
    s.src_size = num(tok[5], len[5]);
    s.seq = tok[6]; s.seq_len = (size_t)len[6];
    while (s.seq_len && (s.seq[s.seq_len - 1] == '\r')) --s.seq_len;
    return true;
}

struct Alignment {            // alignment_t (parallel_file_reader.hpp:19-44) with seqs as one [nl][L] matrix
    int64_t start_pos = 0, chrom_len = 0;
    char strand = '+';
    std::string chrom;
    int64_t L = 0;
    std::vector<uint8_t> seqs;   // [nl][L]
};

class MafFile {
public:
    struct PreLine { int64_t start0; const char *chrom; int chrom_len; };
    struct BlockMeta {
        size_t off = 0, end = 0;
        std::vector<PreLine> pre;        // unmatched `s` lines before the first matched one
        bool has_ref = false;
        uint16_t ref_id = 0;
        int64_t start0 = 0, size = 0, src_size = 0;
        char strand = '+';
        const char *chrom = nullptr; int chrom_len = 0;
        const char *species = nullptr; int species_len = 0;
    };
    struct Chain {
        std::vector<size_t> blocks;
        int64_t start_pos = 0, chrom_len = 0, keep_cols = -1;     // keep_cols >= 0: truncate to that many reference bases
        int64_t ref_cols = 0;                                     // reference bases of the chain (before truncation)
        char strand = '+';
        std::string chrom;
        int ref_id = -1;
    };

    // minus_ref (with concatenate): a chain whose reference row is on '-' is kept as a chain of strand '-' instead of stopping the
    // program, for callers that skip such chains (annotate-with-maf); a block on the other strand than its chain starts a new chain.
    MafFile(const std::string &path, const Model &model, bool concatenate, int threads, bool minus_ref = false)
        : model_(model), concatenate_(concatenate), minus_ref_(minus_ref) {
        fd_ = open(path.c_str(), O_RDONLY);
        if (fd_ < 0) die("Cannot open %s", path.c_str());
        size_ = (size_t)lseek(fd_, 0, SEEK_END);
        if (size_ == 0) { mem_ = nullptr; return; }
        mem_ = (const char *)mmap(nullptr, size_, PROT_READ, MAP_SHARED, fd_, 0);
        if (mem_ == MAP_FAILED) die("Cannot map %s", path.c_str());
        scan_blocks(std::max(1, threads));
        build_chains();
    }
    ~MafFile() {
        if (mem_ && size_) munmap((void *)mem_, size_);
        if (fd_ >= 0) close(fd_);
    }
    size_t file_size() const { return size_; }
    const std::vector<Chain> &chains() const { return chains_; }
    size_t chain_bytes(const Chain &c) const { size_t b = 0; for (size_t i : c.blocks) b += blocks_[i].end - blocks_[i].off; return b; }
    std::vector<std::string> unresolved() const { return std::vector<std::string>(unresolved_.begin(), unresolved_.end()); }

    // Full parse of one chain (thread safe).  species_seen: [nl] flags, may be null.
    void read_chain(const Chain &c, Alignment &aln, std::vector<uint8_t> *species_seen) const {
        const int nl = model_.nl();
        aln.start_pos = c.start_pos; aln.chrom_len = c.chrom_len; aln.strand = c.strand; aln.chrom = c.chrom;
        aln.L = 0; aln.seqs.clear();
        if (c.ref_id < 0) return;
        std::vector<std::string> rows(nl);
        for (std::string &r : rows) r.reserve((size_t)c.ref_cols + (size_t)c.ref_cols / 16 + 64);
        std::string key;
        for (size_t bi : c.blocks) {
            const BlockMeta &b = blocks_[bi];
            const char *p = mem_ + b.off, *end = mem_ + b.end;
            while (p < end) {
                const char *nlp = (const char *)memchr(p, '\n', (size_t)(end - p));
                const char *le = nlp ? nlp : end;
                if (*p == 's') {
                    SLine s;
                    if (parse_s_line(p, le, s)) {
                        const char *dot = (const char *)memchr(s.ident, '.', (size_t)s.ident_len);
                        const int sl = dot ? (int)(dot - s.ident) : s.ident_len;
                        key.assign(s.ident, (size_t)sl);
                        for (char &ch : key) ch = (char)tolower((unsigned char)ch);
                        auto it = model_.seqid_to_phyloid.find(key);
                        if (it != model_.seqid_to_phyloid.end()) {
                            rows[it->second].append(s.seq, s.seq_len);
                            if (species_seen) (*species_seen)[it->second] = 1;
                        }
                    }
                }
                p = le + 1;
            }
            const size_t new_len = rows[c.ref_id].size();                // absent species get N (:603-611)
            for (int i = 0; i < nl; ++i)
                if (rows[i].size() != new_len) {
                    if (rows[i].size() > new_len) die("alignment rows of different length in block at byte %zu", b.off);
                    rows[i].append(new_len - rows[i].size(), 'N');
                }
        }
        // delete the columns where the reference has '-' (:631-669), then cut at the breakpoint + 2
        // (reference gaps are rare, so the kept columns are a few long runs: one memcpy per run and row instead of a byte gather)
        const std::string &ref = rows[c.ref_id];
        std::vector<std::pair<size_t, size_t>> runs;          // [begin, end) of kept alignment columns
        size_t kept = 0;
        const size_t limit = c.keep_cols >= 0 ? (size_t)c.keep_cols : (size_t)-1;
        for (size_t i = 0; i < ref.size() && kept < limit;) {
            const char *gap = (const char *)memchr(ref.data() + i, '-', ref.size() - i);
            size_t e = gap ? (size_t)(gap - ref.data()) : ref.size();
            if (e - i > limit - kept) e = i + (limit - kept);
            if (e > i) { runs.emplace_back(i, e); kept += e - i; }
            i = e;
            while (i < ref.size() && ref[i] == '-') ++i;
        }
        const size_t L = kept;
        aln.L = (int64_t)L;
        aln.seqs.resize((size_t)nl * L);
        for (int s = 0; s < nl; ++s) {
            const char *src = rows[s].data();
            uint8_t *dst = aln.seqs.data() + (size_t)s * L;
            for (const auto &r : runs) { memcpy(dst, src + r.first, r.second - r.first); dst += r.second - r.first; }
        }
    }

    // The same parse, written straight into a caller-owned matrix: row s of the chain goes to dst + s * row_stride, c.ref_cols columns
    // (the reference bases the chain logic counted from the `size` fields).  One pass over the text: per block the reference row (the
    // first row of the model's species, build_chains() insists on that) gives the runs of kept columns, every other row is copied run
    // by run, absent species are filled with 'N'.  Returns the columns written, or -1 if the text disagrees with the size fields
    // (the caller then takes read_chain(), which measures the text as the reference does).
    int64_t read_chain_into(const Chain &c, uint8_t *dst, int64_t row_stride, std::vector<uint8_t> *species_seen) const {
        if (c.ref_id < 0) return 0;
        const int nl = model_.nl();
        const int64_t limit = c.ref_cols;
        int64_t col = 0;
        struct Row { int id; const char *seq; size_t len; };
        std::vector<Row> rows;
        std::vector<uint8_t> present(nl);
        std::vector<std::pair<size_t, size_t>> runs;
        std::string key;
        // Species of the previous block, line by line: consecutive blocks of a MAF list mostly the same species in the same order, so the
        // species token of line k is first compared with what line k of the previous block resolved to (one short memcmp instead of
        // lower-casing + hashing); -2 = "not in the model".
        struct Seen { const char *name; int len; int id; };
        std::vector<Seen> prev_lines, cur_lines;
        for (size_t bi : c.blocks) {
            const BlockMeta &b = blocks_[bi];
            const char *p = mem_ + b.off, *end = mem_ + b.end;
            rows.clear();
            cur_lines.clear();
            std::fill(present.begin(), present.end(), 0);
            const Row *ref = nullptr;
            while (p < end) {
                const char *nlp = (const char *)memchr(p, '\n', (size_t)(end - p));
                const char *le = nlp ? nlp : end;
                if (*p == 's') {
                    // Only two tokens matter here: the species (token 1, up to the first '.') and the sequence text (token 6).  The text
                    // is the last token of a well-formed line, so it is found from the line's end; lines with fewer than seven tokens or
                    // with anything behind the text take the full tokeniser, which is what the scan and read_chain() use.
                    const char *q = p + 1;
                    while (q < le && *q == ' ') ++q;
                    const char *id0 = q;
                    while (q < le && *q != ' ') ++q;
                    const char *id1 = q;
                    const char *e2 = le;
                    while (e2 > id1 && e2[-1] == '\r') --e2;
                    const char *sp = e2 > id1 ? (const char *)memrchr(id1, ' ', (size_t)(e2 - id1)) : nullptr;
                    SLine s;
                    bool ok = false;
                    if (sp && sp + 1 < e2 && p + 1 < le && p[1] == ' ') {
                        // count the tokens between the identifier and the text: exactly four (start, size, strand, srcSize)
                        int ntok = 0;
                        for (const char *r = id1; r < sp;) {
                            while (r < sp && *r == ' ') ++r;
                            if (r >= sp) break;
                            ++ntok;
                            while (r < sp && *r != ' ') ++r;
                        }
                        if (ntok == 4 && id1 > id0) { s.ident = id0; s.ident_len = (int)(id1 - id0); s.seq = sp + 1; s.seq_len = (size_t)(e2 - sp - 1); ok = true; }
                    }
                    if (!ok) ok = parse_s_line(p, le, s);
                    if (ok) {
                        const char *dot = (const char *)memchr(s.ident, '.', (size_t)s.ident_len);
                        const int sl = dot ? (int)(dot - s.ident) : s.ident_len;
                        int id = -1;
                        const size_t k = cur_lines.size();
                        if (k < prev_lines.size() && prev_lines[k].len == sl && memcmp(prev_lines[k].name, s.ident, (size_t)sl) == 0) {
                            id = prev_lines[k].id;
                        } else {
                            key.assign(s.ident, (size_t)sl);
                            for (char &ch : key) ch = (char)tolower((unsigned char)ch);
                            auto it = model_.seqid_to_phyloid.find(key);
                            id = it != model_.seqid_to_phyloid.end() ? (int)it->second : -2;
                        }
                        cur_lines.push_back(Seen{s.ident, sl, id});
                        if (id >= 0) {
                            if (present[id]) die("alignment rows of different length in block at byte %zu", b.off);
                            present[id] = 1;
                            rows.push_back(Row{id, s.seq, s.seq_len});
                            if (species_seen) (*species_seen)[id] = 1;
                        }
                    }
                }
                p = le + 1;
            }
            prev_lines.swap(cur_lines);
            for (const Row &r : rows) if (r.id == c.ref_id) { ref = &r; break; }
            if (!ref) continue;                                   // a block without the reference species adds no column
            const size_t alen = ref->len;
            // runs of kept alignment columns: where the reference has a base (:631-669), up to the breakpoint cut
            runs.clear();
            int64_t kept = 0;
            size_t i = 0;
            while (i < alen && col + kept < limit) {
                const char *gap = (const char *)memchr(ref->seq + i, '-', alen - i);
                size_t e = gap ? (size_t)(gap - ref->seq) : alen;
                if ((int64_t)(e - i) > limit - col - kept) e = i + (size_t)(limit - col - kept);
                if (e > i) { runs.emplace_back(i, e); kept += (int64_t)(e - i); }
                i = e;
                while (i < alen && ref->seq[i] == '-') ++i;
            }
            if (c.keep_cols < 0 && i < alen) return -1;           // more reference bases in the text than the size fields announced
            for (const Row &r : rows) {
                if (r.len > alen) die("alignment rows of different length in block at byte %zu", b.off);
                uint8_t *o = dst + (int64_t)r.id * row_stride + col;
                for (const auto &run : runs) {
                    const size_t a0 = std::min(run.first, r.len), a1 = std::min(run.second, r.len);
                    if (a1 > a0) memcpy(o, r.seq + a0, a1 - a0);
                    if (a1 - a0 < run.second - run.first) memset(o + (a1 - a0), 'N', (run.second - run.first) - (a1 - a0));   // short row: N (:603-611)
                    o += run.second - run.first;
                }
            }
            for (int i = 0; i < nl; ++i)
                if (!present[i]) memset(dst + (int64_t)i * row_stride + col, 'N', (size_t)kept);
            col += kept;
        }
        return col == limit ? col : -1;
    }

private:
    void scan_range(size_t from, size_t to, std::vector<BlockMeta> &out, std::set<std::string> &unres) const {
        // blocks whose "a " line starts in [from, to)
        size_t pos = from;
        // the reference takes any line whose first character is 'a' as a block start (get_char, parallel_file_reader.hpp:476): bare "a",
        // "a\tscore=..." and "a score=..." alike
        auto at_block = [&](size_t p) { return p < size_ && mem_[p] == 'a' && (p == 0 || mem_[p - 1] == '\n'); };
        auto next_block = [&](size_t p) -> size_t {          // first block start >= p
            while (p < size_) {
                if (at_block(p)) return p;
                const char *q = (const char *)memchr(mem_ + p, '\n', size_ - p);
                if (!q) return size_;
                p = (size_t)(q - mem_) + 1;
            }
            return size_;
        };
        if (from > 0) {   // align to a line start
            const char *q = (const char *)memchr(mem_ + from - 1, '\n', size_ - from + 1);
            pos = q ? (size_t)(q - mem_) + 1 : size_;
        }
        pos = next_block(pos);
        std::string key;
        // species of the previous block's `s` lines (see read_chain_into): line k of a block usually names the species line k of the
        // previous block named, and then neither the lower-casing nor the hash lookup is needed
        struct Seen { const char *name; int len; bool known; };
        std::vector<Seen> prev_lines, cur_lines;
        while (pos < to && pos < size_) {
            BlockMeta b;
            b.off = pos;
            const char *q = (const char *)memchr(mem_ + pos, '\n', size_ - pos);
            size_t p = q ? (size_t)(q - mem_) + 1 : size_;
            cur_lines.clear();
            while (p < size_ && !at_block(p)) {
                const char *nlp = (const char *)memchr(mem_ + p, '\n', size_ - p);
                const size_t le = nlp ? (size_t)(nlp - mem_) : size_;
                if (mem_[p] == 's' && !b.has_ref) {
                    SLine s;
                    if (parse_s_line(mem_ + p, mem_ + le, s)) {
                        const char *dot = (const char *)memchr(s.ident, '.', (size_t)s.ident_len);
                        if (!dot) die("expect format species_name.chrom_name in alignment file (byte %zu)", p);
                        const int sl = (int)(dot - s.ident);
                        key.assign(s.ident, (size_t)sl);
                        for (char &ch : key) ch = (char)tolower((unsigned char)ch);
                        auto it = model_.seqid_to_phyloid.find(key);
                        cur_lines.push_back(Seen{s.ident, sl, it != model_.seqid_to_phyloid.end()});
                        if (it == model_.seqid_to_phyloid.end()) {
                            b.pre.push_back(PreLine{s.start0, dot + 1, s.ident_len - sl - 1});
                            unres.insert(key);
                        } else {
                            b.has_ref = true; b.ref_id = it->second;
                            b.start0 = s.start0; b.size = s.size; b.src_size = s.src_size; b.strand = s.strand;
                            b.chrom = dot + 1; b.chrom_len = s.ident_len - sl - 1;
                            b.species = s.ident; b.species_len = sl;
                        }
                    }
                } else if (mem_[p] == 's') {
                    // later rows only matter for the unknown-species warning
                    const char *sp = mem_ + p + 1;
                    while (sp < mem_ + le && *sp == ' ') ++sp;
                    const char *tok_end = sp;
                    while (tok_end < mem_ + le && *tok_end != ' ') ++tok_end;
                    const char *dot = (const char *)memchr(sp, '.', (size_t)(tok_end - sp));
                    if (dot) {
                        const int sl = (int)(dot - sp);
                        const size_t k = cur_lines.size();
                        bool known;
                        if (k < prev_lines.size() && prev_lines[k].len == sl && memcmp(prev_lines[k].name, sp, (size_t)sl) == 0) {
                            known = prev_lines[k].known;
                        } else {
                            key.assign(sp, (size_t)sl);
                            for (char &ch : key) ch = (char)tolower((unsigned char)ch);
                            known = model_.seqid_to_phyloid.count(key) != 0;
                            if (!known) unres.insert(key);
                        }
                        cur_lines.push_back(Seen{sp, sl, known});
                    } else {
                        cur_lines.push_back(Seen{sp, -1, false});
                    }
                }
                p = le + 1;
            }
            b.end = std::min(p, size_);
            out.push_back(std::move(b));
            prev_lines.swap(cur_lines);
            pos = p;
        }
    }

    void scan_blocks(int threads) {
        std::vector<std::vector<BlockMeta>> parts(threads);
        std::vector<std::set<std::string>> unres(threads);
        std::vector<std::thread> th;
        const size_t step = (size_ + threads - 1) / threads;
        for (int t = 0; t < threads; ++t)
            th.emplace_back([&, t] { scan_range(std::min(size_, t * step), std::min(size_, (t + 1) * step), parts[t], unres[t]); });
        for (auto &x : th) x.join();
        for (int t = 0; t < threads; ++t) {
            for (auto &b : parts[t]) blocks_.push_back(std::move(b));
            unresolved_.insert(unres[t].begin(), unres[t].end());
        }
    }

    // get_next_alignment's control flow on the block metadata
    void build_chains() {
        const size_t nb = blocks_.size();
        size_t pos = 0;
        while (pos < nb) {
            Chain c;
            bool first_block = true, abort_next = !concatenate_, reached_bp = false, stop_saving = false;
            size_t saved_pos = pos;
            int64_t prev_cum = 0, cum_after_bp = 0;
            while ((!abort_next || first_block) && pos < nb) {
                if (!stop_saving) { if (reached_bp) stop_saving = true; saved_pos = pos; }
                const size_t bi = pos++;
                const BlockMeta &b = blocks_[bi];
                if (reached_bp && prev_cum >= cum_after_bp + 2) abort_next = true;
                if (!abort_next || first_block) {
                    bool aborted = false;
                    auto contiguous = [&](int64_t start0, const char *chrom, int chrom_len) {
                        return (c.start_pos - 1) + prev_cum == start0 && (size_t)chrom_len == c.chrom.size() && memcmp(chrom, c.chrom.data(), c.chrom.size()) == 0;
                    };
                    if (!first_block) {
                        for (const PreLine &pl : b.pre)
                            if (!contiguous(pl.start0, pl.chrom, pl.chrom_len)) { aborted = true; break; }
                        if (!aborted && b.has_ref && (!contiguous(b.start0, b.chrom, b.chrom_len) || (minus_ref_ && b.strand != c.strand))) aborted = true;
                    }
                    if (aborted) {
                        abort_next = true;
                    } else if (b.has_ref) {
                        const std::string who = std::string(b.species, (size_t)b.species_len) + "." + std::string(b.chrom, (size_t)b.chrom_len);
                        if (c.ref_id == -1 && first_block) {
                            c.start_pos = b.start0 + 1; c.chrom.assign(b.chrom, (size_t)b.chrom_len); c.chrom_len = b.src_size; c.strand = b.strand;
                            c.ref_id = b.ref_id;
                            prev_cum = b.size;
                            if (b.strand != '+' && concatenate_ && !minus_ref_) die("Reference sequence is not on the + strand (%s at position %ld)!", who.c_str(), (long)b.start0);
                            const int64_t prev_end = c.start_pos, new_end = c.start_pos + b.size;
                            if (!reached_bp && prev_end / BREAKPOINT_POS < new_end / BREAKPOINT_POS) { reached_bp = true; cum_after_bp = prev_cum; }
                        } else if (!first_block) {
                            const int64_t prev_end = c.start_pos + prev_cum, new_end = c.start_pos + prev_cum + b.size;
                            prev_cum += b.size;
                            if (!reached_bp && prev_end / BREAKPOINT_POS < new_end / BREAKPOINT_POS) { reached_bp = true; cum_after_bp = prev_cum; }
                            if (c.ref_id != (int)b.ref_id)
                                die("Encountered an alignment block that didn't start with the reference species: %s at position %ld!", who.c_str(), (long)b.start0);
                            if (b.strand != '+' && concatenate_ && !minus_ref_) die("Reference sequence is not on the + strand (%s at position %ld)!", who.c_str(), (long)b.start0);
                        }
                        c.blocks.push_back(bi);
                    } else {
                        // a block without any species of the model contributes nothing
                        if (c.ref_id >= 0 || first_block) c.blocks.push_back(bi);
                    }
                }
                first_block = false;
            }
            if (reached_bp && prev_cum >= cum_after_bp + 2) abort_next = true;
            if (abort_next && concatenate_) pos = saved_pos;
            if (reached_bp && prev_cum > cum_after_bp + 2) c.keep_cols = cum_after_bp + 2;
            c.ref_cols = c.keep_cols >= 0 ? c.keep_cols : prev_cum;
            chains_.push_back(std::move(c));
        }
    }

    const Model &model_;
    bool concatenate_, minus_ref_;
    int fd_ = -1;
    size_t size_ = 0;
    const char *mem_ = nullptr;
    std::vector<BlockMeta> blocks_;
    std::vector<Chain> chains_;
    std::set<std::string> unresolved_;
};

}  // namespace host
