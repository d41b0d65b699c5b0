// transcripts.hpp — the spliced alignments of GFF/GTF transcripts, cut from whole-genome MAF chains (annotate-with-maf).
//
// The MAF files are read with build-tracks' chain semantics (MafFile, concatenate): chain column j is reference position
// start_pos + j.  A position that no chain covers (chromosome absent, or a hole between chains) is N in every row.  Where two chains
// cover a position (the 2 columns a chain keeps past a 1 Mb breakpoint are the next chain's first two), the chain that starts last
// is used; both hold the same bytes.  Chains whose reference row is on '-' are not used.
//
// A transcript with CDS features: the CDS intervals in genomic order, concatenated; reverse-complemented as a whole on '-' (ACGTacgt
// complemented, every other character kept); the phase of the 5'-most CDS dropped from the front.  Region 0 is the whole alignment,
// then one region per CDS feature in file order: its own columns from after its own phase.  A transcript without CDS features is
// its `exon` features (or, without any, its own span) spliced the same way, for the ORF search; its reference row is that of the
// chains its exons fall in (-1: none, -2: they disagree).  phylocsfpp_b200/transcripts.py restates these rules for the tests.
#pragma once

#include <list>

#include "annotate.hpp"
#include "maf.hpp"

namespace host {

struct TxAlignment {
    bool coding = false;
    char strand = '+';
    int ref_row = -1;                                      // -1: no chain covers it, -2: its chains have different reference rows
    int64_t L = 0;
    std::vector<uint8_t> seqs;                             // [nl][L]
    std::vector<std::pair<uint64_t, uint64_t>> segs;       // genomic [begin, end] (1-based) of the alignment's columns, in its order
    std::vector<int64_t> reg_begin, reg_end;               // coding: region 0 = whole, then one per CDS line (file order)
};

class ChainIndex {
public:
    struct Entry { int64_t start, end; int file; size_t chain; int ref_id; };   // reference positions [start, end), 1-based

    ChainIndex(const std::vector<std::string> &paths, const Model &model, int threads) : nl_(model.nl()) {
        for (const std::string &p : paths) {
            mafs_.emplace_back(new MafFile(p, model, true, threads, true));
            const std::vector<MafFile::Chain> &chains = mafs_.back()->chains();
            for (size_t ci = 0; ci < chains.size(); ++ci) {
                const MafFile::Chain &c = chains[ci];
                if (c.ref_id < 0) continue;
                if (c.strand != '+') { ++minus_chains_; continue; }
                by_chrom_[c.chrom].push_back(Entry{c.start_pos, c.start_pos + c.ref_cols, (int)mafs_.size() - 1, ci, c.ref_id});
            }
        }
        for (auto &kv : by_chrom_)
            std::stable_sort(kv.second.begin(), kv.second.end(), [](const Entry &a, const Entry &b) { return a.start < b.start; });
    }
    const std::vector<std::unique_ptr<MafFile>> &mafs() const { return mafs_; }
    int64_t minus_chains() const { return minus_chains_; }
    int nl() const { return nl_; }
    const std::vector<Entry> *chrom(const std::string &name) const {
        auto it = by_chrom_.find(name);
        return it == by_chrom_.end() ? nullptr : &it->second;
    }

private:
    int nl_;
    std::vector<std::unique_ptr<MafFile>> mafs_;
    std::map<std::string, std::vector<Entry>> by_chrom_;
    int64_t minus_chains_ = 0;
};

// The chains a worker has parsed last (most recent first): transcripts near each other in an annotation share their chains.
class ChainCache {
public:
    explicit ChainCache(const ChainIndex &idx, size_t cap = 8) : idx_(idx), cap_(cap) {}
    const Alignment &get(const ChainIndex::Entry &e) {
        for (auto it = lru_.begin(); it != lru_.end(); ++it)
            if (it->first.first == e.file && it->first.second == e.chain) {
                lru_.splice(lru_.begin(), lru_, it);
                return lru_.front().second;
            }
        if (lru_.size() >= cap_) lru_.pop_back();
        lru_.emplace_front(std::make_pair(e.file, e.chain), Alignment{});
        const MafFile &maf = *idx_.mafs()[(size_t)e.file];
        maf.read_chain(maf.chains()[e.chain], lru_.front().second, nullptr);
        return lru_.front().second;
    }

private:
    const ChainIndex &idx_;
    size_t cap_;
    std::list<std::pair<std::pair<int, size_t>, Alignment>> lru_;
};

// Reference positions [b, e] (1-based, inclusive) of `chrom` into columns [d, d + e - b + 1) of the [nl][ld] matrix `out`; the reference
// rows of the chains used are merged into *ref_row (-1 none yet, -2 disagreeing).
inline void extract_interval(const ChainIndex &idx, ChainCache &cache, const std::string &chrom, int64_t b, int64_t e, uint8_t *out,
                             int64_t ld, int64_t d, int *ref_row) {
    const int nl = idx.nl();
    const std::vector<ChainIndex::Entry> *ent = idx.chrom(chrom);
    for (int64_t p = b; p <= e;) {
        // the chain that starts last at or before p covers p if p < its end; a run stops where the next chain starts
        int64_t k = -1, next_start = INT64_MAX;
        if (ent) {
            auto it = std::upper_bound(ent->begin(), ent->end(), p, [](int64_t v, const ChainIndex::Entry &x) { return v < x.start; });
            if (it != ent->end()) next_start = it->start;
            if (it != ent->begin()) k = (int64_t)(it - ent->begin()) - 1;
        }
        const ChainIndex::Entry *c = k >= 0 && p < (*ent)[(size_t)k].end ? &(*ent)[(size_t)k] : nullptr;
        int64_t q = std::min(e + 1, next_start);
        if (c) {
            q = std::min(q, c->end);
            const Alignment &a = cache.get(*c);
            const int64_t j0 = p - c->start, have = std::max<int64_t>(0, std::min<int64_t>(q - p, a.L - j0));
            for (int s = 0; s < nl; ++s) {
                uint8_t *o = out + (size_t)s * ld + d + (p - b);
                if (have) memcpy(o, a.seqs.data() + (size_t)s * a.L + j0, (size_t)have);
                if (have < q - p) memset(o + have, 'N', (size_t)(q - p - have));          // text shorter than its size fields
            }
            *ref_row = *ref_row == -1 ? c->ref_id : (*ref_row == c->ref_id ? *ref_row : -2);
        } else {
            for (int s = 0; s < nl; ++s) memset(out + (size_t)s * ld + d + (p - b), 'N', (size_t)(q - p));
        }
        p = q;
    }
}

inline void reverse_complement(uint8_t *row, int64_t n) {
    static const struct Lut {
        uint8_t t[256];
        Lut() {
            for (int i = 0; i < 256; ++i) t[i] = (uint8_t)i;
            const char *a = "ACGTacgt", *b = "TGCAtgca";
            for (int i = 0; i < 8; ++i) t[(uint8_t)a[i]] = (uint8_t)b[i];
        }
    } lut;
    std::reverse(row, row + n);
    for (int64_t i = 0; i < n; ++i) row[i] = lut.t[row[i]];
}

inline uint8_t cds_phase(const CdsEntry &c) { return c.phase <= 2 ? c.phase : 0; }          // '.' or anything else: 0

// The alignment of transcript t: coding (CDS features) or, with find_orf, its exons.  Returns false for a record that is not scored
// (no `transcript` line, or no CDS without find_orf).
inline bool extract_transcript(const ChainIndex &idx, ChainCache &cache, const GffTranscript &t, bool find_orf, TxAlignment &x) {
    bool has_tx = false;
    for (const auto &ln : t.lines) has_tx |= ln.first == Feature::Transcript;
    if (!has_tx || (t.cds.empty() && !find_orf)) return false;
    const int nl = idx.nl();
    x = TxAlignment{};
    x.coding = !t.cds.empty();
    x.strand = t.strand == '-' ? '-' : '+';
    const bool minus = x.strand == '-';
    std::vector<std::pair<uint64_t, uint64_t>> iv;          // genomic order
    std::vector<size_t> order;                              // coding: CDS line index of iv[k]
    if (x.coding) {
        for (size_t i = 0; i < t.cds.size(); ++i) order.push_back(i);
        std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return t.cds[a].begin < t.cds[b].begin; });
        for (size_t i : order) iv.emplace_back(t.cds[i].begin, t.cds[i].end);
    } else {
        iv = t.exons.empty() ? std::vector<std::pair<uint64_t, uint64_t>>{{t.begin, t.end}} : t.exons;
        std::stable_sort(iv.begin(), iv.end(), [](const std::pair<uint64_t, uint64_t> &a, const std::pair<uint64_t, uint64_t> &b) { return a.first < b.first; });
    }
    std::vector<int64_t> goff(iv.size() + 1, 0), glen(iv.size());
    for (size_t k = 0; k < iv.size(); ++k) {
        glen[k] = iv[k].second >= iv[k].first ? (int64_t)(iv[k].second - iv[k].first + 1) : 0;
        goff[k + 1] = goff[k] + glen[k];
    }
    const int64_t Lraw = goff.back();
    std::vector<uint8_t> raw((size_t)nl * Lraw);
    for (size_t k = 0; k < iv.size(); ++k)
        if (glen[k]) extract_interval(idx, cache, t.chr, (int64_t)iv[k].first, (int64_t)iv[k].second, raw.data(), Lraw, goff[k], &x.ref_row);
    if (minus)
        for (int s = 0; s < nl; ++s) reverse_complement(raw.data() + (size_t)s * Lraw, Lraw);
    int64_t drop = 0;
    if (x.coding) drop = std::min<int64_t>(cds_phase(t.cds[minus ? order.back() : order.front()]), Lraw);
    x.L = Lraw - drop;
    x.seqs.resize((size_t)nl * x.L);
    for (int s = 0; s < nl; ++s) memcpy(x.seqs.data() + (size_t)s * x.L, raw.data() + (size_t)s * Lraw + drop, (size_t)x.L);
    for (size_t k = 0; k < iv.size(); ++k) if (glen[k]) x.segs.push_back(iv[k]);
    if (minus) std::reverse(x.segs.begin(), x.segs.end());
    if (x.coding) {
        x.reg_begin.push_back(0);
        x.reg_end.push_back(x.L);
        std::vector<int64_t> tpos(t.cds.size());          // first column of each CDS line in transcript orientation, before the drop
        for (size_t k = 0; k < order.size(); ++k) tpos[order[k]] = minus ? Lraw - goff[k + 1] : goff[k];
        for (size_t i = 0; i < t.cds.size(); ++i) {
            const size_t k = (size_t)(std::find(order.begin(), order.end(), i) - order.begin());
            const int64_t e = std::max<int64_t>(0, tpos[i] + glen[k] - drop);
            x.reg_begin.push_back(std::min(e, std::max<int64_t>(0, tpos[i] - drop + cds_phase(t.cds[i]))));
            x.reg_end.push_back(e);
        }
    }
    return true;
}

// 1-based genomic position of alignment column j (before any dropped phase: the ORF search runs on exon alignments, which drop none)
inline uint64_t genomic_position(const TxAlignment &x, int64_t j) {
    for (const auto &sg : x.segs) {
        const int64_t n = (int64_t)(sg.second - sg.first + 1);
        if (j < n) return x.strand == '-' ? sg.second - (uint64_t)j : sg.first + (uint64_t)j;
        j -= n;
    }
    return 0;
}

// Polynomial hash of columns [b, e) of every row, row after row: sum of byte_i * P^(i+1) mod 2^64 (numpy computes it in one pass)
inline uint64_t region_hash(const TxAlignment &x, int nl, int64_t b, int64_t e) {
    const uint64_t P = 1099511628211ull;
    uint64_t h = 0, pw = 1;
    for (int s = 0; s < nl; ++s)
        for (int64_t j = b; j < e; ++j) { pw *= P; h += (uint64_t)x.seqs[(size_t)s * x.L + j] * pw; }
    return h;
}

}  // namespace host
