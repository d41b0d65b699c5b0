// annotate.hpp — `annotate-with-tracks`: power-weighted PhyloCSF scores of the CDS features of GFF/GTF files from finished
// bigWig tracks (SURVEY §8 f-4; reference src/phylocsf++annotate_with_tracks.hpp:26-60 count_weighted_scores, :62-218
// run_annotate_with_tracks, :220-305 command line; transcript iterator src/gff_reader.hpp:121-227).
//
// A consumer of the tracks build-tracks writes: pure I/O and float sums, so it stays on the host.  What has to match the
// reference byte for byte is the text of the annotated files, hence:
//   * transcripts are the runs of lines from one `transcript` feature up to the next (gff_reader.hpp:195-203); everything that is
//     not `transcript` / `CDS` is copied through, also when the transcript has no CDS;
//   * the frame track of a CDS: '+': (phase + begin - 1) % 3, '-': 3 + (chrom_len - end - 1 + phase + 1) % 3 with the phase
//     character minus '0' kept as an unsigned byte ('.' = 254) and unsigned 64-bit arithmetic (annotate_with_tracks.hpp:131-135);
//   * all sums are floats accumulated position by position in file order (:36-52), the per-transcript sums are the sums of the
//     per-CDS sums (:148-151); score = Σ v·p / Σ p over positions where both tracks have a value, power = Σ p / #positions;
//   * a chromosome missing from the tracks gives nan / nan (gff_reader.hpp:15-16 defaults);
//   * GFF3 (`key=value`) or GTF (`key "value";`) is detected on the first annotated line of every transcript (common.hpp:98-122).
#pragma once

#include <set>
#include <tuple>

#include "bigwig.hpp"
#include "util.hpp"

namespace host {

struct CdsEntry { uint64_t begin, end; uint8_t phase; float score = NAN, power = NAN; };
enum class Feature { Transcript, Cds, Other };

struct GffTranscript {
    std::string chr;
    char strand = '.';
    uint64_t begin = 0, end = 0;                               // of the `transcript` line
    std::vector<std::pair<uint64_t, uint64_t>> exons;         // `exon` features [begin, end] in file order (their lines stay Other)
    float score = NAN, power = NAN;
    std::vector<CdsEntry> cds;
    std::vector<std::pair<Feature, std::string>> lines;
};

class GffReader {
public:
    explicit GffReader(const std::string &path) {
        FILE *f = fopen(path.c_str(), "rb");
        if (!f) die("Cannot open %s", path.c_str());
        char buf[1 << 16];
        size_t n;
        while ((n = fread(buf, 1, sizeof buf, f)) > 0) text_.append(buf, n);
        fclose(f);
    }
    size_t size() const { return text_.size(); }
    bool ends_with_newline() const { return !text_.empty() && text_.back() == '\n'; }
    size_t pos() const { return pos_; }

    bool next(GffTranscript &t) {
        if (pos_ >= text_.size()) return false;
        int transcripts = 0;
        t.cds.clear();
        t.exons.clear();
        t.lines.clear();
        while (pos_ < text_.size()) {
            size_t le = text_.find('\n', pos_);
            if (le == std::string::npos) le = text_.size();
            // columns 1, 3, 4, 5, 7, 8 (tab separated)
            std::string chr, feature;
            uint64_t begin = 0, end = 0;
            char strand = '.', phase = '.';
            size_t p = pos_;
            for (int col = 1; p < le; ++col) {
                size_t q = text_.find('\t', p);
                if (q == std::string::npos || q > le) q = le;
                switch (col) {
                    case 1: chr.assign(text_, p, q - p); break;
                    case 3: feature.assign(text_, p, q - p); break;
                    case 4: begin = strtoull(text_.c_str() + p, nullptr, 10); break;
                    case 5: end = strtoull(text_.c_str() + p, nullptr, 10); break;
                    case 7: strand = text_[p]; break;
                    case 8: phase = text_[p]; break;
                    default: break;
                }
                p = q + 1;
            }
            if (feature == "transcript" && ++transcripts > 1) break;          // belongs to the next record
            Feature f = Feature::Other;
            if (feature == "transcript") {
                f = Feature::Transcript;
                t.chr = chr;
                t.strand = strand;
                t.begin = begin;
                t.end = end;
            } else if (feature == "CDS") {
                f = Feature::Cds;
                t.cds.push_back(CdsEntry{begin, end, (uint8_t)(phase - '0')});
            } else if (feature == "exon") {
                t.exons.emplace_back(begin, end);
            }
            t.lines.emplace_back(f, text_.substr(pos_, le - pos_));
            pos_ = le + 1;
        }
        return true;
    }

private:
    std::string text_;
    size_t pos_ = 0;
};

inline bool is_gff_line(const std::string &line) {          // common.hpp:98-122
    int col = 1;
    for (size_t i = 0; i < line.size(); ++i) {
        if (col == 9) {
            for (; i < line.size(); ++i) {
                if (line[i] == ' ') return false;
                if (line[i] == '=') return true;
            }
            return true;
        }
        if (line[i] == '\t') ++col;
    }
    return true;
}

struct TrackSet {
    BigWigReader bw[7];          // +1 +2 +3 -1 -2 -3 power
    std::string first_path;
};

// count_weighted_scores (annotate_with_tracks.hpp:26-60)
inline void weighted_scores(float &score_sum, float &weighted_power, float &all_power, uint64_t &count, BigWigReader &track, BigWigReader &power,
                            const std::string &chrom, uint64_t begin, uint64_t end, std::vector<float> &v, std::vector<float> &p) {
    const bool a = track.values(chrom, (uint32_t)begin, (uint32_t)end, v);
    const bool b = power.values(chrom, (uint32_t)begin, (uint32_t)end, p);
    if (!a || !b) return;
    for (size_t i = 0; i < v.size(); ++i) {
        if (!std::isnan(v[i]) && !std::isnan(p[i])) {
            score_sum += v[i] * p[i];
            weighted_power += p[i];
        }
        if (!std::isnan(p[i])) all_power += p[i];
        ++count;
    }
}

inline void annotate_file(const std::string &gff_path, const std::string &output_dir, TrackSet &tracks, std::set<std::string> &missing,
                          const std::string &version_line) {
    GffReader reader(gff_path);
    std::string out_path = output_dir.empty() ? gff_path : output_dir + "/" + gff_path.substr(gff_path.find_last_of('/') == std::string::npos ? 0 : gff_path.find_last_of('/') + 1);
    const size_t dot = out_path.find_last_of('.');
    if (dot == std::string::npos) out_path += ".PhyloCSF++";
    else out_path.insert(dot, ".PhyloCSF++");
    FILE *fo = fopen(out_path.c_str(), "w");
    if (!fo) die("Error creating file %s!", out_path.c_str());
    fputs(version_line.c_str(), fo);
    GffTranscript t;
    std::vector<float> v, p;
    while (reader.next(t)) {
        if (!t.cds.empty()) {
            const BigWigReader::Chrom *chrom = tracks.bw[0].find(t.chr);
            if (!chrom) {
                t.score = t.power = NAN;
                if (missing.insert(t.chr).second) printf("\33[2K\rSequence %s from the GFF file does not occur in the tracks. Skipping ...\n", t.chr.c_str());
            } else {
                const uint64_t chr_len = chrom->len;
                float t_sum = 0.f, t_wpower = 0.f, t_apower = 0.f;
                uint64_t t_count = 0;
                for (CdsEntry &c : t.cds) {
                    const unsigned frame = t.strand == '+' ? (unsigned)((c.phase + c.begin - 1) % 3) : 3u + (unsigned)((chr_len - c.end - 1 + c.phase + 1) % 3);
                    float sum = 0.f, wpower = 0.f, apower = 0.f;
                    uint64_t count = 0;
                    weighted_scores(sum, wpower, apower, count, tracks.bw[frame], tracks.bw[6], t.chr, c.begin - 1, c.end, v, p);
                    c.score = sum / wpower;
                    c.power = count == 0 ? 0.f : apower / count;
                    t_sum += sum; t_wpower += wpower; t_apower += apower; t_count += count;
                }
                t.score = t_sum / t_wpower;
                t.power = t_count == 0 ? 0.f : t_apower / t_count;
            }
        }
        bool first = true, gff = true;
        size_t cds_id = 0;
        for (const auto &ln : t.lines) {
            if (ln.first == Feature::Other || t.cds.empty()) {
                fprintf(fo, "%s\n", ln.second.c_str());
                continue;
            }
            if (first) { first = false; gff = is_gff_line(ln.second); }
            float score, power;
            if (ln.first == Feature::Transcript) { score = t.score; power = t.power; }
            else { score = t.cds[cds_id].score; power = t.cds[cds_id].power; ++cds_id; }
            if (std::isnan(score)) score = NAN;          // never "-nan"
            if (gff) fprintf(fo, "%s;phylocsf_score_weighted_mean=%.3f;phylocsf_power_mean=%.3f\n", ln.second.c_str(), score, power);
            else fprintf(fo, "%s phylocsf_score_weighted_mean \"%.3f\"; phylocsf_power_mean \"%.3f\";\n", ln.second.c_str(), score, power);
        }
    }
    fclose(fo);
}

// The seven track paths from the +1 path ("PhyloCSF+1.bw" -> +2, +3, -1, -2, -3, power), annotate_with_tracks.hpp:254-266
inline std::vector<std::string> track_paths(const std::string &plus1) {
    const size_t at = plus1.find("+1");
    if (at == std::string::npos) die("Could not find '+1' in tracks file name. Expecting a name like 'PhyloCSF+1.bw'.");
    std::vector<std::string> out;
    static const char *suffix[7] = {"+1", "+2", "+3", "-1", "-2", "-3", "power"};
    // the reference replaces two characters at the position of "+1" in the path it has just edited: after "power" (5 characters) it
    // would be off, but power comes last
    for (int i = 0; i < 7; ++i) { std::string s = plus1; s.replace(at, 2, suffix[i]); out.push_back(s); }
    return out;
}

inline bool open_tracks(const std::string &plus1, TrackSet &ts) {
    ts.first_path = plus1;
    const std::vector<std::string> paths = track_paths(plus1);
    for (int i = 0; i < 7; ++i) {
        std::string err;
        if (!ts.bw[i].open(paths[i], err)) {
            const std::string &bp = paths[i];
            if (access(bp.c_str(), F_OK) == 0 && bp.size() >= 4 && bp.compare(bp.size() - 4, 4, ".wig") == 0) {
                printf("\033[31mAn error occurred while opening the PhyloCSF file '%s'.\n\033[0m", bp.c_str());
                printf("It seems you provided a *.wig file. You need to simply index them first with wigToBigWig (or phylocsf_b200 wig-to-bigwig) and then use the *.bw files.\n");
            } else if (access(bp.c_str(), F_OK) == 0) {
                printf("\033[31m%s\n\033[0m", err.c_str());
            } else {
                printf("\033[31mCould not find PhyloCSF track file '%s'.\n\033[0m", bp.c_str());
            }
            return false;
        }
    }
    return true;
}

// ------------------------------------------------------------------------------------------------ wig text -> bigWig
// Streams a fixedStep / variableStep wig file (what build-tracks writes) into a BigWigWriter.  chrom_sizes: "name<TAB>length" lines.
inline std::vector<std::pair<std::string, uint32_t>> read_chrom_sizes(const std::string &path) {
    std::vector<std::pair<std::string, uint32_t>> out;
    FILE *f = fopen(path.c_str(), "r");
    if (!f) die("Cannot open %s", path.c_str());
    char name[1024];
    unsigned long long len;
    while (fscanf(f, "%1023s %llu", name, &len) == 2) out.emplace_back(name, (uint32_t)len);
    fclose(f);
    if (out.empty()) die("%s holds no 'chromosome length' lines", path.c_str());
    return out;
}

inline void wig_to_bigwig(const std::string &wig_path, const std::vector<std::pair<std::string, uint32_t>> &chroms, const std::string &bw_path, bool compress = true) {
    // The file is mapped and indexed run by run first: a bigWig stores its data ordered by chromosome id (= rank of the name in
    // the chromosome tree) and position, a wig file written chromosome file after chromosome file need not be in that order.
    int fd = ::open(wig_path.c_str(), O_RDONLY);
    if (fd < 0) die("Cannot open %s", wig_path.c_str());
    struct stat st;
    fstat(fd, &st);
    const size_t size = (size_t)st.st_size;
    const char *mem = size ? (const char *)mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0) : nullptr;
    ::close(fd);
    if (size && mem == MAP_FAILED) die("Cannot map %s", wig_path.c_str());
    struct Run { std::string chrom; uint32_t rank, start0, step, span; size_t begin, end; };
    std::vector<Run> runs;
    std::map<std::string, uint32_t> rank;
    {
        std::vector<std::string> names;
        for (auto &c : chroms) names.push_back(c.first);
        std::sort(names.begin(), names.end());
        for (size_t i = 0; i < names.size(); ++i) rank[names[i]] = (uint32_t)i;
    }
    for (size_t p = 0; p < size;) {
        const char *nlp = (const char *)memchr(mem + p, '\n', size - p);
        const size_t le = nlp ? (size_t)(nlp - mem) : size;
        if (mem[p] == 'f') {                                          // fixedStep chrom=chr22 start=200002 step=3 span=3
            if (!runs.empty()) runs.back().end = p;
            Run r{"", 0, 0, 1, 1, le + 1, size};
            unsigned long long start1 = 0;
            std::string line(mem + p, le - p);
            char *save = nullptr;          // strtok_r: build-tracks converts its wig files on parallel threads
            for (char *tok = strtok_r(&line[0], " \t\r", &save); tok; tok = strtok_r(nullptr, " \t\r", &save)) {
                if (!strncmp(tok, "chrom=", 6)) r.chrom = tok + 6;
                else if (!strncmp(tok, "start=", 6)) start1 = strtoull(tok + 6, nullptr, 10);
                else if (!strncmp(tok, "step=", 5)) r.step = (uint32_t)strtoul(tok + 5, nullptr, 10);
                else if (!strncmp(tok, "span=", 5)) r.span = (uint32_t)strtoul(tok + 5, nullptr, 10);
            }
            if (r.chrom.empty() || start1 == 0) die("%s: malformed fixedStep line at byte %zu", wig_path.c_str(), p);
            auto it = rank.find(r.chrom);
            if (it == rank.end()) die("%s: chromosome %s is not in the chromosome sizes", wig_path.c_str(), r.chrom.c_str());
            r.rank = it->second;
            r.start0 = (uint32_t)(start1 - 1);
            runs.push_back(r);
        } else if (mem[p] == 'v') {
            die("%s: variableStep wig files are not supported (build-tracks writes fixedStep)", wig_path.c_str());
        } else if (runs.empty() && le > p && mem[p] != '#' && strncmp(mem + p, "track", 5) && strncmp(mem + p, "browser", 7)) {
            die("%s: values before the first fixedStep line", wig_path.c_str());
        }
        p = le + 1;
    }
    std::stable_sort(runs.begin(), runs.end(), [](const Run &a, const Run &b) { return a.rank != b.rank ? a.rank < b.rank : a.start0 < b.start0; });
    BigWigWriter w;
    std::string err;
    if (!w.open(bw_path, chroms, err, compress)) die("%s", err.c_str());
    std::vector<float> vals;
    for (const Run &r : runs) {
        vals.clear();
        for (size_t p = r.begin; p < r.end;) {
            const char *nlp = (const char *)memchr(mem + p, '\n', r.end - p);
            const size_t le = nlp ? (size_t)(nlp - mem) : r.end;
            if (le > p && mem[p] != '#' && mem[p] != '\r') {
                char buf[64];
                const size_t n = std::min<size_t>(le - p, sizeof buf - 1);
                memcpy(buf, mem + p, n);
                buf[n] = 0;
                vals.push_back(strtof(buf, nullptr));
            }
            p = le + 1;
        }
        if (!vals.empty() && !w.add_fixed_step(r.chrom, r.start0, r.step, r.span, vals.data(), vals.size(), err)) die("%s: %s", wig_path.c_str(), err.c_str());
    }
    if (mem) munmap((void *)mem, size);
    if (!w.finish(err)) die("%s: %s", bw_path.c_str(), err.c_str());
}

}  // namespace host
