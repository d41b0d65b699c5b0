// phylocsf_b200 — reference-compatible command line host over libphylocsf_b200.so (include/phylocsf_b200.h).
//
//   phylocsf_b200 build-tracks [OPTIONS] <model> <alignments>...    (reference src/phylocsf++build_tracks.hpp:367-507)
//   phylocsf_b200 score-msa    [OPTIONS] <model> <alignments>...    (reference src/phylocsf++score_msa.hpp:245-385)
//
// The host keeps what the reference keeps on the CPU: option handling (options before positionals,
// src/arg_parse.hpp:111-115; BOOL = 1/true/one, :303), model loading, MAF reading, wig / scores text.  The likelihood
// core is the CUDA library; there is no CPU fallback.  Worker threads parse whole alignment chains, call the C-ABI on
// their GPU (thread t -> GPU t mod --gpus) and format the text; a writer appends the results in file order, so the
// output does not depend on the thread or GPU count (the reference merges its per-job files in job order,
// build_tracks.hpp:27-53,245-259).
// --output-phylo / --output-regions: the PhyloCSF-HMM smoothing of the raw tracks stays on the host (hmm.hpp).
#include <cinttypes>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <cmath>

#include "annotate.hpp"
#include "hmm.hpp"
#include "maf.hpp"
#include "transcripts.hpp"

using namespace host;

namespace {

struct Args {
    std::map<std::string, std::string> opt;
    std::vector<std::string> pos;
    bool has(const std::string &k) const { return opt.count(k) > 0; }
    std::string str(const std::string &k, const std::string &dflt = "") const { auto it = opt.find(k); return it == opt.end() ? dflt : it->second; }
    bool boolean(const std::string &k, bool dflt) const {        // arg_parse.hpp:303
        auto it = opt.find(k);
        if (it == opt.end()) return dflt;
        const std::string v = lower(it->second);
        return v == "1" || v == "true" || v == "one";
    }
    int integer(const std::string &k, int dflt) const { auto it = opt.find(k); return it == opt.end() ? dflt : atoi(it->second.c_str()); }
};

Args parse_args(int argc, char **argv, const std::set<std::string> &known) {
    Args a;
    int i = 2;
    for (; i < argc; ++i) {
        const std::string t = argv[i];
        if (t.rfind("--", 0) != 0) break;
        const std::string k = t.substr(2);
        if (!known.count(k)) die("Unknown option '%s'", t.c_str());
        if (i + 1 >= argc) die("Option '%s' needs a value", t.c_str());
        a.opt[k] = argv[++i];
    }
    for (; i < argc; ++i) {
        if (strncmp(argv[i], "--", 2) == 0) die("Options have to be specified before the positional arguments ('%s')", argv[i]);
        a.pos.push_back(argv[i]);
    }
    return a;
}

uint32_t precision_flag(const Args &a) {
    const std::string p = lower(a.str("precision", "f64"));
    if (p == "f64") return 0;
    if (p == "tc5") return PCSF_TRACKS_TC5;
    die("--precision must be f64 or tc5");
}

int64_t mod3(int64_t x) { x %= 3; return x < 0 ? x + 3 : x; }

// In-order hand-over of per-chain text from the workers to the writer.
struct OrderedSink {
    std::mutex mu;
    std::condition_variable cv;
    std::vector<std::vector<std::string>> slots;      // [chain][stream]
    std::vector<uint8_t> ready;
    void resize(size_t n) { slots.assign(n, {}); ready.assign(n, 0); }
    void put(size_t i, std::vector<std::string> &&v) {
        { std::lock_guard<std::mutex> g(mu); slots[i] = std::move(v); ready[i] = 1; }
        cv.notify_all();
    }
    std::vector<std::string> take(size_t i) {
        std::unique_lock<std::mutex> g(mu);
        cv.wait(g, [&] { return ready[i] != 0; });
        return std::move(slots[i]);
    }
};

// Device models are pooled: two per GPU (one call can copy while the other computes); more host threads inside the library
// would only contend for the device and the driver.  ONE pool over all GPUs, dealt dynamically like the reference's
// `schedule(dynamic, 1)` jobs (build_tracks.hpp:88): a worker takes whichever model is free, on the GPU with the fewest calls in
// flight.  Models join the pool as soon as they exist, so the first groups are scored while the CUDA contexts of the other devices
// are still coming up (eight contexts take ~1.5 s); the output does not depend on who scored what.
struct ModelPool {
    std::mutex mu;
    std::condition_variable cv;
    struct Entry { pcsf_model *m; int dev; };
    std::vector<Entry> free_models, all;
    std::vector<int> busy;          // calls in flight per GPU
    explicit ModelPool(int gpus) : busy(gpus, 0) {}
    void add(pcsf_model *m, int dev) { { std::lock_guard<std::mutex> g(mu); free_models.push_back({m, dev}); all.push_back({m, dev}); } cv.notify_all(); }
    Entry acquire() {
        std::unique_lock<std::mutex> g(mu);
        cv.wait(g, [&] { return !free_models.empty(); });
        size_t best = 0;
        for (size_t i = 1; i < free_models.size(); ++i) if (busy[free_models[i].dev] < busy[free_models[best].dev]) best = i;
        const Entry e = free_models[best];
        free_models.erase(free_models.begin() + (long)best);
        ++busy[e.dev];
        return e;
    }
    void release(const Entry &e) { { std::lock_guard<std::mutex> g(mu); free_models.push_back(e); --busy[e.dev]; } cv.notify_one(); }
    void destroy() { for (const Entry &e : all) pcsf_model_destroy(e.m); all.clear(); free_models.clear(); }
};

int default_gpus() { return std::max(1, pcsf_device_count()); }

// One thread per GPU prepares that GPU's models one after the other (host work: eigensystem, all P(t), tables; then the uploads) and
// hands each to the pool as soon as it exists; `stop` (all groups scored) skips models nobody will need any more.  CUDA contexts are
// brought up two devices at a time (GPU g waits for the first model of GPU g-2): eight contexts created at once all become usable
// together after ~1.5 s (measured: first model after 0.30-0.43 s with one or two devices, 1.45 s with eight), staggered the first
// two devices score while the others are still coming up.  `allowed` is how many devices the job is worth (set after the scan, see
// the caller): devices beyond it are never initialised.
void fill_pool(const Model &model, int gpus, int per_gpu, ModelPool &pool, const std::atomic<bool> &stop, const std::atomic<int> &allowed,
               const std::function<void(pcsf_model *)> &configure) {
    std::vector<std::thread> th;
    std::mutex mu;
    std::condition_variable cv;
    std::vector<char> up(gpus, 0);          // GPU g has its first model (or gave up)
    for (int g = 0; g < gpus; ++g)
        th.emplace_back([&, g] {
            {
                std::unique_lock<std::mutex> l(mu);
                // `allowed` changes once (0 = not decided yet for g >= 2) and `stop` once: poll them with a short timeout
                while (!stop && !((g < 2 || up[g - 2] != 0) && (g < 2 || allowed.load() != 0))) cv.wait_for(l, std::chrono::milliseconds(2));
            }
            const int lim = allowed.load() == 0 ? std::min(gpus, 2) : allowed.load();
            for (int k = 0; k < per_gpu && !stop && g < lim; ++k) {
                pcsf_model *m = create_device_model(model, g);
                configure(m);
                pool.add(m, g);
                if (k == 0) { { std::lock_guard<std::mutex> l(mu); up[g] = 1; } cv.notify_all(); }
            }
            { std::lock_guard<std::mutex> l(mu); up[g] = 1; }
            cv.notify_all();
        });
    for (auto &t : th) t.join();
}

void warn_unresolved(const MafFile &maf) {
    for (const std::string &s : maf.unresolved())
        printf("\033[33mWARNING: Not able to match species %s in alignment file to model (Use `--mapping` to fix it)!\033[0m\n", s.c_str());
}

// --model-info NAME (run.hpp:213-232): the species of a model with their alternative names; no GPU involved.
int print_model_info(const std::string &model_name) {
    Model model;
    load_model(model, model_name, "", "");
    printf("The model %s contains the following species.\n\n", model_name.c_str());
    printf("%35s\t%s\n", "Species name", "Alternative name(s)");
    for (const std::string &label : model.tree.labels) {
        if (label.empty()) continue;
        std::string alt;
        auto it = model.aliases.find(label);
        if (it != model.aliases.end()) for (const std::string &sn : it->second) alt += sn + " ";
        printf("%35s\t%s\n", label.c_str(), alt.c_str());
    }
    return 0;
}

// ------------------------------------------------------------------------------------------- build-tracks
int main_build_tracks(int argc, char **argv) {
    const auto t_entry = std::chrono::steady_clock::now();
    const Args a = parse_args(argc, argv, {"output-raw-phylo", "output-phylo", "output-regions", "power-threshold", "genome-length", "coding-exons",
                                           "threads", "output", "mapping", "species", "gpus", "precision", "model-info", "output-bigwig"});
    if (a.has("model-info")) return print_model_info(a.str("model-info"));          // build_tracks.hpp:401-405
    if (a.pos.size() < 2) die("usage: phylocsf_b200 build-tracks [OPTIONS] <model> <alignments>...");
    const bool keep_raw = a.boolean("output-raw-phylo", true);
    const bool smooth = a.boolean("output-phylo", false), regions = a.boolean("output-regions", false);
    if ((smooth || regions) && (!a.has("genome-length") || !a.has("coding-exons"))) {          // build_tracks.hpp:420-432
        printf("\033[31m%s\n\033[0m", smooth ? "For smoothened tracks (--output-phylo) you need to provide --genome-length and --coding-exons."
                                             : "To generate bed file of potential protein coding regions, you need to provide --genome-length and --coding-exons.");
        return -1;
    }
    const bool raw = keep_raw || smooth || regions;          // the raw tracks are the HMM's input (build_tracks.hpp:109,248)
    // --output-bigwig 1: every wig file written is also indexed as <name>.bw (the reference leaves that to UCSC's wigToBigWig); the
    // chromosome lengths are the srcSize fields of the reference rows
    const bool to_bigwig = a.boolean("output-bigwig", false);
    Hmm hmm_model{};
    if (smooth || regions)          // models.hpp:1760-1764 (the reference estimates only for --output-phylo and leaves the HMM unset for regions alone)
        hmm_model = coding_hmm(estimate_hmm_params(a.str("coding-exons"), (uint32_t)strtoull(a.str("genome-length").c_str(), nullptr, 10)));
    // the reference reads --power-threshold with get_bool (build_tracks.hpp:416-417): anything but 1/true/one gives 0
    const float threshold = a.has("power-threshold") ? (a.boolean("power-threshold", false) ? 1.0f : 0.0f) : 0.1f;
    const int threads = std::max(1, a.integer("threads", (int)std::thread::hardware_concurrency()));
    const int gpus = std::max(1, a.integer("gpus", default_gpus()));          // all visible devices unless told otherwise
    const uint32_t pflag = precision_flag(a);

    Model model;
    load_model(model, a.pos[0], a.str("species"), a.str("mapping"));
    const int nl = model.nl();
    // Start-up overlaps three things: the device models (CUDA context + eigensystems + uploads, two per GPU) are prepared by their own
    // threads while the input files are scanned and cut into chains, and while the page-locked staging slab is allocated.
    const auto t_start = std::chrono::steady_clock::now();
    ModelPool pool(gpus);
    std::atomic<bool> stop_models{false};
    std::atomic<int> allowed_gpus{0};          // decided after the scan: how many devices this input is worth
    const int per_gpu = getenv("PCSF_HOST_MODELS_PER_GPU") ? std::max(1, atoi(getenv("PCSF_HOST_MODELS_PER_GPU"))) : 2;
    const bool dev_timing = getenv("PCSF_HOST_TIMING") != nullptr;          // per-stage CUDA-event times of every library call (diagnostic)
    std::atomic<double> t_first_model{0.0};
    // A group is scored in pieces of PIECE_COLS columns through a small page-locked buffer owned by the worker thread: the piece is
    // copied in BEFORE a model is taken, so a model is held for the library call only (DMA in, kernels, DMA out) and the thread's own
    // copies overlap the calls of the others.  Pinning the workers' whole staging (16 x 82 MB) costs more than DMA copies save on
    // anything but very long runs (see below); 21 MB per thread costs 20 ms each, behind the model preparation.
    const int64_t PIECE_COLS = getenv("PCSF_HOST_PIECE_COLS") ? std::max<int64_t>(1024, atoll(getenv("PCSF_HOST_PIECE_COLS"))) : (1 << 18);
    const size_t pin_in_bytes = ((size_t)nl * (PIECE_COLS + 2) + 255) / 256 * 256, pin_vec_bytes = ((size_t)(PIECE_COLS + 2) * 8 + 255) / 256 * 256;
    const size_t pin_bytes = pin_in_bytes + 3 * pin_vec_bytes;
    std::thread pool_maker([&] {
        fill_pool(model, gpus, per_gpu, pool, stop_models, allowed_gpus, [&](pcsf_model *dm) {
            if (dev_timing) pcsf_set_timing(dm, 1);
            if (getenv("PCSF_HOST_CHUNK_COLS")) pcsf_set_chunk_columns(dm, atoll(getenv("PCSF_HOST_CHUNK_COLS")));
            double expect = 0.0;
            t_first_model.compare_exchange_strong(expect, std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count());
        });
    });
    std::vector<std::vector<uint8_t>> seen(threads, std::vector<uint8_t>(nl, 0));
    double t_parse = 0.0, t_format = 0.0, t_scan = 0.0, t_wait_model = 0.0, t_wait_writer = 0.0;
    double dev_ms[6] = {0, 0, 0, 0, 0, 0};
    int64_t dev_unique = 0, dev_windows = 0;
    static const char *kFrames[6] = {"+1", "+2", "+3", "-1", "-2", "-3"};
    int64_t total_cols = 0;
    double t_gpu = 0.0;

    // All input files are scanned first and their chain groups go into ONE work queue: the workers never wait at a file boundary
    // (chromosome-sized files used to end with a partially filled round of workers each); the writer still emits file after file.
    struct FileCtx { std::string path, out_dir; std::unique_ptr<MafFile> maf; size_t chain0 = 0; };
    struct Group { int file; size_t c0, c1; int64_t col_begin; };          // col_begin: reference columns of all chains before this group
    std::vector<FileCtx> fctx;
    std::vector<Group> groups;
    size_t total_chains = 0;
    int64_t cols_before = 0;
    for (size_t fi = 1; fi < a.pos.size(); ++fi) {
        FileCtx fc;
        fc.path = a.pos[fi];
        fc.out_dir = a.str("output");
        if (fc.out_dir.empty()) {
            const size_t p = fc.path.find_last_of('/');
            fc.out_dir = p == std::string::npos ? "./" : fc.path.substr(0, p);
        } else {
            create_directory(fc.out_dir);
        }
        const auto s0 = std::chrono::steady_clock::now();
        fc.maf.reset(new MafFile(fc.path, model, true, threads));
        t_scan += std::chrono::duration<double>(std::chrono::steady_clock::now() - s0).count();
        warn_unresolved(*fc.maf);
        fc.chain0 = total_chains;
        const std::vector<MafFile::Chain> &chains = fc.maf->chains();
        // consecutive chains are scored in one library call (their columns concatenated; the windows that straddle two
        // chains are computed and ignored): keeps the per-call cost off the many short chains of a gappy file
        const int64_t GROUP_COLS = getenv("PCSF_HOST_GROUP_COLS") ? atoll(getenv("PCSF_HOST_GROUP_COLS")) : (1 << 19);
        size_t g0 = 0;
        int64_t acc = 0;
        for (size_t ci = 0; ci < chains.size(); ++ci) {
            acc += chains[ci].ref_cols + 2;
            if (acc >= GROUP_COLS || ci + 1 == chains.size() || ci + 1 - g0 >= 4096) {
                groups.push_back(Group{(int)fctx.size(), g0, ci + 1, cols_before});
                cols_before += acc;
                g0 = ci + 1; acc = 0;
            }
        }
        total_chains += chains.size();
        fctx.push_back(std::move(fc));
    }
    // How many devices is this input worth?  Bringing a device up costs ~0.4 s during which the calls on the devices already working
    // slow down (measured on the 8-GPU box: 100 M columns take 1.22 s on two devices, 2.2 s when eight are brought up), and a device
    // scores ~60-100 M columns/s through this host: one device per 60 M columns (PCSF_HOST_USE_ALL_GPUS=1: all of --gpus).
    const int gpus_worth = getenv("PCSF_HOST_USE_ALL_GPUS") ? gpus : (int)std::min<int64_t>(gpus, std::max<int64_t>(1, (cols_before + 30000000) / 60000000));
    allowed_gpus = gpus_worth;
    // Staging, one region per worker, sized by the largest group (known exactly from the scan): plain page-aligned memory that the
    // workers parse into and format from.  (Page-locking it was measured in three ways — per thread, as one slab, in place in the
    // background — and always cost more than it saved below ~400 M columns: 1-2 GB/s, serialised in the driver, and the library
    // calls of the other threads crawl meanwhile.  The DMA path comes from the small per-model staging instead.)
    int64_t max_group_cols = 1;
    for (const Group &g : groups) {
        int64_t n = 0;
        const std::vector<MafFile::Chain> &chains = fctx[g.file].maf->chains();
        for (size_t ci = g.c0; ci < g.c1; ++ci) n += chains[ci].ref_id < 0 ? 0 : chains[ci].ref_cols;
        max_group_cols = std::max(max_group_cols, n);
    }
    const size_t mat_bytes = ((size_t)nl * max_group_cols + 4095) / 4096 * 4096, vec_bytes = ((size_t)max_group_cols * 8 + 4095) / 4096 * 4096;
    const size_t per_thread = mat_bytes + 3 * vec_bytes;
    const int slab_threads = (int)std::min<size_t>((size_t)threads, std::max<size_t>(groups.size(), 1));
    std::vector<uint8_t *> slabs(slab_threads, nullptr);
    for (auto &p : slabs)
        if (posix_memalign(reinterpret_cast<void **>(&p), 4096, per_thread) != 0) die("cannot allocate %zu bytes of staging memory", per_thread);
    double t_startup = 0.0;
    const double t_slab = 0.0;
    std::thread pool_waiter([&] {
        pool_maker.join();
        t_startup = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
    });
    OrderedSink sink;
    sink.resize(total_chains);
    std::atomic<size_t> next{0};
    std::atomic<int64_t> cols{0};
    std::vector<std::atomic<int64_t>> gpu_cols(gpus);          // reference columns scored per device (dynamic deal: whichever device has a free model)
    for (auto &g : gpu_cols) g = 0;
    std::mutex gpu_time_mu;
    // back-pressure: the workers run at most this many reference columns ahead of the writer (their finished text waits in memory,
    // about 16 bytes per column for the seven files)
    const int64_t AHEAD_COLS = (int64_t)64 << 20;
    std::mutex written_mu;
    std::condition_variable written_cv;
    int64_t written_cols = 0;
    std::vector<std::thread> workers;
    for (int t = 0; t < threads; ++t)
        workers.emplace_back([&, t] {
                if (t >= slab_threads) return;          // fewer groups than threads
                std::vector<Alignment> alns;
                uint8_t *const my_slab = slabs[t];
                uint8_t *my_pin = nullptr;          // page-locked piece buffer, allocated at the first call (after the thread's first parse)
                std::vector<uint8_t> fallback_mat;          // only for a group whose text disagrees with its size fields
                std::vector<double> fallback_out;
                const uint8_t *src = nullptr;
                double *plus = nullptr, *minus = nullptr, *bls = nullptr;
                double my_gpu = 0.0, my_parse = 0.0, my_fmt = 0.0, my_wait_model = 0.0, my_wait_writer = 0.0;
                auto now = [] { return std::chrono::steady_clock::now(); };
                auto secs = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double>(b - a).count(); };
                for (size_t gi = next++; gi < groups.size(); gi = next++) {
                    const Group &grp = groups[gi];
                    const auto w0 = now();
                    {
                        std::unique_lock<std::mutex> g(written_mu);
                        written_cv.wait(g, [&] { return grp.col_begin <= written_cols + AHEAD_COLS; });
                    }
                    const auto p0 = now();
                    my_wait_writer += secs(w0, p0);
                    MafFile &maf = *fctx[grp.file].maf;
                    const std::vector<MafFile::Chain> &chains = maf.chains();
                    const size_t c0 = grp.c0, c1 = grp.c1, chain0 = fctx[grp.file].chain0;
                    alns.resize(c1 - c0);
                    // The chains of the group side by side in one page-locked [nl][Ltot] matrix, parsed straight into it (the column
                    // count of a chain is known from the scan: its reference bases).  A chain whose text disagrees with its size
                    // fields falls back to the measuring parser, for the whole group.
                    int64_t Ltot = 0;
                    std::vector<int64_t> col0(c1 - c0);
                    for (size_t ci = c0; ci < c1; ++ci) { col0[ci - c0] = Ltot; Ltot += chains[ci].ref_id < 0 ? 0 : chains[ci].ref_cols; }
                    uint8_t *mat = my_slab;
                    bool direct = true;
                    for (size_t ci = c0; ci < c1 && direct; ++ci) {
                        const MafFile::Chain &c = chains[ci];
                        Alignment &aln = alns[ci - c0];
                        aln.start_pos = c.start_pos; aln.chrom_len = c.chrom_len; aln.strand = c.strand; aln.chrom = c.chrom;
                        aln.seqs.clear();
                        aln.L = maf.read_chain_into(c, mat + col0[ci - c0], Ltot, &seen[t]);
                        if (aln.L < 0) direct = false;
                    }
                    if (!direct) {
                        Ltot = 0;
                        for (size_t ci = c0; ci < c1; ++ci) {
                            maf.read_chain(chains[ci], alns[ci - c0], &seen[t]);
                            col0[ci - c0] = Ltot;
                            Ltot += alns[ci - c0].L;
                        }
                        if (Ltot > max_group_cols) {          // measured longer than announced: pageable staging for this one group
                            fallback_mat.resize((size_t)nl * Ltot);
                            mat = fallback_mat.data();
                        }
                        for (size_t k = 0; k < c1 - c0; ++k)
                            for (int s = 0; s < nl; ++s)
                                if (alns[k].L) memcpy(mat + (size_t)s * Ltot + col0[k], alns[k].seqs.data() + (size_t)s * alns[k].L, (size_t)alns[k].L);
                    }
                    if (Ltot > 0) {
                        src = mat;
                        if (Ltot > max_group_cols) {
                            fallback_out.resize((size_t)3 * Ltot);
                            plus = fallback_out.data(); minus = plus + Ltot; bls = minus + Ltot;
                        } else {
                            plus = reinterpret_cast<double *>(my_slab + mat_bytes);
                            minus = reinterpret_cast<double *>(my_slab + mat_bytes + vec_bytes);
                            bls = reinterpret_cast<double *>(my_slab + mat_bytes + 2 * vec_bytes);
                        }
                        const auto p1 = now();
                        my_parse += secs(p0, p1);
                        // piece by piece through a model's page-locked staging: windows [w0, w1) need columns [w0, w1 + 2); the last
                        // piece also takes the trailing columns (BLS is per column).  Every window is scored exactly once, so the result
                        // is that of one call over the whole group.
                        const int64_t Wtot = std::max<int64_t>(Ltot - 2, 0);
                        const uint32_t call_flags = PCSF_TRACKS_BLS | (raw ? PCSF_TRACKS_SCORES : 0) | pflag;
                        for (int64_t w0 = 0; w0 == 0 || w0 < Wtot; w0 += PIECE_COLS) {
                            const int64_t w1 = std::min(Wtot, w0 + PIECE_COLS);
                            const bool last_piece = w1 >= Wtot;
                            const int64_t cend = last_piece ? Ltot : w1 + 2, w = cend - w0;
                            if (!my_pin) {
                                my_pin = static_cast<uint8_t *>(pcsf_alloc_pinned(pin_bytes));
                                if (!my_pin) die("cannot allocate %zu bytes of page-locked memory: %s", pin_bytes, pcsf_last_error());
                            }
                            uint8_t *pin_in = my_pin;
                            double *pin_plus = reinterpret_cast<double *>(my_pin + pin_in_bytes), *pin_minus = reinterpret_cast<double *>(my_pin + pin_in_bytes + pin_vec_bytes),
                                   *pin_bls = reinterpret_cast<double *>(my_pin + pin_in_bytes + 2 * pin_vec_bytes);
                            for (int s2 = 0; s2 < nl; ++s2) memcpy(pin_in + (size_t)s2 * w, src + (size_t)s2 * Ltot + w0, (size_t)w);
                            const auto q0 = now();
                            const ModelPool::Entry me = pool.acquire();
                            const auto g0 = now();
                            my_wait_model += secs(q0, g0);
                            pcsf_tracks_stats cs{};
                            const pcsf_status st = pcsf_tracks(me.m, pin_in, w, w, call_flags, pin_plus, pin_minus, pin_bls, nullptr, &cs);
                            my_gpu += secs(g0, now());
                            pool.release(me);
                            if (st == PCSF_OK) {
                                if (raw && w1 > w0) {
                                    memcpy(plus + w0, pin_plus, (size_t)(w1 - w0) * 8);
                                    memcpy(minus + w0, pin_minus, (size_t)(w1 - w0) * 8);
                                }
                                memcpy(bls + w0, pin_bls, (size_t)(last_piece ? w : w1 - w0) * 8);
                            }
                            if (dev_timing) {
                                std::lock_guard<std::mutex> g(gpu_time_mu);
                                dev_ms[0] += cs.ms_pack; dev_ms[1] += cs.ms_hash; dev_ms[2] += cs.ms_dedup; dev_ms[3] += cs.ms_prune; dev_ms[4] += cs.ms_scatter;
                                dev_ms[5] += cs.ms_bls; dev_unique += cs.n_unique; dev_windows += cs.n_windows;
                            }
                            if (st == PCSF_ERR_BAD_CHAR) { fprintf(stderr, "%s\n", pcsf_last_error()); exit(37); }      // translation.hpp:46-51
                            if (st != PCSF_OK) die("pcsf_tracks: %s", pcsf_last_error());
                            gpu_cols[me.dev] += w1 > w0 ? w1 - w0 : w;
                        }
                        cols += Ltot;
                    }
                    const auto f0 = now();
                    for (size_t ci = c0; ci < c1; ++ci) {
                        const Alignment &aln = alns[ci - c0];
                        const int64_t L = aln.L;
                        std::vector<std::string> text(7);
                        if (L > 0) {
                            const double *pl = plus + col0[ci - c0], *mi = minus + col0[ci - c0], *bl = bls + col0[ci - c0];
                            char hdr[512];
                            // power track (build_tracks.hpp:139-158)
                            {
                                TextOut o(text[0]);
                                const int64_t skip = mod3(3 - aln.start_pos);
                                if (skip + 2 < L) {
                                    snprintf(hdr, sizeof hdr, "fixedStep chrom=%s start=%" PRId64 " step=3 span=3\n", aln.chrom.c_str(), aln.start_pos + skip);
                                    o.text(hdr);
                                }
                                o.room((size_t)(L / 3 + 1) * 8);
                                for (int64_t pos = skip; pos + 2 < L; pos += 3) o.value(4, (float)((bl[pos] + bl[pos + 1] + bl[pos + 2]) / 3.0));
                                o.finish();
                            }
                            // six raw tracks (build_tracks.hpp:160-216; frame arithmetic of update_seqs, parallel_file_reader.hpp:61-113)
                            if (raw) {
                                const float thr3 = threshold * 3;
                                for (int k = 0; k < 6; ++k) {
                                    const bool fwd = k < 3;
                                    const int64_t frame = k % 3 + 1;
                                    int64_t o0, K;
                                    if (fwd) {
                                        const int64_t skip = std::min<int64_t>(mod3(frame - aln.start_pos), L);
                                        o0 = skip; K = (L - skip) / 3;
                                    } else {
                                        const int64_t skip_r = std::min<int64_t>(mod3(frame - (aln.chrom_len - (aln.start_pos + L) + 2)), L);
                                        o0 = (L - skip_r) % 3; K = (L - skip_r) / 3;
                                    }
                                    const double *src_scores = fwd ? pl : mi;
                                    TextOut o(text[1 + k]);
                                    o.room((size_t)(K + 1) * 8);
                                    int64_t prev = -4;
                                    for (int64_t xx = 0; xx < K; ++xx) {
                                        const int64_t off = o0 + 3 * xx;
                                        const float bsum = (float)(bl[off] + bl[off + 1] + bl[off + 2]);
                                        if (bsum < thr3) continue;
                                        const int64_t np = aln.start_pos + off;
                                        if (prev + 3 != np) {
                                            snprintf(hdr, sizeof hdr, "fixedStep chrom=%s start=%" PRId64 " step=3 span=3\n", aln.chrom.c_str(), np);
                                            o.text(hdr);
                                        }
                                        prev = np;
                                        o.value(3, (float)src_scores[off]);
                                    }
                                    o.finish();
                                }
                            }
                        }
                        sink.put(chain0 + ci, std::move(text));
                    }
                    my_fmt += secs(f0, now());
                }
                std::lock_guard<std::mutex> g(gpu_time_mu);
                t_gpu += my_gpu; t_parse += my_parse; t_format += my_fmt; t_wait_model += my_wait_model; t_wait_writer += my_wait_writer;

        });
    for (size_t fi = 0; fi < fctx.size(); ++fi) {
        const std::string &out_dir = fctx[fi].out_dir;
        MafFile &maf = *fctx[fi].maf;
        const std::vector<MafFile::Chain> &chains = maf.chains();
        FILE *files[7];
        const char *mode = fi > 0 ? "a" : "w";          // build_tracks.hpp:245-259: later files append
        files[0] = fopen((out_dir + "/PhyloCSFpower.wig").c_str(), mode);
        for (int k = 0; k < 6; ++k) files[1 + k] = raw ? fopen((out_dir + "/PhyloCSFRaw" + kFrames[k] + ".wig").c_str(), mode) : nullptr;
        if (!files[0] || (raw && !files[1])) die("Error creating output files in '%s'!", out_dir.c_str());
        size_t bytes_done = 0;
        for (size_t ci = 0; ci < chains.size(); ++ci) {
            std::vector<std::string> text = sink.take(fctx[fi].chain0 + ci);
            for (int k = 0; k < 7; ++k) if (files[k] && !text[k].empty()) fwrite(text[k].data(), 1, text[k].size(), files[k]);
            bytes_done += maf.chain_bytes(chains[ci]);
            { std::lock_guard<std::mutex> g(written_mu); written_cols += chains[ci].ref_cols + 2; }
            written_cv.notify_all();
            if ((ci & 15) == 0 || ci + 1 == chains.size()) {
                printf("\33[2K\r");
                if (fctx.size() > 1) printf("File %zu of %zu: ", fi + 1, fctx.size());
                printf("%.2f / %.2f MB (%3.2f %%)\r", bytes_done / 1048576.0, maf.file_size() / 1048576.0, 100.0 * bytes_done / std::max<size_t>(1, maf.file_size()));
                fflush(stdout);
            }
        }
        for (FILE *f : files) if (f) fclose(f);
        // PhyloCSF-HMM over the text of the six raw tracks (build_tracks.hpp:262-348), one thread per track
        if (smooth || regions) {
            printf("\33[2K\rSmoothing scores and/or computing coding-regions ...\r");
            fflush(stdout);
            std::vector<std::thread> sm;
            for (int k = 0; k < 6; ++k)
                sm.emplace_back([&, k] {
                    const std::string rawp = out_dir + "/PhyloCSFRaw" + kFrames[k] + ".wig";
                    FILE *fw = smooth ? fopen((out_dir + "/PhyloCSF" + kFrames[k] + ".wig").c_str(), "w") : nullptr;
                    FILE *fb = regions ? fopen((out_dir + "/PhyloCSF" + kFrames[k] + "Regions.bed").c_str(), "w") : nullptr;
                    if ((smooth && !fw) || (regions && !fb)) die("Error creating output files in '%s'!", out_dir.c_str());
                    hmm_smooth_file(hmm_model, rawp, kFrames[k][0], fw, fb);
                    if (fw) fclose(fw);
                    if (fb) fclose(fb);
                    if (!keep_raw) unlink(rawp.c_str());
                });
            for (auto &t : sm) t.join();
        }
    }
    for (auto &w : workers) w.join();
    stop_models = true;
    pool_waiter.join();
    total_cols += cols;
    if (to_bigwig) {
        std::map<std::string, std::map<std::string, uint32_t>> sizes;          // output directory -> chromosome -> length
        for (const FileCtx &fc : fctx)
            for (const MafFile::Chain &c : fc.maf->chains())
                if (c.ref_id >= 0) { uint32_t &l = sizes[fc.out_dir][c.chrom]; l = std::max<uint32_t>(l, (uint32_t)c.chrom_len); }
        std::vector<std::thread> conv;
        for (const auto &dir : sizes) {
            const std::vector<std::pair<std::string, uint32_t>> chroms(dir.second.begin(), dir.second.end());
            std::vector<std::string> names = {"PhyloCSFpower"};
            for (int k = 0; k < 6; ++k) {
                if (keep_raw) names.push_back(std::string("PhyloCSFRaw") + kFrames[k]);
                if (smooth) names.push_back(std::string("PhyloCSF") + kFrames[k]);
            }
            for (const std::string &n : names)
                conv.emplace_back([=] { wig_to_bigwig(dir.first + "/" + n + ".wig", chroms, dir.first + "/" + n + ".bw"); });
        }
        for (auto &t : conv) t.join();
    }
    const double wall = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
    printf("\nDone!\n");
    if (getenv("PCSF_HOST_STATS")) {
        std::string per_gpu;
        for (int g = 0; g < gpus; ++g) per_gpu += (g ? ", " : "") + std::to_string((long long)gpu_cols[g]);
        printf("{\"columns\": %" PRId64 ", \"seconds\": %.3f, \"columns_per_s\": %.1f, \"threads\": %d, \"gpus\": %d, \"gpus_worth\": %d, \"scan_seconds\": %.3f, "
               "\"first_model_seconds\": %.3f, \"startup_seconds\": %.3f, \"parse_seconds_sum\": %.3f, \"pinned_alloc_seconds\": %.3f, \"wait_model_seconds_sum\": %.3f, \"wait_writer_seconds_sum\": %.3f, "
               "\"gpu_call_seconds_sum\": %.3f, \"format_seconds_sum\": %.3f, \"columns_per_gpu\": [%s]}\n",
               total_cols, wall, total_cols / wall, threads, gpus, gpus_worth, t_scan, t_first_model.load(), t_startup, t_parse, t_slab, t_wait_model, t_wait_writer, t_gpu, t_format, per_gpu.c_str());
    }
    if (dev_timing)
        printf("{\"ms_pack\": %.2f, \"ms_hash\": %.2f, \"ms_dedup\": %.2f, \"ms_prune\": %.2f, \"ms_scatter\": %.2f, \"ms_bls\": %.2f, \"windows\": %" PRId64
               ", \"unique\": %" PRId64 "}\n", dev_ms[0], dev_ms[1], dev_ms[2], dev_ms[3], dev_ms[4], dev_ms[5], dev_windows, dev_unique);
    // species of the model never seen in any alignment (build_tracks.hpp:487-504)
    for (int s = 0; s < nl; ++s) {
        bool any = false;
        for (int t = 0; t < threads; ++t) any |= seen[t][s] != 0;
        if (!any) printf("\033[33mWARNING: species %s from the model was never seen in any alignment.\033[0m\n", model.tree.labels[s].c_str());
    }
    // Everything is on disk.  Tearing down the device models, the staging memory and up to eight CUDA contexts in an orderly fashion
    // costs 0.3-2 s that nobody waits for; the operating system reclaims all of it (PCSF_HOST_ORDERLY_EXIT=1 keeps the teardown, e.g.
    // under compute-sanitizer).
    if (!getenv("PCSF_HOST_ORDERLY_EXIT")) {
        fflush(stdout);
        fflush(stderr);
        _exit(0);
    }
    const auto x0 = std::chrono::steady_clock::now();
    for (int t = 0; t < slab_threads; ++t) free(slabs[t]);
    const auto x1 = std::chrono::steady_clock::now();
    pool.destroy();
    const auto x2 = std::chrono::steady_clock::now();
    fctx.clear();
    const auto x3 = std::chrono::steady_clock::now();
    if (getenv("PCSF_HOST_STATS"))
        printf("{\"teardown_buffers_seconds\": %.3f, \"teardown_models_seconds\": %.3f, \"teardown_files_seconds\": %.3f, \"before_start_seconds\": %.3f}\n",
               std::chrono::duration<double>(x1 - x0).count(), std::chrono::duration<double>(x2 - x1).count(), std::chrono::duration<double>(x3 - x2).count(),
               std::chrono::duration<double>(t_start - t_entry).count());
    return 0;
}

// ---------------------------------------------------------------------------------------------- score-msa
int main_score_msa(int argc, char **argv) {
    const Args a = parse_args(argc, argv, {"strategy", "comp-phylo", "comp-anc", "comp-bls", "threads", "output", "mapping", "species", "gpus",
                                           "genome-length", "coding-exons", "model-info", "frames", "orf", "min-codons", "all-scores"});
    if (a.has("model-info")) return print_model_info(a.str("model-info"));          // score_msa.hpp:291-295
    if (a.pos.size() < 2) die("usage: phylocsf_b200 score-msa [OPTIONS] <model> <alignments>...");
    const std::string strat = lower(a.str("strategy", "mle"));
    pcsf_strategy strategy;
    bool fixed_mean = false;
    if (strat == "mle") strategy = PCSF_STRATEGY_MLE;
    else if (strat == "fixed") strategy = PCSF_STRATEGY_FIXED;
    else if (strat == "omega") strategy = PCSF_STRATEGY_OMEGA;
    else if (strat == "fixed_mean") { strategy = PCSF_STRATEGY_FIXED; fixed_mean = true; }          // score_msa.hpp:314-325
    else { printf("\033[31mPlease choose a valid strategy (MLE, FIXED or OMEGA)!\n\033[0m"); return -1; }
    if (fixed_mean && (!a.has("genome-length") || !a.has("coding-exons"))) {
        printf("\033[31mFor FIXED_MEAN you need to provide --genome-length and --coding-exons.\n\033[0m");
        return -1;
    }
    const bool comp_phylo = a.boolean("comp-phylo", true), comp_anc = a.boolean("comp-anc", false), comp_bls = true;   // no --comp-bls in the reference
    if (strategy == PCSF_STRATEGY_OMEGA && comp_anc) {          // score_msa.hpp:338-342
        printf("\033[31mThe ancestral sequence composition cannot be computed in the Omega mode!\n\033[0m");
        return -1;
    }
    // reading frames / ORFs (pcsf_score_regions): with --frames 1 --orf asis and without --all-scores the command is the plain
    // frame +1 score-msa and takes its path unchanged
    auto strict_int = [&](const char *k, int dflt, int *v) {
        if (!a.has(k)) { *v = dflt; return true; }
        const std::string t = a.str(k);
        char *e = nullptr;
        const long x = strtol(t.c_str(), &e, 10);
        if (t.empty() || *e || x < INT32_MIN || x > INT32_MAX) return false;
        *v = (int)x;
        return true;
    };
    int frames = 1, min_codons = 25;
    if (!strict_int("frames", 1, &frames) || (frames != 1 && frames != 3 && frames != 6)) {
        printf("\033[31m--frames must be 1, 3 or 6!\n\033[0m");
        return -1;
    }
    const std::string orf_s = lower(a.str("orf", "asis"));
    pcsf_orf_mode orf;
    if (orf_s == "asis") orf = PCSF_ORF_ASIS;
    else if (orf_s == "stopstop") orf = PCSF_ORF_STOPSTOP;
    else if (orf_s == "atgstop") orf = PCSF_ORF_ATGSTOP;
    else { printf("\033[31m--orf must be AsIs, StopStop or ATGStop!\n\033[0m"); return -1; }
    if (!strict_int("min-codons", 25, &min_codons) || min_codons < 1) {
        printf("\033[31m--min-codons must be an integer >= 1!\n\033[0m");
        return -1;
    }
    const bool all_scores = a.boolean("all-scores", false);
    const bool regions = frames != 1 || orf != PCSF_ORF_ASIS || all_scores;
    if (regions && fixed_mean) {
        printf("\033[31mFIXED_MEAN cannot be combined with --frames, --orf or --all-scores!\n\033[0m");
        return -1;
    }
    if (regions && !all_scores && !comp_phylo) {
        printf("\033[31mThe best frame or ORF is chosen by its PhyloCSF score: --comp-phylo 0 needs --all-scores 1!\n\033[0m");
        return -1;
    }
    const int threads = std::max(1, a.integer("threads", (int)std::thread::hardware_concurrency()));
    const int gpus = std::max(1, a.integer("gpus", default_gpus()));
    const int workers_n = std::min(threads, 2 * gpus);      // the per-call batch is the unit of GPU work; parsing runs inside the workers

    Model model;
    load_model(model, a.pos[0], a.str("species"), a.str("mapping"));
    const int nl = model.nl();
    Hmm hmm_model{};
    if (fixed_mean) hmm_model = coding_hmm(estimate_hmm_params(a.str("coding-exons"), (uint32_t)strtoull(a.str("genome-length").c_str(), nullptr, 10)));
    const auto t_start = std::chrono::steady_clock::now();
    auto since = [&](std::chrono::steady_clock::time_point a) { return std::chrono::duration<double>(std::chrono::steady_clock::now() - a).count(); };
    std::vector<pcsf_model *> dev(workers_n);
    {
        std::vector<std::thread> th;          // model preparation is host work (eigensystem, all P(t), uploads): one thread per handle
        for (int t = 0; t < workers_n; ++t) th.emplace_back([&, t] { dev[t] = create_device_model(model, t % gpus); });
        for (auto &x : th) x.join();
    }
    const double t_models = since(t_start);
    double t_scan = 0.0, t_parse = 0.0, t_gpu = 0.0, t_format = 0.0;
    std::mutex stat_mu;
    int64_t total_aln = 0;

    for (size_t fi = 1; fi < a.pos.size(); ++fi) {
        const std::string &path = a.pos[fi];
        std::string out_path = a.str("output");
        if (out_path.empty()) out_path = path + ".scores";
        else { create_directory(out_path); const size_t p = path.find_last_of('/'); out_path += "/" + (p == std::string::npos ? path : path.substr(p + 1)) + ".scores"; }
        FILE *out = fopen(out_path.c_str(), "w");
        if (!out) die("Error creating file '%s'!", out_path.c_str());
        fprintf(out, "# PhyloCSF scores computed with PhyloCSF++ v1.2.0 (phylocsf_b200, B200-native likelihood core)\n");
        fprintf(out, "seq\tstart\tend\tstrand");
        if (regions) fprintf(out, "\tframe\torf-start\torf-end");
        if (comp_phylo) fprintf(out, "\tphylocsf-score");
        if (comp_anc) fprintf(out, "\tanc-score");
        if (comp_bls) fprintf(out, "\tbls-score");
        fprintf(out, "\n");

        const auto s0 = std::chrono::steady_clock::now();
        MafFile maf(path, model, false, threads);
        t_scan += since(s0);
        warn_unresolved(maf);
        const std::vector<MafFile::Chain> &chains = maf.chains();
        // alignments per library call (measured on 100 k config-5 alignments, MLE: 4096 ... 131072 per call all take 5.3-5.7 s — the GPU
        // is bound by the evaluations themselves, not by the tail of a call)
        const size_t BATCH = getenv("PCSF_HOST_MSA_BATCH") ? (size_t)atoll(getenv("PCSF_HOST_MSA_BATCH")) : 4096;
        const size_t nbatch = (chains.size() + BATCH - 1) / BATCH;
        OrderedSink sink;
        sink.resize(nbatch);
        std::atomic<size_t> next{0};
        std::vector<std::thread> workers;
        for (int t = 0; t < workers_n; ++t)
            workers.emplace_back([&, t] {
                Alignment aln;
                for (size_t bi = next++; bi < nbatch; bi = next++) {
                    const size_t c0 = bi * BATCH, c1 = std::min(chains.size(), c0 + BATCH);
                    std::vector<uint8_t> blob;
                    std::vector<int64_t> off, len;
                    std::vector<std::string> head;
                    std::vector<int32_t> ref_row;
                    std::vector<int64_t> start_pos;
                    const auto p0 = std::chrono::steady_clock::now();
                    for (size_t ci = c0; ci < c1; ++ci) {
                        if (chains[ci].ref_id < 0) continue;
                        maf.read_chain(chains[ci], aln, nullptr);
                        off.push_back((int64_t)blob.size()); len.push_back(aln.L);
                        ref_row.push_back(chains[ci].ref_id); start_pos.push_back(aln.start_pos);
                        blob.insert(blob.end(), aln.seqs.begin(), aln.seqs.end());
                        char h[600];
                        snprintf(h, sizeof h, "%s\t%" PRId64 "\t%" PRId64 "\t%c", aln.chrom.c_str(), aln.start_pos, aln.start_pos + aln.L - 1, aln.strand);
                        head.push_back(h);
                    }
                    const int n = (int)off.size();
                    std::vector<float> phylo(n, NAN), anc(n, NAN), bls(n, NAN);
                    if (blob.empty()) blob.push_back('N');
                    const double my_parse = since(p0);
                    const auto g0 = std::chrono::steady_clock::now();
                    if (regions) {
                        // one row per region (--all-scores 1) or per alignment (its best region); frame +1..-3 or "." for none,
                        // ORF columns in the coordinates of start / end
                        std::vector<pcsf_region> rg;
                        if (n > 0) {
                            int64_t nr = 0;
                            pcsf_status st = pcsf_score_regions(dev[t], strategy, n, blob.data(), off.data(), len.data(), ref_row.data(), frames, orf,
                                                                min_codons, all_scores ? 0 : 1, comp_anc ? 1 : 0, comp_bls ? 1 : 0, &nr);
                            if (st == PCSF_ERR_BAD_CHAR) { fprintf(stderr, "%s\n", pcsf_last_error()); exit(37); }
                            if (st != PCSF_OK) die("pcsf_score_regions: %s", pcsf_last_error());
                            rg.resize((size_t)nr);
                            if ((st = pcsf_score_regions_get(dev[t], rg.data(), nr)) != PCSF_OK) die("pcsf_score_regions_get: %s", pcsf_last_error());
                        }
                        const double my_gpu = since(g0);
                        const auto f0 = std::chrono::steady_clock::now();
                        std::string text;
                        char v[128];
                        for (const pcsf_region &r : rg) {
                            text += head[r.aln];
                            if (r.frame == 0) text += "\t.\t.\t.";
                            else {
                                snprintf(v, sizeof v, "\t%c%d\t%" PRId64 "\t%" PRId64, r.strand > 0 ? '+' : '-', (int)r.frame,
                                         start_pos[r.aln] + r.col_begin, start_pos[r.aln] + r.col_end - 1);
                                text += v;
                            }
                            if (comp_phylo) { snprintf(v, sizeof v, "\t%.6f", r.phylo); text += v; }
                            if (comp_anc) { snprintf(v, sizeof v, "\t%.6f", r.anc); text += v; }
                            if (comp_bls) { snprintf(v, sizeof v, "\t%.6f", r.bls); text += v; }
                            text += "\n";
                        }
                        std::vector<std::string> one(1);
                        one[0] = std::move(text);
                        sink.put(bi, std::move(one));
                        std::lock_guard<std::mutex> g(stat_mu);
                        t_parse += my_parse; t_gpu += my_gpu; t_format += since(f0); total_aln += n;
                        continue;
                    }
                    if (n > 0) {
                        const pcsf_status st = pcsf_score_msa(dev[t], strategy, n, blob.data(), off.data(), len.data(), (comp_phylo || comp_anc) ? phylo.data() : nullptr,
                                                              comp_anc ? anc.data() : nullptr, comp_bls ? bls.data() : nullptr);
                        if (st == PCSF_ERR_BAD_CHAR) { fprintf(stderr, "%s\n", pcsf_last_error()); exit(37); }
                        if (st != PCSF_OK) die("pcsf_score_msa: %s", pcsf_last_error());
                    }
                    if (fixed_mean && n > 0 && comp_phylo) {
                        // FIXED_MEAN (score_msa.hpp:136-213): the per-codon decibans of frame +1 (run_tracks) go through the
                        // PhyloCSF-HMM as one contiguous run; the score is the mean posterior log-odds, summed in a float.
                        // Per-codon scores come from the tracks entry point on the alignments laid side by side.
                        int64_t Ltot = 0;
                        std::vector<int64_t> col0(n);
                        for (int i = 0; i < n; ++i) { col0[i] = Ltot; Ltot += len[i]; }
                        std::vector<double> plus((size_t)std::max<int64_t>(Ltot - 2, 0)), minus(plus.size());
                        if (Ltot > 2) {
                            std::vector<uint8_t> mat((size_t)nl * Ltot);
                            for (int i = 0; i < n; ++i)
                                for (int sp = 0; sp < nl; ++sp)
                                    if (len[i]) memcpy(mat.data() + (size_t)sp * Ltot + col0[i], blob.data() + off[i] + (size_t)sp * len[i], (size_t)len[i]);
                            const pcsf_status st = pcsf_tracks(dev[t], mat.data(), Ltot, Ltot, PCSF_TRACKS_SCORES, plus.data(), minus.data(), nullptr, nullptr, nullptr);
                            if (st != PCSF_OK) die("pcsf_tracks: %s", pcsf_last_error());
                        }
                        std::vector<double> scores, post;
                        for (int i = 0; i < n; ++i) {
                            scores.clear();
                            for (int64_t k = 0; k < len[i] / 3; ++k) scores.push_back(plus[(size_t)(col0[i] + 3 * k)]);
                            hmm_posterior_coding(hmm_model, scores, post);
                            float sum = 0.0;
                            uint64_t cnt = 0;
                            for (double pc : post) sum += hmm_log_odds(pc);
                            cnt += post.size();
                            phylo[i] = sum / cnt;
                        }
                    }
                    const double my_gpu = since(g0);
                    const auto f0 = std::chrono::steady_clock::now();
                    std::string text;
                    char v[64];
                    for (int i = 0; i < n; ++i) {
                        text += head[i];
                        if (comp_phylo) { snprintf(v, sizeof v, "\t%.6f", phylo[i]); text += v; }
                        if (comp_anc) { snprintf(v, sizeof v, "\t%.6f", anc[i]); text += v; }
                        if (comp_bls) { snprintf(v, sizeof v, "\t%.6f", bls[i]); text += v; }
                        text += "\n";
                    }
                    std::vector<std::string> one(1);
                    one[0] = std::move(text);
                    sink.put(bi, std::move(one));
                    std::lock_guard<std::mutex> g(stat_mu);
                    t_parse += my_parse; t_gpu += my_gpu; t_format += since(f0); total_aln += n;
                }
            });
        for (size_t bi = 0; bi < nbatch; ++bi) {
            std::vector<std::string> text = sink.take(bi);
            fwrite(text[0].data(), 1, text[0].size(), out);
        }
        for (auto &w : workers) w.join();
        fclose(out);
    }
    printf("Done!\n");
    if (getenv("PCSF_HOST_STATS"))
        printf("{\"alignments\": %" PRId64 ", \"seconds\": %.3f, \"model_seconds\": %.3f, \"scan_seconds\": %.3f, \"parse_seconds_sum\": %.3f, "
               "\"gpu_call_seconds_sum\": %.3f, \"format_seconds_sum\": %.3f, \"workers\": %d}\n",
               total_aln, since(t_start), t_models, t_scan, t_parse, t_gpu, t_format, workers_n);
    for (pcsf_model *m : dev) pcsf_model_destroy(m);
    (void)nl;
    return 0;
}

// ------------------------------------------------------------------------------------- dump-alignments
// Test hook (no GPU needed): what the reader hands to the likelihood core, one line per alignment.
int main_dump_alignments(int argc, char **argv) {
    const Args a = parse_args(argc, argv, {"concatenate", "threads", "mapping", "species", "hash"});
    const bool do_hash = a.boolean("hash", true);          // --hash 0: time the reader alone
    if (a.pos.size() < 2) die("usage: phylocsf_b200 dump-alignments [--concatenate BOOL] [--threads INT] <model> <alignments>...");
    Model model;
    load_model(model, a.pos[0], a.str("species"), a.str("mapping"));
    for (size_t fi = 1; fi < a.pos.size(); ++fi) {
        MafFile maf(a.pos[fi], model, a.boolean("concatenate", true), std::max(1, a.integer("threads", 4)));
        Alignment aln;
        for (const MafFile::Chain &c : maf.chains()) {
            maf.read_chain(c, aln, nullptr);
            // the build-tracks workers parse with read_chain_into (straight into their page-locked matrix, row stride != L): it has to
            // give the same bytes whenever it accepts the chain
            if (c.ref_id >= 0) {
                const int64_t stride = c.ref_cols + 5;
                std::vector<uint8_t> direct((size_t)model.nl() * stride, 0);
                const int64_t L2 = maf.read_chain_into(c, direct.data(), stride, nullptr);
                if (L2 >= 0) {
                    if (L2 != aln.L) die("read_chain_into: %" PRId64 " columns, read_chain %" PRId64, L2, aln.L);
                    for (int sidx = 0; sidx < model.nl(); ++sidx)
                        if (aln.L && memcmp(direct.data() + (size_t)sidx * stride, aln.seqs.data() + (size_t)sidx * aln.L, (size_t)aln.L) != 0)
                            die("read_chain_into differs from read_chain in row %d of the chain at %s:%" PRId64, sidx, aln.chrom.c_str(), aln.start_pos);
                } else if (getenv("PCSF_REQUIRE_DIRECT")) {
                    die("read_chain_into refused the chain at %s:%" PRId64, aln.chrom.c_str(), aln.start_pos);
                }
            }
            uint64_t h = 1469598103934665603ull;
            if (do_hash) for (uint8_t b : aln.seqs) { h ^= b; h *= 1099511628211ull; }
            printf("%s\t%" PRId64 "\t%" PRId64 "\t%c\t%" PRId64 "\t%016" PRIx64 "\n", aln.chrom.c_str(), aln.start_pos, aln.chrom_len, aln.strand, aln.L, h);
        }
    }
    return 0;
}

// Test / bench tooling (no GPU needed): a raw [nl][ncols] ASCII matrix (the synthetic workload, phylocsfpp_b200/synth.py) as a MAF file
// with the shape tools/make_synth_maf.py writes for its plain case — blocks of --block columns, a hole of 1..300 bases after every
// --chain columns, species whose cells are all N in a block left out — fast enough for files of 10^8 columns.
int main_matrix_to_maf(int argc, char **argv) {
    const Args a = parse_args(argc, argv, {"block", "chain", "start", "chrom", "skip-bytes"});
    if (a.pos.size() != 4) die("usage: phylocsf_b200 matrix-to-maf [--block INT] [--chain INT] [--start INT] [--chrom NAME] [--skip-bytes INT] <model> <matrix.bin> <ncols> <out.maf>");
    Model model;
    load_model(model, a.pos[0], "", "");
    const int nl = model.nl();
    const int64_t ncols = atoll(a.pos[2].c_str()), block = std::max(1, a.integer("block", 120));
    const int64_t chain = a.has("chain") ? atoll(a.str("chain").c_str()) : 0, start0 = a.has("start") ? atoll(a.str("start").c_str()) : 10000;
    FILE *fi = fopen(a.pos[1].c_str(), "rb");
    if (!fi) die("cannot open %s", a.pos[1].c_str());
    const std::string chrom = a.str("chrom", "chr1");
    if (a.has("skip-bytes")) fseeko(fi, (off_t)atoll(a.str("skip-bytes").c_str()), SEEK_SET);          // e.g. the header of a .npy file
    std::vector<uint8_t> mat((size_t)nl * ncols);
    if (fread(mat.data(), 1, mat.size(), fi) != mat.size()) die("%s is shorter than %d x %" PRId64 " bytes", a.pos[1].c_str(), nl, ncols);
    fclose(fi);
    std::vector<std::string> names(nl);
    for (int s = 0; s < nl; ++s) {
        const std::string &label = model.tree.labels[s];
        auto it = model.aliases.find(label);
        names[s] = (it != model.aliases.end() && !it->second.empty()) ? it->second[0] : label;
    }
    FILE *fo = fopen(a.pos[3].c_str(), "wb");
    if (!fo) die("cannot create %s", a.pos[3].c_str());
    std::vector<char> buf((size_t)16 << 20);
    setvbuf(fo, buf.data(), _IOFBF, buf.size());
    fputs("##maf version=1 scoring=synthetic\n", fo);
    const int64_t src_size = start0 + ncols + ncols / 100 + 400000 + (chain ? (ncols / chain + 1) * 301 : 0);
    int64_t pos = start0, blocks = 0;
    uint64_t lcg = 0x9E3779B97F4A7C15ull;
    for (int64_t c0 = 0; c0 < ncols;) {
        int64_t c1 = std::min(ncols, c0 + block);
        if (chain && c0 / chain != (c1 - 1) / chain) c1 = (c0 / chain + 1) * chain;          // blocks do not straddle a chain boundary
        const int64_t size = c1 - c0;
        fputs("a score=0.0\n", fo);
        for (int s = 0; s < nl; ++s) {
            const uint8_t *row = mat.data() + (size_t)s * ncols + c0;
            if (s == 0) {
                fprintf(fo, "s %s.%s %" PRId64 " %" PRId64 " + %" PRId64 " ", names[0].c_str(), chrom.c_str(), pos, size, src_size);
            } else {
                int64_t nb = 0, nn = 0;
                for (int64_t i = 0; i < size; ++i) { nb += row[i] != '-'; nn += row[i] == 'N'; }
                if (nn == size) continue;
                fprintf(fo, "s %s.scaffold_%d %" PRId64 " %" PRId64 " %c 50000000 ", names[s].c_str(), s, 1000 + c0, nb, "+-"[s % 2]);
            }
            fwrite(row, 1, (size_t)size, fo);
            fputc('\n', fo);
        }
        fputc('\n', fo);
        pos += size;
        ++blocks;
        if (chain && c1 % chain == 0 && c1 < ncols) { lcg = lcg * 6364136223846793005ull + 1442695040888963407ull; pos += 1 + (int64_t)((lcg >> 33) % 300); }
        c0 = c1;
    }
    fclose(fo);
    printf("{\"columns\": %" PRId64 ", \"blocks\": %" PRId64 "}\n", ncols, blocks);
    return 0;
}


// ---------------------------------------------------------------------------------------------- track consumers (SURVEY §8 f-4)
// annotate-with-tracks (reference src/phylocsf++annotate_with_tracks.hpp:220-305): same positionals and --output.
int main_annotate_with_tracks(int argc, char **argv) {
    const Args a = parse_args(argc, argv, {"output"});
    if (a.pos.size() < 2) die("usage: phylocsf_b200 annotate-with-tracks [--output DIR] <PhyloCSF+1.bw> <gff/gtf files>...");
    const std::string out_dir = a.str("output");
    if (!out_dir.empty() && create_directory(out_dir)) printf("Created the output directory.\n");
    TrackSet tracks;
    if (!open_tracks(a.pos[0], tracks)) return -1;
    std::set<std::string> missing;
    const std::string header = "# PhyloCSF scores computed with phylocsf_b200 (PhyloCSF++ compatible) and precomputed tracks " + a.pos[0] + "\n";
    for (size_t i = 1; i < a.pos.size(); ++i) annotate_file(a.pos[i], out_dir, tracks, missing, header);
    printf("\33[2K\rDone!\n");
    return 0;
}

// annotate-with-maf: PhyloCSF scores of the CDS (and of the coding transcripts as a whole) of GFF/GTF files, from spliced alignments
// cut out of whole-genome MAF files (transcripts.hpp); with --find-orf 1, the best ATG-to-stop ORF of every transcript without CDS.
// Every input line is copied; transcript and CDS lines get attributes in the file's syntax.  Batches of transcripts are scored by
// score-msa's worker pattern (one device model per worker, thread t on GPU t mod --gpus) and written in file order.
int main_annotate_with_maf(int argc, char **argv) {
    const Args a = parse_args(argc, argv, {"output", "strategy", "comp-anc", "find-orf", "min-codons", "species", "mapping", "threads", "gpus"});
    if (a.pos.size() < 3)
        die("usage: phylocsf_b200 annotate-with-maf [OPTIONS] <model> <alignments.maf[,more.maf...]> <gff/gtf files>...");
    const std::string strat = lower(a.str("strategy", "mle"));
    pcsf_strategy strategy;
    if (strat == "mle") strategy = PCSF_STRATEGY_MLE;
    else if (strat == "fixed") strategy = PCSF_STRATEGY_FIXED;
    else if (strat == "omega") strategy = PCSF_STRATEGY_OMEGA;
    else { printf("\033[31mPlease choose a valid strategy (MLE, FIXED or OMEGA)!\n\033[0m"); return -1; }
    const bool comp_anc = a.boolean("comp-anc", false), find_orf = a.boolean("find-orf", false);
    if (strategy == PCSF_STRATEGY_OMEGA && comp_anc) {
        printf("\033[31mThe ancestral sequence composition cannot be computed in the Omega mode!\n\033[0m");
        return -1;
    }
    const std::string mc = a.str("min-codons", "25");
    char *mc_end = nullptr;
    const long min_codons = strtol(mc.c_str(), &mc_end, 10);
    if (mc.empty() || *mc_end || min_codons < 1 || min_codons > INT32_MAX) {
        printf("\033[31m--min-codons must be an integer >= 1!\n\033[0m");
        return -1;
    }
    const int threads = std::max(1, a.integer("threads", (int)std::thread::hardware_concurrency()));
    const int gpus = std::max(1, a.integer("gpus", default_gpus()));
    const int workers_n = std::min(threads, 2 * gpus);
    Model model;
    load_model(model, a.pos[0], a.str("species"), a.str("mapping"));
    const auto t_start = std::chrono::steady_clock::now();
    auto since = [](std::chrono::steady_clock::time_point t) { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t).count(); };
    std::vector<pcsf_model *> dev(workers_n);
    std::thread model_maker([&] {
        std::vector<std::thread> th;
        for (int t = 0; t < workers_n; ++t) th.emplace_back([&, t] { dev[t] = create_device_model(model, t % gpus); });
        for (auto &x : th) x.join();
    });
    const ChainIndex idx(split(a.pos[1], ','), model, threads);
    for (const auto &maf : idx.mafs()) warn_unresolved(*maf);
    if (idx.minus_chains())
        printf("\033[33mWARNING: %" PRId64 " alignment chains with the reference on the '-' strand are not used.\033[0m\n", idx.minus_chains());
    const double t_scan = since(t_start);

    struct GffFile { std::string out_path; bool newline_at_end; std::vector<GffTranscript> recs; };
    std::vector<GffFile> files;
    const std::string out_dir = a.str("output");
    if (!out_dir.empty()) create_directory(out_dir);
    for (size_t i = 2; i < a.pos.size(); ++i) {
        const std::string &path = a.pos[i];
        const size_t slash = path.find_last_of('/');
        std::string out = out_dir.empty() ? path : out_dir + "/" + (slash == std::string::npos ? path : path.substr(slash + 1));
        const size_t dot = out.find_last_of('.');
        if (dot == std::string::npos || (out.find_last_of('/') != std::string::npos && dot < out.find_last_of('/'))) out += ".PhyloCSF++maf";
        else out.insert(dot, ".PhyloCSF++maf");
        GffReader reader(path);
        GffFile f{out, reader.ends_with_newline(), {}};
        GffTranscript t;
        while (reader.next(t)) f.recs.push_back(t);
        files.push_back(std::move(f));
    }
    struct Batch { size_t file, r0, r1; };
    const size_t BATCH = getenv("PCSF_HOST_MAF_BATCH") ? std::max<size_t>(1, (size_t)atoll(getenv("PCSF_HOST_MAF_BATCH"))) : 4096;
    std::vector<Batch> batches;
    for (size_t fi = 0; fi < files.size(); ++fi)
        for (size_t r0 = 0; r0 < files[fi].recs.size(); r0 += BATCH) batches.push_back(Batch{fi, r0, std::min(files[fi].recs.size(), r0 + BATCH)});
    const double t_read = since(t_start) - t_scan;
    model_maker.join();

    OrderedSink sink;
    sink.resize(batches.size());
    std::atomic<size_t> next{0};
    std::mutex stat_mu;
    double t_extract = 0.0, t_gpu = 0.0, t_format = 0.0;
    int64_t n_coding = 0, n_orf = 0;
    std::vector<std::thread> workers;
    for (int w = 0; w < workers_n; ++w)
        workers.emplace_back([&, w] {
            ChainCache cache(idx);
            for (size_t bi = next++; bi < batches.size(); bi = next++) {
                const Batch &bt = batches[bi];
                const std::vector<GffTranscript> &recs = files[bt.file].recs;
                const auto p0 = std::chrono::steady_clock::now();
                // coding transcripts: one alignment each, its regions through pcsf_score_given_regions; the others (--find-orf 1): one
                // alignment each through pcsf_score_regions, best ATG-to-stop ORF of frames +1..+3
                std::vector<TxAlignment> tx(bt.r1 - bt.r0);
                std::vector<char> scored(tx.size(), 0);
                std::vector<uint8_t> cblob, oblob;
                std::vector<int64_t> coff, clen, ooff, olen, rbeg, rend;
                std::vector<int32_t> raln, oref;
                std::vector<int64_t> first_region(tx.size(), -1), orf_index(tx.size(), -1);
                // extracted in genomic order: the transcripts of a batch then share the chains the cache holds, however the file is sorted
                std::vector<size_t> by_pos(tx.size());
                for (size_t k = 0; k < tx.size(); ++k) by_pos[k] = k;
                std::stable_sort(by_pos.begin(), by_pos.end(), [&](size_t i, size_t j) {
                    const GffTranscript &a = recs[bt.r0 + i], &b = recs[bt.r0 + j];
                    return a.chr != b.chr ? a.chr < b.chr : a.begin < b.begin;
                });
                for (size_t k : by_pos) {
                    TxAlignment &x = tx[k];
                    if (!extract_transcript(idx, cache, recs[bt.r0 + k], find_orf, x)) continue;
                    scored[k] = 1;
                    if (x.coding) {
                        first_region[k] = (int64_t)rbeg.size();
                        for (size_t r = 0; r < x.reg_begin.size(); ++r) {
                            raln.push_back((int32_t)coff.size()); rbeg.push_back(x.reg_begin[r]); rend.push_back(x.reg_end[r]);
                        }
                        coff.push_back((int64_t)cblob.size()); clen.push_back(x.L);
                        cblob.insert(cblob.end(), x.seqs.begin(), x.seqs.end());
                    } else if (x.ref_row >= 0) {
                        orf_index[k] = (int64_t)ooff.size();
                        ooff.push_back((int64_t)oblob.size()); olen.push_back(x.L); oref.push_back(x.ref_row);
                        oblob.insert(oblob.end(), x.seqs.begin(), x.seqs.end());
                    }
                    std::vector<uint8_t>().swap(x.seqs);
                }
                const double my_extract = since(p0);
                const auto g0 = std::chrono::steady_clock::now();
                const int64_t nr = (int64_t)rbeg.size();
                std::vector<float> phylo(nr, NAN), anc(nr, NAN), bls(nr, NAN);
                if (nr > 0) {
                    const pcsf_status st = pcsf_score_given_regions(dev[w], strategy, (int32_t)coff.size(), cblob.data(), coff.data(), clen.data(), nr,
                                                                    raln.data(), rbeg.data(), rend.data(), phylo.data(), comp_anc ? anc.data() : nullptr,
                                                                    bls.data());
                    if (st == PCSF_ERR_BAD_CHAR) { fprintf(stderr, "%s\n", pcsf_last_error()); exit(37); }
                    if (st != PCSF_OK) die("pcsf_score_given_regions: %s", pcsf_last_error());
                }
                std::vector<pcsf_region> orfs(ooff.size());
                if (!ooff.empty()) {
                    int64_t n = 0;
                    pcsf_status st = pcsf_score_regions(dev[w], strategy, (int32_t)ooff.size(), oblob.data(), ooff.data(), olen.data(), oref.data(), 3,
                                                        PCSF_ORF_ATGSTOP, (int32_t)min_codons, 1, 0, 1, &n);
                    if (st == PCSF_ERR_BAD_CHAR) { fprintf(stderr, "%s\n", pcsf_last_error()); exit(37); }
                    if (st != PCSF_OK) die("pcsf_score_regions: %s", pcsf_last_error());
                    if ((st = pcsf_score_regions_get(dev[w], orfs.data(), n)) != PCSF_OK) die("pcsf_score_regions_get: %s", pcsf_last_error());
                }
                const double my_gpu = since(g0);
                const auto f0 = std::chrono::steady_clock::now();
                std::string text;
                char v[160];
                auto attr = [&](bool gff, const char *key, const char *val) {
                    if (gff) snprintf(v, sizeof v, ";%s=%s", key, val);
                    else snprintf(v, sizeof v, " %s \"%s\";", key, val);
                    text += v;
                };
                auto num = [](char *buf, size_t n, float f) { snprintf(buf, n, "%.6f", std::isnan(f) ? NAN : f); };
                for (size_t k = 0; k < tx.size(); ++k) {
                    const GffTranscript &t = recs[bt.r0 + k];
                    const TxAlignment &x = tx[k];
                    bool first = true, gff = true;
                    size_t cds_id = 0;
                    for (const auto &ln : t.lines) {
                        text += ln.second;
                        const bool tx_line = ln.first == Feature::Transcript;
                        if (scored[k] && (tx_line || (x.coding && ln.first == Feature::Cds))) {
                            if (first) { first = false; gff = is_gff_line(ln.second); }
                            char s[64];
                            if (x.coding) {
                                const int64_t r = first_region[k] + (tx_line ? 0 : (int64_t)(1 + cds_id++));
                                num(s, sizeof s, phylo[r]); attr(gff, "phylocsf_score", s);
                                if (comp_anc) { num(s, sizeof s, anc[r]); attr(gff, "phylocsf_anc", s); }
                                num(s, sizeof s, bls[r]); attr(gff, "phylocsf_bls", s);
                                snprintf(s, sizeof s, "%" PRId64, (rend[r] - rbeg[r]) / 3); attr(gff, "phylocsf_codons", s);
                            } else {
                                const pcsf_region *o = orf_index[k] >= 0 ? &orfs[(size_t)orf_index[k]] : nullptr;
                                const bool found = o && o->frame != 0;
                                num(s, sizeof s, found ? o->phylo : NAN); attr(gff, "phylocsf_orf_score", s);
                                if (found) {
                                    const uint64_t g0p = genomic_position(x, o->col_begin), g1p = genomic_position(x, o->col_end - 1);
                                    snprintf(s, sizeof s, "%" PRIu64, std::min(g0p, g1p)); attr(gff, "phylocsf_orf_start", s);
                                    snprintf(s, sizeof s, "%" PRIu64, std::max(g0p, g1p)); attr(gff, "phylocsf_orf_end", s);
                                    snprintf(s, sizeof s, "%" PRId64, o->codons); attr(gff, "phylocsf_orf_codons", s);
                                } else {
                                    attr(gff, "phylocsf_orf_start", "."); attr(gff, "phylocsf_orf_end", "."); attr(gff, "phylocsf_orf_codons", ".");
                                }
                                num(s, sizeof s, found ? o->bls : NAN); attr(gff, "phylocsf_orf_bls", s);
                            }
                        }
                        text += '\n';
                    }
                }
                std::vector<std::string> one(1);
                one[0] = std::move(text);
                sink.put(bi, std::move(one));
                std::lock_guard<std::mutex> g(stat_mu);
                t_extract += my_extract; t_gpu += my_gpu; t_format += since(f0);
                n_coding += (int64_t)coff.size(); n_orf += (int64_t)ooff.size();
            }
        });
    double t_write = 0.0;
    size_t bi = 0;
    for (const GffFile &f : files) {
        FILE *fo = fopen(f.out_path.c_str(), "w");
        if (!fo) die("Error creating file %s!", f.out_path.c_str());
        for (; bi < batches.size() && batches[bi].file == (size_t)(&f - files.data()); ++bi) {
            std::string text = sink.take(bi)[0];
            const auto w0 = std::chrono::steady_clock::now();
            if (batches[bi].r1 == f.recs.size() && !f.newline_at_end && !text.empty()) text.pop_back();          // the input's last line had none
            fwrite(text.data(), 1, text.size(), fo);
            t_write += since(w0);
        }
        fclose(fo);
    }
    for (auto &w : workers) w.join();
    printf("\33[2K\rDone!\n");
    if (getenv("PCSF_HOST_STATS"))
        printf("{\"transcripts\": %" PRId64 ", \"coding\": %" PRId64 ", \"orf_searched\": %" PRId64 ", \"seconds\": %.3f, \"scan_seconds\": %.3f, "
               "\"gff_read_seconds\": %.3f, \"extract_seconds_sum\": %.3f, \"gpu_call_seconds_sum\": %.3f, \"format_seconds_sum\": %.3f, "
               "\"write_seconds\": %.3f, \"workers\": %d}\n",
               n_coding + n_orf, n_coding, n_orf, since(t_start), t_scan, t_read, t_extract, t_gpu, t_format, t_write, workers_n);
    for (pcsf_model *m : dev) pcsf_model_destroy(m);
    return 0;
}

// Test hook (no GPU needed): the alignments annotate-with-maf scores.  One line per coding transcript and per CDS region, and one per
// transcript without CDS (its exon alignment and the reference row of its chains): file, record, kind, columns, region, FNV-1a hash.
int main_dump_transcripts(int argc, char **argv) {
    const Args a = parse_args(argc, argv, {"threads", "mapping", "species"});
    if (a.pos.size() < 3) die("usage: phylocsf_b200 dump-transcripts [--threads INT] <model> <alignments.maf[,more.maf...]> <gff/gtf files>...");
    Model model;
    load_model(model, a.pos[0], a.str("species"), a.str("mapping"));
    const int nl = model.nl();
    const ChainIndex idx(split(a.pos[1], ','), model, std::max(1, a.integer("threads", 4)));
    printf("# minus_chains %" PRId64 "\n", idx.minus_chains());
    ChainCache cache(idx);
    for (size_t fi = 2; fi < a.pos.size(); ++fi) {
        GffReader reader(a.pos[fi]);
        GffTranscript t;
        TxAlignment x;
        for (size_t rec = 0; reader.next(t); ++rec) {
            if (!extract_transcript(idx, cache, t, true, x)) continue;
            if (!x.coding) {
                printf("%zu\t%zu\texons\t%" PRId64 "\t0\t%" PRId64 "\t%016" PRIx64 "\t%d\n", fi - 2, rec, x.L, x.L, region_hash(x, nl, 0, x.L), x.ref_row);
                continue;
            }
            for (size_t r = 0; r < x.reg_begin.size(); ++r)
                printf("%zu\t%zu\t%s\t%" PRId64 "\t%" PRId64 "\t%" PRId64 "\t%016" PRIx64 "\t.\n", fi - 2, rec, r == 0 ? "transcript" : "CDS", x.L,
                       x.reg_begin[r], x.reg_end[r], region_hash(x, nl, x.reg_begin[r], x.reg_end[r]));
        }
    }
    return 0;
}

// wig-to-bigwig: the step the reference leaves to UCSC's wigToBigWig (README: "wigToBigWig PhyloCSF+1.wig chrom.sizes PhyloCSF+1.bw").
int main_wig_to_bigwig(int argc, char **argv) {
    const Args a = parse_args(argc, argv, {"compress"});
    if (a.pos.size() != 3) die("usage: phylocsf_b200 wig-to-bigwig [--compress BOOL] <in.wig> <chrom.sizes> <out.bw>");
    wig_to_bigwig(a.pos[0], read_chrom_sizes(a.pos[1]), a.pos[2], a.boolean("compress", true));
    return 0;
}

// bigwig-dump: header facts + every interval as bedGraph lines (the text bigWigToBedGraph prints) — what the tests compare.
int main_bigwig_dump(int argc, char **argv) {
    const Args a = parse_args(argc, argv, {"intervals"});
    if (a.pos.size() != 1) die("usage: phylocsf_b200 bigwig-dump [--intervals BOOL] <in.bw>");
    BigWigReader r;
    std::string err;
    if (!r.open(a.pos[0], err)) die("%s", err.c_str());
    const BigWigReader::Summary s = r.summary();
    printf("# version %d zoom_levels %d sections %" PRIu64 " bases_covered %" PRIu64 " min %.6g max %.6g sum %.9g sum_squares %.9g\n", r.version(), r.zoom_levels(),
           r.n_sections(), s.bases_covered, s.min, s.max, s.sum, s.sum_squares);
    for (const auto &c : r.chroms()) printf("# chrom %s id %u length %u\n", c.name.c_str(), c.id, c.len);
    if (a.boolean("intervals", true)) {
        std::vector<std::string> names(r.chroms().size());
        for (const auto &c : r.chroms()) if (c.id < names.size()) names[c.id] = c.name;
        if (!r.for_each_interval([&](uint32_t chrom, uint32_t b, uint32_t e, float v) { printf("%s\t%u\t%u\t%.9g\n", chrom < names.size() ? names[chrom].c_str() : "?", b, e, v); }))
            die("%s: damaged data section", a.pos[0].c_str());
    }
    return 0;
}


// Test / tuning hook (no GPU needed): the reader alone — scan + chain cutting + read_chain_into of every chain into a reused matrix,
// `--threads` workers over the chains; prints seconds and columns/s per phase.
int main_parse_bench(int argc, char **argv) {
    const Args a = parse_args(argc, argv, {"threads", "mapping", "species", "repeat"});
    if (a.pos.size() < 2) die("usage: phylocsf_b200 parse-bench [--threads INT] [--repeat INT] <model> <alignments>...");
    Model model;
    load_model(model, a.pos[0], a.str("species"), a.str("mapping"));
    const int threads = std::max(1, a.integer("threads", 4)), repeat = std::max(1, a.integer("repeat", 1));
    const int nl = model.nl();
    for (size_t fi = 1; fi < a.pos.size(); ++fi) {
        const auto t0 = std::chrono::steady_clock::now();
        MafFile maf(a.pos[fi], model, true, threads);
        const double t_scan = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        const std::vector<MafFile::Chain> &chains = maf.chains();
        int64_t max_cols = 1, total = 0;
        for (const auto &c : chains) { max_cols = std::max(max_cols, c.ref_cols); total += c.ref_id < 0 ? 0 : c.ref_cols; }
        for (int rep = 0; rep < repeat; ++rep) {
            std::atomic<size_t> next{0};
            std::atomic<int64_t> refused{0};
            std::vector<double> secs(threads, 0.0);
            const auto t1 = std::chrono::steady_clock::now();
            std::vector<std::thread> th;
            for (int t = 0; t < threads; ++t)
                th.emplace_back([&, t] {
                    std::vector<uint8_t> mat((size_t)nl * max_cols);
                    const auto b0 = std::chrono::steady_clock::now();
                    for (size_t ci = next++; ci < chains.size(); ci = next++)
                        if (chains[ci].ref_id >= 0 && maf.read_chain_into(chains[ci], mat.data(), chains[ci].ref_cols, nullptr) < 0) ++refused;
                    secs[t] = std::chrono::duration<double>(std::chrono::steady_clock::now() - b0).count();
                });
            for (auto &x : th) x.join();
            const double wall = std::chrono::duration<double>(std::chrono::steady_clock::now() - t1).count();
            double sum = 0;
            for (double x : secs) sum += x;
            printf("{\"file\": \"%s\", \"columns\": %" PRId64 ", \"chains\": %zu, \"threads\": %d, \"scan_seconds\": %.3f, \"parse_wall_seconds\": %.3f, "
                   "\"parse_core_seconds\": %.3f, \"columns_per_core_second\": %.0f, \"refused_chains\": %" PRId64 "}\n",
                   a.pos[fi].c_str(), total, chains.size(), threads, t_scan, wall, sum, total / std::max(sum, 1e-9), (int64_t)refused);
        }
    }
    return 0;
}

// Test hook (no GPU needed): the PhyloCSF-HMM stage alone on existing raw tracks.
int main_smooth_tracks(int argc, char **argv) {
    const Args a = parse_args(argc, argv, {"genome-length", "coding-exons", "output-phylo", "output-regions", "print-hmm"});
    if (a.pos.size() != 2 || !a.has("genome-length") || !a.has("coding-exons"))
        die("usage: phylocsf_b200 smooth-tracks --genome-length INT --coding-exons FILE [--output-phylo BOOL] [--output-regions BOOL] <raw dir> <out dir>");
    const HmmParams hp = estimate_hmm_params(a.str("coding-exons"), (uint32_t)strtoull(a.str("genome-length").c_str(), nullptr, 10));
    const Hmm h = coding_hmm(hp);
    if (a.boolean("print-hmm", false)) {
        printf("coding_prior %.17g\ncoding_codons %.17g\n", hp.coding_prior, hp.coding_codons);
        for (int j = 0; j < 3; ++j) printf("nc %d weight %.17g codons %.17g\n", j, hp.nc_weight[j], hp.nc_codons[j]);
    }
    create_directory(a.pos[1]);
    static const char *kFrames[6] = {"+1", "+2", "+3", "-1", "-2", "-3"};
    for (int k = 0; k < 6; ++k) {
        FILE *fw = a.boolean("output-phylo", true) ? fopen((a.pos[1] + "/PhyloCSF" + kFrames[k] + ".wig").c_str(), "w") : nullptr;
        FILE *fb = a.boolean("output-regions", true) ? fopen((a.pos[1] + "/PhyloCSF" + kFrames[k] + "Regions.bed").c_str(), "w") : nullptr;
        hmm_smooth_file(h, a.pos[0] + "/PhyloCSFRaw" + kFrames[k] + ".wig", kFrames[k][0], fw, fb);
        if (fw) fclose(fw);
        if (fb) fclose(fb);
    }
    return 0;
}

// Test hook: the snprintf-free formatter against the reference's route on n pseudo-random floats + special values.
int main_format_selftest(int argc, char **argv) {
    const long n = argc > 2 ? atol(argv[2]) : 1000000;
    uint64_t x = 0x9E3779B97F4A7C15ull;
    long bad = 0;
    std::string a, b;
    auto check = [&](float v) {
        for (int dec = 3; dec <= 4; ++dec) {
            a.clear(); b.clear();
            my_format(a, dec, v); my_format_printf(b, dec, v);
            if (a != b) { if (bad < 10) printf("mismatch %.9g: '%s' vs '%s'\n", v, a.c_str(), b.c_str()); ++bad; }
            char buf[64];
            const size_t nb = (size_t)(my_format_to(buf, dec, v) - buf);          // the route the build-tracks workers take
            if (nb != b.size() || memcmp(buf, b.data(), nb) != 0) { if (bad < 10) printf("mismatch (my_format_to) %.9g: '%.*s' vs '%s'\n", v, (int)nb, buf, b.c_str()); ++bad; }
        }
    };
    const float special[] = {0.f, -0.f, 0.0625f, 0.1875f, -0.0004f, 0.0005f, 0.00049999f, 1e-30f, -1e-30f, 2.f, 10.f, 0.9995f, 0.99951f, 12345.6789f, -999.9995f,
                             1e10f, 3.4e38f, 0.3125f, 0.4375f, 24.834f, 3.54f, 3999999.75f, 4000000.f, 4.1e6f, -4.1e6f, 99.9995f, 100.f, 9.9995f, 999.9995f, 1000.5f};
    for (float v : special) check(v);
    for (long i = 0; i < n; ++i) {
        x ^= x << 13; x ^= x >> 7; x ^= x << 17;
        const int e = (int)((x >> 40) % 40) - 20;                       // magnitudes 2^-20 .. 2^19
        float v = (float)std::ldexp((double)(x & 0xffffff) / 16777216.0 + 0.5, e);
        if (x & (1ull << 63)) v = -v;
        check(v);
        // exact ties at the rounding position
        check((float)((double)((x >> 8) & 0xfffff) / 2048.0));
    }
    printf("%ld mismatches\n", bad);
    return bad != 0;
}

}  // namespace

int main(int argc, char **argv) {
    if (argc < 2 || !strcmp(argv[1], "--help") || !strcmp(argv[1], "-h")) {
        printf("phylocsf_b200 — B200-native PhyloCSF++ likelihood core behind the reference's command line\n\n"
               "  phylocsf_b200 build-tracks [--output-raw-phylo BOOL] [--output-phylo BOOL] [--output-regions BOOL] [--genome-length INT]\n"
               "                             [--coding-exons FILE] [--power-threshold FLOAT] [--threads INT] [--gpus INT]\n"
               "                             [--precision f64|tc5] [--output-bigwig BOOL] [--output DIR] [--mapping FILE] [--species LIST] <model> <maf>...\n"
               "  phylocsf_b200 score-msa    [--strategy MLE|FIXED|OMEGA|FIXED_MEAN] [--comp-phylo BOOL] [--comp-anc BOOL] [--threads INT] [--gpus INT]\n"
               "                             [--frames 1|3|6] [--orf AsIs|StopStop|ATGStop] [--min-codons INT] [--all-scores BOOL]\n"
               "                             [--output DIR] [--mapping FILE] [--species LIST] <model> <maf>...\n"
               "  phylocsf_b200 annotate-with-tracks [--output DIR] <PhyloCSF+1.bw> <gff/gtf>...\n"
               "  phylocsf_b200 annotate-with-maf [--output DIR] [--strategy MLE|FIXED|OMEGA] [--comp-anc BOOL] [--find-orf BOOL] [--min-codons INT]\n"
               "                             [--species LIST] [--mapping FILE] [--threads INT] [--gpus INT] <model> <maf[,maf...]> <gff/gtf>...\n"
               "  phylocsf_b200 wig-to-bigwig [--compress BOOL] <in.wig> <chrom.sizes> <out.bw>\n");
        return argc < 2 ? 1 : 0;
    }
    const std::string tool = argv[1];
    if (tool == "build-tracks") return main_build_tracks(argc, argv);
    if (tool == "smooth-tracks") return main_smooth_tracks(argc, argv);
    if (tool == "score-msa") return main_score_msa(argc, argv);
    if (tool == "dump-alignments") return main_dump_alignments(argc, argv);
    if (tool == "format-selftest") return main_format_selftest(argc, argv);
    if (tool == "matrix-to-maf") return main_matrix_to_maf(argc, argv);
    if (tool == "parse-bench") return main_parse_bench(argc, argv);
    if (tool == "annotate-with-tracks") return main_annotate_with_tracks(argc, argv);
    if (tool == "annotate-with-maf") return main_annotate_with_maf(argc, argv);
    if (tool == "dump-transcripts") return main_dump_transcripts(argc, argv);
    if (tool == "wig-to-bigwig") return main_wig_to_bigwig(argc, argv);
    if (tool == "bigwig-dump") return main_bigwig_dump(argc, argv);
    die("unknown tool '%s' (build-tracks, score-msa, annotate-with-tracks, annotate-with-maf and wig-to-bigwig are available)", tool.c_str());
}
