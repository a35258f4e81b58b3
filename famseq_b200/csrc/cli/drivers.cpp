// drivers.cpp -- see drivers.hpp.
//
// The reference handles one record at a time (parse, set_LK, calPostProb*, print).  Here the text side
// keeps the reference's record rules and output bytes, but records travel in blocks of up to kBatch lines
// through a three-stage pipeline whose stages overlap:
//     parse(k+1)  ||  engine(k)  ||  format(k-1)  ||  file write
// parse and format are spread over the host threads, the engine stage is one fs_run_pl() / fs_run() call on
// pinned buffers (H2D / kernel / D2H pipelined inside the engine), output order is input order.
// Integer PL fields go to the engine as they stand (uint16, decoded on the device through the engine's
// host-libm table: the host never calls pow for them); anything else (GL, decimals, the LK modes) is decoded on
// the host with libm and takes the FP64 entry.  Phred encoding (log10) stays on the host so that the text is
// byte-identical to the reference's.
#include "drivers.hpp"
#include "../host/format_g.hpp"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <limits>
#include <sstream>
#include <string_view>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <thread>

#include "../../../include/famseq_b200.h"

namespace famseq_cli {

RunStats g_stats;
bool g_engine_failed = false;

namespace {

using sv = std::string_view;
constexpr size_t kBatch = 1u << 17; // record lines per pipeline block
constexpr int kSlots = 4;             // blocks in flight (parse / engine / format + one of slack)

double now() {
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// The reference's split() (normal.cpp:15-53): single-character delimiter, empty fields are kept, a trailing
// delimiter yields a trailing empty field, an empty source yields nothing.
void split(sv src, char tok, std::vector<sv> &out) {
    out.clear();
    if (src.empty()) return;
    size_t head = 0;
    for (;;) {
        const size_t tail = src.find(tok, head);
        if (tail == sv::npos) break;
        out.push_back(src.substr(head, tail - head));
        head = tail + 1;
    }
    out.push_back(src.substr(head));
}

double to_double(sv s) { // atof
    char buf[64];
    const size_t n = std::min(s.size(), sizeof buf - 1);
    std::memcpy(buf, s.data(), n);
    buf[n] = 0;
    return std::strtod(buf, nullptr);
}

int to_int(sv s) { // atoi
    char buf[32];
    const size_t n = std::min(s.size(), sizeof buf - 1);
    std::memcpy(buf, s.data(), n);
    buf[n] = 0;
    return std::atoi(buf);
}

// Reads until end of file with a growing buffer, so that pipes and process substitutions (`-vcfFile <(zcat x.vcf.gz)`,
// which the reference's ifstream/getline accepts) work like regular files; the size of a regular file is only a hint.
bool read_file(const std::string &path, std::string &data) {
    FILE *f = std::fopen(path.c_str(), "rb");
    if (!f) return false;
    size_t hint = 0;
    if (std::fseek(f, 0, SEEK_END) == 0) {
        const long sz = std::ftell(f);
        if (sz > 0) hint = (size_t)sz;
        std::fseek(f, 0, SEEK_SET);
    }
    data.clear();
    size_t got = 0;
    for (;;) {
        if (data.size() - got < (1u << 16)) data.resize(std::max<size_t>({hint + 1, data.size() * 2, (size_t)1 << 20}));
        const size_t n = std::fread(&data[got], 1, data.size() - got, f);
        got += n;
        if (n == 0) break;
    }
    const bool ok = !std::ferror(f);
    std::fclose(f);
    data.resize(got);
    return ok;
}

// The whole input as one string_view: regular files are mapped (no copy; the page faults are taken by the parsing
// threads), anything else (pipes, process substitutions) is read to the end into memory.
class InputFile {
  public:
    ~InputFile() {
        if (map_) munmap(map_, size_);
    }
    bool open(const std::string &path) {
        const int fd = ::open(path.c_str(), O_RDONLY);
        if (fd < 0) return false;
        struct stat st;
        if (fstat(fd, &st) == 0 && S_ISREG(st.st_mode) && st.st_size > 0) {
            void *m = mmap(nullptr, (size_t)st.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
            if (m != MAP_FAILED) {
                map_ = m;
                size_ = (size_t)st.st_size;
                madvise(m, size_, MADV_WILLNEED);
                ::close(fd);
                return true;
            }
        }
        ::close(fd);
        return read_file(path, data_);
    }
    sv view() const { return map_ ? sv(static_cast<const char *>(map_), size_) : sv(data_); }

  private:
    void *map_ = nullptr;
    size_t size_ = 0;
    std::string data_;
};

// getline()-style cursor over an in-memory file.  Mirrors `while(!fin.eof()) getline(fin, line)`: after the last
// newline one more, empty, line is delivered.
struct Lines {
    sv data;
    size_t pos = 0;
    bool done = false;
    explicit Lines(sv d) : data(d) {}
    bool next(sv &line) {
        if (done) return false;
        const void *hit = pos < data.size() ? std::memchr(data.data() + pos, '\n', data.size() - pos) : nullptr;
        if (!hit) {
            line = data.substr(pos);
            done = true;
        } else {
            const size_t nl = (size_t)(static_cast<const char *>(hit) - data.data());
            line = data.substr(pos, nl - pos);
            pos = nl + 1;
        }
        return true;
    }
};

// A PL-like field as the engine's compact input wants it: the whole token is an optionally signed run of digits.
// |value| is returned clamped to 65535 (every PL >= 3237 decodes to exactly 0.0, so the clamp is exact).  False for
// anything else (decimals, exponents, blanks, empty): the caller then takes atof() and the FP64 path.
inline bool integer_field(sv s, uint16_t &out) {
    size_t i = 0;
    if (i < s.size() && (s[i] == '-' || s[i] == '+')) i++;
    if (i == s.size()) return false;
    unsigned v = 0;
    for (; i < s.size(); i++) {
        const unsigned d = (unsigned)(s[i] - '0');
        if (d > 9) return false;
        v = std::min(v * 10 + d, 1000000u);
    }
    out = (uint16_t)std::min(v, 65535u);
    return true;
}

// ostream's default formatting of a double is printf's %g with 6 significant digits (format_g.hpp: same bytes, faster).
void put_number(std::string &out, double v) { famseq::append_g(out, v); }

// file.cpp:702-749: -10*log10(p); +inf is printed as 99999, everything else as its absolute value
void put_phred(std::string &out, double p) {
    const double v = -10 * std::log10(p);
    if (v == std::numeric_limits<double>::infinity())
        out += "99999";
    else
        put_number(out, std::fabs(v));
}

struct BlockResults;

// One Phred column from a device code; the few codes the device left open are looked up (exact double) and formatted here.
void put_phred_code(std::string &out, uint32_t code, int64_t index, const fs_phred_fix *fixes, size_t n_fixes) {
    char buf[16];
    const int n = fs_phred_text(code, buf);
    if (n >= 0) {
        out.append(buf, (size_t)n);
        return;
    }
    const fs_phred_fix *end = fixes + n_fixes;
    const fs_phred_fix *it = std::lower_bound(fixes, end, index, [](const fs_phred_fix &f, int64_t i) { return f.index < i; });
    put_phred(out, it != end && it->index == index ? it->p : std::numeric_limits<double>::quiet_NaN());
}

// GPP, FPP and FGT of one sample (file.cpp:702-761); `off` is the position of the sample's first value in the block
void put_calls(std::string &out, const BlockResults &R, size_t off, uint8_t gt);

const char *kFormatLines =
    "##FORMAT=<ID=FPP,Number=G,Type=Integer,Description=\"Normalized, Phred-scaled for posterior probability calculated by FamSeqPro\">\n"
    "##FORMAT=<ID=FGT,Number=1,Type=String,Description=\"Genotype called by FamSeqPro\">\n";

struct Priors {
    double n[3], k[3], xn[3], xk[3];
};

void fill_params(const CommonOptions &o, fs_params &p, Priors &shown) {
    fs_default_params(&p);
    p.mrate = o.mrate;
    p.lrc = o.lrc;
    auto set = [](const std::vector<double> &src, double *dst) {
        if (src.size() == 3) std::copy(src.begin(), src.end(), dst);
    };
    set(o.geno_prob_n, p.geno_prob_n);
    set(o.geno_prob_k, p.geno_prob_k);
    set(o.geno_prob_xn, p.geno_prob_xn);
    set(o.geno_prob_xk, p.geno_prob_xk);
    std::memcpy(shown.n, p.geno_prob_n, 24);
    std::memcpy(shown.k, p.geno_prob_k, 24);
    std::memcpy(shown.xn, p.geno_prob_xn, 24);
    std::memcpy(shown.xk, p.geno_prob_xk, 24);
}

void put_triplet(std::string &out, const double *v) {
    put_number(out, v[0]); out += ':';
    put_number(out, v[1]); out += ':';
    put_number(out, v[2]);
}

// Maps input columns to ped rows by exact name match, first matching ped row wins (file.cpp:209-220).
struct ColumnMap {
    std::vector<int> ped_row;  // per input column: ped row or -1
    std::vector<int> matched;  // input columns with a ped row, in input order
    std::vector<int> unique;   // per matched column: index into `engine_cols`
    std::vector<int32_t> engine_cols; // distinct ped rows, order of first appearance
    int real_num_ind() const { return (int)matched.size(); }
};

ColumnMap map_columns(const std::vector<sv> &names, size_t first, const PedRows &ped) {
    ColumnMap m;
    for (size_t c = first; c < names.size(); c++) {
        int row = -1;
        for (size_t j = 0; j < ped.name.size(); j++)
            if (names[c] == sv(ped.name[j])) {
                row = (int)j;
                break;
            }
        m.ped_row.push_back(row);
        if (row < 0) continue;
        m.matched.push_back((int)(c - first));
        auto it = std::find(m.engine_cols.begin(), m.engine_cols.end(), row);
        if (it == m.engine_cols.end()) {
            m.unique.push_back((int)m.engine_cols.size());
            m.engine_cols.push_back(row);
        } else
            m.unique.push_back((int)(it - m.engine_cols.begin()));
    }
    return m;
}

// The engine of a run: ONE fs_engine, over one GPU or (fs_create_multi) over several -- every batch is then cut into
// contiguous slices, one per device, inside the engine (variants are independent; the Gibbs sampler's streams are
// keyed by the global variant index, so the output does not depend on the number of devices).
constexpr size_t kMaxPedigreeMembers = 128; // fs_create's limit

struct Engine {
    fs_engine *h = nullptr;
    bool family_bn = false; // -familyBN -method 1: fs_create_cohort_bn, for a ped file of any size
    bool mcmc = false;      // -method 3: fs_create_cohort_mcmc for a ped file past 128 members
    ~Engine() { fs_destroy(h); }
    static std::vector<int> resolve(const std::vector<int> &wanted, int fallback) {
        if (wanted.empty()) return {fallback};
        if (wanted[0] >= 0) return wanted;
        std::vector<int> all;
        for (int d = 0; d < std::max(1, fs_device_count()); d++) all.push_back(d);
        return all;
    }
    bool create(const PedRows &ped, const ColumnMap &cm, const fs_params &prm, const std::vector<int> &devices) {
        std::vector<int32_t> id(ped.id.begin(), ped.id.end()), mo(ped.mother_id.begin(), ped.mother_id.end()),
            fa(ped.father_id.begin(), ped.father_id.end()), ge(ped.gender.begin(), ped.gender.end());
        fs_pedigree fp{(int32_t)id.size(), id.data(), mo.data(), fa.data(), ge.data(), (int32_t)cm.engine_cols.size(),
                       cm.engine_cols.data()};
        // ped files past the 128 members of one pedigree: a cohort of families, each on its own chain (MCMC) or a cohort of
        // loop-free families (ES)
        const bool cohort = id.size() > kMaxPedigreeMembers;
        const int rc = family_bn        ? fs_create_cohort_bn(&fp, &prm, devices.data(), (int)devices.size(), &h)
                       : cohort && mcmc ? fs_create_cohort_mcmc(&fp, &prm, devices.data(), (int)devices.size(), &h)
                       : cohort         ? fs_create_cohort(&fp, &prm, devices.data(), (int)devices.size(), &h)
                                        : fs_create_multi(&fp, &prm, devices.data(), (int)devices.size(), &h);
        if (rc != FS_OK) {
            std::cout << fs_last_error() << std::endl;
            g_engine_failed = true;
            return false;
        }
        return true;
    }
};

// Pinned host buffers of one pipeline slot (fs_alloc_pinned: the engine's copies then run at full PCIe speed and
// asynchronously).  Allocated by the engine stage, i.e. after the CUDA context exists.
struct HostBuffers {
    size_t cap = 0; // variants
    uint16_t *pl = nullptr;
    uint32_t *post32 = nullptr, *single32 = nullptr; // Phred codes (compact blocks)
    double *lk = nullptr, *post = nullptr, *single = nullptr; // FP64 blocks: allocated when the first one comes along
    uint8_t *flags = nullptr, *gt = nullptr, *status = nullptr;
    std::vector<fs_phred_fix> fixes; // values of a compact block the host formats itself, sorted by index
    ~HostBuffers() { release(); }
    void release() {
        fs_free_pinned(pl);
        fs_free_pinned(post32);
        fs_free_pinned(single32);
        fs_free_pinned(lk);
        fs_free_pinned(post);
        fs_free_pinned(single);
        fs_free_pinned(flags);
        fs_free_pinned(gt);
        fs_free_pinned(status);
        pl = nullptr, post32 = single32 = nullptr, lk = post = single = nullptr, flags = gt = status = nullptr, cap = 0;
    }
    bool reserve(size_t variants, size_t S, bool want_lk) {
        if (variants > cap) {
            release();
            cap = std::max(variants, kBatch);
            const size_t n3 = std::max<size_t>(cap * S * 3, 1);
            pl = static_cast<uint16_t *>(fs_alloc_pinned(n3 * sizeof(uint16_t)));
            post32 = static_cast<uint32_t *>(fs_alloc_pinned(n3 * sizeof(uint32_t)));
            single32 = static_cast<uint32_t *>(fs_alloc_pinned(n3 * sizeof(uint32_t)));
            flags = static_cast<uint8_t *>(fs_alloc_pinned(cap));
            gt = static_cast<uint8_t *>(fs_alloc_pinned(std::max<size_t>(cap * S, 1)));
            status = static_cast<uint8_t *>(fs_alloc_pinned(cap));
            if (!pl || !post32 || !single32 || !flags || !gt || !status) return false;
        }
        if (want_lk && !lk) {
            const size_t n3 = std::max<size_t>(cap * S * 3, 1);
            lk = static_cast<double *>(fs_alloc_pinned(n3 * sizeof(double)));
            post = static_cast<double *>(fs_alloc_pinned(n3 * sizeof(double)));
            single = static_cast<double *>(fs_alloc_pinned(n3 * sizeof(double)));
            if (!lk || !post || !single) return false;
        }
        return true;
    }
};

// What a host thread parsed from / formats for its contiguous range of a block.
struct Part {
    std::vector<sv> lines;        // records that produce output, in input order
    std::vector<uint8_t> echo;    // per line: 1 = echoed as it stands (VCF skip rules), 0 = computed
    std::vector<uint16_t> pl;     // compact likelihoods [count][S][3] (while `compact`)
    std::vector<double> lk;       // FP64 likelihoods   [count][S][3] (once a field was not an integer)
    std::vector<uint8_t> flags;   // [count]
    bool compact = true;
    std::string out, warn;
    long long failed = 0;
    size_t first = 0; // index of this part's first computed variant inside the block
    size_t count() const { return flags.size(); }
    void reset() {
        lines.clear(), echo.clear(), pl.clear(), lk.clear(), flags.clear();
        compact = true;
    }
    // a non-integer field was met: continue in FP64 (what is already there decodes through the same table the device uses)
    void widen(const double *table) {
        if (!compact) return;
        lk.resize(pl.size());
        for (size_t k = 0; k < pl.size(); k++) lk[k] = table[pl[k]];
        pl.clear();
        compact = false;
    }
};

struct Block {
    std::vector<sv> lines;
    std::vector<Part> parts;
    size_t total = 0;
    long long v_offset = 0;
    bool compact = true;
    size_t n_fixes = 0;
    HostBuffers buf;
};

// Bounded FIFO between two pipeline stages; close() wakes everybody up (end of input or failure).
template <class T> class Channel {
  public:
    bool push(T v) {
        std::unique_lock<std::mutex> lk(m_);
        if (closed_) return false;
        q_.push_back(v);
        cv_.notify_all();
        return true;
    }
    bool pop(T &v) {
        std::unique_lock<std::mutex> lk(m_);
        cv_.wait(lk, [this] { return closed_ || !q_.empty(); });
        if (q_.empty()) return false;
        v = q_.front();
        q_.pop_front();
        return true;
    }
    void close() {
        std::lock_guard<std::mutex> lk(m_);
        closed_ = true;
        cv_.notify_all();
    }

  private:
    std::mutex m_;
    std::condition_variable cv_;
    std::deque<T> q_;
    bool closed_ = false;
};

// Number of host threads for parsing / formatting: FAMSEQ_THREADS or the hardware concurrency (at most 64).
int host_threads() {
    int n = (int)std::thread::hardware_concurrency();
    if (const char *env = std::getenv("FAMSEQ_THREADS")) n = std::atoi(env);
    return std::max(1, std::min(n, 64));
}

template <class F> void run_parallel(int n, F f) {
    std::vector<std::thread> pool;
    for (int t = 1; t < n; t++) pool.emplace_back(f, t);
    f(0);
    for (auto &th : pool) th.join();
}

// Output file writer on its own thread: formatted blocks are queued in order and written while the next block is
// being parsed, computed and formatted.  The queue is bounded (the producer waits when the disk is slower).
class AsyncWriter {
  public:
    explicit AsyncWriter(FILE *f) : f_(f), th_([this] { loop(); }) {}
    ~AsyncWriter() { close(); }
    void push(std::string &&s) {
        if (s.empty()) return;
        std::unique_lock<std::mutex> lk(m_);
        cv_space_.wait(lk, [this] { return q_.size() < 256; });
        q_.push_back(std::move(s));
        cv_data_.notify_one();
    }
    bool close() { // drains the queue; the caller closes the FILE.  False when a write failed (disk full, ...)
        {
            std::lock_guard<std::mutex> lk(m_);
            if (done_) return !failed_;
            done_ = true;
        }
        cv_data_.notify_one();
        th_.join();
        return !failed_;
    }

  private:
    void loop() {
        for (;;) {
            std::string s;
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_data_.wait(lk, [this] { return done_ || !q_.empty(); });
                if (q_.empty()) return;
                s = std::move(q_.front());
                q_.pop_front();
            }
            cv_space_.notify_one();
            if (!failed_ && std::fwrite(s.data(), 1, s.size(), f_) != s.size()) failed_ = true; // keep draining so the producer never blocks
        }
    }
    FILE *f_;
    bool failed_ = false; // written by the writer thread, read after join()
    std::mutex m_;
    std::condition_variable cv_data_, cv_space_;
    std::deque<std::string> q_;
    bool done_ = false;
    std::thread th_;
};

// fs_create (CUDA context, pedigree compilers) on its own thread, so that it overlaps the parsing of the first block.
class EngineStart {
  public:
    EngineStart(Engine &e, const PedRows &ped, const ColumnMap &cm, const fs_params &prm, std::vector<int> devices)
        : th_([&e, &ped, &cm, &prm, devices, this] { ok_ = e.create(ped, cm, prm, devices); }) {}
    ~EngineStart() { wait(); }
    bool wait() {
        if (th_.joinable()) th_.join();
        return ok_;
    }

  private:
    bool ok_ = false;
    std::thread th_;
};

// The record pipeline shared by the two drivers.
//   accept(line): 0 = the input ends here, 1 = a record, 2 = skip the line
//   parse(part, lines, n, compact): fills `part` from n record lines; with compact = true it returns false as soon as a
//                                   likelihood field is not an integer (the range is then parsed again in FP64)
//   format(part, results): writes part.out / part.warn / part.failed from the engine's results of the part's block
struct BlockResults {
    const double *post, *single;       // FP64 blocks
    const uint32_t *post32, *single32; // compact blocks: Phred codes from the device
    const fs_phred_fix *fixes;         // ... and the few values it left to the host, sorted by index
    size_t n_fixes;
    const uint8_t *gt, *status;
    bool compact;
};
void put_calls(std::string &out, const BlockResults &R, size_t off, uint8_t gt) {
    static const char sep[3] = {',', ',', ':'};
    if (R.compact) {
        for (int g = 0; g < 3; g++) {
            put_phred_code(out, R.single32[off + g], (int64_t)(off + g) + FS_PHRED_FIX_SINGLE, R.fixes, R.n_fixes);
            out += sep[g];
        }
        for (int g = 0; g < 3; g++) {
            put_phred_code(out, R.post32[off + g], (int64_t)(off + g), R.fixes, R.n_fixes);
            out += sep[g];
        }
    } else {
        for (int g = 0; g < 3; g++) {
            put_phred(out, R.single[off + g]);
            out += sep[g];
        }
        for (int g = 0; g < 3; g++) {
            put_phred(out, R.post[off + g]);
            out += sep[g];
        }
    }
    out += gt == 0 ? "0/0\t" : (gt == 1 ? "0/1\t" : "1/1\t"); // file.cpp:750-761: anything but 0 and 1 prints 1/1
}

struct PipelineSetup {
    Engine *engine;
    EngineStart *start;
    int S, method, burn, rep;
    unsigned long long seed;
    AsyncWriter *writer;
};

template <class Accept, class Parse, class Format>
bool run_pipeline(Lines &in, const PipelineSetup &ps, Accept accept, Parse parse, Format format) {
    const int n_threads = host_threads();
    const size_t S = (size_t)ps.S;
    std::vector<Block> blocks((size_t)kSlots);
    Channel<Block *> free_q, engine_q, format_q;
    for (Block &b : blocks) {
        b.parts.resize((size_t)n_threads);
        free_q.push(&b);
    }
    std::atomic<bool> ok{true};
    auto abort_all = [&]() {
        ok = false;
        free_q.close();
        engine_q.close();
        format_q.close();
    };

    // ---- stage A: cut the input into blocks and parse them ---------------------------------------------------
    std::thread stage_a([&] {
        long long v_offset = 0;
        bool eof = false;
        Block *b = nullptr;
        while (!eof && free_q.pop(b)) {
            const double t0 = now();
            b->lines.clear();
            sv line;
            while (b->lines.size() < kBatch) {
                if (!in.next(line)) {
                    eof = true;
                    break;
                }
                const int what = accept(line);
                if (what == 0) {
                    eof = true;
                    break;
                }
                if (what == 1) b->lines.push_back(line);
            }
            if (b->lines.empty()) break;
            g_stats.records += (long long)b->lines.size();
            run_parallel(n_threads, [&](int t) {
                const size_t lo = b->lines.size() * (size_t)t / n_threads, hi = b->lines.size() * (size_t)(t + 1) / n_threads;
                Part &P = b->parts[t];
                P.reset();
                if (!parse(P, b->lines.data() + lo, hi - lo, true)) {
                    P.reset();
                    P.compact = false;
                    parse(P, b->lines.data() + lo, hi - lo, false);
                }
            });
            b->total = 0;
            b->compact = true;
            for (Part &P : b->parts) {
                P.first = b->total;
                b->total += P.count();
                b->compact = b->compact && (P.compact || P.count() == 0);
            }
            b->v_offset = v_offset;
            v_offset += (long long)b->total;
            g_stats.parse_s += now() - t0;
            if (!engine_q.push(b)) break;
        }
        engine_q.close();
    });

    // ---- stage B: one engine call per block on pinned buffers ----------------------------------------------------
    std::thread stage_b([&] {
        std::vector<double> table;
        Block *b = nullptr;
        while (engine_q.pop(b)) {
            if (b->total) {
                double t0 = now();
                const bool ready = ps.start->wait();
                g_stats.start_wait_s += now() - t0;
                if (!ready) break;
                t0 = now();
                const bool reserved = b->buf.reserve(b->total, S, !b->compact);
                g_stats.alloc_s += now() - t0;
                if (!reserved) {
                    std::cout << "Cannot allocate pinned host memory for a block of " << b->total << " variants" << std::endl;
                    g_engine_failed = true;
                    break;
                }
                if (!b->compact && table.empty()) {
                    table.resize(FS_PL_TABLE_SIZE);
                    fs_get_pl_table(ps.engine->h, table.data());
                }
                for (Part &P : b->parts) {
                    if (!P.count()) continue;
                    std::memcpy(b->buf.flags + P.first, P.flags.data(), P.count());
                    const size_t n3 = P.count() * S * 3, off = P.first * S * 3;
                    if (b->compact)
                        std::memcpy(b->buf.pl + off, P.pl.data(), n3 * sizeof(uint16_t));
                    else if (P.compact)
                        for (size_t k = 0; k < n3; k++) b->buf.lk[off + k] = table[P.pl[k]];
                    else
                        std::memcpy(b->buf.lk + off, P.lk.data(), n3 * sizeof(double));
                }
                int rc;
                if (b->compact) { // integer PL fields up, Phred codes down: 2 and 4 bytes per value instead of 8 and 8
                    int64_t n_fixes = 0;
                    b->buf.fixes.resize(std::max<size_t>(b->buf.fixes.size(), 4096));
                    rc = fs_run_pl_phred(ps.engine->h, ps.method, (int64_t)b->total, b->buf.pl, b->buf.flags, ps.burn, ps.rep, ps.seed, b->v_offset,
                                         b->buf.post32, b->buf.single32, b->buf.gt, b->buf.status, b->buf.fixes.data(), (int64_t)b->buf.fixes.size(), &n_fixes);
                    if (rc == FS_OK && n_fixes > (int64_t)b->buf.fixes.size()) { // more exceptions than room (NaN-ridden input): once more with room for all
                        b->buf.fixes.resize((size_t)n_fixes);
                        rc = fs_run_pl_phred(ps.engine->h, ps.method, (int64_t)b->total, b->buf.pl, b->buf.flags, ps.burn, ps.rep, ps.seed, b->v_offset,
                                             b->buf.post32, b->buf.single32, b->buf.gt, b->buf.status, b->buf.fixes.data(), (int64_t)b->buf.fixes.size(), &n_fixes);
                    }
                    b->n_fixes = rc == FS_OK ? (size_t)n_fixes : 0;
                    std::sort(b->buf.fixes.begin(), b->buf.fixes.begin() + (long)b->n_fixes,
                              [](const fs_phred_fix &x, const fs_phred_fix &y) { return x.index < y.index; });
                    g_stats.phred_fixes += (long long)b->n_fixes;
                } else {
                    rc = fs_run(ps.engine->h, ps.method, (int64_t)b->total, b->buf.lk, b->buf.flags, ps.burn, ps.rep, ps.seed, b->v_offset, b->buf.post,
                                b->buf.single, b->buf.gt, b->buf.status);
                }
                g_stats.engine_s += now() - t0;
                if (!g_stats.batches) g_stats.first_engine_s = now() - t0;
                g_stats.kernel_ms += fs_last_kernel_ms(ps.engine->h);
                g_stats.batches++;
                if (b->compact) g_stats.compact_batches++;
                if (rc != FS_OK) {
                    std::cout << fs_last_error() << std::endl;
                    g_engine_failed = true;
                    break;
                }
            }
            if (!format_q.push(b)) break;
            b = nullptr;
        }
        if (g_engine_failed || !ok) abort_all();
        format_q.close();
    });

    // ---- stage C (this thread): format and hand to the writer, in order ------------------------------------------
    {
        Block *b = nullptr;
        while (format_q.pop(b)) {
            const double t0 = now();
            const BlockResults res{b->buf.post, b->buf.single, b->buf.post32, b->buf.single32, b->buf.fixes.data(), b->compact ? b->n_fixes : 0,
                                   b->buf.gt, b->buf.status, b->compact};
            run_parallel(n_threads, [&](int t) { format(b->parts[t], res); });
            for (Part &P : b->parts) {
                ps.writer->push(std::move(P.out));
                P.out.clear();
                if (!P.warn.empty()) std::cout << P.warn << std::flush;
                g_stats.failed += P.failed;
            }
            g_stats.computed += (long long)b->total;
            g_stats.write_s += now() - t0;
            if (!free_q.push(b)) break;
        }
    }
    if (g_engine_failed) abort_all();
    free_q.close();
    stage_a.join();
    stage_b.join();
    // an input without records still reports a pedigree the engine rejects
    const double t0 = now();
    const bool ready = ps.start->wait();
    g_stats.start_wait_s += now() - t0;
    return ok && ready && !g_engine_failed;
}


void emit_stats() {
    if (!std::getenv("FAMSEQ_STATS")) return;
    std::fprintf(stderr,
                 "{\"records\": %lld, \"computed\": %lld, \"failed\": %lld, \"batches\": %lld, \"compact_batches\": %lld, \"phred_fixes\": %lld, \"parse_s\": %.4f, "
                 "\"engine_s\": %.4f, \"alloc_s\": %.4f, \"first_engine_s\": %.4f, \"kernel_ms\": %.3f, \"write_s\": %.4f, \"read_s\": %.4f, \"start_wait_s\": %.4f, "
                 "\"drain_s\": %.4f, \"total_s\": %.4f}\n",
                 g_stats.records, g_stats.computed, g_stats.failed, g_stats.batches, g_stats.compact_batches, g_stats.phred_fixes, g_stats.parse_s, g_stats.engine_s,
                 g_stats.alloc_s, g_stats.first_engine_s, g_stats.kernel_ms, g_stats.write_s, g_stats.read_s, g_stats.start_wait_s, g_stats.drain_s, g_stats.total_s);
}

} // namespace

// --------------------------------------------------------------------------------------------------------
bool read_ped(const std::string &path, PedRows &out) {
    std::ifstream fin(path.c_str());
    if (!fin.is_open()) {
        std::cout << "Cannot open " << path << std::endl;
        return false;
    }
    std::string line;
    std::getline(fin, line); // one header line
    out = PedRows();
    while (!fin.eof()) {
        std::getline(fin, line);
        if (line.size() < 2) break;
        int id = 0, mid = 0, fid = 0, gender = 0;
        std::string name;
        std::istringstream in(line);
        in >> id >> mid >> fid >> gender >> name;
        out.id.push_back(id);
        out.mother_id.push_back(mid);
        out.father_id.push_back(fid);
        out.gender.push_back(gender);
        out.name.push_back(name);
    }
    return true;
}

int engine_method(const CommonOptions &opt) { return opt.peel_loops && opt.method == 1 ? FS_METHOD_BN_PEEL : opt.method; }

bool check_family(const PedRows &ped, bool family_bn, bool mcmc, bool peel) {
    if (peel && family_bn) {
        std::cout << "-peelLoops and -familyBN cannot be used together: -peelLoops computes the Bayesian network of the whole "
                     "ped file (at most " << kMaxPedigreeMembers << " individuals) by conditioned peeling." << std::endl;
        return false;
    }
    if (peel && ped.id.size() > kMaxPedigreeMembers) {
        std::cout << "-peelLoops takes ped files of at most " << kMaxPedigreeMembers << " individuals; this one has "
                  << ped.id.size() << ". Use -familyBN for ped files of many families." << std::endl;
        return false;
    }
    std::vector<int32_t> id(ped.id.begin(), ped.id.end()), mo(ped.mother_id.begin(), ped.mother_id.end()),
        fa(ped.father_id.begin(), ped.father_id.end()), ge(ped.gender.begin(), ped.gender.end());
    fs_pedigree fp{(int32_t)id.size(), id.data(), mo.data(), fa.data(), ge.data(), 0, nullptr};
    fs_engine *h = nullptr;
    const int host_only = -1;
    const bool cohort = id.size() > kMaxPedigreeMembers;
    const int rc = family_bn        ? fs_create_cohort_bn(&fp, nullptr, &host_only, 1, &h)
                   : cohort && mcmc ? fs_create_cohort_mcmc(&fp, nullptr, &host_only, 1, &h)
                   : cohort         ? fs_create_cohort(&fp, nullptr, &host_only, 1, &h)
                                    : fs_create(&fp, nullptr, -1, &h);
    // the conditioned program is refused (too many loop breakers, too long) at run time, so ask for it here
    const int prc = rc == FS_OK && peel ? fs_get_bn_peel_program(h, nullptr, 0, nullptr, nullptr, nullptr, 0, nullptr, nullptr) : rc;
    fs_destroy(h);
    if (prc != FS_OK && rc == FS_OK) {
        std::cout << fs_last_error() << std::endl;
        std::cout << "Cannot initiate family. Please check ped file." << std::endl;
        return false;
    }
    if (rc == FS_OK) return true;
    if (rc == FS_E_GENDER)
        std::cerr << fs_last_error() << std::endl; // family.cpp:208,213 write to cerr
    else
        std::cout << fs_last_error() << std::endl;
    std::cout << "Cannot initiate family. Please check ped file." << std::endl; // file.cpp:1922
    return false;
}

// --------------------------------------------------------------------------------------------------------
// FamSeq vcf
// --------------------------------------------------------------------------------------------------------
namespace {

int chrom_number(sv chrom) { // file.cpp:460-466
    if (chrom.substr(0, 3) == "chr") return to_int(chrom.substr(3));
    return to_int(chrom);
}

bool is_x(sv c) { return c == "X" || c == "chrX" || c == "CHRX"; }

} // namespace

bool run_vcf(const VcfOptions &opt, const PedRows &ped) {
    const double t_start = now();
    g_stats = RunStats();
    const std::string &vcf_name = opt.vcf_files[0];
    bool var_only = opt.var_only, all_line = opt.all_line;
    if (opt.diff_only) { // file.cpp:124-128
        all_line = false;
        var_only = true;
    }
    fs_params prm;
    Priors pri;
    fill_params(opt, prm, pri);

    std::thread warm([&opt] { fs_warmup(opt.device); }); // CUDA context creation overlaps reading the input
    struct Joiner {
        std::thread &t;
        ~Joiner() { if (t.joinable()) t.join(); }
    } warm_joiner{warm};
    InputFile input;
    const double t_read = now();
    if (!input.open(vcf_name)) {
        std::cout << "Cannot open " << vcf_name << std::endl;
        return false;
    }
    const sv data = input.view();
    g_stats.read_s = now() - t_read;
    FILE *fout = std::fopen(opt.output.c_str(), "wb");
    if (!fout) {
        std::cout << "Cannot open " << opt.output << std::endl;
        return false;
    }
    std::string out;
    out.reserve(1 << 24);

    // ---- pass 1: header echo with a one-line delay, tag injection (file.cpp:143-196) ---------------------
    auto fs_info_lines = [&]() {
        out += "##FS mutation rate=";
        put_number(out, prm.mrate);
        out += " \n##FS genotype frequency in pupulation (Rare): ";
        put_triplet(out, pri.n);
        out += "\n##FS genotype frequency in population (Common): ";
        put_triplet(out, pri.k);
        out += "\n##FS genotype frequency for chromosome X of male in population (Rare): ";
        put_triplet(out, pri.xn);
        out += "\n##FS genotype frequency for chromosome X of male in population (Common): ";
        put_triplet(out, pri.xk);
        out += "\n";
    };
    sv title;
    {
        bool want_info = true, want_tag = true;
        Lines in(data);
        sv line;
        while (in.next(line)) {
            if (!line.empty() && line[0] == '#') {
                if (title.size() > 2) {
                    out.append(title);
                    out += '\n';
                    if (title.substr(2, 6) == "FORMAT" && line.size() >= 2 && line.substr(2, 4) == "INFO" && want_tag) {
                        out += "##FORMAT=<ID=GPP,Number=G,Type=Integer,Description=\"Normalized, Phred-scaled for posterior "
                               "probability calculated by individual-based Method\">\n";
                        out += kFormatLines;
                        want_tag = false;
                    }
                    if (line.size() >= 2 && line.substr(2, 6) == "contig" && want_info) {
                        fs_info_lines();
                        want_info = false;
                    }
                }
                title = line;
                continue;
            }
            if (want_tag) {
                out += "##FORMAT=<ID=GPP,Number=G,Type=Integer,Description=\"Normalized, Phred-scaled for posterior "
                       "probability calbulated by Single Method\">\n";
                out += kFormatLines;
            }
            if (want_info) fs_info_lines();
            break;
        }
    }
    std::vector<sv> names;
    split(title, '\t', names);
    if (names.size() < 9) {
        std::cout << "Cannot find the #CHROM header line in " << vcf_name << std::endl;
        std::fclose(fout);
        return false;
    }
    for (int i = 0; i < 9; i++) {
        out.append(names[i]);
        out += '\t';
    }
    const ColumnMap cm = map_columns(names, 9, ped);
    for (int c : cm.matched) {
        out.append(names[9 + c]);
        out += '\t';
    }
    out += '\n';
    const int S = (int)cm.engine_cols.size();
    const int real_num_ind = cm.real_num_ind();

    // ---- optional -l location file (file.cpp:235-298) --------------------------------------------------------
    std::vector<std::vector<int>> location;
    const bool use_location = !opt.location_file.empty();
    if (use_location) {
        std::string ldata;
        if (!read_file(opt.location_file, ldata)) {
            std::cout << "Cannot open " << opt.location_file << std::endl;
            std::fclose(fout);
            return false;
        }
        location.assign(25, {});
        Lines in(ldata);
        sv line;
        std::vector<sv> f;
        while (in.next(line)) {
            if (line.size() < 2) break;
            split(line, '\t', f);
            int chr = f[0] == "X" ? 23 : f[0] == "Y" ? 24 : f[0] == "MT" ? 25 : to_int(f[0]);
            if (chr <= 0 || chr > 25 || f.size() < 2) continue;
            const int pos = to_int(f[1]);
            if (pos == 0) continue;
            location[chr - 1].push_back(pos);
        }
        for (auto &v : location) std::sort(v.begin(), v.end());
    }

    Engine eng;
    eng.family_bn = opt.family_bn && opt.method == 1;
    eng.mcmc = opt.method == 3;
    EngineStart eng_start(eng, ped, cm, prm, Engine::resolve(opt.devices, opt.device)); // joined before the first engine call (or at the end of an empty input)
    int burn = opt.num_burn_in, rep = opt.num_rep; // file.cpp:644-656
    if (burn < 0) burn = 1000 * real_num_ind;
    if (rep < 0) rep = 20000 * real_num_ind;

    // ---- pass 2: records ---------------------------------------------------------------------------------------
    // Parsing (tokenise, skip rules, PL fields) and formatting (Phred encode, "%g") are spread over host threads, each
    // owning a contiguous range of a block; see run_pipeline.
    auto parse_range = [&](Part &P, const sv *lines, size_t n, bool compact) -> bool {
        std::vector<sv> col, fmt, sub, pl;
        for (size_t li = 0; li < n; li++) {
            const sv line = lines[li];
            split(line, '\t', col);
            if (col.size() < 9 + cm.ped_row.size()) continue; // malformed record: the reference would read out of bounds
            const sv chrom = col[0], ref = col[3], alt = col[4];
            if (use_location) { // file.cpp:318-360
                int chr = (chrom == "X" || chrom == "chrX") ? 23 : (chrom == "Y" || chrom == "chrY") ? 24 : chrom == "MT" ? 25 : chrom_number(chrom);
                if (chr <= 0 || chr > 25) continue;
                const int pos = to_int(col[1]);
                if (pos == 0) continue;
                if (!std::binary_search(location[chr - 1].begin(), location[chr - 1].end(), pos)) continue;
            }
            auto echo = [&]() {
                P.lines.push_back(line);
                P.echo.push_back(1);
            };
            auto skip = [&]() {
                if (all_line) echo();
            };
            if (ref == "." || ref == "-") { skip(); continue; }
            if (ref.size() != 1 || alt.size() != 1) { skip(); continue; }
            if (var_only && (alt == "." || alt == "-")) continue;
            if (chrom == "Y" || chrom == "chrY") { skip(); continue; }
            if (chrom == "MT") { skip(); continue; }
            const int chr = chrom_number(chrom);
            if (!((0 < chr && chr < 23) || is_x(chrom))) { skip(); continue; }
            const bool known = col[2] != ".";
            const bool chrx = is_x(chrom);
            int n_miss = 0;
            for (int m : cm.matched) n_miss += col[9 + m].size() < 5;
            if (n_miss == real_num_ind) { skip(); continue; }
            split(col[8], ':', fmt);
            int ind_pl = -1;
            for (size_t i = 0; i < fmt.size(); i++)
                if (fmt[i] == "PL" || fmt[i] == "GL") ind_pl = (int)i; // the last one wins; GL is decoded like PL
            if (ind_pl < 0) { // no likelihoods: the record is echoed whatever -a says (file.cpp:541-555)
                echo();
                continue;
            }
            // likelihoods: pow(10, -|PL|/10); missing or malformed sample fields keep (1,1,1) (file.cpp:565-593, :794-831).
            // Compact: the integer itself (0 = likelihood 1), decoded on the device through the engine's libm-built table.
            size_t base;
            if (compact) {
                base = P.pl.size();
                P.pl.resize(base + (size_t)S * 3, 0);
            } else {
                base = P.lk.size();
                P.lk.resize(base + (size_t)S * 3, 1.0);
            }
            for (size_t k = 0; k < cm.matched.size(); k++) {
                const sv field = col[9 + cm.matched[k]];
                const size_t at = base + (size_t)cm.unique[k] * 3;
                if (n_miss > 0 && field.size() < 5) {
                    for (int j = 0; j < 3; j++) {
                        if (compact)
                            P.pl[at + j] = 0;
                        else
                            P.lk[at + j] = 1.0;
                    }
                    continue;
                }
                split(field, ':', sub);
                if (sub.size() != fmt.size()) continue;
                split(sub[ind_pl], ',', pl);
                for (size_t j = 0; j < 3 && j < pl.size(); j++) {
                    if (compact) {
                        if (!integer_field(pl[j], P.pl[at + j])) return false; // GL, decimals, ...: this range goes the FP64 way
                    } else {
                        P.lk[at + j] = std::pow(10.0, -std::fabs(to_double(pl[j])) / 10.0);
                    }
                }
            }
            P.flags.push_back((uint8_t)((known ? FS_FLAG_KNOWN : 0) | (chrx ? FS_FLAG_CHRX : 0)));
            P.lines.push_back(line);
            P.echo.push_back(0);
        }
        return true;
    };

    auto format_range = [&](Part &P, const BlockResults &R) {
        std::vector<sv> col, fmt;
        std::string &o = P.out;
        o.clear();
        P.warn.clear();
        P.failed = 0;
        size_t v = P.first;
        for (size_t li = 0; li < P.lines.size(); li++) {
            const sv line = P.lines[li];
            split(line, '\t', col);
            if (P.echo[li]) { // first nine columns and the matched samples, each followed by a tab
                for (int i = 0; i < 9; i++) {
                    o.append(col[i]);
                    o += '\t';
                }
                for (int m : cm.matched) {
                    o.append(col[9 + m]);
                    o += '\t';
                }
                o += '\n';
                continue;
            }
            split(col[8], ':', fmt);
            for (int i = 0; i < 8; i++) {
                o.append(col[i]);
                o += '\t';
            }
            o.append(col[8]);
            o += ":GPP:FPP:FGT\t";
            const bool failed = R.status[v] != 0;
            if (failed) { // file.cpp:607-619
                P.warn += "Warning: this variant hasn't been calculated: \n";
                P.warn.append(line);
                P.warn += '\n';
                P.failed++;
            }
            bool any_missing = false;
            for (int m : cm.matched) any_missing |= col[9 + m].size() < 5;
            for (size_t k = 0; k < cm.matched.size(); k++) {
                const sv field = col[9 + cm.matched[k]];
                if (failed) {
                    o.append(field);
                    o += ":NA:NA:NA\t";
                    continue;
                }
                if (any_missing && field.size() < 5) { // file.cpp:927-933
                    for (size_t j = 0; j < fmt.size(); j++) o += "NA:";
                } else {
                    o.append(field);
                    o += ':';
                }
                const size_t off = (v * S + cm.unique[k]) * 3;
                put_calls(o, R, off, R.gt[v * S + cm.unique[k]]);
            }
            o += '\n';
            v++;
        }
    };

    AsyncWriter writer(fout);
    writer.push(std::move(out)); // header
    out.clear();
    Lines in(data);
    // the reference stops at the first line shorter than two characters; header lines are not records
    auto accept = [](sv line) { return line.size() < 2 ? 0 : (line[0] == '#' ? 2 : 1); };
    const PipelineSetup setup{&eng, &eng_start, S, engine_method(opt), burn, rep, opt.seed, &writer};
    bool ok = run_pipeline(in, setup, accept, parse_range, format_range);
    {
        const double t0 = now();
        const bool written = writer.close();
        g_stats.drain_s = now() - t0;
        if ((std::fclose(fout) != 0 || !written) && ok) {
            std::cout << "Cannot write " << opt.output << std::endl;
            ok = false;
        }
    }
    g_stats.total_s = now() - t_start;
    emit_stats();
    return ok;
}

// --------------------------------------------------------------------------------------------------------
// FamSeq LK
// --------------------------------------------------------------------------------------------------------
bool run_lk(const LkOptions &opt, const PedRows &ped) {
    const double t_start = now();
    g_stats = RunStats();
    fs_params prm;
    Priors pri;
    fill_params(opt, prm, pri);
    std::thread warm([&opt] { fs_warmup(opt.device); }); // CUDA context creation overlaps reading the input
    struct Joiner {
        std::thread &t;
        ~Joiner() { if (t.joinable()) t.join(); }
    } warm_joiner{warm};
    InputFile input;
    if (!input.open(opt.lk_file)) {
        std::cout << "Cannot open " << opt.lk_file << std::endl;
        return false;
    }
    const sv data = input.view();
    FILE *fout = std::fopen(opt.output.c_str(), "wb");
    if (!fout) {
        std::cout << "Cannot open " << opt.output << std::endl;
        return false;
    }
    std::string out;
    out.reserve(1 << 24);
    Lines in(data);
    sv title;
    in.next(title);
    // file.cpp:1664-1669
    out += "##FORMAT=<ID=GPP,Number=G,Type=Integer,Description=\"Normalized, Phred-scaled for posterior probability "
           "calculated by individual-base Method\">\n";
    out += kFormatLines;
    out += "##FS mutation rate=";
    put_number(out, prm.mrate);
    out += " \n##FS genotype frequency in pupulation: ";
    put_triplet(out, pri.n);
    out += "\n";
    std::vector<sv> names;
    split(title, '\t', names);
    const ColumnMap cm = map_columns(names, 0, ped);
    out += "#FORMAT\t";
    for (int c : cm.matched) {
        out.append(names[c]);
        out += '\t';
    }
    out += '\n';
    const int S = (int)cm.engine_cols.size();

    Engine eng;
    eng.family_bn = opt.family_bn && opt.method == 1;
    eng.mcmc = opt.method == 3;
    EngineStart eng_start(eng, ped, cm, prm, Engine::resolve(opt.devices, opt.device)); // joined before the first engine call (or at the end of an empty input)

    // decoding and formatting are spread over host threads (see run_vcf / run_pipeline).  The LK driver calls the engine
    // with Known = false, chrType = 0 (file.cpp:1751,1768,1785): flags stay 0.  Phred-scaled rows (-lkType PS) of
    // non-negative integers go to the engine as they stand, like VCF PL fields; everything else is decoded here.
    auto parse_range = [&](Part &P, const sv *rows, size_t n, bool compact) -> bool {
        std::vector<sv> col, pl;
        if (compact && opt.lk_type != 4) return false;
        for (size_t li = 0; li < n; li++) {
            split(rows[li], '\t', col);
            if (col.size() < cm.ped_row.size()) continue; // malformed row: the reference would read out of bounds
            size_t base;
            if (compact) {
                base = P.pl.size();
                P.pl.resize(base + (size_t)S * 3, 0);
            } else {
                base = P.lk.size();
                P.lk.resize(base + (size_t)S * 3, 1.0);
            }
            for (size_t k = 0; k < cm.matched.size(); k++) {
                const size_t at = base + (size_t)cm.unique[k] * 3;
                split(col[cm.matched[k]], ',', pl);
                for (size_t j = 0; j < 3 && j < pl.size(); j++) {
                    if (compact) { // pow(10, -x/10) of a non-negative integer x: the table entry x
                        if (pl[j].empty() || pl[j][0] == '-' || !integer_field(pl[j], P.pl[at + j])) return false;
                        continue;
                    }
                    const double x = to_double(pl[j]);
                    switch (opt.lk_type) { // file.cpp:1719-1738
                    case 2: P.lk[at + j] = std::pow(10.0, x); break;
                    case 3: P.lk[at + j] = std::exp(x); break;
                    case 4: P.lk[at + j] = std::pow(10.0, -x / 10.0); break;
                    default: P.lk[at + j] = x; break;
                    }
                }
            }
            P.flags.push_back(0);
            P.lines.push_back(rows[li]);
        }
        return true;
    };
    auto format_range = [&](Part &P, const BlockResults &R) {
        std::vector<sv> col;
        std::string &o = P.out;
        o.clear();
        P.warn.clear();
        P.failed = 0;
        size_t v = P.first;
        for (const sv row : P.lines) {
            split(row, '\t', col);
            o += "LK:GPP:FPP:FGT\t";
            const bool failed = R.status[v] != 0;
            if (failed) {
                P.warn += "Warning: this variant hasn't been calculated: \n";
                P.warn.append(row);
                P.warn += '\n';
                P.failed++;
            }
            for (size_t k = 0; k < cm.matched.size(); k++) {
                o.append(col[cm.matched[k]]);
                if (failed) {
                    o += ":NA:NA:NA\t";
                    continue;
                }
                o += ':';
                const size_t off = (v * S + cm.unique[k]) * 3;
                put_calls(o, R, off, R.gt[v * S + cm.unique[k]]);
            }
            o += '\n';
            v++;
        }
    };

    AsyncWriter writer(fout);
    writer.push(std::move(out)); // header
    out.clear();
    auto accept = [](sv line) { return line.size() < 2 ? 0 : 1; };
    const PipelineSetup setup{&eng, &eng_start, S, engine_method(opt), opt.num_burn_in, opt.num_rep, opt.seed, &writer};
    bool ok = run_pipeline(in, setup, accept, parse_range, format_range);
    {
        const double t0 = now();
        const bool written = writer.close();
        g_stats.drain_s = now() - t0;
        if ((std::fclose(fout) != 0 || !written) && ok) {
            std::cout << "Cannot write " << opt.output << std::endl;
            ok = false;
        }
    }
    g_stats.total_s = now() - t_start;
    emit_stats();
    return ok;
}

} // namespace famseq_cli
