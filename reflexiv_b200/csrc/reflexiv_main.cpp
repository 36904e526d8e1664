// reflexiv_main.cpp -- `reflexiv` command-line driver on top of libreflexiv_cuda (C ABI only).
//
// Mirrors, for the `run` and `counter` commands:
//   bin/reflexiv:209-267                     command word, `--x [v]` (Spark) vs `-x [v]` (Reflexiv) option split
//   main/Main.java:57-79, MainOfCounter.java:58-80
//   util/Parameter.java:311-611, util/ParameterOfCounter.java:205-390   option names, defaults, exit code 0 on errors
//   pipeline/ReflexivDataFrameCounter.java:222-233   <out>/Count_<k>/part-*.csv[.gz] + _SUCCESS
//   pipeline/ReflexivDSMain.java:331-354, 706-710    <out>/part-00000 (or <out>/Assemble_<k>/ with -kmerc)
// The reference's driver is Java; a JDK is not available in this image, so the host side above the C ABI is C++
// (INTEGRATION.md shows the JNI / Panama binding a Java driver would use instead).
#include <dirent.h>
#include <fcntl.h>
#include <glob.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <time.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/reflexiv_cuda.h"

static void info(const char* msg) {  // util/InfoDumper.java: "Reflexiv HH:mm:ss msg"
    time_t t = time(nullptr);
    struct tm tmv;
    localtime_r(&t, &tmv);
    printf("Reflexiv %02d:%02d:%02d %s\n", tmv.tm_hour, tmv.tm_min, tmv.tm_sec, msg);
    fflush(stdout);
}

static const char* HELP =
    "usage: reflexiv <run|counter|sort> [--spark-options ignored] -fastq <glob> -outfile <dir> [-kmer 31] [-cover 2]\n"
    "       [-maxcov 10000000] [-error 8] [-clipf N] [-clipe N] [-mincontig 500] [-miniter 15] [-maxiter 150]\n"
    "       [-partition N] [-partitionredu 200] [-kmerc <Count_k csv glob>] [-infmt fmt] [-bubble] [-gzip] [-cache]\n"
    "       [-stitch]  (with -kmerc AND -fastq: low-coverage reads bridge contig ends, ReflexivDSMain.java:585-672)\n"
    "       sort: -kmerc <Count_k csv glob> -outfile <dir> -kmer k [-maxcov N] [-error 8] [-klist 23,31,...] [-accurate]\n"
    "             writes <dir>/Count_<k>_sorted (rows KMER,1|left|right)\n";

struct Opt { bool has_arg; };
static std::map<std::string, Opt> run_options() {
    std::map<std::string, Opt> m;
    for (const char* n : {"fastq", "paired", "single", "inter", "fasta", "infmt", "reads", "contig", "kmerc", "outfile", "kmer", "klist",
                          "overlap", "miniter", "maxiter", "clipf", "clipe", "cover", "maxcov", "error", "minlength", "mincontig",
                          "partition", "partitionredu", "sbin", "mode"})
        m[n] = Opt{true};
    for (const char* n : {"gzip", "bubble", "stitch", "accurate", "cache", "version", "h", "help"}) m[n] = Opt{false};
    return m;
}
static std::map<std::string, Opt> counter_options() {
    std::map<std::string, Opt> m;
    for (const char* n : {"fastq", "fasta", "infmt", "reads", "outfile", "kmer", "overlap", "clipf", "clipe", "cover", "maxcov", "minlength",
                          "partition", "partitionredu"})
        m[n] = Opt{true};
    for (const char* n : {"gzip", "cache", "version", "h", "help"}) m[n] = Opt{false};
    return m;
}

static int bad_params(const std::string& why) {  // Parameter.java:601-611: message, stack trace, exit code 0
    info("Parameter settings incorrect.");
    fprintf(stderr, "%s\n", why.c_str());
    return 0;
}

// ---- input files (SURVEY 8f-3) -----------------------------------------------------------------------------------
// spark.read().text(glob) reads every matching file as its own set of partitions, in parallel
// (ReflexivDataFrameCounter.java:161-188, ReflexivDSMain.java:188).  Here: a few host threads inflate .gz files ahead
// of the consumer (zlib), plain files are mapped, and the consumer takes the files in path order -- one rfx_push_fastq
// per file, so the host never holds more than the look-ahead window and the GPU parses file i while i+1.. inflate.
static bool ends_with(const std::string& s, const char* suf) {
    const size_t n = strlen(suf);
    return s.size() > n && s.compare(s.size() - n, n, suf) == 0;
}

struct InputFile {
    std::string path;
    std::string data;            // inflated text, or a plain file that had to be copied
    const char* map = nullptr;   // plain file mapped read-only
    size_t map_len = 0;
    bool ok = false, done = false;
    const char* bytes() const { return map ? map : data.data(); }
    size_t size() const { return map ? map_len : data.size(); }
    void release() {
        if (map) munmap(const_cast<char*>(map), map_len);
        map = nullptr; map_len = 0;
        std::string().swap(data);
    }
};

// Hadoop's LineRecordReader (the reference's text source) ends a line at "\n", "\r\n" and at a lone "\r".  The library
// takes "\n" and "\r\n"; a file with classic-Mac line ends would silently parse as one long line, so it is refused.
// Looked for in the first 64 KB (a line-end convention holds for a whole file).
static bool has_lone_cr(const char* d, size_t n) {
    if (n > 65536) n = 65536;
    for (size_t i = 0; i + 1 < n; i++)
        if (d[i] == '\r' && d[i + 1] != '\n') return true;
    return false;
}
static bool load_file_raw(InputFile& f);
static bool load_file(InputFile& f) {
    if (!load_file_raw(f)) return false;
    const char* d = f.map ? f.map : f.data.data();
    const size_t n = f.map ? f.map_len : f.data.size();
    if (n && has_lone_cr(d, n)) {
        fprintf(stderr, "%s: lone '\\r' line ends (classic Mac text) are not supported; convert with tr '\\r' '\\n'\n", f.path.c_str());
        return false;
    }
    return true;
}
static bool load_file_raw(InputFile& f) {
    if (ends_with(f.path, ".4mc")) {
        fprintf(stderr, "%s: 4mc input needs hadoop-4mc; decompress first or use gzip / plain text\n", f.path.c_str());
        return false;
    }
    if (!ends_with(f.path, ".gz")) {
        const int fd = open(f.path.c_str(), O_RDONLY);
        if (fd < 0) return false;
        struct stat st;
        if (fstat(fd, &st) != 0) { close(fd); return false; }
        if (st.st_size == 0) { close(fd); return true; }
        void* m = mmap(nullptr, (size_t)st.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
        close(fd);
        if (m != MAP_FAILED) {
            if (static_cast<const char*>(m)[st.st_size - 1] == '\n') {
                madvise(m, (size_t)st.st_size, MADV_SEQUENTIAL);
                f.map = static_cast<const char*>(m); f.map_len = (size_t)st.st_size;
                return true;
            }
            f.data.assign(static_cast<const char*>(m), (size_t)st.st_size);  // no final newline: a copy that gets one
            munmap(m, (size_t)st.st_size);
            f.data.push_back('\n');
            return true;
        }
    }
    gzFile g = gzopen(f.path.c_str(), "rb");  // zlib reads plain files transparently (mmap failed: pipes, odd file systems)
    if (!g) return false;
    gzbuffer(g, 1u << 20);
    std::vector<char> buf(4u << 20);
    int n;
    while ((n = gzread(g, buf.data(), (unsigned)buf.size())) > 0) f.data.append(buf.data(), (size_t)n);
    int zerr = Z_OK;
    gzerror(g, &zerr);
    const bool ok = gzclose(g) == Z_OK && n == 0 && (zerr == Z_OK || zerr == Z_STREAM_END);  // Z_BUF_ERROR: the stream ends early
    if (!f.data.empty() && f.data.back() != '\n') f.data.push_back('\n');
    return ok;
}

static bool expand_inputs(const std::string& pattern, std::vector<std::string>& files) {
    glob_t g;
    std::vector<std::string> paths;
    if (glob(pattern.c_str(), 0, nullptr, &g) == 0)
        for (size_t i = 0; i < g.gl_pathc; i++) paths.push_back(g.gl_pathv[i]);
    globfree(&g);
    if (paths.empty()) { fprintf(stderr, "Input path does not exist: %s\n", pattern.c_str()); return false; }
    std::sort(paths.begin(), paths.end());
    for (const std::string& p : paths) {
        struct stat st;
        if (stat(p.c_str(), &st) == 0 && S_ISDIR(st.st_mode)) {
            std::vector<std::string> inner;
            if (DIR* d = opendir(p.c_str())) {
                while (dirent* e = readdir(d))
                    if (e->d_name[0] != '_' && e->d_name[0] != '.') inner.push_back(p + "/" + e->d_name);
                closedir(d);
            }
            std::sort(inner.begin(), inner.end());
            files.insert(files.end(), inner.begin(), inner.end());
        } else files.push_back(p);
    }
    return true;
}

// Hands the files matching `pattern` to `consume(bytes, len)` in path order; up to `ahead` files are being read or
// wait decoded at any time.  Returns false on the first file that cannot be read or that `consume` rejects.
static bool stream_inputs(const std::string& pattern, const std::function<bool(const char*, size_t)>& consume) {
    std::vector<std::string> paths;
    if (!expand_inputs(pattern, paths)) return false;
    std::vector<InputFile> files(paths.size());
    for (size_t i = 0; i < paths.size(); i++) files[i].path = paths[i];
    unsigned hw = std::thread::hardware_concurrency();
    size_t ahead = hw ? hw : 4;
    if (const char* e = getenv("REFLEXIV_READERS")) ahead = (size_t)std::max(1, atoi(e));
    ahead = std::min<size_t>(std::min<size_t>(ahead, 16), files.size());
    std::mutex mu;
    std::condition_variable cv;
    size_t next = 0, consumed = 0;
    bool stop = false;
    auto worker = [&]() {
        for (;;) {
            size_t i;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return stop || next >= files.size() || next < consumed + ahead; });
                if (stop || next >= files.size()) return;
                i = next++;
            }
            const bool ok = load_file(files[i]);
            {
                std::lock_guard<std::mutex> lk(mu);
                files[i].ok = ok; files[i].done = true;
            }
            cv.notify_all();
        }
    };
    std::vector<std::thread> pool;
    for (size_t t = 0; t < ahead; t++) pool.emplace_back(worker);
    bool ok = true;
    for (size_t i = 0; i < files.size() && ok; i++) {
        {
            std::unique_lock<std::mutex> lk(mu);
            cv.wait(lk, [&] { return files[i].done; });
        }
        if (!files[i].ok) { fprintf(stderr, "reflexiv: cannot read %s\n", files[i].path.c_str()); ok = false; }
        else if (files[i].size() && !consume(files[i].bytes(), files[i].size())) ok = false;
        files[i].release();
        {
            std::lock_guard<std::mutex> lk(mu);
            consumed = i + 1;
        }
        cv.notify_all();
    }
    {
        std::lock_guard<std::mutex> lk(mu);
        stop = true;
    }
    cv.notify_all();
    for (std::thread& t : pool) t.join();
    for (InputFile& f : files) f.release();
    return ok;
}

static bool write_out(const std::string& path, const char* data, size_t n, bool gz) {
    if (gz) {
        gzFile f = gzopen((path + ".gz").c_str(), "wb");
        if (!f) return false;
        size_t off = 0;
        while (off < n) { int w = gzwrite(f, data + off, (unsigned)std::min<size_t>(n - off, 1u << 30)); if (w <= 0) { gzclose(f); return false; } off += (size_t)w; }
        return gzclose(f) == Z_OK;
    }
    FILE* f = fopen(path.c_str(), "wb");
    if (!f) return false;
    bool ok = fwrite(data, 1, n, f) == n;
    return fclose(f) == 0 && ok;
}

static int fail(rfx_ctx* c, const char* what) {
    fprintf(stderr, "reflexiv: %s: %s\n", what, rfx_last_error(c));
    if (c) rfx_destroy(c);
    return 1;
}

// One worker's share of the rows: [data + from, data + to), both on line starts.  No allocation per row.
static bool parse_count_rows(const char* data, size_t from, size_t to, int k, int minc, int maxc, std::vector<uint64_t>& keys, std::vector<uint32_t>& counts) {
    const int words = k <= 31 ? 1 : k / 32 + 1, res = k % 32;
    size_t pos = from;
    while (pos < to) {
        const char* nl = static_cast<const char*>(memchr(data + pos, '\n', to - pos));
        size_t end = nl ? (size_t)(nl - data) : to;
        size_t b = pos, e = end;
        pos = end + 1;
        if (e > b && data[e - 1] == '\r') e--;
        if (b == e) continue;
        if (data[b] == '(') b++;
        if (e > b && data[e - 1] == ')') e--;
        const char* cm = static_cast<const char*>(memchr(data + b, ',', e - b));
        if (!cm || (cm - (data + b)) < k) return false;
        const char* num = cm + 1;
        const size_t nd = (size_t)(data + e - num);
        long cover = 0;
        if (nd >= 10) cover = 1000000000L;  // ReflexivDSMain.java:3895-3910
        else for (size_t i = 0; i < nd; i++) { if (num[i] < '0' || num[i] > '9') break; cover = cover * 10 + (num[i] - '0'); }
        if (cover < minc || cover > maxc) continue;  // ReflexivDSMain.java:405-412
        unsigned __int128 v = 0;
        for (int i = 0; i < k; i++) { const char ch = data[b + i]; v = (v << 2) | (ch == 'A' ? 0 : ch == 'C' ? 1 : ch == 'G' ? 2 : 3); }
        if (words == 1) keys.push_back((uint64_t)v);
        else { keys.push_back((uint64_t)(v >> (2 * res))); keys.push_back((uint64_t)v & ((res ? ((uint64_t)1 << (2 * res)) : 1) - 1)); }
        counts.push_back((uint32_t)cover);
    }
    return true;
}

// KmerBinarizer input: `KMER,count` or legacy `(KMER,count)`, ReflexivDSMain.java:3872-3948.  Large tables are cut at line
// starts into one piece per host thread (Spark parses every partition of the CSV on its own core); row order is kept.
// The -kmerc paths parse on the device (rfx_load_counts_csv); this host parser is the reference the tests compare that against.
[[maybe_unused]] static bool parse_counts(const char* data, size_t n, int k, int minc, int maxc, std::vector<uint64_t>& keys, std::vector<uint32_t>& counts) {
    unsigned T = std::thread::hardware_concurrency();
    if (const char* e = getenv("REFLEXIV_READERS")) T = (unsigned)std::max(1, atoi(e));
    if (T > 32) T = 32;
    if (T <= 1 || n < (4u << 20)) return parse_count_rows(data, 0, n, k, minc, maxc, keys, counts);
    std::vector<size_t> cut(T + 1, n);
    cut[0] = 0;
    for (unsigned t = 1; t < T; t++) {
        size_t c = std::max(cut[t - 1], n / T * t);
        const char* nl = c < n ? static_cast<const char*>(memchr(data + c, '\n', n - c)) : nullptr;
        cut[t] = nl ? (size_t)(nl - data) + 1 : n;
    }
    std::vector<std::vector<uint64_t>> pk(T);
    std::vector<std::vector<uint32_t>> pc(T);
    std::vector<char> ok(T, 1);
    std::vector<std::thread> pool;
    for (unsigned t = 0; t < T; t++)
        pool.emplace_back([&, t] { ok[t] = parse_count_rows(data, cut[t], cut[t + 1], k, minc, maxc, pk[t], pc[t]) ? 1 : 0; });
    for (std::thread& th : pool) th.join();
    for (unsigned t = 0; t < T; t++) {
        if (!ok[t]) return false;
        keys.insert(keys.end(), pk[t].begin(), pk[t].end());
        counts.insert(counts.end(), pc[t].begin(), pc[t].end());
    }
    return true;
}

// ---- outputs (one part file per rank, as Spark writes one per partition) -----------------------------------------------
static bool write_csv_part(rfx_ctx* c, bool sorter, const std::string& target, int rank, bool gz) {
    uint64_t nbytes = 0;
    auto csv_fn = sorter ? rfx_sorted_csv : rfx_counts_csv;
    if (csv_fn(c, nullptr, 0, &nbytes) != RFX_OK) return false;
    std::vector<char> csv(nbytes ? nbytes : 1);
    if (nbytes && csv_fn(c, csv.data(), nbytes, &nbytes) != RFX_OK) return false;
    char name[128];
    snprintf(name, sizeof(name), "/part-%05d-%08lx-%04x-%04x-%04x-%012lx-c000.csv", rank, (unsigned long)time(nullptr) & 0xffffffffUL, rand() & 0xffff,
             rand() & 0xffff, rand() & 0xffff, ((unsigned long)rand() << 16 ^ (unsigned long)rand()) & 0xffffffffffffUL);
    if (!write_out(target + name, csv.data(), nbytes, gz)) { fprintf(stderr, "reflexiv: cannot write %s\n", target.c_str()); return false; }
    return true;
}
// DSKmerToContig + changeLine + TagRowContigID, ReflexivDSMain.java:743-794, 717-725; ids continue from id_base
static bool write_contig_part(rfx_ctx* c, const std::string& target, int rank, uint64_t id_base, bool gz, uint64_t* n_out) {
    uint64_t n = 0, total = 0;
    if (rfx_contigs_size(c, &n, &total) != RFX_OK) return false;
    std::vector<char> bases(total ? total : 1);
    std::vector<uint64_t> offs(n + 1);
    std::vector<int32_t> left(n ? n : 1), right(n ? n : 1);
    if (rfx_contigs_copy(c, bases.data(), offs.data(), left.data(), right.data()) != RFX_OK) return false;
    std::string out;
    out.reserve(total + total / 100 + 64 * n + 16);
    for (uint64_t i = 0; i < n; i++) {
        const uint64_t len = offs[i + 1] - offs[i];
        char head[96];
        snprintf(head, sizeof(head), ">Contig-%llu-(%d,%d)-%llu\n", (unsigned long long)len, left[i], right[i], (unsigned long long)(id_base + i));
        out += head;
        for (uint64_t j = 0; j < len; j += 100) {
            out.append(bases.data() + offs[i] + j, (size_t)std::min<uint64_t>(100, len - j));
            out.push_back('\n');
        }
    }
    char name[32];
    snprintf(name, sizeof(name), "/part-%05d", rank);
    if (!write_out(target + name, out.data(), out.size(), gz)) { fprintf(stderr, "reflexiv: cannot write %s\n", target.c_str()); return false; }
    if (n_out) *n_out = n;
    return true;
}
static void clear_dir(const std::string& target) {  // SaveMode.Overwrite
    if (DIR* d = opendir(target.c_str())) {
        while (dirent* e = readdir(d))
            if (e->d_name[0] != '.' || strlen(e->d_name) > 2) remove((target + "/" + e->d_name).c_str());
        closedir(d);
    }
}

// ---- --gpus N: one context per rank, ranks are host threads; the library's sharded calls do the exchange over peer memory ----
// Where a 4-line FASTQ text may be cut: in front of a line that starts with '@' whose second-next line starts with '+'
// (a quality line may start with '@' too, but then the second-next line is a sequence).
static size_t record_start_near(const char* d, size_t n, size_t pos) {
    if (pos >= n) return n;
    const size_t limit = std::min(n, pos + ((size_t)4 << 20));
    const char* nl = static_cast<const char*>(memchr(d + pos, '\n', n - pos));
    while (nl && (size_t)(nl - d) + 1 < limit) {
        const size_t l0 = (size_t)(nl - d) + 1;
        const char* n1 = static_cast<const char*>(memchr(d + l0, '\n', n - l0));
        const char* n2 = n1 ? static_cast<const char*>(memchr(n1 + 1, '\n', n - (size_t)(n1 + 1 - d))) : nullptr;
        if (d[l0] == '@' && n2 && (size_t)(n1 + 1 - d) < n && n1[1] != '+' && n2[1] == '+') return l0;
        nl = n1;
    }
    return n;  // no safe cut nearby: the rest stays with the previous rank
}
struct Rank {
    rfx_ctx* c = nullptr;
    std::vector<std::pair<const char*, size_t>> parts;
    int rc = RFX_OK;
    const char* what = "";
};
// Contexts for n_gpus ranks (fewer devices than ranks: ranks share devices, how a one-GPU box runs this path), each with its
// peer-visible arena, connected to each other.  On failure everything is destroyed and false returned.
static void destroy_ranks(std::vector<Rank>& R) {
    for (auto& k : R) if (k.c) rfx_destroy(k.c);
    R.clear();
}
static bool open_ranks(int n_gpus, rfx_params p, std::vector<Rank>& R) {
    int32_t n_dev = 0;
    if (rfx_device_count(&n_dev) != RFX_OK || n_dev < 1) { fprintf(stderr, "reflexiv: no CUDA device\n"); return false; }
    R.assign(n_gpus, Rank());
    const int dev0 = p.device;
    for (int r = 0; r < n_gpus; r++) {
        p.device = (dev0 + r) % n_dev;
        if (rfx_create(&R[r].c, &p) != RFX_OK) { fprintf(stderr, "reflexiv: rfx_create (rank %d): %s\n", r, rfx_last_error(nullptr)); destroy_ranks(R); return false; }
    }
    uint64_t arena = getenv("REFLEXIV_ARENA_MB") ? (uint64_t)atoll(getenv("REFLEXIV_ARENA_MB")) << 20 : 0;
    if (!arena && n_dev < n_gpus) { fprintf(stderr, "reflexiv: %d ranks on %d device(s): set REFLEXIV_ARENA_MB (device memory per rank)\n", n_gpus, n_dev); destroy_ranks(R); return false; }
    std::vector<unsigned char> blobs((size_t)n_gpus * RFX_SHARD_HANDLE_BYTES);
    for (int r = 0; r < n_gpus; r++) {
        if (rfx_shard_init(R[r].c, r, n_gpus, arena) != RFX_OK || rfx_shard_export(R[r].c, blobs.data() + (size_t)r * RFX_SHARD_HANDLE_BYTES) != RFX_OK) {
            fprintf(stderr, "reflexiv: rfx_shard_init (rank %d): %s\n", r, rfx_last_error(R[r].c)); destroy_ranks(R); return false;
        }
    }
    for (int r = 0; r < n_gpus; r++)
        if (rfx_shard_connect(R[r].c, blobs.data(), n_gpus) != RFX_OK) { fprintf(stderr, "reflexiv: rfx_shard_connect (rank %d): %s\n", r, rfx_last_error(R[r].c)); destroy_ranks(R); return false; }
    return true;
}
// the collective stages, one thread per rank; false (every failure reported) if a rank failed
static bool run_ranks(std::vector<Rank>& R, const std::function<void(Rank&, int)>& body) {
    std::vector<std::thread> th;
    for (int r = 0; r < (int)R.size(); r++) th.emplace_back([&, r] { body(R[r], r); });
    for (auto& t : th) t.join();
    bool ok = true;
    for (int r = 0; r < (int)R.size(); r++)
        if (R[r].rc != RFX_OK) { fprintf(stderr, "reflexiv: %s (rank %d): %s\n", R[r].what, r, rfx_last_error(R[r].c)); ok = false; }
    return ok;
}
// what a rank writes: its contigs (Assemble_<k> or the run's output directory), its Count_<k> rows or its Count_<k>_sorted rows
enum class Output { contigs, counts, sorted };
// one part file per rank (contig ids continue across ranks) + _SUCCESS
static int write_ranks(std::vector<Rank>& R, Output what, const std::string& outdir, const std::string& target, bool gz) {
    const int n_gpus = (int)R.size();
    mkdir(outdir.c_str(), 0755);
    mkdir(target.c_str(), 0755);
    if (what != Output::contigs) clear_dir(target);
    uint64_t id_base = 0, n_sorted = 0;
    rfx_stats_t tot;
    memset(&tot, 0, sizeof(tot));
    for (int r = 0; r < n_gpus; r++) {
        uint64_t n = 0;
        const bool ok = what == Output::contigs ? write_contig_part(R[r].c, target, r, id_base, gz, &n)
                                                : write_csv_part(R[r].c, what == Output::sorted, target, r, gz) && (what != Output::sorted || rfx_sorted_size(R[r].c, &n) == RFX_OK);
        if (!ok) { fprintf(stderr, "reflexiv: writing the output of rank %d failed: %s\n", r, rfx_last_error(R[r].c)); destroy_ranks(R); return 1; }
        if (what == Output::contigs) id_base += n;
        else n_sorted += n;
        rfx_stats_t s;
        rfx_stats(R[r].c, &s);
        tot.n_reads += s.n_reads; tot.n_instances += s.n_instances; tot.n_distinct += s.n_distinct; tot.n_rows += s.n_rows; tot.n_contigs += s.n_contigs;
    }
    FILE* okf = fopen((target + "/_SUCCESS").c_str(), "wb");
    if (okf) fclose(okf);
    rfx_shard_stats_t sh;
    rfx_shard_stats(R[0].c, &sh);
    char msg[512];
    snprintf(msg, sizeof(msg), "done on %d ranks: %llu reads, %llu k-mers, %llu distinct, %llu rows, %llu %s; rank 0: %llu neighbour probes answered by a peer, %.2f ms in barriers",
             n_gpus, (unsigned long long)tot.n_reads, (unsigned long long)tot.n_instances, (unsigned long long)tot.n_distinct, (unsigned long long)tot.n_rows,
             (unsigned long long)(what == Output::sorted ? n_sorted : tot.n_contigs), what == Output::sorted ? "sorted rows" : "contigs", (unsigned long long)sh.n_remote_probes, sh.ms_comm);
    info(msg);
    destroy_ranks(R);
    return 0;
}
static int run_sharded(int n_gpus, rfx_params p, bool counter, const std::string& pattern, const std::string& outdir, const std::string& target, bool gz) {
    std::vector<Rank> R;
    if (!open_ranks(n_gpus, p, R)) return 1;
    // input: every file is cut into n_gpus runs of whole records (`run`) or whole lines (`counter`); rank r takes the r-th run of every file
    bool push_ok = true;
    const bool read_ok = stream_inputs(pattern, [&](const char* data, size_t n) {
        std::vector<size_t> cut(n_gpus + 1, n);
        cut[0] = 0;
        for (int r = 1; r < n_gpus; r++) {
            size_t want = n / n_gpus * r;
            if (want < cut[r - 1]) want = cut[r - 1];
            if (counter) {
                const char* nl = want < n ? static_cast<const char*>(memchr(data + want, '\n', n - want)) : nullptr;
                cut[r] = nl ? (size_t)(nl - data) + 1 : n;
            } else cut[r] = record_start_near(data, n, want);
        }
        // the pushes of one file run concurrently, one thread per rank, before the reader hands out the next file
        std::vector<std::thread> th;
        for (int r = 0; r < n_gpus; r++)
            th.emplace_back([&, r] {
                if (cut[r + 1] > cut[r] && R[r].rc == RFX_OK) {
                    R[r].rc = rfx_push_fastq(R[r].c, reinterpret_cast<const uint8_t*>(data + cut[r]), cut[r + 1] - cut[r]);
                    R[r].what = "rfx_push_fastq";
                }
            });
        for (auto& t : th) t.join();
        for (auto& k : R) push_ok = push_ok && k.rc == RFX_OK;
        return push_ok;
    });
    if (!read_ok || !push_ok) {
        for (int r = 0; r < n_gpus; r++) if (R[r].rc != RFX_OK) fprintf(stderr, "reflexiv: %s (rank %d): %s\n", R[r].what, r, rfx_last_error(R[r].c));
        destroy_ranks(R);
        return 1;
    }
    const bool ok = run_ranks(R, [&](Rank& k, int) {
        k.what = "rfx_count_sharded";
        if ((k.rc = rfx_count_sharded(k.c)) != RFX_OK) return;
        if (!counter) { k.what = "rfx_assemble_sharded"; k.rc = rfx_assemble_sharded(k.c); }
    });
    if (!ok) { destroy_ranks(R); return 1; }
    return write_ranks(R, counter ? Output::counts : Output::contigs, outdir, target, counter && gz);  // -gzip applies to contigs from a count table only
}
// The arguments of the Count_<k>_sorted stage (`sort`): E is rfx_params.min_error_coverage
struct SortStage {
    double min_repeat_fold;
    int32_t max_kmer_size;
    bool k_listed;  // k is in -klist: otherwise no row takes part (ReflexivDSKmerLeftAndRightSorting.java:1695)
};
// `run -kmerc <glob> --gpus N` / `sort -kmerc <glob> --gpus N`: every file is cut into N runs of whole lines and rank r parses its run
// on its own device (rfx_load_counts_csv, appended to an empty table), rfx_shard_table sends every row to the owner of its minimiser
// bin, then the sharded assembly or (sort != nullptr) the sharded Count_<k>_sorted stage.  Rows kept: min_count..max_count.
static int run_kmerc_sharded(int n_gpus, rfx_params p, const SortStage* sort, int64_t min_count, int64_t max_count, const std::string& pattern,
                             const std::string& outdir, const std::string& target, bool gz) {
    std::vector<Rank> R;
    if (!open_ranks(n_gpus, p, R)) return 1;
    for (Rank& k : R) {
        k.what = "rfx_load_counts_csv";
        k.rc = rfx_load_counts_csv(k.c, nullptr, 0, min_count, max_count, 0);
    }
    bool load_ok = true;
    for (Rank& k : R) load_ok = load_ok && k.rc == RFX_OK;
    const bool read_ok = load_ok && stream_inputs(pattern, [&](const char* data, size_t n) {
        std::vector<size_t> cut(n_gpus + 1, n);
        cut[0] = 0;
        for (int r = 1; r < n_gpus; r++) {
            const size_t want = std::max(cut[r - 1], n / n_gpus * r);
            const char* nl = want < n ? static_cast<const char*>(memchr(data + want, '\n', n - want)) : nullptr;
            cut[r] = nl ? (size_t)(nl - data) + 1 : n;
        }
        std::vector<std::thread> th;
        for (int r = 0; r < n_gpus; r++)
            th.emplace_back([&, r] {
                if (cut[r + 1] > cut[r] && R[r].rc == RFX_OK) R[r].rc = rfx_load_counts_csv(R[r].c, reinterpret_cast<const uint8_t*>(data + cut[r]), cut[r + 1] - cut[r], min_count, max_count, 1);
            });
        for (auto& t : th) t.join();
        for (auto& k : R) load_ok = load_ok && k.rc == RFX_OK;
        return load_ok;
    });
    if (!read_ok || !load_ok) {
        for (int r = 0; r < n_gpus; r++) if (R[r].rc != RFX_OK) fprintf(stderr, "reflexiv: %s (rank %d): %s\n", R[r].what, r, rfx_last_error(R[r].c));
        destroy_ranks(R);
        return 1;
    }
    const bool ok = run_ranks(R, [&](Rank& k, int) {
        k.what = "rfx_shard_table";
        if ((k.rc = rfx_shard_table(k.c)) != RFX_OK) return;
        if (sort) {
            k.what = "rfx_sort_kmers_sharded";
            k.rc = rfx_sort_kmers_sharded(k.c, p.min_error_coverage, sort->min_repeat_fold, sort->max_kmer_size);
        } else {
            k.what = "rfx_assemble_sharded";
            k.rc = rfx_assemble_sharded(k.c);
        }
    });
    if (!ok) { destroy_ranks(R); return 1; }
    return write_ranks(R, sort ? Output::sorted : Output::contigs, outdir, target, gz);
}

int main(int argc, char** argv) {
    if (argc < 2) { fputs(HELP, stdout); return 1; }
    const std::string cmd = argv[1];
    // `sort` is not a command of bin/reflexiv: it runs the one stage of the multi-k workflows that is on the GPU path
    // (Pipelines.reflexivLeftAndRightSortingPipe, Count_<k> -> Count_<k>_sorted) on its own, with the `run` option names
    if (cmd != "run" && cmd != "counter" && cmd != "sort") {
        fprintf(stderr, "reflexiv: command '%s' is outside the GPU path (supported: run, counter, sort)\n", cmd.c_str());
        fputs(HELP, stdout);
        return 1;
    }
    const bool counter = cmd == "counter", sorter = cmd == "sort";
    // bin/reflexiv:209-238: `--x [value]` belongs to spark-submit, `-x [value]` to Reflexiv
    // ... of which this driver reads one: `--gpus N` (what `--master local[N]` is to the reference; also REFLEXIV_GPUS)
    std::vector<std::string> own;
    int n_gpus = getenv("REFLEXIV_GPUS") ? atoi(getenv("REFLEXIV_GPUS")) : 1;
    for (int i = 2; i < argc; i++) {
        std::string a = argv[i];
        const bool next_is_value = i + 1 < argc && argv[i + 1][0] != '-';
        if (a.rfind("--", 0) == 0) {
            if (a == "--gpus" && next_is_value) n_gpus = atoi(argv[i + 1]);
            if (next_is_value) i++;
            continue;
        }
        if (a[0] == '-') { own.push_back(a); if (next_is_value) own.push_back(argv[++i]); }
    }
    info(counter ? "Reflexiv counter initiating ... " : sorter ? "Reflexiv k-mer sorting initiating ... " : "Reflexiv main initiating ... ");
    info("interpreting parameters.");
    const auto table = counter ? counter_options() : run_options();
    std::map<std::string, std::string> v;
    for (size_t i = 0; i < own.size(); i++) {
        std::string name = own[i].substr(own[i].find_first_not_of('-'));
        auto it = table.find(name);
        if (it == table.end()) return bad_params("Unrecognized option: " + own[i]);
        if (it->second.has_arg) {
            if (i + 1 >= own.size()) return bad_params("Missing argument for option: " + name);
            v[name] = own[++i];
        } else v[name] = "1";
    }
    if (v.count("help") || v.count("h")) { fputs(HELP, stdout); return 0; }
    if (v.count("version")) return 0;

    rfx_params p;
    rfx_params_default(&p);
    std::string err;
    auto geti = [&](const char* n, int32_t& dst, long lo, long hi) {
        if (!v.count(n)) return true;
        char* e = nullptr;
        long x = strtol(v[n].c_str(), &e, 0);
        if (!e || *e) { err = std::string("For input string: \"") + v[n] + "\""; return false; }
        if (x < lo || x > hi) { err = std::string("Parameter ") + n + " out of range"; return false; }
        dst = (int32_t)x;
        return true;
    };
    if (!geti("kmer", p.kmer_size, -2147483647L, 2147483647L) || !geti("partition", p.partitions, 0, 2147483647L) ||
        !geti("partitionredu", p.shuffle_partitions, 0, 2147483647L) || !geti("miniter", p.min_iter, 0, 2147483647L) ||
        !geti("maxiter", p.max_iter, -2147483647L, 100000) || !geti("clipf", p.front_clip, 1, 2147483647L) ||
        !geti("clipe", p.end_clip, 1, 2147483647L) || !geti("cover", p.min_kmer_coverage, 0, 2147483647L) ||
        !geti("maxcov", p.max_kmer_coverage, 0, 2147483647L) || !geti("error", p.min_error_coverage, 0, 2147483647L) ||
        !geti("mincontig", p.min_contig, 0, 2147483647L))
        return bad_params(err);
    if (v.count("bubble")) p.bubble = 0;
    const bool gz = v.count("gzip") > 0;
    const std::string infmt = v.count("infmt") ? v["infmt"] : "4mc";
    // -kmerc wins over -fastq (Pipelines.java:83-84: inputKmerPath != null -> assemblyFromKmer()); with both, the FASTQ is
    // only read by the -stitch branch (Parameter.java:571-575, ReflexivDSMain.java:599)
    const bool from_kmer = !counter && v.count("kmerc");
    const bool stitch = from_kmer && !sorter && v.count("stitch");
    if (sorter && !from_kmer) { fputs(HELP, stdout); return 0; }
    if (!v.count("fastq") && !from_kmer) { fputs(HELP, stdout); return 0; }  // Parameter.java:565-568
    // -klist / -accurate: Parameter.java:362-387, 417-420 (read by the sorted stage only)
    std::vector<int> klist;
    {
        const std::string ks = v.count("klist") ? v["klist"] : "23,31,41,53,67,81,95";  // DefaultParam.java:87
        size_t pos = 0;
        while (pos <= ks.size()) {
            size_t end = ks.find(',', pos);
            if (end == std::string::npos) end = ks.size();
            char* e = nullptr;
            const std::string tok = ks.substr(pos, end - pos);
            const long x = strtol(tok.c_str(), &e, 0);
            if (tok.empty() || !e || *e) return bad_params("For input string: \"" + tok + "\"");
            klist.push_back((int)x);
            pos = end + 1;
        }
    }
    const double min_repeat_fold = v.count("accurate") ? 2.0 : 1.5;  // DefaultParam.java:107
    const SortStage sort_stage{min_repeat_fold, klist.back() /* param.kmerListInt[last], :445 */, std::find(klist.begin(), klist.end(), p.kmer_size) != klist.end()};
    if (!v.count("outfile")) { info("Output file not set of -outfile options"); return 0; }
    const std::string outdir = v["outfile"];
    p.counter_mode = counter ? 1 : 0;
    p.fastq_mode = counter ? (infmt == "line" ? RFX_FASTQ_LINE : RFX_FASTQ_COUNTER) : RFX_FASTQ_RUN;
    if (const char* d = getenv("REFLEXIV_DEVICE")) p.device = atoi(d);

    const std::string target = counter ? outdir + "/Count_" + std::to_string(p.kmer_size)
                               : sorter ? outdir + "/Count_" + std::to_string(p.kmer_size) + "_sorted"
                                        : (from_kmer ? outdir + "/Assemble_" + std::to_string(p.kmer_size) : outdir);
    struct stat stt;
    if (!counter && !sorter && stat(target.c_str(), &stt) == 0) {  // Hadoop FileAlreadyExistsException in saveAsTextFile
        fprintf(stderr, "reflexiv: output directory %s already exists\n", target.c_str());
        return 1;
    }

    if (n_gpus > 1 && stitch) { fprintf(stderr, "reflexiv: --gpus applies to runs from reads (-fastq), to -kmerc runs without -stitch and to sort; this one runs on one GPU\n"); n_gpus = 1; }
    if (n_gpus > RFX_SHARD_MAX_RANKS) { fprintf(stderr, "reflexiv: --gpus %d: at most %d\n", n_gpus, RFX_SHARD_MAX_RANKS); return 1; }
    // the rows a -kmerc table keeps: run cover <= count <= maxcov (ReflexivDSMain.java:405-412), sort count <= maxcov only
    // (ReflexivDSKmerLeftAndRightSorting.java:186-193) and only k-mers whose length is in the list (:1695): with k outside -klist every
    // row is still checked and none is kept
    const int64_t min_count = !sorter ? (int64_t)p.min_kmer_coverage : sort_stage.k_listed ? (int64_t)INT32_MIN : INT64_MAX;
    const int64_t max_count = p.max_kmer_coverage;
    if (n_gpus > 1) {
        info("Initiating CUDA contexts ...");
        if (from_kmer) return run_kmerc_sharded(n_gpus, p, sorter ? &sort_stage : nullptr, min_count, max_count, v["kmerc"], outdir, target, gz);
        return run_sharded(n_gpus, p, counter, v["fastq"], outdir, target, gz);
    }
    info("Initiating CUDA context ...");
    rfx_ctx* c = nullptr;
    if (rfx_create(&c, &p) != RFX_OK) return fail(nullptr, "rfx_create");
    if (from_kmer) {
        // every file parsed on the device as it arrives: the first call replaces the table, the others append
        bool load_ok = true, loaded = false;
        const bool read_ok = stream_inputs(v["kmerc"], [&](const char* data, size_t n) {
            load_ok = rfx_load_counts_csv(c, reinterpret_cast<const uint8_t*>(data), n, min_count, max_count, loaded ? 1 : 0) == RFX_OK;
            loaded = true;
            return load_ok;
        });
        if (!load_ok) return fail(c, "rfx_load_counts_csv");
        if (!read_ok) { rfx_destroy(c); return 1; }
        if (!loaded && rfx_load_counts_csv(c, nullptr, 0, min_count, max_count, 0) != RFX_OK) return fail(c, "rfx_load_counts_csv");  // only empty files
    } else {
        bool push_ok = true, pushed = false;
        const bool read_ok = stream_inputs(v["fastq"], [&](const char* data, size_t n) {
            push_ok = rfx_push_fastq(c, reinterpret_cast<const uint8_t*>(data), n) == RFX_OK;
            pushed = true;
            return push_ok;
        });
        if (!push_ok) return fail(c, "rfx_push_fastq");
        if (!read_ok) { rfx_destroy(c); return 1; }
        if (!pushed && rfx_push_fastq(c, reinterpret_cast<const uint8_t*>(""), 0) != RFX_OK) return fail(c, "rfx_push_fastq");  // only empty files
        if (rfx_count(c) != RFX_OK) return fail(c, "rfx_count");
    }
    mkdir(outdir.c_str(), 0755);
    if (counter || sorter) {
        if (sorter && rfx_sort_kmers(c, p.min_error_coverage, sort_stage.min_repeat_fold, sort_stage.max_kmer_size) != RFX_OK)
            return fail(c, "rfx_sort_kmers");
        mkdir(target.c_str(), 0755);
        clear_dir(target);
        if (!write_csv_part(c, sorter, target, 0, gz)) return fail(c, sorter ? "rfx_sorted_csv" : "rfx_counts_csv");
    } else {
        if (stitch) {
            // ReflexivDSMain.java:585-672: probes from the contig ends, the reads scanned for fragments, contigs joined
            if (!v.count("fastq")) { fprintf(stderr, "reflexiv: -stitch reads the FASTQ a second time (ReflexivDSMain.java:599): give -fastq\n"); rfx_destroy(c); return 1; }
            if (rfx_stitch_begin(c) != RFX_OK) return fail(c, "rfx_stitch_begin");
            bool push_ok = true;
            const bool read_ok = stream_inputs(v["fastq"], [&](const char* data, size_t n) {
                push_ok = rfx_push_fastq(c, reinterpret_cast<const uint8_t*>(data), n) == RFX_OK;
                return push_ok;
            });
            if (!push_ok) return fail(c, "rfx_push_fastq");
            if (!read_ok) { rfx_destroy(c); return 1; }
            if (rfx_stitch_finish(c) != RFX_OK) return fail(c, "rfx_stitch_finish");
            rfx_stitch_stats_t ss;
            rfx_stitch_stats(c, &ss);
            char m2[256];
            snprintf(m2, sizeof(m2), "stitch: %llu probes, %llu reads scanned, %llu fragments, %llu kept, %llu records stitched", (unsigned long long)ss.n_probes,
                     (unsigned long long)ss.n_reads, (unsigned long long)ss.n_fragments, (unsigned long long)ss.n_after_pass1, (unsigned long long)ss.n_stitched);
            info(m2);
        } else if (rfx_assemble(c) != RFX_OK) return fail(c, "rfx_assemble");
        mkdir(target.c_str(), 0755);
        if (!write_contig_part(c, target, 0, 0, gz && from_kmer, nullptr)) return fail(c, "rfx_contigs_copy");
    }
    FILE* ok = fopen((target + "/_SUCCESS").c_str(), "wb");
    if (ok) fclose(ok);
    rfx_stats_t s;
    rfx_stats(c, &s);
    char msg[512];
    snprintf(msg, sizeof(msg), "done: %llu reads, %llu k-mers, %llu distinct, %llu rows, %llu contigs; GPU ms parse %.2f partition %.2f count %.2f graph %.2f extend %.2f contigs %.2f",
             (unsigned long long)s.n_reads, (unsigned long long)s.n_instances, (unsigned long long)s.n_distinct, (unsigned long long)s.n_rows,
             (unsigned long long)s.n_contigs, s.ms_parse, s.ms_partition, s.ms_count, s.ms_graph, s.ms_extend, s.ms_contigs);
    info(msg);
    rfx_destroy(c);
    return 0;
}
