// stitch_align_cli.cpp — `stitch align` re-hosted on the B200 library: the reference's command line
// (fg-stitch-cli/src/commands/align.rs:94-275: same long/short flags and defaults), its input handling
// (FASTA/FASTQ, optionally gzip: fg-stitch-lib/src/align/io.rs:39-146, util/target_seq.rs:69-123), its
// "align a run of identical sequences once" rule (align.rs:364-375, io.rs:118-146), its output order
// (= input order, io.rs:161-175) and its output contract: a BAM stream on stdout (BGZF, level
// `--compression`, default 0) holding @HD / @SQ / @PG and the records of SamRecordFormatter::format, or the
// same as SAM text with --sam.  Everything between reading a batch and writing its records goes through
// the C ABI of include/stitch_b200.h (stitch_create / stitch_align_batch / stitch_format_sam): this file
// contains no alignment arithmetic and there is no CPU fallback.
//
// Pipeline (align.rs:338-441, io.rs:149-246 of the reference: a reader thread, aligner threads, an ordered writer): a
// reader thread parses and groups the input into batches and feeds a bounded queue; one worker thread per device context
// pulls batches as it becomes free (no lock-step rounds), aligns and formats them; the writer thread puts the finished
// batches back into input order, encodes BAM / BGZF and writes.  GPUs never wait for parsing, compression or each other.
// --pre-align runs the library's own pre-alignment (k-mer seeding on the GPU; the reference delegates it to the `bio`
// crate: parity unpinned, DESIGN.md section 9).
// The library is loaded at run time (STITCH_B200_LIB / STITCH_B200_PREFIX select another build of the same
// ABI: the CPU tests point it at the emulator of the kernels, tests/emul).
#include <dlfcn.h>
#include <unistd.h>
#include <zlib.h>

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstring>
#include <deque>
#include <map>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "../../include/stitch_b200.h"

namespace {

[[noreturn]] void die(const std::string &msg) {
    std::fprintf(stderr, "stitch-b200: %s\n", msg.c_str());
    std::exit(2);
}

// ---------------------------------------------------------------------------------------------
// the C ABI, bound at run time
// ---------------------------------------------------------------------------------------------
struct Api {
    void *h = nullptr;
    decltype(&stitch_create) create;
    decltype(&stitch_align_batch) align_batch;
    decltype(&stitch_format_sam) format_sam;
    decltype(&stitch_free_text) free_text;
    decltype(&stitch_free_results) free_results;
    decltype(&stitch_destroy) destroy;
    decltype(&stitch_last_error) last_error;
    decltype(&stitch_results_prealign) results_prealign;
    template <typename F> void bind(F &f, const std::string &prefix, const char *name) {
        f = reinterpret_cast<F>(dlsym(h, (prefix + name).c_str()));
        if (!f) die("symbol " + prefix + name + " not found in the alignment library");
    }
    void load(const char *argv0) {
        std::string path;
        if (const char *e = std::getenv("STITCH_B200_LIB")) path = e;
        else {
            std::string self = argv0;
            char buf[4096];
            const ssize_t n = readlink("/proc/self/exe", buf, sizeof(buf) - 1);
            if (n > 0) { buf[n] = 0; self = buf; }
            const size_t slash = self.rfind('/');
            path = (slash == std::string::npos ? std::string(".") : self.substr(0, slash)) + "/libstitch_b200.so";
        }
        h = dlopen(path.c_str(), RTLD_NOW | RTLD_LOCAL);
        if (!h) die(std::string("cannot load ") + path + ": " + dlerror());
        const char *pe = std::getenv("STITCH_B200_PREFIX");
        const std::string prefix = pe ? pe : "stitch_";
        bind(create, prefix, "create"); bind(align_batch, prefix, "align_batch"); bind(format_sam, prefix, "format_sam");
        bind(free_text, prefix, "free_text"); bind(free_results, prefix, "free_results"); bind(destroy, prefix, "destroy");
        bind(last_error, prefix, "last_error"); bind(results_prealign, prefix, "results_prealign");
    }
};

// ---------------------------------------------------------------------------------------------
// FASTA / FASTQ records (plain or gzip: zlib reads both)
// ---------------------------------------------------------------------------------------------
struct Record { std::string head, seq, qual; bool has_qual = false; };

class FastxReader {
  public:
    FastxReader(const std::string &path, bool fastq) : fastq_(fastq) {
        gz_ = gzopen(path.c_str(), "rb");
        if (!gz_) die("cannot open " + path);
        gzbuffer(gz_, 1 << 20);
    }
    ~FastxReader() { if (gz_) gzclose(gz_); }
    bool next(Record &r) {
        std::string line;
        if (pending_.empty()) { do { if (!getline(line)) return false; } while (line.empty()); }
        else { line.swap(pending_); pending_.clear(); }
        const char tag = fastq_ ? '@' : '>';
        if (line[0] != tag) die(std::string("malformed ") + (fastq_ ? "FASTQ" : "FASTA") + " record header: " + line);
        r.head = line.substr(1); r.seq.clear(); r.qual.clear(); r.has_qual = fastq_;
        if (fastq_) {
            // sequence lines up to '+', then as many quality characters as bases (multi-line FASTQ allowed)
            while (getline(line) && (line.empty() || line[0] != '+')) r.seq += line;
            while (r.qual.size() < r.seq.size() && getline(line)) r.qual += line;
            if (r.qual.size() != r.seq.size()) die("FASTQ record " + r.head + ": sequence and quality lengths differ");
        } else {
            while (getline(line)) {
                if (!line.empty() && line[0] == '>') { pending_ = line; break; }
                r.seq += line;
            }
        }
        return true;
    }

  private:
    bool getline(std::string &out) {
        out.clear();
        char buf[1 << 16];
        bool any = false;
        while (gzgets(gz_, buf, sizeof(buf))) {
            any = true;
            size_t n = std::strlen(buf);
            const bool eol = n && buf[n - 1] == '\n';
            if (eol) --n;
            if (n && buf[n - 1] == '\r') --n;
            out.append(buf, n);
            if (eol) return true;
        }
        return any;
    }
    gzFile gz_ = nullptr;
    bool fastq_;
    std::string pending_;
};

std::string upper(std::string s) {
    for (char &c : s) if (c >= 'a' && c <= 'z') c = (char)(c - 32);
    return s;
}
std::string first_word(const std::string &s) {
    size_t e = 0;
    while (e < s.size() && s[e] != ' ' && s[e] != '\t') ++e;
    return s.substr(0, e);
}

// ---------------------------------------------------------------------------------------------
// BAM / BGZF
// ---------------------------------------------------------------------------------------------
// BGZF blocks (<= 0xff00 payload bytes each) of a byte range, appended to `out`.  Blocks are independent, so every batch is
// compressed by the formatter thread that encoded it and the writer only copies bytes to the stream.
void bgzf_compress(const uint8_t *p, size_t n, int level, std::vector<uint8_t> &out) {
    constexpr size_t BLOCK = 0xff00;
    while (n) {
        const size_t take = std::min(n, BLOCK);
        const size_t at = out.size();
        out.resize(at + BLOCK + 1024);
        z_stream zs{};
        if (deflateInit2(&zs, level, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) die("zlib: deflateInit2 failed");
        zs.next_in = const_cast<uint8_t *>(p); zs.avail_in = (uInt)take;
        zs.next_out = out.data() + at + 18; zs.avail_out = (uInt)(BLOCK + 1024 - 18 - 8);
        if (deflate(&zs, Z_FINISH) != Z_STREAM_END) die("zlib: deflate failed");
        const size_t clen = zs.total_out;
        deflateEnd(&zs);
        const size_t bsize = 18 + clen + 8;
        const uint8_t hdr[18] = {31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 'B', 'C', 2, 0, (uint8_t)((bsize - 1) & 255), (uint8_t)((bsize - 1) >> 8)};
        std::memcpy(out.data() + at, hdr, 18);
        const uint32_t crc = (uint32_t)crc32(crc32(0L, Z_NULL, 0), p, (uInt)take), isz = (uint32_t)take;
        for (int k = 0; k < 4; ++k) { out[at + 18 + clen + k] = (uint8_t)(crc >> (8 * k)); out[at + 22 + clen + k] = (uint8_t)(isz >> (8 * k)); }
        out.resize(at + bsize);
        p += take; n -= take;
    }
}
void write_all(FILE *f, const uint8_t *p, size_t n) { if (n && std::fwrite(p, 1, n, f) != n) die("write failed"); }
void bgzf_finish(FILE *f) {
    static const uint8_t eof[28] = {31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 66, 67, 2, 0, 27, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    write_all(f, eof, 28);
    std::fflush(f);
}

void put32(std::vector<uint8_t> &v, uint32_t x) { for (int k = 0; k < 4; ++k) v.push_back((uint8_t)(x >> (8 * k))); }
void put16(std::vector<uint8_t> &v, uint32_t x) { v.push_back((uint8_t)x); v.push_back((uint8_t)(x >> 8)); }

int reg2bin(int64_t beg, int64_t end) {   // SAM specification, section 5.3
    --end;
    if (beg >> 14 == end >> 14) return (int)(((1 << 15) - 1) / 7 + (beg >> 14));
    if (beg >> 17 == end >> 17) return (int)(((1 << 12) - 1) / 7 + (beg >> 17));
    if (beg >> 20 == end >> 20) return (int)(((1 << 9) - 1) / 7 + (beg >> 20));
    if (beg >> 23 == end >> 23) return (int)(((1 << 6) - 1) / 7 + (beg >> 23));
    if (beg >> 26 == end >> 26) return (int)(((1 << 3) - 1) / 7 + (beg >> 26));
    return 0;
}

std::vector<std::string> split_tab(const std::string &s) {
    std::vector<std::string> f;
    size_t b = 0;
    for (;;) {
        const size_t e = s.find('\t', b);
        f.push_back(s.substr(b, e == std::string::npos ? std::string::npos : e - b));
        if (e == std::string::npos) break;
        b = e + 1;
    }
    return f;
}

// One SAM text line -> one BAM record (block_size included).
std::vector<uint8_t> bam_record(const std::string &line, const std::vector<std::string> &ref_names) {
    const std::vector<std::string> f = split_tab(line);
    if (f.size() < 11) die("internal: SAM line with fewer than 11 fields");
    auto ref_id = [&](const std::string &name, int32_t same) -> int32_t {
        if (name == "*") return -1;
        if (name == "=") return same;
        for (size_t k = 0; k < ref_names.size(); ++k) if (ref_names[k] == name) return (int32_t)k;
        die("internal: unknown reference " + name);
    };
    const int32_t rid = ref_id(f[2], -1), pos = (int32_t)std::stol(f[3]) - 1;
    const uint32_t flag = (uint32_t)std::stoul(f[1]), mapq = (uint32_t)std::stoul(f[4]);
    std::vector<uint32_t> cigar;
    int64_t ref_len = 0;
    if (f[5] != "*") {
        static const char *OPS = "MIDNSHP=X";
        size_t k = 0;
        while (k < f[5].size()) {
            uint64_t n = 0;
            while (k < f[5].size() && f[5][k] >= '0' && f[5][k] <= '9') n = n * 10 + (uint64_t)(f[5][k++] - '0');
            const char *p = std::strchr(OPS, f[5][k++]);
            if (!p) die("internal: bad CIGAR " + f[5]);
            const uint32_t op = (uint32_t)(p - OPS);
            cigar.push_back((uint32_t)(n << 4) | op);
            if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) ref_len += (int64_t)n;
        }
    }
    if (cigar.size() > 65535) die("a record has more than 65535 CIGAR operations (CG tag not implemented)");
    const std::string &seq = f[9], &qual = f[10];
    const uint32_t l_seq = seq == "*" ? 0u : (uint32_t)seq.size();
    std::vector<uint8_t> r;
    put32(r, 0);   // block_size, patched below
    put32(r, (uint32_t)rid); put32(r, (uint32_t)pos);
    r.push_back((uint8_t)(f[0].size() + 1)); r.push_back((uint8_t)mapq);
    put16(r, (uint32_t)reg2bin(pos < 0 ? 0 : pos, pos < 0 ? 1 : pos + (ref_len > 0 ? ref_len : 1)));
    put16(r, (uint32_t)cigar.size()); put16(r, flag); put32(r, l_seq);
    put32(r, (uint32_t)ref_id(f[6], rid)); put32(r, (uint32_t)((int32_t)std::stol(f[7]) - 1)); put32(r, (uint32_t)(int32_t)std::stol(f[8]));
    r.insert(r.end(), f[0].begin(), f[0].end()); r.push_back(0);
    for (uint32_t c : cigar) put32(r, c);
    static const char *NT16 = "=ACMGRSVTWYHKDBN";
    for (uint32_t k = 0; k < l_seq; k += 2) {
        // (the 4-bit codes have no case: soft-masked bases encode as their upper-case letters, as in htslib)
        auto code = [&](char c) -> uint8_t { if (c >= 'a' && c <= 'z') c = (char)(c - 32); const char *p = std::strchr(NT16, c); return (uint8_t)(p && c ? p - NT16 : 15); };
        r.push_back((uint8_t)((code(seq[k]) << 4) | (k + 1 < l_seq ? code(seq[k + 1]) : 0)));
    }
    if (qual == "*") r.insert(r.end(), l_seq, 0xff);
    else for (uint32_t k = 0; k < l_seq; ++k) r.push_back((uint8_t)(qual[k] - 33));
    for (size_t t = 11; t < f.size(); ++t) {   // TAG:TYPE:VALUE
        const std::string &s = f[t];
        if (s.size() < 5 || s[2] != ':' || s[4] != ':') die("internal: bad SAM tag " + s);
        r.push_back((uint8_t)s[0]); r.push_back((uint8_t)s[1]);
        const std::string v = s.substr(5);
        switch (s[3]) {
            case 'i': {   // smallest integer type that holds the value (as htslib does)
                const long long x = std::stoll(v);
                if (x >= 0) {
                    if (x <= 255) { r.push_back('C'); r.push_back((uint8_t)x); }
                    else if (x <= 65535) { r.push_back('S'); put16(r, (uint32_t)x); }
                    else { r.push_back('I'); put32(r, (uint32_t)x); }
                } else {
                    if (x >= -128) { r.push_back('c'); r.push_back((uint8_t)(int8_t)x); }
                    else if (x >= -32768) { r.push_back('s'); put16(r, (uint32_t)(int16_t)x); }
                    else { r.push_back('i'); put32(r, (uint32_t)(int32_t)x); }
                }
                break;
            }
            case 'A': r.push_back('A'); r.push_back((uint8_t)v[0]); break;
            case 'f': { r.push_back('f'); const float x = std::stof(v); uint32_t u; std::memcpy(&u, &x, 4); put32(r, u); break; }
            case 'Z': r.push_back('Z'); r.insert(r.end(), v.begin(), v.end()); r.push_back(0); break;
            default: die("internal: SAM tag type not handled: " + s);
        }
    }
    const uint32_t bs = (uint32_t)r.size() - 4;
    for (int k = 0; k < 4; ++k) r[k] = (uint8_t)(bs >> (8 * k));
    return r;
}

// ---------------------------------------------------------------------------------------------
// command line (align.rs:94-275)
// ---------------------------------------------------------------------------------------------
struct Args {
    std::string reads_fastq, reads_fasta, ref_fasta;
    bool double_strand = false, decompress = false, pre_align = false, pre_align_subset = true, soft_clip = false, use_eq_and_x = false, circular = false,
         filter_secondary = false, suboptimal = false, sam = false;
    int threads = 2, match_score = 1, mismatch_score = -4, gap_open = -6, gap_extend = -2, jump_score = -10, mode = STITCH_MODE_LOCAL,
        pick_primary = 0, compression = 0, gpus = 1, device = 0;
    bool has_same = false, has_opp = false, has_inter = false;
    int jump_same = 0, jump_opp = 0, jump_inter = 0;
    unsigned circular_slop = 20, batch = 2048, kmer = 12, band = 50;
    int pre_align_min_score = 100, pre_align_scoring = STITCH_PREALIGN_KMER;
    float filter_secondary_pct = 10.0f, suboptimal_pct = 20.0f;
    std::string command_line;
};

bool parse_bool(const std::string &v) {
    if (v == "true" || v == "1") return true;
    if (v == "false" || v == "0") return false;
    die("expected true or false, got " + v);
}
int parse_mode(std::string v) {
    for (char &c : v) if (c >= 'A' && c <= 'Z') c = (char)(c + 32);
    std::string w;
    for (char c : v) if (c != '-' && c != '_') w += c;
    if (w == "local") return STITCH_MODE_LOCAL;
    if (w == "querylocal") return STITCH_MODE_QUERY_LOCAL;
    if (w == "targetlocal") return STITCH_MODE_TARGET_LOCAL;
    if (w == "global") return STITCH_MODE_GLOBAL;
    die("unknown alignment mode " + v);
}

void usage() {
    std::fputs(
        "stitch-b200 align: `stitch align` on NVIDIA B200 (same options as fulcrumgenomics/stitch)\n"
        "  -f, --reads-fastq <FASTQ> | -a, --reads-fasta <FASTA>   reads (plain or gzip)\n"
        "  -r, --ref-fasta <FASTA>          reference contigs\n"
        "  -d, --double-strand  -C, --circular  --circular-slop <20>\n"
        "  -m, --mode <local|query-local|target-local|global>      [local]\n"
        "  -A <1> -B <-4> -O <-6> -E <-2> -J <-10>  --jump-score-same-contig-and-strand <J>\n"
        "  --jump-score-same-contig-opposite-strand <J>  --jump-score-inter-contig <J>\n"
        "  -S, --soft-clip  -X, --use-eq-and-x  -P, --pick-primary <query-length|score>\n"
        "  --filter-secondary [--filter-secondary-pct <10>]  --suboptimal [--suboptimal-pct <20>]\n"
        "  -c, --compression <0>            BGZF level of the BAM written to stdout\n"
        "  -t, --threads <2>                formatter threads (SAM records + BAM encoding; alignment runs on the GPU)\n"
        "  -p, --pre-align                  pre-align reads (k-mer seeding on the GPU) and align only those reaching the score\n"
        "  -k, --k <12>  -w, --w <50>  -s, --pre-align-min-score <100>  -x, --pre-align-subset-contigs <true>\n"
        "extras: --sam (SAM text instead of BAM)  --gpus <1>  --device <0>  --batch <2048>\n"
        "  --pre-align-scoring <kmer|banded>  [kmer] score of -p: bases covered by exact k-mer hits in the best band, or\n"
        "                                   the best local affine-gap alignment inside that band\n", stderr);
}

Args parse(int argc, char **argv) {
    Args a;
    for (int k = 0; k < argc; ++k) { if (k) a.command_line += ' '; a.command_line += argv[k]; }
    int i = 1;
    if (i < argc && std::string(argv[i]) == "align") ++i;
    auto value = [&](const std::string &flag, const std::string &inline_v, bool has_inline) -> std::string {
        if (has_inline) return inline_v;
        if (i + 1 >= argc) die("option " + flag + " needs a value");
        return argv[++i];
    };
    for (; i < argc; ++i) {
        std::string arg = argv[i], inl;
        bool has_inl = false;
        if (arg.rfind("--", 0) == 0) {
            const size_t eq = arg.find('=');
            if (eq != std::string::npos) { inl = arg.substr(eq + 1); arg = arg.substr(0, eq); has_inl = true; }
        }
        // boolean flags: bare, or with an explicit true/false (clap's default_value = "false" flags take no value;
        // --pre-align-subset-contigs takes one)
        auto flag = [&](bool &dst) { dst = has_inl ? parse_bool(inl) : true; };
        if (arg == "-h" || arg == "--help") { usage(); std::exit(0); }
        else if (arg == "-f" || arg == "--reads-fastq") a.reads_fastq = value(arg, inl, has_inl);
        else if (arg == "-a" || arg == "--reads-fasta") a.reads_fasta = value(arg, inl, has_inl);
        else if (arg == "-r" || arg == "--ref-fasta") a.ref_fasta = value(arg, inl, has_inl);
        else if (arg == "-d" || arg == "--double-strand") flag(a.double_strand);
        else if (arg == "-t" || arg == "--threads") a.threads = std::stoi(value(arg, inl, has_inl));
        else if (arg == "-z" || arg == "--decompress") flag(a.decompress);
        else if (arg == "-p" || arg == "--pre-align") flag(a.pre_align);
        else if (arg == "-k" || arg == "--k") a.kmer = (unsigned)std::stoul(value(arg, inl, has_inl));
        else if (arg == "-w" || arg == "--w") a.band = (unsigned)std::stoul(value(arg, inl, has_inl));
        else if (arg == "-s" || arg == "--pre-align-min-score") a.pre_align_min_score = std::stoi(value(arg, inl, has_inl));
        else if (arg == "-x" || arg == "--pre-align-subset-contigs") a.pre_align_subset = parse_bool(value(arg, inl, has_inl));   // takes a value (align.rs:144-146)
        else if (arg == "-S" || arg == "--soft-clip") flag(a.soft_clip);
        else if (arg == "-X" || arg == "--use-eq-and-x") flag(a.use_eq_and_x);
        else if (arg == "-A" || arg == "--match-score") a.match_score = std::stoi(value(arg, inl, has_inl));
        else if (arg == "-B" || arg == "--mismatch-score") a.mismatch_score = std::stoi(value(arg, inl, has_inl));
        else if (arg == "-O" || arg == "--gap-open") a.gap_open = std::stoi(value(arg, inl, has_inl));
        else if (arg == "-E" || arg == "--gap-extend") a.gap_extend = std::stoi(value(arg, inl, has_inl));
        else if (arg == "-J" || arg == "--jump-score") a.jump_score = std::stoi(value(arg, inl, has_inl));
        else if (arg == "--jump-score-same-contig-and-strand") { a.jump_same = std::stoi(value(arg, inl, has_inl)); a.has_same = true; }
        else if (arg == "--jump-score-same-contig-opposite-strand") { a.jump_opp = std::stoi(value(arg, inl, has_inl)); a.has_opp = true; }
        else if (arg == "--jump-score-inter-contig") { a.jump_inter = std::stoi(value(arg, inl, has_inl)); a.has_inter = true; }
        else if (arg == "-m" || arg == "--mode") a.mode = parse_mode(value(arg, inl, has_inl));
        else if (arg == "-P" || arg == "--pick-primary") {
            std::string v = value(arg, inl, has_inl);
            for (char &c : v) if (c >= 'A' && c <= 'Z') c = (char)(c + 32);
            if (v == "score") a.pick_primary = 1; else if (v == "query-length" || v == "querylength") a.pick_primary = 0; else die("unknown --pick-primary " + v);
        }
        else if (arg == "-C" || arg == "--circular") flag(a.circular);
        else if (arg == "--circular-slop") a.circular_slop = (unsigned)std::stoul(value(arg, inl, has_inl));
        else if (arg == "--filter-secondary") flag(a.filter_secondary);
        else if (arg == "--filter-secondary-pct") a.filter_secondary_pct = std::stof(value(arg, inl, has_inl));
        else if (arg == "--suboptimal") flag(a.suboptimal);
        else if (arg == "--suboptimal-pct") a.suboptimal_pct = std::stof(value(arg, inl, has_inl));
        else if (arg == "-c" || arg == "--compression") a.compression = std::stoi(value(arg, inl, has_inl));
        else if (arg == "--sam") a.sam = true;
        else if (arg == "--gpus") a.gpus = std::stoi(value(arg, inl, has_inl));
        else if (arg == "--device") a.device = std::stoi(value(arg, inl, has_inl));
        else if (arg == "--batch") a.batch = (unsigned)std::stoul(value(arg, inl, has_inl));
        else if (arg == "--pre-align-scoring") {
            const std::string v = value(arg, inl, has_inl);
            if (v == "kmer") a.pre_align_scoring = STITCH_PREALIGN_KMER;
            else if (v == "banded") a.pre_align_scoring = STITCH_PREALIGN_BANDED;
            else die("unknown --pre-align-scoring " + v + " (expected kmer or banded)");
        }
        else die("unknown option " + arg + " (see --help)");
    }
    if (a.reads_fastq.empty() == a.reads_fasta.empty()) die("Must specify exactly one of --reads-fastq or --reads-fasta");
    if (a.ref_fasta.empty()) die("--ref-fasta is required");
    if (a.match_score <= 0) die("--match-score must be positive");
    if (a.mismatch_score >= 0 || a.gap_open >= 0 || a.gap_extend >= 0 || a.jump_score >= 0) die("mismatch, gap and jump scores must be negative");
    if (a.compression < 0 || a.compression > 9) die("--compression must be 0..9");
    if (a.gpus < 1 || a.batch < 1) die("--gpus and --batch must be positive");
    return a;
}

// One batch of input records on one device context: align the unique sequences, format every record.
struct Batch {
    uint64_t seq_no = 0;
    std::vector<Record> recs;
    std::vector<uint32_t> uniq_of;     // record -> aligned (de-duplicated) sequence
    stitch_ctx *ctx = nullptr;         // the context that aligned it
    stitch_results *res = nullptr;
    std::vector<std::string> lines;    // SAM text lines (--sam)
    std::vector<uint8_t> bam;          // encoded BAM records, back to back
    uint64_t n_records = 0;
    std::string error;
};

// Stage 2 (one thread per device context): align the unique sequences of the batch.
void align_stage(const Api &api, stitch_ctx *ctx, Batch &b) {
    // a run of consecutive records with the same (upper-cased) sequence is aligned once (align.rs:364-375)
    b.uniq_of.resize(b.recs.size());
    std::vector<std::string> seqs;
    for (size_t k = 0; k < b.recs.size(); ++k) {
        std::string u = upper(b.recs[k].seq);
        if (seqs.empty() || seqs.back() != u) seqs.push_back(std::move(u));
        b.uniq_of[k] = (uint32_t)seqs.size() - 1;
    }
    std::string blob;
    std::vector<uint64_t> offs(seqs.size() + 1, 0);
    for (size_t k = 0; k < seqs.size(); ++k) { blob += seqs[k]; offs[k + 1] = blob.size(); }
    b.ctx = ctx;
    if (api.align_batch(ctx, reinterpret_cast<const uint8_t *>(blob.data()), offs.data(), (uint32_t)seqs.size(), nullptr, 0, &b.res) != STITCH_OK) {
        b.error = api.last_error(ctx);
        b.res = nullptr;
    }
}

// Stage 3 (--threads formatter threads): the SAM records of every read of the batch (host work: it overlaps the next
// batch's alignment on the device), encoded as BAM unless --sam.
void format_stage(const Api &api, const stitch_sam_opts &so, const std::vector<std::string> &names, bool sam, int level, Batch &b) {
    if (!b.res) return;
    for (size_t k = 0; k < b.recs.size() && b.error.empty(); ++k) {
        const Record &r = b.recs[k];
        char *text = nullptr;
        int32_t pre_score = 0;
        const int has_pre = api.results_prealign(b.res, b.uniq_of[k], &pre_score);   // the Option<i32> of Aligners::align (mod.rs:338-339)
        // SEQ / QUAL of the records are the read as given (SamRecordFormatter::format uses fastq.seq(), mod.rs:630; only the
        // alignment sees the upper-cased copy, mod.rs:243)
        if (api.format_sam(b.ctx, b.res, b.uniq_of[k], r.head.c_str(), reinterpret_cast<const uint8_t *>(r.seq.data()),
                           r.has_qual ? reinterpret_cast<const uint8_t *>(r.qual.data()) : nullptr, (uint32_t)r.seq.size(), has_pre, pre_score, &so, &text) != STITCH_OK) {
            b.error = api.last_error(b.ctx);
            break;
        }
        const char *p = text ? text : "";
        while (*p) {
            const char *e = std::strchr(p, '\n');
            std::string line = e ? std::string(p, e) : std::string(p);
            if (sam) b.lines.push_back(std::move(line));
            else { const std::vector<uint8_t> rec = bam_record(line, names); b.bam.insert(b.bam.end(), rec.begin(), rec.end()); }
            ++b.n_records;
            if (!e) break;
            p = e + 1;
        }
        api.free_text(text);
    }
    api.free_results(b.res);
    b.res = nullptr;
    std::vector<Record>().swap(b.recs);
    if (!sam && !b.bam.empty()) {   // BGZF here, in parallel: the writer only copies
        std::vector<uint8_t> z;
        z.reserve(b.bam.size() + b.bam.size() / 512 + 64);
        bgzf_compress(b.bam.data(), b.bam.size(), level, z);
        b.bam.swap(z);
    }
}

// Bounded hand-over between the pipeline stages.
template <typename T>
class Channel {
  public:
    explicit Channel(size_t cap) : cap_(cap) {}
    void push(T v) {
        std::unique_lock<std::mutex> l(m_);
        not_full_.wait(l, [&] { return q_.size() < cap_; });
        q_.push_back(std::move(v));
        not_empty_.notify_one();
    }
    bool pop(T &v) {   // false: closed and drained
        std::unique_lock<std::mutex> l(m_);
        not_empty_.wait(l, [&] { return !q_.empty() || closed_; });
        if (q_.empty()) return false;
        v = std::move(q_.front()); q_.pop_front();
        not_full_.notify_one();
        return true;
    }
    void close() { std::lock_guard<std::mutex> l(m_); closed_ = true; not_empty_.notify_all(); }

  private:
    std::mutex m_;
    std::condition_variable not_full_, not_empty_;
    std::deque<T> q_;
    size_t cap_;
    bool closed_ = false;
};

}  // namespace

int main(int argc, char **argv) {
    const auto t_start = std::chrono::steady_clock::now();
    auto since_start = [&] { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count(); };
    const Args a = parse(argc, argv);
    Api api;
    api.load(argv[0]);
    // STITCH_CLI_TIMING=1: one JSON line on stderr at exit (where the wall clock of the process goes: start-up, the span
    // in which the devices align, the busy time of every stage)
    const bool timing = std::getenv("STITCH_CLI_TIMING") != nullptr;
    std::atomic<uint64_t> align_busy_us{0}, format_busy_us{0}, write_busy_us{0}, reads_aligned{0};
    std::mutex span_m;
    double t_ctx_ready = 0, t_first_align = -1, t_last_align = 0;

    // reference contigs: upper-cased, name = first word of the header (target_seq.rs:99-121)
    std::vector<std::string> names, seqs;
    {
        FastxReader rf(a.ref_fasta, false);
        Record r;
        while (rf.next(r)) { names.push_back(first_word(r.head)); seqs.push_back(upper(r.seq)); }
        if (names.empty()) die("no contigs in " + a.ref_fasta);
    }
    std::vector<stitch_contig> contigs(names.size());
    for (size_t k = 0; k < names.size(); ++k) {
        contigs[k].name = names[k].c_str();
        contigs[k].fwd = reinterpret_cast<const uint8_t *>(seqs[k].data());
        contigs[k].len = (uint32_t)seqs[k].size();
    }
    stitch_opts o{};
    o.mode = a.mode; o.match_score = a.match_score; o.mismatch_score = a.mismatch_score; o.gap_open = a.gap_open; o.gap_extend = a.gap_extend;
    o.jump_same = a.has_same ? a.jump_same : a.jump_score; o.jump_opp = a.has_opp ? a.jump_opp : a.jump_score;
    o.jump_inter = a.has_inter ? a.jump_inter : a.jump_score;
    o.double_strand = a.double_strand; o.circular = a.circular; o.suboptimal = a.suboptimal;
    o.circular_slop = a.circular_slop; o.suboptimal_pct = a.suboptimal_pct;
    o.pre_align = a.pre_align; o.pre_align_subset_contigs = a.pre_align_subset; o.kmer_size = a.kmer; o.band_width = a.band;
    o.pre_align_min_score = a.pre_align_min_score; o.pre_align_scoring = (uint8_t)a.pre_align_scoring;
    stitch_sam_opts so{};
    so.soft_clip = a.soft_clip; so.use_eq_and_x = a.use_eq_and_x; so.pick_primary = (uint8_t)a.pick_primary;
    so.filter_secondary = a.filter_secondary; so.filter_secondary_pct = a.filter_secondary_pct;

    // one context per device, created concurrently (driver initialisation and the contig upload of every device overlap)
    std::vector<stitch_ctx *> ctxs((size_t)a.gpus, nullptr);
    {
        std::vector<std::string> errs((size_t)a.gpus);
        std::vector<std::thread> th;
        for (int g = 0; g < a.gpus; ++g)
            th.emplace_back([&, g] {
                if (api.create(&o, contigs.data(), (uint32_t)contigs.size(), a.device + g, &ctxs[(size_t)g]) != STITCH_OK)
                    errs[(size_t)g] = std::string("cannot create the aligner on device ") + std::to_string(a.device + g) + ": " + api.last_error(nullptr);
            });
        for (auto &t : th) t.join();
        for (const auto &e : errs) if (!e.empty()) die(e);
    }
    t_ctx_ready = since_start();

    // header: @HD, one @SQ per contig, @PG (align.rs:393-416)
    std::string header = "@HD\tVN:1.6\n";
    for (size_t k = 0; k < names.size(); ++k) header += "@SQ\tSN:" + names[k] + "\tLN:" + std::to_string(seqs[k].size()) + "\n";
    header += "@PG\tID:stitch\tPN:stitch\tVN:b200-0.1.0\tCL:" + a.command_line + "\n";
    std::setvbuf(stdout, nullptr, _IOFBF, 8u << 20);
    if (a.sam) std::fputs(header.c_str(), stdout);
    else {
        std::vector<uint8_t> h = {'B', 'A', 'M', 1};
        put32(h, (uint32_t)header.size()); h.insert(h.end(), header.begin(), header.end());
        put32(h, (uint32_t)names.size());
        for (size_t k = 0; k < names.size(); ++k) {
            put32(h, (uint32_t)names[k].size() + 1); h.insert(h.end(), names[k].begin(), names[k].end()); h.push_back(0);
            put32(h, (uint32_t)seqs[k].size());
        }
        std::vector<uint8_t> z;
        bgzf_compress(h.data(), h.size(), a.compression, z);
        write_all(stdout, z.data(), z.size());
    }

    const int n_fmt = std::max(std::max(1, a.threads), 2 * a.gpus);   // (two formatters keep up with one B200 on 10 kb reads)
    Channel<std::unique_ptr<Batch>> to_align((size_t)a.gpus * 2), to_format((size_t)a.gpus * 2 + (size_t)n_fmt), to_write((size_t)a.gpus * 4 + 4);
    std::mutex err_m;
    std::string first_error;
    auto fail = [&](const std::string &e) { std::lock_guard<std::mutex> l(err_m); if (first_error.empty()) first_error = e; };

    // reader: batches of >= --batch records; a run of identical sequences is never split across batches (io.rs:126-146)
    std::thread reader([&] {
        FastxReader reads(a.reads_fastq.empty() ? a.reads_fasta : a.reads_fastq, !a.reads_fastq.empty());
        Record carry; bool have_carry = false, eof = false;
        uint64_t seq_no = 0;
        while (!eof) {
            std::unique_ptr<Batch> b(new Batch());
            b->seq_no = seq_no++;
            if (have_carry) { b->recs.push_back(std::move(carry)); have_carry = false; }
            Record r;
            for (;;) {
                if (!reads.next(r)) { eof = true; break; }
                if (b->recs.size() >= a.batch && upper(r.seq) != upper(b->recs.back().seq)) { carry = std::move(r); have_carry = true; break; }
                b->recs.push_back(std::move(r));
            }
            if (!b->recs.empty()) to_align.push(std::move(b)); else --seq_no;
        }
        to_align.close();
    });
    // aligners: one per device context, each pulls the next batch as soon as it is free
    std::vector<std::thread> workers;
    for (int g = 0; g < a.gpus; ++g)
        workers.emplace_back([&, g] {
            std::unique_ptr<Batch> b;
            while (to_align.pop(b)) {
                const double t0 = since_start();
                align_stage(api, ctxs[(size_t)g], *b);
                const double t1 = since_start();
                align_busy_us += (uint64_t)((t1 - t0) * 1e6); reads_aligned += b->recs.size();
                { std::lock_guard<std::mutex> l(span_m); if (t_first_align < 0 || t0 < t_first_align) t_first_align = t0; if (t1 > t_last_align) t_last_align = t1; }
                if (!b->error.empty()) fail(b->error);
                to_format.push(std::move(b));
            }
        });
    // formatters (-t): SAM records + BAM encoding, off the aligners' threads
    std::vector<std::thread> formatters;
    for (int t = 0; t < n_fmt; ++t)
        formatters.emplace_back([&] {
            std::unique_ptr<Batch> b;
            while (to_format.pop(b)) {
                const double t0 = since_start();
                format_stage(api, so, names, a.sam, a.compression, *b);
                format_busy_us += (uint64_t)((since_start() - t0) * 1e6);
                if (!b->error.empty()) fail(b->error);
                to_write.push(std::move(b));
            }
        });
    // writer: input order restored, BGZF and the output stream
    uint64_t n_lines = 0, n_batches = 0;
    std::thread writer([&] {
        std::map<uint64_t, std::unique_ptr<Batch>> pending;
        uint64_t next = 0;
        std::unique_ptr<Batch> b;
        while (to_write.pop(b)) {
            pending[b->seq_no] = std::move(b);
            const double t0 = since_start();
            for (auto it = pending.find(next); it != pending.end(); it = pending.find(next)) {
                if (a.sam) for (const std::string &line : it->second->lines) { std::fputs(line.c_str(), stdout); std::fputc('\n', stdout); }
                else write_all(stdout, it->second->bam.data(), it->second->bam.size());
                n_lines += it->second->n_records; ++n_batches;
                pending.erase(it); ++next;
            }
            write_busy_us += (uint64_t)((since_start() - t0) * 1e6);
        }
    });
    reader.join();
    for (auto &t : workers) t.join();
    to_format.close();
    for (auto &t : formatters) t.join();
    to_write.close();
    writer.join();
    if (!first_error.empty()) die("alignment failed: " + first_error);
    if (a.sam) std::fflush(stdout); else bgzf_finish(stdout);
    for (stitch_ctx *c : ctxs) api.destroy(c);
    if (timing) {
        const double span = t_last_align - t_first_align, wall = since_start();
        std::fprintf(stderr, "stitch-b200 timing: {\"wall_s\": %.3f, \"contexts_ready_s\": %.3f, \"first_align_s\": %.3f, \"last_align_s\": %.3f, "
                             "\"align_span_s\": %.3f, \"reads\": %llu, \"reads_per_s_in_align_span\": %.1f, \"gpus\": %d, \"align_busy_s\": %.3f, "
                             "\"format_threads\": %d, \"format_busy_s\": %.3f, \"write_busy_s\": %.3f}\n",
                     wall, t_ctx_ready, t_first_align, t_last_align, span, (unsigned long long)reads_aligned.load(),
                     span > 0 ? (double)reads_aligned.load() / span : 0.0, a.gpus, align_busy_us.load() * 1e-6, n_fmt, format_busy_us.load() * 1e-6,
                     write_busy_us.load() * 1e-6);
    }
    std::fprintf(stderr, "stitch-b200: wrote %llu records of %llu batches\n", (unsigned long long)n_lines, (unsigned long long)n_batches);
    return 0;
}
