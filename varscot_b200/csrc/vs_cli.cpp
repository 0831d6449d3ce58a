// varscot_b200/csrc/vs_cli.cpp — the two executables of the read_mapping stage as library calls.
//
//   vs_bidir_index_main   mirrors VARSCOT_pipeline/read_mapping/bidir_index.cpp:10-52
//                         (-G/--genome fa|fasta|fastq, -I/--index prefix; stdout lines :42,:49)
//   vs_bidir_mapping_main mirrors VARSCOT_pipeline/read_mapping/bidir_mapping.cpp:190-312
//                         (-G -I -R -M -T -O -P; range check :234-238; stdout lines :265,:269;
//                          exit codes :219-220,:237,:301-305; header-less SAM :298-309)
// The argv contract is what VARSCOT_pipeline/VARSCOT:296-314 passes.  The "index" written at the
// -I prefix is the bit-sliced packed text (<prefix>.vsidx), not an FM index.
#include "vs_internal.h"
#include <algorithm>
#include <cctype>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <string>
#include <thread>
#include <fcntl.h>
#include <sys/file.h>
#include <unistd.h>
#include <unistd.h>
#include <vector>

namespace {

// ---- FASTA ----------------------------------------------------------------------------------
// SeqAn readRecord semantics as used by the reference: id = the whole header line after '>'
// (bidir_mapping.cpp:272-280), sequence = every non-whitespace character up to the next header.
struct FastaSink {
    std::function<void(const std::string &)> header;
    std::function<void(const char *, size_t)> seq;
    std::function<void()> end_record;
};

bool read_fasta(const std::string &path, const FastaSink &sink, std::string &err)
{
    FILE *f = fopen(path.c_str(), "rb");
    if (!f) { err = "cannot open " + path; return false; }
    std::vector<char> buf(8u << 20);
    std::string hdr;
    bool in_header = false, at_line_start = true, have_record = false;
    size_t got;
    while ((got = fread(buf.data(), 1, buf.size(), f)) > 0) {
        const char *b = buf.data();
        size_t i = 0;
        while (i < got) {
            if (in_header) {
                const char *nl = (const char *)memchr(b + i, '\n', got - i);
                size_t e = nl ? (size_t)(nl - b) : got;
                hdr.append(b + i, e - i);
                i = e;
                if (nl) {
                    while (!hdr.empty() && (hdr.back() == '\r' || hdr.back() == '\n')) hdr.pop_back();
                    sink.header(hdr);
                    hdr.clear();
                    in_header = false; at_line_start = true; have_record = true;
                    ++i;
                }
                continue;
            }
            // sequence data runs to the next '>' that opens a line; whole spans (newlines included) go to the sink
            size_t j = i;
            bool header_found = false;
            while (j < got) {
                const char *gt = (const char *)memchr(b + j, '>', got - j);
                if (!gt) { j = got; break; }
                size_t g = (size_t)(gt - b);
                bool line_start = g == 0 ? at_line_start : (g == i ? at_line_start : b[g - 1] == '\n');
                if (line_start) { j = g; header_found = true; break; }
                j = g + 1;                                   // a '>' inside a line is just a (non-ACGT) character
            }
            if (j > i) {
                if (have_record) sink.seq(b + i, j - i);
                at_line_start = b[j - 1] == '\n';
            }
            i = j;
            if (header_found) {
                if (have_record) sink.end_record();
                in_header = true;
                ++i;
            }
        }
    }
    fclose(f);
    if (in_header) { sink.header(hdr); have_record = true; }
    if (have_record) sink.end_record();
    return true;
}

struct PackedText {
    vs_packer *packer = nullptr;
    void *owner = nullptr;             // buffer of a loaded .vsidx
    vs_text_view v{};
    std::vector<std::string> names;
    ~PackedText() { vs_packer_free(packer); vs_free(owner); }
};

bool pack_fasta(const std::string &path, PackedText &t, bool want_names, std::string &err)
{
    t.packer = vs_packer_new();
    if (!t.packer) { err = "out of memory"; return false; }
    int rc = VS_OK;
    FastaSink sink;
    sink.header = [&](const std::string &h) { if (want_names) t.names.push_back(h); };
    sink.seq = [&](const char *s, size_t n) { if (rc == VS_OK) rc = vs_packer_append(t.packer, s, n); };
    sink.end_record = [&]() { if (rc == VS_OK) rc = vs_packer_end_contig(t.packer); };
    if (!read_fasta(path, sink, err)) return false;
    if (rc == VS_OK) rc = vs_packer_finish(t.packer, &t.v);
    if (rc != VS_OK) { err = "packing failed (out of memory?)"; return false; }
    return true;
}

bool read_names(const std::string &path, std::vector<std::string> &names, std::string &err)
{
    FastaSink sink;
    sink.header = [&](const std::string &h) { names.push_back(h); };
    sink.seq = [](const char *, size_t) {};
    sink.end_record = []() {};
    return read_fasta(path, sink, err);
}

// ---- argument parsing (SeqAn ArgumentParser look-alike) ----------------------------------------
struct Opt {
    char s; const char *l; bool required; bool has_value; std::string value; bool seen = false;
    std::vector<std::string> exts;   // valid file extensions (setValidValues)
};

bool has_ext(const std::string &path, const std::vector<std::string> &exts)
{
    if (exts.empty()) return true;
    std::string low = path;
    std::transform(low.begin(), low.end(), low.begin(), [](unsigned char c) { return (char)std::tolower(c); });
    for (const auto &e : exts) {
        std::string suf = "." + e;
        if (low.size() >= suf.size() && low.compare(low.size() - suf.size(), suf.size(), suf) == 0) return true;
    }
    return false;
}

// returns 0 ok, 1 parse error, 2 help/version shown
int parse_args(const char *prog, int argc, char **argv, std::vector<Opt> &opts, const char *desc)
{
    for (int i = 1; i < argc; ++i) {
        std::string a = argv[i];
        if (a == "-h" || a == "--help") {
            printf("%s\n\n%s\n\nOPTIONS\n", prog, desc);
            for (auto &o : opts) printf("    -%c, --%s%s%s\n", o.s, o.l, o.has_value ? " ARG" : "", o.required ? " (required)" : "");
            return 2;
        }
        if (a == "--version") { printf("%s version: varscot-b200 0.1\n", prog); return 2; }
        Opt *hit = nullptr;
        std::string inline_val; bool has_inline = false;
        if (a.size() >= 3 && a[0] == '-' && a[1] == '-') {
            std::string name = a.substr(2);
            size_t eq = name.find('=');
            if (eq != std::string::npos) { inline_val = name.substr(eq + 1); name = name.substr(0, eq); has_inline = true; }
            for (auto &o : opts) if (name == o.l) hit = &o;
        } else if (a.size() == 2 && a[0] == '-') {
            for (auto &o : opts) if (a[1] == o.s) hit = &o;
        }
        if (!hit) { fprintf(stderr, "%s: illegal option -- %s\n", prog, a.c_str()); return 1; }
        if (hit->has_value) {
            if (has_inline) hit->value = inline_val;
            else if (i + 1 < argc) hit->value = argv[++i];
            else { fprintf(stderr, "%s: option requires an argument -- %s\n", prog, a.c_str()); return 1; }
        }
        hit->seen = true;
    }
    for (auto &o : opts) {
        if (o.required && !o.seen) { fprintf(stderr, "%s: option -%c/--%s is required but was not set\n", prog, o.s, o.l); return 1; }
        if (o.seen && !has_ext(o.value, o.exts)) {
            fprintf(stderr, "%s: the given path '%s' does not have a valid file extension for -%c/--%s\n", prog, o.value.c_str(), o.s, o.l);
            return 1;
        }
    }
    return 0;
}

bool parse_int(const std::string &s, long &v)
{
    if (s.empty()) return false;
    char *end = nullptr;
    v = strtol(s.c_str(), &end, 10);
    return end && *end == 0;
}

Opt *find_opt(std::vector<Opt> &opts, char s) { for (auto &o : opts) if (o.s == s) return &o; return nullptr; }

// positions inside a sequence are 32-bit (SAM POS, vs_record.pos): true if every contig holds at most 2^32 bases
bool contigs_fit(const char *prog, const vs_text_view &v)
{
    for (uint32_t c = 0; c < v.n_contigs; ++c)
        if (v.contig_off[c + 1] - v.contig_off[c] > (1ull << 32)) {
            fprintf(stderr, "%s: sequence %u has more than 4 giga bases (2^32); a single sequence may not be longer\n", prog, c);
            return false;
        }
    return true;
}

// Several mapper processes run concurrently (VARSCOT:321-322 runs two, parallel.py:17 up to 48 pipelines).  Each process
// takes an advisory lock (flock on /tmp/varscot_b200_gpu<i>.lock, held until it exits) on the first free device,
// starting at pid % n: concurrent processes land on different GPUs as long as there are free ones, and share them
// evenly afterwards.  VARSCOT_DEVICE pins the choice.
int first_device()
{
    static int chosen = -2;
    if (chosen != -2) return chosen;
    int n = vs_device_count();
    if (n <= 0) return chosen = -1;
    if (const char *e = getenv("VARSCOT_DEVICE")) { int i = atoi(e); if (i >= 0 && i < n) return chosen = i; }
    const int start = (int)((unsigned)getpid() % (unsigned)n);
    for (int j = 0; j < n; ++j) {
        const int d = (start + j) % n;
        const std::string path = "/tmp/varscot_b200_gpu" + std::to_string(d) + ".lock";
        int fd = open(path.c_str(), O_CREAT | O_RDWR, 0666);
        if (fd < 0) continue;
        if (flock(fd, LOCK_EX | LOCK_NB) == 0) return chosen = d;      // the descriptor stays open: the lock lives as long as the process
        close(fd);
    }
    return chosen = start;
}

std::vector<int> choose_devices(uint64_t n_bases)
{
    // small texts stay on ONE device so that concurrent processes spread out; big texts are sharded over several
    int n = vs_device_count();
    std::vector<int> d;
    if (n <= 0) return d;
    const int first = first_device();
    if (getenv("VARSCOT_DEVICE")) { d.push_back(first); return d; }
    int want = (int)std::min<uint64_t>((uint64_t)n, std::max<uint64_t>(1, n_bases / (512ull << 20)));
    if (const char *e = getenv("VARSCOT_GPUS")) { int g = atoi(e); if (g >= 1) want = std::min(g, n); }
    for (int i = 0; i < want; ++i) d.push_back((first + i) % n);
    return d;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
extern "C" int vs_bidir_index_main(int argc, char **argv)
{
    const char *prog = "bidir_index";
    std::vector<Opt> opts = {
        {'G', "genome", true, true, "", false, {"fa", "fasta", "fastq"}},
        {'I', "index", true, true, "", false, {}},
    };
    int pr = parse_args(prog, argc, argv, opts,
                        "VARSCOT - Index Creation (B200 build): packs a multi-sequence FASTA (Dna5: A, C, G, T, N) into the "
                        "bit-sliced text the GPU scan reads. Any total length; each sequence at most 4 giga bases (2^32).");
    if (pr == 2) return 0;
    if (pr == 1) return 1;
    std::string genome = find_opt(opts, 'G')->value, index = find_opt(opts, 'I')->value;
    if (has_ext(genome, {"fastq"})) { fprintf(stderr, "%s: FASTQ input is not supported by this build; convert to FASTA\n", prog); return 1; }
    PackedText t;
    std::string err;
    const auto t0 = std::chrono::steady_clock::now();
    if (!pack_fasta(genome, t, true, err)) { fprintf(stderr, "%s: %s\n", prog, err.c_str()); return 1; }
    const auto t1 = std::chrono::steady_clock::now();
    if (!contigs_fit(prog, t.v)) return 1;
    printf("Number of sequences: %u\n", t.v.n_contigs);
    fflush(stdout);
    if (vs_text_save(index.c_str(), &t.v) != VS_OK) {
        fprintf(stderr, "%s: %s\n", prog, vs_last_error(nullptr));
        return 1;
    }
    // contig ids next to the packed text (<prefix>.vsnames, one header line per contig): bidir_mapping then does not have
    // to re-read a multi-gigabyte FASTA just for its ids (the reference does, bidir_mapping.cpp:272-280)
    if (FILE *nf = fopen((index + ".vsnames").c_str(), "wb")) {
        for (const std::string &n : t.names) { fwrite(n.data(), 1, n.size(), nf); fputc('\n', nf); }
        fclose(nf);
    }
    if (getenv("VARSCOT_VERBOSE"))
        fprintf(stderr, "%s: packed %llu bases in %.2f s, wrote the index in %.2f s\n", prog, (unsigned long long)t.v.n_bases,
                std::chrono::duration<double>(t1 - t0).count(), std::chrono::duration<double>(std::chrono::steady_clock::now() - t1).count());
    printf("Index created successfully\n");
    return 0;
}

extern "C" int vs_bidir_mapping_main(int argc, char **argv)
{
    const char *prog = "bidir_mapping";
    std::vector<Opt> opts = {
        {'G', "genome", true, true, "", false, {"fa", "fasta"}},
        {'I', "index", true, true, "", false, {}},
        {'R', "reads", true, true, "", false, {"fa", "fasta"}},
        {'M', "mismatches", true, true, "", false, {}},
        {'T', "threads", false, true, "1", false, {}},
        {'O', "output", false, true, "", false, {"sam", "bam"}},
        {'P', "pam", false, true, "", false, {}},
        {'S', "md-style", false, true, "seqan", false, {}},     // extension: seqan | samtools (SURVEY.md R9)
    };
    int pr = parse_args(prog, argc, argv, opts,
                        "Read mapper for CRISPR-Cas9 off-targets (B200 build). Only supports Dna4 reads (everything else than ACGT "
                        "will be converted to A). All reads must have the same length (23). Texts of any total length; each sequence at "
                        "most 4 giga bases (2^32).");
    if (pr == 2) return 0;
    if (pr == 1) return 1;
    long mism = 0, threads = 1;
    if (!parse_int(find_opt(opts, 'M')->value, mism)) { fprintf(stderr, "%s: the given value '%s' for -M is not an integer\n", prog, find_opt(opts, 'M')->value.c_str()); return 1; }
    if (!parse_int(find_opt(opts, 'T')->value, threads)) { fprintf(stderr, "%s: the given value for -T is not an integer\n", prog); return 1; }
    if (mism < 0 || mism > 8) { fprintf(stderr, "Error: Maximum number of mismatches must lie between 0 and 8.\n"); return 1; }
    std::string genome = find_opt(opts, 'G')->value, index = find_opt(opts, 'I')->value, reads = find_opt(opts, 'R')->value;
    std::string output = find_opt(opts, 'O')->value, pam = find_opt(opts, 'P')->value, mdst = find_opt(opts, 'S')->value;
    int md_style = mdst == "samtools" ? VS_MD_SAMTOOLS : VS_MD_SEQAN;

    // additional PAM (bidir_mapping.cpp:240-247): a Dna5String compared with the 2-base window end, so only a
    // two-letter ACGT string can ever match anything
    int extra_pam = -1;
    if (!pam.empty()) {
        auto code = [](char c) { switch (std::toupper((unsigned char)c)) { case 'A': return 0; case 'C': return 1; case 'G': return 2; case 'T': case 'U': return 3; default: return 4; } };
        if (pam.size() == 2 && code(pam[0]) < 4 && code(pam[1]) < 4) extra_pam = 4 * code(pam[0]) + code(pam[1]);
        else fprintf(stderr, "%s: warning: additional PAM '%s' can never match a 2-base window without N; ignored\n", prog, pam.c_str());
    }

    // CUDA context creation takes 0.3-4 s: start it now, in the background, on the device a small text will use, and
    // read the inputs meanwhile (choose_devices() picks pid % n_gpus first)
    std::thread warm([] {
        const int dev = first_device();
        if (dev >= 0) vs_warmup_device(dev);
    });
    struct Joiner { std::thread &t; ~Joiner() { if (t.joinable()) t.join(); } } joiner{warm};

    // reads: StringSet<DnaString> (bidir_mapping.cpp:256,263-264): non-ACGT -> A
    std::vector<std::string> ids;
    std::vector<uint8_t> guides;
    {
        std::string cur, err;
        FastaSink sink;
        sink.header = [&](const std::string &h) { ids.push_back(h); cur.clear(); };
        sink.seq = [&](const char *s, size_t n) { for (size_t i = 0; i < n; ++i) if (!isspace((unsigned char)s[i])) cur.push_back(s[i]); };
        bool bad = false;
        sink.end_record = [&]() {
            if (cur.size() != VS_GLEN) { bad = true; return; }
            for (char c : cur) {
                uint8_t v;
                switch (std::toupper((unsigned char)c)) { case 'C': v = 1; break; case 'G': v = 2; break; case 'T': case 'U': v = 3; break; default: v = 0; }
                guides.push_back(v);
            }
        };
        if (!read_fasta(reads, sink, err)) { fprintf(stderr, "%s: %s\n", prog, err.c_str()); return 1; }
        if (bad) { fprintf(stderr, "%s: all reads must be %d nt long (guide + PAM)\n", prog, VS_GLEN); return 1; }
    }
    const auto tm0 = std::chrono::steady_clock::now();
    printf("Reads loaded (total: %zu).\n", ids.size());
    fflush(stdout);

    // "index": the packed text cached by bidir_index at the -I prefix; if it is absent or unreadable, pack -G now
    PackedText t;
    std::string err;
    bool from_cache = vs_text_load(index.c_str(), &t.v, &t.owner) == VS_OK;
    if (from_cache) {
        // contig ids: from <index>.vsnames when bidir_index left one that matches, else from the genome FASTA with the
        // sequences discarded (bidir_mapping.cpp:272-280)
        if (FILE *nf = fopen((index + ".vsnames").c_str(), "rb")) {
            char *line = nullptr; size_t cap = 0; ssize_t len;
            while ((len = getline(&line, &cap, nf)) >= 0) {
                while (len > 0 && (line[len - 1] == '\n' || line[len - 1] == '\r')) --len;
                t.names.emplace_back(line, (size_t)len);
            }
            free(line);
            fclose(nf);
            if (t.names.size() != t.v.n_contigs) t.names.clear();
        }
        if (t.names.empty() && !read_names(genome, t.names, err)) { fprintf(stderr, "%s: %s\n", prog, err.c_str()); return 1; }
        if (t.names.size() != t.v.n_contigs) {
            fprintf(stderr, "%s: index %s.vsidx has %u sequences but %s has %zu; re-run bidir_index\n", prog, index.c_str(), t.v.n_contigs, genome.c_str(), t.names.size());
            return 1;
        }
    } else {
        fprintf(stderr, "%s: note: no packed text at %s.vsidx (%s); packing %s now\n", prog, index.c_str(), vs_last_error(nullptr), genome.c_str());
        if (!pack_fasta(genome, t, true, err)) { fprintf(stderr, "%s: %s\n", prog, err.c_str()); return 1; }
    }
    if (!contigs_fit(prog, t.v)) return 1;
    printf("Index loaded.\n");
    fflush(stdout);
    const auto tm1 = std::chrono::steady_clock::now();

    // output is opened only after all work in the reference (bidir_mapping.cpp:298-305); failing early is equivalent for the caller
    FILE *out = fopen(output.c_str(), "wb");
    if (!out) { fprintf(stderr, "ERROR: Could not open output path.\n"); return 1; }

    // the scan: every device resolves its hits to (contig, pos), sorts them into the reference's emission order and reads each
    // hit's genome window; the host merges the shards' lists a range of guides at a time, applies the primary / secondary rule and
    // formats the range's SAM on the -T host threads (MD:Z from the windows) while the devices score the next range.
    // VARSCOT_RECORDS_PER_DELIVERY: records per range (0 = the library's default).
    const int host_threads = (int)std::min<long>(64, std::max<long>(1, threads));
    const uint32_t n_guides = (uint32_t)ids.size();
    struct Writer {
        FILE *out;
        const std::vector<std::string> &ids, &names;
        const std::vector<uint8_t> &guides;
        int md_style, host_threads;
        bool write_failed = false;
        uint64_t deliveries = 0, largest = 0;
        std::vector<std::string> parts;
        // SAM text: batches of records are formatted by the host threads into per-thread buffers and written in order
        int write(const vs_record *rec, const uint64_t *win, uint64_t n)
        {
            ++deliveries;
            largest = std::max(largest, n);
            const size_t batch = (size_t)host_threads * 65536;
            parts.resize((size_t)host_threads);
            for (size_t b0 = 0; b0 < n; b0 += batch) {
                const size_t b1 = std::min<size_t>(n, b0 + batch);
                auto format = [&](int ti) {
                    std::string &o = parts[(size_t)ti];
                    o.clear();
                    const size_t r0 = b0 + (b1 - b0) * (size_t)ti / (size_t)host_threads, r1 = b0 + (b1 - b0) * (size_t)(ti + 1) / (size_t)host_threads;
                    std::vector<char> buf(1 << 12);
                    for (size_t i = r0; i < r1; ++i) {
                        const vs_record &r = rec[i];
                        char md[64];
                        const uint8_t *g = guides.data() + (size_t)r.guide * VS_GLEN;
                        vs_md_from_window(win[i], g, (r.flag >> 4) & 1, md_style, md);
                        const std::string &qn = ids[r.guide], &rn = names[r.contig];
                        if (buf.size() < qn.size() + rn.size() + 256) buf.resize(qn.size() + rn.size() + 256);
                        int len = vs_format_sam(&r, qn.c_str(), rn.c_str(), g, md, buf.data(), buf.size());
                        if (len > 0) o.append(buf.data(), (size_t)len);
                    }
                };
                if (host_threads == 1) format(0);
                else {
                    std::vector<std::thread> th;
                    for (int ti = 0; ti < host_threads; ++ti) th.emplace_back(format, ti);
                    for (auto &x : th) x.join();
                }
                for (const std::string &o : parts)
                    if (!o.empty() && fwrite(o.data(), 1, o.size(), out) != o.size()) { write_failed = true; return 1; }
            }
            return 0;
        }
        static int sink(void *user, const vs_record *rec, const uint64_t *win, uint64_t n, uint32_t, uint32_t)
        {
            return static_cast<Writer *>(user)->write(rec, win, n);
        }
    } writer{out, ids, t.names, guides, md_style, host_threads};
    uint64_t coll = 0;
    if (n_guides && t.v.n_bases) {
        std::vector<int> devices = choose_devices(t.v.n_bases);
        if (devices.empty()) { fprintf(stderr, "%s: no usable CUDA device: %s (this build has no CPU path)\n", prog, vs_last_error(nullptr)); fclose(out); return 1; }
        const char *rpd = getenv("VARSCOT_RECORDS_PER_DELIVERY");
        vs_scan_stats st;
        int rc = vs_map_records_stream(&t.v, guides.data(), n_guides, (int)mism, extra_pam, devices.data(), (int)devices.size(), host_threads,
                                       rpd ? strtoull(rpd, nullptr, 10) : 0, 1, &Writer::sink, &writer, &coll, &st);
        if (writer.write_failed) { fprintf(stderr, "%s: write error\n", prog); fclose(out); return 1; }
        if (rc != VS_OK) { fprintf(stderr, "%s: scan failed: %s\n", prog, vs_last_error(nullptr)); fclose(out); return 1; }
        if (getenv("VARSCOT_VERBOSE"))
            for (int dv : devices) fprintf(stderr, "%s: scanning on device %d\n", prog, dv);
        if (getenv("VARSCOT_VERBOSE"))
            fprintf(stderr, "%s: %zu device(s), %.3f ms upload+scan (extract %.3f, score %.3f, resolve+sort %.3f; %.1f MB H2D), %llu candidates, %llu hits, "
                            "%llu deliveries (largest %llu records)\n", prog,
                    devices.size(), st.total_ms, st.extract_ms, st.score_ms, st.resolve_ms, st.h2d_bytes / 1e6,
                    (unsigned long long)(st.n_cand_fwd + st.n_cand_rev), (unsigned long long)st.n_hits, (unsigned long long)writer.deliveries,
                    (unsigned long long)writer.largest);
    }
    const auto tm2 = std::chrono::steady_clock::now();
    if (coll) fprintf(stderr, "%s: note: %llu records share a (contig id mod 65536, position) key; the reference's uint16 map key would have kept one of each\n", prog, (unsigned long long)coll);
    if (fclose(out) != 0) { fprintf(stderr, "%s: write error\n", prog); return 1; }
    if (getenv("VARSCOT_VERBOSE")) {
        auto sec = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double>(b - a).count(); };
        fprintf(stderr, "%s: wall: load %.3f s, device (context + upload + scan) overlapped with resolve + SAM %.3f s, close %.3f s\n", prog,
                sec(tm0, tm1), sec(tm1, tm2), sec(tm2, std::chrono::steady_clock::now()));
    }
    return 0;
}
