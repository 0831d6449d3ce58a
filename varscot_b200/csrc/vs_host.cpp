// varscot_b200/csrc/vs_host.cpp — host half of the C ABI in include/varscot_scan.h:
// text packer (the B200 analogue of bidir_index.cpp:36-47), packed-text cache, hit resolution
// (std::map order + primary/secondary flags of bidir_mapping.cpp:154,164-187), MD/SAM formatting
// (:111-123, :177-187) and text sharding across devices.  No search arithmetic lives here: hits
// come only from the CUDA kernels (vs_device.cu); nothing in this file can substitute for them.
#include "vs_internal.h"
#include <algorithm>
#include <atomic>
#include <emmintrin.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <vector>

// ------------------------------------------------------------------------------------------------
// alphabet: SeqAn Dna5 for the text (R6): A,C,G,T(U) case-insensitive -> 0..3, everything else N (4);
// whitespace is not sequence.  SKIP = 255.
namespace {
struct Lut {
    uint8_t t[256];
    Lut()
    {
        for (int i = 0; i < 256; ++i) t[i] = 4;
        t[(int)'A'] = t[(int)'a'] = 0; t[(int)'C'] = t[(int)'c'] = 1; t[(int)'G'] = t[(int)'g'] = 2;
        t[(int)'T'] = t[(int)'t'] = 3; t[(int)'U'] = t[(int)'u'] = 3;
        t[(int)' '] = t[(int)'\t'] = t[(int)'\n'] = t[(int)'\r'] = t[(int)'\v'] = t[(int)'\f'] = 255;
    }
};
const Lut g_lut;
}  // namespace

// Window masks of one word from the N plane and the contig-end plane (n0/e0 = this word, n1/e1 = the next):
//   iv: any N in [p, p+23)  or  any contig end in [p, p+22)   (R1, R3)
//   lw: the window is valid and its last base (p+22) is a contig end   (R4)
static inline vs_masks masks_of(uint32_t n0, uint32_t n1, uint32_t e0, uint32_t e1)
{
    uint64_t N = ((uint64_t)n1 << 32) | n0, E = ((uint64_t)e1 << 32) | e0;
    uint64_t t = N | (N >> 1); t |= t >> 2; t |= t >> 4; t |= t >> 8;      // OR over 16 consecutive
    uint64_t n23 = t | (t >> 7);                                             // OR over 23
    uint64_t e = E | (E >> 1); e |= e >> 2; e |= e >> 4; e |= e >> 8;
    uint64_t e22 = e | (e >> 6);                                             // OR over 22
    vs_masks m;
    m.iv = (uint32_t)(n23 | e22);
    m.lw = (uint32_t)(E >> 22) & ~m.iv;
    return m;
}

extern "C" int vs_masks_from_planes(const uint32_t *nm, const uint32_t *em, uint64_t n_words, vs_masks *out)
{
    if ((!nm || !em || !out) && n_words) return VS_ERR_ARG;
    for (uint64_t w = 0; w < n_words; ++w) out[w] = masks_of(nm[w], nm[w + 1], em[w], em[w + 1]);
    return VS_OK;
}

extern "C" int vs_masks_sparse(const vs_masks *masks, uint64_t n_words, vs_mask_entry **out, uint64_t *n_out)
{
    if (!out || !n_out || (!masks && n_words)) return VS_ERR_ARG;
    uint64_t n = 0;
    for (uint64_t w = 0; w < n_words; ++w) n += (masks[w].iv | masks[w].lw) != 0;
    vs_mask_entry *e = (vs_mask_entry *)malloc((n ? n : 1) * sizeof(vs_mask_entry));
    if (!e) return VS_ERR_NOMEM;
    uint64_t i = 0;
    for (uint64_t w = 0; w < n_words; ++w)
        if (masks[w].iv | masks[w].lw) e[i++] = vs_mask_entry{(uint32_t)w, masks[w].iv, masks[w].lw};
    *out = e; *n_out = n;
    return VS_OK;
}

// Compact mask source (include/varscot_scan.h): runs of equal non-zero words for the N plane; for the contig-end plane
// a decision per block of VS_EM_BLOCK words: as one code byte per word (+ runs for the words with several bits) when
// that is smaller than listing the block's non-zero words as 12-byte runs.
static void append_run(std::vector<vs_plane_run> &runs, uint64_t w, uint32_t v)
{
    if (!runs.empty() && runs.back().value == v && (uint64_t)runs.back().word + runs.back().count == w) runs.back().count++;
    else runs.push_back(vs_plane_run{(uint32_t)w, 1u, v});
}

static int build_mask_source(const uint32_t *nm, const uint32_t *em, uint64_t n_words, std::vector<vs_plane_run> &nm_runs,
                             std::vector<vs_plane_run> &em_runs, std::vector<uint8_t> &em_dense, std::vector<uint8_t> &em_code)
{
    const uint64_t n = n_words + 1, n_blocks = (n + VS_EM_BLOCK - 1) / VS_EM_BLOCK;
    try {
        nm_runs.clear(); em_runs.clear();
        em_dense.assign(n_blocks, 0);
        em_code.assign(n, (uint8_t)VS_EM_NONE);
        for (uint64_t w = 0; w < n; ++w)
            if (nm[w]) append_run(nm_runs, w, nm[w]);
        std::vector<vs_plane_run> all, multi;
        for (uint64_t b = 0; b < n_blocks; ++b) {
            const uint64_t w0 = b * VS_EM_BLOCK, w1 = std::min<uint64_t>(n, w0 + VS_EM_BLOCK);
            all.clear(); multi.clear();
            for (uint64_t w = w0; w < w1; ++w)
                if (em[w]) {
                    append_run(all, w, em[w]);
                    if (em[w] & (em[w] - 1)) append_run(multi, w, em[w]);
                }
            const bool coded = all.size() * sizeof(vs_plane_run) > (w1 - w0) + multi.size() * sizeof(vs_plane_run);
            em_dense[b] = coded ? 1 : 0;
            if (coded)
                for (uint64_t w = w0; w < w1; ++w)
                    if (em[w] && !(em[w] & (em[w] - 1))) em_code[w] = (uint8_t)__builtin_ctz(em[w]);
            const std::vector<vs_plane_run> &keep = coded ? multi : all;
            em_runs.insert(em_runs.end(), keep.begin(), keep.end());
        }
    } catch (...) { return VS_ERR_NOMEM; }
    return VS_OK;
}

extern "C" int vs_mask_source_build(const uint32_t *nm, const uint32_t *em, uint64_t n_words, vs_mask_source *out)
{
    if (!nm || !em || !out) return VS_ERR_ARG;
    memset(out, 0, sizeof(*out));
    std::vector<vs_plane_run> nr, er;
    std::vector<uint8_t> ed, ec;
    int r = build_mask_source(nm, em, n_words, nr, er, ed, ec);
    if (r != VS_OK) return r;
    out->em_code = (uint8_t *)malloc(ec.size() ? ec.size() : 1);
    out->em_dense = (uint8_t *)malloc(ed.size() ? ed.size() : 1);
    out->nm_runs = (vs_plane_run *)malloc((nr.size() ? nr.size() : 1) * sizeof(vs_plane_run));
    out->em_runs = (vs_plane_run *)malloc((er.size() ? er.size() : 1) * sizeof(vs_plane_run));
    if (!out->em_code || !out->em_dense || !out->nm_runs || !out->em_runs) { vs_mask_source_free(out); return VS_ERR_NOMEM; }
    if (!ec.empty()) memcpy(out->em_code, ec.data(), ec.size());
    if (!ed.empty()) memcpy(out->em_dense, ed.data(), ed.size());
    if (!nr.empty()) memcpy(out->nm_runs, nr.data(), nr.size() * sizeof(vs_plane_run));
    if (!er.empty()) memcpy(out->em_runs, er.data(), er.size() * sizeof(vs_plane_run));
    out->n_nm_runs = nr.size(); out->n_em_runs = er.size(); out->n_em_blocks = ed.size();
    return VS_OK;
}

extern "C" void vs_mask_source_free(vs_mask_source *s)
{
    if (!s) return;
    free(s->em_code); free(s->em_dense); free(s->nm_runs); free(s->em_runs);
    memset(s, 0, sizeof(*s));
}

struct vs_packer {
    std::vector<vs_bases> bases;
    std::vector<uint32_t> nm, em;
    std::vector<vs_masks> masks;
    std::vector<vs_mask_entry> sparse;
    std::vector<vs_plane_run> nm_runs, em_runs;      // compact mask source
    std::vector<uint8_t> em_dense, em_code;
    std::vector<uint64_t> off{0};
    uint64_t n = 0;
    bool finalized = false;
};

extern "C" vs_packer *vs_packer_new(void) { return new (std::nothrow) vs_packer(); }
extern "C" void vs_packer_free(vs_packer *p) { delete p; }

extern "C" int vs_packer_append(vs_packer *p, const char *chars, size_t len)
{
    if (!p || (!chars && len)) return VS_ERR_ARG;
    if (p->finalized) { vs_set_last_error("vs_packer_append: packer already finished"); return VS_ERR_ARG; }
    uint64_t need = ((p->n + len + 31) >> 5) + 1;
    if (p->bases.size() < need) {
        try {
            uint64_t cap = std::max<uint64_t>(need, p->bases.size() * 2);
            p->bases.resize(cap, vs_bases{0, 0}); p->nm.resize(cap, 0u); p->em.resize(cap, 0u);
        } catch (...) { return VS_ERR_NOMEM; }
    }
    vs_bases *B = p->bases.data();
    uint32_t *NM = p->nm.data();
    uint64_t n = p->n;
    size_t i = 0;
    // SSE2 fast path: 16 characters at a time when none of them is whitespace (a FASTA line is 60-80 such characters)
    const __m128i fold = _mm_set1_epi8((char)0xDF), cA = _mm_set1_epi8('A'), cC = _mm_set1_epi8('C'), cG = _mm_set1_epi8('G'),
                  cT = _mm_set1_epi8('T'), cU = _mm_set1_epi8('U'), lim = _mm_set1_epi8(0x21);
    while (i + 16 <= len) {
        const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i *>(chars + i));
        // characters below 0x21 (whitespace, control) or above 0x7F end the clean run of this block
        const uint32_t stop = (uint32_t)_mm_movemask_epi8(_mm_cmpgt_epi8(lim, c));
        const uint32_t k = stop ? (uint32_t)__builtin_ctz(stop) : 16u;
        if (k) {
            const uint32_t keep = (1u << k) - 1u;
            const __m128i u = _mm_and_si128(c, fold);
            const __m128i tu = _mm_or_si128(_mm_cmpeq_epi8(u, cT), _mm_cmpeq_epi8(u, cU));
            const __m128i isC = _mm_cmpeq_epi8(u, cC), isG = _mm_cmpeq_epi8(u, cG);
            const uint32_t valid = (uint32_t)_mm_movemask_epi8(_mm_or_si128(_mm_or_si128(_mm_cmpeq_epi8(u, cA), isC), _mm_or_si128(isG, tu)));
            const uint64_t h = (uint64_t)((uint32_t)_mm_movemask_epi8(_mm_or_si128(isG, tu)) & keep) << (n & 31);
            const uint64_t l = (uint64_t)((uint32_t)_mm_movemask_epi8(_mm_or_si128(isC, tu)) & keep) << (n & 31);
            const uint64_t m = (uint64_t)(~valid & keep) << (n & 31);
            const uint64_t w = n >> 5;
            B[w].hi |= (uint32_t)h; B[w].lo |= (uint32_t)l; NM[w] |= (uint32_t)m;
            if ((n & 31) + k > 32) { B[w + 1].hi |= (uint32_t)(h >> 32); B[w + 1].lo |= (uint32_t)(l >> 32); NM[w + 1] |= (uint32_t)(m >> 32); }
            n += k; i += k;
        }
        if (stop) {                                         // the stopping character itself: skip whitespace, anything else is N
            if (g_lut.t[(uint8_t)chars[i]] != 255) { NM[n >> 5] |= 1u << (n & 31); ++n; }
            ++i;
        }
    }
    for (; i < len; ++i) {
        uint8_t c = g_lut.t[(uint8_t)chars[i]];
        if (c == 255) continue;
        uint32_t bit = 1u << (n & 31);
        if (c & 2) B[n >> 5].hi |= bit;
        if (c & 1) B[n >> 5].lo |= bit;
        if (c & 4) NM[n >> 5] |= bit;
        ++n;
    }
    p->n = n;
    return VS_OK;
}

extern "C" int vs_packer_end_contig(vs_packer *p)
{
    if (!p || p->finalized) return VS_ERR_ARG;
    if (p->n > p->off.back()) {
        uint64_t last = p->n - 1;
        p->em[last >> 5] |= 1u << (last & 31);
    }
    p->off.push_back(p->n);
    return VS_OK;
}

extern "C" int vs_packer_finish(vs_packer *p, vs_text_view *out)
{
    if (!p || !out) return VS_ERR_ARG;
    const uint64_t nw = (p->n + 31) >> 5;
    if (!p->finalized) {
        try {
            p->bases.resize(nw + 1, vs_bases{0, 0}); p->nm.resize(nw + 1, 0u); p->em.resize(nw + 1, 0u);
            p->bases[nw] = vs_bases{0, 0};
            if (p->n & 31) p->nm[nw - 1] |= ~0u << (p->n & 31);     // padding past the end reads as N
            p->nm[nw] = ~0u; p->em[nw] = 0;
            p->masks.resize(nw);
            vs_masks_from_planes(p->nm.data(), p->em.data(), nw, p->masks.data());
            for (uint64_t w = 0; w < nw; ++w)
                if (p->masks[w].iv | p->masks[w].lw) p->sparse.push_back(vs_mask_entry{(uint32_t)w, p->masks[w].iv, p->masks[w].lw});
            if (build_mask_source(p->nm.data(), p->em.data(), nw, p->nm_runs, p->em_runs, p->em_dense, p->em_code) != VS_OK) return VS_ERR_NOMEM;
            std::vector<uint32_t>().swap(p->nm);
            std::vector<uint32_t>().swap(p->em);
        } catch (...) { return VS_ERR_NOMEM; }
        p->finalized = true;
    }
    out->n_bases = p->n; out->n_words = nw; out->n_contigs = (uint32_t)(p->off.size() - 1); out->reserved = 0;
    out->contig_off = p->off.data(); out->bases = p->bases.data(); out->masks = p->masks.data();
    out->sparse = p->sparse.data(); out->n_sparse = p->sparse.size();
    out->em_code = p->em_code.data(); out->em_dense = p->em_dense.data();
    out->nm_runs = p->nm_runs.data(); out->em_runs = p->em_runs.data();
    out->n_nm_runs = p->nm_runs.size(); out->n_em_runs = p->em_runs.size();
    return VS_OK;
}

extern "C" int vs_pack_text_planes(const char *ascii, uint64_t n_bases, const uint64_t *contig_off, uint32_t n_contigs,
                                   vs_bases *out_bases, uint32_t *out_nm, uint32_t *out_em)
{
    if (!out_bases || !out_nm || !out_em || (!ascii && n_bases) || (!contig_off && n_contigs)) return VS_ERR_ARG;
    if (n_contigs && (contig_off[0] != 0 || contig_off[n_contigs] != n_bases)) {
        vs_set_last_error("vs_pack_text: offsets must start at 0 and end at n_bases");
        return VS_ERR_ARG;
    }
    const uint64_t nw = (n_bases + 31) >> 5;
    memset(out_bases, 0, (nw + 1) * sizeof(vs_bases));
    memset(out_nm, 0, (nw + 1) * sizeof(uint32_t));
    memset(out_em, 0, (nw + 1) * sizeof(uint32_t));
    for (uint64_t i = 0; i < n_bases; ++i) {
        uint8_t c = g_lut.t[(uint8_t)ascii[i]];
        if (c == 255) c = 4;              // whitespace inside a pre-split text is just a non-base
        uint32_t bit = 1u << (i & 31);
        if (c & 2) out_bases[i >> 5].hi |= bit;
        if (c & 1) out_bases[i >> 5].lo |= bit;
        if (c & 4) out_nm[i >> 5] |= bit;
    }
    for (uint32_t c = 0; c < n_contigs; ++c) {
        if (contig_off[c + 1] < contig_off[c]) { vs_set_last_error("vs_pack_text: offsets must be non-decreasing"); return VS_ERR_ARG; }
        if (contig_off[c + 1] > contig_off[c]) {
            uint64_t last = contig_off[c + 1] - 1;
            out_em[last >> 5] |= 1u << (last & 31);
        }
    }
    if (n_bases & 31) out_nm[nw - 1] |= ~0u << (n_bases & 31);     // padding past the end reads as N
    out_nm[nw] = ~0u;
    return VS_OK;
}

extern "C" int vs_pack_text(const char *ascii, uint64_t n_bases, const uint64_t *contig_off, uint32_t n_contigs,
                            vs_bases *out_bases, vs_masks *out_masks)
{
    if (!out_masks && n_bases) return VS_ERR_ARG;
    const uint64_t nw = (n_bases + 31) >> 5;
    std::vector<uint32_t> nm, em;
    try { nm.assign(nw + 1, 0u); em.assign(nw + 1, 0u); } catch (...) { return VS_ERR_NOMEM; }
    int r = vs_pack_text_planes(ascii, n_bases, contig_off, n_contigs, out_bases, nm.data(), em.data());
    if (r != VS_OK) return r;
    return vs_masks_from_planes(nm.data(), em.data(), nw, out_masks);
}

// ------------------------------------------------------------------------------------------------
// packed-text cache: <prefix>.vsidx.  Format 003: header, source header, offsets, bases, then
//   * a view WITH a compact mask source (what bidir_index writes): em_code, em_dense, nm_runs, em_runs — the window masks
//     are not stored; the device computes them during the upload (the file is half the size: 0.27 B per base);
//   * a view without one: masks, sparse masks.
// All sections are 16-byte aligned.  (Format 002 of round 1 — no source header — is no longer read: re-run bidir_index.)
namespace {
struct IdxHeader {
    char magic[8];
    uint64_t n_bases;
    uint64_t n_sparse;
    uint32_t n_contigs;
    uint32_t flags;          // 003: bit 0 = compact mask source stored (and masks / sparse masks are not)
};
struct IdxSourceHeader {    // 003 only, directly after IdxHeader
    uint64_t n_nm_runs, n_em_runs;
};
const char IDX_MAGIC3[8] = {'V', 'S', 'I', 'D', 'X', '0', '0', '3'};
inline uint64_t pad16(uint64_t x) { return (x + 15) & ~15ull; }
inline bool has_source(const vs_text_view *t) { return t->em_code && t->em_dense; }

// planes from a compact mask source (the host twin of k_fill_runs / k_expand_em_code), then the masks
int masks_from_source(const vs_text_view *t, vs_masks *out)
{
    const uint64_t n = t->n_words + 1;
    std::vector<uint32_t> nm, em;
    try { nm.assign(n, 0u); em.assign(n, 0u); } catch (...) { return VS_ERR_NOMEM; }
    auto fill = [&](const vs_plane_run *r, uint64_t cnt, std::vector<uint32_t> &plane) {
        for (uint64_t i = 0; i < cnt; ++i) {
            if ((uint64_t)r[i].word + r[i].count > n) return false;
            std::fill(plane.begin() + r[i].word, plane.begin() + r[i].word + r[i].count, r[i].value);
        }
        return true;
    };
    if (!fill(t->nm_runs, t->n_nm_runs, nm)) return VS_ERR_IO;
    for (uint64_t w = 0; w < n; ++w)
        if (t->em_dense[w / VS_EM_BLOCK] && t->em_code[w] < 32) em[w] = 1u << t->em_code[w];
    if (!fill(t->em_runs, t->n_em_runs, em)) return VS_ERR_IO;
    return vs_masks_from_planes(nm.data(), em.data(), t->n_words, out);
}
}  // namespace

// window masks of a view on the host: copied, or rebuilt from the compact mask source when the view carries no masks
extern "C" int vs_text_masks(const vs_text_view *t, vs_masks *out)
{
    if (!t || (!out && t->n_words)) return VS_ERR_ARG;
    if (t->masks) { memcpy(out, t->masks, t->n_words * sizeof(vs_masks)); return VS_OK; }
    if (!has_source(t)) return VS_ERR_ARG;
    return masks_from_source(t, out);
}

// vs_text_load maps the cache file; vs_free() has to know which pointers are mappings (and how long they are)
namespace {
std::mutex g_maps_mu;
std::unordered_map<void *, size_t> g_maps;
}

extern "C" int vs_text_save(const char *prefix, const vs_text_view *t)
{
    if (!prefix || !t || !t->contig_off || (!t->bases) || (!t->masks && !has_source(t) && t->n_words)) return VS_ERR_ARG;
    std::string path = std::string(prefix) + ".vsidx";
    FILE *f = fopen(path.c_str(), "wb");
    if (!f) { vs_set_last_error(("cannot open " + path + " for writing").c_str()); return VS_ERR_IO; }
    const bool src = has_source(t);
    vs_mask_entry *tmp = nullptr;
    const vs_mask_entry *sp = t->sparse;
    uint64_t nsp = t->n_sparse;
    if (src) { sp = nullptr; nsp = 0; }
    else if (!sp && t->n_words) { if (vs_masks_sparse(t->masks, t->n_words, &tmp, &nsp) != VS_OK) { fclose(f); return VS_ERR_NOMEM; } sp = tmp; }
    IdxHeader h;
    memcpy(h.magic, IDX_MAGIC3, 8);
    h.n_bases = t->n_bases; h.n_sparse = nsp; h.n_contigs = t->n_contigs; h.flags = src ? 1u : 0u;
    IdxSourceHeader sh{src ? t->n_nm_runs : 0, src ? t->n_em_runs : 0};
    static const char zeros[16] = {0};
    auto put = [&](const void *p, uint64_t bytes) {
        bool ok = bytes == 0 || fwrite(p, 1, bytes, f) == bytes;
        uint64_t pad = pad16(bytes) - bytes;
        return ok && (pad == 0 || fwrite(zeros, 1, pad, f) == pad);
    };
    bool ok = put(&h, sizeof(h)) && put(&sh, sizeof(sh)) && put(t->contig_off, ((uint64_t)t->n_contigs + 1) * 8) &&
              put(t->bases, (t->n_words + 1) * sizeof(vs_bases));
    if (ok && src)
        ok = put(t->em_code, t->n_words + 1) && put(t->em_dense, (t->n_words + VS_EM_BLOCK) / VS_EM_BLOCK) &&
             put(t->nm_runs, sh.n_nm_runs * sizeof(vs_plane_run)) && put(t->em_runs, sh.n_em_runs * sizeof(vs_plane_run));
    else if (ok)
        ok = put(t->masks, t->n_words * sizeof(vs_masks)) && put(sp, nsp * sizeof(vs_mask_entry));
    ok = (fclose(f) == 0) && ok;
    free(tmp);
    if (!ok) { vs_set_last_error(("short write to " + path).c_str()); return VS_ERR_IO; }
    return VS_OK;
}

// The cache file is MAPPED, not read: the view points into the page cache, nothing is copied and nothing is built on the host
// (a file written by bidir_index holds bases + mask source; the device computes the window masks during the upload).  A mapper
// process runs one scan and exits, so the text is deliberately not page-locked: locking 1 GB costs several times what the
// pageable H2D path loses (measured with the page-locked variant of round 2: 1.8 s of load for a 0.07 s scan).
extern "C" int vs_text_load(const char *prefix, vs_text_view *out, void **owner)
{
    if (!prefix || !out || !owner) return VS_ERR_ARG;
    *owner = nullptr;
    memset(out, 0, sizeof(*out));
    std::string path = std::string(prefix) + ".vsidx";
    int fd = open(path.c_str(), O_RDONLY);
    if (fd < 0) { vs_set_last_error(("cannot open " + path).c_str()); return VS_ERR_IO; }
    struct stat sb;
    if (fstat(fd, &sb) != 0 || (uint64_t)sb.st_size < pad16(sizeof(IdxHeader)) + pad16(sizeof(IdxSourceHeader))) {
        close(fd); vs_set_last_error((path + " is not a VSIDX003 packed text").c_str()); return VS_ERR_IO;
    }
    const uint64_t fsize = (uint64_t)sb.st_size;
    // MAP_POPULATE: the page tables are filled here — in the executables while the CUDA context is being created on another thread —
    // instead of fault by fault inside the driver's staging copies of the upload
    char *base = (char *)mmap(nullptr, fsize, PROT_READ, MAP_PRIVATE | MAP_POPULATE, fd, 0);
    if (base == MAP_FAILED) base = (char *)mmap(nullptr, fsize, PROT_READ, MAP_PRIVATE, fd, 0);
    close(fd);
    if (base == MAP_FAILED) { vs_set_last_error(("cannot map " + path).c_str()); return VS_ERR_IO; }
    auto bad = [&](const std::string &why, int code) { munmap(base, fsize); memset(out, 0, sizeof(*out)); vs_set_last_error((path + why).c_str()); return code; };
    IdxHeader h;
    IdxSourceHeader sh;
    memcpy(&h, base, sizeof(h));
    if (memcmp(h.magic, IDX_MAGIC3, 8) != 0) return bad(" is not a VSIDX003 packed text", VS_ERR_IO);
    memcpy(&sh, base + pad16(sizeof(h)), sizeof(sh));
    const bool src = (h.flags & 1u) != 0;
    const uint64_t nw = (h.n_bases + 31) >> 5;
    const uint64_t s_off = pad16(((uint64_t)h.n_contigs + 1) * 8), s_b = pad16((nw + 1) * sizeof(vs_bases));
    const uint64_t s_m = src ? 0 : pad16(nw * sizeof(vs_masks)), s_s = src ? 0 : pad16(h.n_sparse * sizeof(vs_mask_entry));
    const uint64_t s_em = src ? pad16(nw + 1) : 0, s_ed = src ? pad16((nw + VS_EM_BLOCK) / VS_EM_BLOCK) : 0,
                   s_nr = src ? pad16(sh.n_nm_runs * sizeof(vs_plane_run)) : 0, s_er = src ? pad16(sh.n_em_runs * sizeof(vs_plane_run)) : 0;
    const uint64_t data_at = pad16(sizeof(h)) + pad16(sizeof(sh));
    if (data_at + s_off + s_b + s_m + s_s + s_em + s_ed + s_nr + s_er > fsize) return bad(" is truncated", VS_ERR_IO);
    char *p = base + data_at;
    const uint64_t *off = (const uint64_t *)p;
    if (off[h.n_contigs] != h.n_bases) return bad(" is truncated", VS_ERR_IO);
    out->n_bases = h.n_bases; out->n_words = nw; out->n_contigs = h.n_contigs;
    out->contig_off = off;
    out->bases = (const vs_bases *)(p + s_off);
    char *tail = p + s_off + s_b;
    if (src) {
        out->em_code = (const uint8_t *)tail;
        out->em_dense = (const uint8_t *)(tail + s_em);
        out->nm_runs = (const vs_plane_run *)(tail + s_em + s_ed);
        out->em_runs = (const vs_plane_run *)(tail + s_em + s_ed + s_nr);
        out->n_nm_runs = sh.n_nm_runs; out->n_em_runs = sh.n_em_runs;
        // the runs are trusted by the upload: check them here
        bool good = true;
        for (uint64_t i = 0; i < sh.n_nm_runs && good; ++i) good = (uint64_t)out->nm_runs[i].word + out->nm_runs[i].count <= nw + 1;
        for (uint64_t i = 0; i < sh.n_em_runs && good; ++i) good = (uint64_t)out->em_runs[i].word + out->em_runs[i].count <= nw + 1;
        if (!good) return bad(" holds a corrupt mask source", VS_ERR_IO);
    } else {
        out->masks = (const vs_masks *)tail;
        out->sparse = (const vs_mask_entry *)(tail + s_m);
        out->n_sparse = h.n_sparse;
    }
    { std::lock_guard<std::mutex> lk(g_maps_mu); g_maps[base] = fsize; }
    *owner = base;
    return VS_OK;
}

extern "C" void vs_free(void *p)
{
    if (!p) return;
    size_t len = 0;
    {
        std::lock_guard<std::mutex> lk(g_maps_mu);
        auto it = g_maps.find(p);
        if (it != g_maps.end()) { len = it->second; g_maps.erase(it); }
    }
    if (len) munmap(p, len); else free(p);
}

// ------------------------------------------------------------------------------------------------
// hit resolution
namespace {
struct SortRec {
    uint64_t k1;   // guide << 17 | strand << 16 | (contig & 0xFFFF)
    uint64_t k2;   // pos << 32 | (contig >> 16) << 8 | mm
    uint32_t contig;
};
inline bool operator<(const SortRec &a, const SortRec &b) { return a.k1 != b.k1 ? a.k1 < b.k1 : a.k2 < b.k2; }
}  // namespace

// Hits -> records in the reference's emission order.  Three steps, the first and last parallel over `n_threads`:
//   1. global position -> (contig, pos) by binary search, sort key (guide, strand, id & 0xFFFF, pos, id >> 16);
//   2. counting sort by pass = (guide, strand) (single pass over the keys);
//   3. per pass: sort by the std::map key and walk it with the running-best rule of bidir_mapping.cpp:164-187.  A pass
//      occupies the same index range before and after step 3, so passes are independent.
extern "C" int vs_resolve_hits_mt(const vs_hit *hits, uint64_t n, const uint64_t *contig_off, uint32_t n_contigs,
                                  vs_record *out, uint64_t *key16_collisions, int n_threads)
{
    if ((n && (!hits || !out)) || !contig_off || n_contigs == 0) return n ? VS_ERR_ARG : VS_OK;
    if (key16_collisions) *key16_collisions = 0;
    if (n == 0) return VS_OK;
    if (n_threads < 1) n_threads = 1;
    if ((uint64_t)n_threads > n / 4096 + 1) n_threads = (int)(n / 4096 + 1);
    std::vector<SortRec> v, v2;
    try { v.resize(n); v2.resize(n); } catch (...) { return VS_ERR_NOMEM; }
    const uint64_t *ob = contig_off, *oe = contig_off + n_contigs + 1;
    std::vector<int> bad((size_t)n_threads, 0);
    std::vector<uint64_t> max_pass((size_t)n_threads, 0);
    auto run = [&](auto fn) {
        if (n_threads == 1) { fn(0); return; }
        std::vector<std::thread> th;
        for (int t = 0; t < n_threads; ++t) th.emplace_back(fn, t);
        for (auto &x : th) x.join();
    };
    run([&](int t) {
        const uint64_t b0 = n * (uint64_t)t / (uint64_t)n_threads, b1 = n * (uint64_t)(t + 1) / (uint64_t)n_threads;
        uint64_t mp = 0;
        for (uint64_t i = b0; i < b1; ++i) {
            const uint64_t gp = hits[i].pos;
            // last contig c with off[c] <= gp (empty contigs share an offset; the non-empty one is the last)
            const uint64_t *it = std::upper_bound(ob, oe, gp);
            if (it == ob || it == oe) { bad[(size_t)t] = 1; return; }
            const uint32_t c = (uint32_t)(it - ob - 1);
            const uint32_t pos = (uint32_t)(gp - contig_off[c]);
            const uint32_t info = hits[i].info;
            const uint64_t guide = info >> 8, strand = (info >> 7) & 1, mm = info & 0xF;
            v[i].k1 = (guide << 17) | (strand << 16) | (c & 0xFFFFu);
            v[i].k2 = ((uint64_t)pos << 32) | ((uint64_t)(c >> 16) << 8) | mm;
            v[i].contig = c;
            mp = std::max(mp, (guide << 1) | strand);
        }
        max_pass[(size_t)t] = mp;
    });
    for (int t = 0; t < n_threads; ++t) if (bad[(size_t)t]) { vs_set_last_error("vs_resolve_hits: hit position outside the text"); return VS_ERR_ARG; }
    const uint64_t n_pass = *std::max_element(max_pass.begin(), max_pass.end()) + 1;
    std::vector<uint64_t> start;
    try { start.assign(n_pass + 1, 0); } catch (...) { return VS_ERR_NOMEM; }
    for (uint64_t i = 0; i < n; ++i) start[(v[i].k1 >> 16) + 1]++;
    for (uint64_t p = 0; p < n_pass; ++p) start[p + 1] += start[p];
    {
        std::vector<uint64_t> cur(start.begin(), start.end() - 1);
        for (uint64_t i = 0; i < n; ++i) v2[cur[v[i].k1 >> 16]++] = v[i];
    }
    std::vector<SortRec>().swap(v);
    std::vector<uint64_t> coll((size_t)n_threads, 0);
    std::atomic<uint64_t> next{0};
    run([&](int t) {
        uint64_t c = 0;
        for (;;) {
            const uint64_t p0 = next.fetch_add(64);
            if (p0 >= n_pass) break;
            for (uint64_t p = p0; p < std::min(n_pass, p0 + 64); ++p) {
                const uint64_t i = start[p], j = start[p + 1];
                if (i == j) continue;
                std::sort(v2.begin() + (long)i, v2.begin() + (long)j);
                uint64_t w = i, best = i;
                auto emit = [&](const SortRec &r, uint16_t secondary) {
                    vs_record &o = out[w++];
                    o.guide = (uint32_t)(r.k1 >> 17);
                    o.contig = r.contig;
                    o.pos = (uint32_t)(r.k2 >> 32);
                    o.mm = (uint8_t)(r.k2 & 0xF);
                    o.flag = (uint16_t)(secondary | (((r.k1 >> 16) & 1) ? 16 : 0));
                    o.pad = 0;
                };
                for (uint64_t x = i + 1; x < j; ++x) {
                    if (v2[x].k1 == v2[x - 1].k1 && (v2[x].k2 >> 32) == (v2[x - 1].k2 >> 32)) ++c;   // same (id16, pos): uint16 key collision
                    if ((v2[x].k2 & 0xF) >= (v2[best].k2 & 0xF)) emit(v2[x], 256);
                    else { emit(v2[best], 256); best = x; }
                }
                emit(v2[best], 0);
            }
        }
        coll[(size_t)t] = c;
    });
    if (key16_collisions) for (uint64_t c : coll) *key16_collisions += c;
    return VS_OK;
}

extern "C" int vs_resolve_hits(const vs_hit *hits, uint64_t n, const uint64_t *contig_off, uint32_t n_contigs,
                               vs_record *out, uint64_t *key16_collisions)
{
    return vs_resolve_hits_mt(hits, n, contig_off, n_contigs, out, key16_collisions, 1);
}

// Merge of the device-sorted lists of the shards (vs_scan_resolved).  Every list is ascending in (guide, strand, contig &
// 0xFFFF, pos); the lists are cut at the same pass boundaries into n_threads ranges of passes, each range is gathered
// into its final place in `out`'s index space, sorted when more than one list contributed (or when records tie on the
// 16-bit key: the order among those is by the full contig id), and walked with the running-best rule of
// bidir_mapping.cpp:164-187.
extern "C" int vs_merge_resolved(const vs_loc_hit *const *lists, const uint64_t *counts, int n_lists,
                                 vs_record *out, uint64_t *key16_collisions, int n_threads)
{
    if (key16_collisions) *key16_collisions = 0;
    if (n_lists < 0 || (n_lists && (!lists || !counts))) return VS_ERR_ARG;
    uint64_t total = 0;
    int biggest = 0;
    for (int l = 0; l < n_lists; ++l) {
        if (counts[l] && !lists[l]) return VS_ERR_ARG;
        total += counts[l];
        if (counts[l] > counts[biggest]) biggest = l;
    }
    if (total == 0) return VS_OK;
    if (!out) return VS_ERR_ARG;
    if (n_threads < 1) n_threads = 1;
    if ((uint64_t)n_threads > total / 2048 + 1) n_threads = (int)(total / 2048 + 1);
    auto pass_of = [](const vs_loc_hit &h) { return (uint64_t)(h.info >> 7); };                 // guide << 1 | strand
    // pass boundaries of the thread ranges: quantiles of the biggest list
    std::vector<uint64_t> cut((size_t)n_threads + 1, 0);
    cut[(size_t)n_threads] = ~0ull;
    for (int t = 1; t < n_threads; ++t) cut[(size_t)t] = pass_of(lists[biggest][counts[biggest] * (uint64_t)t / (uint64_t)n_threads]);
    // start of every range in every list (first record whose pass is >= the cut), and in the output
    std::vector<uint64_t> at((size_t)(n_threads + 1) * (size_t)n_lists, 0), out_at((size_t)n_threads + 1, 0);
    for (int t = 0; t <= n_threads; ++t)
        for (int l = 0; l < n_lists; ++l) {
            const vs_loc_hit *b = lists[l], *e = lists[l] + counts[l];
            const uint64_t i = t == n_threads ? counts[l] : (uint64_t)(std::partition_point(b, e, [&](const vs_loc_hit &h) { return pass_of(h) < cut[(size_t)t]; }) - b);
            at[(size_t)t * (size_t)n_lists + (size_t)l] = i;
            out_at[(size_t)t] += i;
        }
    std::vector<uint64_t> coll((size_t)n_threads, 0);
    std::vector<int> rc((size_t)n_threads, VS_OK);
    constexpr uint64_t KEY48 = (1ull << 49) - 1;                                                  // strand, contig & 0xFFFF, pos
    // Per thread: a k-way merge of its ranges of the lists (each ascending; ties on the 16-bit key are not ordered inside a
    // list, so a run of equal keys is collected and ordered by the full contig id before it is emitted), streamed straight
    // into the running-best walk — no copy of the hits, no sort.
    auto work = [&](int t) {
        const uint64_t o0 = out_at[(size_t)t], o1 = out_at[(size_t)t + 1];
        if (o1 == o0) return;
        struct Head { const vs_loc_hit *p, *e; };
        std::vector<Head> heads;
        for (int l = 0; l < n_lists; ++l) {
            const vs_loc_hit *b = lists[l] + at[(size_t)t * (size_t)n_lists + (size_t)l], *e = lists[l] + at[(size_t)(t + 1) * (size_t)n_lists + (size_t)l];
            if (b < e) heads.push_back(Head{b, e});
        }
        uint64_t w = o0, c = 0;
        auto emit = [&](const vs_loc_hit &h, uint16_t secondary) {
            vs_record &o = out[w++];
            o.guide = h.info >> 8;
            o.contig = h.contig;
            o.pos = (uint32_t)h.key;
            o.mm = (uint8_t)(h.info & 0x7F);
            o.flag = (uint16_t)(secondary | ((h.info & 0x80) ? 16 : 0));
            o.pad = 0;
        };
        // running-best walk (bidir_mapping.cpp:164-187), fed one record at a time in emission-key order
        bool have_best = false;
        vs_loc_hit best{};
        uint64_t cur_pass = ~0ull;
        auto feed = [&](const vs_loc_hit &h) {
            const uint64_t p = pass_of(h);
            if (p != cur_pass) {
                if (have_best) emit(best, 0);
                best = h; have_best = true; cur_pass = p;
                return;
            }
            if ((h.info & 0x7F) >= (best.info & 0x7F)) emit(h, 256);
            else { emit(best, 256); best = h; }
        };
        // records sharing (pass, strand, contig & 0xFFFF, pos) — a uint16 key collision, rare — are ordered by the full contig id:
        // one record is held back until the next one shows a different key
        std::vector<vs_loc_hit> ties;
        bool have_prev = false;
        vs_loc_hit prev{};
        uint64_t prev_pass = 0, prev_key = 0;
        auto flush_ties = [&]() {
            if (!ties.empty()) {
                ties.push_back(prev);
                std::sort(ties.begin(), ties.end(), [](const vs_loc_hit &a, const vs_loc_hit &b) { return a.contig < b.contig; });
                c += ties.size() - 1;
                for (const vs_loc_hit &h : ties) feed(h);
                ties.clear();
            } else if (have_prev) feed(prev);
            have_prev = false;
        };
        auto take = [&](const vs_loc_hit &h, uint64_t p, uint64_t k) {
            if (have_prev && p == prev_pass && k == prev_key) { ties.push_back(prev); prev = h; return; }
            flush_ties();
            prev = h; prev_pass = p; prev_key = k; have_prev = true;
        };
        if (heads.size() == 1) {
            for (const vs_loc_hit *p = heads[0].p; p < heads[0].e; ++p) take(*p, pass_of(*p), p->key & KEY48);
        } else {
            // k-way merge by linear selection over the cached keys of the heads (k = number of shards, a handful)
            const size_t k = heads.size();
            std::vector<uint64_t> hp(k), hk(k);
            for (size_t i = 0; i < k; ++i) { hp[i] = pass_of(*heads[i].p); hk[i] = heads[i].p->key & KEY48; }
            size_t live = k;
            while (live) {
                size_t m = 0;
                for (size_t i = 1; i < k; ++i)
                    if (hp[i] < hp[m] || (hp[i] == hp[m] && hk[i] < hk[m])) m = i;
                take(*heads[m].p, hp[m], hk[m]);
                if (++heads[m].p < heads[m].e) { hp[m] = pass_of(*heads[m].p); hk[m] = heads[m].p->key & KEY48; }
                else { hp[m] = ~0ull; hk[m] = ~0ull; --live; }
            }
        }
        flush_ties();
        if (have_best) emit(best, 0);
        coll[(size_t)t] = c;
        if (w != o1) rc[(size_t)t] = VS_ERR_ARG;             // a list was not ascending
    };
    if (n_threads == 1) work(0);
    else {
        std::vector<std::thread> th;
        for (int t = 0; t < n_threads; ++t) th.emplace_back(work, t);
        for (auto &x : th) x.join();
    }
    for (int t = 0; t < n_threads; ++t) if (rc[(size_t)t] != VS_OK) return rc[(size_t)t];
    if (key16_collisions) for (uint64_t c : coll) *key16_collisions += c;
    return VS_OK;
}

static inline int base_at(const vs_bases *bases, uint64_t p)
{
    const vs_bases &w = bases[p >> 5];
    uint32_t b = (uint32_t)(p & 31);
    return (int)(((w.hi >> b) & 1) << 1 | ((w.lo >> b) & 1));     // hits never contain N
}

extern "C" int vs_md_string(const vs_bases *words, uint64_t gpos, const uint8_t *guide, int strand, int md_style, char *out)
{
    if (!words || !guide || !out) return VS_ERR_ARG;
    static const char L[4] = {'A', 'C', 'G', 'T'};
    int n = 0, run = 0;
    bool in_match = false, any = false;
    for (int i = 0; i < VS_GLEN; ++i) {
        int g = strand ? 3 - guide[VS_GLEN - 1 - i] : guide[i];   // pattern of the pass, genome-forward orientation
        int t = base_at(words, gpos + i);
        if (t == g) { ++run; in_match = true; any = true; continue; }
        // mismatch column: genome character (row 0 of the Align at bidir_mapping.cpp:117)
        if (md_style == VS_MD_SAMTOOLS) n += sprintf(out + n, "%d", run);
        else if (in_match) n += sprintf(out + n, "%d", run);
        out[n++] = L[t];
        run = 0; in_match = false; any = true;
    }
    if (md_style == VS_MD_SAMTOOLS || in_match) n += sprintf(out + n, "%d", run);
    (void)any;
    out[n] = 0;
    return VS_OK;
}

extern "C" int vs_format_sam(const vs_record *r, const char *qname, const char *rname, const uint8_t *guide,
                             const char *md, char *buf, size_t buflen)
{
    if (!r || !qname || !rname || !guide || !md || !buf) return -1;
    static const char L[4] = {'A', 'C', 'G', 'T'};
    char seq[VS_GLEN + 1];
    for (int i = 0; i < VS_GLEN; ++i) seq[i] = L[guide[i] & 3];   // SEQ is always the original guide, bidir_mapping.cpp:106-108
    seq[VS_GLEN] = 0;
    int n = snprintf(buf, buflen, "%s\t%u\t%s\t%u\t255\t23M\t*\t0\t0\t%s\tIIIIIIIIIIIIIIIIIIIIIII\tNM:i:%u\tMD:Z:%s\n",
                     qname, (unsigned)r->flag, rname, r->pos + 1u, seq, (unsigned)r->mm, md);
    if (n < 0 || (size_t)n >= buflen) return -1;
    return n;
}

// ------------------------------------------------------------------------------------------------
// sharding across devices: contiguous word ranges, no collective, hits concatenated on the host
namespace vs {

constexpr uint64_t SHARD_TILE = 256;      // shard starts are tile-aligned

std::vector<uint64_t> shard_bounds(uint64_t n_words, int n)
{
    if (n < 1) n = 1;
    std::vector<uint64_t> b((size_t)n + 1, 0);
    const uint64_t tile = SHARD_TILE;
    uint64_t tiles = (n_words + tile - 1) / tile;
    for (int i = 0; i <= n; ++i) {
        uint64_t t = tiles * (uint64_t)i / (uint64_t)n;
        b[(size_t)i] = std::min(n_words, t * tile);
    }
    b[(size_t)n] = n_words;
    return b;
}

std::vector<uint64_t> shard_plan(uint64_t n_words, int n_devices)
{
    if (n_devices < 1) n_devices = 1;
    uint64_t n = (uint64_t)n_devices;
    if (n_words * 32 > (1ull << 32)) {
        const uint64_t tiles = (n_words + SHARD_TILE - 1) / SHARD_TILE, per = VS_MAX_SHARD_WORDS / SHARD_TILE;
        n = std::max<uint64_t>(n, (tiles + per - 1) / per);            // no shard gets more than `per` tiles
        n = (n + n_devices - 1) / n_devices * n_devices;
    }
    return shard_bounds(n_words, (int)n);
}

// times of scans that ran at the same time on different devices: the slowest; of shards one device scanned one after
// the other (`sequential`): the sum
static void add_stats(vs_scan_stats *agg, const vs_scan_stats &s, bool sequential = false)
{
    const auto t = [sequential](float a, float b) { return sequential ? a + b : std::max(a, b); };
    agg->upload_ms = t(agg->upload_ms, s.upload_ms); agg->extract_ms = t(agg->extract_ms, s.extract_ms);
    agg->score_ms = t(agg->score_ms, s.score_ms); agg->total_ms = t(agg->total_ms, s.total_ms);
    agg->resolve_ms = t(agg->resolve_ms, s.resolve_ms);
    agg->n_cand_fwd += s.n_cand_fwd; agg->n_cand_rev += s.n_cand_rev;
    agg->n_blocks_fwd += s.n_blocks_fwd; agg->n_blocks_rev += s.n_blocks_rev;
    agg->n_hits += s.n_hits; agg->launches += s.launches; agg->score_launches += s.score_launches;
    agg->h2d_bytes += s.h2d_bytes; agg->d2h_bytes += s.d2h_bytes; agg->n_chunks += s.n_chunks; agg->redo_chunks += s.redo_chunks;
    agg->guide_passes = std::max(agg->guide_passes, s.guide_passes);
}

// One host thread + one context per device; the shards of the plan b (a multiple of the device count) are dealt out in
// contiguous runs, and each device scans its run one shard after the other on its context.  `run(s, ctx, w0, n)` scans
// shard s.
template <class Run>
static int for_each_shard(const std::vector<uint64_t> &b, const std::vector<int> &devices, vs_scan_stats *agg, std::string &err, Run run)
{
    const int nd = (int)devices.size(), per = (int)(b.size() - 1) / nd;
    std::vector<int> rc((size_t)nd, VS_OK);
    std::vector<std::string> errs((size_t)nd);
    std::vector<vs_scan_stats> st((size_t)nd);
    auto work = [&](int i) {
        vs_ctx *ctx = nullptr;
        memset(&st[(size_t)i], 0, sizeof(vs_scan_stats));
        int r = VS_OK;
        for (int s = i * per; s < (i + 1) * per && r == VS_OK; ++s) {
            const uint64_t w0 = b[(size_t)s], w1 = b[(size_t)s + 1];
            if (w1 <= w0) continue;
            if (!ctx) r = vs_ctx_create(devices[(size_t)i], &ctx);
            vs_scan_stats one;
            memset(&one, 0, sizeof(one));
            if (r == VS_OK) r = run(s, ctx, w0, w1 - w0, &one);
            if (r == VS_OK) add_stats(&st[(size_t)i], one, true);
        }
        if (r != VS_OK) errs[(size_t)i] = vs_last_error(ctx);
        rc[(size_t)i] = r;
        vs_ctx_destroy(ctx);
    };
    if (nd == 1) work(0);
    else {
        std::vector<std::thread> th;
        for (int i = 0; i < nd; ++i) th.emplace_back(work, i);
        for (auto &t : th) t.join();
    }
    if (agg) memset(agg, 0, sizeof(*agg));
    for (int i = 0; i < nd; ++i) {
        if (rc[(size_t)i] != VS_OK) { err = "device " + std::to_string(devices[(size_t)i]) + ": " + errs[(size_t)i]; return rc[(size_t)i]; }
        if (agg) add_stats(agg, st[(size_t)i]);
    }
    return VS_OK;
}

static std::vector<int> or_device0(const std::vector<int> &devices) { return devices.empty() ? std::vector<int>{0} : devices; }

int scan_text_sharded(const vs_text_view &text, const std::vector<int> &devices_in,
                      const uint8_t *guides, uint32_t n_guides, int k, int extra_pam,
                      std::vector<vs_hit> &hits, vs_scan_stats *agg, std::string &err)
{
    const std::vector<int> devices = or_device0(devices_in);
    const std::vector<uint64_t> b = shard_plan(text.n_words, (int)devices.size());
    std::vector<std::vector<vs_hit>> part(b.size() - 1);
    int rc = for_each_shard(b, devices, agg, err, [&](int i, vs_ctx *ctx, uint64_t w0, uint64_t n, vs_scan_stats *st) {
        uint64_t cnt = 0;
        std::vector<vs_hit> &h = part[(size_t)i];
        h.resize(1u << 16);
        vs_ctx_set_option(ctx, VS_OPT_KEEP_INDEX, 0);
        int r = vs_scan_text(ctx, &text, w0, n, guides, n_guides, k, extra_pam, h.data(), h.size(), &cnt, st);
        if (r == VS_ERR_OVERFLOW && st->guide_passes <= 1) {
            h.resize(cnt);
            r = vs_scan_fetch(ctx, h.data(), h.size(), &cnt);
        }
        if (r == VS_OK) h.resize(cnt);
        return r;
    });
    hits.clear();
    if (rc != VS_OK) return rc;
    for (auto &p : part) hits.insert(hits.end(), p.begin(), p.end());
    return VS_OK;
}

// the same with the hits resolved and sorted on every device (vs_scan_resolved): one list per shard, ready for vs_merge_resolved
int scan_text_sharded_resolved(const vs_text_view &text, const std::vector<int> &devices_in,
                               const uint8_t *guides, uint32_t n_guides, int k, int extra_pam,
                               std::vector<std::vector<vs_loc_hit>> &lists, vs_scan_stats *agg, std::string &err)
{
    const std::vector<int> devices = or_device0(devices_in);
    const std::vector<uint64_t> b = shard_plan(text.n_words, (int)devices.size());
    lists.assign(b.size() - 1, {});
    struct Sink {
        static int put(void *user, const vs_loc_hit *h, uint64_t n, uint32_t, uint32_t)
        {
            auto *v = static_cast<std::vector<vs_loc_hit> *>(user);
            try { v->insert(v->end(), h, h + n); } catch (...) { return 1; }
            return 0;
        }
    };
    return for_each_shard(b, devices, agg, err, [&](int i, vs_ctx *ctx, uint64_t w0, uint64_t n, vs_scan_stats *st) {
        uint64_t cnt = 0;
        vs_ctx_set_option(ctx, VS_OPT_KEEP_INDEX, 0);
        return vs_scan_resolved(ctx, &text, w0, n, guides, n_guides, k, extra_pam, nullptr, 0, &cnt, &Sink::put, &lists[(size_t)i], st);
    });
}

}  // namespace vs

extern "C" int vs_map_packed(const vs_text_view *text, const uint8_t *guides, uint32_t n_guides,
                             int k, int extra_pam, const int *devices, int n_devices,
                             vs_hit **hits, uint64_t *n_hits, vs_scan_stats *stats)
{
    if (!hits || !n_hits || !text) return VS_ERR_ARG;
    *hits = nullptr; *n_hits = 0;
    if (text->n_words * 32 > (1ull << 32)) {
        vs_set_last_error("vs_map_packed: unordered hits carry global 32-bit positions, which end at 4 Gbases of text: use vs_map_records");
        return VS_ERR_ARG;
    }
    std::vector<int> dev;
    for (int i = 0; i < n_devices && devices; ++i) dev.push_back(devices[i]);
    std::vector<vs_hit> h;
    std::string err;
    int rc = vs::scan_text_sharded(*text, dev, guides, n_guides, k, extra_pam, h, stats, err);
    if (rc != VS_OK) { vs_set_last_error(err.c_str()); return rc; }
    if (!h.empty()) {
        vs_hit *o = (vs_hit *)malloc(h.size() * sizeof(vs_hit));
        if (!o) return VS_ERR_NOMEM;
        memcpy(o, h.data(), h.size() * sizeof(vs_hit));
        *hits = o;
    }
    *n_hits = h.size();
    return VS_OK;
}

extern "C" int vs_map_records(const vs_text_view *text, const uint8_t *guides, uint32_t n_guides,
                              int k, int extra_pam, const int *devices, int n_devices, int n_threads,
                              vs_record **records, uint64_t *n_records, uint64_t *key16_collisions, vs_scan_stats *stats)
{
    if (!records || !n_records || !text) return VS_ERR_ARG;
    *records = nullptr; *n_records = 0;
    std::vector<int> dev;
    for (int i = 0; i < n_devices && devices; ++i) dev.push_back(devices[i]);
    std::vector<std::vector<vs_loc_hit>> lists;
    std::string err;
    int rc = vs::scan_text_sharded_resolved(*text, dev, guides, n_guides, k, extra_pam, lists, stats, err);
    if (rc != VS_OK) { vs_set_last_error(err.c_str()); return rc; }
    std::vector<const vs_loc_hit *> ptr;
    std::vector<uint64_t> cnt;
    uint64_t total = 0;
    for (auto &l : lists) { ptr.push_back(l.data()); cnt.push_back(l.size()); total += l.size(); }
    if (total == 0) return VS_OK;
    vs_record *o = (vs_record *)malloc(total * sizeof(vs_record));
    if (!o) return VS_ERR_NOMEM;
    rc = vs_merge_resolved(ptr.data(), cnt.data(), (int)ptr.size(), o, key16_collisions, n_threads);
    if (rc != VS_OK) { free(o); return rc; }
    *records = o; *n_records = total;
    return VS_OK;
}

extern "C" int vs_shard_bounds(uint64_t n_words, int n_shards, uint64_t *out)
{
    if (!out || n_shards < 1) return VS_ERR_ARG;
    std::vector<uint64_t> b = vs::shard_bounds(n_words, n_shards);
    for (int i = 0; i <= n_shards; ++i) out[i] = b[(size_t)i];
    return VS_OK;
}
