/*
 * include/varscot_scan.h — C ABI of the B200-native off-target scan ("read_mapping" hot path).
 *
 * The reference has no in-process API for this path: its boundary is two executables,
 * `bidir_index` and `bidir_mapping` (VARSCOT_pipeline/read_mapping/bidir_index.cpp:10-52,
 * bidir_mapping.cpp:190-312), called by the driver script (VARSCOT_pipeline/VARSCOT:296-314).
 * This header is the layer those two executables (and any FFI binding: ctypes, cgo, JNI) sit on.
 * Plain C types only; caller-owned host buffers; callee-owned device buffers; int error codes.
 *
 * Entry point                      replaces (reference file:line)
 * -------------------------------  -----------------------------------------------------------------
 * vs_packer_* / vs_pack_text /     bidir_index.cpp:36-47  readRecords -> Dna5 StringSet -> indexCreate
 * vs_masks_from_planes / _sparse /
 * vs_mask_source_build
 * vs_text_save / vs_text_load      bidir_index.cpp:47 save(index, path); bidir_mapping.cpp:268 open(index, path)
 * vs_ctx_create / vs_text_upload   bidir_mapping.cpp:268  index resident in RAM -> packed text resident in HBM
 * vs_scan / vs_scan_text           bidir_mapping.cpp:285-295 omp-parallel loop over guides calling
 *                                  searchAndVerifyEntireRead -> searchAndVerify (:31-148, :150-188):
 *                                  seed search + verify delegate, for both strands
 * vs_scan_resolved                 the same + the std::map<TOccType,..> order of :13,154 (contig lookup and sort on the device)
 * vs_resolve_hits / vs_merge_resolved  bidir_mapping.cpp:154,164-187  std::map order + primary/secondary flags
 * vs_mapper_*                      bidir_mapping.cpp:268-295 with the index kept open across many guide sets
 * vs_md_string / vs_format_sam     bidir_mapping.cpp:111-123 getMDString + tags; :177-187 write(.., Sam())
 * vs_bidir_index_main              bidir_index.cpp:10-52   main (argv contract)
 * vs_bidir_mapping_main            bidir_mapping.cpp:190-312 main (argv contract, stdout lines, exit codes)
 * vs_vcf_loader_main               variant_processing/vcf_loader.cpp:11-77 (+ process_vcf.h, overlap_sequences.h, write_fasta.h)
 * vs_fasta_writer_main             variant_processing/fasta_writer.cpp:8-41 (+ extract_fasta_ontargets.h)
 * vs_bam_merger_main,              variant_processing/bam_merger.cpp:8-62, bam_merger_ref_only.cpp:8-55 (+ merge_output_bam.h,
 * vs_bam_merger_ref_only_main      filter_output_bam.h, feature_matrix.h, mit_score.h)
 */
#ifndef VARSCOT_SCAN_H
#define VARSCOT_SCAN_H
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VS_GLEN 23            /* guide length incl. PAM (CIGAR 23M hard-coded at bidir_mapping.cpp:102) */
#define VS_MAX_MISMATCHES 8   /* bidir_mapping.cpp:234-238 */

enum {
    VS_OK = 0,
    VS_ERR_ARG = 1,
    VS_ERR_CUDA = 2,
    VS_ERR_NOMEM = 3,
    VS_ERR_OVERFLOW = 4,     /* caller's hit buffer too small; *n_hits holds the required count */
    VS_ERR_NODEVICE = 5,
    VS_ERR_IO = 6
};

/* ---- packed text ---------------------------------------------------------------------------
 * The text (all contigs concatenated, "ConcatDirect" as bidir_index.cpp:12) is stored bit-sliced, 32 bases per
 * word, base j of a word in bit j, as a structure of arrays:
 *   bases[w] = {hi, lo}  the two bits of the Dna code (A=00, C=01, G=10, T=11); N and padding are 00
 *   masks[w] = {iv, lw}  per WINDOW START p = 32 w + j:
 *                iv: the 23-base window at p is not scannable — it contains an N (anything outside ACGT/U, R6),
 *                    runs over the end of its contig, or runs past the end of the text (R1, R3)
 *                lw: the window ends exactly on the last base of its contig (R4: bidir_mapping.cpp:51 lets only
 *                    the second-half seed reach it)
 * n_words = ceil(n_bases/32).  bases carries ONE extra all-zero pad word (bases[n_words]) so that word w+1 is
 * readable for every w < n_words; masks has n_words entries.  `sparse` optionally lists the non-zero mask words
 * in ascending word order: uploads then move only those over PCIe.
 */
typedef struct { uint32_t hi, lo; } vs_bases;
typedef struct { uint32_t iv, lw; } vs_masks;
typedef struct { uint32_t word, iv, lw; } vs_mask_entry;

/* ---- compact mask source (optional) ---------------------------------------------------------
 * The window masks are a function of two bit planes (one bit per base, n_words + 1 words each): the N plane `nm`
 * (base is not A/C/G/T; the padding after the last base reads as N) and the contig-end plane `em` (base is the last
 * of its contig) — see vs_masks_from_planes().  A view that carries them in the compact form below lets the device
 * compute the masks itself, so an upload moves only the planes: N runs of a genome collapse to a few runs, and a
 * swarm of short contigs (variant segments) costs 4 B per word (`em`) instead of 8 B (masks).
 *   run   {word, count, value}: words [word, word + count) of the plane all equal `value` (non-zero)
 *   nm_runs : every non-zero word of nm, in ascending order
 *   em_code : one byte per word of em: the index of the word's only set bit, or VS_EM_NONE when the word is zero or has
 *             several bits set; read only for the blocks flagged in em_dense (a contig of >= 32 bases puts at most one end
 *             into a word, so a swarm of 45-base contigs costs one byte per 32 bases)
 *   em_dense: one byte per block of VS_EM_BLOCK words; 1 = the block travels as em_code, 0 = its non-zero words are in em_runs
 *   em_runs : ascending; every non-zero word of a block with em_dense == 0, and the words with several bits of the others
 * A view carries the source iff em_code and em_dense are set (nm_runs / em_runs may be NULL when their counts are 0);
 * otherwise uploads use masks / sparse. */
#define VS_EM_BLOCK 4096
#define VS_EM_NONE 32
typedef struct { uint32_t word, count, value; } vs_plane_run;

typedef struct {
    uint64_t n_bases;
    uint64_t n_words;
    uint32_t n_contigs;
    uint32_t reserved;
    const uint64_t      *contig_off;   /* n_contigs + 1 */
    const vs_bases      *bases;        /* n_words + 1 */
    const vs_masks      *masks;        /* n_words */
    const vs_mask_entry *sparse;       /* n_sparse entries, or NULL */
    uint64_t n_sparse;
    /* compact mask source, or all NULL / 0 */
    const uint8_t       *em_code;      /* n_words + 1 */
    const uint8_t       *em_dense;     /* ceil((n_words + 1) / VS_EM_BLOCK) */
    const vs_plane_run  *nm_runs;
    const vs_plane_run  *em_runs;
    uint64_t n_nm_runs, n_em_runs;
} vs_text_view;

/* Build the compact mask source from the two planes (n_words + 1 words each).  The members of *out are malloc'd;
 * release them with vs_mask_source_free. */
typedef struct {
    uint8_t        *em_code;
    uint8_t        *em_dense;
    vs_plane_run   *nm_runs;
    vs_plane_run   *em_runs;
    uint64_t n_nm_runs, n_em_runs, n_em_blocks;
} vs_mask_source;
int  vs_mask_source_build(const uint32_t *nm, const uint32_t *em, uint64_t n_words, vs_mask_source *out);
void vs_mask_source_free(vs_mask_source *s);

typedef struct vs_packer vs_packer;
vs_packer *vs_packer_new(void);
void       vs_packer_free(vs_packer *p);
/* append raw sequence characters (whitespace, incl. newlines, is skipped) */
int        vs_packer_append(vs_packer *p, const char *chars, size_t n);
/* close the current contig (contigs of length 0 are kept: they occupy an id, SeqAn StringSet semantics) */
int        vs_packer_end_contig(vs_packer *p);
/* finish: computes the window masks and their sparse form; the view's pointers stay valid until vs_packer_free */
int        vs_packer_finish(vs_packer *p, vs_text_view *out);

/* one-shot: ASCII text of all contigs concatenated + n_contigs+1 offsets -> bases[ceil(n/32)+1], masks[ceil(n/32)] */
int vs_pack_text(const char *ascii, uint64_t n_bases, const uint64_t *contig_off, uint32_t n_contigs,
                 vs_bases *out_bases, vs_masks *out_masks);
/* the same, returning the N plane and the contig-end plane (n_words + 1 words each) instead of the masks */
int vs_pack_text_planes(const char *ascii, uint64_t n_bases, const uint64_t *contig_off, uint32_t n_contigs,
                        vs_bases *out_bases, uint32_t *out_nm, uint32_t *out_em);
/* window masks from an N plane and a contig-end plane (both n_words + 1 words, the extra word is read as padding) */
int vs_masks_from_planes(const uint32_t *nm, const uint32_t *em, uint64_t n_words, vs_masks *out);
/* sparse form of a mask array: malloc'd list of the non-zero words (release with vs_free) */
int vs_masks_sparse(const vs_masks *masks, uint64_t n_words, vs_mask_entry **out, uint64_t *n_out);

/* packed-text cache at the -I prefix (file <prefix>.vsidx) */
int vs_text_save(const char *prefix, const vs_text_view *text);
/* window masks of a view on the host: a copy of text->masks, or — for a view that carries only the compact mask source
 * (what vs_text_load returns for a cache written by bidir_index) — rebuilt from it.  out: n_words entries. */
int vs_text_masks(const vs_text_view *text, vs_masks *out);
/* loads into ONE malloc'd buffer (returned in *owner, release with vs_free) that the view points into */
int vs_text_load(const char *prefix, vs_text_view *out, void **owner);
void vs_free(void *p);

/* ---- device context ------------------------------------------------------------------------- */
typedef struct vs_ctx vs_ctx;

int  vs_device_count(void);                     /* >= 0, or -VS_ERR_* */
int  vs_ctx_create(int device, vs_ctx **ctx);   /* one context per device per host thread */
void vs_ctx_destroy(vs_ctx *ctx);
const char *vs_last_error(const vs_ctx *ctx);   /* ctx may be NULL: last error of the calling thread */
/* words per pipeline chunk (default 4 Mi words = 128 Mi bases); tests shrink it to cross chunk borders */
int  vs_ctx_set_chunk_words(vs_ctx *ctx, uint64_t chunk_words);

/* Limits.  A text of any length is accepted; a contig holds at most 2^32 bases (positions inside a contig are 32-bit).
 * Positions inside a context are 32-bit and relative to the shard's origin: 0 — they are global — for every shard of a
 * text within 4 Gbases and for a shard that ends at least 32 bases below 2^32; the shard's first base otherwise.  Such a
 * shard (one that reaches beyond 2^32 - 32 in a text longer than 4 Gbases) holds at most VS_MAX_SHARD_WORDS words.
 * vs_scan_resolved, vs_map_records and the executables serve every text; the unordered calls (vs_scan, vs_scan_text,
 * vs_scan_fetch, vs_map_packed) report global 32-bit positions and return VS_ERR_ARG beyond that domain (a text longer
 * than 4 Gbases, or a resident shard whose origin is not 0). */
#define VS_MAX_SHARD_WORDS ((1ull << 27) - 256)      /* 2^32 - 8192 bases, a whole number of 256-word tiles */

/* Make words [first_word, first_word + n_words) of the text resident on the device (+ one halo word of bases).
 * Window STARTS in those words are owned by this context; hit positions are 32 * first_word + local - origin (global
 * for every text within 4 Gbases, see the limits above). */
int vs_text_upload(vs_ctx *ctx, const vs_text_view *text, uint64_t first_word, uint64_t n_words);

/* page-locked host memory for fast uploads / hit downloads */
void *vs_host_alloc(size_t bytes);
void  vs_host_free(void *p);

typedef struct {
    uint32_t pos;    /* start position in the concatenated text (global: the unordered calls serve texts within 4 Gbases) */
    uint32_t info;   /* guide << 8 | strand << 7 | mm  (strand 1 = reverse pass, flag bit 16) */
} vs_hit;

typedef struct {
    float    upload_ms, extract_ms, score_ms, total_ms;  /* CUDA-event times; extract/score are sums over chunks */
    uint64_t n_cand_fwd, n_cand_rev;                      /* PAM-valid, N-free windows per strand */
    uint64_t n_blocks_fwd, n_blocks_rev;                  /* 32-candidate blocks scored per strand */
    uint64_t n_hits;
    uint64_t h2d_bytes, d2h_bytes;                        /* bytes this call moved over PCIe */
    uint32_t launches;                                    /* kernels launched by this call */
    uint32_t score_launches;
    uint32_t n_chunks;
    uint32_t redo_chunks;                                 /* passes repeated because a device buffer was too small (0 on uniform text) */
    float    resolve_ms;                                  /* device-side hit resolution + sort + download (vs_scan_resolved) */
    uint32_t index_reused;                                /* 1: the resident candidate index was scored, nothing was extracted; 2: its bucketed form */
    uint32_t guide_passes;                                /* passes over the candidate index (guide super-chunks) */
    float    index_build_ms;                              /* building the bucketed index (the scan that builds it pays once) */
} vs_scan_stats;

/* ---- resident candidate index ---------------------------------------------------------------------------------
 * The first scan of a resident text extracts the PAM-valid windows of both strands into a candidate store (bit-sliced
 * blocks of 32) that stays in HBM: the analogue of the reference's split between bidir_index (bidir_index.cpp:45-47,
 * build once) and bidir_mapping (bidir_mapping.cpp:268, open and search).  Later scans with the same PAM set score the
 * store directly.  It is dropped by a new upload, a different -P, vs_index_drop(), or kept off with VS_OPT_KEEP_INDEX 0. */
#define VS_OPT_KEEP_INDEX   1     /* 0 / 1 (default 1) */
#define VS_OPT_HIT_CAPACITY 2     /* entries of the device hit buffer; 0 (default) = sized from k, the PAM set and the shard */
#define VS_OPT_BUCKET_INDEX 3     /* 0 never / 1 (default) where it pays (>= 256 guides, or >= 64 guides on a large shard) / 2 always: when a resident index is scanned a second time,
                                   * regroup its candidates by the PAM dinucleotide + the six bases next to it, so that later scans
                                   * score 9-15 instead of 19 positions per window and guide (vs_scan_stats.index_reused == 2) */
int vs_ctx_set_option(vs_ctx *ctx, int option, int64_t value);
int vs_index_drop(vs_ctx *ctx);

/* Scan the RESIDENT text for every window within k mismatches of each guide, both strands (rules R1-R4,
 * SURVEY.md section 8a).  guides: n_guides x 23 Dna codes (0..3).  extra_pam: -1 or 4*x+y for -P XY.
 * Hits arrive UNORDERED.  If more than out_cap hits exist returns VS_ERR_OVERFLOW with *n_hits = needed;
 * the hits stay on the device and vs_scan_fetch() retrieves them without rescanning. */
int vs_scan(vs_ctx *ctx, const uint8_t *guides, uint32_t n_guides, int k, int extra_pam,
            vs_hit *out, uint64_t out_cap, uint64_t *n_hits, vs_scan_stats *stats);
/* Same, reading the text from HOST memory: the upload of chunk i+1 overlaps the scan of chunk i (the text is
 * resident afterwards).  This is the end-to-end call the executables use. */
int vs_scan_text(vs_ctx *ctx, const vs_text_view *text, uint64_t first_word, uint64_t n_words,
                 const uint8_t *guides, uint32_t n_guides, int k, int extra_pam,
                 vs_hit *out, uint64_t out_cap, uint64_t *n_hits, vs_scan_stats *stats);
int vs_scan_fetch(vs_ctx *ctx, vs_hit *out, uint64_t out_cap, uint64_t *n_hits);

/* ---- scans that resolve and sort their hits on the device ---------------------------------------------------
 * The contig of every hit is looked up on the device (contig starts derived from the contig-end plane, or uploaded when
 * the view has no mask source) and the hits are radix-sorted into the reference's emission order
 * (guide; forward pass then reverse pass; std::map key (contig & 0xFFFF, pos), bidir_mapping.cpp:13,154,285-295), so the
 * host only merges the lists of the shards (vs_merge_resolved).  The text view must carry contig_off.
 *   key    = (guide - guide_lo of the delivery) << 49 | strand << 48 | (contig & 0xFFFF) << 32 | pos in contig
 *   contig = full 32-bit id;  info = guide << 8 | strand << 7 | mm  (as vs_hit)
 * Guides are processed in super-chunks sized to the device hit buffer (one for configs 1-4); with a `sink` every
 * super-chunk is handed over as soon as it is sorted (host memory stays O(super-chunk), config 5), otherwise the lists
 * are concatenated in `out` (guide-ascending, so the concatenation is sorted as a whole). */
typedef struct { uint64_t key; uint32_t contig; uint32_t info; } vs_loc_hit;
typedef int (*vs_hit_sink)(void *user, const vs_loc_hit *hits, uint64_t n, uint32_t guide_lo, uint32_t guide_hi);   /* non-zero aborts */
/* text == NULL: scan the resident shard (first_word / n_words ignored); otherwise upload + scan as vs_scan_text */
int vs_scan_resolved(vs_ctx *ctx, const vs_text_view *text, uint64_t first_word, uint64_t n_words,
                     const uint8_t *guides, uint32_t n_guides, int k, int extra_pam,
                     vs_loc_hit *out, uint64_t out_cap, uint64_t *n_hits, vs_hit_sink sink, void *user, vs_scan_stats *stats);
/* page-lock / unlock memory the caller owns (e.g. a shared-memory segment the hits are downloaded into) */
int vs_host_register(void *p, size_t bytes);
int vs_host_unregister(void *p);

/* Convenience used by the executables and bindings: shard a packed text by word ranges over the given
 * devices (devices == NULL or n_devices == 0 -> device 0; one host thread + one context per device, no
 * collective), scan, and return all hits unordered in a malloc'd array (release with vs_free).
 * Texts within 4 Gbases only (VS_ERR_ARG beyond: use vs_map_records). */
int vs_map_packed(const vs_text_view *text, const uint8_t *guides, uint32_t n_guides,
                  int k, int extra_pam, const int *devices, int n_devices,
                  vs_hit **hits, uint64_t *n_hits, vs_scan_stats *stats);

/* Shard plan used by vs_map_packed and by one-process-per-GPU callers: out[0..n] are word indices, shard i owns the
 * window starts of words [out[i], out[i+1]) and reads one halo word after them.  Tile-aligned, balanced. */
int vs_shard_bounds(uint64_t n_words, int n_shards, uint64_t *out);

/* ---- host-side resolution ------------------------------------------------------------------- */
typedef struct {
    uint32_t guide;
    uint32_t contig;   /* full 32-bit id */
    uint32_t pos;      /* 0-based inside the contig */
    uint16_t flag;     /* 0 / 16 / 256 / 272 */
    uint8_t  mm;
    uint8_t  pad;
} vs_record;

/* Sort hits into the reference's emission order (guide; forward pass then reverse pass; std::map key order
 * (contig & 0xFFFF, pos) extended by contig >> 16) and apply the running-best primary/secondary rule.
 * out must hold n records.  *key16_collisions counts records the reference's uint16 key would have merged. */
int vs_resolve_hits(const vs_hit *hits, uint64_t n, const uint64_t *contig_off, uint32_t n_contigs,
                    vs_record *out, uint64_t *key16_collisions);
/* the same with n_threads host threads (the executables pass -T): the contig lookup and the per-pass sorts run in parallel */
int vs_resolve_hits_mt(const vs_hit *hits, uint64_t n, const uint64_t *contig_off, uint32_t n_contigs,
                       vs_record *out, uint64_t *key16_collisions, int n_threads);

/* Merge the sorted lists of n_lists shards (vs_scan_resolved) into records in emission order and apply the running-best
 * primary/secondary rule (bidir_mapping.cpp:164-187).  out must hold the sum of the counts. */
int vs_merge_resolved(const vs_loc_hit *const *lists, const uint64_t *counts, int n_lists,
                      vs_record *out, uint64_t *key16_collisions, int n_threads);

/* The whole mapping step of the executables: shard, scan with device-side resolution, merge; records in emission order
 * in a malloc'd array (release with vs_free).  A text within 4 Gbases gets one shard per device (vs_shard_bounds); a
 * longer one max(n_devices, ceil(n_words / VS_MAX_SHARD_WORDS)) shards rounded up to a multiple of n_devices, which every
 * device scans one after the other. */
int vs_map_records(const vs_text_view *text, const uint8_t *guides, uint32_t n_guides,
                   int k, int extra_pam, const int *devices, int n_devices, int n_threads,
                   vs_record **records, uint64_t *n_records, uint64_t *key16_collisions, vs_scan_stats *stats);

/* ---- resident mapper ------------------------------------------------------------------------------------------
 * vs_map_records with the text kept in HBM between calls: a caller that maps many guide sets against one genome (a guide
 * screen, a service, a batch that keeps the reference loaded) pays the upload once, the extraction of the candidate index
 * once per PAM set, and from the second call on scores the bucketed index wherever VS_OPT_BUCKET_INDEX's default policy
 * builds it.  Beyond 4 Gbases every device keeps all of its shards resident at once. */
typedef struct vs_mapper vs_mapper;
/* Shard `text` over the devices exactly as vs_map_records does (vs_shard_bounds within 4 Gbases, one shard per device;
 * several per device beyond) and upload every shard to a context of its own that keeps its candidate index (devices == NULL
 * or n_devices == 0 -> device 0).  The view's host buffers are read during this call only and may be released afterwards;
 * the view must carry contig_off.  Before anything is uploaded, the device memory every device's shards will need (text,
 * masks, the plain and the bucketed candidate store at the densest PAM set, the scan scratch of every context) is compared
 * with its free memory: VS_ERR_NOMEM, with the bytes needed and free in vs_last_error(NULL), when it does not fit.  A failed
 * upload releases everything and names the device and the shard.  VS_ERR_NODEVICE without a device. */
int  vs_mapper_create(const vs_text_view *text, const int *devices, int n_devices, vs_mapper **out);
/* Same arguments and results as vs_map_records, against the resident shards: records in emission order (malloc'd, release
 * with vs_free).  The first call, and the first after a change of extra_pam, extracts the candidate index from the resident
 * text; later calls score it.  stats: index_reused is the least over the shards (2 only when every shard scored its bucketed
 * index), index_build_ms sums over a device's shards and takes the slowest device.  An argument error returns VS_ERR_ARG and
 * leaves the resident shards and indexes as they were; so does a call made while another one runs on the same mapper. */
int  vs_mapper_map(vs_mapper *m, const uint8_t *guides, uint32_t n_guides, int k, int extra_pam, int n_threads,
                   vs_record **records, uint64_t *n_records, uint64_t *key16_collisions, vs_scan_stats *stats);
/* ---- streamed records ------------------------------------------------------------------------------------------
 * The records of vs_mapper_map / vs_map_records delivered a range of whole guides at a time, in emission order, while the
 * devices score the next range: host memory stays bounded by the delivery size instead of growing with the whole map.  The
 * concatenated deliveries are, byte for byte, the records the one-shot call returns.
 *   records_per_delivery  target records per delivery; 0 = 32 Mi.  A delivery holds whole guides (the flags are per guide
 *                         and strand) and at most this many records, except a single guide denser than it, which comes alone.
 *                         Ranges are sized from the expected hit density first, then from the hits per guide just scanned.
 *   with_windows          also deliver each record's 23-base genome window, read on the device beside the sorted hit:
 *                         bits 2 i .. 2 i + 1 = Dna code (A 0, C 1, G 2, T 3) of genome base pos + i of the record's contig,
 *                         forward orientation.  vs_md_from_window turns it into the record's MD:Z without the host text.
 *   sink                  called on the calling thread, one delivery at a time, guides ascending and contiguous from 0 to
 *                         n_guides (a range without records is delivered too, with n = 0).  Record guide ids are absolute.
 *                         The pointers are valid during the call only.  A non-zero return stops the call: no further sink
 *                         call is made, the devices are drained, and the call returns VS_ERR_ARG ("the sink aborted").
 * Host memory in flight: about 3 x records_per_delivery x (16 + 8 with_windows) bytes (the sorted lists of the range being
 * delivered and of the range being scanned, and the merged delivery), plus every context's pinned staging of its largest
 * super-chunk.  key16_collisions and stats are sums over the deliveries (times: device times summed over the ranges). */
typedef int (*vs_record_sink)(void *user, const vs_record *records, const uint64_t *windows /* NULL unless asked */,
                              uint64_t n, uint32_t guide_lo, uint32_t guide_hi);          /* non-zero aborts */
/* The resident mapper's shards scan every range; the one-call-at-a-time rule of vs_mapper_map applies, and an abort leaves the
 * resident shards and indexes as they were. */
int vs_mapper_map_stream(vs_mapper *m, const uint8_t *guides, uint32_t n_guides, int k, int extra_pam, int n_threads,
                         uint64_t records_per_delivery, int with_windows, vs_record_sink sink, void *user,
                         uint64_t *key16_collisions, vs_scan_stats *stats);
/* Shards as vs_map_records.  With one shard per device every device keeps its context for the whole call: the first range
 * streams the upload and extracts the candidate index, later ranges score the resident index.  With several shards per device
 * (texts beyond 4 Gbases on few devices) every range uploads each shard again: that cost is paid only when the map needs more
 * than one delivery. */
int vs_map_records_stream(const vs_text_view *text, const uint8_t *guides, uint32_t n_guides, int k, int extra_pam,
                          const int *devices, int n_devices, int n_threads, uint64_t records_per_delivery, int with_windows,
                          vs_record_sink sink, void *user, uint64_t *key16_collisions, vs_scan_stats *stats);

/* shards held; bytes of device memory the mapper's contexts hold now, and the create-time estimate (all devices; an upper
 * bound for scans that keep up to 16 Mi hits per shard and pass, of up to 4096 guides) */
int  vs_mapper_info(const vs_mapper *m, uint32_t *n_shards, uint64_t *device_bytes, uint64_t *planned_bytes);
void vs_mapper_destroy(vs_mapper *m);

#define VS_MD_SEQAN 0
#define VS_MD_SAMTOOLS 1
/* MD:Z value for the window at global position gpos against guide (codes) on the given strand. out >= 64 bytes. */
int vs_md_string(const vs_bases *bases, uint64_t gpos, const uint8_t *guide, int strand, int md_style, char *out);
/* MD:Z from a delivered window (vs_record_sink): the same string vs_md_string writes for that record. out >= 64 bytes. */
int vs_md_from_window(uint64_t window, const uint8_t *guide, int strand, int md_style, char *out);
/* one 13-column SAM line (R9) incl. '\n'; returns the length written (excluding NUL), or -1 if buflen is too small */
int vs_format_sam(const vs_record *r, const char *qname, const char *rname, const uint8_t *guide,
                  const char *md, char *buf, size_t buflen);

/* ---- the two executables as library calls ---------------------------------------------------- */
int vs_bidir_index_main(int argc, char **argv);
int vs_bidir_mapping_main(int argc, char **argv);
/* row f1 (producer of the variant segments): `vcf_loader FILE.vcf SNPGENOME.fa GENOME.fa SAMPLE SEQLENGTH THREADS`,
 * VARSCOT_pipeline/variant_processing/vcf_loader.cpp:11-77 (host only, no GPU involved) */
int vs_vcf_loader_main(int argc, char **argv);
/* row f4 (producer of the guide FASTA): `fasta_writer OUTPUT1.fa OUTPUT2.fa ONTARGETS.bed GENOME.fa`,
 * VARSCOT_pipeline/variant_processing/fasta_writer.cpp:8-41 (host only) */
int vs_fasta_writer_main(int argc, char **argv);
/* row f3 (consumers of the mapper's SAM): `bam_merger RESULT.txt FEATURES.txt REF.sam SNP.sam TARGETS.bed GENOME.fa SNP.fa
 * TUSCAN.txt K SEQLENGTH THREADS MIT` and `bam_merger_ref_only RESULT.txt FEATURES.txt REF.sam TARGETS.bed GENOME.fa TUSCAN.txt
 * K SEQLENGTH MIT`, VARSCOT_pipeline/variant_processing/bam_merger.cpp:8-62, bam_merger_ref_only.cpp:8-55 (host only) */
int vs_bam_merger_main(int argc, char **argv);
int vs_bam_merger_ref_only_main(int argc, char **argv);

/* ---- microbenchmarks used by bench.py for the roofline denominators ---------------------------- */
/* thread-level LOP3 instructions per second of the device (alu pipe), and LDS 32-bit lane-words per second */
int vs_measure_int_peaks(vs_ctx *ctx, double *lop3_per_s, double *lds_words_per_s);

#ifdef __cplusplus
}
#endif
#endif
