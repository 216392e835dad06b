/* pp_abi.h — C ABI of polypolish-b200 (libpolypolish_b200.so).
 *
 * The reference (rrwick/Polypolish v0.6.1) is a monolithic Rust binary with no plugin/FFI surface, so the
 * drop-in boundary is cut at the function seams of its hot path (SURVEY.md §8b); each entry point below
 * names the reference function(s) it replaces.  Everything text-shaped (SAM/FASTA) stays on the host side of
 * the boundary; everything from packed records to polished bytes runs as sm_100a kernels.
 *
 * Conventions: plain pointers and sizes, no C++/torch types; the caller owns every host buffer; the library
 * owns all device memory and streams inside pp_ctx; integer return codes (0 = ok, <0 = error) and
 * pp_last_error() for the message; no exceptions or exit() cross the boundary.  A pp_ctx is single-threaded
 * (the reference is single-threaded); multi-GPU = one ctx per GPU, one host thread (or process) each.
 * There is no CPU fallback: every compute entry point fails with PP_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef PP_ABI_H
#define PP_ABI_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PP_OK 0
#define PP_ERR_CUDA (-1)   /* CUDA runtime/driver failure, or no usable device */
#define PP_ERR_ARG (-2)    /* malformed arguments (null pointers, sizes out of range, capacity too small) */
#define PP_ERR_INPUT (-3)  /* the reference's quit_with_error / panic cases; message = the reference's text */
#define PP_ERR_NOMEM (-4)
#define PP_ERR_IO (-5)

typedef struct pp_ctx pp_ctx; /* opaque; one per (host thread, GPU) */

int pp_create(int device, pp_ctx** out);
void pp_destroy(pp_ctx* ctx);
const char* pp_last_error(const pp_ctx* ctx); /* ctx-owned, valid until the next call on ctx */
const char* pp_version(void);                 /* "0.6.1-b200" : tracks main.rs:24-25 crate version */

/* Pinned host memory for the SoA arrays (H2D at full PCIe rate). Plain malloc'd buffers also work. */
void* pp_host_alloc(size_t bytes);
void pp_host_free(void* p);

/* ------------------------------------------------------------------------------------------------------
 * Packed alignments (struct-of-arrays), in SAM order: (file index, line index).  ORDER IS SEMANTICALLY
 * SIGNIFICANT: the reference sums the f64 depth sequentially in this order (pileup.rs:64).
 * Replaces the in-memory `Alignment` of alignment.rs:33-43 as produced by Alignment::new (alignment.rs:49-98).
 * ---------------------------------------------------------------------------------------------------- */
#define PP_CONTIG_UNKNOWN 0xFFFFFFFFu /* RNAME not in the assembly: an error only if the alignment is "good" (alignment.rs:298-300) */

#define PP_FLAG_REVERSE 0x01 /* SAM flag 16 (alignment.rs:151-153) */
#define PP_FLAG_ZPFAIL  0x02 /* a ZP:Z:fail tag was present (alignment.rs:72-74) */
#define PP_FLAG_SEQSTAR 0x04 /* SEQ was "*": the sequence is the read group's source sequence (alignment.rs:290-295,311-322) */
#define PP_FLAG_RC      0x08 /* use the reverse complement of the pooled sequence (alignment.rs:161-167) */
#define PP_FLAG_NOSEQ   0x10 /* no record of the group carried a sequence (only legal when the group is skipped by --careful) */
#define PP_FLAG_GHOST   0x20 /* record of a read that lives on another GPU's contigs: counts for goodness / k / --careful,
                                adds nothing to the pileup (contig sharding, pp_shards_build) */
#define PP_FLAG_ESC     0x40 /* seq_bits == 2 only: the sequence has a base other than A, C, G, T and lives in esc_pool (4-bit
                                codes); seq_off then counts esc_pool blocks */
#define PP_FLAG_NEWGROUP 0x80 /* seq_bits == 2 only, and only where read_id == NULL: the first record of a read group (read_id is then
                                 rebuilt on the device as the number of such records so far, minus one) */

/* CIGAR op codes in cigar_ops (BAM numbering): len << 4 | op.  Zero-length ops are dropped by the packer
 * (they contribute nothing to the expanded CIGAR of alignment.rs:325-346). */
#define PP_OP_M 0
#define PP_OP_I 1
#define PP_OP_D 2
#define PP_OP_N 3
#define PP_OP_S 4
#define PP_OP_H 5
#define PP_OP_P 6
#define PP_OP_EQ 7
#define PP_OP_X 8

#define PP_SEQ_BLOCK 32 /* every pooled sequence starts on a 32-base boundary (16 B in 4-bit mode) */

typedef struct {
  uint64_t n_aln;            /* aligned records (flag&4 == 0), all SAM files concatenated in CLI order        */
  uint64_t n_reads;          /* number of read groups = max(read_id)+1                                        */
  const uint32_t* contig;    /* [n_aln] contig index, or PP_CONTIG_UNKNOWN                                    */
  const uint32_t* ref_start; /* [n_aln] 0-based (POS-1, POS 0 stays 0: alignment.rs:58-61)                    */
  const uint32_t* read_id;   /* [n_aln] group id; a group = maximal run of consecutive equal QNAMEs
                                (alignment.rs:255-263); ids are dense and non-decreasing                     */
  const uint32_t* seq_off;   /* [n_aln] start of the sequence in seq_pool, in units of PP_SEQ_BLOCK bases     */
  const uint16_t* seq_len;   /* [n_aln] bases                                                                 */
  const uint32_t* cigar_off; /* [n_aln] first op in cigar_ops                                                 */
  const uint16_t* n_cigar;   /* [n_aln] ops                                                                   */
  const uint32_t* nm;        /* [n_aln] NM:i value (last one wins, alignment.rs:68-71)                        */
  const uint8_t* flags;      /* [n_aln] PP_FLAG_*                                                             */
  uint64_t n_cigar_ops;
  const uint32_t* cigar_ops; /* pool                                                                          */
  uint32_t seq_bits;         /* 4: BAM nibble codes "=ACMGRSVTWYHKDBN", 2 per byte, low nibble first, code 0
                                never used; 8: upper-cased ASCII bytes (any read with a character outside the
                                15 letters forces 8-bit mode so that parity holds for arbitrary SEQ bytes);
                                2: the wire format of pp_alignments_to_2bit - A,C,G,T = 0..3, 4 per byte, low bits
                                first, 8 bytes per PP_SEQ_BLOCK (same block numbering as the 4-bit pool); sequences
                                with any other base are PP_FLAG_ESC records in esc_pool.  Expanded to 4-bit on the
                                device right after the upload: 38 % fewer bytes cross PCIe.  In this format two arrays
                                may be NULL because the device can rebuild them: cigar_off (= exclusive prefix sums of
                                n_cigar, when the ops lie in record order without gaps) and read_id (PP_FLAG_NEWGROUP) */
  uint64_t seq_pool_bytes;
  const uint8_t* seq_pool;   /* 16-byte aligned                                                               */
  uint64_t esc_pool_bytes;   /* seq_bits == 2: 4-bit sequences of the PP_FLAG_ESC records (else 0 / NULL)        */
  const uint8_t* esc_pool;
} pp_alignments;

/* The 2-bit wire format of a 4-bit batch (host side, done once per batch like the packing itself): *out shares every array
 * with `in` except flags, seq_off, seq_pool and esc_pool, which belong to *owner (free with pp_2bit_free).  PP_ERR_ARG unless
 * in->seq_bits == 4. */
typedef struct pp_2bit pp_2bit;
int pp_alignments_to_2bit(const pp_alignments* in, pp_alignments* out, pp_2bit** owner);
void pp_2bit_free(pp_2bit* owner);

/* The assembly: Pileup::new input (pileup.rs:178-187) as loaded by misc::load_fasta (misc.rs:38-167). */
typedef struct {
  uint32_t n_contigs;
  const uint64_t* off;  /* [n_contigs+1] start of each contig in bases; off[n_contigs] = total bp (< 2^32-64) */
  const uint8_t* bases; /* upper-cased ASCII, contigs concatenated                                            */
} pp_contigs;

/* polish options (main.rs:78-108; validation polish.rs:277-287 is done by the caller-facing layers) */
typedef struct {
  double fraction_invalid; /* -i, default 0.2 */
  double fraction_valid;   /* -v, default 0.5 */
  uint32_t max_errors;     /* -m, default 10  */
  uint32_t min_depth;      /* -d, default 5   */
  int32_t careful;         /* --careful       */
} pp_polish_params;

#define PP_N_STAGES 8
typedef struct {
  float total_ms;               /* CUDA-event time of the whole device path of this call            */
  float stage_ms[PP_N_STAGES];  /* 0 reset (chain heads, status), 1 classify (fallback k pre-pass, normally 0), 2 goodness / k of every
                                   alignment under the call's options, 3 tile (CIGAR walk, pileup in shared memory, ordered depth,
                                   vote), 4 compaction, 5 unused, 6 h2d (pp_polish: upload + position binning of the dataset), 7 d2h */
  uint32_t launches;            /* kernels of this library launched during the call                 */
  uint32_t reserved;
} pp_timing;

typedef struct {
  /* caller-allocated outputs (may be NULL to leave the result on the device; fetch later) */
  uint64_t* out_off;    /* [n_contigs+1] start of each polished contig in out_bases                  */
  uint8_t* out_bases;   /* polished bases, '-' already removed (polish.rs:188), contigs concatenated */
  uint64_t out_cap;     /* capacity of out_bases in bytes                                            */
  uint64_t* changed;    /* [n_contigs] positions with status Changed (polish.rs:173-176), may be NULL */
  uint64_t* zero_depth; /* [n_contigs] positions with depth == 0 (polish.rs:178-180), may be NULL     */
  double* total_depth;  /* [n_contigs] sum over positions of the f64 depth (polish.rs:177; mean read depth of the log =
                           total_depth / contig length), may be NULL.  Per-position depths are the reference's exactly; their
                           sum is accumulated in parallel, so it can differ from the reference's sequential sum in the last bits */
  /* filled by the library */
  uint64_t out_len;     /* total polished bases (if > out_cap nothing was copied: PP_ERR_ARG)        */
  uint64_t n_aln_used;  /* Σ good alignments (alignment.rs:304, polish.rs:121)                       */
  int64_t error_aln;    /* for PP_ERR_INPUT raised by one alignment: its index, else -1              */
  pp_timing timing;
} pp_polish_result;

/* One call = process_one_read for every group (alignment.rs:275-305) + Pileup::add_alignment for every good
 * alignment (pileup.rs:189-200, alignment.rs:175-201,364-378) + PileupBase::get_polished_seq for every
 * position (pileup.rs:67-134) + the '-' stripping join of polish_one_sequence (polish.rs:185-188).
 * Host buffers in, host buffers out; H2D/D2H inside. */
int pp_polish(pp_ctx* ctx, const pp_contigs* contigs, const pp_alignments* alns,
              const pp_polish_params* params, pp_polish_result* result);

/* Device-resident variant (kernel-path timing; repeated polishing with different options):
 * upload once, polish many times, fetch when wanted. */
int pp_dataset_upload(pp_ctx* ctx, const pp_contigs* contigs, const pp_alignments* alns);
int pp_polish_resident(pp_ctx* ctx, const pp_polish_params* params, pp_polish_result* result);


/* Per-position record of the last polish on ctx, for the --debug TSV (polish.rs:230-266, pileup.rs:137-166).
 * Recording is off by default (it costs 56 B per position); switch it on before the polish call. */
typedef struct {
  double depth;                 /* pileup.rs:31 */
  uint32_t valid_threshold, invalid_threshold;  /* pileup.rs:70-72 */
  uint32_t count[6];            /* A, C, G, T, "-", and the draft's own base when it is not A/C/G/T */
  uint32_t n_other;             /* entries carrying any other allele (their distinct strings: pp_polish_debug_alleles) */
  uint32_t new_node;            /* node index of the emitted allele when it is an "other" allele, else 0xFFFFFFFF */
  uint8_t original;             /* pileup.rs:30 */
  uint8_t status;               /* 0 low_depth 1 none 2 multiple 3 too_close 4 kept 5 changed (pileup.rs:18-25,156-163) */
  uint8_t new_char;             /* emitted single character ('-' for a deletion) when new_node == 0xFFFFFFFF */
  uint8_t pad[5];
} pp_debug_pos;
typedef struct {                /* one distinct "other" allele of one position */
  uint64_t sig;                 /* 4-bit mode: low nibble = length (1..15) then one BAM code per nibble; 8-bit mode: low byte =
                                   length (1..7) then one byte per base; length field 0 = too long, read it through val */
  uint64_t val;                 /* alignment index << 32 | start in the (strand-corrected) read << 16 | length */
  uint32_t count;
  uint32_t next;                /* next node of the same position, 0xFFFFFFFF = end */
} pp_debug_node;
int pp_polish_set_debug(pp_ctx* ctx, int on /* 1 record, 2 stop recording but keep the last records, 0 off */);
int pp_polish_debug_fetch(pp_ctx* ctx, uint64_t first_pos, uint64_t n_pos, pp_debug_pos* out);
/* head[p] = 1 + index of the first node of global position p (0 = none); nodes[0..*n_nodes) */
int pp_polish_debug_alleles(pp_ctx* ctx, uint32_t* head /* [total bp] */, pp_debug_node* nodes, uint64_t node_cap, uint64_t* n_nodes);

/* ------------------------------------------------------------------------------------------------------
 * filter (filter.rs).  One record per ALIGNED line of one mate's SAM file, in file order.
 * Replaces get_insert_size_thresholds (filter.rs:148-186) and alignment_pass_qc (filter.rs:352-377).
 * ---------------------------------------------------------------------------------------------------- */
typedef struct {
  uint64_t n;
  const uint32_t* name_id;   /* [n] id of QNAME, shared between the two mates (filter.rs:133-135,322-326) */
  const uint32_t* contig;    /* [n] id of RNAME (string equality, filter.rs:161,369)                        */
  const uint32_t* ref_start; /* [n] 0-based                                                                  */
  const uint32_t* ref_end;   /* [n] Alignment::get_ref_end (alignment.rs:138-149)                            */
  const uint8_t* flags;      /* [n] bit0 = reverse strand                                                     */
} pp_filter_mate;

typedef struct {
  int32_t orientation;  /* -1 auto, 0 fr, 1 rf, 2 ff, 3 rr, 4 = any other user string (matches nothing) */
  double low_pct;       /* --low, default 0.1  */
  double high_pct;      /* --high, default 99.9 */
  uint64_t n_names;     /* name ids are < n_names */
} pp_filter_params;

typedef struct {
  uint8_t* pass1;       /* [m1.n] caller-allocated: 1 = line written verbatim, 0 = "\tZP:Z:fail" appended */
  uint8_t* pass2;       /* [m2.n] */
  uint32_t low, high;   /* insert-size thresholds (filter.rs:179-180) */
  int32_t orientation;  /* chosen orientation 0..3 (or 4) */
  uint64_t pairs[4];    /* fr, rf, ff, rr pair counts (filter.rs:223-226) */
  uint64_t n_pass;      /* filter.rs:345 pass counts, both mates */
  pp_timing timing;
} pp_filter_result;

int pp_filter(pp_ctx* ctx, const pp_filter_mate* m1, const pp_filter_mate* m2,
              const pp_filter_params* params, pp_filter_result* result);

/* ------------------------------------------------------------------------------------------------------
 * Host layer (text <-> packed), exported so that the CLI, the Python mirror and a Rust host share one
 * implementation.  No GPU needed for these.
 * ---------------------------------------------------------------------------------------------------- */
typedef struct pp_fasta pp_fasta;
/* misc::load_fasta (misc.rs:38-167): plain or gzip (magic 1f 8b), upper-cased, checks of misc.rs:56-75. */
pp_fasta* pp_fasta_load(const char* path, char* err, size_t errcap);
void pp_fasta_free(pp_fasta* f);
void pp_fasta_view(const pp_fasta* f, pp_contigs* out);
const char* pp_fasta_name(const pp_fasta* f, uint32_t i);
const char* pp_fasta_description(const pp_fasta* f, uint32_t i);

typedef struct pp_pack pp_pack;
/* SAM text -> pp_alignments.  Restates the text side of add_to_pileup (alignment.rs:225-272) and
 * Alignment::new (alignment.rs:49-98): line skipping, column checks, NM / ZP tags, CIGAR validation,
 * QNAME grouping, source sequence of SEQ="*" records. */
pp_pack* pp_pack_create(const pp_fasta* f, int careful);
void pp_pack_free(pp_pack* p);
/* A BAM file (recognised by content: a BGZF block that inflates to "BAM\1", never by its name; pipes are always SAM) is parsed as
 * its SAM text: the stored header text, then one line per record (SAMv1 §4.2's columns with the NM and ZP tags, a CG:B:I array in
 * place of the long-CIGAR placeholder), so results, messages and "(line N)" numbers are those of that text.  PP_ERR_IO, with a
 * message naming the file, for what only BAM can get wrong: not BGZF, a CRC32 / ISIZE mismatch, a record past its block_size or
 * past the end of the data, a refID / next_refID out of range, malformed optional fields, no BGZF end-of-file block. */
int pp_pack_add_sam_file(pp_pack* p, const char* path);                        /* PP_OK / PP_ERR_INPUT / PP_ERR_IO */
/* big files are parsed by several host threads (same result, same errors); 0 threads = one per hardware thread */
int pp_pack_set_threads(pp_pack* p, uint32_t n_threads, uint64_t min_chunk_bytes);
int pp_pack_add_sam_text(pp_pack* p, const char* text, size_t len, const char* name_for_errors);
/* one logical SAM file fed in chunks of whole lines (a host reading a pipe; the synthetic generator) */
int pp_pack_stream_begin(pp_pack* p, const char* name_for_errors);
int pp_pack_stream_feed(pp_pack* p, const char* text, size_t len);
int pp_pack_stream_end(pp_pack* p);
int pp_pack_finish(pp_pack* p, pp_alignments* out);                             /* arrays owned by p */
const char* pp_pack_error(const pp_pack* p);
/* name of the RNAME of alignment i when contig[i] == PP_CONTIG_UNKNOWN, and the QNAME of alignment i */
const char* pp_pack_unknown_ref(const pp_pack* p, uint64_t aln);
const char* pp_pack_read_name(const pp_pack* p, uint64_t aln);
int pp_pack_cigar_string(const pp_pack* p, uint64_t aln, char* out, size_t cap); /* rebuilt from the packed ops */
/* per file: aligned records and read groups (the stderr line of polish.rs:117-119) */
int pp_pack_file_stats(const pp_pack* p, uint32_t file, uint64_t* alignments, uint64_t* reads);

/* ------------------------------------------------------------------------------------------------------
 * SAM text -> packed alignments ON THE DEVICE (SURVEY.md §8f-1).  Same result as pp_pack_* + pp_dataset_upload, bit for bit
 * (Alignment::new alignment.rs:49-98, get_expanded_cigar :325-346, the grouping of add_to_pileup :238-263 and the
 * SEQ="*" handling of process_one_read :275-295), but the parse runs in HBM: the host only streams the file's bytes.
 *   pp_tok_begin(ctx, assembly, careful, 4)  ->  pp_tok_add_file / pp_tok_add_text per SAM, in order  ->  pp_tok_finish
 *   ->  pp_polish_resident.
 * Return values beyond PP_OK / PP_ERR_*:
 *   PP_TOK_HOST   the text holds something the device tokeniser leaves to the host packer (a malformed line, a read group
 *                 without SEQ, an empty file, a size limit): run pp_pack_* on the same input, which yields the result
 *                 or the reference's own error message.  Not an error by itself.
 *   PP_TOK_NEED8  a SEQ character outside "ACMGRSVTWYHKDBN" while seq_bits == 4: start again with seq_bits = 8.
 * After either, the construction is abandoned (pp_tok_begin starts a new one).
 * ---------------------------------------------------------------------------------------------------- */
#define PP_TOK_HOST 1
#define PP_TOK_NEED8 2
typedef struct {
  uint64_t lines, alignments, reads;   /* of this file (alignment.rs:266-271's log line) */
  float h2d_ms;                        /* wall time of getting the text into HBM (file read + pinned staging + PCIe) */
  float device_ms;                     /* CUDA-event time of the tokeniser kernels */
  uint32_t launches;
  uint64_t h2d_bytes;                  /* bytes that crossed PCIe for this file (less than its size when QUAL was dropped) */
} pp_tok_stats;
int pp_tok_begin(pp_ctx* ctx, const pp_fasta* assembly, int careful, int seq_bits /* 4 | 8 */);
int pp_tok_add_text(pp_ctx* ctx, const char* text, size_t len, pp_tok_stats* stats /* may be NULL */);
/* A BAM file (as in pp_pack_add_sam_file) is inflated on the host, its image crosses PCIe and is decoded one record per thread;
 * the result is the same as for its SAM text.  Its stats count records as lines, and h2d_ms covers read, inflate, record walk
 * and PCIe.  Anything the host must word (a structural fault included) is PP_TOK_HOST.  pp_tok_prefetch of a BAM does nothing. */
int pp_tok_add_file(pp_ctx* ctx, const char* path, pp_tok_stats* stats /* may be NULL */);
/* Several files in order, pipelined: file i+1 streams into a second text buffer while file i is tokenised.  SAM and BAM may mix. */
int pp_tok_add_files(pp_ctx* ctx, const char* const* paths, int n_paths, pp_tok_stats* stats /* [n_paths] or NULL */);
/* Optional, any time after pp_create: start streaming `path` into HBM in the background (one outstanding upload);
 * the next pp_tok_add_file(s) that starts with the same path picks it up.  Lets the upload overlap the FASTA load. */
int pp_tok_prefetch(pp_ctx* ctx, const char* path);
/* Optional, after pp_tok_begin: total bytes of all the files to come, so that the arrays are sized once. */
int pp_tok_expect(pp_ctx* ctx, uint64_t total_text_bytes);
int pp_tok_finish(pp_ctx* ctx);        /* the tokenised alignments + the assembly become the resident dataset */
/* Optional, between pp_tok_begin and pp_tok_finish: this context keeps only a SHARD of the assembly (contig sharding without the
 * host in the middle: every GPU tokenises the text itself, over its own PCIe link).  local_of[c], c < the assembly's contig count:
 * the contig's index inside shard_contigs, or 0xFFFFFFFF = another shard's.  At pp_tok_finish the records of foreign contigs
 * become PP_FLAG_GHOST records (they still count for goodness / k / --careful, exactly like pp_shards_build's), the others are
 * renumbered, and shard_contigs replaces the assembly as the resident draft.  takes_unknown: the one shard that keeps records whose
 * RNAME is not in the assembly, so that the reference's error is raised once.  The arrays are copied during the call. */
int pp_tok_set_shard(pp_ctx* ctx, const uint32_t* local_of, uint32_t n_contigs_total, const pp_contigs* shard_contigs, int takes_unknown);
/* n byte ranges of a SAM file for n GPUs: cuts[0] = 0, cuts[n] = the file size, every other cut is the start of a line whose QNAME
 * differs from the line before it, so that no read group (alignment.rs:214-272) is split.  PP_ERR_IO: not a plain file / a line longer
 * than 1 MiB.  (pp_polish_files_multi gives range g of every file to GPU g, then the GPUs exchange read groups by contig.) */
int pp_sam_split_ranges(const char* path, int n, uint64_t* cuts /* [n + 1] */);   /* SAM only: PP_ERR_IO for a BAM file */
/* Multi-GPU ingestion, the building blocks of pp_polish_files_multi (polish.rs:109-134 load_alignments over N GPUs).  Per context g:
 *   pp_tok_begin -> pp_tok_set_ranges(off, len, n_files): this context reads only bytes [off[f], off[f] + len[f]) of file f
 *   (range g of pp_sam_split_ranges) -> pp_tok_add_files(the same n_files paths on every context).
 * Then ONE call for all contexts, instead of pp_tok_finish: pp_tok_exchange_finish hands every read group, whole, to each GPU that
 * owns a contig one of its records lies on (owner[c] = context of contig c, local_of[g][c] = index of contig c inside
 * shard_contigs[g] or 0xFFFFFFFF; peer copies on the device, global SAM order = (file, range, line)), marks the foreign records
 * PP_FLAG_GHOST, installs shard_contigs[g] as context g's draft and bins: every context is then ready for pp_polish_resident.
 * PP_TOK_HOST: more than 32 contexts / 64 files, or something the host path must look at.  n_aln_total = aligned records read. */
/* (SAM only: pp_tok_add_files answers PP_TOK_HOST when a file of a ranged list is BAM; pp_polish_files_multi cuts BAM files by record.) */
int pp_tok_set_ranges(pp_ctx* ctx, const uint64_t* off, const uint64_t* len, int n_files);
int pp_tok_exchange_finish(pp_ctx* const* ctxs, int n_ctx, const uint32_t* owner, uint32_t n_contigs_total, const uint32_t* const* local_of,
                           const pp_contigs* shard_contigs /* [n_ctx] */, uint64_t* n_aln_total);
/* Which parser pp_polish_files uses for its SAM files: 0 (default) the device tokeniser, with the host packer taking over
 * on PP_TOK_HOST and for --debug / multi-GPU runs; 1 the host packer only.  Both give the same bytes. */
int pp_set_parser(pp_ctx* ctx, int mode);
int pp_get_parser(const pp_ctx* ctx);
/* Host threads pp_tok_add_file uses to stream a file into HBM (pread -> pinned slot -> PCIe); 0 = a quarter of the cores, 2..16. */
int pp_tok_set_readers(pp_ctx* ctx, int n);
/* Optional (default 0): pp_tok_add_file(s) / pp_tok_prefetch stage the text with QUAL (column 11: 45 % of a bwa-mem line,
 * never read by polish, alignment.rs:49-98) replaced by "*", so that 40 % less crosses PCIe.  Same arrays, same result; it pays
 * only where the PCIe link is narrower than what the reader threads can strip (measured on this pod: 20-30 ms instead of
 * 13-20 ms per 626 MB file, i.e. slower).  `filter`, which reproduces its input lines, always uploads byte for byte.  With it on,
 * the line count in pp_tok_stats includes one comment line per upload slice. */
int pp_tok_set_strip_qual(pp_ctx* ctx, int on);
/* The resident dataset read back (tests: equality with the host packer's arrays).  pp_dataset_sizes fills the counts of
 * `out`; pp_dataset_download copies into the caller's arrays (same counts; NULL pointers are skipped). */
int pp_dataset_sizes(pp_ctx* ctx, pp_alignments* out);
int pp_dataset_download(pp_ctx* ctx, const pp_alignments* into);

/* Contig sharding across GPUs (one pp_ctx per GPU, no collective): whole contigs per shard, each with its alignments
 * in SAM order; reads that also map to another shard's contigs keep their k through PP_FLAG_GHOST records. */
typedef struct pp_shards pp_shards;
pp_shards* pp_shards_build(const pp_contigs* contigs, const pp_alignments* alns, uint32_t n_shards);
/* the same with the contig -> shard assignment given by the caller (NULL = the sharder's own longest-processing-time packing) and,
 * when only_shard >= 0, only that shard built (the others stay empty): one rank of a multi-process run builds just its own. */
pp_shards* pp_shards_build_assigned(const pp_contigs* contigs, const pp_alignments* alns, uint32_t n_shards,
                                    const uint32_t* shard_of_contig, int32_t only_shard);
int pp_shards_get(const pp_shards* s, uint32_t i, pp_contigs* contigs, pp_alignments* alns,
                  const uint32_t** contig_map /* original index of each shard contig */, uint64_t* n_home);
void pp_shards_free(pp_shards* s);

/* Whole commands (the functions the CLI calls; same behaviour, error text and exit status as the
 * reference's polish::polish (polish.rs:26-38) and filter::filter (filter.rs:26-37)).
 * out_fasta receives exactly what the reference prints to stdout; free with pp_free.
 * pp_polish_files parses its SAM files with the device tokeniser (pp_tok_*) unless pp_set_parser(ctx, 1), a --debug run, or
 * PP_TOK_HOST / a data error send it through pp_pack_*.  Any of `sams` may be a BAM file instead (pp_pack_add_sam_file): same output,
 * log and errors as its SAM text. */
int pp_polish_files(pp_ctx* ctx, const char* assembly, const char* const* sams, int n_sams,
                    const pp_polish_params* params, const char* debug_path, char** out_fasta,
                    uint64_t* out_len, int verbose /* 1: reference-style log on stderr */);
/* the same command over several GPUs of one box: contigs shard across ctxs[0..n_ctx) (one host thread per GPU); every GPU tokenises
 * its byte range of every SAM file and the read groups change GPUs on the device (pp_tok_set_ranges / pp_tok_exchange_finish).  A BAM
 * file is inflated once on the host and every GPU decodes its range of the records, cut between read groups. */
int pp_polish_files_multi(pp_ctx* const* ctxs, int n_ctx, const char* assembly, const char* const* sams, int n_sams,
                          const pp_polish_params* params, const char* debug_path, char** out_fasta,
                          uint64_t* out_len, int verbose);
/* `polypolish filter` (filter.rs:26-37).  With pp_set_parser(ctx, 0) (default) the SAM text stays on the device from parse to
 * write (quick parse alignment.rs:102-149, QNAME/RNAME interning = the keys of filter.rs:110-145, pp_filter's kernels on the
 * arrays in place, output text of filter.rs:296-349 assembled in HBM); anything unusual, and pp_set_parser(ctx, 1), use the host
 * text code.  Same bytes and messages either way. */
int pp_filter_files(pp_ctx* ctx, const char* in1, const char* in2, const char* out1, const char* out2,
                    const char* orientation, double low, double high, int verbose);
/* `polypolish filter` followed by `polypolish polish` on its output, as ONE call (SURVEY.md §8f-2): both SAM files cross PCIe once,
 * the filter's verdict stays in HBM as the ZP flag of the tokenised records (what the ZP:Z:fail tag carries through the intermediate
 * files: filter.rs:334-342, alignment.rs:72-74), and the polished FASTA is byte for byte that of the two commands.  out1 / out2 may
 * be NULL: the filtered SAM files are then not written at all.  Anything unusual falls back to the two commands through files. */
int pp_filter_polish_files(pp_ctx* ctx, const char* assembly, const char* in1, const char* in2, const char* out1, const char* out2,
                           const char* orientation, double low, double high, const pp_polish_params* params, char** out_fasta,
                           uint64_t* out_len, int verbose);
void pp_free(void* p);

/* ------------------------------------------------------------------------------------------------------
 * Synthetic inputs (measurement / test support; SURVEY.md §8d).  Deterministic in `seed`.
 * ---------------------------------------------------------------------------------------------------- */
typedef struct {
  uint64_t seed;
  uint32_t n_contigs;
  uint32_t read_len;          /* 150 */
  uint64_t contig_len;        /* truth bases per contig */
  double depth;               /* mean read depth */
  double insert_mean, insert_sd; /* 400, 40 (clipped to [200,700]) */
  double draft_error_rate;    /* 1e-4 per bp: 50 % substitutions, 25 % / 25 % 1-bp indels */
  double seq_sub_rate;        /* 2e-3 per base */
  double seq_indel_rate;      /* 1e-4 per base */
  double repeat_fraction;     /* 0.03 of the genome in repeat families with 7,5,3,2,4 copies */
  double clip_rate, highnm_rate, unaligned_rate; /* 0.005 each */
} pp_synth_params;
typedef struct pp_synth pp_synth;
pp_synth* pp_synth_create(const pp_synth_params* prm);
/* the same, plus repeat families (3, 2, 5, 7 copies) whose copies lie on DIFFERENT contigs, covering `cross_contig_fraction`
 * of the assembly: reads in them multi-map across contigs, so under contig sharding their k spans GPUs (BASELINE config 5). */
pp_synth* pp_synth_create_shared(const pp_synth_params* prm, double cross_contig_fraction);
/* cross-contig data sets only: restrict the generated reads to those with a record on a contig of `shard` (contig i belongs to
 * shard_of_contig[i], or i % n_shards when NULL); n_shards = 0 switches the restriction off.  What is emitted is, record for
 * record, what pp_shards_build_assigned gives that shard from the whole data set - a rank of an N-GPU run can build its share of
 * BASELINE config 5 without generating the other ranks' reads. */
int pp_synth_set_shard_filter(pp_synth* s, uint32_t n_shards, uint32_t shard, const uint32_t* shard_of_contig);
/* worker threads of pp_synth_write_sam / pp_synth_feed_pack for data sets with per-pair streams (pp_synth_create_shared with a
 * cross-contig fraction > 0); 0 = one per hardware thread.  The bytes produced do not depend on it. */
int pp_synth_set_threads(pp_synth* s, uint32_t n_threads);
void pp_synth_free(pp_synth* s);
uint64_t pp_synth_total_bp(const pp_synth* s);    /* draft bases */
uint64_t pp_synth_n_pairs(const pp_synth* s);
int pp_synth_write_fasta(const pp_synth* s, const char* path, int truth /* 0 = draft */);
int pp_synth_write_sam(const pp_synth* s, int mate /* 1 | 2 */, const char* path);
/* the same records as BAM (BGZF, level 6, with the end-of-file block), compressed on the worker threads of pp_synth_set_threads */
int pp_synth_write_bam(const pp_synth* s, int mate /* 1 | 2 */, const char* path);
pp_fasta* pp_synth_fasta(const pp_synth* s);      /* the draft as a loaded assembly (free with pp_fasta_free) */
int pp_synth_feed_pack(const pp_synth* s, int mate, pp_pack* pack); /* same text, streamed into the packer */

#ifdef __cplusplus
}
#endif
#endif /* PP_ABI_H */
