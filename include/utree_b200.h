/* utree_b200.h -- C ABI of the B200-native SEARCH_GG hot path.
 *
 * The reference (knights-lab/UTree, itree.c) has no library/FFI interface
 * ("Gutted the API because nobody (would) use(d) it", itree.c:27-29); its
 * search binary is main() -> XT_read32() -> XT_doSearch32().  This header is
 * the boundary a maintainer would bind instead of those two calls: plain C,
 * pointers and sizes only, int return codes (0 = ok), no exceptions, no CPU
 * fallback -- every entry point fails with UTB_ERR_CUDA when no sm_100 device
 * is usable.  INTEGRATION.md shows the replacement main().
 *
 *   reference                                this header
 *   ---------------------------------------  ---------------------------------
 *   XT_read32()            itree.c:733-828   utb_ctr_open + utb_db_upload
 *   readSamplesFPdelim()   itree.c:1202-1223 (inside utb_ctr_open)
 *   XT_doSearch32()        itree.c:833-1108  utb_search_file / utb_search_mem
 *     XT_INITIATE_WS       itree.c:860-901     framing kernels (exact host reader behind them;
 *                                              FASTQ, wrapped FASTA: utb_searcher_set_input)
 *     XT_WORD_SEARCH       itree.c:903-933     pack + sieve kernels
 *     XT_getIX32/xtSuffixBS itree.c:699-730    table lookup kernel (or the probe sequence verbatim)
 *     full aufbau vote     itree.c:1028-1098   vote kernels
 *     fprintf lines        itree.c:1032-1096   format kernels
 *   main() search branch   itree.c:1357-1377 utb_main
 */
#ifndef UTREE_B200_H
#define UTREE_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- error codes (never exceptions) -------------------------------------- */
enum {
    UTB_OK = 0,
    UTB_ERR_ARG = 1,      /* bad argument                                     */
    UTB_ERR_IO = 2,       /* cannot open / short read                         */
    UTB_ERR_FORMAT = 3,   /* malformed CTR, FASTA or FASTQ                    */
    UTB_ERR_NOMEM = 4,
    UTB_ERR_CUDA = 5,     /* CUDA runtime error or no usable device           */
    UTB_ERR_LIMIT = 6     /* input exceeds a documented limit                 */
};
/* Thread-local message for the last failing call on this thread. */
const char *utb_last_error(void);

/* ---- CTR database on the host (App. A of SURVEY.md) ----------------------- */
typedef struct utb_ctr utb_ctr;
/* Parses header, BinIx, record blob and label tail (itree.c:733-828,
 * 1154-1223).  The file stays mapped; nothing is copied until upload. */
int utb_ctr_open(const char *path, utb_ctr **out);
void utb_ctr_close(utb_ctr *ctr);
uint64_t utb_ctr_num_nodes(const utb_ctr *ctr);   /* metadata[3]              */
uint32_t utb_ctr_ix_bytes(const utb_ctr *ctr);    /* sizeof(IXTYPE): 2 or 4   */
uint32_t utb_ctr_binix_bytes(const utb_ctr *ctr); /* on-disk entry: 4 or 8    */
uint32_t utb_ctr_max_ix(const utb_ctr *ctr);      /* sampIX+1 (itree.c:855)   */
uint64_t utb_ctr_last_bin(const utb_ctr *ctr);    /* BinIx[2^24] (itree.c:792)*/
const char *utb_ctr_label(const utb_ctr *ctr, uint32_t ix);
uint32_t utb_ctr_label_rank(const utb_ctr *ctr, uint32_t ix); /* strcmp order */

/* ---- CTR resident in one GPU's HBM ---------------------------------------- */
typedef struct utb_db utb_db;
int utb_device_count(int *n);
/* Copies prefix index, packed records and label table to `device`.  The host
 * views stay caller-owned.  The returned handle is bound to that device. */
int utb_db_upload(const utb_ctr *ctr, int device, utb_db **out);
void utb_db_free(utb_db *db);
uint64_t utb_db_hbm_bytes(const utb_db *db);
/* 1 when every bucket of the CTR is strictly sorted (what utree-compress
 * emits; the first-bin quirk is handled), so the record words are distinct
 * and the sector hash table (+ sieve) is in use; 0 when the reference's probe
 * sequence is emulated verbatim on the on-disk image. */
int utb_db_lookup_mode(const utb_db *db);
/* A second GPU gets the finished tables from an uploaded one by peer copy
 * (NVLink) instead of a second upload (SURVEY 8e). */
int utb_db_clone(const utb_db *src, int device, utb_db **out);
int utb_db_device(const utb_db *db);

/* ---- per-read result record (what the vote leaves for the formatter) ------ */
enum { UTB_NONE = 0, UTB_STAR = 1, UTB_WALK = 2 };
#define UTB_CUT_EMPTY 0xFFFFFFFFu   /* dv == -1: empty taxonomy               */
#define UTB_CUT_FULL  0xFFFFFFFEu   /* dv == -2: whole label                  */
typedef struct {
    uint32_t kind;    /* UTB_NONE: no line; STAR: "...\t*"; WALK: "...\tsl;ol" */
    uint32_t label;   /* label id whose string / prefix is printed            */
    uint32_t cut;     /* WALK: bytes of the label to print, or EMPTY / FULL   */
    uint32_t found;   /* foundUniq                                            */
    uint32_t uix;     /* distinct labels hit                                  */
    uint32_t sl, ol;  /* WALK only                                            */
    uint32_t _pad;
} utb_result;

/* ---- batches: one stream slot = pinned staging + device buffers ----------- */
typedef struct utb_batch utb_batch;
/* max_bytes: raw FASTA bytes per batch; max_reads: records per batch. */
int utb_batch_create(utb_db *db, size_t max_bytes, size_t max_reads, utb_batch **out);
void utb_batch_destroy(utb_batch *b);
/* Pinned staging the caller fills before submit: raw bytes (sequence lines
 * anywhere inside, headers may stay in between), and per read the byte offset
 * and length of its trimmed sequence line.  Lengths are limited to 16777214
 * bases (LINELEN, itree.c:836). */
char *utb_batch_bytes(utb_batch *b);
uint64_t *utb_batch_seq_off(utb_batch *b);
uint32_t *utb_batch_seq_len(utb_batch *b);
size_t utb_batch_max_bytes(const utb_batch *b);
size_t utb_batch_max_reads(const utb_batch *b);
/* Number of 32-base position slots a read of `len` bases occupies on the
 * device; a batch may not exceed utb_batch_max_slots() in total. */
uint64_t utb_read_slots(uint32_t len);
uint64_t utb_batch_max_slots(const utb_batch *b);
/* Asynchronous: H2D copy, pack, lookup, vote, D2H of results on the batch's
 * stream.  The caller must not touch the pinned staging until wait returns. */
int utb_batch_submit(utb_batch *b, size_t n_bytes, size_t n_reads, int do_rc);
/* Blocks until the batch is done; *results points at n_reads records in
 * pinned memory, valid until the next submit on this batch. */
int utb_batch_wait(utb_batch *b, const utb_result **results);
/* Pinned, per read: where its name sits in the raw bytes.  The search
 * pipeline fills them for the format kernels, which build the output LINES
 * (itree.c:1032, 1040, 1096) on the device. */
uint32_t *utb_batch_name_off(utb_batch *b);
uint32_t *utb_batch_name_len(utb_batch *b);
/* Re-runs only the device stages on the inputs already resident from the last
 * submit (no PCIe traffic) `iters` times and reports CUDA-event milliseconds
 * per stage, summed over iters: ms[0]=pack ms[1]=lookup ms[2]=vote ms[3]=total.
 * Also reports how many kernels were launched. */
int utb_batch_rerun_device(utb_batch *b, int iters, float ms[4], uint64_t *launches);
/* Counters of the last submit: valid 32-mer windows x strands (= lookups). */
int utb_batch_counts(utb_batch *b, uint64_t *lookups, uint64_t *hits);
/* Two-phase lookup detail of the last run: ms[0] sieve kernel, ms[1] survivor
 * kernel; sectors[0] lookups the sieve answered (one 16-byte block is fetched
 * per POSITION and serves both strands), sectors[1] table sectors the exact
 * lookup touched.  ms and sectors[0] are zero when the single lookup kernel
 * ran (sieve off). */
int utb_batch_lookup_detail(utb_batch *b, float ms[2], uint64_t sectors[2]);

/* ---- stage-level entry points (parity tests call the kernels 1:1) --------- */
/* words[n] (host) -> ix[n] (host): label id or 0xFFFFFFFF, exactly
 * XT_getIX32 (itree.c:720-730). */
int utb_lookup_words(utb_db *db, const uint64_t *words, size_t n, uint32_t *ix);
/* One trimmed sequence (host) -> for every base position i the forward and
 * reverse-complement 32-mer words and a valid flag (itree.c:906-926).
 * fwd/rc/valid have room for len entries; entries i > len-32 are invalid. */
int utb_pack_sequence(utb_db *db, const char *seq, uint32_t len,
                      uint64_t *fwd, uint64_t *rc, uint8_t *valid);
/* hits (host; label ids, 0xFFFFFFFF = miss) of n_reads reads laid out
 * back to back, read r owning hits[off[r] .. off[r+1]) -> vote results
 * (itree.c:1028-1098). */
int utb_vote_hits(utb_db *db, const uint32_t *hits, const uint64_t *off,
                  size_t n_reads, utb_result *results);
/* The same vote through the representation the batch pipeline uses (per read
 * the list of the labels that hit, misses left out; thread-per-read kernel, with
 * the warp and block kernels behind it for label-rich and long reads). */
int utb_vote_hits_sparse(utb_db *db, const uint32_t *hits, const uint64_t *off,
                         size_t n_reads, utb_result *results);

/* ---- host stages (no GPU involved; CPU tests drive them directly) --------- */
/* The reference's record reader (itree.c:866-890) over a byte buffer: lines
 * are taken strictly in pairs, name = bytes after '>' up to the first ' ',
 * '\n' or NUL, sequence = the line cut at a NUL, minus one '\n' and one '\r'.
 * Fills one entry per complete record (at most max_reads), *used = byte after
 * the last framed record.  A malformed record stops the framing: the records
 * before it are valid, the call returns UTB_ERR_FORMAT and *ref_exit = 2. */
int utb_frame_records(const char *buf, size_t n, int eof, int threads, size_t max_reads,
                      uint64_t *seq_off, uint32_t *seq_len, uint32_t *name_off, uint32_t *name_len,
                      size_t *n_reads, size_t *used, int *ref_exit);
/* The FASTQ twin of utb_frame_records (strict 4-line records, see
 * utb_searcher_set_input): per read also the offset of its quality line,
 * whose length equals seq_len.  On a malformed record the call returns
 * UTB_ERR_FORMAT, the records before it are valid, *err_record is its
 * 1-based number and *err_code one of UTB_FQ_*; otherwise both are 0. */
enum {
    UTB_FQ_NOHEADER = 1,     /* header line does not begin with '@'              */
    UTB_FQ_NOSEPARATOR = 2,  /* third line does not begin with '+'               */
    UTB_FQ_QUALLEN = 3,      /* quality length differs from sequence length      */
    UTB_FQ_TOOLONG = 4,      /* a line of UTB_LINELEN (16777216) bytes or more   */
    UTB_FQ_TRUNCATED = 5     /* the input ends inside a record                   */
};
int utb_frame_fastq_records(const char *buf, size_t n, int eof, int threads, size_t max_reads,
                            uint64_t *seq_off, uint32_t *seq_len, uint64_t *qual_off, uint32_t *name_off, uint32_t *name_len,
                            size_t *n_reads, size_t *used, size_t *err_record, int *err_code);
/* The wrapped-FASTA framer (UTB_INPUT_FASTA_WRAPPED, see utb_searcher_set_input):
 * the joined sequence of read r is seq_out[seq_off[r] .. +seq_len[r]), the
 * reads back to back; seq_cap >= n is required (a joined sequence is never
 * longer than its lines).  With eof = 0 the record after the last header line
 * is carried: *used stops before it, since without the next header it is not
 * known to be complete.  At most max_reads records are framed.  On a malformed
 * record the call returns UTB_ERR_FORMAT, the records before it are valid,
 * *err_record is its 1-based number and *err_code one of UTB_FW_*; otherwise
 * both are 0. */
enum {
    UTB_FW_NOHEADER = 1,     /* the input does not begin with '>'                */
    UTB_FW_TOOLONG = 4       /* a line of UTB_LINELEN (16777216) bytes or more,
                              * or a joined sequence of more than 16777214 bases */
};
int utb_frame_wrapped_records(const char *buf, size_t n, int eof, int threads, size_t max_reads,
                              char *seq_out, size_t seq_cap, uint64_t *seq_off, uint32_t *seq_len,
                              uint32_t *name_off, uint32_t *name_len,
                              size_t *n_reads, size_t *used, size_t *err_record, int *err_code);
/* The reference's output lines (itree.c:1032, 1040, 1096) for n_reads result
 * records; names are taken from bytes[name_off[r] .. +name_len[r]). */
int utb_format_results(const utb_ctr *ctr, const char *bytes, const uint32_t *name_off, const uint32_t *name_len,
                       const utb_result *results, size_t n_reads, char *out, size_t out_cap, size_t *out_len);

/* ---- whole search (XT_doSearch32 + output, itree.c:833-1108) -------------- */
typedef struct {
    uint64_t reads;        /* records parsed ("Searched N queries")            */
    uint64_t good_finds;   /* reads with >= 1 hit ("Good finds: N")            */
    uint64_t lookups;      /* valid windows x strands                          */
    uint64_t hits;
    uint64_t batches;
    uint64_t kernel_launches;
    uint64_t h2d_bytes, d2h_bytes;
    uint64_t out_bytes;
    double seconds_total;  /* wall, excludes DB upload                         */
    double seconds_device; /* sum of CUDA-event time over batches (all GPUs)   */
    /* where the two host threads' wall time went (seconds) */
    double rd_wait_slot, rd_fill, rd_frame, rd_submit;   /* reader team leader   */
    double fm_wait_gpu, fm_format, fm_emit;              /* formatter team leader */
} utb_stats;

typedef struct utb_searcher utb_searcher;
/* devices[n_devices]: GPUs to shard batches over (DB replicated on each).
 * host_threads: framing/formatting workers (the CLI's [threads] argument). */
int utb_searcher_create(const utb_ctr *ctr, const int *devices, int n_devices,
                        int host_threads, utb_searcher **out);
void utb_searcher_destroy(utb_searcher *s);
/* FASTA in a file -> output file, lines in input order (== reference at
 * threads=1).  Returns UTB_OK, or UTB_ERR_FORMAT with *ref_exit set to the
 * reference's exit code (2) after writing every line that precedes the bad
 * record, as the reference does. */
int utb_search_file(utb_searcher *s, const char *fasta_path, const char *out_path,
                    int do_rc, utb_stats *stats, int *ref_exit);
/* Same with host buffers: fasta[n] in (a page-locked buffer is copied to the
 * devices from where it lies), *out / *out_len = the output text.  The text
 * lives in a page-locked arena that BELONGS TO THE SEARCHER (the devices copy
 * their lines straight into it): it stays valid until the next search on this
 * searcher or utb_searcher_destroy, and is kept between searches.  utb_free is
 * a no-op kept for the round-1 ABI. */
int utb_search_mem(utb_searcher *s, const char *fasta, size_t n, int do_rc,
                   char **out, size_t *out_len, utb_stats *stats, int *ref_exit);
void utb_free(void *p);

/* The reference CLI contract (itree.c:1357-1377, SURVEY App. C): argv parse,
 * stdout banner, exit codes.  Returns the process exit code. */
int utb_main(int argc, char **argv);

/* ---- the non-GG search binary (utree-search, itree.c with -D SEARCH; SURVEY 8f-3) ---- */
/* Same loader, packing and lookups; the slide skips PACKSIZE/SPARSITY - 1 = 7
 * windows after every hit (itree.c:948-951) and the vote is the shallow top-2
 * plurality of itree.c:969-1007 with its 4-column "%f" line.  That vote is
 * single-threaded in the reference and reads one entry past the hit list of
 * a read (itree.c:982), i.e. depends on the reads before it: the device looks
 * up and selects, the formatter thread votes read by read.  Call before the
 * first search; utb_search_file / utb_search_mem then produce that output. */
int utb_searcher_set_shallow(utb_searcher *s, int on);
int utb_main_shallow(int argc, char **argv);

/* ---- input format ----------------------------------------------------------- */
/* utb_search_file / utb_search_mem read linearised FASTA (two lines per
 * record) by default.  UTB_INPUT_FASTQ switches them to strict 4-line FASTQ:
 *   header     begins with '@'; the name is the bytes after it up to the first
 *              ' ' or the newline (a tab does not end it; with CRLF input a
 *              '\r' stays in a name without a space, as for FASTA);
 *   sequence   one trailing '\r' trimmed; a byte that is not ACGTacgt breaks
 *              windows, as for FASTA;
 *   separator  begins with '+'; the rest of the line is ignored;
 *   quality    one trailing '\r' trimmed; its length must equal the sequence
 *              length; its bytes are not otherwise checked.
 * Every line is shorter than 16777216 bytes.  Wrapped (multi-line) FASTQ is a
 * format error.  An empty sequence with an empty quality is a read without
 * windows.  The last record may lack its final '\n' (not when its quality line
 * is empty).  A NUL byte is an ordinary byte: it stays in a name and, in a
 * sequence, breaks windows like any byte that is not a base (the FASTA reader
 * instead cuts the name and the sequence line at a NUL, as the reference's
 * strlen() does).  For input without NUL bytes the output is byte for byte
 * that of the same search on the FASTA made of each record's header (with '>'
 * for '@') and sequence line.  A
 * malformed record is handled as for FASTA: every line of the records before
 * it is written, the search returns UTB_ERR_FORMAT with *ref_exit = 2, and
 * utb_last_error() names the 1-based record and the rule (UTB_FQ_*).
 * min_qual = q > 0 (FASTQ only, q <= 222): a base whose quality byte is below
 * 33 + q counts as 'N', so every window over it is skipped.  The caller's
 * buffer is never modified.  Call before a search, like
 * utb_searcher_set_shallow; memory the FASTQ path needs is allocated here.
 *
 * UTB_INPUT_FASTA_WRAPPED (min_qual must be 0) reads FASTA whose sequences
 * span any number of lines, as genomes and assemblies are usually written:
 *   records    a header is a line that begins with '>'; every following line
 *              up to the next header, or to the end of the input, belongs to
 *              that record's sequence.  Lines may have any length (ragged
 *              widths are fine).
 *   name       as for FASTA: the bytes after '>' up to the first ' ' or the
 *              line end; a '\r' stays in a name that has no space.
 *   sequence   the record's non-header lines concatenated, each without its
 *              '\n' and one '\r' directly before the line end (or before the
 *              end of the input).  Empty lines add nothing.  Any other byte is
 *              kept: a '>' inside a line, ';' or a NUL is an ordinary byte and
 *              breaks windows like any byte that is not a base.
 *   empty      a header followed by another header, or by the end of the
 *              input, is a read without windows.  The last line may lack its
 *              '\n'.
 * Malformed input: the input does not begin with '>' (a leading blank line
 * included; UTB_FW_NOHEADER), or a line of 16777216 bytes or more counting its
 * '\n', or a joined sequence of more than 16777214 bases (UTB_FW_TOOLONG).  It
 * is handled as for FASTQ: every line of the records before the bad one is
 * written, the search returns UTB_ERR_FORMAT with *ref_exit = 2, and
 * utb_last_error() names the 1-based record and the rule.  A record larger
 * than the batch buffer in bytes (lines averaging under about 1.5 bases, or
 * millions of blank lines, below the base limit) is refused with the
 * pipeline's "record larger than the batch buffer" error; batches are grown to
 * at least 64 MiB + 4 KiB here.  For input without NUL bytes the output is
 * byte for byte that of the same search in UTB_INPUT_FASTA mode on lin(input),
 * which writes each record's header line unchanged, then its joined sequence,
 * then '\n' (GG and shallow, RC on and off, one or many devices).  The
 * sequences are joined on the device; the caller's buffer is never written,
 * and what this input needs is allocated here, not inside a search. */
enum { UTB_INPUT_FASTA = 0, UTB_INPUT_FASTQ = 1, UTB_INPUT_FASTA_WRAPPED = 2 };
int utb_searcher_set_input(utb_searcher *s, int format, uint32_t min_qual);

/* ---- utree-compress equivalent (XT_cmp32, itree.c:1234-1315; SURVEY 8f-2) -- */
/* .ubt -> .ctr, byte-identical to the reference compressor (first-bin quirk
 * included).  Host only. */
int utb_compress_ubt(const char *ubt_path, const char *ctr_path, uint64_t *n_records, uint32_t *n_labels);
/* The COMPRESS binary's CLI contract (itree.c:1352-1355). */
int utb_compress_main(int argc, char **argv);

/* ---- utree-build_gg equivalent (itree.c:501-635, 268-307, 1317-1343; SURVEY 8f-4) ---- */
typedef struct {
    uint64_t map_bytes, map_lines;   /* "Parsed map. N bytes, M lines."                     */
    uint64_t sequences;              /* FASTA records                                       */
    uint64_t kmers_seen;             /* k-mer occurrences that pass the complevel rule      */
    uint64_t kmers_made;             /* distinct words ("Done with sequence parse: N k-mers made") */
    uint64_t records;                /* good words written ("Total nodes in tree")          */
    uint32_t labels;                 /* label ids handed out, superseded ones included      */
} utb_build_stats;
/* FASTA (one header + one sequence line per genome) + two-column map (name <tab> label)
 * -> .ubt (+ <out>.gg.log), byte-identical to the reference builder for complevel 0..4: the
 * k-mers are extracted, stably sorted and relabelled on `device`; gg = 0 gives the plain
 * BUILD rule (a second label makes a word bad).  *ref_exit: the reference's exit code for
 * malformed input (1, 2, 4). */
int utb_build_ubt(const char *fasta_path, const char *map_path, const char *out_path, uint32_t complevel, int gg, int ix_bytes,
                  int device, utb_build_stats *st, int *ref_exit);
/* The BUILD_GG binary's CLI contract (itree.c:1379-1408). */
int utb_build_main(int argc, char **argv);

/* ---- measurement helpers --------------------------------------------------- */
/* Random 32-byte-sector gather bandwidth over a working set of ws_bytes on
 * `device` (the roofline denominator of SURVEY 8d).  loads: sectors read. */
int utb_measure_rand32(int device, uint64_t ws_bytes, uint64_t loads, int iters,
                       double *gbs);

#ifdef __cplusplus
}
#endif
#endif
