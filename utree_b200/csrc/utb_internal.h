/* utb_internal.h -- shared between the host C files and the CUDA TU. */
#ifndef UTB_INTERNAL_H
#define UTB_INTERNAL_H
#include "../../include/utree_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

#define UTB_NUMBINS ((1u << 24) + 1u)   /* itree.c:693 */
#define UTB_LINELEN 16777216u           /* itree.c:836 */
#define UTB_MAXSEQ (UTB_LINELEN - 2u)   /* longest sequence line the reference handles */
#define UTB_BAD32 0xFFFFFFFFu

/* Host view of a CTR file (memory-mapped; label table parsed). */
struct utb_ctr {
    int fd;
    void *map;
    size_t map_len;
    uint64_t num_nodes;
    uint32_t ix_bytes;      /* 2 / 4 */
    uint32_t binix_bytes;   /* 4 / 8 */
    uint32_t sz;            /* 5 + ix_bytes */
    uint32_t max_ix;        /* number of distinct labels */
    const uint8_t *binix_raw;   /* UTB_NUMBINS entries of binix_bytes */
    const uint8_t *recs;        /* num_nodes * sz bytes */
    uint64_t last_bin;
    /* label table: NUL-terminated strings back to back, padded */
    char *blob;
    size_t blob_len;
    uint32_t *off;          /* max_ix + 1 offsets into blob */
    uint32_t *rank;         /* rank[ix]: position of label ix in strcmp order */
    uint32_t *by_rank;      /* inverse permutation */
};

void utb_set_error(const char *fmt, ...);

/* What a batch hands back to the host. */
typedef enum {
    UTB_OUT_RESULTS,      /* one utb_result per read (utb_batch_submit / utb_batch_wait) */
    UTB_OUT_TEXT,         /* the output lines, kept on the device (utb_batch_wait_len, then _text_to / _text_piece) */
    UTB_OUT_SELECTIONS    /* non-GG mode: the ids each read selected (utb_batch_wait_shallow) */
} utb_batch_out;

/* What the search pipeline (pipeline.c) uses of kernels.cu beyond the public header. */
int utb_batch_prepare(utb_batch *b, utb_batch_out out, int chunked);
int utb_batch_submit_ex(utb_batch *b, const char *src, size_t n_bytes, size_t n_reads, int do_rc, utb_batch_out out, uint64_t total_groups);
int utb_batch_submit_chunk(utb_batch *b, const char *src, size_t n_bytes, size_t n_reads, int do_rc, utb_batch_out out);
int utb_batch_set_input(utb_batch *b, int format, uint32_t min_qual, int chunked);   /* format: UTB_INPUT_* */
uint64_t *utb_batch_qual_off(utb_batch *b);   /* pinned, per read: where its quality line starts (FASTQ batches) */
char *utb_batch_join(utb_batch *b);           /* pinned, max_bytes: the joined sequences of a host-framed wrapped-FASTA batch */
int utb_batch_frame_error(const utb_batch *b, size_t *record, int *code);
size_t utb_batch_reads(const utb_batch *b);
uint64_t utb_batch_launches(const utb_batch *b);
int utb_batch_last_ms(utb_batch *b, float ms[4]);
int utb_batch_wait_len(utb_batch *b, size_t *len, uint64_t *good_finds);
int utb_batch_text_to(utb_batch *b, char *dst, size_t len);
int utb_batch_text_piece(utb_batch *b, size_t off, size_t *len, const char **piece);
int utb_batch_wait_shallow(utb_batch *b, const uint32_t **sel_cnt, const uint32_t **sel, size_t *sel_total,
                           const uint32_t **name_off, const uint32_t **name_len);
int utb_batch_sync(utb_batch *b);
/* Sample profile of the later submits of a text batch: mode 0 off, 1 with the text, 2 instead of it (the format
 * kernels do not run).  The first mode != 0 allocates a key table for max_keys distinct keys per batch. */
int utb_batch_set_profile(utb_batch *b, int mode, size_t max_keys);
/* After utb_batch_wait_len: the batch's (key = label << 32 | printed length, reads) pairs, *n of them. */
int utb_batch_profile(utb_batch *b, const uint64_t **pairs, size_t *n);
/* The most reads per batch, at most max_reads, for which the worst-case output text of a batch of max_bytes raw
 * bytes (every read printing its name and the longest label, max_label bytes with the NUL) fits the 32-bit offsets
 * of the format kernels; 0 if none does. */
size_t utb_text_max_reads(size_t max_bytes, size_t max_reads, size_t max_label);
int utb_host_ptr_is_pinned(const void *p);
int utb_pinned_alloc(size_t n, void **out);
void utb_pinned_free(void *p);

/* ctr_loader.c: the header of a CTR that utb_ctr_open refused as truncated, for the CLI's messages. */
int utb_ctr_probe(const char *path, uint64_t md[4], uint64_t *binix_read);

#ifdef __cplusplus
}
#endif
#endif
