/* pipeline.c -- host side of the search: FASTA framer (the reference's record
 * reader XT_INITIATE_WS, itree.c:860-901), batch scheduler over one or more
 * GPUs, and the ordered output formatter (the fprintf lines of itree.c:1032,
 * 1040, 1096).
 *
 * Two thread teams share the [threads] the CLI is given:
 *   reader team    -- fills the pinned staging buffer of the next free batch
 *                     slot straight from the input (parallel pread / memcpy),
 *                     frames the records in place (parallel newline count,
 *                     then parallel record parse keyed by line parity), and
 *                     submits the batch.  No per-read copies: the device gets
 *                     the file bytes as they are plus one (offset, length)
 *                     pair per read.
 *   formatter team -- waits for batches in sequence order and moves the lines
 *                     the device built for each to the output, in order
 *                     (parallel pwrite / memcpy; a page-locked output arena
 *                     takes them straight from the device).
 * Slots are dealt round-robin over the devices, the database being replicated
 * on each, so multi-GPU needs no collective: the ordered merge is the only
 * cross-device step (SURVEY 8e).
 */
#define _GNU_SOURCE
#define _FILE_OFFSET_BITS 64
#include "utb_internal.h"
#include <errno.h>
#include <fcntl.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/syscall.h>
#include <sys/vfs.h>
#include <time.h>
#include <unistd.h>

#define SLOTS_PER_DEVICE 4                         /* measured on B200, ms per 10 M reads (profiles/r02_e2e_sweep.txt): 2 slots 42.9, 3: 36.0, 4: 35.5, 5: 38.0, 6: 37.6 */
#define DEFAULT_BATCH_BYTES ((size_t)128 << 20)   /* ~2.3 ms of PCIe per batch: launch and sync costs are a few percent of that */
#define RAMP_BYTES ((size_t)32 << 20)              /* first / last batches: small, so the pipeline fills and drains fast */
#define MAX_TEAM 64
#define MAX_RECORD(lines) ((lines) * (size_t)UTB_LINELEN + 4096)   /* a record of maximal lines, and slack */

/* ---- thread team: leader + helpers, fork/join with barriers ----------------- */
typedef void (*team_fn)(void *ctx, int part, int nparts);
typedef struct {
    int n;                      /* members including the leader */
    pthread_t th[MAX_TEAM];
    pthread_barrier_t start, end;
    team_fn fn;
    void *ctx;
    volatile int quit;
    struct team_arg { void *team; int id; } arg[MAX_TEAM];
} team_t;

static void *team_helper(void *a_) {
    struct team_arg *a = (struct team_arg *)a_;
    team_t *t = (team_t *)a->team;
    int id = a->id;
    for (;;) {
        pthread_barrier_wait(&t->start);
        if (t->quit) break;
        t->fn(t->ctx, id, t->n);
        pthread_barrier_wait(&t->end);
    }
    return NULL;
}
static int team_init(team_t *t, int n) {
    memset(t, 0, sizeof *t);
    if (n < 1) n = 1;
    if (n > MAX_TEAM) n = MAX_TEAM;
    t->n = n;
    if (n == 1) return 0;
    pthread_barrier_init(&t->start, NULL, (unsigned)n);
    pthread_barrier_init(&t->end, NULL, (unsigned)n);
    for (int i = 1; i < n; ++i) {
        t->arg[i].team = t; t->arg[i].id = i;
        if (pthread_create(&t->th[i], NULL, team_helper, &t->arg[i])) return -1;
    }
    return 0;
}
static void team_run(team_t *t, team_fn fn, void *ctx) {
    if (t->n == 1) { fn(ctx, 0, 1); return; }
    t->fn = fn; t->ctx = ctx;
    pthread_barrier_wait(&t->start);
    fn(ctx, 0, t->n);
    pthread_barrier_wait(&t->end);
}
static void team_destroy(team_t *t) {
    if (t->n <= 1) return;
    t->quit = 1;
    pthread_barrier_wait(&t->start);
    for (int i = 1; i < t->n; ++i) pthread_join(t->th[i], NULL);
    pthread_barrier_destroy(&t->start);
    pthread_barrier_destroy(&t->end);
}

/* ---- searcher ----------------------------------------------------------------- */
typedef struct {
    utb_batch *b;
    int dev_index;
    size_t n_bytes, n_reads;
    uint32_t *name_off, *name_len;
    uint64_t first_read;           /* global index of the slot's first read */
    uint64_t src_off;              /* offset in the input stream of the batch's first byte */
    const char *host_bytes;        /* where this batch's raw bytes live on the host (staging, or the caller's pinned buffer) */
    int state;                     /* 0 free, 1 submitted */
} slot_t;

struct utb_searcher {
    const utb_ctr *ctr;
    int n_devices;
    int *devices;
    utb_db **dbs;
    int n_slots;
    slot_t *slots;
    int host_threads;
    size_t batch_bytes, batch_reads, ramp_bytes;
    size_t max_label;              /* longest label incl. NUL */
    int verbose;                   /* CLI: progress lines on stdout */
    int device_frame;              /* records framed on the GPU (default): the host only cuts chunks at a "\n>" */
    int shallow;                   /* the non-GG binary's search (-D SEARCH): SPARSITY-skip slide + shallow vote (utb_searcher_set_shallow) */
    uint32_t *horses; size_t horses_cap;   /* its AllTheKingsHorses (itree.c:970): survives from read to read within a search */
    uint32_t *tally;               /* its Hashes (itree.c:971) */
    char *arena; size_t arena_cap; /* page-locked output of utb_search_mem: the devices copy their text straight into it; valid until
                                    * the next search on this searcher or its destruction */
    int spread;                    /* more than one physical GPU: page-locked buffers are interleaved over the NUMA nodes */
    int format;                    /* UTB_INPUT_FASTA, _FASTQ (4-line) or _FASTA_WRAPPED (utb_searcher_set_input) */
    uint32_t min_qual;             /* FASTQ: bases with a quality byte below 33 + min_qual count as 'N' (0: off) */
};

static double now_s(void) {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

/* A searcher over several GPUs: its page-locked buffers (batch staging, output arena) are read and written by all of
 * them, so their pages are spread over the NUMA nodes instead of landing on the node of the thread that happened to
 * allocate them (one socket's memory controllers would carry every GPU's DMA).  Best effort: a kernel that refuses
 * set_mempolicy (seccomp) leaves the default placement. */
static void mem_interleave(int on) {
#ifdef SYS_set_mempolicy
    unsigned long mask = 0;
    if (on) {
        FILE *f = fopen("/sys/devices/system/node/online", "r");
        if (!f) return;
        int a, b; char sep;
        while (fscanf(f, "%d", &a) == 1) {
            b = a;
            if (fscanf(f, "%c", &sep) == 1 && sep == '-') { if (fscanf(f, "%d", &b) != 1) b = a; if (fscanf(f, "%c", &sep) != 1) sep = 0; }
            for (int n = a; n <= b && n < 64; ++n) mask |= 1ul << n;
            if (sep != ',') break;
        }
        fclose(f);
        if (!(mask & (mask - 1))) return;                          /* one node: nothing to spread */
    }
    (void)syscall(SYS_set_mempolicy, on ? 3 /* MPOL_INTERLEAVE */ : 0 /* MPOL_DEFAULT */, on ? &mask : NULL, on ? 65ul : 0ul);
#else
    (void)on;
#endif
}

/* the output lines of a batch are built on the device: long labels take fewer reads per batch */
static size_t batch_reads_for(utb_searcher *s) {
    s->batch_reads = utb_text_max_reads(s->batch_bytes, s->batch_bytes / 64, s->max_label);
    return s->batch_reads;
}
/* (Re)creates the batches of every slot with s->batch_bytes, prepared for the searcher's mode: nothing is allocated
 * inside a search.  All or nothing: the new batches replace the old ones only when every one of them could be made. */
static int slots_create(utb_searcher *s) {
    utb_batch **nb = (utb_batch **)calloc((size_t)s->n_slots, sizeof(utb_batch *));
    if (!nb) { utb_set_error("out of memory"); return UTB_ERR_NOMEM; }
    int rc = UTB_OK;
    for (int i = 0; i < s->n_slots && !rc; ++i) {
        if (s->spread) mem_interleave(1);
        rc = utb_batch_create(s->dbs[i % s->n_devices], s->batch_bytes, s->batch_reads, &nb[i]);
        if (!rc) rc = utb_batch_prepare(nb[i], UTB_OUT_TEXT, s->device_frame);
        if (!rc && s->shallow) rc = utb_batch_prepare(nb[i], UTB_OUT_SELECTIONS, s->device_frame);
        if (!rc && s->format != UTB_INPUT_FASTA) rc = utb_batch_set_input(nb[i], s->format, s->min_qual, s->device_frame);
        if (s->spread) mem_interleave(0);
    }
    for (int i = 0; i < s->n_slots; ++i) {
        slot_t *sl = &s->slots[i];
        if (rc) { utb_batch_destroy(nb[i]); continue; }
        utb_batch_destroy(sl->b);
        sl->b = nb[i];
        sl->dev_index = i % s->n_devices;
        sl->name_off = utb_batch_name_off(sl->b);                  /* pinned: the device formatter reads them too */
        sl->name_len = utb_batch_name_len(sl->b);
    }
    free(nb);
    return rc;
}

int utb_searcher_create(const utb_ctr *ctr, const int *devices, int n_devices,
                        int host_threads, utb_searcher **out) {
    if (!ctr || !out || n_devices < 1 || !devices) { utb_set_error("utb_searcher_create: bad argument"); return UTB_ERR_ARG; }
    *out = NULL;
    utb_searcher *s = (utb_searcher *)calloc(1, sizeof(*s));
    if (!s) { utb_set_error("out of memory"); return UTB_ERR_NOMEM; }
    s->ctr = ctr; s->n_devices = n_devices; s->host_threads = host_threads < 1 ? 1 : host_threads;
    const char *e = getenv("UTB_BATCH_MB");
    s->batch_bytes = e && atoi(e) > 0 ? (size_t)atoi(e) << 20 : DEFAULT_BATCH_BYTES;
    if (s->batch_bytes < MAX_RECORD(2)) s->batch_bytes = MAX_RECORD(2);   /* one max record must fit */
    e = getenv("UTB_HOST_FRAME");
    s->device_frame = !(e && atoi(e) != 0);
    for (uint32_t i = 0; i < ctr->max_ix; ++i) {
        size_t l = ctr->off[i + 1] - ctr->off[i];
        if (l > s->max_label) s->max_label = l;
    }
    if (!batch_reads_for(s)) { free(s); utb_set_error("batch too large for device-side formatting"); return UTB_ERR_LIMIT; }
    s->devices = (int *)malloc(sizeof(int) * (size_t)n_devices);
    s->dbs = (utb_db **)calloc((size_t)n_devices, sizeof(utb_db *));
    e = getenv("UTB_SLOTS");                                       /* stream slots per device (tuning) */
    int spd = e && atoi(e) >= 2 && atoi(e) <= 8 ? atoi(e) : SLOTS_PER_DEVICE;
    s->n_slots = n_devices * spd;
    e = getenv("UTB_RAMP_MB");
    s->ramp_bytes = e && atoi(e) > 0 ? (size_t)atoi(e) << 20 : RAMP_BYTES;
    s->slots = (slot_t *)calloc((size_t)s->n_slots, sizeof(slot_t));
    if (!s->devices || !s->dbs || !s->slots) { utb_searcher_destroy(s); utb_set_error("out of memory"); return UTB_ERR_NOMEM; }
    /* one upload + table build (PCIe); a repeated device shares that handle, every further GPU gets the
     * finished tables by peer copy over NVLink (SURVEY 8e) */
    for (int d = 1; d < n_devices; ++d) if (devices[d] != devices[0]) s->spread = 1;
    { const char *sp = getenv("UTB_NUMA_SPREAD"); if (sp) s->spread = atoi(sp) != 0; }
    for (int d = 0; d < n_devices; ++d) {
        s->devices[d] = devices[d];
        int rc = UTB_OK, shared = -1;
        for (int e = 0; e < d; ++e) if (devices[e] == devices[d]) { shared = e; break; }
        if (shared >= 0) s->dbs[d] = s->dbs[shared];
        else if (d == 0) rc = utb_db_upload(ctr, devices[d], &s->dbs[d]);
        else rc = utb_db_clone(s->dbs[0], devices[d], &s->dbs[d]);
        if (rc) { s->n_devices = d; utb_searcher_destroy(s); return rc; }
    }
    int rc = slots_create(s);
    if (rc) { utb_searcher_destroy(s); return rc; }
    *out = s;
    return UTB_OK;
}

/* Switches the searcher to what the reference's OTHER search binary computes (utree-search, itree.c built with
 * -D SEARCH): the slide skips 7 windows after every hit (itree.c:948-951) and the vote is the shallow top-2
 * plurality of itree.c:969-1007, whose result for a read depends on the reads before it.  The device looks up and
 * selects; the order-dependent vote and the "%f" column are done by the formatter thread, read by read. */
int utb_searcher_set_shallow(utb_searcher *s, int on) {
    if (!s) { utb_set_error("utb_searcher_set_shallow: null searcher"); return UTB_ERR_ARG; }
    s->shallow = on ? 1 : 0;
    if (!on) return UTB_OK;
    if (!s->tally) s->tally = (uint32_t *)calloc(s->ctr->max_ix ? s->ctr->max_ix : 1, sizeof(uint32_t));
    if (!s->tally) { utb_set_error("out of memory"); return UTB_ERR_NOMEM; }
    for (int i = 0; i < s->n_slots; ++i) {
        int rc = utb_batch_prepare(s->slots[i].b, UTB_OUT_SELECTIONS, s->device_frame);
        if (rc) return rc;
    }
    return UTB_OK;
}

int utb_searcher_set_input(utb_searcher *s, int format, uint32_t min_qual) {
    if (!s || format < UTB_INPUT_FASTA || format > UTB_INPUT_FASTA_WRAPPED || (format != UTB_INPUT_FASTQ && min_qual) || min_qual > 222) {
        utb_set_error("utb_searcher_set_input: bad argument (format %d, min_qual %u)", format, min_qual);
        return UTB_ERR_ARG;
    }
    /* on failure the searcher keeps its batches and its format */
    const int old_format = s->format;
    const uint32_t old_qual = s->min_qual;
    /* a batch must hold one FASTQ record of four maximal lines; wrapped FASTA takes the same floor */
    if (format != UTB_INPUT_FASTA && s->batch_bytes < MAX_RECORD(4)) {
        const size_t keep = s->batch_bytes;
        s->batch_bytes = MAX_RECORD(4);
        int rc = batch_reads_for(s) ? UTB_OK : UTB_ERR_LIMIT;
        if (rc) utb_set_error("batch too large for device-side formatting");
        s->format = format; s->min_qual = min_qual;
        if (!rc) rc = slots_create(s);
        if (rc) { s->batch_bytes = keep; batch_reads_for(s); s->format = old_format; s->min_qual = old_qual; }
        return rc;
    }
    for (int i = 0; i < s->n_slots; ++i) {
        int rc = utb_batch_set_input(s->slots[i].b, format, min_qual, s->device_frame);
        if (rc) {                                                  /* back to the old format: allocates nothing */
            for (int j = 0; j < i; ++j) (void)utb_batch_set_input(s->slots[j].b, old_format, old_qual, s->device_frame);
            return rc;
        }
    }
    s->format = format; s->min_qual = min_qual;
    return UTB_OK;
}

void utb_searcher_destroy(utb_searcher *s) {
    if (!s) return;
    if (s->slots) for (int i = 0; i < s->n_slots; ++i) utb_batch_destroy(s->slots[i].b);
    if (s->dbs) for (int d = 0; d < s->n_devices; ++d) {
        int shared = 0;
        for (int e = 0; e < d; ++e) if (s->dbs[e] == s->dbs[d]) shared = 1;
        if (!shared) utb_db_free(s->dbs[d]);
    }
    utb_pinned_free(s->arena);
    free(s->horses); free(s->tally);
    free(s->slots); free(s->dbs); free(s->devices); free(s);
}

/* ---- input source ---------------------------------------------------------------- */
typedef struct {
    int fd;                 /* >= 0: file */
    int seekable;           /* regular file: parallel pread */
    off_t file_off, file_size;
    const char *mem;        /* else memory */
    size_t mem_len, mem_pos;
    int eof;
} source_t;

typedef struct { source_t *src; char *dst; size_t n; int failed; } fill_ctx;
static void fill_part(void *c_, int part, int nparts) {
    fill_ctx *c = (fill_ctx *)c_;
    size_t a = c->n * (size_t)part / (size_t)nparts, b = c->n * (size_t)(part + 1) / (size_t)nparts;
    if (c->src->fd < 0) { memcpy(c->dst + a, c->src->mem + c->src->mem_pos + a, b - a); return; }
    while (a < b) {
        ssize_t k = pread(c->src->fd, c->dst + a, b - a, c->src->file_off + (off_t)a);
        if (k < 0) { if (errno == EINTR) continue; c->failed = 1; return; }
        if (k == 0) { c->failed = 1; return; }
        a += (size_t)k;
    }
}
/* Reads up to cap bytes into dst; returns bytes read or -1. */
static ssize_t src_fill(source_t *s, team_t *team, char *dst, size_t cap) {
    if (s->eof || !cap) return 0;
    if (s->fd >= 0 && !s->seekable) {                 /* pipe / fifo: plain reads */
        size_t got = 0;
        while (got < cap) {
            ssize_t k = read(s->fd, dst + got, cap - got);
            if (k < 0) { if (errno == EINTR) continue; return -1; }
            if (k == 0) { s->eof = 1; break; }
            got += (size_t)k;
        }
        return (ssize_t)got;
    }
    size_t left = s->fd >= 0 ? (size_t)(s->file_size - s->file_off) : s->mem_len - s->mem_pos;
    size_t n = left < cap ? left : cap;
    fill_ctx c = {s, dst, n, 0};
    if (n) team_run(team, fill_part, &c);
    if (c.failed) return -1;
    if (s->fd >= 0) s->file_off += (off_t)n; else s->mem_pos += n;
    if (n == left) s->eof = 1;
    return (ssize_t)n;
}

/* ---- output sink -------------------------------------------------------------------- */
/* memory sink: the searcher's page-locked arena.  The text of a batch goes from the device straight to its
 * final place in it (utb_batch_text_to): no staging buffer, no host memcpy.  The arena is kept for the next
 * search of this searcher (page-locking ~1 GB costs far more than a search). */
typedef struct {
    int fd;                 /* >= 0: file sink; < 0: memory sink */
    utb_searcher *s;
    size_t off;             /* bytes emitted so far */
    size_t hint;            /* expected output size (first allocation) */
    int failed;
    /* file sinks.  stream: not seekable (pipe, tty): plain sequential write().  mapped: a file on a memory
     * file system is written through a moving shared mapping -- pwrite()s to one file serialise on the inode
     * lock (~2.7 GB/s whatever the thread count), page faults of a mapping do not.  Otherwise parallel pwrite. */
    int stream, mapped;
    char *map; size_t map_lo, map_hi, file_len;
} sink_t;
#define SINK_WINDOW ((size_t)256 << 20)

static void sink_unmap(sink_t *k) {
    if (k->map) munmap(k->map, k->map_hi - k->map_lo);
    k->map = NULL; k->map_lo = k->map_hi = 0;
}
/* file sink: sets up how the file is written (after open) */
static void sink_open_file(sink_t *k) {
    struct stat st;
    if (fstat(k->fd, &st) || !S_ISREG(st.st_mode)) { k->stream = 1; return; }
    const char *e = getenv("UTB_OUT_MMAP");
    int want = -1;
    if (e) want = atoi(e) != 0;
    struct statfs fs;
    if (want < 0) want = !fstatfs(k->fd, &fs) && (fs.f_type == 0x01021994 /* tmpfs */ || fs.f_type == 0x858458f6 /* ramfs */);
    if (want && (fcntl(k->fd, F_GETFL) & O_ACCMODE) == O_RDWR) k->mapped = 1;
}
/* at the end of the search: the file gets its true length */
static int sink_close_file(sink_t *k) {
    int bad = 0;
    if (k->mapped || k->file_len) {
        sink_unmap(k);
        if (k->file_len != k->off && ftruncate(k->fd, (off_t)k->off)) bad = 1;
    }
    return bad;
}
/* writes n bytes at file offset o (any thread of a team; stream sinks: the caller keeps them in order) */
static void sink_put(sink_t *k, const char *p, size_t n, size_t o) {
    if (k->fd < 0) { memcpy(k->s->arena + o, p, n); return; }
    if (k->map && o >= k->map_lo && o + n <= k->map_hi) { memcpy(k->map + (o - k->map_lo), p, n); return; }
    while (n) {
        ssize_t w = k->stream ? write(k->fd, p, n) : pwrite(k->fd, p, n, (off_t)o);
        if (w < 0) { if (errno == EINTR) continue; k->failed = 1; return; }
        p += w; o += (size_t)w; n -= (size_t)w;
    }
}

static int sink_reserve(sink_t *k, size_t upto) {
    if (k->fd >= 0) {
        if (!k->mapped || upto <= k->map_hi) return 0;
        /* move the window: [off rounded down to a page, at least SINK_WINDOW further); the file grows with it (sparse) */
        sink_unmap(k);
        const size_t pg = (size_t)sysconf(_SC_PAGESIZE) - 1;       /* a mapping starts on a page of the file */
        const size_t lo = k->off & ~pg;
        size_t hi = lo + SINK_WINDOW;
        if (hi < upto) hi = (upto + pg) & ~pg;
        if (hi > k->file_len) {
            struct statfs fs;                                      /* a store into a mapping of a full file system is a SIGBUS, not an error code */
            if (fstatfs(k->fd, &fs) || (size_t)fs.f_bavail * (size_t)fs.f_bsize < 2 * (hi - lo) || ftruncate(k->fd, (off_t)hi)) { k->mapped = 0; return 0; }
            k->file_len = hi;
        }
        void *m = mmap(NULL, hi - lo, PROT_READ | PROT_WRITE, MAP_SHARED, k->fd, (off_t)lo);
        if (m == MAP_FAILED) { k->mapped = 0; return 0; }          /* pwrite from here on; the file is cut to its length at the end */
        k->map = (char *)m; k->map_lo = lo; k->map_hi = hi;
        return 0;
    }
    utb_searcher *s = k->s;
    if (upto <= s->arena_cap) return 0;
    size_t nc = s->arena_cap ? s->arena_cap + s->arena_cap / 2 : (k->hint > ((size_t)1 << 24) ? k->hint : (size_t)1 << 24);
    if (nc < upto) nc = upto + upto / 4;
    void *m = NULL;
    if (s->spread) mem_interleave(1);
    int arc = utb_pinned_alloc(nc, &m);
    if (s->spread) mem_interleave(0);
    if (arc) { k->failed = 1; return -1; }
    if (s->arena) {
        for (int i = 0; i < s->n_slots; ++i) utb_batch_sync(s->slots[i].b);   /* copies still in flight into the old arena */
        memcpy(m, s->arena, k->off);
        utb_pinned_free(s->arena);
    }
    s->arena = (char *)m; s->arena_cap = nc;
    return 0;
}
/* Kept for callers of the round-1 ABI: the output of utb_search_mem belongs to the searcher (see above). */
void utb_free(void *p) { (void)p; }

/* ---- shared run state ------------------------------------------------------------------ */
typedef struct {
    utb_searcher *s;
    sink_t *sink;
    team_t fmt_team;
    pthread_mutex_t mu;
    pthread_cond_t cv;
    uint64_t submitted;     /* batches handed to the devices */
    uint64_t consumed;      /* batches the formatter is done with */
    int discard;            /* a device-framed batch held a malformed record: output from restart_seq on is dropped, */
    uint64_t restart_seq;   /* the reader rewinds to that batch and frames the rest on the host (exact error path)    */
    uint64_t reads_done;    /* records of the batches consumed so far (device-framed batches report their count on completion) */
    int done_reading;
    int error;              /* sticky UTB_ERR_* from the device side */
    char errmsg[512];
    utb_stats st;
    /* UTB_TIMELINE=1: per-batch host timestamps (s since start) for the first 64 batches */
    double t0, tl_submit[64], tl_framed[64], tl_gpu_done[64], tl_emitted[64]; size_t tl_reads[64];
} run_t;

/* ---- formatter ----------------------------------------------------------------------------- */
static inline char *put_u32(char *p, uint32_t v) {
    char t[10]; int n = 0;
    do { t[n++] = (char)('0' + v % 10u); v /= 10u; } while (v);
    while (n) *p++ = t[--n];
    return p;
}

/* One line per read with >= 1 hit, reads [0, n); shapes of itree.c:1032, 1040, 1096.  out has room for every
 * name plus n * (max_label + 64) + 64 bytes.  Returns the length written. */
static size_t fmt_lines(const utb_ctr *c, const char *bytes, const uint32_t *name_off, const uint32_t *name_len,
                        const utb_result *res, size_t n, char *out) {
    char *p = out;
    for (size_t r = 0; r < n; ++r) {
        const utb_result *v = &res[r];
        if (v->kind == UTB_NONE) continue;
        memcpy(p, bytes + name_off[r], name_len[r]); p += name_len[r];
        *p++ = '\t';
        const char *lab = c->blob + c->off[v->label];
        size_t ll = c->off[v->label + 1] - c->off[v->label] - 1;
        if (v->kind == UTB_WALK) {
            if (v->cut == UTB_CUT_EMPTY) ll = 0;                   /* dv == -1: "" (itree.c:1087) */
            else if (v->cut != UTB_CUT_FULL && v->cut < ll) ll = v->cut;   /* first dv bytes (itree.c:1088) */
        }
        memcpy(p, lab, ll); p += ll;
        *p++ = '\t';
        p = put_u32(p, v->found); *p++ = '\t';
        p = put_u32(p, v->uix); *p++ = '\t';
        if (v->kind == UTB_STAR) *p++ = '*';
        else { p = put_u32(p, v->sl); *p++ = ';'; p = put_u32(p, v->ol); }
        *p++ = '\n';
    }
    return (size_t)(p - out);
}

typedef struct { sink_t *sink; const char *text; size_t len, off; } copy_ctx;
static void copy_part(void *c_, int part, int nparts) {
    copy_ctx *c = (copy_ctx *)c_;
    size_t a = c->len * (size_t)part / (size_t)nparts, b = c->len * (size_t)(part + 1) / (size_t)nparts;
    if (a != b) sink_put(c->sink, c->text + a, b - a, c->off + a);
}
static void copy_all(team_t *team, copy_ctx *c) {
    if (c->sink->fd >= 0 && c->sink->stream) sink_put(c->sink, c->text, c->len, c->off);
    else team_run(team, copy_part, c);
}

/* The shallow vote of the non-GG binary, read by read in input order (itree.c:979-1003).  sel_cnt[r] ids per read,
 * back to back in sel, are what its slide appended to AllTheKingsHorses; `if (!kingsMen++)` (itree.c:982) never
 * fires but bumps the count, so the tally runs over ONE MORE entry: whatever an earlier read of this search left
 * at that index (0 if none did).  Lines go to *buf (*cap bytes, grown as needed). */
static int shallow_vote(utb_searcher *s, const slot_t *sl, const uint32_t *sel_cnt, const uint32_t *sel, size_t sel_total,
                        char **buf, size_t *cap, size_t *n_out, uint64_t *good_out) {
    const utb_ctr *c = s->ctr;
    size_t need = 64;
    for (size_t r = 0; r < sl->n_reads; ++r) if (sel_cnt[r]) need += sl->name_len[r] + s->max_label + 48;
    if (need > *cap) {
        free(*buf);
        *cap = need + (need >> 2);
        *buf = (char *)malloc(*cap);
        if (!*buf) { *cap = 0; utb_set_error("out of memory (formatter)"); return UTB_ERR_NOMEM; }
    }
    char *p = *buf;
    uint64_t good = 0;
    size_t at = 0;
    uint32_t *tally = s->tally;
    for (size_t r = 0; r < sl->n_reads; ++r) {
        const size_t n = sel_cnt[r];
        if (!n) continue;                                          /* itree.c:979 */
        if (at + n > sel_total) { utb_set_error("selected-hit list shorter than its counts"); return UTB_ERR_LIMIT; }
        if (n + 1 > s->horses_cap) {                               /* the reference's array is one zero-filled 2 x 16 Mi block */
            size_t nc = s->horses_cap ? s->horses_cap : 1024;
            while (nc < n + 1) nc <<= 1;
            uint32_t *h = (uint32_t *)realloc(s->horses, nc * sizeof(uint32_t));
            if (!h) { utb_set_error("out of memory (formatter)"); return UTB_ERR_NOMEM; }
            memset(h + s->horses_cap, 0, (nc - s->horses_cap) * sizeof(uint32_t));
            s->horses = h; s->horses_cap = nc;
        }
        uint32_t *horses = s->horses;
        memcpy(horses, sel + at, n * sizeof(uint32_t));            /* itree.c:951 */
        at += n;
        ++good;                                                    /* itree.c:980 */
        const size_t men = n + 1;                                  /* itree.c:982 */
        for (size_t i = 0; i < men; ++i) ++tally[horses[i]];       /* itree.c:984-985 */
        uint32_t most = 0, second = 0, most_ix = 0;
        for (size_t i = 0; i < men; ++i) {                         /* itree.c:988-997 */
            const uint32_t h = tally[horses[i]];
            if (h > most) { second = most; most_ix = horses[i]; most = h; }
            else if (h > second) second = h;
            tally[horses[i]] = 0;
        }
        if (most < 2 || most < 2 * second) { --good; continue; }   /* itree.c:1000: TOLERANCE_THRESHOLD 2, SLACK 2 */
        memcpy(p, sl->host_bytes + sl->name_off[r], sl->name_len[r]); p += sl->name_len[r];
        *p++ = '\t';
        const char *lab = c->blob + c->off[most_ix];
        const size_t ll = c->off[most_ix + 1] - c->off[most_ix] - 1;
        memcpy(p, lab, ll); p += ll;
        p += sprintf(p, "\t%f\t%d\n", (double)1 - (double)second / most, (int)most);   /* itree.c:1002 */
    }
    *n_out = (size_t)(p - *buf);
    *good_out = good;
    return UTB_OK;
}

static void *formatter_main(void *arg) {
    run_t *R = (run_t *)arg;
    utb_searcher *s = R->s;
    char *vote_buf = NULL; size_t vote_cap = 0;                    /* the non-GG mode's lines */
    const int direct = R->sink->fd < 0;                            /* device text -> its final place in the arena */
    for (uint64_t seq = 0;; ++seq) {
        pthread_mutex_lock(&R->mu);
        while (R->submitted <= seq && !R->done_reading) pthread_cond_wait(&R->cv, &R->mu);
        int have = R->submitted > seq;
        pthread_mutex_unlock(&R->mu);
        if (!have) break;
        slot_t *sl = &s->slots[seq % (uint64_t)s->n_slots];
        const char *text = NULL; size_t text_len = 0; uint64_t good = 0;
        double tw = now_s();
        const uint32_t *sel_cnt = NULL, *sel = NULL; size_t sel_total = 0;
        int rc = s->shallow ? utb_batch_wait_shallow(sl->b, &sel_cnt, &sel, &sel_total, NULL, NULL)
                            : utb_batch_wait_len(sl->b, &text_len, &good);
        R->st.fm_wait_gpu += now_s() - tw;
        if (seq < 64) R->tl_gpu_done[seq] = now_s() - R->t0;
        if (rc && !R->error) { R->error = rc; snprintf(R->errmsg, sizeof R->errmsg, "%s", utb_last_error()); }
        sl->n_reads = utb_batch_reads(sl->b);                      /* device-framed: the count came back with the results */
        sl->first_read = R->reads_done;
        pthread_mutex_lock(&R->mu);
        if (!rc && !R->discard && utb_batch_frame_error(sl->b, NULL, NULL)) { R->discard = 1; R->restart_seq = seq; }
        const int discard = R->discard;
        pthread_mutex_unlock(&R->mu);
        if (discard) rc = -1;                                      /* nothing of this batch is emitted or counted */
        if (!rc && s->shallow) {
            double tf = now_s();
            size_t n_out = 0;
            int r2 = shallow_vote(s, sl, sel_cnt, sel, sel_total, &vote_buf, &vote_cap, &n_out, &good);
            if (r2 && !R->error) { R->error = r2; snprintf(R->errmsg, sizeof R->errmsg, "%s", utb_last_error()); }
            R->st.fm_format += now_s() - tf;
            tf = now_s();
            if (!r2 && n_out && !sink_reserve(R->sink, R->sink->off + n_out)) {
                sink_put(R->sink, vote_buf, n_out, R->sink->off);
                R->sink->off += n_out;
                R->st.out_bytes += n_out;
            }
            R->st.good_finds += good;
            R->st.fm_emit += now_s() - tf;
            R->st.d2h_bytes += sl->n_reads * 12 + sel_total * 4 + 4 * 1024 * 8 + 16;
        } else if (!rc) {
            double tf = now_s();
            if (text_len && !sink_reserve(R->sink, R->sink->off + text_len)) {
                if (direct) {
                    int r2 = utb_batch_text_to(sl->b, s->arena + R->sink->off, text_len);
                    if (r2 && !R->error) { R->error = r2; snprintf(R->errmsg, sizeof R->errmsg, "%s", utb_last_error()); }
                } else for (size_t o = 0; o < text_len && !R->error;) {   /* file sink: through the slot's page-locked staging */
                    size_t len = text_len - o;
                    int r2 = utb_batch_text_piece(sl->b, o, &len, &text);
                    if (r2) { R->error = r2; snprintf(R->errmsg, sizeof R->errmsg, "%s", utb_last_error()); break; }
                    copy_ctx cc = {R->sink, text, len, R->sink->off + o};
                    copy_all(&R->fmt_team, &cc);
                    o += len;
                }
                R->sink->off += text_len;
                R->st.out_bytes += text_len;
            }
            R->st.good_finds += good;
            R->st.fm_emit += now_s() - tf;
            R->st.d2h_bytes += text_len + 4 * 1024 * 8 + 16;
        }
        if (!rc) {
            uint64_t lk = 0, ht = 0; float ms[4] = {0, 0, 0, 0};
            utb_batch_counts(sl->b, &lk, &ht);
            utb_batch_last_ms(sl->b, ms);
            R->st.lookups += lk; R->st.hits += ht;
            R->st.seconds_device += 1e-3 * (double)ms[3];
            R->reads_done += sl->n_reads;
            if (s->verbose) {   /* itree.c:878 */
                uint64_t a = sl->first_read, b = sl->first_read + sl->n_reads;
                for (uint64_t m = (a >> 20) + 1; (m << 20) <= b; ++m)
                    printf("Searched %llu queries...\n", (unsigned long long)(m << 20));
            }
        }
        if (seq < 64) R->tl_emitted[seq] = now_s() - R->t0;
        pthread_mutex_lock(&R->mu);
        sl->state = 0;
        R->consumed = seq + 1;
        pthread_cond_broadcast(&R->cv);
        pthread_mutex_unlock(&R->mu);
    }
    free(vote_buf);
    return NULL;
}

/* ---- framer ----------------------------------------------------------------------------------- */
/* The reference reads lines strictly in pairs (itree.c:869-871): line 2r is
 * the header of record r, line 2r+1 its sequence, whatever they contain.  So
 * a line's role follows from its index, which a parallel newline count gives:
 * pass 1 counts '\n' per segment, pass 2 lets every worker parse the records
 * whose header line starts right after a newline of its own segment. */
enum { FE_NONE = 0, FE_NOHEADER, FE_SEQ_GT, FE_EMPTY, FE_TOOLONG };
typedef struct {
    const char *buf; size_t fill; int eof;
    uint64_t *seq_off; uint32_t *seq_len; uint32_t *name_off, *name_len;
    uint64_t *qual_off;            /* FASTQ */
    char *join;                    /* wrapped FASTA: the joined sequences */
    size_t hfirst[MAX_TEAM];       /* wrapped FASTA: first header of each segment (fill: none) */
    uint64_t jsum[MAX_TEAM];       /* wrapped FASTA: sequence bytes of each worker's records, then where they go */
    size_t err_at[MAX_TEAM];       /* wrapped FASTA: where each worker's first bad record starts */
    size_t n_valid;                /* wrapped FASTA: records before the first bad one */
    size_t cnt[MAX_TEAM];          /* newlines per segment (wrapped FASTA: headers) */
    size_t base[MAX_TEAM];         /* newlines before the segment (wrapped FASTA: headers) */
    size_t n_rec;                  /* complete records in the buffer (clamped to max_rec) */
    size_t max_rec;                /* capacity of the per-read arrays */
    size_t err_rec[MAX_TEAM]; int err_code[MAX_TEAM];
    size_t end_of_records;         /* byte after the last complete record */
    /* newline index (fast path): positions of every '\n', per segment, in one arena */
    uint32_t *idx; size_t idx_cap;                 /* arena and its size in entries */
    size_t idx_off[MAX_TEAM], idx_room[MAX_TEAM];  /* region of each segment */
    int has_nul[MAX_TEAM], idx_overflow[MAX_TEAM];
    size_t nl_total;
    uint64_t groups[MAX_TEAM];                     /* 32-base position groups of the records each worker framed */
    int groups_valid;
} frame_ctx;

static void count_part(void *c_, int part, int nparts) {
    frame_ctx *c = (frame_ctx *)c_;
    size_t a = c->fill * (size_t)part / (size_t)nparts, b = c->fill * (size_t)(part + 1) / (size_t)nparts;
    size_t n = 0;
    const char *p = c->buf + a, *e = c->buf + b;
    while (p < e) {
        const char *q = (const char *)memchr(p, '\n', (size_t)(e - p));
        if (!q) break;
        ++n; p = q + 1;
    }
    c->cnt[part] = n;
}

/* Parses record r whose header line starts at s (itree.c:879-890). */
static inline size_t parse_record(frame_ctx *c, size_t r, size_t s, int *err) {
    const char *buf = c->buf;
    size_t fill = c->fill;
    const char *h = buf + s;
    const char *hnl = (const char *)memchr(h, '\n', fill - s);
    size_t sstart = (size_t)(hnl - buf) + 1;                       /* r < n_rec guarantees both lines exist */
    const char *sq = buf + sstart;
    const char *snl = sstart < fill ? (const char *)memchr(sq, '\n', fill - sstart) : NULL;
    size_t send = snl ? (size_t)(snl - buf) + 1 : fill;            /* one past the line incl. '\n' */
    *err = FE_NONE;
    if (sstart - s >= UTB_LINELEN || send - sstart >= UTB_LINELEN) { *err = FE_TOOLONG; return send; }
    if (*h != '>') { *err = FE_NOHEADER; return send; }            /* itree.c:880 */
    if (*sq == '>') { *err = FE_SEQ_GT; return send; }             /* itree.c:886 */
    size_t length = send - sstart;
    const char *nul = (const char *)memchr(sq, 0, length);                     /* strlen(): itree.c:887 */
    if (nul) length = (size_t)(nul - sq);
    if (!length) { *err = FE_EMPTY; return send; }                 /* itree.c:888 */
    if (sq[length - 1] == '\n') --length;                          /* itree.c:889 */
    if (length && sq[length - 1] == '\r') --length;                /* itree.c:890 */
    /* name: after '>' up to the first ' ', '\n' or NUL (itree.c:881-882) */
    size_t hl = sstart - s, nl = 1;
    while (nl < hl && h[nl] && h[nl] != ' ' && h[nl] != '\n') ++nl;
    c->name_off[r] = (uint32_t)(s + 1);
    c->name_len[r] = (uint32_t)(nl - 1);
    c->seq_off[r] = sstart;
    c->seq_len[r] = (uint32_t)length;
    return send;
}

static void frame_part(void *c_, int part, int nparts) {
    frame_ctx *c = (frame_ctx *)c_;
    size_t a = c->fill * (size_t)part / (size_t)nparts, b = c->fill * (size_t)(part + 1) / (size_t)nparts;
    c->err_rec[part] = (size_t)-1; c->err_code[part] = FE_NONE;
    /* first line start owned by this segment, and its line index */
    size_t s, L;
    if (part == 0) { s = 0; L = 0; }
    else {
        const char *q = a < b ? (const char *)memchr(c->buf + a, '\n', b - a) : NULL;
        if (!q) return;
        s = (size_t)(q - c->buf) + 1; L = c->base[part] + 1;
    }
    for (;;) {
        if (L & 1) {                                               /* a sequence line: its record belongs to whoever owns the header */
            if (s >= b) return;
            const char *q = (const char *)memchr(c->buf + s, '\n', b - s);
            if (!q) return;
            s = (size_t)(q - c->buf) + 1; ++L;
            continue;
        }
        size_t r = L >> 1;
        if (r >= c->n_rec) return;
        int err;
        size_t send = parse_record(c, r, s, &err);
        if (err) { if (r < c->err_rec[part]) { c->err_rec[part] = r; c->err_code[part] = err; } }
        if (r == c->n_rec - 1) c->end_of_records = send;
        /* the next header starts after the sequence line's newline: ours iff that newline is in [a, b) */
        if (send > b || send == 0 || c->buf[send - 1] != '\n') return;
        if (send - 1 < a) return;
        s = send; L += 2;
        if (s > c->fill) return;
    }
}


/* Pass 1 (fast path): one sweep records the position of every newline of the
 * segment and notes whether a NUL byte occurs (AVX2 when the CPU has it). */
#if defined(__x86_64__)
#include <immintrin.h>
__attribute__((target("avx2")))
static size_t index_avx2(const char *buf, size_t a, size_t b, uint32_t *out, size_t room, int *has_nul) {
    const __m256i nl = _mm256_set1_epi8('\n'), zero = _mm256_setzero_si256();
    __m256i accz = zero;
    size_t n = 0, i = a;
    for (; i + 32 <= b; i += 32) {
        __m256i v = _mm256_loadu_si256((const __m256i *)(buf + i));
        uint32_t m = (uint32_t)_mm256_movemask_epi8(_mm256_cmpeq_epi8(v, nl));
        accz = _mm256_or_si256(accz, _mm256_cmpeq_epi8(v, zero));
        while (m) {
            if (n < room) out[n] = (uint32_t)(i + (size_t)__builtin_ctz(m));
            ++n; m &= m - 1;
        }
    }
    int z = _mm256_movemask_epi8(accz) != 0;
    for (; i < b; ++i) {
        if (buf[i] == '\n') { if (n < room) out[n] = (uint32_t)i; ++n; }
        else if (!buf[i]) z = 1;
    }
    *has_nul = z;
    return n;
}
#endif
static size_t index_scalar(const char *buf, size_t a, size_t b, uint32_t *out, size_t room, int *has_nul) {
    size_t n = 0;
    const char *p = buf + a, *e = buf + b;
    while (p < e) {
        const char *q = (const char *)memchr(p, '\n', (size_t)(e - p));
        if (!q) break;
        if (n < room) out[n] = (uint32_t)(q - buf);
        ++n; p = q + 1;
    }
    *has_nul = memchr(buf + a, 0, b - a) != NULL;
    return n;
}
static void index_part(void *c_, int part, int nparts) {
    frame_ctx *c = (frame_ctx *)c_;
    size_t a = c->fill * (size_t)part / (size_t)nparts, b = c->fill * (size_t)(part + 1) / (size_t)nparts;
    /* arena share proportional to the segment: one newline per 8 bytes, plus slack */
    c->idx_off[part] = a / 8 + 64 * (size_t)part;
    c->idx_room[part] = (b - a) / 8 + 64;
    if (c->idx_off[part] + c->idx_room[part] > c->idx_cap) c->idx_room[part] = c->idx_off[part] < c->idx_cap ? c->idx_cap - c->idx_off[part] : 0;
    uint32_t *out = c->idx + c->idx_off[part];
    size_t n;
#if defined(__x86_64__)
    if (__builtin_cpu_supports("avx2")) n = index_avx2(c->buf, a, b, out, c->idx_room[part], &c->has_nul[part]);
    else
#endif
        n = index_scalar(c->buf, a, b, out, c->idx_room[part], &c->has_nul[part]);
    c->cnt[part] = n;
    c->idx_overflow[part] = n > c->idx_room[part];
}

/* Pass 2 (fast path): records are dealt to the workers by index; line 2r / 2r+1
 * boundaries come from the newline index, no byte is scanned twice.  Only valid
 * when the buffer holds no NUL byte (strlen() semantics are then the identity). */
static void frame_indexed_part(void *c_, int part, int nparts) {
    frame_ctx *c = (frame_ctx *)c_;
    const size_t r0 = c->n_rec * (size_t)part / (size_t)nparts, r1 = c->n_rec * (size_t)(part + 1) / (size_t)nparts;
    c->err_rec[part] = (size_t)-1; c->err_code[part] = FE_NONE; c->groups[part] = 0;
    if (r0 >= r1) return;
    const char *buf = c->buf;
    /* cursor over the global newline sequence: segment sp, local index sk */
    size_t i = r0 ? 2 * r0 - 1 : 0;                /* first newline needed: the one before header r0 (or newline 0) */
    int sp = 0;
    while (sp + 1 < nparts && c->base[sp + 1] <= i) ++sp;
    size_t sk = i - c->base[sp];
#define NEXT_NL(var) do { while (sk >= c->cnt[sp]) { ++sp; sk = 0; } (var) = c->idx[c->idx_off[sp] + sk]; ++sk; ++i; } while (0)
    size_t hs = 0;
    if (r0) { size_t prev; NEXT_NL(prev); hs = prev + 1; }
    uint64_t groups = 0;
    for (size_t r = r0; r < r1; ++r) {
        size_t hn, send, line_end;
        NEXT_NL(hn);
        const size_t ss = hn + 1;
        if (i < c->nl_total) { size_t sn; NEXT_NL(sn); line_end = sn; send = sn + 1; }
        else { line_end = c->fill; send = c->fill; }           /* last line without '\n' (EOF) */
        int err = FE_NONE;
        if (ss - hs >= UTB_LINELEN || send - ss >= UTB_LINELEN) err = FE_TOOLONG;
        else if (buf[hs] != '>') err = FE_NOHEADER;             /* itree.c:880 */
        else if (buf[ss] == '>' && ss < c->fill) err = FE_SEQ_GT;   /* itree.c:886 */
        if (err) { c->err_rec[part] = r; c->err_code[part] = err; break; }
        size_t length = line_end - ss;
        if (length && buf[ss + length - 1] == '\r') --length;   /* itree.c:890 */
        size_t nl = hs + 1;                                     /* name: up to the first ' ' or the newline (itree.c:881) */
        while (nl < hn && buf[nl] != ' ') ++nl;
        c->name_off[r] = (uint32_t)(hs + 1);
        c->name_len[r] = (uint32_t)(nl - hs - 1);
        c->seq_off[r] = ss;
        c->seq_len[r] = (uint32_t)length;
        groups += utb_read_slots((uint32_t)length);
        if (r == c->n_rec - 1) c->end_of_records = send;
        hs = send;
    }
#undef NEXT_NL
    c->groups[part] = groups;
}

static const char *fe_text(int code) {
    switch (code) {
    case FE_NOHEADER: return "ERROR: no header '>'";
    case FE_SEQ_GT: return "ERROR: sequence begins '>'";
    case FE_EMPTY: return "ERROR: empty query line";
    default: return "ERROR: line longer than the reference reader's 16777215-byte limit";
    }
}


/* Frames buf[0..fill): on return *n_out records are valid (those before the
 * first malformed one), *used is the byte after the last complete record,
 * *err is FE_* of the record at index *n_out (or FE_NONE), *dangling tells
 * that at EOF a header line is left without its sequence line. */
static void frame_buffer(team_t *team, frame_ctx *F, size_t *n_out, size_t *n_complete, size_t *used, int *err, int *dangling) {
    int indexed = F->idx != NULL && F->fill < 0xFFFFFFFFull;
    if (indexed) team_run(team, index_part, F); else team_run(team, count_part, F);
    size_t nl_total = 0;
    for (int p = 0; p < team->n; ++p) {
        F->base[p] = nl_total; nl_total += F->cnt[p];
        if (indexed && (F->idx_overflow[p] || F->has_nul[p])) indexed = 0;    /* dense newlines or a NUL: exact byte-wise path */
    }
    F->nl_total = nl_total;
    size_t n_lines = nl_total + ((F->eof && F->fill && F->buf[F->fill - 1] != '\n') ? 1 : 0);   /* a last line without '\n' counts at EOF */
    F->n_rec = n_lines / 2;
    *dangling = F->eof && (n_lines & 1);                       /* header whose sequence fgets fails (itree.c:871-872) */
    if (F->n_rec > F->max_rec) { F->n_rec = F->max_rec; *dangling = 0; }   /* the rest comes back with the carry */
    F->end_of_records = 0;
    for (int p = 0; p < team->n; ++p) { F->err_rec[p] = (size_t)-1; F->err_code[p] = FE_NONE; F->groups[p] = 0; }
    if (F->n_rec) team_run(team, indexed ? frame_indexed_part : frame_part, F);
    size_t n = F->n_rec; *err = FE_NONE;
    for (int p = 0; p < team->n; ++p) if (F->err_rec[p] < n) { n = F->err_rec[p]; *err = F->err_code[p]; }
    F->groups_valid = indexed && n == F->n_rec;                /* per-worker sums cover exactly the framed records */
    *n_out = n; *n_complete = F->n_rec; *used = F->end_of_records;
}

/* ---- FASTQ framer ------------------------------------------------------------------------------ */
/* Strict 4-line records: line 4r is the header of record r, 4r+1 its sequence, 4r+2 the separator, 4r+3 the
 * quality, whatever they contain.  As for FASTA a line's role follows from its index: count_part counts the
 * newlines per segment, then every worker parses the records whose header line starts right after a newline of
 * its own segment.  The rules and their order are those of frame_parse_fastq_kernel, so a chunk the device
 * flagged is re-framed here with the same verdict. */
static inline size_t fq_line(const frame_ctx *c, size_t s, size_t *end) {   /* start of the next line; *end: the '\n' or fill */
    const char *q = s < c->fill ? (const char *)memchr(c->buf + s, '\n', c->fill - s) : NULL;
    *end = q ? (size_t)(q - c->buf) : c->fill;
    return q ? *end + 1 : c->fill;
}
/* Parses record r whose header line starts at hs; returns the byte after its quality line. */
static size_t fq_record(frame_ctx *c, size_t r, size_t hs, int *err) {
    const char *buf = c->buf;
    size_t hn, sn, pn, qn;
    const size_t ss = fq_line(c, hs, &hn), ps = fq_line(c, ss, &sn), qs = fq_line(c, ps, &pn), next = fq_line(c, qs, &qn);
    size_t length = sn - ss, qlength = qn - qs;
    if (length && buf[ss + length - 1] == '\r') --length;
    if (qlength && buf[qs + qlength - 1] == '\r') --qlength;
    *err = FE_NONE;
    if (ss - hs >= UTB_LINELEN || ps - ss >= UTB_LINELEN || qs - ps >= UTB_LINELEN || next - qs >= UTB_LINELEN) *err = UTB_FQ_TOOLONG;
    else if (buf[hs] != '@') *err = UTB_FQ_NOHEADER;
    else if (buf[ps] != '+') *err = UTB_FQ_NOSEPARATOR;
    else if (qlength != length) *err = UTB_FQ_QUALLEN;
    if (*err) return next;
    size_t e = hs + 1;                                             /* name: up to the first ' ' or the newline, as for FASTA */
    while (e < hn && buf[e] != ' ') ++e;
    c->name_off[r] = (uint32_t)(hs + 1);
    c->name_len[r] = (uint32_t)(e - hs - 1);
    c->seq_off[r] = ss; c->seq_len[r] = (uint32_t)length; c->qual_off[r] = qs;
    return next;
}
static void fq_part(void *c_, int part, int nparts) {
    frame_ctx *c = (frame_ctx *)c_;
    size_t a = c->fill * (size_t)part / (size_t)nparts, b = c->fill * (size_t)(part + 1) / (size_t)nparts;
    c->err_rec[part] = (size_t)-1; c->err_code[part] = FE_NONE; c->groups[part] = 0;
    size_t s, L;                                                   /* first line start owned by this segment, and its index */
    if (part == 0) { s = 0; L = 0; }
    else {
        const char *q = a < b ? (const char *)memchr(c->buf + a, '\n', b - a) : NULL;
        if (!q) return;
        s = (size_t)(q - c->buf) + 1; L = c->base[part] + 1;
    }
    while (L & 3) {                                                /* not a header line: its record belongs to an earlier segment */
        const char *q = s < b ? (const char *)memchr(c->buf + s, '\n', b - s) : NULL;
        if (!q) return;
        s = (size_t)(q - c->buf) + 1; ++L;
    }
    uint64_t groups = 0;
    for (size_t r = L >> 2; r < c->n_rec; ++r) {
        int err;
        const size_t next = fq_record(c, r, s, &err);
        if (err) { c->err_rec[part] = r; c->err_code[part] = err; break; }
        groups += utb_read_slots(c->seq_len[r]);
        if (r == c->n_rec - 1) c->end_of_records = next;
        if (next > b || c->buf[next - 1] != '\n') break;          /* the next header is ours iff this record's last newline is in [a, b) */
        s = next;
    }
    c->groups[part] = groups;
}
static const char *fq_text(int code) {
    switch (code) {
    case UTB_FQ_NOHEADER: return "ERROR: FASTQ header line does not begin with '@'";
    case UTB_FQ_NOSEPARATOR: return "ERROR: FASTQ separator line does not begin with '+'";
    case UTB_FQ_QUALLEN: return "ERROR: FASTQ quality length differs from the sequence length";
    case UTB_FQ_TRUNCATED: return "ERROR: truncated FASTQ record";
    default: return "ERROR: line longer than the reference reader's 16777215-byte limit";
    }
}
/* Frames buf[0..fill) as FASTQ: on return *n_out records are valid (those before the first malformed one), *used
 * is the byte after the last complete record, *err is UTB_FQ_* of the record at index *n_out (or FE_NONE); an input
 * that ends inside a record is UTB_FQ_TRUNCATED at index *n_complete. */
static void fq_buffer(team_t *team, frame_ctx *F, size_t *n_out, size_t *n_complete, size_t *used, int *err) {
    team_run(team, count_part, F);
    size_t nl_total = 0;
    for (int p = 0; p < team->n; ++p) { F->base[p] = nl_total; nl_total += F->cnt[p]; }
    const size_t n_lines = nl_total + ((F->eof && F->fill && F->buf[F->fill - 1] != '\n') ? 1 : 0);   /* a last line without '\n' counts at EOF */
    F->n_rec = n_lines / 4;
    int truncated = F->eof && (n_lines & 3);
    if (F->n_rec > F->max_rec) { F->n_rec = F->max_rec; truncated = 0; }   /* the rest comes back with the carry */
    F->end_of_records = 0;
    for (int p = 0; p < team->n; ++p) { F->err_rec[p] = (size_t)-1; F->err_code[p] = FE_NONE; F->groups[p] = 0; }
    if (F->n_rec) team_run(team, fq_part, F);
    size_t n = F->n_rec; *err = FE_NONE;
    for (int p = 0; p < team->n; ++p) if (F->err_rec[p] < n) { n = F->err_rec[p]; *err = F->err_code[p]; }
    if (!*err && truncated) *err = UTB_FQ_TRUNCATED;
    F->groups_valid = n == F->n_rec;                               /* per-worker sums cover exactly the framed records */
    *n_out = n; *n_complete = F->n_rec; *used = F->end_of_records;
}

/* ---- wrapped FASTA framer ---------------------------------------------------------------------- */
/* A header is a line that begins with '>', a record its header and every line up to the next header.  A line's
 * role follows from its first byte, so pass 1 lets every worker count the headers that start in its segment; pass
 * 2 parses the records whose header lies in the segment, walking past its end as far as the record goes, and sums
 * their sequence bytes; pass 3 copies each worker's sequences to where the sums of the workers before it put them.
 * The rules are those of wrap_keep_kernel and wrap_record_kernel, so a chunk the device flagged is re-framed here
 * with the same verdict. */
static void wr_count_part(void *c_, int part, int nparts) {
    frame_ctx *c = (frame_ctx *)c_;
    const size_t a = c->fill * (size_t)part / (size_t)nparts, b = c->fill * (size_t)(part + 1) / (size_t)nparts;
    size_t n = 0, first = c->fill;
    if (a == 0 && b > 0 && c->buf[0] == '>') { n = 1; first = 0; }
    const char *p = c->buf + (a ? a - 1 : 0), *e = c->buf + (b ? b - 1 : 0);   /* a '\n' in [a-1, b-1): a line starts in [a, b) */
    while (p < e) {
        const char *q = (const char *)memchr(p, '\n', (size_t)(e - p));
        if (!q) break;
        if (q[1] == '>') { if (!n) first = (size_t)(q + 1 - c->buf); ++n; }
        p = q + 1;
    }
    c->cnt[part] = n; c->hfirst[part] = first;
}
/* The record whose header starts at hs: *name_end ends its name, *len is the length of its joined sequence (which
 * is written to dst unless that is NULL), *err a UTB_FW_* code or FE_NONE.  Returns where the next record starts. */
static size_t wr_record(const frame_ctx *c, size_t hs, char *dst, size_t *name_end, uint64_t *len, int *err) {
    const char *buf = c->buf;
    const size_t fill = c->fill;
    const char *q = (const char *)memchr(buf + hs, '\n', fill - hs);
    const size_t hn = q ? (size_t)(q - buf) : fill;
    size_t s = q ? hn + 1 : fill;
    *err = s - hs >= UTB_LINELEN ? UTB_FW_TOOLONG : FE_NONE;
    size_t e = hs + 1;                                             /* name: up to the first ' ' or the line end, as for FASTA */
    while (e < hn && buf[e] != ' ') ++e;
    *name_end = e;
    uint64_t n = 0;
    while (s < fill && buf[s] != '>') {                            /* the sequence lines */
        const char *r = (const char *)memchr(buf + s, '\n', fill - s);
        const size_t end = r ? (size_t)(r - buf) : fill, next = r ? end + 1 : fill;
        if (next - s >= UTB_LINELEN) *err = UTB_FW_TOOLONG;
        size_t k = end - s;
        if (k && buf[end - 1] == '\r') --k;                        /* one '\r' before the line end or the end of the input */
        if (dst) memcpy(dst + n, buf + s, k);
        n += k;
        s = next;
    }
    if (n > UTB_MAXSEQ) *err = UTB_FW_TOOLONG;
    *len = n;
    return s;
}
static void wr_part(void *c_, int part, int nparts) {
    frame_ctx *c = (frame_ctx *)c_;
    (void)nparts;
    c->err_rec[part] = (size_t)-1; c->err_code[part] = FE_NONE; c->groups[part] = 0; c->jsum[part] = 0;
    const size_t r1 = c->base[part] + c->cnt[part] < c->n_rec ? c->base[part] + c->cnt[part] : c->n_rec;
    uint64_t groups = 0, js = 0;
    size_t hs = c->hfirst[part];
    for (size_t r = c->base[part]; r < r1; ++r) {
        size_t ne; uint64_t len; int err;
        const size_t next = wr_record(c, hs, NULL, &ne, &len, &err);
        if (err) { c->err_rec[part] = r; c->err_code[part] = err; c->err_at[part] = hs; break; }
        c->name_off[r] = (uint32_t)(hs + 1);
        c->name_len[r] = (uint32_t)(ne - hs - 1);
        c->seq_len[r] = (uint32_t)len;
        groups += utb_read_slots((uint32_t)len); js += len;
        if (r == c->n_rec - 1) c->end_of_records = next;
        hs = next;                                                 /* the next header: this worker's while r + 1 < r1 */
    }
    c->groups[part] = groups; c->jsum[part] = js;
}
static void wr_copy_part(void *c_, int part, int nparts) {
    frame_ctx *c = (frame_ctx *)c_;
    (void)nparts;
    const size_t r1 = c->base[part] + c->cnt[part] < c->n_valid ? c->base[part] + c->cnt[part] : c->n_valid;
    uint64_t at = c->jsum[part];
    for (size_t r = c->base[part]; r < r1; ++r) {
        size_t ne; uint64_t len; int err;
        c->seq_off[r] = at;
        (void)wr_record(c, (size_t)c->name_off[r] - 1, c->join + at, &ne, &len, &err);
        at += len;
    }
}
static const char *wr_text(int code) {
    return code == UTB_FW_NOHEADER ? "ERROR: wrapped FASTA input does not begin with '>'"
                                   : "ERROR: line of 16777216 bytes or more, or sequence of more than 16777214 bases";
}
/* Frames buf[0..fill) as wrapped FASTA into F->join: on return *n_out records are valid (those before the first
 * malformed one), *n_complete were framed (without EOF the record after the last header is carried), *used is the
 * byte after the last of them (a malformed record: where it starts), *err is UTB_FW_* of the record at index
 * *n_out or FE_NONE. */
static void wr_buffer(team_t *team, frame_ctx *F, size_t *n_out, size_t *n_complete, size_t *used, int *err) {
    *n_out = *n_complete = *used = 0; *err = FE_NONE;
    F->end_of_records = 0; F->groups_valid = 0;
    if (!F->fill) return;
    if (F->buf[0] != '>') { *err = UTB_FW_NOHEADER; return; }
    team_run(team, wr_count_part, F);
    size_t h = 0;
    for (int p = 0; p < team->n; ++p) { F->base[p] = h; h += F->cnt[p]; }
    F->n_rec = F->eof ? h : h - 1;                                 /* buf[0] is a header, so h >= 1 */
    if (F->n_rec > F->max_rec) F->n_rec = F->max_rec;              /* the rest comes back with the carry */
    for (int p = 0; p < team->n; ++p) { F->err_rec[p] = (size_t)-1; F->err_code[p] = FE_NONE; F->groups[p] = 0; F->jsum[p] = 0; }
    if (F->n_rec) team_run(team, wr_part, F);
    size_t n = F->n_rec, at = 0;
    for (int p = 0; p < team->n; ++p) if (F->err_rec[p] < n) { n = F->err_rec[p]; *err = F->err_code[p]; at = F->err_at[p]; }
    uint64_t j = 0;
    for (int p = 0; p < team->n; ++p) { const uint64_t k = F->jsum[p]; F->jsum[p] = j; j += k; }
    F->n_valid = n;
    if (n) team_run(team, wr_copy_part, F);
    F->groups_valid = n == F->n_rec;
    *n_out = n; *n_complete = F->n_rec; *used = *err ? at : F->end_of_records;
}

/* Host-stage entry points (CPU-only tests drive the framer and the formatter through these). */
int utb_frame_records(const char *buf, size_t n, int eof, int threads, size_t max_reads,
                      uint64_t *seq_off, uint32_t *seq_len, uint32_t *name_off, uint32_t *name_len,
                      size_t *n_reads, size_t *used, int *ref_exit) {
    if ((!buf && n) || !seq_off || !seq_len || !name_off || !name_len || !n_reads || !used) { utb_set_error("utb_frame_records: null argument"); return UTB_ERR_ARG; }
    if (ref_exit) *ref_exit = 0;
    *n_reads = 0; *used = 0;
    if (!n) return UTB_OK;
    team_t team;
    if (team_init(&team, threads)) { utb_set_error("cannot start worker threads"); return UTB_ERR_NOMEM; }
    frame_ctx F;
    memset(&F, 0, sizeof F);
    F.buf = buf; F.fill = n; F.eof = eof; F.max_rec = max_reads;
    F.idx_cap = n / 8 + 64 * (size_t)MAX_TEAM + 64;
    F.idx = (uint32_t *)malloc(F.idx_cap * sizeof(uint32_t));     /* NULL: the byte-wise path is used */
    F.seq_off = seq_off; F.seq_len = seq_len; F.name_off = name_off; F.name_len = name_len;
    size_t nr, nc, u; int err, dangling;
    frame_buffer(&team, &F, &nr, &nc, &u, &err, &dangling);
    team_destroy(&team);
    free(F.idx);
    *n_reads = nr; *used = u;
    if (err) { utb_set_error("%s [L %zu]", fe_text(err), nr + 1); if (ref_exit) *ref_exit = 2; return UTB_ERR_FORMAT; }
    if (dangling) { utb_set_error("ERROR: can't read sequence L %zu", nr); if (ref_exit) *ref_exit = 2; return UTB_ERR_FORMAT; }
    return UTB_OK;
}

int utb_frame_fastq_records(const char *buf, size_t n, int eof, int threads, size_t max_reads,
                            uint64_t *seq_off, uint32_t *seq_len, uint64_t *qual_off, uint32_t *name_off, uint32_t *name_len,
                            size_t *n_reads, size_t *used, size_t *err_record, int *err_code) {
    if ((!buf && n) || !seq_off || !seq_len || !qual_off || !name_off || !name_len || !n_reads || !used) {
        utb_set_error("utb_frame_fastq_records: null argument"); return UTB_ERR_ARG;
    }
    *n_reads = 0; *used = 0;
    if (err_record) *err_record = 0;
    if (err_code) *err_code = 0;
    if (!n) return UTB_OK;
    team_t team;
    if (team_init(&team, threads)) { utb_set_error("cannot start worker threads"); return UTB_ERR_NOMEM; }
    frame_ctx F;
    memset(&F, 0, sizeof F);
    F.buf = buf; F.fill = n; F.eof = eof; F.max_rec = max_reads;
    F.seq_off = seq_off; F.seq_len = seq_len; F.qual_off = qual_off; F.name_off = name_off; F.name_len = name_len;
    size_t nr, nc, u; int err;
    fq_buffer(&team, &F, &nr, &nc, &u, &err);
    team_destroy(&team);
    *n_reads = nr; *used = u;
    if (!err) return UTB_OK;
    if (err_record) *err_record = nr + 1;
    if (err_code) *err_code = err;
    utb_set_error("%s [record %zu]", fq_text(err), nr + 1);
    return UTB_ERR_FORMAT;
}

int utb_frame_wrapped_records(const char *buf, size_t n, int eof, int threads, size_t max_reads,
                              char *seq_out, size_t seq_cap, uint64_t *seq_off, uint32_t *seq_len,
                              uint32_t *name_off, uint32_t *name_len,
                              size_t *n_reads, size_t *used, size_t *err_record, int *err_code) {
    if ((!buf && n) || (!seq_out && n) || !seq_off || !seq_len || !name_off || !name_len || !n_reads || !used) {
        utb_set_error("utb_frame_wrapped_records: null argument"); return UTB_ERR_ARG;
    }
    if (seq_cap < n) { utb_set_error("utb_frame_wrapped_records: seq_cap %zu is less than the %zu input bytes", seq_cap, n); return UTB_ERR_ARG; }
    *n_reads = 0; *used = 0;
    if (err_record) *err_record = 0;
    if (err_code) *err_code = 0;
    if (!n) return UTB_OK;
    team_t team;
    if (team_init(&team, threads)) { utb_set_error("cannot start worker threads"); return UTB_ERR_NOMEM; }
    frame_ctx F;
    memset(&F, 0, sizeof F);
    F.buf = buf; F.fill = n; F.eof = eof; F.max_rec = max_reads; F.join = seq_out;
    F.seq_off = seq_off; F.seq_len = seq_len; F.name_off = name_off; F.name_len = name_len;
    size_t nr, nc, u; int err;
    wr_buffer(&team, &F, &nr, &nc, &u, &err);
    team_destroy(&team);
    *n_reads = nr; *used = u;
    if (!err) return UTB_OK;
    if (err_record) *err_record = nr + 1;
    if (err_code) *err_code = err;
    utb_set_error("%s [record %zu]", wr_text(err), nr + 1);
    return UTB_ERR_FORMAT;
}

int utb_format_results(const utb_ctr *ctr, const char *bytes, const uint32_t *name_off, const uint32_t *name_len,
                       const utb_result *results, size_t n_reads, char *out, size_t out_cap, size_t *out_len) {
    if (!ctr || !bytes || !name_off || !name_len || !results || !out || !out_len) { utb_set_error("utb_format_results: null argument"); return UTB_ERR_ARG; }
    size_t max_label = 0, need = n_reads * 64 + 64;                /* name + label + 4 tabs + 4 numbers + newline */
    for (uint32_t i = 0; i < ctr->max_ix; ++i) { size_t l = ctr->off[i + 1] - ctr->off[i]; if (l > max_label) max_label = l; }
    for (size_t r = 0; r < n_reads; ++r) need += name_len[r] + max_label;
    char *buf = (char *)malloc(need);
    if (!buf) { utb_set_error("out of memory (formatter)"); return UTB_ERR_NOMEM; }
    const size_t len = fmt_lines(ctr, bytes, name_off, name_len, results, n_reads, buf);
    int rc = UTB_OK;
    if (len > out_cap) { utb_set_error("utb_format_results: output needs %zu bytes", len); rc = UTB_ERR_LIMIT; }
    else memcpy(out, buf, len);
    *out_len = len;
    free(buf);
    return rc;
}

/* Where the device fast path cuts a FASTQ chunk: right before the last line L that begins with '@' and whose line
 * L+2 begins with '+' (0: none).  In well-formed input the header lines pass.  A quality line that begins with '@'
 * fails, because its line L+2 is the next record's sequence line (unless that begins with '+').  The cut is only a
 * guess: by induction the chunk starts on a header line, so a cut before a line whose index is not a multiple of 4
 * leaves a line count that is not one either; frame_setup_kernel<4> rejects such a chunk (FRE_CHUNK) and the
 * reader rewinds to it with the host framer, which takes every line's role from its index.  A cut before a line
 * whose index is a multiple of 4 is a record boundary of the strict 4-line framing, whatever the line holds.  So
 * correctness never rests on the cut, only the speed does. */
static size_t fastq_cut(const char *buf, size_t fill) {
    size_t next1 = 0, next2 = 0;                                   /* starts of the two lines after the candidate (0: none) */
    for (size_t hi = fill - 1; hi > 0;) {                          /* newline at index < fill - 1: a line starts after it */
        const char *q = (const char *)memrchr(buf, '\n', hi);
        if (!q) break;
        const size_t i = (size_t)(q - buf), L = i + 1;
        if (buf[L] == '@' && next2 && buf[next2] == '+') return L;
        next2 = next1; next1 = L;
        hi = i;
    }
    return 0;
}

static int run_search(utb_searcher *s, source_t *src, sink_t *sink, int do_rc, utb_stats *stats, int *ref_exit) {
    run_t R;
    memset(&R, 0, sizeof R);
    R.s = s; R.sink = sink;
    pthread_mutex_init(&R.mu, NULL);
    pthread_cond_init(&R.cv, NULL);
    if (ref_exit) *ref_exit = 0;
    double t0 = now_s();
    R.t0 = t0;
    uint64_t launches0 = 0;
    for (int i = 0; i < s->n_slots; ++i) { s->slots[i].state = 0; launches0 += utb_batch_launches(s->slots[i].b); }
    if (s->shallow && s->horses) memset(s->horses, 0, s->horses_cap * sizeof(uint32_t));   /* every search starts like a fresh process */
    /* split the host threads between the two teams */
    /* with the lines built on the device the formatter only moves finished text: most threads frame */
    int T = s->host_threads, n_fm = T >= 4 ? T / 2 : 1, n_rd = T >= 4 ? T - n_fm : 1;
    team_t rd_team;
    if (team_init(&rd_team, n_rd) || team_init(&R.fmt_team, n_fm)) { utb_set_error("cannot start worker threads"); return UTB_ERR_NOMEM; }
    pthread_t fmt;
    if (pthread_create(&fmt, NULL, formatter_main, &R)) { utb_set_error("cannot start formatter thread"); return UTB_ERR_NOMEM; }

    char *carry = (char *)malloc(s->batch_bytes);
    size_t carry_len = 0;
    /* newline-index arena of the framer (one newline per 8 bytes; denser input takes the byte-wise path) */
    size_t idx_cap = s->batch_bytes / 8 + 64 * (size_t)MAX_TEAM + 64;
    uint32_t *idx = (uint32_t *)malloc(idx_cap * sizeof(uint32_t));
    /* a caller buffer that is already page-locked is framed in place and copied to the device from where it
     * lies: no staging memcpy, no carry (batches are just consecutive ranges of it) */
    const int zero_copy = src->fd < 0 && src->mem_len && utb_host_ptr_is_pinned(src->mem) &&
                          utb_host_ptr_is_pinned(src->mem + src->mem_len - 1);
    int rc = UTB_OK, fmt_err = 0, chunked = 0;                    /* chunked: device-framed batches may still be in flight */
    char fmt_msg[256] = "";
    uint64_t seq = 0, n_reads_total = 0, consumed = 0;
    /* device-side framing needs an input that can be rewound if a malformed record turns up */
    int device_frame = s->device_frame && (src->fd < 0 || src->seekable);
    double rd_t[4] = {0, 0, 0, 0};
    if (!carry) { rc = UTB_ERR_NOMEM; utb_set_error("out of memory (carry)"); }
read_loop:
    while (!rc) {
        slot_t *sl = &s->slots[seq % (uint64_t)s->n_slots];
        double tp = now_s();
        pthread_mutex_lock(&R.mu);
        while (sl->state != 0 && !R.discard) pthread_cond_wait(&R.cv, &R.mu);
        if (R.discard) {
            /* A device-framed batch held a malformed record.  Let the formatter drain (and drop) what is in
             * flight, rewind the input to the start of that batch and frame the rest with the host reader,
             * which reproduces the reference's partial output, message and exit code exactly. */
            while (R.consumed < R.submitted) pthread_cond_wait(&R.cv, &R.mu);
            const slot_t *ks = &s->slots[R.restart_seq % (uint64_t)s->n_slots];
            consumed = ks->src_off; n_reads_total = R.reads_done;   /* the batches before it were counted, none from it on */
            if (src->fd >= 0) { src->file_off = (off_t)consumed; src->eof = src->file_off >= src->file_size; }
            else { src->mem_pos = (size_t)consumed; src->eof = src->mem_pos >= src->mem_len; }
            carry_len = 0; device_frame = 0; chunked = 0; R.discard = 0;
            fmt_err = 0; fmt_msg[0] = 0;                           /* an error met further down the input is met again, in order */
            pthread_mutex_unlock(&R.mu);
            continue;
        }
        int dev_err = R.error;
        pthread_mutex_unlock(&R.mu);
        rd_t[0] += now_s() - tp; tp = now_s();
        if (dev_err) break;
        const char *buf = utb_batch_bytes(sl->b);
        size_t cap = utb_batch_max_bytes(sl->b), fill = carry_len;
        /* batch-size schedule: ramp up (64, 64, 128 MiB, then full) and, when the input size is known, down again */
        const size_t RAMP = s->ramp_bytes;
        if (cap > 2 * RAMP) {
            size_t want = seq < 2 ? RAMP : seq == 2 ? 2 * RAMP : cap;
            size_t left = src->fd < 0 ? src->mem_len - src->mem_pos : src->seekable ? (size_t)(src->file_size - src->file_off) : (size_t)-1;
            if (left != (size_t)-1 && left + carry_len <= 3 * RAMP) want = RAMP;
            else if (left != (size_t)-1 && left + carry_len < want + 2 * RAMP && want > 2 * RAMP) want = left + carry_len - 2 * RAMP;
            if (want < carry_len + 4096) want = carry_len + 4096;  /* a carried partial record must be able to complete */
            if (want < MAX_RECORD(s->format != UTB_INPUT_FASTA ? 4 : 2)) want = MAX_RECORD(s->format != UTB_INPUT_FASTA ? 4 : 2);
            if (want < cap) cap = want;
        }
        if (zero_copy) {
            buf = src->mem + src->mem_pos;
            fill = src->mem_len - src->mem_pos < cap ? src->mem_len - src->mem_pos : cap;
            if (src->mem_pos + fill == src->mem_len) src->eof = 1;
        } else {
            if (carry_len) memcpy(utb_batch_bytes(sl->b), carry, carry_len);
            carry_len = 0;
            ssize_t k = src_fill(src, &rd_team, utb_batch_bytes(sl->b) + fill, cap - fill);
            if (k < 0) { rc = UTB_ERR_IO; utb_set_error("read error on input: %s", strerror(errno)); break; }
            fill += (size_t)k;
        }
        rd_t[1] += now_s() - tp; tp = now_s();
        if (!fill) break;                                          /* clean EOF */

        sl->src_off = consumed;
        const utb_batch_out out = s->shallow ? UTB_OUT_SELECTIONS : UTB_OUT_TEXT;   /* the text stays on the device until the formatter knows where it goes */
        if (device_frame && fill >= 2 && fill < 0xFFFFFFFFull) {
            /* Fast path: the host does not look at the bytes.  In a well-formed file exactly the header lines
             * begin with '>' (itree.c:880, 886), so the chunk is cut right before the last line that does (at the
             * end of the input: after the final newline) and goes to the GPU as it is; the device counts the
             * lines, checks that they pair up and that every record is well formed, and frames them.  Nothing is
             * waited for: if the check fails the formatter drops the batches from that one on and this loop
             * rewinds to it with the exact host reader.  Left to the host reader from the start: a last line
             * without '\n', a chunk without a second header. */
            size_t used = 0;
            if (src->eof) { if (buf[fill - 1] == '\n') used = fill; }
            else if (s->format == UTB_INPUT_FASTQ) used = fastq_cut(buf, fill);
            else for (size_t hi = fill - 1; hi > 0;) {             /* newline at index < fill - 1 followed by '>' (wrapped FASTA:
                                                                    * always a header, so the chunk ends on a record boundary) */
                const char *q = (const char *)memrchr(buf, '\n', hi);
                if (!q) break;
                const size_t i = (size_t)(q - buf);
                if (buf[i + 1] == '>') { used = i + 1; break; }
                hi = i;
            }
            if (used >= 2) {
                sl->n_reads = 0; sl->host_bytes = buf; sl->n_bytes = used;
                consumed += used;
                if (zero_copy) { src->mem_pos += used; if (src->mem_pos < src->mem_len) src->eof = 0; }
                else if (used < fill) { carry_len = fill - used; memcpy(carry, buf + used, carry_len); }
                rd_t[2] += now_s() - tp; tp = now_s();
                if (seq < 64) { R.tl_framed[seq] = now_s() - t0; R.tl_reads[seq] = 0; }
                int r2 = utb_batch_submit_chunk(sl->b, zero_copy ? buf : NULL, used, 0, do_rc, out);
                if (r2) { rc = r2; break; }
                R.st.h2d_bytes += used;
                chunked = 1;
                if (seq < 64) R.tl_submit[seq] = now_s() - t0;
                pthread_mutex_lock(&R.mu);
                sl->state = 1;
                R.submitted = ++seq;
                pthread_cond_broadcast(&R.cv);
                pthread_mutex_unlock(&R.mu);
                rd_t[3] += now_s() - tp;
                if (src->eof && !carry_len) break;
                continue;
            }
        }
        if (chunked) {
            /* the host reader numbers its records (error messages carry the line count): the batches in
             * flight report theirs on completion, so let them finish first */
            pthread_mutex_lock(&R.mu);
            while (R.consumed < R.submitted) pthread_cond_wait(&R.cv, &R.mu);
            const int again = R.discard;
            n_reads_total = R.reads_done;
            pthread_mutex_unlock(&R.mu);
            chunked = 0;
            if (again) continue;                                   /* the top of the loop rewinds; this chunk is read again */
        }
        frame_ctx F;
        memset(&F, 0, sizeof F);
        F.buf = buf; F.fill = fill; F.eof = src->eof; F.max_rec = utb_batch_max_reads(sl->b);
        F.idx = idx; F.idx_cap = idx ? idx_cap : 0;
        F.seq_off = utb_batch_seq_off(sl->b); F.seq_len = utb_batch_seq_len(sl->b);
        F.name_off = sl->name_off; F.name_len = sl->name_len;
        size_t n, n_complete, end_of_records; int err_code, dangling = 0;
        if (s->format == UTB_INPUT_FASTQ) {                        /* a truncated record is an error like any other */
            F.qual_off = utb_batch_qual_off(sl->b);
            fq_buffer(&rd_team, &F, &n, &n_complete, &end_of_records, &err_code);
            if (err_code) { fmt_err = 1; snprintf(fmt_msg, sizeof fmt_msg, "%s [record %llu]", fq_text(err_code), (unsigned long long)(n_reads_total + n + 1)); }
        } else if (s->format == UTB_INPUT_FASTA_WRAPPED) {        /* the sequences are joined into the slot's second staging buffer */
            F.join = utb_batch_join(sl->b);
            wr_buffer(&rd_team, &F, &n, &n_complete, &end_of_records, &err_code);
            if (err_code) { fmt_err = 1; snprintf(fmt_msg, sizeof fmt_msg, "%s [record %llu]", wr_text(err_code), (unsigned long long)(n_reads_total + n + 1)); }
        } else {
            frame_buffer(&rd_team, &F, &n, &n_complete, &end_of_records, &err_code, &dangling);
            if (err_code) { fmt_err = 1; snprintf(fmt_msg, sizeof fmt_msg, "%s [L %llu]", fe_text(err_code), (unsigned long long)(n_reads_total + n + 1)); }
        }
        /* capacity: reads and 32-base position groups */
        size_t max_reads = utb_batch_max_reads(sl->b);
        uint64_t max_slots = utb_batch_max_slots(sl->b), groups = 0;
        int cut = 0;
        if (n > max_reads) { n = max_reads; cut = 1; }
        int groups_known = 0;
        if (F.groups_valid && !cut) {                              /* the workers summed the groups while framing */
            for (int p = 0; p < rd_team.n; ++p) groups += F.groups[p];
            groups_known = groups <= max_slots;
        }
        if (!groups_known) {
            groups = 0;
            for (size_t r = 0; r < n; ++r) {
                uint64_t g = utb_read_slots(F.seq_len[r]);
                if (groups + g > max_slots) { n = r; cut = 1; break; }
                groups += g;
            }
        }
        if (cut) fmt_err = 0;                                      /* the bad record, if any, comes back with the carry */
        size_t used = (n == n_complete) ? end_of_records : (size_t)sl->name_off[n] - 1;
        if (!fmt_err && !cut && dangling && n == n_complete) {
            fmt_err = 1;
            snprintf(fmt_msg, sizeof fmt_msg, "ERROR: can't read sequence L %llu", (unsigned long long)(n_reads_total + n));
        }
        if (!fmt_err && n == 0 && !cut && !src->eof && fill == cap) {
            fmt_err = 1;
            snprintf(fmt_msg, sizeof fmt_msg, "ERROR: record larger than the %zu-byte batch buffer", cap);
        }
        sl->n_reads = n;
        sl->host_bytes = buf;
        sl->n_bytes = fmt_err ? fill : used;
        sl->first_read = n_reads_total;
        n_reads_total += n;
        consumed += fmt_err ? fill : used;
        if (zero_copy) { src->mem_pos += fmt_err ? fill : used; if (src->mem_pos < src->mem_len) src->eof = 0; }
        else if (!fmt_err && used < fill) { carry_len = fill - used; memcpy(carry, buf + used, carry_len); }
        rd_t[2] += now_s() - tp; tp = now_s();
        if (seq < 64) { R.tl_framed[seq] = now_s() - t0; R.tl_reads[seq] = n; }
        if (n) {
            /* every sequence lies inside the first n_bytes of the buffer */
            int r2 = utb_batch_submit_ex(sl->b, zero_copy ? buf : NULL, fmt_err ? fill : used, n, do_rc, out,
                                         groups_known && !cut ? groups : 0);
            if (r2) { rc = r2; break; }
            R.st.h2d_bytes += (fmt_err ? fill : used) + n * 24 + 4;
            if (seq < 64) R.tl_submit[seq] = now_s() - t0;
            pthread_mutex_lock(&R.mu);
            sl->state = 1;
            R.submitted = ++seq;
            pthread_cond_broadcast(&R.cv);
            pthread_mutex_unlock(&R.mu);
        }
        rd_t[3] += now_s() - tp;
        if (fmt_err) break;
        if (src->eof && !carry_len) break;
    }
    if (!rc && chunked) {
        /* the reader is done (input exhausted, or a format error of its own), but a device-framed batch still in
         * flight may hold an EARLIER malformed record: that one decides the output, the message and the line number */
        pthread_mutex_lock(&R.mu);
        while (R.consumed < R.submitted) pthread_cond_wait(&R.cv, &R.mu);
        const int again = R.discard;
        pthread_mutex_unlock(&R.mu);
        chunked = 0;
        if (again) goto read_loop;                                 /* the top of the loop rewinds and forgets the later error */
    }
    free(idx);
    pthread_mutex_lock(&R.mu);
    R.done_reading = 1;
    pthread_cond_broadcast(&R.cv);
    pthread_mutex_unlock(&R.mu);
    pthread_join(fmt, NULL);
    team_destroy(&rd_team);
    team_destroy(&R.fmt_team);
    free(carry);
    pthread_mutex_destroy(&R.mu);
    pthread_cond_destroy(&R.cv);
    if (!rc && R.error) { rc = R.error; utb_set_error("%s", R.errmsg); }
    if (!rc && sink->failed) { rc = UTB_ERR_IO; utb_set_error("write error on output"); }
    for (int i = 0; i < s->n_slots; ++i) {                        /* text copies into the output arena still in flight */
        int r3 = utb_batch_sync(s->slots[i].b);
        if (r3 && !rc) rc = r3;
    }
    R.st.reads = R.reads_done;
    R.st.batches = seq;
    for (int i = 0; i < s->n_slots; ++i) R.st.kernel_launches += utb_batch_launches(s->slots[i].b);
    R.st.kernel_launches -= launches0;
    R.st.seconds_total = now_s() - t0;
    if (getenv("UTB_TIMELINE")) {
        fprintf(stderr, "utree-b200 timeline (ms): batch reads framed submitted gpu_done emitted\n");
        for (uint64_t i = 0; i < seq && i < 64; ++i)
            fprintf(stderr, "  %2llu %8zu %8.2f %8.2f %8.2f %8.2f\n", (unsigned long long)i, R.tl_reads[i], 1e3 * R.tl_framed[i],
                    1e3 * R.tl_submit[i], 1e3 * R.tl_gpu_done[i], 1e3 * R.tl_emitted[i]);
        fprintf(stderr, "  total %.2f ms\n", 1e3 * R.st.seconds_total);
    }
    R.st.rd_wait_slot = rd_t[0]; R.st.rd_fill = rd_t[1]; R.st.rd_frame = rd_t[2]; R.st.rd_submit = rd_t[3];
    if (stats) *stats = R.st;
    if (!rc && fmt_err) {
        utb_set_error("%s", fmt_msg);
        if (ref_exit) *ref_exit = 2;                               /* itree.c:872-888 */
        return UTB_ERR_FORMAT;
    }
    return rc;
}

int utb_search_file(utb_searcher *s, const char *fasta_path, const char *out_path,
                    int do_rc, utb_stats *stats, int *ref_exit) {
    if (!s || !fasta_path || !out_path) { utb_set_error("utb_search_file: null argument"); return UTB_ERR_ARG; }
    if (ref_exit) *ref_exit = 0;
    int fd = open(fasta_path, O_RDONLY);
    if (fd < 0) { utb_set_error("Invalid input files"); if (ref_exit) *ref_exit = 1; return UTB_ERR_IO; }   /* itree.c:835 */
    int fo = open(out_path, O_RDWR | O_CREAT | O_TRUNC, 0644);   /* read access only for the shared mapping of sink_reserve */
    if (fo < 0) fo = open(out_path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (fo < 0) { close(fd); utb_set_error("cannot open output file %s", out_path); if (ref_exit) *ref_exit = 1; return UTB_ERR_IO; }
    source_t src; memset(&src, 0, sizeof src); src.fd = fd;
    struct stat st;
    if (!fstat(fd, &st) && S_ISREG(st.st_mode)) { src.seekable = 1; src.file_size = st.st_size; if (!st.st_size) src.eof = 1; }
    sink_t sink; memset(&sink, 0, sizeof sink); sink.fd = fo; sink.s = s;
    sink_open_file(&sink);
    int rc = run_search(s, &src, &sink, do_rc, stats, ref_exit);
    int bad = sink_close_file(&sink);
    if ((close(fo) || bad) && !rc) { rc = UTB_ERR_IO; utb_set_error("write error on output"); }
    close(fd);
    return rc;
}

int utb_search_mem(utb_searcher *s, const char *fasta, size_t n, int do_rc,
                   char **out, size_t *out_len, utb_stats *stats, int *ref_exit) {
    if (!s || (!fasta && n) || !out || !out_len) { utb_set_error("utb_search_mem: null argument"); return UTB_ERR_ARG; }
    source_t src; memset(&src, 0, sizeof src); src.fd = -1; src.mem = fasta; src.mem_len = n; src.eof = n == 0;
    sink_t sink; memset(&sink, 0, sizeof sink); sink.fd = -1; sink.s = s;
    sink.hint = n / 2 + n / 4 + ((size_t)1 << 20);                 /* typical output: about half the FASTA */
    int rc = run_search(s, &src, &sink, do_rc, stats, ref_exit);
    *out = sink.off ? s->arena : NULL; *out_len = sink.off;
    return rc;
}

/* ---- CLI (itree.c:1357-1377; stdout lines of SURVEY App. C) -------------------------------------- */
static const char *TYPEARR[9] = {"NA", "uint8_t", "uint16_t", "NA", "uint32_t", "NA", "NA", "NA", "uint64_t"};

static int main_impl(int argc, char **argv, int gg);
int utb_main(int argc, char **argv) { return main_impl(argc, argv, 1); }
/* the non-GG binary (makefile: utree-search, -D SEARCH): same argv / banner / exit codes, shallow vote */
int utb_main_shallow(int argc, char **argv) { return main_impl(argc, argv, 0); }
static int main_impl(int argc, char **argv, int gg) {
    if (argc < 4) {                                                /* itree.c:1358-1360 */
        printf("[v2.0RF SigNature Edition] usage: xtree-search%s compTree.ctr fastaToSearch.fa output.txt [threads] [SPEED <X>] [RC]\n", gg ? "GG" : "");
        return 1;
    }
    printf("This is UTree [v2.0RF SigNature Edition]\n");
    int do_rc = !strcmp(argv[argc - 1], "RC");                     /* itree.c:1362-1364 */
    argc -= do_rc;
    int speed = 0;
    if (!strcmp(argv[argc - 2], "SPEED")) { speed = atoi(argv[argc - 1]); argc -= 2; }
    printf("Reverse complement consideration is %sabled.\n", do_rc ? "en" : "dis");
    printf("Searching at speed %d.\n", speed);
    long ncpu = sysconf(_SC_NPROCESSORS_ONLN);
    int threads = argc >= 5 ? atoi(argv[4]) : (int)(ncpu > 0 ? ncpu : 1);   /* itree.c:1368 */
    printf("Using up to %d threads.\n", threads);

    utb_ctr *ctr = NULL;
    int rc = utb_ctr_open(argv[1], &ctr);
    if (rc == UTB_ERR_FORMAT && !strcmp(utb_last_error(), "Error in reading tree.")) {
        /* truncated tree: XT_read32 prints what it has got so far, then the message, and exits 3 (itree.c:754-768) */
        uint64_t md[4], got = 0;
        if (!utb_ctr_probe(argv[1], md, &got)) {
            puts(md[3] < 0xFFFFFFFFull ? "Using 32-bit counters" : "Holey smokes, a tree of over 4 billion k-mers. Here goes...");
            printf("%llu elements read.\n", (unsigned long long)got);
            printf("Nodes in input tree: %llu (PACKSIZE=%u, CNTTYPE=%s, IXTYPE=%s, SZ=%d)\n", (unsigned long long)md[3], 32u, "NA",
                   TYPEARR[md[2]], (int)(5 + md[2]));
        }
        puts("Error in reading tree.");
        return 3;
    }
    if (rc) { puts(utb_last_error()); return 0; }                  /* itree.c:735, 738, 750: exit(0) */
    if (ctr->num_nodes < 0xFFFFFFFFull) puts("Using 32-bit counters");   /* itree.c:754-755 */
    else puts("Holey smokes, a tree of over 4 billion k-mers. Here goes...");
    printf("%llu elements read.\n", (unsigned long long)UTB_NUMBINS);     /* itree.c:761 */
    printf("Nodes in input tree: %llu (PACKSIZE=%u, CNTTYPE=%s, IXTYPE=%s, SZ=%d)\n",   /* itree.c:764 */
           (unsigned long long)ctr->num_nodes, 32u, "NA", TYPEARR[ctr->ix_bytes], (int)ctr->sz);
    printf("Read %llu nodes.\n", (unsigned long long)ctr->num_nodes);     /* itree.c:769 */
    if (ctr->last_bin != ctr->num_nodes)                           /* itree.c:792-793 */
        printf("Warning: detected nodes %u != %u\n", (unsigned)ctr->last_bin, (unsigned)ctr->num_nodes);

    int ndev = 0, devs[64];
    rc = utb_device_count(&ndev);
    if (rc) { fprintf(stderr, "utree-b200: %s\n", utb_last_error()); utb_ctr_close(ctr); return 4; }
    int n = 0;
    const char *e = getenv("UTB_DEVICES");                         /* e.g. "0,1,2,3"; default: all visible */
    if (e && *e) {
        char *dup = strdup(e), *save = NULL;
        for (char *t = strtok_r(dup, ",", &save); t && n < 64; t = strtok_r(NULL, ",", &save)) devs[n++] = atoi(t);
        free(dup);
    } else for (; n < ndev && n < 64; ++n) devs[n] = n;
    utb_searcher *s = NULL;
    rc = utb_searcher_create(ctr, devs, n, threads, &s);
    if (rc) { fprintf(stderr, "utree-b200: %s\n", utb_last_error()); utb_ctr_close(ctr); return rc == UTB_ERR_NOMEM ? 3 : 4; }
    if (!gg) rc = utb_searcher_set_shallow(s, 1);
    if (rc) { fprintf(stderr, "utree-b200: %s\n", utb_last_error()); utb_searcher_destroy(s); utb_ctr_close(ctr); return rc == UTB_ERR_NOMEM ? 3 : 4; }
    puts("Tree read.");                                            /* itree.c:826 */
    fflush(stdout);
    s->verbose = 1;
    utb_stats st;
    int ref_exit = 0;
    rc = utb_search_file(s, argv[2], argv[3], do_rc, &st, &ref_exit);
    if (rc == UTB_ERR_IO && ref_exit == 1) { puts(utb_last_error()); utb_searcher_destroy(s); utb_ctr_close(ctr); return 1; }
    if (rc == UTB_ERR_FORMAT && ref_exit) {                        /* output so far is on disk, as after the reference's exit() */
        fflush(stdout);
        fprintf(stderr, "%s\n", utb_last_error());
        utb_searcher_destroy(s); utb_ctr_close(ctr);
        return ref_exit;
    }
    if (rc) { fprintf(stderr, "utree-b200: %s\n", utb_last_error()); utb_searcher_destroy(s); utb_ctr_close(ctr); return 4; }
    printf("Good finds: %llu\n", (unsigned long long)st.good_finds);       /* itree.c:1106 */
    printf("Searched %llu queries\n", (unsigned long long)st.reads);       /* itree.c:1375 */
    if (getenv("UTB_STATS"))
        fprintf(stderr, "utree-b200: %d GPU(s), %llu batches, %llu lookups, %llu hits, %.3f s total, %.3f s device\n",
                n, (unsigned long long)st.batches, (unsigned long long)st.lookups, (unsigned long long)st.hits,
                st.seconds_total, st.seconds_device);
    utb_searcher_destroy(s);
    utb_ctr_close(ctr);
    return 0;
}
