// kernels.cu -- sm_100a device side of the SEARCH_GG hot path + the thin C ABI
// over it (utb_db_*, utb_batch_*, stage-level entry points).
//
// Data layout in HBM (DESIGN.md "Data layout"):
//   binix   : the CTR prefix index exactly as on disk, (2^24+1) x 4 B
//             (8 B when numNodes >= 2^32-1)                  itree.c:756-759
//   recs    : the CTR record blob exactly as on disk, numNodes x SZ bytes,
//             SZ = 5-byte suffix + IXTYPE id, + 32 B slack   itree.c:766
//             (kept for irregular CTRs only; regular ones are re-keyed once at
//             upload into ktab, a sector hash table, and get the sieve, a
//             minimizer-keyed blocked Bloom filter -- see DevDB)
//   labels  : blob of NUL-terminated strings, off[], rank[], by_rank[]
// Per batch (one stream slot):
//   raw     : the FASTA bytes as read from the file (headers included)
//   nl      : positions of the newlines (device-side framing)
//   seq_off/seq_len/name_off/name_len/grp_off : where each read's lines sit, and
//             the first 32-base group it owns in the packed "super-sequence"
//   pk/bad  : 2-bit codes (u64 per 32 bases, first base most significant, the
//             k-mer word order of itree.c:924) and a bad-base bit mask.  Every
//             read is padded to a multiple of 32 positions with >= 1 bad
//             position, so a 32-mer window can never straddle two reads.
//   pl      : the same bases as two bit planes per group (sieve on; the sieve kernel's input)
//   hits    : sieve on (GG path): per read the labels of its hits back to back from the read's first slot, hcnt[read]
//             of them; otherwise one u32 per (position, strand), with a 1-bit-per-slot hitmap in the non-GG path
//   results : one utb_result per read;  text : the output lines
//
// Kernels: nl_count / nl_index / frame_parse (XT_INITIATE_WS, itree.c:860-901),
// pack_kernel (XT_WORD_SEARCH's 2-bit packing, itree.c:919-926), sieve_kernel
// (membership pre-filter, one 8-byte fetch per position for both strands, one DRAM
// line per ~9 positions) and queue_lookup_kernel (XT_getIX32 + xtSuffixBS on the
// survivors, itree.c:699-730), lookup_kernel (the same without pre-filter, or the
// reference's exact probe sequence), vote_thread / vote_warp / vote_block (full
// aufbau vote, itree.c:1028-1098), fmt_* (the fprintf lines, itree.c:1032-1096).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "utb_internal.h"

#define SUFMASK 0xFFFFFFFFFFull
#define HIT_MISS 0xFFFFFFFFu   // looked up, not found (BAD_IX widened)
#define HIT_NOWIN 0xFFFFFFFEu  // no valid 32-mer window here: no lookup made

#define CK(call)                                                                 \
    do {                                                                         \
        cudaError_t e_ = (call);                                                 \
        if (e_ != cudaSuccess) {                                                 \
            utb_set_error("CUDA error %s at %s:%d (%s)", cudaGetErrorName(e_),   \
                          __FILE__, __LINE__, cudaGetErrorString(e_));           \
            return UTB_ERR_CUDA;                                                 \
        }                                                                        \
    } while (0)

// ---------------------------------------------------------------------------
// device-side database view (passed by value to kernels)
// ---------------------------------------------------------------------------
struct DevDB {
    const uint32_t *binix32;   // one of binix32 / binix64 is non-null while the on-disk image is resident
    const uint64_t *binix64;
    const uint8_t *recs;
    uint64_t num_nodes;
    uint32_t sz;               // 7 or 9
    uint32_t ix_bytes;         // 2 or 4
    uint32_t max_ix;
    const char *blob;
    const uint32_t *off;
    const uint32_t *rank;
    const uint32_t *by_rank;
    uint32_t quirk_bin;        // bucket whose record 0 is the folded foreign record (SURVEY 0 #4), else 0xFFFFFFFF
    // regular CTRs only: the records re-keyed into a sector hash table (binix / recs are then freed)
    const uint64_t *ktab;      // kt_sectors x 32 bytes: 4 entries of 8 bytes (uint16_t labels) or 3 wide entries (uint32_t labels)
    uint32_t kt_wide;          // IXTYPE uint32_t: three entries per sector, the label id inside
    uint64_t kt_sectors;
    // membership pre-filter over all record words: blocked Bloom, line chosen by the word's minimizer
    const uint2 *sieve;        // sv_lines x 16 blocks of 8 bytes
    uint32_t sv_lines;         // < 2^28
};

struct utb_db {
    int device;
    DevDB d;
    int regular;               // every bucket strictly sorted (modulo quirk_bin): the record words are distinct, a hash table is exact
    int use_table;             // lookup variant in use: 1 sector hash table (+ sieve), 0 the reference's probe sequence
    void *binix, *recs, *blob, *off, *rank, *by_rank, *ktab, *sieve;
    int sieve_mode;            // 0 off, 1 always, 2 auto (on while the observed hit rate is low)
    volatile double ema_hit_rate;   // of the batches seen so far (written by the formatter thread, read at submit)
    size_t max_label;          // longest label, bytes
    uint64_t hbm_bytes;
    int sm_count;              // multiprocessors of the device (grid sizing)
    size_t nb_binix, nb_recs, nb_blob, nb_lab, nb_ktab, nb_sieve;   // bytes behind the device pointers (utb_db_clone)
    int l2_window;             // reference probe sequence only: persisting-L2 window over binix configured
    size_t l2_window_bytes;
    float l2_hit_ratio;
};

// ---------------------------------------------------------------------------
// pack: raw bytes -> 2-bit groups + bad mask
// ---------------------------------------------------------------------------
// One thread per 32-base group.  The 32 bytes are fetched with nine aligned
// 32-bit loads (neighbouring threads share cache lines, so the raw bytes move
// once from L2), classified four at a time with byte-SIMD compares.
// returns the 2-bit codes of the four bytes, one per byte (a 0, c 1, g 2, t 3)
__device__ __forceinline__ uint32_t classify4(uint32_t w, uint32_t &badbits) {
    const uint32_t u = w | 0x20202020u;                            // fold case (itree.c:114-117)
    // bits 1 and 2 of the letter give its code: a 0x61 -> 0, c 0x63 -> 1, g 0x67 -> 2, t 0x74 -> 3 (C2Xb, itree.c:110-121)
    const uint32_t code = ((u >> 1) ^ (u >> 2)) & 0x03030303u;
    // a byte is a base iff it IS the letter of its code: 0x61 + {0, 2, 6, 0x13}[code], built bytewise from the code's two bits
    const uint32_t c0 = code & 0x01010101u, c1 = (code >> 1) & 0x01010101u;
    const uint32_t both = c0 & c1;
    const uint32_t expect = 0x61616161u + (((c0 | c1) << 1) | ((c1 & ~c0) << 2)) + both * 0x11u;
    const uint32_t x = u ^ expect;                                  // nonzero byte = not ACGTacgt
    const uint32_t inval = ((((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) >> 7) & 0x01010101u;
    badbits = (inval * 0x01020408u) >> 24;                          // bit j = byte j is not a base
    return code;
}

// reverse complement of a 32-mer word: reverse the 2-bit fields of ~w
__device__ __forceinline__ uint64_t revcomp_word(uint64_t w) {
    uint64_t x = __brevll(~w);
    return ((x >> 1) & 0x5555555555555555ull) | ((x & 0x5555555555555555ull) << 1);
}
// The bit planes of a 32-mer: one u64, code bit 1 of every base in the upper 32 bits, code bit 0 in the lower 32,
// base 0 the most significant bit of both.  A window at any offset is then one funnel shift per plane, and the
// reverse complement of a plane is ~__brev(plane).  The word is the planes' bit interleave (bit 1 of a code odd).
__device__ __forceinline__ uint64_t word_to_planes(uint64_t w) {   // perfect unshuffle: odd bits up, even bits down
    uint64_t t;
    t = (w ^ (w >> 1)) & 0x2222222222222222ull; w ^= t ^ (t << 1);
    t = (w ^ (w >> 2)) & 0x0C0C0C0C0C0C0C0Cull; w ^= t ^ (t << 2);
    t = (w ^ (w >> 4)) & 0x00F000F000F000F0ull; w ^= t ^ (t << 4);
    t = (w ^ (w >> 8)) & 0x0000FF000000FF00ull; w ^= t ^ (t << 8);
    t = (w ^ (w >> 16)) & 0x00000000FFFF0000ull; w ^= t ^ (t << 16);
    return w;
}
__device__ __forceinline__ uint64_t planes_to_word(uint64_t w) {   // perfect shuffle: the inverse, steps in reverse order
    uint64_t t;
    t = (w ^ (w >> 16)) & 0x00000000FFFF0000ull; w ^= t ^ (t << 16);
    t = (w ^ (w >> 8)) & 0x0000FF000000FF00ull; w ^= t ^ (t << 8);
    t = (w ^ (w >> 4)) & 0x00F000F000F000F0ull; w ^= t ^ (t << 4);
    t = (w ^ (w >> 2)) & 0x0C0C0C0C0C0C0C0Cull; w ^= t ^ (t << 2);
    t = (w ^ (w >> 1)) & 0x2222222222222222ull; w ^= t ^ (t << 1);
    return w;
}
// The read that owns group g0 + lane, for a warp that takes the 32 groups from g0 on (warp-uniform call, g0 < the
// batch's groups): the largest r with grp_off[r] <= g0 by one bisection per warp; every read owns >= 1 group, so the
// reads of the other 31 groups start at one of the next 31 boundaries: a coalesced load of those, a warp-wide OR of
// "a read starts at group g0 + j", and a population count give each lane its read
__device__ __forceinline__ uint32_t group_read(const uint32_t *__restrict__ grp_off, uint32_t n_reads, uint32_t g0, uint32_t lane) {
    uint32_t lo = 0, hi = n_reads;                                 // invariant: grp_off[lo] <= g0 < grp_off[hi]
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (__ldg(grp_off + mid) <= g0) lo = mid; else hi = mid;
    }
    const uint32_t nb = lo + 1u + lane;                            // boundary held by this lane
    const uint32_t bnd = nb < n_reads ? __ldg(grp_off + nb) : 0xFFFFFFFFu;
    const uint32_t starts = __reduce_or_sync(0xFFFFFFFFu, bnd - g0 < 32u ? 1u << (bnd - g0) : 0u);
    return lo + __popc(starts & (0xFFFFFFFFu >> (31u - lane)));    // boundaries at groups g0 + 1 .. g0 + lane
}
#define PK_GUARD 8u               // all-bad groups behind the last read: the sieve kernel walks whole tiles without bounds checks
// WORDS: write pk (the 2-bit words, read by the sieve-off lookup, the non-GG selection and expand_windows_kernel);
// PLANES: write pl (the bit planes, read by the sieve kernel).  rid (optional): the read every group belongs to
template <bool WORDS, bool PLANES>
__global__ void __launch_bounds__(256)
pack_kernel(const uint8_t *__restrict__ raw, const uint64_t *__restrict__ seq_off,
            const uint32_t *__restrict__ seq_len, const uint32_t *__restrict__ grp_off,
            uint32_t n_reads, uint32_t n_groups, const uint32_t *__restrict__ dims,
            uint64_t *__restrict__ pk, uint32_t *__restrict__ bad, uint64_t *__restrict__ pl, uint32_t *__restrict__ rid) {
    if (dims) { n_reads = dims[0]; n_groups = dims[1]; }          // device-side framing: the host only knows upper bounds
    const uint32_t lane = threadIdx.x & 31u;
    // a warp takes 32 consecutive groups per round (warp-uniform loop)
    for (uint64_t gw = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) & ~31ull; gw < (uint64_t)n_groups + PK_GUARD; gw += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t g = (uint32_t)gw + lane;
        const uint32_t lo = (uint32_t)gw < n_groups ? group_read(grp_off, n_reads, (uint32_t)gw, lane) : 0u;
        if (g >= n_groups + PK_GUARD) continue;
        if (g >= n_groups) {                                       // guard groups: all positions bad
            if (WORDS) pk[g] = 0;
            if (PLANES) pl[g] = 0;
            bad[g] = 0xFFFFFFFFu;
            continue;
        }
        uint32_t k = g - __ldg(grp_off + lo);
        uint32_t len = __ldg(seq_len + lo);
        if (rid) rid[g] = lo;                                      // group -> read (phase B files a hit under its read)
        uint32_t b0 = k * 32u;
        uint32_t nv = len > b0 ? min(32u, len - b0) : 0u;  // real bases in this group
        uint64_t word = 0;
        uint32_t p1 = 0, p0 = 0;                                   // the planes, first base most significant
        uint32_t badm = 0;
        if (nv) {
            uint64_t a = __ldg(seq_off + lo) + b0;
            const uint32_t *p = reinterpret_cast<const uint32_t *>(raw + (a & ~3ull));
            uint32_t sh = (uint32_t)(a & 3u) * 8u;
            uint32_t nw = (nv + 3u) >> 2;                  // 4-byte words that hold real bases
            uint32_t prev = __ldg(p);
#pragma unroll
            for (uint32_t j = 0; j < 8; ++j) {
                uint32_t cur = (j < nw) ? __ldg(p + j + 1) : 0u;   // p[j+1] only if word j is needed
                uint32_t w = __funnelshift_r(prev, cur, sh);
                prev = cur;
                uint32_t bb;
                const uint32_t code = classify4(w, bb);
                // first base most significant: b0 << 6 | b1 << 4 | b2 << 2 | b3, resp. b0 << 3 | b1 << 2 | b2 << 1 | b3 per plane
                if (WORDS) word = (word << 8) | ((code * 0x40100401u) >> 24);
                if (PLANES) {
                    p1 = (p1 << 4) | ((((code >> 1) & 0x01010101u) * 0x08040201u) >> 24);
                    p0 = (p0 << 4) | (((code & 0x01010101u) * 0x08040201u) >> 24);
                }
                badm |= bb << (4u * j);
            }
        }
        if (nv < 32u) badm |= 0xFFFFFFFFu << nv;           // padding positions are bad
        if (WORDS) pk[g] = word;
        if (PLANES) pl[g] = ((uint64_t)p1 << 32) | p0;
        bad[g] = badm;
    }
}

// ---------------------------------------------------------------------------
// window extraction (shared by lookup and the stage-level test kernel)
// ---------------------------------------------------------------------------
__device__ __forceinline__ bool window_at(const uint64_t *__restrict__ pk, const uint32_t *__restrict__ bad,
                                          uint32_t pos, uint64_t &w) {
    uint32_t g = pos >> 5, o = pos & 31u;
    uint64_t hi = pk[g], lo = pk[g + 1];                          // const __restrict__ global pointers still compile to LDG.CONSTANT
    uint32_t bh = bad[g], bl = bad[g + 1];
    uint32_t wb = o ? ((bh >> o) | (bl << (32u - o))) : bh;
    w = o ? ((hi << (2u * o)) | (lo >> (64u - 2u * o))) : hi;
    return wb == 0;
}


// ---------------------------------------------------------------------------
// lookup: XT_getIX32 + xtSuffixBS, the reference's probe sequence verbatim
// ---------------------------------------------------------------------------
// Records are byte-packed (SZ = 7 or 9) so a suffix starts at any byte; its 5
// bytes always fall inside two consecutive aligned 32-bit words, which are the
// only bytes fetched (no sector is touched that the reference would not touch).
__device__ __forceinline__ uint64_t load_suffix(const uint8_t *__restrict__ recs, uint64_t byte_addr) {
    const uint32_t *p = reinterpret_cast<const uint32_t *>(recs + (byte_addr & ~3ull));
    uint32_t w0 = __ldg(p), w1 = __ldg(p + 1);
    uint32_t sh = (uint32_t)(byte_addr & 3u) * 8u;
    uint64_t v = ((uint64_t)w1 << 32) | w0;
    return (v >> sh) & SUFMASK;
}

__device__ __forceinline__ uint32_t load_ix(const DevDB &db, uint64_t rec) {
    const uint8_t *r = db.recs + rec * db.sz + 5;
    uint32_t v = (uint32_t)__ldg(r) | ((uint32_t)__ldg(r + 1) << 8);
    if (db.ix_bytes == 4) v |= ((uint32_t)__ldg(r + 2) << 16) | ((uint32_t)__ldg(r + 3) << 24);
    return v;
}

struct Probe {            // state of one in-flight xtSuffixBS
    uint64_t pos, size, suf;
    bool live;            // bucket non-empty
};

__device__ __forceinline__ void probe_begin(const DevDB &db, uint64_t word, Probe &q) {
    uint64_t p = word >> 40;
    uint64_t a, b;
    if (db.binix32) { a = __ldg(db.binix32 + p); b = __ldg(db.binix32 + p + 1); }
    else { a = __ldg(db.binix64 + p); b = __ldg(db.binix64 + p + 1); }
    q.suf = word & SUFMASK;
    q.live = a < b;                                    // itree.c:726
    // a CTR whose index points past the blob would make the reference read
    // out of bounds; clamp so the device never does
    if (b > db.num_nodes) q.live = false;
    q.pos = a;
    q.size = q.live ? b - a - 1 : 0;                   // itree.c:728
}

template <int N>
__device__ __forceinline__ void probe_run(const DevDB &db, Probe (&q)[N]) {
    // Lock-step binary searches: every round issues the N independent loads
    // first, then resolves the N compares (itree.c:701-705).
    for (;;) {
        bool any = false;
#pragma unroll
        for (int i = 0; i < N; ++i) any |= q[i].size != 0;
        if (!any) break;
        uint64_t v[N], h[N];
#pragma unroll
        for (int i = 0; i < N; ++i) {
            h[i] = q[i].size >> 1;
            v[i] = q[i].size ? load_suffix(db.recs, (q[i].pos + h[i] + 1) * db.sz) : 0;
        }
#pragma unroll
        for (int i = 0; i < N; ++i) {
            if (q[i].size) {
                if (v[i] <= q[i].suf) { q[i].pos += h[i] + 1; q[i].size -= h[i] + 1; }
                else q[i].size = h[i];
            }
        }
    }
}

__device__ __forceinline__ uint32_t probe_end(const DevDB &db, const Probe &q) {
    if (!q.live) return HIT_MISS;
    if (load_suffix(db.recs, q.pos * db.sz) != q.suf) return HIT_MISS;   // itree.c:706
    uint32_t ix = load_ix(db, q.pos);
    return ix < db.max_ix ? ix : HIT_MISS;                                // itree.c:929
}


// ---- sector hash table (regular CTRs only) -----------------------------------
// What bounds an exact lookup on the device is the chain of dependent random
// DRAM accesses (profiles/r01_*: the reference's bisection makes ~8 round trips,
// index -> interpolated key window -> aux still 3).  For a regular CTR (every
// bucket strictly sorted -- verified on the device at upload -- so all record
// words are distinct and any exact membership test returns what xtSuffixBS
// returns) the records are therefore re-keyed once, at load time, into an open-
// addressing table whose bucket is one 32-byte sector:
//     h = mix64(word)  (a bijection)      home sector = floor(h * S / 2^64)
//     entry (8 B) = low 48 bits of h << 16 | tag        4 entries per sector
// uint16_t labels: tag = 0xFFFF - id (never 0: 0xFFFE/0xFFFF are the builder's
// sentinels, itree.c:105-107).  uint32_t labels: THREE entries per sector with the
// id inside (words 0-2 the ids, 3-5 the low 32 bits of the remainders, 6-7 their
// upper 16 bits and three "occupied" bits) -- a parallel id array costs a second
// random access per hit, which is what bound the lookups on uint32_t trees
// (profiles/r02_*: 22 ms of a 44 ms step).  An entry that does not fit its home sector goes to the
// next one (linear probing over sectors, displacement <= KT_MAXD, load <= 0.5),
// so a lookup is ONE random 32-byte access (1.06 on average) with no index in
// front of it.  Uniqueness of the 48-bit remainder: an entry found within
// KT_MAXD sectors of the probe's home has a hash within (KT_MAXD+1) * 2^64 / S
// <= 2^48 of the probe's (S >= KT_MIN_SECTORS), so equal low 48 bits mean equal
// hashes, hence equal words.
#define KT_MAXD 63u
#define KT_MIN_SECTORS ((uint64_t)(KT_MAXD + 1u) << 16)
__device__ __forceinline__ uint64_t mix64(uint64_t x) {           // murmur3 finaliser: invertible
    x ^= x >> 33; x *= 0xFF51AFD7ED558CCDull;
    x ^= x >> 33; x *= 0xC4CEB9FE1A85EC53ull;
    return x ^ (x >> 33);
}
// uint32_t labels (see above).  Sector as two uint4: a = {id0, id1, id2, lo0}, b = {lo1, lo2, hi0 | hi1 << 16, hi2 | occupied << 16}
__device__ __forceinline__ uint32_t kt_lookup_wide(const DevDB &db, uint64_t word, uint32_t *sect) {
    const uint64_t h = mix64(word);
    const uint32_t lo = (uint32_t)h, hi = (uint32_t)(h >> 32) & 0xFFFFu;
    uint64_t s = __umul64hi(h, db.kt_sectors);
    uint32_t ns = 0, r = HIT_MISS;
    for (uint32_t d = 0; d <= KT_MAXD; ++d) {
        const uint4 *p = reinterpret_cast<const uint4 *>(db.ktab + s * 4);
        const uint4 a = __ldg(p), b = __ldg(p + 1);
        ++ns;
        const uint32_t occ = b.w >> 16;
        uint32_t ix = HIT_MISS;
        bool found = false;
        if ((occ & 1u) && a.w == lo && (b.z & 0xFFFFu) == hi) { ix = a.x; found = true; }
        if ((occ & 2u) && b.x == lo && (b.z >> 16) == hi) { ix = a.y; found = true; }
        if ((occ & 4u) && b.y == lo && (b.w & 0xFFFFu) == hi) { ix = a.z; found = true; }
        if (found) { r = ix < db.max_ix ? ix : HIT_MISS; break; }   // itree.c:929
        if (occ != 7u) break;                                      // a free slot: the word was never displaced past here
        if (++s == db.kt_sectors) s = 0;
    }
    if (sect) *sect = ns;
    return r;
}
// sect (optional): 32-byte sectors this lookup touched
__device__ __forceinline__ uint32_t kt_lookup(const DevDB &db, uint64_t word, uint32_t *sect = nullptr) {
    if (db.kt_wide) return kt_lookup_wide(db, word, sect);
    const uint64_t h = mix64(word), rem = h << 16;
    uint64_t s = __umul64hi(h, db.kt_sectors);
    uint32_t ns = 0, r = HIT_MISS;
    for (uint32_t d = 0; d <= KT_MAXD; ++d) {
        const ulonglong2 *p = reinterpret_cast<const ulonglong2 *>(db.ktab + s * 4);
        const ulonglong2 a = __ldg(p), b = __ldg(p + 1);
        const uint64_t e[4] = {a.x, a.y, b.x, b.y};
        ++ns;
        int at = -1;
        uint32_t tag = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) if (e[j] && ((e[j] ^ rem) >> 16) == 0) { at = j; tag = (uint32_t)(e[j] & 0xFFFFu); }
        if (at >= 0) {
            const uint32_t ix = 0xFFFFu - tag;
            r = ix < db.max_ix ? ix : HIT_MISS;                    // itree.c:929
            break;
        }
        if (!(e[0] && e[1] && e[2] && e[3])) break;                // a free slot: the word was never displaced past here
        if (++s == db.kt_sectors) s = 0;
    }
    if (sect) *sect = ns;
    return r;
}
// G lanes per prefix bin walk the bin's records (bins are taken as the index gives them, itree.c:722-726)
template <int G>
__global__ void __launch_bounds__(256)
ktab_build_kernel(DevDB db, unsigned long long *__restrict__ ktab, uint32_t wide, uint64_t n_sectors,
                  uint32_t *__restrict__ overflow) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t p = t / G;
    const uint32_t gl = (uint32_t)(t % G);
    if (p >= UTB_NUMBINS - 1) return;
    uint64_t a, b;
    if (db.binix32) { a = db.binix32[p]; b = db.binix32[p + 1]; }
    else { a = db.binix64[p]; b = db.binix64[p + 1]; }
    if (a >= b || b > db.num_nodes) return;
    if ((uint32_t)p == db.quirk_bin) ++a;                          // the folded record is unreachable for xtSuffixBS (SURVEY 0 #4)
    for (uint64_t i = a + gl; i < b; i += G) {
        const uint64_t word = (p << 40) | load_suffix(db.recs, i * db.sz);
        const uint32_t ix = load_ix(db, i);
        const uint64_t h = mix64(word);
        uint64_t s = __umul64hi(h, n_sectors);
        bool placed = false;
        if (wide) {
            if (ix >= db.max_ix) continue;                         // never passes ix < maxIX (itree.c:929): as good as absent
            for (uint32_t d = 0; d <= KT_MAXD && !placed; ++d) {
                uint32_t *w = reinterpret_cast<uint32_t *>(ktab + s * 4);
#pragma unroll
                for (uint32_t j = 0; j < 3 && !placed; ++j) {
                    const uint32_t bit = 1u << (16u + j);
                    if (w[7] & bit) continue;
                    if (atomicOr(w + 7, bit) & bit) continue;      // somebody else took it
                    w[j] = ix; w[3 + j] = (uint32_t)h;
                    const uint32_t hi = (uint32_t)(h >> 32) & 0xFFFFu;
                    if (j == 0) atomicOr(w + 6, hi); else if (j == 1) atomicOr(w + 6, hi << 16); else atomicOr(w + 7, hi);
                    placed = true;
                }
                if (!placed && ++s == n_sectors) s = 0;
            }
        } else {
            const unsigned long long entry = (h << 16) | (unsigned long long)(0xFFFFu - (ix & 0xFFFFu));
            if (ix >= 0xFFFEu) continue;                           // sentinel ids never pass ix < maxIX (itree.c:929)
            for (uint32_t d = 0; d <= KT_MAXD && !placed; ++d) {
#pragma unroll
                for (int j = 0; j < 4 && !placed; ++j) {
                    if (ktab[s * 4 + j]) continue;
                    if (atomicCAS(ktab + s * 4 + j, 0ull, entry) == 0ull) placed = true;
                }
                if (!placed && ++s == n_sectors) s = 0;
            }
        }
        if (!placed) atomicAdd(overflow, 1u);
    }
}

// Load-time check of the invariant the table relies on.
// out[0] buckets with a disorder past their first pair (or an index beyond the blob)
// out[1] buckets whose only disorder is record0 >= record1   out[2] smallest such bin
// out[3] first non-empty bin
__global__ void __launch_bounds__(256)
verify_kernel(DevDB db, unsigned long long *__restrict__ out) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= UTB_NUMBINS - 1) return;
    uint64_t a, b;
    if (db.binix32) { a = db.binix32[p]; b = db.binix32[p + 1]; }
    else { a = db.binix64[p]; b = db.binix64[p + 1]; }
    if (a >= b) return;                                            // empty for XT_getIX32 (itree.c:726)
    if (b > db.num_nodes) { atomicAdd(out + 0, 1ull); return; }
    atomicMin(out + 3, (unsigned long long)p);
    uint64_t prev = load_suffix(db.recs, a * db.sz);
    bool first_bad = false, rest_bad = false;
    for (uint64_t i = a + 1; i < b; ++i) {
        uint64_t cur = load_suffix(db.recs, i * db.sz);
        if (cur <= prev) { if (i == a + 1) first_bad = true; else rest_bad = true; }
        prev = cur;
    }
    if (rest_bad) atomicAdd(out + 0, 1ull);
    else if (first_bad) { atomicAdd(out + 1, 1ull); atomicMin(out + 2, (unsigned long long)p); }
}

// ---- minimizer-keyed sieve (membership pre-filter) -------------------------------
// Most 32-mers of a read are not in a sampled tree (complevel 2 keeps 1/16 of the
// k-mers), so a blocked Bloom filter over the record words, built on the device at
// upload, answers "certainly absent" before the exact table is touched.  No false
// negatives, so a filtered miss is a miss of XT_getIX32 too; positives take the
// exact path.  What one random filter probe per position costs on B200 is one
// 128-byte DRAM line fill (profiles/r01_membench*): 47.5 G fills/s, 25 ms for the
// 1.19 G positions of 10 M reads.  So the LINE of a word is not chosen by the word
// but by its MINIMIZER: the smallest hash among the canonical 16-mers (min of a
// 16-mer and its reverse complement) inside the 32-mer.  Consecutive windows of a
// read share their minimizer for 9 positions on average (density 2/(w+1), w = 17),
// and lane = position, so the 32 probes of a warp instruction fall into ~4.4 lines
// which the L1 coalesces into as many requests: one DRAM line per ~9 positions, no
// partitioning pass, nothing that depends on the batch size.  The minimizer is
// strand-neutral (itree.c:887-898 makes every window be searched on both strands),
// so x and revcomp(x) share the line; inside it the 8-byte BLOCK (16 per line) is
// chosen by a strand-neutral hash and the eight BITS, one in each byte of the
// block, by x itself: one 8-byte load per position answers both strands, and the
// two mask words of a strand cost two PRMTs (byte table 1 << n, selected by 3-bit
// fields of a hash) -- the kernel is bound by the integer pipe, not by memory
// (profiles/r02_*, r03_*).  Lines hold SV_RPL records on average (~43 bits per record:
// ~0.04 % false positives, the spread of the line loads included).
// Every function here takes a 32-mer as its bit planes x1 (code bit 1 of each base) and x0 (code bit 0), base 0 the
// most significant bit (word_to_planes): the sieve kernel builds a window with one funnel shift per plane and the
// reverse complement of a plane is ~__brev(plane).  The build, the sieve kernel and the stage-level lookups all call
// these, so the three cannot disagree on a hash.  A 16-mer (planes a1, a0 of 16 bits) is keyed as
// a1[15:8] | a0 | a1[7:0], most significant first: one PRMT from the upper halves of the planes, and a layout that a
// bit reversal maps onto itself, so the reverse complement of a key is ~__brev(key).
#define SV_W 17u                // 16-mers per 32-mer
#define SV_RPL 24u              // records per 128-byte line
__device__ __forceinline__ uint32_t sv_kmer16(uint32_t x1, uint32_t x0) { return __byte_perm(x1, x0, 0x3762); }   // the 16-mer at offset 0
__device__ __forceinline__ uint32_t sv_rc16(uint32_t m) { return ~__brev(m); }   // the key of its reverse complement
__device__ __forceinline__ uint32_t sv_mhash(uint32_t m, uint32_t r) {   // order key of a 16-mer m with reverse complement r
    uint32_t a = m < r ? m : r;
    a *= 0x9E3779B1u; a ^= a >> 15; a *= 0x85EBCA77u;
    return a;
}
__device__ __forceinline__ uint32_t sv_line(uint32_t mv, uint32_t n_lines) {   // n_lines < 2^28: a block index fits 32 bits
    uint32_t t = mv * 0xB5297A4Du; t ^= t >> 16; t *= 0x68E31DA5u;           // the minimum of 17 hashes is small: spread it again
    return __umulhi(t, n_lines);
}
// h0 / h16: order keys of the first and the last 16-mer of the word -- the reverse complement swaps the two, so
// the block is the same for both strands (and independent of the line, which the minimum of all 17 keys picks)
__device__ __forceinline__ uint32_t sv_block(uint32_t h0, uint32_t h16) { return (h0 ^ h16) >> 28; }
// the word's two mask words: one bit in each of the block's 8 bytes
__device__ __forceinline__ uint2 sv_masks(uint32_t x1, uint32_t x0) {
    uint32_t e = x1 * 0xC2B2AE3Du + x0 * 0x27D4EB2Fu;
    e ^= e >> 15;
    const uint32_t s0 = __umulhi(e, 0x165667B1u) & 0x7777u, s1 = __umulhi(e, 0x9E3779B1u) & 0x7777u;   // 4 x 3-bit byte selectors each
    return make_uint2(__byte_perm(0x08040201u, 0x80402010u, s0), __byte_perm(0x08040201u, 0x80402010u, s1));
}
__device__ __forceinline__ bool sv_test(const uint2 &v, uint32_t x1, uint32_t x0) {
    const uint2 m = sv_masks(x1, x0);
    return ((~v.x & m.x) | (~v.y & m.y)) == 0u;
}
// (line, block) of one word, the slow way (build, stage-level lookups): all 17 16-mers
__device__ __forceinline__ uint32_t sv_index(const DevDB &db, uint32_t x1, uint32_t x0) {
    uint32_t mv = 0xFFFFFFFFu, h0 = 0, h16 = 0;
#pragma unroll
    for (uint32_t j = 0; j < SV_W; ++j) {
        const uint32_t m = sv_kmer16(x1 << j, x0 << j);
        const uint32_t h = sv_mhash(m, sv_rc16(m));
        mv = h < mv ? h : mv;
        if (j == 0) h0 = h;
        if (j == SV_W - 1) h16 = h;
    }
    return (sv_line(mv, db.sv_lines) << 4) | sv_block(h0, h16);
}
__device__ __forceinline__ bool sv_maybe(const DevDB &db, uint64_t word) {   // word: the 2-bit form
    const uint64_t x = word_to_planes(word);
    const uint32_t x1 = (uint32_t)(x >> 32), x0 = (uint32_t)x;
    return sv_test(__ldg(db.sieve + sv_index(db, x1, x0)), x1, x0);
}
template <int G>
__global__ void __launch_bounds__(256)
sieve_build_kernel(DevDB db, uint32_t *__restrict__ sieve) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t p = t / G;
    const uint32_t gl = (uint32_t)(t % G);
    if (p >= UTB_NUMBINS - 1) return;
    uint64_t a, b;
    if (db.binix32) { a = db.binix32[p]; b = db.binix32[p + 1]; }
    else { a = db.binix64[p]; b = db.binix64[p + 1]; }
    if (a >= b || b > db.num_nodes) return;
    if ((uint32_t)p == db.quirk_bin) ++a;                          // the folded record is unreachable anyway
    for (uint64_t i = a + gl; i < b; i += G) {
        const uint64_t x = word_to_planes((p << 40) | load_suffix(db.recs, i * db.sz));
        const uint32_t x1 = (uint32_t)(x >> 32), x0 = (uint32_t)x;
        uint32_t *blk = sieve + 2ull * sv_index(db, x1, x0);
        const uint2 m = sv_masks(x1, x0);
        atomicOr(blk + 0, m.x); atomicOr(blk + 1, m.y);
    }
}

// One thread per (position, strand) of the packed super-sequence: lanes 2k and
// 2k+1 look up the forward and the reverse-complement word of window k, so the
// hit slots of a warp are 32 consecutive u32.  No block-level synchronisation;
// lookups and hits are counted per warp into COUNTER_SLOTS spread counters that
// the host sums.  TABLE: the sector hash table (regular CTRs with the sieve
// switched off: dense trees where most lookups hit); else the reference's probe
// sequence on the on-disk records (irregular CTRs, UTB_LOOKUP=exact).
#define COUNTER_SLOTS 1024
template <int NSTR, bool TABLE>
__global__ void __launch_bounds__(256, 6)
lookup_kernel(DevDB db, const uint64_t *__restrict__ pk, const uint32_t *__restrict__ bad,
              uint32_t n_pos, const uint32_t *__restrict__ n_groups_dev, uint32_t *__restrict__ hits, unsigned long long *__restrict__ counters) {
    if (n_groups_dev) n_pos = *n_groups_dev * 32u;
    const uint64_t slot = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t pos = (uint32_t)(NSTR == 2 ? slot >> 1 : slot);
    uint64_t w = 0;
    const bool valid = pos < n_pos && window_at(pk, bad, pos, w);
    uint32_t r = HIT_NOWIN, ns = 0;
    if (valid) {
        if (NSTR == 2 && (slot & 1)) w = revcomp_word(w);
        if (TABLE) r = kt_lookup(db, w, &ns);
        else {
            Probe q[1];
            probe_begin(db, w, q[0]);
            probe_run<1>(db, q);
            r = probe_end(db, q[0]);
        }
    }
    if (pos < n_pos) hits[slot] = r;
    const uint32_t nv = __popc(__ballot_sync(0xFFFFFFFFu, valid));
    const uint32_t nh = __popc(__ballot_sync(0xFFFFFFFFu, r < HIT_NOWIN));
    for (int o = 16; o; o >>= 1) ns += __shfl_xor_sync(0xFFFFFFFFu, ns, o);
    if ((threadIdx.x & 31u) == 0) {
        const uint32_t c = blockIdx.x & (COUNTER_SLOTS - 1);
        if (nv) atomicAdd(counters + c, (unsigned long long)nv);
        if (nh) atomicAdd(counters + COUNTER_SLOTS + c, (unsigned long long)nh);
        if (ns) atomicAdd(counters + 3 * COUNTER_SLOTS + c, (unsigned long long)ns);
    }
}

// ---- two-phase lookup (sieve on) ----------------------------------------------------
// In one fused kernel every warp waits for its slowest lane, i.e. for the one
// or two lanes per warp whose word passes the sieve and goes on to the table,
// while the other ~30 lanes idle.  So the work is split into two dense passes:
// phase A (sieve_kernel) tests every window against the sieve and appends the
// survivors to a queue through per-warp chunks; phase B (queue_lookup_kernel)
// runs the exact lookup over the queue with every lane busy.
#define Q_CHUNK 128u              // queue slots a warp reserves per atomic (>= 64: two ballots per step)
#define Q_INVALID 0xFFFFFFFFu
// A warp's private window into the survivor queue: the global counter sees one
// atomic per Q_CHUNK survivors instead of one per warp-step.
struct WarpQueue {
    uint64_t base;
    uint32_t used;
    bool have;
};
__device__ __forceinline__ void wq_init(WarpQueue &q) { q.base = 0; q.used = Q_CHUNK; q.have = false; }
__device__ __forceinline__ void wq_retire(const WarpQueue &q, uint32_t lane, uint32_t *__restrict__ q_slots) {
    if (q.have) for (uint32_t j = q.used + lane; j < Q_CHUNK; j += 32) q_slots[q.base + j] = Q_INVALID;   // pad the tail
}
// make room for c more entries (warp-uniform call); q_cap is a multiple of Q_CHUNK
__device__ __forceinline__ void wq_reserve(WarpQueue &q, uint32_t c, uint32_t lane, uint32_t *__restrict__ q_slots,
                                           unsigned long long *__restrict__ q_count, uint64_t q_cap) {
    if (q.used + c <= Q_CHUNK) return;
    wq_retire(q, lane, q_slots);
    unsigned long long nb = 0;
    if (lane == 0) nb = atomicAdd(q_count, (unsigned long long)Q_CHUNK);
    q.base = __shfl_sync(0xFFFFFFFFu, nb, 0);
    q.used = 0;
    q.have = q.base + Q_CHUNK <= q_cap;                            // beyond capacity: the caller resolves inline
}
// Where the labels of the hits go.  List mode (cnt != null, the GG path): appended to the hit list of the READ the slot
// belongs to -- the list starts at the read's first slot in `hits`, cnt[read] counts it; rid maps a 32-position
// group to its read.  The vote then reads one or two sectors per read instead of a hit map plus one gather per hit,
// and phase B writes next to what it wrote before instead of read-modify-writing a random line of `hits` and one of
// the map per hit.  Scatter mode (cnt == null, the non-GG path, which needs positions): hits[slot] + a bit in hitmap.
struct HitSink {
    uint32_t *hits;
    uint32_t *hitmap;
    const uint32_t *rid, *grp_off;
    uint32_t *cnt;
    uint32_t sh;                                                    // log2(slots per group): 5 + (strands == 2)
};
__device__ __forceinline__ void sink_put(const HitSink &k, uint32_t slot, uint32_t r) {   // one hit, any thread
    if (k.cnt) {
        const uint32_t rd = __ldg(k.rid + (slot >> k.sh));
        k.hits[((uint64_t)__ldg(k.grp_off + rd) << k.sh) + atomicAdd(k.cnt + rd, 1u)] = r;
    } else { k.hits[slot] = r; atomicOr(k.hitmap + (slot >> 5), 1u << (slot & 31u)); }
}
// queue overflow: the exact lookup right here (rare); x: the window's planes
__device__ __noinline__ uint32_t resolve_inline(const DevDB &db, uint64_t x, uint32_t slot, const HitSink &sink) {
    const uint32_t r = kt_lookup(db, planes_to_word(x));
    if (r == HIT_MISS) return 0;
    sink_put(sink, slot, r);
    return 1;
}
// Appends the survivors of one warp step (warp-uniform call).  w / rc: the planes of the window and of its reverse
// complement; the queue keeps planes, phase B turns them into words (only ~2.5 % of the windows get there).
template <int NSTR>
__device__ __forceinline__ uint32_t emit_survivors(const DevDB &db, WarpQueue &wq, uint32_t lane, bool passF, bool passR, uint64_t w, uint64_t rc,
                                                   uint32_t pos, uint64_t *__restrict__ q_words, uint32_t *__restrict__ q_slots,
                                                   unsigned long long *__restrict__ q_count, uint64_t q_cap, const HitSink &sink) {
    const uint32_t bF = __ballot_sync(0xFFFFFFFFu, passF);
    const uint32_t bR = NSTR == 2 ? __ballot_sync(0xFFFFFFFFu, passR) : 0u;
    const uint32_t cF = __popc(bF), c = cF + __popc(bR);
    uint32_t nh = 0;
    if (!c) return 0;
    wq_reserve(wq, c, lane, q_slots, q_count, q_cap);
    const uint32_t lt = (1u << lane) - 1u;
    if (wq.have) {
        const uint64_t at = wq.base + wq.used;
        if (passF) { const uint64_t i = at + __popc(bF & lt); q_words[i] = w; q_slots[i] = pos * NSTR; }
        if (passR) { const uint64_t i = at + cF + __popc(bR & lt); q_words[i] = rc; q_slots[i] = pos * NSTR + 1u; }
    } else {
        if (passF) nh += resolve_inline(db, w, pos * NSTR, sink);
        if (passR) nh += resolve_inline(db, rc, pos * NSTR + 1u, sink);
    }
    wq.used += c;
    return nh;
}

// Phase A.  Persistent warps; every warp owns a contiguous range of 32-position steps (one step = one
// group of the packed stream, lane = position) and walks it SV_U steps at a time.  Per step a lane
// builds its window -- one funnel shift per plane of two consecutive groups of the plane stream pl --
// and the hash of the canonical 16-mer that STARTS at its position; the minimizer of a window is the
// minimum of the 17 hashes at positions p .. p+16, taken across lanes with shuffles (doubling: 2, 4, 8,
// 16, 17), where positions beyond lane 31 belong to the next step -- which is computed one tile ahead
// and carried over, so nothing is computed twice.  The reverse complement of a window is derived only
// where its strand is tested.
// template parameters of sieve_kernel: SV_U steps per tile (= filter loads in flight per lane), SV_MINB CTAs per SM
// the register budget is sized for (launch_stages uses U = 6 at 3 CTAs per SM; the measurements are at the launch)
#define SV_DEAD 0xFFFFFFFFu       // SvStep.blk of a position without a valid window
struct SvStep { uint32_t w1, w0, h, blk; };                       // window planes, 16-mer hash, SV_DEAD or (later) block in the line
// cur / next: groups s and s + 1 of pl, bh / bl: of bad
__device__ __forceinline__ void sv_step(uint64_t cur, uint64_t next, uint32_t bh, uint32_t bl, uint32_t lane, SvStep &s) {
    s.w1 = __funnelshift_l((uint32_t)(next >> 32), (uint32_t)(cur >> 32), lane);
    s.w0 = __funnelshift_l((uint32_t)next, (uint32_t)cur, lane);
    const uint32_t m = sv_kmer16(s.w1, s.w0);
    s.h = sv_mhash(m, sv_rc16(m));
    s.blk = __funnelshift_r(bh, bl, lane) == 0u ? 0u : SV_DEAD;   // a bad base in the 32 positions from here: no window
}
// x[u][lane] -> value of the (virtual) array x at index 32 * u + lane + D; the last array only serves lanes that stay inside it
template <int D, int SV_U>
__device__ __forceinline__ void sv_shifted(const uint32_t (&x)[SV_U + 1], uint32_t (&y)[SV_U + 1], uint32_t lane) {
    uint32_t rot[SV_U + 1];
#pragma unroll
    for (int u = 0; u <= SV_U; ++u) rot[u] = __shfl_sync(0xFFFFFFFFu, x[u], (lane + D) & 31u);
    const bool same = lane + D < 32u;
#pragma unroll
    for (int u = 0; u < SV_U; ++u) y[u] = same ? rot[u] : rot[u + 1];
    y[SV_U] = rot[SV_U];
}
__device__ __forceinline__ void sv_prefetch(const void *p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
template <int NSTR, int SV_U, int SV_MINB>
__global__ void __launch_bounds__(256, SV_MINB)
sieve_kernel(DevDB db, const uint64_t *__restrict__ pl, const uint32_t *__restrict__ bad, uint32_t n_pos,
             const uint32_t *__restrict__ n_groups_dev, unsigned long long *__restrict__ counters,
             uint64_t *__restrict__ q_words, uint32_t *__restrict__ q_slots, unsigned long long *__restrict__ q_count,
             uint64_t q_cap, const HitSink sink) {
    if (n_groups_dev) n_pos = *n_groups_dev * 32u;
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t n_steps = n_pos >> 5;                           // n_pos is a multiple of 32; PK_GUARD all-bad groups follow group n_steps - 1
    const uint32_t n_warps = gridDim.x * (blockDim.x >> 5), wid = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    uint32_t per = (n_steps + n_warps - 1) / n_warps;
    per = (per + SV_U - 1) / SV_U * SV_U;
    const uint64_t s0 = (uint64_t)wid * per;
    const uint32_t s1 = s0 + per < n_steps ? (uint32_t)(s0 + per) : n_steps;
    const uint2 *__restrict__ sieve = db.sieve;
    const uint32_t n_lines = db.sv_lines;
    WarpQueue wq;
    wq_init(wq);
    uint32_t nv = 0, nh = 0;
    if (s0 < s1) {
        SvStep st[SV_U + 1];
        // groups s and s + 1 feed step s; the pair is carried from step to step (one 8-byte and one 4-byte load per step).
        // A tile may run past s1 only at the very end of the batch, into the guard groups: no bounds checks in the loop.
        uint64_t cur = __ldg(pl + s0), next = __ldg(pl + s0 + 1);
        uint32_t bh = __ldg(bad + s0), bl = __ldg(bad + s0 + 1);
        sv_step(cur, next, bh, bl, lane, st[0]);
        for (uint32_t s = (uint32_t)s0; s < s1; s += SV_U) {
            {   // both streams are read front to back: ask for the lines two ahead (a line of pl feeds 16 steps)
                const uint32_t pf = s + 32u < n_steps ? s + 32u : n_steps;
                sv_prefetch(pl + pf); sv_prefetch(bad + pf);
            }
#pragma unroll
            for (int u = 1; u <= SV_U; ++u) {
                cur = next; bh = bl;
                next = __ldg(pl + s + u + 1); bl = __ldg(bad + s + u + 1);
                sv_step(cur, next, bh, bl, lane, st[u]);
            }
            // minimizer = min of the 17 hashes at q .. q+16: windows of 3, then 9 (3 + 3 + 3), then 17 (9 + 9, one shared)
            uint32_t x[SV_U + 1], y1[SV_U + 1], y2[SV_U + 1];
#pragma unroll
            for (int u = 0; u <= SV_U; ++u) x[u] = st[u].h;
            sv_shifted<16, SV_U>(x, y1, lane);                                           // the window's last 16-mer
#pragma unroll
            for (int u = 0; u < SV_U; ++u) st[u].blk |= sv_block(x[u], y1[u]);          // SV_DEAD stays SV_DEAD
            sv_shifted<1, SV_U>(x, y1, lane); sv_shifted<2, SV_U>(x, y2, lane);
#pragma unroll
            for (int u = 0; u <= SV_U; ++u) x[u] = __vimin3_u32(x[u], y1[u], y2[u]);     // [q, q+2]
            sv_shifted<3, SV_U>(x, y1, lane); sv_shifted<6, SV_U>(x, y2, lane);
#pragma unroll
            for (int u = 0; u <= SV_U; ++u) x[u] = __vimin3_u32(x[u], y1[u], y2[u]);     // [q, q+8]
            sv_shifted<8, SV_U>(x, y1, lane);
#pragma unroll
            for (int u = 0; u < SV_U; ++u) x[u] = x[u] < y1[u] ? x[u] : y1[u];           // [q, q+16]
            uint2 v[SV_U];
#pragma unroll
            for (int u = 0; u < SV_U; ++u) {
                v[u] = make_uint2(0, 0);
                if (st[u].blk != SV_DEAD) v[u] = __ldg(sieve + ((sv_line(x[u], n_lines) << 4) | st[u].blk));
            }
#pragma unroll
            for (int u = 0; u < SV_U; ++u) {
                const bool live = st[u].blk != SV_DEAD;
                if (__any_sync(0xFFFFFFFFu, live)) {               // the padding group behind every read holds no window at all
                    const uint32_t r1 = ~__brev(st[u].w1), r0 = ~__brev(st[u].w0);   // the reverse complement's planes
                    const bool tF = sv_test(v[u], st[u].w1, st[u].w0), tR = NSTR == 2 && sv_test(v[u], r1, r0);
                    nh += emit_survivors<NSTR>(db, wq, lane, live & tF, live & tR, ((uint64_t)st[u].w1 << 32) | st[u].w0, ((uint64_t)r1 << 32) | r0,
                                               (s + u) * 32u + lane, q_words, q_slots, q_count, q_cap, sink);
                    nv += live ? NSTR : 0;                         // nothing is stored for a miss
                }
            }
            st[0] = st[SV_U];
        }
    }
    wq_retire(wq, lane, q_slots);
    for (int o = 16; o; o >>= 1) { nv += __shfl_xor_sync(0xFFFFFFFFu, nv, o); nh += __shfl_xor_sync(0xFFFFFFFFu, nh, o); }
    if (lane == 0) {
        const uint32_t cs = (blockIdx.x * 8 + (threadIdx.x >> 5)) & (COUNTER_SLOTS - 1);
        if (nv) atomicAdd(counters + cs, (unsigned long long)nv);
        if (nh) atomicAdd(counters + COUNTER_SLOTS + cs, (unsigned long long)nh);
    }
}

// Phase B: one survivor per thread, ONE random 32-byte table access each (no chain to wait for).  LISTS: the hits
// of a warp that belong to the same read (neighbours in the queue do) reserve their places in that read's list
// with one atomic and store side by side.
template <bool LISTS>
__global__ void __launch_bounds__(256, 6)
queue_lookup_kernel(DevDB db, const uint64_t *__restrict__ q_words, const uint32_t *__restrict__ q_slots,
                    const unsigned long long *__restrict__ q_count, uint64_t q_cap,
                    const HitSink sink, unsigned long long *__restrict__ counters) {
    const uint64_t n = *q_count < q_cap ? *q_count : q_cap;       // both multiples of Q_CHUNK: every entry below n was written
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint32_t lane = threadIdx.x & 31u;
    uint32_t nh = 0, nsect = 0;
    // n and the stride are multiples of 32: the lanes of a warp leave the loop together
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t slot = q_slots[i];
        uint32_t r = HIT_MISS;
        if (slot != Q_INVALID) {                                   // else: padding of a retired chunk
            uint32_t sc;
            r = kt_lookup(db, planes_to_word(q_words[i]), &sc);   // the queue holds planes (see emit_survivors)
            nsect += sc;
        }
        const bool hit = r != HIT_MISS;
        nh += hit;
        if (!LISTS) {
            if (hit) { sink.hits[slot] = r; atomicOr(sink.hitmap + (slot >> 5), 1u << (slot & 31u)); }
            continue;
        }
        if (!__any_sync(0xFFFFFFFFu, hit)) continue;
        const uint32_t rd = hit ? __ldg(sink.rid + (slot >> sink.sh)) : 0xFFFFFFFFu;
        const uint32_t peers = __match_any_sync(0xFFFFFFFFu, rd);
        const uint32_t leader = (uint32_t)__ffs(peers) - 1u;
        uint32_t base = 0;
        if (hit && lane == leader) base = atomicAdd(sink.cnt + rd, (uint32_t)__popc(peers));
        base = __shfl_sync(0xFFFFFFFFu, base, leader);
        if (hit) sink.hits[((uint64_t)__ldg(sink.grp_off + rd) << sink.sh) + base + __popc(peers & ((1u << lane) - 1u))] = r;
    }
    for (int o = 16; o; o >>= 1) { nh += __shfl_xor_sync(0xFFFFFFFFu, nh, o); nsect += __shfl_xor_sync(0xFFFFFFFFu, nsect, o); }
    if (lane == 0) {
        const uint32_t c = blockIdx.x & (COUNTER_SLOTS - 1);
        if (nh) atomicAdd(counters + COUNTER_SLOTS + c, (unsigned long long)nh);
        if (nsect) atomicAdd(counters + 3 * COUNTER_SLOTS + c, (unsigned long long)nsect);
    }
}

// stage-level: words[] -> ix[] (utb_lookup_words)
template <bool TABLE>
__global__ void lookup_words_kernel(DevDB db, const uint64_t *__restrict__ words, uint64_t n, uint32_t *__restrict__ ix) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (TABLE) {
        if (db.sieve && !sv_maybe(db, words[i])) { ix[i] = HIT_MISS; return; }
        ix[i] = kt_lookup(db, words[i]);
        return;
    }
    Probe q[1];
    probe_begin(db, words[i], q[0]);
    probe_run<1>(db, q);
    ix[i] = probe_end(db, q[0]);
}


// stage-level: expose every window of the packed stream (utb_pack_sequence)
__global__ void expand_windows_kernel(const uint64_t *__restrict__ pk, const uint32_t *__restrict__ bad, uint32_t n_pos,
                                      uint64_t *__restrict__ fwd, uint64_t *__restrict__ rc, uint8_t *__restrict__ valid) {
    uint32_t pos = blockIdx.x * blockDim.x + threadIdx.x;
    if (pos >= n_pos) return;
    uint64_t w;
    bool ok = window_at(pk, bad, pos, w);
    fwd[pos] = ok ? w : 0;
    rc[pos] = ok ? revcomp_word(w) : 0;
    valid[pos] = ok;
}

// ---------------------------------------------------------------------------
// vote (itree.c:1028-1098)
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cutoff_of(uint32_t x) {   // itree.c:1044-1046
    uint32_t c = x - x / 4u;
    c += ((x >> 1) >= c);
    return c;
}

// itree.c:1060-1061 for one thread: the first t' >= t with s1[t'] == 0 || s1[t'] != s2[t'] || s1[t'] == ';', and the two
// characters there.  Both strings start at a multiple of 8 bytes and are NUL-padded to the next one (the device blob,
// the staged copy), and agree below t: eight characters per step from the same offset in both.
__device__ __forceinline__ unsigned long long nz_bytes(unsigned long long v) {    // bit 7 of every nonzero byte
    return (((v & 0x7F7F7F7F7F7F7F7Full) + 0x7F7F7F7F7F7F7F7Full) | v) & 0x8080808080808080ull;
}
__device__ __forceinline__ uint32_t scan_token(const char *s1, const char *s2, uint32_t t, char &a, char &b) {
    uint32_t tb = t & ~7u;
    unsigned long long keep = ~0ull << (8u * (t & 7u));
    for (;;) {
        const unsigned long long x1 = *reinterpret_cast<const unsigned long long *>(s1 + tb);
        const unsigned long long x2 = *reinterpret_cast<const unsigned long long *>(s2 + tb);
        const unsigned long long stop = ((nz_bytes(x1) & nz_bytes(x1 ^ 0x3B3B3B3B3B3B3B3Bull)) ^ 0x8080808080808080ull | nz_bytes(x1 ^ x2)) & keep;
        if (stop) {
            const uint32_t k = ((uint32_t)__ffsll((long long)stop) - 1u) >> 3;
            a = (char)(x1 >> (8u * k)); b = (char)(x2 >> (8u * k));
            return tb + k;
        }
        tb += 8u; keep = ~0ull;
    }
}

// The aufbau walk, executed by one converged warp; every lane carries the same
// scalar state, the character scans are done 32 bytes at a time with ballots.
// T_lab/T_cnt: the distinct labels of the read in strcmp order with counts
// (shared or global memory).
__device__ void walk_warp(const DevDB &db, const uint32_t *T_lab, const uint32_t *T_cnt,
                          uint32_t uix, uint32_t n, utb_result *out) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t EMPTY = 0xFFFFFFFFu;
    uint32_t cutoff = cutoff_of(n), st = 0, ed = uix, dv = EMPTY, orun = n, sl = 0, ol = 0;
    for (;;) {                                                      // itree.c:1047
        uint32_t run = T_cnt[st], td = dv;
        for (uint32_t z = st + 1; z < ed; ++z) {                    // itree.c:1050
            const char *s1 = db.blob + __ldg(db.off + T_lab[z - 1]);
            const char *s2 = db.blob + __ldg(db.off + T_lab[z]);
            if (!s1[dv + (dv == EMPTY)]) {                          // itree.c:1052
                run = T_cnt[z]; st = z;
                orun -= T_cnt[z - 1];
                cutoff = cutoff_of(orun);
                continue;
            }
            // itree.c:1060-1061: first td >= dv+1 with s1[td]==0 || s1[td]!=s2[td] || s1[td]==';'
            uint32_t t0 = dv + 1u;
            char a, b;
            for (;;) {
                char ca = s1[t0 + lane], cb = s2[t0 + lane];
                uint32_t m = __ballot_sync(0xFFFFFFFFu, ca == 0 || ca != cb || ca == ';');
                if (m) {
                    int src = __ffs(m) - 1;
                    td = t0 + (uint32_t)src;
                    a = (char)__shfl_sync(0xFFFFFFFFu, (int)ca, src);
                    b = (char)__shfl_sync(0xFFFFFFFFu, (int)cb, src);
                    break;
                }
                t0 += 32u;
            }
            if (a == b) run += T_cnt[z];                            // itree.c:1062
            else if ((!a && b == ';') ||
                     ((a == ';' || !a) && td > 0 && s1[td - 1] == '_')) {   // itree.c:1063
                run = T_cnt[z]; st = z;
                orun -= T_cnt[z - 1];
                cutoff = cutoff_of(orun);
            }
            else if (run >= cutoff) { ed = z; break; }              // itree.c:1068
            else { run = T_cnt[z]; st = z; }                        // itree.c:1069
        }
        sl = run; ol = orun;                                        // itree.c:1071
        if (run < cutoff) break;                                    // itree.c:1072
        if (st + 1 >= ed) {                                         // itree.c:1073-1080
            if (T_cnt[ed - 1] >= cutoff) dv = 0xFFFFFFFEu;
            break;
        }
        orun = run; dv = td; cutoff = cutoff_of(run);               // itree.c:1082-1085
    }
    if (lane == 0) {
        out->kind = UTB_WALK; out->label = T_lab[ed - 1]; out->cut = dv;
        out->found = n; out->uix = uix; out->sl = sl; out->ol = ol; out->_pad = 0;
    }
}

struct VoteIn {            // where a read's hits live
    const uint32_t *hits = nullptr;
    const uint32_t *grp_off = nullptr;   // batch mode: position space
    const uint32_t *seq_len = nullptr;
    const uint64_t *off = nullptr;       // stage-level mode: explicit ranges (overrides batch mode)
    uint32_t nstr = 1;
    // two-phase lookup: the survivor kernel appends the labels of a read's hits back to back from the read's first
    // slot and counts them here (any order: the vote is over a multiset); null: one entry per (position, strand)
    const uint32_t *cnt = nullptr;
    // non-GG mode (needs the positions): one bit per slot that holds a label; hits[] is only valid where it is set
    const uint32_t *hitmap = nullptr;
};
__device__ __forceinline__ void vote_range(const VoteIn &in, uint32_t r, uint64_t &start, uint64_t &count) {
    if (in.off) { start = in.off[r]; count = in.off[r + 1] - start; return; }
    start = (uint64_t)__ldg(in.grp_off + r) * 32u * in.nstr;
    if (in.cnt) { count = in.cnt[r]; return; }
    uint32_t len = __ldg(in.seq_len + r);
    uint64_t nwin = len >= 32u ? len - 31u : 0u;
    count = nwin * in.nstr;
}
#define VW_SLOTS 64u            // distinct labels a warp can hold in shared memory
#define VW_MAXHITS 4096u        // entries a single warp will scan (longer reads hold more labels than a warp's table anyway)
#define VW_WARPS 8

// Warp per read: hits -> (label,count) multiset in a shared-memory hash table
// (warp-aggregated with match_any), sorted by label rank, then the walk.
// Reads that are too long or have too many distinct labels are queued for
// vote_block_kernel.
struct VoteWarpSmem { uint32_t *key, *cnt, *rk, *lab, *tc; };
__device__ void vote_warp_read(const DevDB &db, const VoteIn &in, uint32_t r, utb_result *__restrict__ results,
                               uint32_t *__restrict__ gen_list, uint32_t *__restrict__ gen_count,
                               unsigned long long *__restrict__ counters, const VoteWarpSmem &sm) {
    const uint32_t lane = threadIdx.x & 31u;
    uint64_t start, count;
    vote_range(in, r, start, count);
    utb_result *out = results + r;
    if (count > VW_MAXHITS) {
        if (lane == 0) gen_list[atomicAdd(gen_count, 1u)] = r;
        return;
    }
    uint32_t *key = sm.key, *cnt = sm.cnt;
    key[lane] = UTB_BAD32; key[lane + 32] = UTB_BAD32;
    cnt[lane] = 0; cnt[lane + 32] = 0;
    __syncwarp();
    uint32_t n = 0;
    bool overflow = false;
    {
    // dense: 128 slots per round (one uint4 per lane); a round without a label costs one ballot
    const uint32_t mis = (uint32_t)((4u - (start & 3u)) & 3u);     // slots before the first 16-byte boundary
    for (uint64_t base = 0; base < count + 128; base += 128) {
        uint32_t hv[4];
        if (base == 0) {                                           // unaligned head: up to 3 slots, scalar
#pragma unroll
            for (int c = 0; c < 4; ++c) hv[c] = HIT_NOWIN;
            if (lane < mis && lane < count) hv[0] = __ldg(in.hits + start + lane);
        } else {
            const uint64_t i0 = mis + (base - 128) + 4ull * lane;   // aligned body
            if (i0 + 4 <= count) {
                const uint4 q4 = __ldg(reinterpret_cast<const uint4 *>(in.hits + start + i0));
                hv[0] = q4.x; hv[1] = q4.y; hv[2] = q4.z; hv[3] = q4.w;
            } else {
#pragma unroll
                for (int c = 0; c < 4; ++c) hv[c] = i0 + c < count ? __ldg(in.hits + start + i0 + c) : HIT_NOWIN;
            }
            if (mis + (base - 128) >= count) break;
        }
        const bool any4 = hv[0] < db.max_ix || hv[1] < db.max_ix || hv[2] < db.max_ix || hv[3] < db.max_ix;
        if (!__any_sync(0xFFFFFFFFu, any4)) continue;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const uint32_t h = hv[c];
            const bool ok = h < db.max_ix;
            const uint32_t okm = __ballot_sync(0xFFFFFFFFu, ok);
            if (!okm) continue;
            n += __popc(okm);
            const uint32_t peers = __match_any_sync(0xFFFFFFFFu, h);
            if (ok && (uint32_t)(__ffs(peers) - 1) == lane) {      // one lane per distinct label
                uint32_t cc = __popc(peers), slot = (h * 2654435761u) >> 26;   // 6 bits
                for (uint32_t tries = 0;; ++tries) {
                    if (tries == VW_SLOTS) { overflow = true; break; }
                    uint32_t old = atomicCAS(&key[slot], UTB_BAD32, h);
                    if (old == UTB_BAD32 || old == h) { atomicAdd(&cnt[slot], cc); break; }
                    slot = (slot + 1) & (VW_SLOTS - 1);
                }
            }
            __syncwarp();
        }
    }
    }
    if (__any_sync(0xFFFFFFFFu, overflow)) {
        if (lane == 0) gen_list[atomicAdd(gen_count, 1u)] = r;
        return;
    }
    if (n == 0) {
        if (lane == 0) { out->kind = UTB_NONE; out->label = 0; out->cut = 0; out->found = 0; out->uix = 0; out->sl = 0; out->ol = 0; out->_pad = 0; }
        return;
    }
    uint32_t k0 = key[lane], k1 = key[lane + 32];
    uint32_t m0 = __ballot_sync(0xFFFFFFFFu, k0 != UTB_BAD32), m1 = __ballot_sync(0xFFFFFFFFu, k1 != UTB_BAD32);
    uint32_t uix = __popc(m0) + __popc(m1);
    if (lane == 0) atomicAdd(counters + 2 * COUNTER_SLOTS + (blockIdx.x & (COUNTER_SLOTS - 1)), 1ull);   // good finds (itree.c:1029)
    if (uix == 1) {                                                // itree.c:1031-1032, 1039-1040
        uint32_t lab = m0 ? __shfl_sync(0xFFFFFFFFu, k0, __ffs(m0) - 1) : __shfl_sync(0xFFFFFFFFu, k1, __ffs(m1) - 1);
        if (lane == 0) { out->kind = UTB_STAR; out->label = lab; out->cut = 0; out->found = n; out->uix = 1; out->sl = 0; out->ol = 0; out->_pad = 0; }
        return;
    }
    // sort the entries by label rank (strcmp order, itree.c:1041): compact the occupied slots first -- a read
    // typically holds 2-3 labels, so ranking costs uix compares per entry instead of a sweep over all 64 slots
    uint32_t *rk = sm.rk, *T_lab = sm.lab, *T_cnt = sm.tc;
    const uint32_t r0 = k0 != UTB_BAD32 ? __ldg(db.rank + k0) : UTB_BAD32;
    const uint32_t r1 = k1 != UTB_BAD32 ? __ldg(db.rank + k1) : UTB_BAD32;
    const uint32_t lt = (1u << lane) - 1u;
    const uint32_t i0 = __popc(m0 & lt), i1 = __popc(m0) + __popc(m1 & lt);
    if (k0 != UTB_BAD32) rk[i0] = r0;
    if (k1 != UTB_BAD32) rk[i1] = r1;
    __syncwarp();
    uint32_t p0 = 0, p1 = 0;
    for (uint32_t j = 0; j < uix; ++j) { const uint32_t x = rk[j]; p0 += x < r0; p1 += x < r1; }
    if (k0 != UTB_BAD32) { T_lab[p0] = k0; T_cnt[p0] = cnt[lane]; }
    if (k1 != UTB_BAD32) { T_lab[p1] = k1; T_cnt[p1] = cnt[lane + 32]; }
    __syncwarp();
    walk_warp(db, T_lab, T_cnt, uix, n, out);
}
// Persistent over `list` (reads deferred by vote_thread_kernel), or over all reads when list is null.
__global__ void __launch_bounds__(VW_WARPS * 32)
vote_warp_kernel(DevDB db, VoteIn in, uint32_t n_reads, const uint32_t *__restrict__ dims, const uint32_t *__restrict__ list, const uint32_t *__restrict__ list_count,
                 utb_result *__restrict__ results, uint32_t *__restrict__ gen_list, uint32_t *__restrict__ gen_count,
                 unsigned long long *__restrict__ counters) {
    __shared__ uint32_t s_key[VW_WARPS][VW_SLOTS], s_cnt[VW_WARPS][VW_SLOTS];
    __shared__ uint32_t s_rk[VW_WARPS][VW_SLOTS], s_lab[VW_WARPS][VW_SLOTS], s_tc[VW_WARPS][VW_SLOTS];
    const uint32_t wib = threadIdx.x >> 5;
    const VoteWarpSmem sm = {s_key[wib], s_cnt[wib], s_rk[wib], s_lab[wib], s_tc[wib]};
    if (dims) n_reads = dims[0];
    const uint32_t total = list ? *list_count : n_reads;
    for (uint32_t i = blockIdx.x * VW_WARPS + wib; i < total; i += gridDim.x * VW_WARPS) {
        vote_warp_read(db, in, list ? list[i] : i, results, gen_list, gen_count, counters, sm);
        __syncwarp();
    }
}

// ---- thread per read (the common case) ----------------------------------------------
// A 150-base read holds a handful of hits on 1-3 distinct labels; a warp per read spends ~800 issue
// slots on it, almost all of them with one useful lane (the aufbau walk compares two label strings
// character by character).  Here every lane walks its own read: the read's hit list (one or two
// sectors, written back to back by the survivor kernel) -> (label, count) pairs kept in registers,
// sorted by label rank -> the same walk as walk_warp, scalar.  Reads with more than VT_K distinct
// labels or more than VT_MAXHITS entries are deferred to vote_warp_kernel through `list`.
#define VT_K 6u
#define VT_THREADS 128
#define VT_MAXHITS 512u
__device__ __forceinline__ void walk_thread(const DevDB &db, const uint32_t *T_lab, const uint32_t *T_cnt,   // [k * VT_THREADS]
                                            uint32_t uix, uint32_t n, utb_result *out) {
#define TL(z) T_lab[(z) * VT_THREADS]
#define TC(z) T_cnt[(z) * VT_THREADS]
    const uint32_t EMPTY = 0xFFFFFFFFu;
    uint32_t cutoff = cutoff_of(n), st = 0, ed = uix, dv = EMPTY, orun = n, sl = 0, ol = 0;
    for (;;) {                                                      // itree.c:1047
        uint32_t run = TC(st), td = dv;
        for (uint32_t z = st + 1; z < ed; ++z) {                    // itree.c:1050
            const char *s1 = db.blob + __ldg(db.off + TL(z - 1));
            const char *s2 = db.blob + __ldg(db.off + TL(z));
            if (!s1[dv + (dv == EMPTY)]) {                          // itree.c:1052
                run = TC(z); st = z;
                orun -= TC(z - 1);
                cutoff = cutoff_of(orun);
                continue;
            }
            // itree.c:1060-1061: first td >= dv+1 with s1[td]==0 || s1[td]!=s2[td] || s1[td]==';'
            char a, b;
            td = scan_token(s1, s2, dv + 1u, a, b);
            if (a == b) run += TC(z);                               // itree.c:1062
            else if ((!a && b == ';') ||
                     ((a == ';' || !a) && td > 0 && s1[td - 1] == '_')) {   // itree.c:1063
                run = TC(z); st = z;
                orun -= TC(z - 1);
                cutoff = cutoff_of(orun);
            }
            else if (run >= cutoff) { ed = z; break; }              // itree.c:1068
            else { run = TC(z); st = z; }                           // itree.c:1069
        }
        sl = run; ol = orun;                                        // itree.c:1071
        if (run < cutoff) break;                                    // itree.c:1072
        if (st + 1 >= ed) {                                         // itree.c:1073-1080
            if (TC(ed - 1) >= cutoff) dv = 0xFFFFFFFEu;
            break;
        }
        orun = run; dv = td; cutoff = cutoff_of(run);               // itree.c:1082-1085
    }
    out->kind = UTB_WALK; out->label = TL(ed - 1); out->cut = dv;
    out->found = n; out->uix = uix; out->sl = sl; out->ol = ol; out->_pad = 0;
#undef TL
#undef TC
}
__global__ void __launch_bounds__(VT_THREADS)
vote_thread_kernel(DevDB db, VoteIn in, uint32_t n_reads, const uint32_t *__restrict__ dims, utb_result *__restrict__ results,
                   uint32_t *__restrict__ list, uint32_t *__restrict__ list_count, unsigned long long *__restrict__ counters) {
    if (dims) n_reads = dims[0];
    __shared__ uint32_t s_lab[VT_K * VT_THREADS], s_cnt[VT_K * VT_THREADS];
    __shared__ uint32_t s_good;
    const uint32_t tid = threadIdx.x;
    uint32_t good = 0;
    if (tid == 0) s_good = 0;
    __syncthreads();
    for (uint64_t base = (uint64_t)blockIdx.x * VT_THREADS; base < n_reads; base += (uint64_t)gridDim.x * VT_THREADS) {
        const uint32_t r = (uint32_t)base + tid;                   // the shared rows are private to a thread: no barrier between rounds
        if (r >= n_reads) break;
        uint64_t start, count;
        vote_range(in, r, start, count);
        bool defer = count > VT_MAXHITS;
        uint32_t lab[VT_K], cnt[VT_K], n = 0, uix = 0;
#pragma unroll
        for (uint32_t k = 0; k < VT_K; ++k) { lab[k] = UTB_BAD32; cnt[k] = 0; }
        if (!defer) {
            const uint32_t *hp = in.hits + start;
            for (uint32_t i = 0; i < (uint32_t)count; ++i) {
                const uint32_t h = __ldg(hp + i);
                if (h >= db.max_ix) continue;
                ++n;
                bool seen = false;
#pragma unroll
                for (uint32_t k = 0; k < VT_K; ++k) if (lab[k] == h) { ++cnt[k]; seen = true; }
                if (!seen) {
                    if (uix == VT_K) { defer = true; break; }
#pragma unroll
                    for (uint32_t k = 0; k < VT_K; ++k) if (k == uix) { lab[k] = h; cnt[k] = 1; }
                    ++uix;
                }
            }
        }
        utb_result *out = results + r;
        if (defer) list[atomicAdd(list_count, 1u)] = r;
        else if (n == 0) { out->kind = UTB_NONE; out->label = 0; out->cut = 0; out->found = 0; out->uix = 0; out->sl = 0; out->ol = 0; out->_pad = 0; }
        else {
            ++good;                                                 // good finds (itree.c:1029)
            if (uix == 1) {                                         // itree.c:1031-1032, 1039-1040
                out->kind = UTB_STAR; out->label = lab[0]; out->cut = 0; out->found = n; out->uix = 1; out->sl = 0; out->ol = 0; out->_pad = 0;
            } else {
                // sort by label rank (strcmp order, itree.c:1041): insertion sort over at most VT_K entries
                uint32_t rk[VT_K];
#pragma unroll
                for (uint32_t k = 0; k < VT_K; ++k) rk[k] = k < uix ? __ldg(db.rank + lab[k]) : UTB_BAD32;
#pragma unroll
                for (uint32_t i = 1; i < VT_K; ++i)
#pragma unroll
                    for (uint32_t j = i; j > 0; --j)
                        if (rk[j] < rk[j - 1]) {
                            uint32_t t = rk[j]; rk[j] = rk[j - 1]; rk[j - 1] = t;
                            t = lab[j]; lab[j] = lab[j - 1]; lab[j - 1] = t;
                            t = cnt[j]; cnt[j] = cnt[j - 1]; cnt[j - 1] = t;
                        }
#pragma unroll
                for (uint32_t k = 0; k < VT_K; ++k) { s_lab[k * VT_THREADS + tid] = lab[k]; s_cnt[k * VT_THREADS + tid] = cnt[k]; }
                walk_thread(db, s_lab + tid, s_cnt + tid, uix, n, out);
            }
        }
    }
    for (int o = 16; o; o >>= 1) good += __shfl_xor_sync(0xFFFFFFFFu, good, o);
    if ((tid & 31u) == 0 && good) atomicAdd(&s_good, good);
    __syncthreads();
    if (tid == 0 && s_good) atomicAdd(counters + 2 * COUNTER_SLOTS + (blockIdx.x & (COUNTER_SLOTS - 1)), (unsigned long long)s_good);
}

// ---- long queries and label-rich reads ---------------------------------------------------
// Reads the warp kernel defers (more than VW_MAXHITS entries or more than VW_SLOTS distinct
// labels) are voted from a dense per-label histogram in global memory; the labels a read touches
// are appended to a list the moment their count leaves zero, so what follows costs O(touched
// labels), not O(max_ix): the list is sorted by label rank in shared memory (itree.c:1041), the
// counts are gathered and the scratch is left clean, then the same walk runs.
//   vote_block_kernel   one CTA per read, CTA-private scratch; reads with more than `split_slots`
//                       entries (north_star: "long and whole-genome queries split across
//                       blocks and merged") are handed on to
//   vote_big_count_kernel  the hit list of every such read is cut into chunks of 32 * VBIG_CHUNK_WORDS
//                       entries which the whole grid accumulates into that read's histogram, and
//   vote_big_finish_kernel one CTA per read merges: sort, gather, walk.
#define VB_THREADS 256
#define VB_PER_SM 4
#define VB_SORT_MAX 2048u           // touched labels sorted in shared memory; beyond: sweep over all labels in rank order
#define VBIG_CHUNK_WORDS 2048u      // x 32 = 65,536 entries of a read's hits a CTA accumulates at a time
#define VBIG_POOL_MAX 2048u         // split reads a batch can hold scratch for
#define VL_CACHE 64u                // per-CTA (label, count) pairs gathered in shared memory before they go to the histogram
struct VoteLong {
    uint32_t *hist, *tlab, *tcnt;                       // [CTAs of vote_block_kernel][max_ix]
    uint32_t *big_hist, *big_tlab, *big_tcnt;           // [pool][max_ix]
    uint32_t *big_list;                                 // [pool] read index
    uint32_t *big_state;                                // [0] split reads of the batch, then per read: touched labels, hits
    uint32_t *work;                                     // [0] next entry of the deferral list a CTA of vote_block_kernel takes
    uint32_t pool;
    uint32_t sort_max;                                  // <= VB_SORT_MAX (tests lower it to reach the sweep)
    unsigned long long split_slots;
};
// A read hits few distinct labels (its own lineage), thousands of times: the hits are gathered in a small
// shared-memory table first (CAS on the key, add on the count) and only its entries go to the global
// histogram -- a dependent global atomic per hit was what bound this kernel (profiles/r02_*: 24.6 ms of a
// 59 ms LONG step).  A label that finds no room in its four probes goes to the histogram directly.
struct VlCache { uint32_t key[VL_CACHE]; uint32_t cnt[VL_CACHE]; };
__device__ __forceinline__ void vl_cache_clear(VlCache &c) {
    for (uint32_t i = threadIdx.x; i < VL_CACHE; i += blockDim.x) { c.key[i] = UTB_BAD32; c.cnt[i] = 0; }
}
__device__ __forceinline__ void vl_add(VlCache &c, uint32_t h, uint32_t k, uint32_t *__restrict__ hist, uint32_t *__restrict__ tlab, uint32_t *nt) {
    uint32_t s = (h * 2654435761u) >> 26;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const uint32_t old = atomicCAS(&c.key[s], UTB_BAD32, h);
        if (old == UTB_BAD32 || old == h) { atomicAdd(&c.cnt[s], k); return; }
        s = (s + 1u) & (VL_CACHE - 1u);
    }
    if (atomicAdd(&hist[h], k) == 0u) tlab[atomicAdd(nt, 1u)] = h;
}
// block-wide, between two barriers: the table's entries into the histogram; labels met for the first time are
// appended to tlab through *nt
__device__ __forceinline__ void vl_flush(VlCache &c, uint32_t *__restrict__ hist, uint32_t *__restrict__ tlab, uint32_t *nt) {
    for (uint32_t i = threadIdx.x; i < VL_CACHE; i += blockDim.x) {
        const uint32_t h = c.key[i], k = c.cnt[i];
        if (h != UTB_BAD32 && k && atomicAdd(&hist[h], k) == 0u) tlab[atomicAdd(nt, 1u)] = h;
        c.key[i] = UTB_BAD32; c.cnt[i] = 0;
    }
}
// Adds the labels of entries [32 * w0, 32 * w1) of one read's hits through the table.  Block-wide call; returns this
// thread's hits.  The caller flushes.
__device__ __forceinline__ uint32_t vl_accumulate(const DevDB &db, const VoteIn &in, uint64_t start, uint64_t count, uint64_t w0, uint64_t w1,
                                                  VlCache &cache, uint32_t *__restrict__ hist, uint32_t *__restrict__ tlab, uint32_t *nt) {
    const uint32_t tid = threadIdx.x, lane = tid & 31u;
    uint32_t n_local = 0;
    const uint64_t lo = w0 * 32u, hi = w1 * 32u < count ? w1 * 32u : count;
    for (uint64_t base = lo; base < hi; base += VB_THREADS) {
        const uint64_t i = base + tid;
        const uint32_t h = i < hi ? __ldg(in.hits + start + i) : HIT_NOWIN;
        const bool ok = h < db.max_ix;
        const uint32_t peers = __match_any_sync(0xFFFFFFFFu, h);   // a long read names its own lineage over and over: one add per distinct label of the warp
        if (ok && (uint32_t)(__ffs(peers) - 1) == lane) vl_add(cache, h, (uint32_t)__popc(peers), hist, tlab, nt);
        n_local += ok;
    }
    return n_local;
}
struct VlSmem { unsigned long long key[VB_SORT_MAX]; uint32_t warp[VB_THREADS / 32]; uint32_t base; };
// The walk compares neighbouring label strings level by level: a chain of dependent loads (label id -> offset ->
// characters) per comparison, ~2 us each from global memory with one warp at work -- 250 us for a read that touched a
// hundred labels, which is what the long-query vote spent its time on.  So the whole CTA first stages ids, counts
// and strings in shared memory (the sort keys' space is free by then), and the walk runs on that copy.
#define VL_STAGE_MAX 512u           // labels
#define VL_STR_BYTES 24576u         // their strings, NULs included
struct VlStage { uint32_t off[VL_STAGE_MAX + 1], lab[VL_STAGE_MAX], cnt[VL_STAGE_MAX]; };
static_assert(sizeof(VlStage) <= sizeof(unsigned long long) * VB_SORT_MAX, "VlStage lives in VlSmem::key");
// The walk over the staged copy, one warp, 32 neighbour pairs at a time.  What the reference decides for a pair
// (z-1, z) at a level -- the first string ended (K), same token (S), a new run that also shrinks the outer run (O),
// different token (D) -- depends only on the two strings and the level's depth dv, so every lane classifies its own
// pair (a short scalar scan over one token); the sequential state of itree.c:1050-1070 then is a segmented sum of the
// counts (a new segment wherever the class is not S), a prefix sum of what K / O pairs take off the outer run, and
// the walk stops at the first D pair whose run so far reaches the cutoff of the outer run so far.  Same results as
// walk_warp, about a tenth of its instructions for a read that touched hundreds of labels.
__device__ void walk_warp_staged(const VlStage *sg, const char *str, uint32_t uix, uint32_t n, utb_result *out) {
    const uint32_t lane = threadIdx.x & 31u, FULL = 0xFFFFFFFFu, EMPTY = 0xFFFFFFFFu;
    enum { CLS_S = 0, CLS_K = 1, CLS_O = 2, CLS_D = 3 };
    const uint32_t *T_cnt = sg->cnt, *S_off = sg->off;
    uint32_t st = 0, ed = uix, dv = EMPTY, orun = n, sl = 0, ol = 0, cutoff;
    for (;;) {                                                      // itree.c:1047
        uint32_t run = T_cnt[st], td = dv;
        const uint32_t ed0 = ed;
        for (uint32_t zb = st + 1; zb < ed0; zb += 32u) {           // itree.c:1050
            const uint32_t z = zb + lane;
            const bool valid = z < ed0;
            uint32_t cls = CLS_S, tdz = 0, cz = 0, cprev = 0;
            if (valid) {
                cz = T_cnt[z]; cprev = T_cnt[z - 1];
                const char *s1 = str + S_off[z - 1], *s2 = str + S_off[z];
                if (!s1[dv + (dv == EMPTY)]) cls = CLS_K;           // itree.c:1052
                else {
                    char a, b;
                    const uint32_t t = scan_token(s1, s2, dv + 1u, a, b);   // itree.c:1060-1061
                    tdz = t;
                    if (a == b) cls = CLS_S;                        // itree.c:1062
                    else if ((!a && b == ';') || ((a == ';' || !a) && t > 0 && s1[t - 1] == '_')) cls = CLS_O;   // itree.c:1063
                    else cls = CLS_D;                               // itree.c:1068-1069
                }
            }
            const uint32_t hm = __ballot_sync(FULL, valid && cls != CLS_S);          // pairs that start a new run
            const uint32_t nk = __ballot_sync(FULL, valid && cls != CLS_K);          // pairs that set td
            uint32_t pv = cz, ps = (cls == CLS_K || cls == CLS_O) ? cprev : 0u;      // inclusive prefix sums over the lanes
#pragma unroll
            for (uint32_t o = 1; o < 32u; o <<= 1) {
                const uint32_t t1 = __shfl_up_sync(FULL, pv, o), t2 = __shfl_up_sync(FULL, ps, o);
                if (lane >= o) { pv += t1; ps += t2; }
            }
            const uint32_t lower = hm & (0xFFFFFFFFu >> (31u - lane));               // run starts at lanes <= this one
            const int hs = lower ? 31 - __clz(lower) : -1;
            const uint32_t before_hs = __shfl_sync(FULL, pv - cz, hs < 0 ? 0 : hs);
            const uint32_t run_z = hs < 0 ? run + pv : pv - before_hs;               // run / outer run after pair z
            const uint32_t orun_z = orun - ps;
            uint32_t run_b = __shfl_up_sync(FULL, run_z, 1), orun_b = __shfl_up_sync(FULL, orun_z, 1);   // ... and before it
            if (lane == 0) { run_b = run; orun_b = orun; }
            const uint32_t bm = __ballot_sync(FULL, valid && cls == CLS_D && run_b >= cutoff_of(orun_b));
            if (bm) {                                               // itree.c:1068: the run ends before pair zb + L
                const uint32_t L = (uint32_t)__ffs(bm) - 1u;
                ed = zb + L;
                run = __shfl_sync(FULL, run_b, L); orun = __shfl_sync(FULL, orun_b, L);
                const uint32_t hb = hm & ((1u << L) - 1u);
                if (hb) st = zb + (31u - (uint32_t)__clz(hb));
                td = __shfl_sync(FULL, tdz, L);
                break;
            }
            run = __shfl_sync(FULL, run_z, 31); orun = __shfl_sync(FULL, orun_z, 31);
            if (hm) st = zb + (31u - (uint32_t)__clz(hm));
            if (nk) td = __shfl_sync(FULL, tdz, 31 - __clz(nk));
        }
        cutoff = cutoff_of(orun);                                   // the cutoff always is that of the outer run (itree.c:1044-1046, 1055, 1066, 1085)
        sl = run; ol = orun;                                        // itree.c:1071
        if (run < cutoff) break;                                    // itree.c:1072
        if (st + 1 >= ed) {                                         // itree.c:1073-1080
            if (T_cnt[ed - 1] >= cutoff) dv = 0xFFFFFFFEu;
            break;
        }
        orun = run; dv = td;                                        // itree.c:1082-1085
    }
    if (lane == 0) {
        out->kind = UTB_WALK; out->label = sg->lab[ed - 1]; out->cut = dv;
        out->found = n; out->uix = uix; out->sl = sl; out->ol = ol; out->_pad = 0;
    }
}
// block-wide; false (block-uniform): too many labels or bytes, walk from global memory
__device__ bool vl_stage(const DevDB &db, const uint32_t *tlab, const uint32_t *tcnt, uint32_t uix, VlSmem &sm, char *str) {
    if (uix > VL_STAGE_MAX) return false;
    VlStage *sg = reinterpret_cast<VlStage *>(sm.key);
    const uint32_t tid = threadIdx.x, lane = tid & 31u, wid = tid >> 5;
    for (uint32_t i = tid; i < uix; i += VB_THREADS) { sg->lab[i] = tlab[i]; sg->cnt[i] = tcnt[i]; }
    for (uint32_t i = wid; i < uix; i += VB_THREADS / 32) {        // lengths, NUL included: a warp per label
        const char *p = db.blob + __ldg(db.off + tlab[i]);
        uint32_t t0 = 0, len;
        for (;;) {
            const uint32_t m = __ballot_sync(0xFFFFFFFFu, p[t0 + lane] == 0);   // the blob is padded: reading on past the NUL is fine
            if (m) { len = t0 + (uint32_t)__ffs(m); break; }
            t0 += 32u;
        }
        if (lane == 0) sg->off[i + 1] = (len + 7u) & ~7u;          // staged like the blob: multiples of 8, NUL-padded
    }
    __syncthreads();
    if (wid == 0) {                                                // lengths -> offsets
        uint32_t carry = 0;
        for (uint32_t base = 0; base < uix; base += 32u) {
            const uint32_t i = base + lane;
            uint32_t v = i < uix ? sg->off[i + 1] : 0u;
            for (uint32_t o = 1; o < 32u; o <<= 1) { const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, v, o); if (lane >= o) v += t; }
            if (i < uix) sg->off[i + 1] = carry + v;
            carry += __shfl_sync(0xFFFFFFFFu, v, 31);
        }
        if (lane == 0) { sg->off[0] = 0; sm.base = carry; }
    }
    __syncthreads();
    if (sm.base + 32u > VL_STR_BYTES) return false;                // the walk reads up to 31 bytes past a NUL
    for (uint32_t i = wid; i < uix; i += VB_THREADS / 32) {
        const char *p = db.blob + __ldg(db.off + sg->lab[i]);
        const uint32_t a = sg->off[i], len = sg->off[i + 1] - a;       // the blob's own padding comes along
        for (uint32_t j = lane; j < len; j += 32u) str[a + j] = p[j];
    }
    __syncthreads();
    return true;
}
// hist holds the label counts of one read, tlab[0 .. nt) the labels touched (any order), n the hits.  Block-wide.
__device__ void vl_finish(const DevDB &db, uint32_t *hist, uint32_t *tlab, uint32_t *tcnt, uint32_t nt, uint32_t n, uint32_t sort_max,
                          utb_result *out, unsigned long long *__restrict__ counters, VlSmem &sm, char *str) {
    const uint32_t tid = threadIdx.x, lane = tid & 31u, wid = tid >> 5;
    if (n == 0) {                                                  // block-uniform
        if (tid == 0) { out->kind = UTB_NONE; out->label = 0; out->cut = 0; out->found = 0; out->uix = 0; out->sl = 0; out->ol = 0; out->_pad = 0; }
        return;
    }
    __threadfence();
    __syncthreads();
    uint32_t uix;
    if (nt <= sort_max) {
        // sort the touched labels by rank (strcmp order, itree.c:1041): bitonic network over rank << 32 | label
        uint32_t np2 = 2;
        while (np2 < nt) np2 <<= 1;
        for (uint32_t i = tid; i < np2; i += VB_THREADS) {
            unsigned long long k = ~0ull;
            if (i < nt) { const uint32_t lab = __ldcg(tlab + i); k = ((unsigned long long)__ldg(db.rank + lab) << 32) | lab; }
            sm.key[i] = k;
        }
        __syncthreads();
        for (uint32_t k2 = 2; k2 <= np2; k2 <<= 1)
            for (uint32_t j = k2 >> 1; j; j >>= 1) {
                for (uint32_t i = tid; i < np2; i += VB_THREADS) {
                    const uint32_t l = i ^ j;
                    if (l > i) {
                        const unsigned long long a = sm.key[i], c = sm.key[l];
                        const bool up = (i & k2) == 0;
                        if ((a > c) == up) { sm.key[i] = c; sm.key[l] = a; }
                    }
                }
                __syncthreads();
            }
        for (uint32_t i = tid; i < nt; i += VB_THREADS) {
            const uint32_t lab = (uint32_t)sm.key[i];
            tlab[i] = lab; tcnt[i] = __ldcg(hist + lab);          // L2 view: the counts were made by atomics
            hist[lab] = 0;                                         // leave the scratch clean
        }
        uix = nt;
    } else {
        // very many labels: compaction of the whole label space in rank order (itree.c:1036-1041 produce exactly this list)
        if (tid == 0) sm.base = 0;
        __syncthreads();
        for (uint32_t r0 = 0; r0 < db.max_ix; r0 += VB_THREADS) {
            const uint32_t rr = r0 + tid;
            const uint32_t lab = rr < db.max_ix ? __ldg(db.by_rank + rr) : 0;
            const uint32_t c = rr < db.max_ix ? __ldcg(hist + lab) : 0;
            const uint32_t bal = __ballot_sync(0xFFFFFFFFu, c != 0);
            if (lane == 0) sm.warp[wid] = __popc(bal);
            __syncthreads();
            uint32_t wbase = sm.base;
            for (uint32_t w = 0; w < wid; ++w) wbase += sm.warp[w];
            if (c) {
                const uint32_t p = wbase + __popc(bal & ((1u << lane) - 1u));
                tlab[p] = lab; tcnt[p] = c;
                hist[lab] = 0;
            }
            __syncthreads();
            if (tid == 0) { uint32_t t = 0; for (uint32_t w = 0; w < VB_THREADS / 32; ++w) t += sm.warp[w]; sm.base += t; }
            __syncthreads();
        }
        uix = sm.base;
    }
    __threadfence();
    __syncthreads();
    const bool staged = uix > 1 && vl_stage(db, tlab, tcnt, uix, sm, str);
    if (wid == 0) {
        if (lane == 0) atomicAdd(counters + 2 * COUNTER_SLOTS + (blockIdx.x & (COUNTER_SLOTS - 1)), 1ull);   // good finds (itree.c:1029)
        if (uix == 1) {                                            // itree.c:1031-1032, 1039-1040
            if (lane == 0) { out->kind = UTB_STAR; out->label = tlab[0]; out->cut = 0; out->found = n; out->uix = 1; out->sl = 0; out->ol = 0; out->_pad = 0; }
        } else if (staged) {
            walk_warp_staged(reinterpret_cast<const VlStage *>(sm.key), str, uix, n, out);
        } else walk_warp(db, tlab, tcnt, uix, n, out);
    }
    __syncthreads();
}
__global__ void __launch_bounds__(VB_THREADS)
vote_block_kernel(DevDB db, VoteIn in, utb_result *__restrict__ results,
                  const uint32_t *__restrict__ gen_list, const uint32_t *__restrict__ gen_count,
                  VoteLong vl, unsigned long long *__restrict__ counters) {
    __shared__ VlSmem sm;
    __shared__ VlCache cache;
    __shared__ __align__(8) char str[VL_STR_BYTES];
    __shared__ uint32_t s_nt, s_n, s_big, s_qi;
    const uint32_t tid = threadIdx.x, lane = tid & 31u;
    uint32_t *hist = vl.hist + (size_t)blockIdx.x * db.max_ix;
    uint32_t *tlab = vl.tlab + (size_t)blockIdx.x * db.max_ix;
    uint32_t *tcnt = vl.tcnt + (size_t)blockIdx.x * db.max_ix;
    const uint32_t total = *gen_count;
    vl_cache_clear(cache);
    for (;;) {                                                     // reads differ a hundredfold in length: whoever is free takes the next one
        __syncthreads();
        if (tid == 0) s_qi = atomicAdd(vl.work, 1u);
        __syncthreads();
        const uint32_t qi = s_qi;
        if (qi >= total) break;
        const uint32_t r = gen_list[qi];
        uint64_t start, count;
        vote_range(in, r, start, count);
        if (tid == 0) {
            s_nt = 0; s_n = 0; s_big = 0;
            if (count > vl.split_slots) {                          // split across the grid (scratch permitting)
                const uint32_t bi = atomicAdd(vl.big_state, 1u);
                if (bi < vl.pool) { vl.big_list[bi] = r; s_big = 1; }
            }
        }
        __syncthreads();
        if (s_big) continue;
        uint32_t n_local = vl_accumulate(db, in, start, count, 0, (count + 31) >> 5, cache, hist, tlab, &s_nt);
        for (int o = 16; o; o >>= 1) n_local += __shfl_xor_sync(0xFFFFFFFFu, n_local, o);
        if (lane == 0 && n_local) atomicAdd(&s_n, n_local);
        __syncthreads();
        vl_flush(cache, hist, tlab, &s_nt);
        __syncthreads();
        vl_finish(db, hist, tlab, tcnt, s_nt, s_n, vl.sort_max, results + r, counters, sm, str);
    }
}
__global__ void __launch_bounds__(VB_THREADS)
vote_big_count_kernel(DevDB db, VoteIn in, VoteLong vl) {
    __shared__ VlCache cache;
    const uint32_t n_big = min(*vl.big_state, vl.pool), lane = threadIdx.x & 31u;
    vl_cache_clear(cache);
    __syncthreads();
    for (uint32_t bi = 0; bi < n_big; ++bi) {
        uint64_t start, count;
        vote_range(in, vl.big_list[bi], start, count);
        const uint64_t n_words = (count + 31) >> 5, n_chunks = (n_words + VBIG_CHUNK_WORDS - 1) / VBIG_CHUNK_WORDS;
        uint32_t *hist = vl.big_hist + (size_t)bi * db.max_ix, *tlab = vl.big_tlab + (size_t)bi * db.max_ix;
        uint32_t n_local = 0;
        bool any = false;
        // the chunks of consecutive reads start at different CTAs, so short tails do not pile up on CTA 0
        for (uint64_t c = (blockIdx.x + gridDim.x - (bi * 61u) % gridDim.x) % gridDim.x; c < n_chunks; c += gridDim.x) {
            const uint64_t w0 = c * VBIG_CHUNK_WORDS, w1 = w0 + VBIG_CHUNK_WORDS < n_words ? w0 + VBIG_CHUNK_WORDS : n_words;
            n_local += vl_accumulate(db, in, start, count, w0, w1, cache, hist, tlab, vl.big_state + 1 + 2 * bi);
            any = true;
        }
        if (any) {                                                 // block-uniform: the chunk loop's bounds are
            __syncthreads();
            vl_flush(cache, hist, tlab, vl.big_state + 1 + 2 * bi);
            __syncthreads();
        }
        for (int o = 16; o; o >>= 1) n_local += __shfl_xor_sync(0xFFFFFFFFu, n_local, o);
        if (lane == 0 && n_local) atomicAdd(vl.big_state + 2 + 2 * bi, n_local);
    }
}
__global__ void __launch_bounds__(VB_THREADS)
vote_big_finish_kernel(DevDB db, VoteLong vl, utb_result *__restrict__ results, unsigned long long *__restrict__ counters) {
    __shared__ VlSmem sm;
    __shared__ __align__(8) char str[VL_STR_BYTES];
    const uint32_t n_big = min(*vl.big_state, vl.pool);
    for (uint32_t bi = blockIdx.x; bi < n_big; bi += gridDim.x)
        vl_finish(db, vl.big_hist + (size_t)bi * db.max_ix, vl.big_tlab + (size_t)bi * db.max_ix, vl.big_tcnt + (size_t)bi * db.max_ix,
                  vl.big_state[1 + 2 * bi], vl.big_state[2 + 2 * bi], vl.sort_max, results + vl.big_list[bi], counters, sm, str);
}

// ---------------------------------------------------------------------------
// the non-GG binary (-D SEARCH): the ids its slide collects (itree.c:903-933 with XT_SHALLOWVOTE, :948-951)
// ---------------------------------------------------------------------------
// After a hit the reference's loop index jumps PACKSIZE / SPARSITY - 1 = 7 windows ahead -- and its rolling
// word does not follow: `w <<= (i-z-1) << 1` (itree.c:920) shifts by 7 bases on top of the 8 per-base shifts
// of the inner loop, so the word looked up at z + 8 is the last 17 bases before the hit, seven A's, and the 8
// new bases; the stray A's stay in the word for 24 more windows.  What is looked up after a hit at window end
// z is therefore: 24 CORRUPTED words at z + 8 .. z + 31 (each can hit by accident, which corrupts the word
// again), then the true windows from z + 32 on; an ambiguous base (and the 'N' between the read and its
// reverse complement, itree.c:892) restarts with a clean word.  A lookup is a pure function of its word, so
// the true windows are taken from the hit map the GG path fills anyway (every window was looked up), and only
// the corrupted stretches are emulated word by word with direct lookups.  One thread per read walks the two
// halves of the text in order: forward windows left to right, then the windows of the reverse-complement
// text, i.e. the reverse-strand slots right to left.  The ids land in the read's own stretch of a gapped
// buffer (a kept hit uses up >= 8 text positions, so a quarter of the read's slots is room enough);
// shallow_compact_kernel packs them.
struct ShallowRead {
    const uint64_t *pk; const uint32_t *bad;                       // packed stream
    uint64_t pos0;                                                  // first position of the read in it
    uint32_t L, nwin, nstr;
    uint64_t start;                                                 // first lookup slot of the read
};
// base at text position t of half `strand` (strand 1: the reverse-complement text); false: not ACGT
__device__ __forceinline__ bool sh_base(const ShallowRead &R, uint32_t strand, uint32_t t, uint32_t &c) {
    const uint64_t pos = R.pos0 + (strand ? R.L - 1u - t : t);
    const uint64_t g = pos >> 5; const uint32_t o = (uint32_t)pos & 31u;
    if ((R.bad[g] >> o) & 1u) return false;
    c = (uint32_t)(R.pk[g] >> (62u - 2u * o)) & 3u;
    if (strand) c = 3u - c;
    return true;
}
__device__ __forceinline__ uint32_t lookup_any(const DevDB &db, uint64_t w) {
    if (db.ktab) return (db.sieve && !sv_maybe(db, w)) ? HIT_MISS : kt_lookup(db, w);
    Probe q[1];
    probe_begin(db, w, q[0]);
    probe_run<1>(db, q);
    return probe_end(db, q[0]);
}
// first true window of this half, at text index >= from, that hit: its index (nwin if none) and its label
__device__ __forceinline__ uint32_t sh_next_hit(const DevDB &db, const VoteIn &in, const ShallowRead &R, uint32_t strand, uint32_t from, uint32_t &label) {
    if (from >= R.nwin) return R.nwin;
    if (in.hitmap) {
        const uint32_t *hm = in.hitmap + (R.start >> 5);            // start is a multiple of 32
        if (!strand) {
            uint64_t slot = (uint64_t)from * R.nstr;
            const uint64_t end = (uint64_t)R.nwin * R.nstr;
            const uint32_t lanes = R.nstr == 2 ? 0x55555555u : 0xFFFFFFFFu;
            for (uint64_t w = slot >> 5; w * 32 < end; ++w) {
                uint32_t m = __ldg(hm + w) & lanes;
                if (w == slot >> 5) m &= 0xFFFFFFFFu << (slot & 31u);
                while (m) {
                    const uint32_t bit = __ffs(m) - 1u; m &= m - 1u;
                    const uint64_t sl = w * 32 + bit;
                    if (sl >= end) return R.nwin;
                    const uint32_t h = __ldg(in.hits + R.start + sl);
                    if (h < db.max_ix) { label = h; return (uint32_t)(sl / R.nstr); }
                }
            }
            return R.nwin;
        }
        // reverse-complement text: window q of it is the reverse-strand slot of forward position nwin - 1 - q
        int64_t slot = (int64_t)(R.nwin - 1u - from) * 2 + 1;
        for (int64_t w = slot >> 5; w >= 0; --w) {
            uint32_t m = __ldg(hm + w) & 0xAAAAAAAAu;
            if (w == slot >> 5 && (slot & 31) != 31) m &= (1u << ((slot & 31) + 1)) - 1u;
            while (m) {
                const uint32_t bit = 31u - __clz(m); m &= ~(1u << bit);
                const uint64_t sl = (uint64_t)w * 32 + bit;
                const uint32_t h = __ldg(in.hits + R.start + sl);
                if (h < db.max_ix) { label = h; return R.nwin - 1u - (uint32_t)(sl >> 1); }
            }
        }
        return R.nwin;
    }
    for (uint32_t t = from; t < R.nwin; ++t) {                      // dense hit slots (sieve off / probe sequence)
        const uint32_t pos = strand ? R.nwin - 1u - t : t;
        const uint32_t h = __ldg(in.hits + R.start + (uint64_t)pos * R.nstr + strand);
        if (h < db.max_ix) { label = h; return t; }
    }
    return R.nwin;
}
__global__ void __launch_bounds__(128)
shallow_select_kernel(DevDB db, VoteIn in, const uint64_t *__restrict__ pk, const uint32_t *__restrict__ bad, uint32_t n_reads,
                      const uint32_t *__restrict__ dims, uint32_t *__restrict__ sel_cnt, uint32_t *__restrict__ sel_gap) {
    if (dims) n_reads = dims[0];
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_reads; r += (uint64_t)gridDim.x * blockDim.x) {
        ShallowRead R;
        uint64_t count;
        vote_range(in, (uint32_t)r, R.start, count);
        R.pk = pk; R.bad = bad; R.nstr = in.nstr;
        R.L = __ldg(in.seq_len + r); R.nwin = R.L >= 32u ? R.L - 31u : 0u;
        R.pos0 = (uint64_t)__ldg(in.grp_off + r) * 32u;
        uint32_t *out = sel_gap + (R.start >> 2);
        uint32_t n = 0;
        for (uint32_t strand = 0; strand < R.nstr && R.nwin; ++strand) {
            uint32_t from = 0;                                      // first true window that may be looked up next
            for (;;) {
                uint32_t lab;
                const uint32_t p = sh_next_hit(db, in, R, strand, from, lab);
                if (p >= R.nwin) break;
                out[n++] = lab;                                     // itree.c:951
                // the true word of that window, then the reference's arithmetic from there on
                uint64_t w = 0;
                {
                    const uint32_t fp = strand ? R.nwin - 1u - p : p;
                    window_at(pk, bad, (uint32_t)(R.pos0 + fp), w);
                    if (strand) w = revcomp_word(w);
                }
                uint32_t z = p + 31u;                               // text index of the hit's last base
                bool half_done = false;
                for (;;) {                                          // one corrupted stretch per round
                    uint32_t i = z + 8u;                            // itree.c:950 + the loop's ++i
                    if (i >= R.L) { half_done = true; break; }      // forward half: the 'N' follows; reverse half / no RC: i < length fails
                    w <<= 14;                                       // itree.c:920 with i - z - 1 = 7
                    bool clean = false;
                    for (uint32_t j = z + 1u; j <= i; ++j) {        // itree.c:922-925
                        uint32_t c;
                        if (!sh_base(R, strand, j, c)) { from = j + 1u; clean = true; break; }   // a clean word restarts after the bad base
                        w = (w << 2) | c;
                    }
                    if (clean) break;
                    bool again = false;
                    for (uint32_t left = 24u;;) {                   // windows z + 8 .. z + 31 carry the stray A's
                        const uint32_t h = lookup_any(db, w);
                        if (h < db.max_ix) { out[n++] = h; z = i; again = true; break; }   // an accidental hit: corrupted again from here
                        if (--left == 0u) { from = i + 1u - 31u; clean = true; break; }    // the next window is a true one
                        ++i;
                        if (i >= R.L) { half_done = true; break; }
                        uint32_t c;
                        if (!sh_base(R, strand, i, c)) { from = i + 1u; clean = true; break; }
                        w = (w << 2) | c;
                    }
                    if (!again) break;
                }
                if (half_done) break;
            }
        }
        sel_cnt[r] = n;
    }
}
// gapped -> packed: one thread per read
__global__ void __launch_bounds__(128)
shallow_compact_kernel(VoteIn in, uint32_t n_reads, const uint32_t *__restrict__ dims, const uint32_t *__restrict__ sel_cnt,
                       const uint32_t *__restrict__ sel_off, const uint32_t *__restrict__ sel_gap, uint32_t *__restrict__ sel) {
    if (dims) n_reads = dims[0];
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_reads; r += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t start, count;
        vote_range(in, (uint32_t)r, start, count);
        const uint32_t *src = sel_gap + (start >> 2);
        uint32_t *dst = sel + sel_off[r];
        for (uint32_t k = 0, n = sel_cnt[r]; k < n; ++k) dst[k] = src[k];
    }
}

// ---------------------------------------------------------------------------
// output text on the device (the fprintf lines of itree.c:1032, 1040, 1096)
// ---------------------------------------------------------------------------
// Formatting on the host would compete with the framer for a handful of cores
// (16 for 8 GPUs on the test box), so the lines are produced here: per-read length,
// exclusive scan, then one warp per read copies name, label prefix and the
// numeric tail.  The host only moves the finished text to the sink.
__device__ __forceinline__ uint32_t dec_digits(uint32_t v) {
    return v < 10u ? 1u : v < 100u ? 2u : v < 1000u ? 3u : v < 10000u ? 4u : v < 100000u ? 5u : v < 1000000u ? 6u :
           v < 10000000u ? 7u : v < 100000000u ? 8u : v < 1000000000u ? 9u : 10u;
}
// strlen of a label: the blob keeps every string at a multiple of 8 bytes, NUL-padded to the next (>= 1 NUL), so the
// length is the string's span minus the NULs at the end of its last 8-byte word
__device__ __forceinline__ uint32_t label_len(const DevDB &db, uint32_t label) {
    const uint32_t a = __ldg(db.off + label), b = __ldg(db.off + label + 1);
    const unsigned long long nz = nz_bytes(*reinterpret_cast<const unsigned long long *>(db.blob + b - 8u));
    return b - a - 8u + (nz ? (uint32_t)(64 - __clzll((long long)nz)) >> 3 : 0u);
}
__device__ __forceinline__ uint32_t tax_len_of(const DevDB &db, const utb_result &v) {
    uint32_t ll = label_len(db, v.label);
    if (v.kind == UTB_WALK) {
        if (v.cut == UTB_CUT_EMPTY) ll = 0;                        // dv == -1 (itree.c:1087)
        else if (v.cut != UTB_CUT_FULL && v.cut < ll) ll = v.cut;  // first dv bytes (itree.c:1088)
    }
    return ll;
}
__global__ void __launch_bounds__(256)
fmt_len_kernel(DevDB db, const utb_result *__restrict__ res, const uint32_t *__restrict__ name_len, uint32_t n_reads,
               const uint32_t *__restrict__ dims, uint32_t *__restrict__ line_len) {
    if (dims) n_reads = dims[0];
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_reads; r += (uint64_t)gridDim.x * blockDim.x) {
        const utb_result v = res[r];
        uint32_t n = 0;
        if (v.kind != UTB_NONE) {
            n = __ldg(name_len + r) + 1u + tax_len_of(db, v) + 1u + dec_digits(v.found) + 1u + dec_digits(v.uix) + 1u;
            n += v.kind == UTB_STAR ? 1u : dec_digits(v.sl) + 1u + dec_digits(v.ol);
            n += 1u;
        }
        line_len[r] = n;
    }
}
// exclusive scan of u32 (n up to 2^31): block sums, scan of the sums by one block, local scan + base.
// MAX: the exclusive max-scan instead (identity 0), in the same three kernels
#define SCAN_TILE 2048u
template <bool MAX> __device__ __forceinline__ uint32_t scan_op(uint32_t a, uint32_t b) { return MAX ? max(a, b) : a + b; }
template <bool MAX>
__global__ void __launch_bounds__(256)
scan_sums_kernel(const uint32_t *__restrict__ in, uint32_t n, const uint32_t *__restrict__ n_dev, uint32_t n_tiles, uint32_t *__restrict__ sums) {
    if (n_dev) n = *n_dev;
    __shared__ uint32_t sh[8];
    for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {   // n_tiles covers the host's upper bound of n: tiles past n sum to 0
        const uint32_t base = t * SCAN_TILE;
        uint32_t acc = 0;
        for (uint32_t i = threadIdx.x; i < SCAN_TILE; i += 256) if (base + i < n) acc = scan_op<MAX>(acc, in[base + i]);
        for (int o = 16; o; o >>= 1) acc = scan_op<MAX>(acc, __shfl_xor_sync(0xFFFFFFFFu, acc, o));
        if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
        __syncthreads();
        if (threadIdx.x == 0) { uint32_t x = 0; for (int w = 0; w < 8; ++w) x = scan_op<MAX>(x, sh[w]); sums[t] = x; }
        __syncthreads();
    }
}
template <bool MAX>
__global__ void __launch_bounds__(1024)
scan_top_kernel(uint32_t *__restrict__ sums, uint32_t nb, uint32_t *__restrict__ total) {
    __shared__ uint32_t sh[1024];
    uint32_t carry = 0;
    for (uint32_t base = 0; base < nb; base += 1024) {
        uint32_t i = base + threadIdx.x, v = i < nb ? sums[i] : 0;
        sh[threadIdx.x] = v;
        __syncthreads();
        for (uint32_t o = 1; o < 1024; o <<= 1) {
            uint32_t t = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
            __syncthreads();
            sh[threadIdx.x] = scan_op<MAX>(sh[threadIdx.x], t);
            __syncthreads();
        }
        if (MAX) { if (i < nb) sums[i] = max(carry, threadIdx.x ? sh[threadIdx.x - 1] : 0u); carry = max(carry, sh[1023]); }
        else {
            if (i < nb) sums[i] = carry + sh[threadIdx.x] - v;       // exclusive
            carry += sh[1023];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}
template <bool MAX>
__global__ void __launch_bounds__(256)
scan_apply_kernel(const uint32_t *__restrict__ in, uint32_t n, const uint32_t *__restrict__ n_dev, uint32_t n_tiles,
                  const uint32_t *__restrict__ sums, uint32_t *__restrict__ out) {
    if (n_dev) n = *n_dev;
    __shared__ uint32_t sh[8];
    __shared__ uint32_t run;
    for (uint32_t t = blockIdx.x; t < n_tiles && t * SCAN_TILE < n; t += gridDim.x) {
        const uint32_t base = t * SCAN_TILE;
        if (threadIdx.x == 0) run = sums[t];
        __syncthreads();
        for (uint32_t c = 0; c < SCAN_TILE; c += 256) {
            const uint32_t i = base + c + threadIdx.x;
            const uint32_t v = i < n ? in[i] : 0;
            uint32_t x = v;
            for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o); if ((threadIdx.x & 31) >= (uint32_t)o) x = scan_op<MAX>(x, y); }
            if ((threadIdx.x & 31) == 31) sh[threadIdx.x >> 5] = x;
            __syncthreads();
            uint32_t wbase = run;
            for (uint32_t w = 0; w < (threadIdx.x >> 5); ++w) wbase = scan_op<MAX>(wbase, sh[w]);
            if (MAX) {                                                 // exclusive: the inclusive value of the lane before
                const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, 1);
                if (i < n) out[i] = max(wbase, (threadIdx.x & 31) ? y : 0u);
            } else if (i < n) out[i] = wbase + x - v;
            __syncthreads();
            if (threadIdx.x == 255) run = scan_op<MAX>(wbase, x);
            __syncthreads();
        }
    }
}
__device__ __forceinline__ uint32_t put_dec(char *p, uint32_t v) {
    const uint32_t n = dec_digits(v);
    for (uint32_t i = n; i; --i) { p[i - 1] = (char)('0' + v % 10u); v /= 10u; }
    return n;
}
__global__ void __launch_bounds__(256)
slots_kernel(const uint32_t *__restrict__ seq_len, uint32_t n, uint32_t *__restrict__ slots) {
    uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) slots[r] = (seq_len[r] + 1u + 31u) / 32u;           // utb_read_slots
}
// ---- device-side framing (SURVEY 8f-1) ---------------------------------------------
// The host only counts the newlines of a chunk (which fixes the number of complete
// records and where the last one ends, itree.c:869-871: lines are read strictly in
// pairs); everything per read -- where its header and sequence lines start, the name
// (itree.c:879-882), the CR/LF trimming (itree.c:889-890) and the format checks
// (itree.c:880, 886) -- happens here, on the bytes that were copied to the device
// anyway.  Three kernels: newline count per 16 KB block, exclusive scan of the block
// counts (scan_top_kernel), newline positions + record parse.
#define FR_BPT 64u              // bytes per thread
#define FR_BLOCK (256u * FR_BPT)
#define FR_ERR_NONE 0xFFFFFFFFu
enum { FRE_NOHEADER = 1, FRE_SEQ_GT = 2, FRE_TOOLONG = 4, FRE_CHUNK = 7 };   // 1, 2, 4: codes as in pipeline.c (FE_*); 7: the chunk as a whole
// bit j of the result: byte j of the 64 bytes at p is '\n' (bytes at or beyond n_bytes never match);
// *nul (optional): whether one of those bytes is 0
__device__ __forceinline__ uint64_t nl_mask64(const uint8_t *__restrict__ raw, uint64_t at, uint64_t n_bytes, bool *nul = nullptr) {
    uint64_t m = 0, z = 0;
    if (nul) *nul = false;
    if (at >= n_bytes) return 0;
    const uint4 *p = reinterpret_cast<const uint4 *>(raw + at);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint4 v = __ldg(p + q);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t e = __vcmpeq4(w[k], 0x0A0A0A0Au) & 0x01010101u;
            m |= (uint64_t)((e * 0x01020408u) >> 24) << (16 * q + 4 * k);
            if (nul) { const uint32_t e0 = __vcmpeq4(w[k], 0u) & 0x01010101u; z |= (uint64_t)((e0 * 0x01020408u) >> 24) << (16 * q + 4 * k); }
        }
    }
    const uint64_t left = n_bytes - at;
    if (left < 64) { m &= (1ull << left) - 1ull; z &= (1ull << left) - 1ull; }
    if (nul) *nul = z != 0;
    return m;
}
__global__ void __launch_bounds__(256)
nl_count_kernel(const uint8_t *__restrict__ raw, uint64_t n_bytes, uint32_t *__restrict__ blk_cnt, uint32_t *__restrict__ nul_flag) {
    __shared__ uint32_t sh[8];
    const uint64_t at = ((uint64_t)blockIdx.x * 256u + threadIdx.x) * FR_BPT;
    bool nul;
    uint32_t c = __popcll(nl_mask64(raw, at, n_bytes, &nul));
    if (__any_sync(0xFFFFFFFFu, nul) && (threadIdx.x & 31) == 0) atomicOr(nul_flag, 1u);
    for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) { uint32_t t = 0; for (int w = 0; w < 8; ++w) t += sh[w]; blk_cnt[blockIdx.x] = t; }
}
// blk_off: exclusive scan of blk_cnt.  nl[i] = position of newline i, for i < limit (LPR lines per record of dims[0]).
template <uint32_t LPR>
__global__ void __launch_bounds__(256)
nl_index_kernel(const uint8_t *__restrict__ raw, uint64_t n_bytes, const uint32_t *__restrict__ blk_off,
                uint32_t limit, const uint32_t *__restrict__ dims, uint32_t *__restrict__ nl) {
    if (dims) limit = LPR * dims[0];
    __shared__ uint32_t sh[8];
    const uint64_t at = ((uint64_t)blockIdx.x * 256u + threadIdx.x) * FR_BPT;
    uint64_t m = nl_mask64(raw, at, n_bytes);
    const uint32_t c = __popcll(m), lane = threadIdx.x & 31u;
    uint32_t x = c;
    for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, x, o); if (lane >= (uint32_t)o) x += t; }
    if (lane == 31) sh[threadIdx.x >> 5] = x;
    __syncthreads();
    uint32_t i = blk_off[blockIdx.x] + x - c;
    for (uint32_t w = 0; w < (threadIdx.x >> 5); ++w) i += sh[w];
    while (m && i < limit) {
        nl[i++] = (uint32_t)(at + (uint32_t)(__ffsll((long long)m) - 1));
        m &= m - 1;
    }
}
// One thread per record r: header line = (nl[2r-1], nl[2r]], sequence line = (nl[2r], nl[2r+1]].
// The first malformed record (smallest r) is reported in *err as r << 3 | code; the host then
// re-frames from this batch on with its own exact reader, which reproduces the reference's message
// and partial output.
__global__ void __launch_bounds__(256)
frame_parse_kernel(const uint8_t *__restrict__ raw, const uint32_t *__restrict__ nl, uint32_t n_reads, const uint32_t *__restrict__ dims,
                   uint64_t *__restrict__ seq_off, uint32_t *__restrict__ seq_len,
                   uint32_t *__restrict__ name_off, uint32_t *__restrict__ name_len,
                   uint32_t *__restrict__ slots, uint32_t *__restrict__ err) {
    if (dims) n_reads = dims[0];
    for (uint64_t r64 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r64 < n_reads; r64 += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t r = (uint32_t)r64;
        const uint32_t hs = r ? nl[2 * r - 1] + 1u : 0u, hn = nl[2 * r], ss = hn + 1u, sn = nl[2 * r + 1];
        uint32_t code = 0;
        if (ss - hs >= UTB_LINELEN || sn + 1u - ss >= UTB_LINELEN) code = FRE_TOOLONG;
        else if (raw[hs] != '>') code = FRE_NOHEADER;              // itree.c:880
        else if (raw[ss] == '>') code = FRE_SEQ_GT;                // itree.c:886
        if (code) atomicMin(err, (r << 3) | code);
        uint32_t length = sn - ss;
        if (length && raw[ss + length - 1] == '\r') --length;      // itree.c:890
        uint32_t e = hs + 1u;                                      // name: up to the first ' ' or the newline (itree.c:881)
        while (e < hn && raw[e] != ' ') ++e;
        seq_off[r] = ss; seq_len[r] = length;
        name_off[r] = hs + 1u; name_len[r] = e - hs - 1u;
        slots[r] = (length + 1u + 31u) / 32u;                      // utb_read_slots
    }
}
// Chunk-level verdict of the device-side framing.  The reader cuts a chunk right before a line that begins with
// '>' (in a well-formed file exactly the header lines do, itree.c:880, 886), so a chunk holds whole records iff
// its newline count is even; with that, no NUL byte (strlen() semantics, itree.c:887) and every record well formed
// (frame_parse_kernel), the next chunk starts on a header line again -- by induction the framing equals the
// reference's strictly pairwise fgets (itree.c:869-871).  Anything else is reported as record 0 / FRE_CHUNK and
// the host re-reads from this chunk on with its exact reader.  LPR: lines per record, 2 for FASTA; 4 for FASTQ,
// where the same induction holds with "a multiple of 4" (the cut rule is argued in pipeline.c, fastq_cut).
template <uint32_t LPR>
__global__ void frame_setup_kernel(const uint32_t *__restrict__ info, uint32_t max_reads, uint32_t *__restrict__ dims, uint32_t *__restrict__ err) {
    const uint32_t n_lines = info[0], nul = info[1];
    const bool bad = nul || (n_lines % LPR) || !n_lines || (n_lines / LPR) > max_reads;
    dims[0] = bad ? 0u : n_lines / LPR;
    if (bad) atomicMin(err, (uint32_t)FRE_CHUNK);
}
// One thread per FASTQ record r: lines 4r .. 4r+3 are its header, sequence, separator and quality line, line i
// being (nl[i-1], nl[i]].  The rules, and the order in which they are checked, are the host framer's
// (pipeline.c, fq_record): the host re-frames a flagged chunk and reports the error itself.
__global__ void __launch_bounds__(256)
frame_parse_fastq_kernel(const uint8_t *__restrict__ raw, const uint32_t *__restrict__ nl, uint32_t n_reads, const uint32_t *__restrict__ dims,
                         uint64_t *__restrict__ seq_off, uint32_t *__restrict__ seq_len, uint64_t *__restrict__ qual_off,
                         uint32_t *__restrict__ name_off, uint32_t *__restrict__ name_len,
                         uint32_t *__restrict__ slots, uint32_t *__restrict__ err) {
    if (dims) n_reads = dims[0];
    for (uint64_t r64 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r64 < n_reads; r64 += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t r = (uint32_t)r64;
        const uint32_t hs = r ? nl[4 * r - 1] + 1u : 0u, hn = nl[4 * r], ss = hn + 1u, sn = nl[4 * r + 1];
        const uint32_t ps = sn + 1u, pn = nl[4 * r + 2], qs = pn + 1u, qn = nl[4 * r + 3];
        uint32_t length = sn - ss, qlength = qn - qs;
        if (length && raw[ss + length - 1] == '\r') --length;
        if (qlength && raw[qs + qlength - 1] == '\r') --qlength;
        uint32_t code = 0;
        if (hn + 1u - hs >= UTB_LINELEN || sn + 1u - ss >= UTB_LINELEN || pn + 1u - ps >= UTB_LINELEN || qn + 1u - qs >= UTB_LINELEN)
            code = UTB_FQ_TOOLONG;
        else if (raw[hs] != '@') code = UTB_FQ_NOHEADER;
        else if (raw[ps] != '+') code = UTB_FQ_NOSEPARATOR;
        else if (qlength != length) code = UTB_FQ_QUALLEN;
        if (code) { atomicMin(err, (r << 3) | code); length = 0; } // a flagged record gets no bases: its quality line may be
                                                                   // shorter, and qual_mask_kernel reads seq_len quality bytes
        uint32_t e = hs + 1u;                                      // name: up to the first ' ' or the newline, as for FASTA
        while (e < hn && raw[e] != ' ') ++e;
        seq_off[r] = ss; seq_len[r] = length; qual_off[r] = qs;
        name_off[r] = hs + 1u; name_len[r] = e - hs - 1u;
        slots[r] = (length + 1u + 31u) / 32u;                      // utb_read_slots
    }
}
// Quality masking (FASTQ with min_qual > 0): every base whose quality byte is below 33 + min_qual becomes 'N' in
// the device copy of the input, so pack_kernel marks it bad and the slide skips every window over it, as it does
// for any byte that is not a base (itree.c:919-926).  One thread per 32-base group with pack_kernel's group -> read
// mapping: a read is spread over as many threads as it has groups, however long it is.  thr4: 33 + min_qual in
// every byte.  Only sequence bytes are written, and quality bytes are only read.
__global__ void __launch_bounds__(256)
qual_mask_kernel(uint8_t *raw, const uint64_t *__restrict__ seq_off, const uint64_t *__restrict__ qual_off,
                 const uint32_t *__restrict__ seq_len, const uint32_t *__restrict__ grp_off,
                 uint32_t n_reads, uint32_t n_groups, const uint32_t *__restrict__ dims, uint32_t thr4) {
    if (dims) { n_reads = dims[0]; n_groups = dims[1]; }
    const uint32_t lane = threadIdx.x & 31u;
    for (uint64_t gw = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) & ~31ull; gw < n_groups; gw += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t g = (uint32_t)gw + lane;
        const uint32_t lo = group_read(grp_off, n_reads, (uint32_t)gw, lane);
        if (g >= n_groups) continue;
        const uint32_t b0 = (g - __ldg(grp_off + lo)) * 32u, len = __ldg(seq_len + lo);
        const uint32_t nv = len > b0 ? min(32u, len - b0) : 0u;    // real bases in this group
        if (!nv) continue;
        const uint64_t a = __ldg(qual_off + lo) + b0;
        const uint32_t *p = reinterpret_cast<const uint32_t *>(raw + (a & ~3ull));
        const uint32_t sh = (uint32_t)(a & 3u) * 8u, nw = (nv + 3u) >> 2;
        uint32_t prev = p[0], m = 0;
        for (uint32_t j = 0; j < nw; ++j) {
            const uint32_t cur = p[j + 1];
            const uint32_t lt = __vcmpltu4(__funnelshift_r(prev, cur, sh), thr4) & 0x01010101u;
            m |= ((lt * 0x01020408u) >> 24) << (4u * j);           // bit i: base b0 + i is masked
            prev = cur;
        }
        if (nv < 32u) m &= (1u << nv) - 1u;
        uint8_t *s = raw + __ldg(seq_off + lo) + b0;
        for (; m; m &= m - 1u) s[__ffs(m) - 1] = 'N';
    }
}

// ---- wrapped FASTA (UTB_INPUT_FASTA_WRAPPED) ----------------------------------------------------------------
// A record is a header line (a line that begins with '>') and every line up to the next header; its sequence is
// the concatenation of those lines without their '\n' and one '\r' before it.  No newline index: a chunk may hold
// n_bytes / 2 lines.  Everything is per 64-byte tile (nl_mask64's unit), one thread per tile:
//   wrap_tile_kernel   last line start and header count per tile
//   max-scan / sum-scan  -> the line in force at each tile's start, the index of its first record
//   wrap_keep_kernel   which bytes are sequence bytes (kmask), their count per tile, the long-line rule, and
//                      where every header starts (name_off)
//   sum-scan           -> where each tile's sequence bytes go in d_join
//   wrap_join_kernel   the sequence bytes, packed into d_join (stores coalesced per warp)
//   wrap_record_kernel one thread per record: name, seq_off / seq_len (from kmask, O(1)), the base limit, slots
// The reader cuts a chunk right before a line that begins with '>', which in wrapped FASTA always starts a record:
// by induction every chunk starts on a header and ends with '\n'.  A chunk that does not begin with '>', or holds
// more headers than the batch has reads, is flagged FRE_CHUNK and re-framed by the host (pipeline.c, wr_buffer),
// which applies the same rules.
struct WrapTile { uint64_t nl, ls, hs, cr; };   // newlines, line starts, header starts, '\r' bytes of one tile
__device__ __forceinline__ WrapTile wrap_tile(const uint8_t *__restrict__ raw, uint64_t at, uint64_t n_bytes) {
    WrapTile w = {0, 0, 0, 0};
    if (at >= n_bytes) return w;
    uint64_t gt = 0;
    const uint4 *p = reinterpret_cast<const uint4 *>(raw + at);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint4 v = __ldg(p + q);
        const uint32_t x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t sh = 16 * q + 4 * k;
            w.nl |= (uint64_t)(((__vcmpeq4(x[k], 0x0A0A0A0Au) & 0x01010101u) * 0x01020408u) >> 24) << sh;
            w.cr |= (uint64_t)(((__vcmpeq4(x[k], 0x0D0D0D0Du) & 0x01010101u) * 0x01020408u) >> 24) << sh;
            gt |= (uint64_t)(((__vcmpeq4(x[k], 0x3E3E3E3Eu) & 0x01010101u) * 0x01020408u) >> 24) << sh;
        }
    }
    const uint64_t left = n_bytes - at, valid = left < 64 ? (1ull << left) - 1ull : ~0ull;
    const uint64_t first = at == 0 || raw[at - 1] == '\n';          // byte at starts a line
    w.nl &= valid; w.cr &= valid;
    w.ls = ((w.nl << 1) | first) & valid;
    w.hs = w.ls & gt;
    return w;
}
__global__ void __launch_bounds__(256)
wrap_tile_kernel(const uint8_t *__restrict__ raw, uint64_t n_bytes, uint32_t n_tiles,
                 uint32_t *__restrict__ last_ls, uint32_t *__restrict__ hdr_cnt, uint32_t *__restrict__ err) {
    const uint32_t t = blockIdx.x * 256u + threadIdx.x;
    if (t >= n_tiles) return;
    const uint64_t at = (uint64_t)t * 64u;
    const WrapTile w = wrap_tile(raw, at, n_bytes);
    last_ls[t] = w.ls ? (uint32_t)(at + 63u - (uint32_t)__clzll((long long)w.ls)) : 0u;   // 0: none (the max-scan's identity)
    hdr_cnt[t] = __popcll(w.hs);
    if (t == 0 && raw[0] != '>') atomicMin(err, (uint32_t)FRE_CHUNK);
}
// ls_in[t]: start of the line in force at tile t's first byte (exclusive max-scan of last_ls); rec0[t]: records
// that start before tile t (exclusive sum-scan of hdr_cnt).  kmask[t]: the tile's sequence bytes -- not in a header
// line, not '\n', not a '\r' right before '\n'.
__global__ void __launch_bounds__(256)
wrap_keep_kernel(const uint8_t *__restrict__ raw, uint64_t n_bytes, uint32_t n_tiles, const uint32_t *__restrict__ ls_in,
                 const uint32_t *__restrict__ rec0, const uint32_t *__restrict__ dims, uint64_t *__restrict__ kmask,
                 uint32_t *__restrict__ keep_cnt, uint32_t *__restrict__ name_off, uint32_t *__restrict__ err) {
    const uint32_t t = blockIdx.x * 256u + threadIdx.x;
    if (t >= n_tiles) return;
    const uint64_t at = (uint64_t)t * 64u;
    const WrapTile w = wrap_tile(raw, at, n_bytes);
    const uint32_t lin = ls_in[t], r0 = rec0[t], n_reads = dims[0];
    // in-header-line mask: every byte takes the header flag of the nearest line start at or before it (segmented
    // copy by doubling; bit 0 is seeded from the line in force when no line starts there)
    uint64_t f = w.ls | 1ull, v = w.hs | ((!(w.ls & 1ull) && raw[lin] == '>') ? 1ull : 0ull);
#pragma unroll
    for (int s = 1; s < 64; s <<= 1) { v = (v & f) | ((v << s) & ~f); f |= f << s; }
    const uint64_t left = n_bytes - at;
    const uint64_t ends = (w.nl >> 1) | (left > 64 ? (uint64_t)(raw[at + 64] == '\n') << 63 : 1ull << (left - 1));   // byte before a line end
    const uint64_t valid = left < 64 ? (1ull << left) - 1ull : ~0ull;
    const uint64_t k = ~v & ~w.nl & ~(w.cr & ends) & valid;
    kmask[t] = k;
    keep_cnt[t] = __popcll(k);
    // a line of UTB_LINELEN bytes or more, counting its '\n': only the tile's first newline can end a line that
    // starts before the tile; its record is the last one that starts before it
    if (w.nl) {
        const uint32_t j = __ffsll((long long)w.nl) - 1;
        if (!(w.ls & ((2ull << j) - 1ull)) && at + j + 1u - lin >= UTB_LINELEN && r0)
            atomicMin(err, ((r0 - 1u) << 3) | UTB_FW_TOOLONG);
    }
    uint32_t r = r0;
    for (uint64_t h = w.hs; h && r < n_reads; h &= h - 1ull, ++r) name_off[r] = (uint32_t)(at + __ffsll((long long)h));   // the byte after '>'
}
// Packs the sequence bytes of the block's 256 tiles into join: each thread takes 4 bytes at a stride of 1 KiB, so a
// warp's stores fall into a few consecutive sectors.
__global__ void __launch_bounds__(256)
wrap_join_kernel(const uint8_t *__restrict__ raw, uint64_t n_bytes, uint32_t n_tiles, const uint64_t *__restrict__ kmask,
                 const uint32_t *__restrict__ join_off, uint8_t *__restrict__ join) {
    __shared__ uint64_t km[256];
    __shared__ uint32_t jo[256];
    const uint32_t t0 = blockIdx.x * 256u;
    if (t0 + threadIdx.x < n_tiles) { km[threadIdx.x] = kmask[t0 + threadIdx.x]; jo[threadIdx.x] = join_off[t0 + threadIdx.x]; }
    __syncthreads();
    const uint64_t base = (uint64_t)t0 * 64u;
#pragma unroll 4
    for (uint32_t c = 0; c < FR_BLOCK; c += 1024u) {
        const uint32_t o = c + 4u * threadIdx.x, lt = o >> 6, sh = o & 63u;
        if (base + o >= n_bytes) break;
        const uint64_t m = km[lt];
        uint32_t bits = (uint32_t)(m >> sh) & 0xFu;
        if (!bits) continue;
        const uint32_t x = *reinterpret_cast<const uint32_t *>(raw + base + o);
        uint32_t d = jo[lt] + __popcll(m & ((1ull << sh) - 1ull));
        for (; bits; bits &= bits - 1u) join[d++] = (uint8_t)(x >> (8u * (__ffs(bits) - 1u)));
    }
}
__device__ __forceinline__ uint32_t wrap_join_at(const uint64_t *__restrict__ kmask, const uint32_t *__restrict__ join_off, uint32_t p) {
    return join_off[p >> 6] + __popcll(kmask[p >> 6] & ((1ull << (p & 63u)) - 1ull));   // sequence bytes before byte p
}
// One thread per record r: its header starts at name_off[r] - 1; a header line holds no sequence byte, so the
// record's sequence starts at the join offset of its header and ends at the next record's (or the total).
__global__ void __launch_bounds__(256)
wrap_record_kernel(const uint8_t *__restrict__ raw, uint64_t n_bytes, const uint64_t *__restrict__ kmask,
                   const uint32_t *__restrict__ join_off, const uint32_t *__restrict__ join_total, uint32_t n_reads,
                   const uint32_t *__restrict__ dims, uint64_t *__restrict__ seq_off, uint32_t *__restrict__ seq_len,
                   const uint32_t *__restrict__ name_off, uint32_t *__restrict__ name_len,
                   uint32_t *__restrict__ slots, uint32_t *__restrict__ err) {
    if (dims) n_reads = dims[0];
    for (uint64_t r64 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r64 < n_reads; r64 += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t r = (uint32_t)r64, hs = name_off[r] - 1u;
        const uint32_t so = wrap_join_at(kmask, join_off, hs);
        const uint32_t eo = r + 1u < n_reads ? wrap_join_at(kmask, join_off, name_off[r + 1u] - 1u) : *join_total;
        uint32_t length = eo - so;
        if (length > UTB_MAXSEQ) { atomicMin(err, (r << 3) | UTB_FW_TOOLONG); length = 0; }
        uint32_t e = hs + 1u;                                      // name: up to the first ' ' or the newline, as for FASTA
        while (e < n_bytes && raw[e] != ' ' && raw[e] != '\n') ++e;
        seq_off[r] = so; seq_len[r] = length;
        name_len[r] = e - hs - 1u;
        slots[r] = (length + 1u + 31u) / 32u;                      // utb_read_slots
    }
}

#define FW_WARPS 8
__global__ void __launch_bounds__(FW_WARPS * 32)
fmt_write_kernel(DevDB db, const utb_result *__restrict__ res, const uint8_t *__restrict__ raw,
                 const uint32_t *__restrict__ name_off, const uint32_t *__restrict__ name_len,
                 const uint32_t *__restrict__ line_off, uint32_t n_reads, const uint32_t *__restrict__ dims, char *__restrict__ text) {
    if (dims) n_reads = dims[0];
    __shared__ char s_tail[FW_WARPS][48];
    const uint32_t lane = threadIdx.x & 31u, wib = threadIdx.x >> 5;
    for (uint64_t r = (uint64_t)blockIdx.x * FW_WARPS + wib; r < n_reads; r += (uint64_t)gridDim.x * FW_WARPS) {
        const utb_result v = res[r];
        if (v.kind == UTB_NONE) continue;
        char *out = text + line_off[r];
        const uint32_t nl = __ldg(name_len + r), tl = tax_len_of(db, v);
        const uint8_t *nm = raw + __ldg(name_off + r);
        const char *lab = db.blob + __ldg(db.off + v.label);
        uint32_t tn = 0;
        __syncwarp();                                              // the previous round's readers of s_tail are done
        if (lane == 0) {                                           // "\t<found>\t<uix>\t*\n" or "...\t<sl>;<ol>\n"
            char *t = s_tail[wib];
            t[tn++] = '\t'; tn += put_dec(t + tn, v.found);
            t[tn++] = '\t'; tn += put_dec(t + tn, v.uix);
            t[tn++] = '\t';
            if (v.kind == UTB_STAR) t[tn++] = '*';
            else { tn += put_dec(t + tn, v.sl); t[tn++] = ';'; tn += put_dec(t + tn, v.ol); }
            t[tn++] = '\n';
        }
        tn = __shfl_sync(0xFFFFFFFFu, tn, 0);
        __syncwarp();
        for (uint32_t i = lane; i < nl; i += 32) out[i] = (char)nm[i];
        if (lane == 0) out[nl] = '\t';
        for (uint32_t i = lane; i < tl; i += 32) out[nl + 1 + i] = lab[i];
        for (uint32_t i = lane; i < tn; i += 32) out[nl + 1 + tl + i] = s_tail[wib][i];
    }
}

// ---------------------------------------------------------------------------
// random-sector gather microbenchmark (roofline denominator, SURVEY 8d)
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
rand32_kernel(const uint8_t *__restrict__ buf, uint64_t n_sectors, uint32_t per_thread, uint64_t seed,
              unsigned long long *__restrict__ sink) {
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t x = (t + 1) * 0x9E3779B97F4A7C15ull + seed;
    uint64_t acc = 0;
    for (uint32_t k = 0; k < per_thread; k += 8) {
        uint64_t v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            x ^= x >> 12; x ^= x << 25; x ^= x >> 27;              // xorshift64*
            uint64_t s = __umul64hi(x * 0x2545F4914F6CDD1Dull, n_sectors);   // uniform in [0, n_sectors)
            v[j] = __ldg(reinterpret_cast<const uint64_t *>(buf + s * 32));
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) acc += v[j];
    }
    if (acc == 0x123456789ull) atomicAdd(sink, 1ull);              // keep the loads alive
}

// ---------------------------------------------------------------------------
// C ABI: database residency
// ---------------------------------------------------------------------------
extern "C" int utb_device_count(int *n) {
    if (!n) { utb_set_error("utb_device_count: null argument"); return UTB_ERR_ARG; }
    *n = 0;
    cudaError_t e = cudaGetDeviceCount(n);
    if (e != cudaSuccess || *n <= 0) {
        *n = 0;
        utb_set_error("no CUDA device available (%s); there is no CPU fallback", cudaGetErrorString(e));
        return UTB_ERR_CUDA;
    }
    return UTB_OK;
}

static int check_device(int device) {
    int n = 0;
    int rc = utb_device_count(&n);
    if (rc) return rc;
    if (device < 0 || device >= n) { utb_set_error("device %d out of range (have %d)", device, n); return UTB_ERR_ARG; }
    cudaDeviceProp p;
    CK(cudaGetDeviceProperties(&p, device));
    if (p.major < 10) {
        utb_set_error("device %d is sm_%d%d; this library is built for sm_100a only", device, p.major, p.minor);
        return UTB_ERR_CUDA;
    }
    return UTB_OK;
}

// host (pageable / mmap'ed) -> device: UP_THREADS workers, each with its own pinned bounce buffer and
// stream, take the chunks round-robin, so the page-cache copies run in parallel and overlap the PCIe
// copies (one thread and one memcpy moved ~3 GB/s: 2.4 s for an 8 GB tree)
#include <pthread.h>
#define UP_CHUNK ((size_t)32 << 20)
#define UP_THREADS 6
struct up_job { int device; char *dst; const char *src; size_t n; int t, nt; int rc; char err[256]; };
static void *up_worker(void *a_) {
    up_job *j = (up_job *)a_;
    void *pin = nullptr; cudaStream_t st = nullptr; cudaEvent_t ev = nullptr;
    cudaError_t e = cudaSetDevice(j->device);
    if (e == cudaSuccess) e = cudaMallocHost(&pin, UP_CHUNK);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    for (size_t o = (size_t)j->t * UP_CHUNK; e == cudaSuccess && o < j->n; o += (size_t)j->nt * UP_CHUNK) {
        const size_t c = j->n - o < UP_CHUNK ? j->n - o : UP_CHUNK;
        e = cudaEventSynchronize(ev);                              // the previous copy out of this buffer is done
        if (e != cudaSuccess) break;
        memcpy(pin, j->src + o, c);
        e = cudaMemcpyAsync(j->dst + o, pin, c, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaEventRecord(ev, st);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { j->rc = UTB_ERR_CUDA; snprintf(j->err, sizeof j->err, "CUDA error %s during upload (%s)", cudaGetErrorName(e), cudaGetErrorString(e)); }
    if (ev) cudaEventDestroy(ev);
    if (st) cudaStreamDestroy(st);
    if (pin) cudaFreeHost(pin);
    return nullptr;
}
static int upload_streamed(int device, void *dst, const void *src, size_t n) {
    int nt = (int)((n + UP_CHUNK - 1) / UP_CHUNK);
    if (nt > UP_THREADS) nt = UP_THREADS;
    if (nt < 1) return UTB_OK;
    up_job job[UP_THREADS];
    pthread_t th[UP_THREADS];
    int started = 0, rc = UTB_OK;
    for (int t = 0; t < nt; ++t) {
        job[t].device = device; job[t].dst = (char *)dst; job[t].src = (const char *)src; job[t].n = n; job[t].t = t; job[t].nt = nt; job[t].rc = UTB_OK;
        if (t == nt - 1 || pthread_create(&th[t], nullptr, up_worker, &job[t])) { up_worker(&job[t]); if (t != nt - 1) job[t].t = -1; }   // last share (or a failed spawn) runs here
        else ++started;
    }
    for (int t = 0; t < nt; ++t) {
        if (t != nt - 1 && job[t].t >= 0) pthread_join(th[t], nullptr);
        if (job[t].rc && !rc) { rc = job[t].rc; utb_set_error("%s", job[t].err); }
    }
    (void)started;
    return rc;
}

static int db_upload_impl(const utb_ctr *ctr, int device, utb_db *db);
extern "C" int utb_db_upload(const utb_ctr *ctr, int device, utb_db **out) {
    if (!ctr || !out) { utb_set_error("utb_db_upload: null argument"); return UTB_ERR_ARG; }
    *out = nullptr;
    int rc = check_device(device);
    if (rc) return rc;
    CK(cudaSetDevice(device));
    utb_db *db = (utb_db *)calloc(1, sizeof(utb_db));
    if (!db) { utb_set_error("out of memory"); return UTB_ERR_NOMEM; }
    db->device = device;
    db->ema_hit_rate = -1.0;                                       // no batch seen yet: the first one sets it
    rc = db_upload_impl(ctr, device, db);
    if (rc) { utb_db_free(db); return rc; }                        // device buffers allocated so far are released
    *out = db;
    return UTB_OK;
}
// errors inside db_upload_impl / utb_db_clone: everything allocated so far hangs off `db`, which the caller frees
static int db_build_tables(utb_db *db, size_t nb_binix, size_t nb_recs);
static int db_upload_impl(const utb_ctr *ctr, int device, utb_db *db) {
    int rc;
    const size_t nb_binix = (size_t)UTB_NUMBINS * ctr->binix_bytes;
    const size_t nb_recs = (size_t)(ctr->num_nodes * ctr->sz);
    const size_t nl = ctr->max_ix;
    if (cudaDeviceGetAttribute(&db->sm_count, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || db->sm_count < 1) { cudaGetLastError(); db->sm_count = 148; }
    CK(cudaMalloc(&db->binix, nb_binix + 64));
    CK(cudaMalloc(&db->recs, nb_recs + 64));                       // +slack: itree.c:766
    // the label strings, each at a multiple of 8 bytes and NUL-padded to the next one: the vote's walk compares two
    // labels eight characters per step from the same offset in both (scan_token)
    size_t blob8 = 0;
    for (size_t i = 0; i < nl; ++i) blob8 += ((size_t)(ctr->off[i + 1] - ctr->off[i]) + 7) & ~(size_t)7;
    if (blob8 + 64 >= ((size_t)1 << 32)) { utb_set_error("label strings exceed 4 GB"); return UTB_ERR_LIMIT; }
    char *h_blob = (char *)calloc(blob8 + 64, 1);
    uint32_t *h_off = (uint32_t *)malloc((nl + 1) * 4);
    if (!h_blob || !h_off) { free(h_blob); free(h_off); utb_set_error("out of memory"); return UTB_ERR_NOMEM; }
    {
        size_t at = 0;
        for (size_t i = 0; i < nl; ++i) {
            const size_t l = ctr->off[i + 1] - ctr->off[i];
            h_off[i] = (uint32_t)at;
            memcpy(h_blob + at, ctr->blob + ctr->off[i], l);
            at += (l + 7) & ~(size_t)7;
        }
        h_off[nl] = (uint32_t)at;
    }
    struct HostTmp { char *b; uint32_t *o; ~HostTmp() { free(b); free(o); } } host_tmp{h_blob, h_off};
    CK(cudaMalloc(&db->blob, blob8 + 64));
    CK(cudaMalloc(&db->off, (nl + 1) * 4));
    CK(cudaMalloc(&db->rank, (nl + 1) * 4));
    CK(cudaMalloc(&db->by_rank, (nl + 1) * 4));
    CK(cudaMemset((char *)db->binix + nb_binix, 0, 64));
    CK(cudaMemset((char *)db->recs + nb_recs, 0, 64));
    rc = upload_streamed(device, db->binix, ctr->binix_raw, nb_binix); if (rc) return rc;
    rc = upload_streamed(device, db->recs, ctr->recs, nb_recs); if (rc) return rc;
    CK(cudaMemcpy(db->blob, h_blob, blob8 + 64, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(db->off, h_off, (nl + 1) * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(db->rank, ctr->rank, nl * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(db->by_rank, ctr->by_rank, nl * 4, cudaMemcpyHostToDevice));
    db->nb_binix = nb_binix; db->nb_recs = nb_recs; db->nb_blob = blob8 + 64; db->nb_lab = (nl + 1) * 4;
    db->d.binix32 = ctr->binix_bytes == 4 ? (const uint32_t *)db->binix : nullptr;
    db->d.binix64 = ctr->binix_bytes == 8 ? (const uint64_t *)db->binix : nullptr;
    db->d.recs = (const uint8_t *)db->recs;
    db->d.num_nodes = ctr->num_nodes;
    db->d.sz = ctr->sz; db->d.ix_bytes = ctr->ix_bytes; db->d.max_ix = ctr->max_ix;
    db->d.blob = (const char *)db->blob;
    db->d.off = (const uint32_t *)db->off;
    db->d.rank = (const uint32_t *)db->rank;
    db->d.by_rank = (const uint32_t *)db->by_rank;
    for (size_t i = 0; i < nl; ++i) { size_t l = ctr->off[i + 1] - ctr->off[i]; if (l > db->max_label) db->max_label = l; }
    return db_build_tables(db, nb_binix, nb_recs);
}
template <typename F> static void launch_per_bin(uint64_t n_records, F f) {
    // lanes per prefix bin: about half the mean bucket (1 .. 32)
    const uint64_t mean = n_records >> 24;
    int g = 1;
    while (g < 32 && (uint64_t)g * 2 <= mean) g <<= 1;
    f(g, (unsigned)(((uint64_t)(UTB_NUMBINS - 1) * g + 255) / 256));
}
static int db_build_tables(utb_db *db, size_t nb_binix, size_t nb_recs) {
    const size_t fixed = db->nb_blob + 3 * db->nb_lab;
    db->hbm_bytes = nb_binix + nb_recs + fixed;
    // Is the CTR regular (what utree-compress emits: every bucket strictly sorted, at most the first-bin
    // quirk)?  Then the record words are distinct and a hash table answers exactly what xtSuffixBS
    // answers; otherwise keep the reference's probe sequence on the on-disk image.
    {
        db->d.quirk_bin = 0xFFFFFFFFu;
        unsigned long long *d_out, h_out[4] = {0, 0, ~0ull, ~0ull};
        CK(cudaMalloc(&d_out, 32));
        cudaError_t e = cudaMemcpy(d_out, h_out, 32, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) { verify_kernel<<<(UTB_NUMBINS - 1 + 255) / 256, 256>>>(db->d, d_out); e = cudaGetLastError(); }
        if (e == cudaSuccess) e = cudaMemcpy(h_out, d_out, 32, cudaMemcpyDeviceToHost);
        cudaFree(d_out);
        CK(e);
        db->regular = h_out[0] == 0 && (h_out[1] == 0 || (h_out[1] == 1 && h_out[2] == h_out[3]));
        if (db->regular && h_out[1] == 1) db->d.quirk_bin = (uint32_t)h_out[2];
        const char *lk = getenv("UTB_LOOKUP");                      // "exact" forces the reference probe sequence
        db->use_table = db->regular && !(lk && !strcmp(lk, "exact"));
    }
    // sector hash table at load <= 0.5 (4 entries per sector, 3 with uint32_t labels); grown if a record cannot be placed within KT_MAXD sectors
    const uint64_t n = db->d.num_nodes;
    const uint32_t wide = db->d.ix_bytes == 4;
    uint64_t sectors = wide ? n / 3 * 2 + 1 : n / 2 + 1;
    if (sectors < KT_MIN_SECTORS) sectors = KT_MIN_SECTORS;
    uint32_t table_failed = 0;                                      // records the table could not place at its largest size
    if (db->use_table) {
        uint32_t *d_ovf;
        CK(cudaMalloc(&d_ovf, 4));
        for (int attempt = 0;; ++attempt) {
            cudaError_t e = cudaMalloc(&db->ktab, sectors * 32);
            if (e == cudaSuccess) e = cudaMemset(db->ktab, 0, sectors * 32);
            if (e == cudaSuccess) e = cudaMemset(d_ovf, 0, 4);
            if (e != cudaSuccess) { cudaFree(d_ovf); CK(e); }
            DevDB dd = db->d;
            unsigned long long *kt = (unsigned long long *)db->ktab;
            launch_per_bin(n, [&](int g, unsigned blocks) {
                switch (g) {
                case 1: ktab_build_kernel<1><<<blocks, 256>>>(dd, kt, wide, sectors, d_ovf); break;
                case 2: ktab_build_kernel<2><<<blocks, 256>>>(dd, kt, wide, sectors, d_ovf); break;
                case 4: ktab_build_kernel<4><<<blocks, 256>>>(dd, kt, wide, sectors, d_ovf); break;
                case 8: ktab_build_kernel<8><<<blocks, 256>>>(dd, kt, wide, sectors, d_ovf); break;
                case 16: ktab_build_kernel<16><<<blocks, 256>>>(dd, kt, wide, sectors, d_ovf); break;
                default: ktab_build_kernel<32><<<blocks, 256>>>(dd, kt, wide, sectors, d_ovf); break;
                }
            });
            uint32_t ovf = 0;
            e = cudaGetLastError();
            if (e == cudaSuccess) e = cudaMemcpy(&ovf, d_ovf, 4, cudaMemcpyDeviceToHost);
            if (e != cudaSuccess) { cudaFree(d_ovf); CK(e); }
            if (!ovf) break;
            cudaFree(db->ktab); db->ktab = nullptr;
            if (attempt == 3) { table_failed = ovf; break; }
            sectors += sectors / 2;
        }
        cudaFree(d_ovf);
        // Records whose hashes crowd one stretch of sectors more than 1.5^3 growth spreads them: the CTR is
        // still valid, so search it with the reference probe sequence on the on-disk image (still resident
        // here) instead of refusing it.  It gets the same L2 set-up as an irregular CTR below.
        if (table_failed) db->use_table = 0;
    }
    if (db->use_table) {
        db->d.ktab = (const uint64_t *)db->ktab; db->d.kt_wide = wide; db->d.kt_sectors = sectors;
        db->nb_ktab = sectors * 32;
        const char *bm = getenv("UTB_SIEVE");                      // 0 off, 1 always, default auto
        db->sieve_mode = bm ? (atoi(bm) == 0 ? 0 : atoi(bm) == 1 ? 1 : 2) : 2;
        if (db->sieve_mode) {
            // SV_RPL records per 128-byte line = ~43 bits per record: ~0.04 % false positives
            uint64_t lines = n / SV_RPL + 1024;
            if (lines >= ((uint64_t)1 << 28)) lines = ((uint64_t)1 << 28) - 1;   // > 6.4 G records: more records per line, more false positives
            CK(cudaMalloc(&db->sieve, lines * 128));
            CK(cudaMemset(db->sieve, 0, lines * 128));
            db->d.sv_lines = (uint32_t)lines;
            DevDB dd = db->d;
            uint32_t *sv = (uint32_t *)db->sieve;
            launch_per_bin(n, [&](int g, unsigned blocks) {
                switch (g) {
                case 1: sieve_build_kernel<1><<<blocks, 256>>>(dd, sv); break;
                case 2: sieve_build_kernel<2><<<blocks, 256>>>(dd, sv); break;
                case 4: sieve_build_kernel<4><<<blocks, 256>>>(dd, sv); break;
                case 8: sieve_build_kernel<8><<<blocks, 256>>>(dd, sv); break;
                case 16: sieve_build_kernel<16><<<blocks, 256>>>(dd, sv); break;
                default: sieve_build_kernel<32><<<blocks, 256>>>(dd, sv); break;
                }
            });
            CK(cudaGetLastError());
            CK(cudaDeviceSynchronize());
            db->d.sieve = (const uint2 *)db->sieve;
            db->nb_sieve = lines * 128;
        }
        CK(cudaDeviceSynchronize());
        CK(cudaFree(db->recs)); CK(cudaFree(db->binix));           // the on-disk image is no longer needed
        db->recs = db->binix = nullptr; db->d.recs = nullptr; db->d.binix32 = nullptr; db->d.binix64 = nullptr;
        db->nb_recs = db->nb_binix = 0;
        db->hbm_bytes = db->nb_ktab + db->nb_sieve + fixed;
    } else {
        // Reference probe sequence: the hot prefix table pinned in L2 -- reserve persisting lines for the
        // index so the record traffic does not evict it (applied per stream in utb_batch_create).
        cudaDeviceProp p;
        CK(cudaGetDeviceProperties(&p, db->device));
        if (p.persistingL2CacheMaxSize > 0 && p.accessPolicyMaxWindowSize > 0) {
            size_t want = nb_binix < (size_t)p.persistingL2CacheMaxSize ? nb_binix : (size_t)p.persistingL2CacheMaxSize;
            if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) == cudaSuccess) {
                db->l2_window = 1;
                db->l2_window_bytes = nb_binix < (size_t)p.accessPolicyMaxWindowSize ? nb_binix : (size_t)p.accessPolicyMaxWindowSize;
                // a window larger than the set-aside would thrash it: persist only the fraction that fits
                db->l2_hit_ratio = want >= db->l2_window_bytes ? 1.0f : (float)((double)want / (double)db->l2_window_bytes);
            } else cudaGetLastError();
        }
    }
    if (getenv("UTB_STATS")) {
        char why[96] = "";
        if (table_failed) snprintf(why, sizeof why, " (sector hash table not built: %u records unplaced)", table_failed);
        fprintf(stderr, "utree-b200: device %d: %s%s, %.2f GB resident (table %.2f GB, sieve %.2f GB)\n", db->device,
                db->use_table ? "sector hash table" : "reference probe sequence", why, db->hbm_bytes / 1e9,
                db->nb_ktab / 1e9, db->nb_sieve / 1e9);
    }
    return UTB_OK;
}

// A second GPU gets the finished tables from the first one over NVLink (peer copy) instead of a
// second PCIe upload and rebuild (SURVEY 8e).
extern "C" int utb_db_clone(const utb_db *src, int device, utb_db **out) {
    if (!src || !out) { utb_set_error("utb_db_clone: null argument"); return UTB_ERR_ARG; }
    *out = nullptr;
    int rc = check_device(device);
    if (rc) return rc;
    CK(cudaSetDevice(device));
    utb_db *db = (utb_db *)calloc(1, sizeof(utb_db));
    if (!db) { utb_set_error("out of memory"); return UTB_ERR_NOMEM; }
    *db = *src;
    db->device = device;
    db->binix = db->recs = db->blob = db->off = db->rank = db->by_rank = db->ktab = db->sieve = nullptr;
    if (cudaDeviceGetAttribute(&db->sm_count, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || db->sm_count < 1) { cudaGetLastError(); db->sm_count = 148; }
    int can = 0;
    if (cudaDeviceCanAccessPeer(&can, device, src->device) == cudaSuccess && can) {
        cudaError_t e = cudaDeviceEnablePeerAccess(src->device, 0);
        if (e != cudaSuccess) cudaGetLastError();                   // already enabled, or staged through the host by the runtime
    } else cudaGetLastError();
    struct { void **dst; void *from; size_t n; } parts[] = {
        {&db->binix, src->binix, src->nb_binix ? src->nb_binix + 64 : 0}, {&db->recs, src->recs, src->nb_recs ? src->nb_recs + 64 : 0},
        {&db->blob, src->blob, src->nb_blob}, {&db->off, src->off, src->nb_lab}, {&db->rank, src->rank, src->nb_lab},
        {&db->by_rank, src->by_rank, src->nb_lab}, {&db->ktab, src->ktab, src->nb_ktab},
        {&db->sieve, src->sieve, src->nb_sieve}};
    cudaError_t e = cudaSuccess;
    for (size_t i = 0; i < sizeof parts / sizeof parts[0] && e == cudaSuccess; ++i) {
        if (!parts[i].n || !parts[i].from) continue;
        e = cudaMalloc(parts[i].dst, parts[i].n);
        if (e == cudaSuccess) e = cudaMemcpyPeer(*parts[i].dst, device, parts[i].from, src->device, parts[i].n);
    }
    if (e != cudaSuccess) {
        utb_set_error("CUDA error %s cloning the tree to device %d (%s)", cudaGetErrorName(e), device, cudaGetErrorString(e));
        utb_db_free(db);
        return UTB_ERR_CUDA;
    }
    db->d.binix32 = src->d.binix32 ? (const uint32_t *)db->binix : nullptr;
    db->d.binix64 = src->d.binix64 ? (const uint64_t *)db->binix : nullptr;
    db->d.recs = (const uint8_t *)db->recs;
    db->d.blob = (const char *)db->blob; db->d.off = (const uint32_t *)db->off;
    db->d.rank = (const uint32_t *)db->rank; db->d.by_rank = (const uint32_t *)db->by_rank;
    db->d.ktab = (const uint64_t *)db->ktab; db->d.sieve = (const uint2 *)db->sieve;
    if (db->l2_window && cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, db->l2_window_bytes) != cudaSuccess) { cudaGetLastError(); db->l2_window = 0; }
    *out = db;
    return UTB_OK;
}

extern "C" void utb_db_free(utb_db *db) {
    if (!db) return;
    cudaSetDevice(db->device);
    cudaFree(db->binix); cudaFree(db->recs); cudaFree(db->blob); cudaFree(db->ktab); cudaFree(db->sieve);
    cudaFree(db->off); cudaFree(db->rank); cudaFree(db->by_rank);
    free(db);
}
extern "C" uint64_t utb_db_hbm_bytes(const utb_db *db) { return db ? db->hbm_bytes : 0; }
extern "C" int utb_db_lookup_mode(const utb_db *db) { return db ? db->use_table : 0; }
extern "C" int utb_db_device(const utb_db *db) { return db ? db->device : -1; }

// ---------------------------------------------------------------------------
// scratch + launch of the long-read vote (vote_block / vote_big_* kernels)
// ---------------------------------------------------------------------------
struct vote_scratch { VoteLong vl; unsigned n_cta; };
static void vs_free(vote_scratch *vs) {
    cudaFree(vs->vl.hist); cudaFree(vs->vl.tlab); cudaFree(vs->vl.tcnt);
    cudaFree(vs->vl.big_hist); cudaFree(vs->vl.big_tlab); cudaFree(vs->vl.big_tcnt); cudaFree(vs->vl.big_list); cudaFree(vs->vl.big_state); cudaFree(vs->vl.work);
    memset(vs, 0, sizeof *vs);
}
// max_bytes: raw bytes a batch can hold -- a read of more than max_bytes / pool bases cannot occur more than pool times
static int vs_alloc(const utb_db *db, size_t max_bytes, vote_scratch *vs) {
    memset(vs, 0, sizeof *vs);
    const size_t nl = db->d.max_ix ? db->d.max_ix : 1;
    vs->n_cta = (unsigned)db->sm_count * VB_PER_SM;
    size_t pool = ((size_t)384 << 20) / (12 * nl);                 // at most 384 MB of histograms for the split reads of a batch
    if (pool > VBIG_POOL_MAX) pool = VBIG_POOL_MAX;
    if (pool < 1) pool = 1;
    vs->vl.pool = (uint32_t)pool;
    // entries (hits in list mode, lookup slots otherwise) beyond which a read is split across the grid; when more than
    // `pool` reads of a batch qualify the rest are voted by one CTA each, as the shorter ones are
    vs->vl.split_slots = (size_t)128 << 10;
    (void)max_bytes;
    const char *e = getenv("UTB_VOTE_SPLIT_SLOTS");                // tests: a small threshold sends short "long" reads through the split path
    if (e && atoll(e) > 0) vs->vl.split_slots = (unsigned long long)atoll(e);
    vs->vl.sort_max = VB_SORT_MAX;
    e = getenv("UTB_VOTE_SORT_MAX");
    if (e && atoi(e) >= 0 && (uint32_t)atoi(e) < VB_SORT_MAX) vs->vl.sort_max = (uint32_t)atoi(e);
    cudaError_t err = cudaMalloc(&vs->vl.hist, (size_t)vs->n_cta * nl * 4);
    if (err == cudaSuccess) err = cudaMalloc(&vs->vl.tlab, (size_t)vs->n_cta * nl * 4);
    if (err == cudaSuccess) err = cudaMalloc(&vs->vl.tcnt, (size_t)vs->n_cta * nl * 4);
    if (err == cudaSuccess) err = cudaMalloc(&vs->vl.big_hist, pool * nl * 4);
    if (err == cudaSuccess) err = cudaMalloc(&vs->vl.big_tlab, pool * nl * 4);
    if (err == cudaSuccess) err = cudaMalloc(&vs->vl.big_tcnt, pool * nl * 4);
    if (err == cudaSuccess) err = cudaMalloc(&vs->vl.big_list, pool * 4);
    if (err == cudaSuccess) err = cudaMalloc(&vs->vl.big_state, (1 + 2 * pool) * 4);
    if (err == cudaSuccess) err = cudaMalloc(&vs->vl.work, 4);
    if (err == cudaSuccess) err = cudaMemset(vs->vl.hist, 0, (size_t)vs->n_cta * nl * 4);      // the kernels leave the histograms zeroed
    if (err == cudaSuccess) err = cudaMemset(vs->vl.big_hist, 0, pool * nl * 4);
    if (err != cudaSuccess) { vs_free(vs); CK(err); }
    return UTB_OK;
}
static int launch_long_vote(const utb_db *db, const VoteIn &in, utb_result *results, const uint32_t *gen_list, const uint32_t *gen_count,
                            vote_scratch *vs, unsigned long long *counters, cudaStream_t st) {
    CK(cudaMemsetAsync(vs->vl.big_state, 0, (1 + 2 * (size_t)vs->vl.pool) * 4, st));
    CK(cudaMemsetAsync(vs->vl.work, 0, 4, st));
    vote_block_kernel<<<vs->n_cta, VB_THREADS, 0, st>>>(db->d, in, results, gen_list, gen_count, vs->vl, counters);
    vote_big_count_kernel<<<(unsigned)db->sm_count * 4, VB_THREADS, 0, st>>>(db->d, in, vs->vl);
    vote_big_finish_kernel<<<vs->vl.pool < (uint32_t)db->sm_count ? vs->vl.pool : (unsigned)db->sm_count, VB_THREADS, 0, st>>>(db->d, vs->vl, results, counters);
    CK(cudaGetLastError());
    return UTB_OK;
}

// ---------------------------------------------------------------------------
// C ABI: batches
// ---------------------------------------------------------------------------

struct utb_batch {
    utb_db *db;
    cudaStream_t st;
    cudaEvent_t done, ev[7];
    size_t max_bytes, max_reads;
    uint64_t max_groups;
    // pinned host
    char *h_bytes; uint64_t *h_seq_off; uint32_t *h_seq_len; uint32_t *h_grp_off;
    utb_result *h_results; unsigned long long *h_counters;
    uint32_t *h_name_off, *h_name_len; char *h_text; uint32_t *h_text_len; size_t text_cap, h_text_cap;   // device-side formatting
    // device
    uint8_t *d_raw; uint64_t *d_seq_off; uint32_t *d_seq_len; uint32_t *d_grp_off;
    uint64_t *d_pk; uint32_t *d_bad; uint32_t *d_hits; uint64_t *d_pl;
    utb_result *d_results; uint32_t *d_gen_list; uint32_t *d_gen_count; uint32_t *d_warp_list; uint32_t *d_warp_count;
    uint32_t *d_name_off, *d_name_len, *d_line_len, *d_line_off, *d_scan_sums, *d_text_len; char *d_text;
    utb_batch_out out;
    unsigned long long *d_counters;   // [4][COUNTER_SLOTS]: lookups, hits, good finds, exact-path sectors (summed on the host)
    vote_scratch vs;
    uint32_t *d_sel_cnt, *d_sel_off, *d_sel, *d_sel_gap, *d_sel_total, *h_sel_cnt, *h_sel, *h_sel_total; size_t sel_cap;   // non-GG mode (UTB_OUT_SELECTIONS)
    uint64_t *d_qwords; uint32_t *d_qslots; unsigned long long *d_qcount; uint64_t q_cap;   // filter survivors (window planes, slots)
    uint32_t *d_hitmap;
    uint32_t *d_rid, *d_hcnt;     // group -> read, hits per read (list mode of the survivor kernel)
    // last submit
    size_t n_reads; uint32_t n_groups; int do_rc; int in_flight; int used_sieve, used_lists;
    uint64_t launches;
    // device-side framing
    uint32_t *d_nl, *d_blk, *d_frame_err, *h_frame_err; int framed_on_device;
    uint32_t *d_frame_info;                                        // [0] newlines of the chunk, [1] NUL seen
    uint32_t *d_dims, *h_dims; const uint32_t *dims_dev;           // [0] records, [1] position groups of the batch as the device derived them
    size_t nl_cap;                                                 // entries of d_nl
    // FASTQ input (utb_batch_set_input): per read the offset of its quality line; min_qual > 0 masks low-quality bases
    int fastq; uint32_t min_qual;
    uint64_t *h_qual_off, *d_qual_off;
    // wrapped FASTA (utb_batch_set_input): pack_kernel reads the joined sequence bytes d_join instead of d_raw; a
    // host-framed batch brings them in h_join.  Device framing: per 64-byte tile last line start, line in force,
    // header count, first record, sequence-byte count, join offset (d_wt, 6 x wt_cap) and sequence-byte mask
    int wrapped; const uint8_t *d_pack;                            // pack_kernel's input: d_raw, or d_join
    char *h_join; uint8_t *d_join;
    uint32_t *d_wt, *d_wsums, *d_wtotal; uint64_t *d_kmask; size_t wt_cap;
};

extern "C" uint64_t utb_read_slots(uint32_t len) { return ((uint64_t)len + 1 + 31) / 32; }
extern "C" uint64_t utb_batch_max_slots(const utb_batch *b) { return b->max_groups; }
extern "C" char *utb_batch_bytes(utb_batch *b) { return b->h_bytes; }
extern "C" uint64_t *utb_batch_seq_off(utb_batch *b) { return b->h_seq_off; }
extern "C" uint32_t *utb_batch_seq_len(utb_batch *b) { return b->h_seq_len; }
extern "C" size_t utb_batch_max_bytes(const utb_batch *b) { return b->max_bytes; }
extern "C" size_t utb_batch_max_reads(const utb_batch *b) { return b->max_reads; }

extern "C" void utb_batch_destroy(utb_batch *b) {
    if (!b) return;
    cudaSetDevice(b->db->device);
    if (b->st) cudaStreamSynchronize(b->st);
    cudaFreeHost(b->h_bytes); cudaFreeHost(b->h_seq_off); cudaFreeHost(b->h_seq_len); cudaFreeHost(b->h_grp_off);
    cudaFreeHost(b->h_results); cudaFreeHost(b->h_counters);
    cudaFreeHost(b->h_name_off); cudaFreeHost(b->h_name_len); cudaFreeHost(b->h_text); cudaFreeHost(b->h_text_len);
    cudaFree(b->d_name_off); cudaFree(b->d_name_len); cudaFree(b->d_line_len); cudaFree(b->d_line_off); cudaFree(b->d_scan_sums);
    cudaFree(b->d_text_len); cudaFree(b->d_text);
    cudaFree(b->d_raw); cudaFree(b->d_seq_off); cudaFree(b->d_seq_len); cudaFree(b->d_grp_off);
    cudaFree(b->d_pk); cudaFree(b->d_bad); cudaFree(b->d_hits); cudaFree(b->d_results); cudaFree(b->d_pl);
    cudaFree(b->d_gen_list); cudaFree(b->d_gen_count); cudaFree(b->d_warp_list); cudaFree(b->d_warp_count); cudaFree(b->d_counters);
    vs_free(&b->vs);
    cudaFree(b->d_sel_cnt); cudaFree(b->d_sel_off); cudaFree(b->d_sel); cudaFree(b->d_sel_gap); cudaFree(b->d_sel_total);
    cudaFreeHost(b->h_sel_cnt); cudaFreeHost(b->h_sel); cudaFreeHost(b->h_sel_total);
    cudaFree(b->d_qwords); cudaFree(b->d_qslots); cudaFree(b->d_qcount); cudaFree(b->d_hitmap); cudaFree(b->d_rid); cudaFree(b->d_hcnt);
    cudaFree(b->d_nl); cudaFree(b->d_blk); cudaFree(b->d_frame_err); cudaFreeHost(b->h_frame_err);
    cudaFree(b->d_frame_info); cudaFree(b->d_dims); cudaFreeHost(b->h_dims);
    cudaFreeHost(b->h_qual_off); cudaFree(b->d_qual_off);
    cudaFreeHost(b->h_join); cudaFree(b->d_join); cudaFree(b->d_wt); cudaFree(b->d_wsums); cudaFree(b->d_wtotal); cudaFree(b->d_kmask);
    if (b->done) cudaEventDestroy(b->done);
    for (int i = 0; i < 7; ++i) if (b->ev[i]) cudaEventDestroy(b->ev[i]);
    if (b->st) cudaStreamDestroy(b->st);
    free(b);
}

extern "C" int utb_batch_create(utb_db *db, size_t max_bytes, size_t max_reads, utb_batch **out) {
    if (!db || !out || !max_bytes || !max_reads) { utb_set_error("utb_batch_create: bad argument"); return UTB_ERR_ARG; }
    *out = nullptr;
    if (max_bytes + 32 * max_reads >= ((uint64_t)1 << 32) - 4096) {
        utb_set_error("batch too large: positions must fit 32 bits"); return UTB_ERR_LIMIT;
    }
    CK(cudaSetDevice(db->device));
    utb_batch *b = (utb_batch *)calloc(1, sizeof(utb_batch));
    if (!b) { utb_set_error("out of memory"); return UTB_ERR_NOMEM; }
    b->db = db; b->max_bytes = max_bytes; b->max_reads = max_reads;
    // every read owns ceil((len+1)/32) <= len/32 + 1 groups
    b->max_groups = max_bytes / 32 + max_reads + 1;
    size_t npos = (size_t)b->max_groups * 32;
#define BK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { utb_set_error("CUDA error %s at %s:%d (%s)", cudaGetErrorName(e_), __FILE__, __LINE__, cudaGetErrorString(e_)); utb_batch_destroy(b); return UTB_ERR_CUDA; } } while (0)
    BK(cudaStreamCreateWithFlags(&b->st, cudaStreamNonBlocking));
    BK(cudaEventCreateWithFlags(&b->done, cudaEventDisableTiming));
    for (int i = 0; i < 7; ++i) BK(cudaEventCreate(&b->ev[i]));
    BK(cudaMallocHost(&b->h_bytes, max_bytes + 64));
    BK(cudaMallocHost(&b->h_seq_off, max_reads * 8));
    BK(cudaMallocHost(&b->h_seq_len, max_reads * 4));
    BK(cudaMallocHost(&b->h_grp_off, (max_reads + 1) * 4));
    BK(cudaMallocHost(&b->h_results, max_reads * sizeof(utb_result)));
    BK(cudaMallocHost(&b->h_counters, 4 * COUNTER_SLOTS * 8));
    BK(cudaMallocHost(&b->h_name_off, (max_reads + 1) * 4));
    BK(cudaMallocHost(&b->h_name_len, (max_reads + 1) * 4));
    BK(cudaMallocHost(&b->h_text_len, 4));
    BK(cudaMalloc(&b->d_name_off, (max_reads + 1) * 4));
    BK(cudaMalloc(&b->d_name_len, (max_reads + 1) * 4));
    BK(cudaMalloc(&b->d_line_len, (max_reads + 1) * 4));
    BK(cudaMalloc(&b->d_line_off, (max_reads + 1) * 4));
    BK(cudaMalloc(&b->d_scan_sums, (max_reads / SCAN_TILE + 2) * 4));
    BK(cudaMalloc(&b->d_text_len, 4));
    BK(cudaMalloc(&b->d_dims, 8));
    BK(cudaMallocHost(&b->h_dims, 8));
    BK(cudaMalloc(&b->d_raw, max_bytes + 128));
    BK(cudaMalloc(&b->d_seq_off, max_reads * 8));
    BK(cudaMalloc(&b->d_seq_len, max_reads * 4));
    BK(cudaMalloc(&b->d_grp_off, (max_reads + 1) * 4));
    BK(cudaMalloc(&b->d_pk, (b->max_groups + PK_GUARD + 2) * 8));
    BK(cudaMalloc(&b->d_bad, (b->max_groups + PK_GUARD + 2) * 4));
    BK(cudaMalloc(&b->d_hits, npos * 2 * 4));
    BK(cudaMalloc(&b->d_results, max_reads * sizeof(utb_result)));
    BK(cudaMalloc(&b->d_gen_list, max_reads * 4));
    BK(cudaMalloc(&b->d_gen_count, 4));
    BK(cudaMalloc(&b->d_warp_list, max_reads * 4));
    BK(cudaMalloc(&b->d_warp_count, 4));
    BK(cudaMalloc(&b->d_counters, 4 * COUNTER_SLOTS * 8));
    if (vs_alloc(db, max_bytes, &b->vs)) { utb_batch_destroy(b); return UTB_ERR_CUDA; }
    BK(cudaMemset(b->d_raw, 0, max_bytes + 128));
    b->d_pack = b->d_raw;
    if (db->sieve) {                                               // queue for a quarter of the lookup slots; overflow resolves inline
        b->q_cap = npos * 2 / 4 + 4096;
        const char *qc = getenv("UTB_QCAP");                       // tests: a tiny queue forces the overflow path
        if (qc && atoll(qc) > 0) b->q_cap = (uint64_t)atoll(qc);
        b->q_cap = (b->q_cap + Q_CHUNK - 1) / Q_CHUNK * Q_CHUNK;    // whole chunks: the consumer reads [0, min(count, cap)) and every entry of it is written
        BK(cudaMalloc(&b->d_qwords, b->q_cap * 8));
        BK(cudaMalloc(&b->d_qslots, b->q_cap * 4));
        BK(cudaMemset(b->d_qslots, 0xFF, b->q_cap * 4));            // Q_INVALID
        BK(cudaMalloc(&b->d_qcount, 8));
        BK(cudaMalloc(&b->d_hitmap, (npos * 2 / 32 + 8) * 4));
        BK(cudaMalloc(&b->d_pl, (b->max_groups + PK_GUARD + 2) * 8));
        BK(cudaMalloc(&b->d_rid, (b->max_groups + PK_GUARD + 2) * 4));
        BK(cudaMalloc(&b->d_hcnt, (max_reads + 1) * 4));
    }
    if (db->l2_window) {
        cudaStreamAttrValue a;
        memset(&a, 0, sizeof a);
        a.accessPolicyWindow.base_ptr = db->binix;
        a.accessPolicyWindow.num_bytes = db->l2_window_bytes;
        a.accessPolicyWindow.hitRatio = db->l2_hit_ratio;
        a.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        a.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        if (cudaStreamSetAttribute(b->st, cudaStreamAttributeAccessPolicyWindow, &a) != cudaSuccess) cudaGetLastError();
    }
#undef BK
    *out = b;
    return UTB_OK;
}

// grid of a grid-stride kernel: enough CTAs for n items of `per` each, at most `waves` CTAs per SM
static unsigned gs_grid(const utb_batch *b, uint64_t n, uint32_t per, unsigned waves) {
    const uint64_t need = (n + per - 1) / per, cap = (uint64_t)b->db->sm_count * waves;
    return (unsigned)(need < cap ? (need ? need : 1) : cap);
}

// launches the device stages on b->st; if timed, records ev[0..4] around them
static int launch_stages(utb_batch *b, bool timed) {
    const DevDB &d = b->db->d;
    const uint32_t n_reads = (uint32_t)b->n_reads, n_groups = b->n_groups;
    const uint32_t n_pos = n_groups * 32u;
    const uint32_t nstr = b->do_rc ? 2u : 1u;
    CK(cudaMemsetAsync(b->d_gen_count, 0, 4, b->st));
    CK(cudaMemsetAsync(b->d_counters, 0, 4 * COUNTER_SLOTS * 8, b->st));
    // sieve on while misses dominate (it only adds a fetch to lookups that hit)
    const bool sieve = b->db->sieve && (b->db->sieve_mode == 1 || (b->db->sieve_mode == 2 && b->db->ema_hit_rate < 0.40));
    const bool two_phase = b->db->use_table && sieve;              // the sieve kernel reads pl; everything else reads pk
    if (timed) CK(cudaEventRecord(b->ev[0], b->st));
    if (n_reads) {
        const unsigned grid = gs_grid(b, (uint64_t)n_groups + PK_GUARD, 256, 32);
        if (!two_phase) pack_kernel<true, false><<<grid, 256, 0, b->st>>>(b->d_pack, b->d_seq_off, b->d_seq_len, b->d_grp_off,
                                                                        n_reads, n_groups, b->dims_dev, b->d_pk, b->d_bad, nullptr, b->d_rid);
        else if (b->out == UTB_OUT_SELECTIONS) pack_kernel<true, true><<<grid, 256, 0, b->st>>>(b->d_pack, b->d_seq_off, b->d_seq_len, b->d_grp_off,
                                                                        n_reads, n_groups, b->dims_dev, b->d_pk, b->d_bad, b->d_pl, b->d_rid);
        else pack_kernel<false, true><<<grid, 256, 0, b->st>>>(b->d_pack, b->d_seq_off, b->d_seq_len, b->d_grp_off,
                                                             n_reads, n_groups, b->dims_dev, nullptr, b->d_bad, b->d_pl, b->d_rid);
        b->launches++;
    }
    if (timed) CK(cudaEventRecord(b->ev[1], b->st));
    if (n_pos) {
        const unsigned nb = (unsigned)(((uint64_t)n_pos * nstr + 255) / 256);
        const unsigned sms = (unsigned)b->db->sm_count;
        b->used_sieve = sieve; b->used_lists = 0;
        if (two_phase) {
            CK(cudaMemsetAsync(b->d_qcount, 0, 8, b->st));
            // hits are sparse (only sieve survivors that really match).  GG path: the survivor kernel files every label
            // under its read (list mode, see HitSink); non-GG path: by slot, flagged in a 1-bit-per-slot map
            HitSink sink;
            sink.hits = b->d_hits; sink.sh = nstr == 2 ? 6u : 5u;
            const bool lists = b->out != UTB_OUT_SELECTIONS;
            if (lists) { sink.hitmap = nullptr; sink.rid = b->d_rid; sink.grp_off = b->d_grp_off; sink.cnt = b->d_hcnt;
                         CK(cudaMemsetAsync(b->d_hcnt, 0, ((size_t)n_reads + 1) * 4, b->st)); }
            else { sink.hitmap = b->d_hitmap; sink.rid = nullptr; sink.grp_off = nullptr; sink.cnt = nullptr;
                   CK(cudaMemsetAsync(b->d_hitmap, 0, ((size_t)n_pos * nstr / 32 + 4) * 4, b->st)); }
            b->used_lists = lists;
            if (timed) CK(cudaEventRecord(b->ev[4], b->st));
            // persistent: MINB CTAs per SM, every warp a contiguous range of steps (small batches: one tile per warp)
            // measured on B200 (1000 W), 10 M x 150 bp, windows from bit planes (profiles/r03_bench_l2s_*): U = 6 steps per
            // tile at 3 CTAs per SM (80 registers, no spills) 7.86 ms; (6, 4) 7.98 (64 registers, 88 B spilled); (8, 3)
            // 8.03 (32 B spilled).  Before, from 2-bit words (r02_sieve_variants.txt): (6, 3) 8.54; (5, 3) 8.60; (4, 3)
            // 8.81; (4, 4) 8.98; (6, 2) 9.66 -- instructions per step, not occupancy, decide
            constexpr unsigned U = 6, MINB = 3;
            const unsigned wb = (n_groups + 8u * U - 1) / (8u * U);
            const unsigned pb = wb < sms * MINB ? (wb ? wb : 1u) : sms * MINB;
            const uint32_t *sv_groups = b->dims_dev ? b->dims_dev + 1 : nullptr;
            if (nstr == 2) sieve_kernel<2, U, MINB><<<pb, 256, 0, b->st>>>(d, b->d_pl, b->d_bad, n_pos, sv_groups, b->d_counters, b->d_qwords, b->d_qslots, b->d_qcount, b->q_cap, sink);
            else sieve_kernel<1, U, MINB><<<pb, 256, 0, b->st>>>(d, b->d_pl, b->d_bad, n_pos, sv_groups, b->d_counters, b->d_qwords, b->d_qslots, b->d_qcount, b->q_cap, sink);
            if (timed) CK(cudaEventRecord(b->ev[5], b->st));
            if (lists) queue_lookup_kernel<true><<<sms * 6, 256, 0, b->st>>>(d, b->d_qwords, b->d_qslots, b->d_qcount, b->q_cap, sink, b->d_counters);
            else queue_lookup_kernel<false><<<sms * 6, 256, 0, b->st>>>(d, b->d_qwords, b->d_qslots, b->d_qcount, b->q_cap, sink, b->d_counters);
            b->launches++;
        } else if (b->db->use_table) {
            if (nstr == 2) lookup_kernel<2, true><<<nb, 256, 0, b->st>>>(d, b->d_pk, b->d_bad, n_pos, b->dims_dev ? b->dims_dev + 1 : nullptr, b->d_hits, b->d_counters);
            else lookup_kernel<1, true><<<nb, 256, 0, b->st>>>(d, b->d_pk, b->d_bad, n_pos, b->dims_dev ? b->dims_dev + 1 : nullptr, b->d_hits, b->d_counters);
        } else {
            if (nstr == 2) lookup_kernel<2, false><<<nb, 256, 0, b->st>>>(d, b->d_pk, b->d_bad, n_pos, b->dims_dev ? b->dims_dev + 1 : nullptr, b->d_hits, b->d_counters);
            else lookup_kernel<1, false><<<nb, 256, 0, b->st>>>(d, b->d_pk, b->d_bad, n_pos, b->dims_dev ? b->dims_dev + 1 : nullptr, b->d_hits, b->d_counters);
        }
        b->launches++;
    }
    if (timed) CK(cudaEventRecord(b->ev[2], b->st));
    if (n_reads && b->out == UTB_OUT_SELECTIONS) {
        // non-GG mode: no vote on the device (it depends on the order of the reads, itree.c:982); the ids the
        // reference's skipping slide would have collected, per read, compacted: count -> scan -> fill
        VoteIn in;
        in.hits = b->d_hits; in.grp_off = b->d_grp_off; in.seq_len = b->d_seq_len; in.off = nullptr; in.nstr = nstr;
        in.hitmap = b->used_sieve ? b->d_hitmap : nullptr;
        const uint32_t nt = (n_reads + SCAN_TILE - 1) / SCAN_TILE;
        shallow_select_kernel<<<gs_grid(b, n_reads, 128, 32), 128, 0, b->st>>>(d, in, b->d_pk, b->d_bad, n_reads, b->dims_dev, b->d_sel_cnt, b->d_sel_gap);
        scan_sums_kernel<false><<<gs_grid(b, nt, 1, 8), 256, 0, b->st>>>(b->d_sel_cnt, n_reads, b->dims_dev, nt, b->d_scan_sums);
        scan_top_kernel<false><<<1, 1024, 0, b->st>>>(b->d_scan_sums, nt, b->d_sel_total);
        scan_apply_kernel<false><<<gs_grid(b, nt, 1, 8), 256, 0, b->st>>>(b->d_sel_cnt, n_reads, b->dims_dev, nt, b->d_scan_sums, b->d_sel_off);
        shallow_compact_kernel<<<gs_grid(b, n_reads, 128, 32), 128, 0, b->st>>>(in, n_reads, b->dims_dev, b->d_sel_cnt, b->d_sel_off, b->d_sel_gap, b->d_sel);
        b->launches += 5;
    } else if (n_reads) {
        VoteIn in;
        in.hits = b->d_hits; in.grp_off = b->d_grp_off; in.seq_len = b->d_seq_len; in.off = nullptr; in.nstr = nstr;
        in.cnt = b->used_lists ? b->d_hcnt : nullptr;
        if (in.cnt) {
            // thread per read for the common case; label-rich or long reads fall through to the warp kernel
            // (and from there to the block kernel) by way of device-side lists
            CK(cudaMemsetAsync(b->d_warp_count, 0, 4, b->st));
            vote_thread_kernel<<<gs_grid(b, n_reads, VT_THREADS, 32), VT_THREADS, 0, b->st>>>(
                d, in, n_reads, b->dims_dev, b->d_results, b->d_warp_list, b->d_warp_count, b->d_counters);
            vote_warp_kernel<<<(unsigned)b->db->sm_count * 6, VW_WARPS * 32, 0, b->st>>>(
                d, in, n_reads, b->dims_dev, b->d_warp_list, b->d_warp_count, b->d_results, b->d_gen_list, b->d_gen_count, b->d_counters);
            b->launches++;
        } else
            vote_warp_kernel<<<gs_grid(b, n_reads, VW_WARPS, 32), VW_WARPS * 32, 0, b->st>>>(
                d, in, n_reads, b->dims_dev, nullptr, nullptr, b->d_results, b->d_gen_list, b->d_gen_count, b->d_counters);
        int rv = launch_long_vote(b->db, in, b->d_results, b->d_gen_list, b->d_gen_count, &b->vs, b->d_counters, b->st);
        if (rv) return rv;
        b->launches += 4;
    }
    if (timed) CK(cudaEventRecord(b->ev[3], b->st));
    CK(cudaGetLastError());
    return UTB_OK;
}

// Text buffers (the device-resident measurement batches never format): d_text holds the worst case (every read
// prints its name and the longest label); the page-locked staging h_text, through which file sinks take the text
// piece by piece, is sized for the typical output (about half the input) -- page-locking is the slow part.
static size_t text_bytes(size_t max_bytes, size_t max_reads, size_t max_label) {
    return max_bytes + max_reads * (max_label + 48) + 64;
}
#define TEXT_LIMIT (((size_t)1 << 32) - 1)                         // the format kernels address the text with 32 bits
extern "C" size_t utb_text_max_reads(size_t max_bytes, size_t max_reads, size_t max_label) {
    const size_t fixed = text_bytes(max_bytes, 0, max_label);
    if (fixed > TEXT_LIMIT) return 0;
    const size_t fit = (TEXT_LIMIT - fixed) / (max_label + 48);
    return fit < max_reads ? fit : max_reads;
}
static int ensure_text_buffers(utb_batch *b) {
    if (b->d_text) return UTB_OK;
    const size_t cap = text_bytes(b->max_bytes, b->max_reads, b->db->max_label);
    if (cap > TEXT_LIMIT) { utb_set_error("batch too large for device-side formatting"); return UTB_ERR_LIMIT; }
    const size_t hcap = b->max_bytes / 2 + ((size_t)8 << 20) < cap ? b->max_bytes / 2 + ((size_t)8 << 20) : cap;
    CK(cudaMalloc(&b->d_text, cap));
    CK(cudaMallocHost(&b->h_text, hcap));
    b->text_cap = cap; b->h_text_cap = hcap;
    return UTB_OK;
}
static int ensure_shallow_buffers(utb_batch *b);

static int submit_impl(utb_batch *b, const char *src, size_t n_bytes, size_t n_reads, int do_rc, utb_batch_out out, uint64_t total_groups);
static int finish_submit(utb_batch *b);
extern "C" int utb_batch_submit(utb_batch *b, size_t n_bytes, size_t n_reads, int do_rc) {
    return submit_impl(b, nullptr, n_bytes, n_reads, do_rc, UTB_OUT_RESULTS, 0);
}
// Pipeline-internal variant: `src` (pinned host memory, or NULL for the batch's own staging) holds the raw
// bytes; total_groups != 0 means the caller already summed utb_read_slots() over the reads, so the
// per-read offsets are scanned on the device instead of in a serial host loop.
extern "C" int utb_batch_submit_ex(utb_batch *b, const char *src, size_t n_bytes, size_t n_reads, int do_rc,
                                   utb_batch_out out, uint64_t total_groups) {
    return submit_impl(b, src, n_bytes, n_reads, do_rc, out, total_groups);
}
extern "C" int utb_host_ptr_is_pinned(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return 0; }
    return a.type == cudaMemoryTypeHost;
}
// page-locked host memory visible to every device (the searcher's output arena)
extern "C" int utb_pinned_alloc(size_t n, void **out) {
    if (!out || !n) { utb_set_error("utb_pinned_alloc: bad argument"); return UTB_ERR_ARG; }
    *out = nullptr;
    cudaError_t e = cudaHostAlloc(out, n, cudaHostAllocPortable);
    if (e != cudaSuccess) { cudaGetLastError(); utb_set_error("cannot page-lock %zu bytes (%s)", n, cudaGetErrorString(e)); return UTB_ERR_NOMEM; }
    return UTB_OK;
}
extern "C" void utb_pinned_free(void *p) { if (p) cudaFreeHost(p); }
extern "C" uint32_t *utb_batch_name_off(utb_batch *b) { return b->h_name_off; }
extern "C" uint32_t *utb_batch_name_len(utb_batch *b) { return b->h_name_len; }

// FASTQ with min_qual > 0: low-quality bases of the device copy become 'N' (after grp_off, before pack_kernel)
static int launch_mask(utb_batch *b) {
    const uint32_t thr = 33u + b->min_qual;
    qual_mask_kernel<<<gs_grid(b, (uint64_t)b->n_groups, 256, 32), 256, 0, b->st>>>(
        b->d_raw, b->d_seq_off, b->d_qual_off, b->d_seq_len, b->d_grp_off, (uint32_t)b->n_reads, b->n_groups, b->dims_dev, thr * 0x01010101u);
    b->launches++;
    CK(cudaGetLastError());
    return UTB_OK;
}

static int submit_impl(utb_batch *b, const char *src, size_t n_bytes, size_t n_reads, int do_rc, utb_batch_out out, uint64_t total_groups) {
    if (!b) { utb_set_error("utb_batch_submit: null batch"); return UTB_ERR_ARG; }
    if (n_bytes > b->max_bytes || n_reads > b->max_reads) { utb_set_error("utb_batch_submit: batch over capacity"); return UTB_ERR_LIMIT; }
    CK(cudaSetDevice(b->db->device));
    // position space: read r owns groups [grp_off[r], grp_off[r+1])
    uint64_t g = total_groups;
    if (!total_groups) for (size_t r = 0; r < n_reads; ++r) {
        uint32_t len = b->h_seq_len[r];
        if (len > UTB_MAXSEQ) { utb_set_error("read %zu: %u bases exceeds the 16777214-base limit", r, len); return UTB_ERR_LIMIT; }
        if (b->h_seq_off[r] + len > n_bytes) { utb_set_error("read %zu: sequence outside the batch bytes", r); return UTB_ERR_ARG; }
        b->h_grp_off[r] = (uint32_t)g;
        g += utb_read_slots(len);
    }
    if (g > b->max_groups) { utb_set_error("utb_batch_submit: %llu position groups exceed capacity %llu", (unsigned long long)g, (unsigned long long)b->max_groups); return UTB_ERR_LIMIT; }
    if (g * 32ull * (do_rc ? 2u : 1u) >= 0xFFFFFFFFull) {          // a lookup slot (position x strand) is addressed with 32 bits
        utb_set_error("utb_batch_submit: %llu positions x %d strands exceed the 32-bit slot space", (unsigned long long)(g * 32ull), do_rc ? 2 : 1);
        return UTB_ERR_LIMIT;
    }
    if (!total_groups) b->h_grp_off[n_reads] = (uint32_t)g;
    b->n_reads = n_reads; b->n_groups = (uint32_t)g; b->do_rc = do_rc ? 1 : 0;
    b->out = out; b->dims_dev = nullptr; b->framed_on_device = 0;
    if (out == UTB_OUT_SELECTIONS) {                               // non-GG mode: the names stay with the host framer
        int rt = ensure_shallow_buffers(b);
        if (rt) return rt;
    } else if (out == UTB_OUT_TEXT) {
        int rt = ensure_text_buffers(b);
        if (rt) return rt;
        if (n_reads) {
            CK(cudaMemcpyAsync(b->d_name_off, b->h_name_off, n_reads * 4, cudaMemcpyHostToDevice, b->st));
            CK(cudaMemcpyAsync(b->d_name_len, b->h_name_len, n_reads * 4, cudaMemcpyHostToDevice, b->st));
        }
    }
    b->d_pack = b->wrapped ? b->d_join : b->d_raw;
    if (n_reads) {
        CK(cudaMemcpyAsync(b->d_raw, src ? src : b->h_bytes, n_bytes, cudaMemcpyHostToDevice, b->st));
        if (b->wrapped) {                                          // the host framer joined the sequences back to back
            const uint64_t nj = b->h_seq_off[n_reads - 1] + b->h_seq_len[n_reads - 1];
            if (nj) CK(cudaMemcpyAsync(b->d_join, b->h_join, nj, cudaMemcpyHostToDevice, b->st));
        }
        CK(cudaMemcpyAsync(b->d_seq_off, b->h_seq_off, n_reads * 8, cudaMemcpyHostToDevice, b->st));
        CK(cudaMemcpyAsync(b->d_seq_len, b->h_seq_len, n_reads * 4, cudaMemcpyHostToDevice, b->st));
        if (!total_groups) CK(cudaMemcpyAsync(b->d_grp_off, b->h_grp_off, (n_reads + 1) * 4, cudaMemcpyHostToDevice, b->st));
        else {                                                     // grp_off = exclusive scan of the per-read slot counts
            const uint32_t n = (uint32_t)n_reads, nt = (n + SCAN_TILE - 1) / SCAN_TILE;
            slots_kernel<<<(n + 255) / 256, 256, 0, b->st>>>(b->d_seq_len, n, b->d_line_len);
            scan_sums_kernel<false><<<gs_grid(b, nt, 1, 8), 256, 0, b->st>>>(b->d_line_len, n, nullptr, nt, b->d_scan_sums);
            scan_top_kernel<false><<<1, 1024, 0, b->st>>>(b->d_scan_sums, nt, b->d_text_len);
            scan_apply_kernel<false><<<gs_grid(b, nt, 1, 8), 256, 0, b->st>>>(b->d_line_len, n, nullptr, nt, b->d_scan_sums, b->d_grp_off);
            b->launches += 4;
        }
        if (b->fastq && b->min_qual) {
            CK(cudaMemcpyAsync(b->d_qual_off, b->h_qual_off, n_reads * 8, cudaMemcpyHostToDevice, b->st));
            int rm = launch_mask(b);
            if (rm) return rm;
        }
    }
    return finish_submit(b);
}

// device stages + (text | result records | selections) + counters back to the host, all on the batch's stream
static int finish_submit(utb_batch *b) {
    const size_t n_reads = b->n_reads;                             // device-side framing: an upper bound (the device holds the count)
    int rc = launch_stages(b, true);
    if (rc) return rc;
    if (b->out == UTB_OUT_SELECTIONS) {
        // per-read counts, the total, and (device-framed batches) where the names are; the id list follows in the wait
        if (n_reads) {
            CK(cudaMemcpyAsync(b->h_sel_cnt, b->d_sel_cnt, n_reads * 4, cudaMemcpyDeviceToHost, b->st));
            if (b->dims_dev) {
                CK(cudaMemcpyAsync(b->h_name_off, b->d_name_off, n_reads * 4, cudaMemcpyDeviceToHost, b->st));
                CK(cudaMemcpyAsync(b->h_name_len, b->d_name_len, n_reads * 4, cudaMemcpyDeviceToHost, b->st));
            }
        }
        CK(cudaMemcpyAsync(b->h_sel_total, b->d_sel_total, 4, cudaMemcpyDeviceToHost, b->st));
    } else if (b->out == UTB_OUT_TEXT) {
        // lines built on the device: lengths -> exclusive scan -> one warp per read writes its line
        const uint32_t n = (uint32_t)n_reads, nt = (n + SCAN_TILE - 1) / SCAN_TILE;
        CK(cudaMemsetAsync(b->d_text_len, 0, 4, b->st));
        if (n) {
            fmt_len_kernel<<<gs_grid(b, n, 256, 16), 256, 0, b->st>>>(b->db->d, b->d_results, b->d_name_len, n, b->dims_dev, b->d_line_len);
            scan_sums_kernel<false><<<gs_grid(b, nt, 1, 8), 256, 0, b->st>>>(b->d_line_len, n, b->dims_dev, nt, b->d_scan_sums);
            scan_top_kernel<false><<<1, 1024, 0, b->st>>>(b->d_scan_sums, nt, b->d_text_len);
            scan_apply_kernel<false><<<gs_grid(b, nt, 1, 8), 256, 0, b->st>>>(b->d_line_len, n, b->dims_dev, nt, b->d_scan_sums, b->d_line_off);
            fmt_write_kernel<<<gs_grid(b, n, FW_WARPS, 32), FW_WARPS * 32, 0, b->st>>>(
                b->db->d, b->d_results, b->d_raw, b->d_name_off, b->d_name_len, b->d_line_off, n, b->dims_dev, b->d_text);
            b->launches += 5;
            CK(cudaGetLastError());
        }
        CK(cudaMemcpyAsync(b->h_text_len, b->d_text_len, 4, cudaMemcpyDeviceToHost, b->st));
    } else if (n_reads) CK(cudaMemcpyAsync(b->h_results, b->d_results, n_reads * sizeof(utb_result), cudaMemcpyDeviceToHost, b->st));
    if (b->dims_dev) CK(cudaMemcpyAsync(b->h_dims, b->d_dims, 8, cudaMemcpyDeviceToHost, b->st));
    CK(cudaMemcpyAsync(b->h_counters, b->d_counters, 4 * COUNTER_SLOTS * 8, cudaMemcpyDeviceToHost, b->st));
    CK(cudaEventRecord(b->done, b->st));
    b->in_flight = 1;
    return UTB_OK;
}

// Chunk submit (pipeline-internal): the host has not looked at the bytes beyond cutting the chunk right before
// a line that starts with '>' (or at the end of the input); the chunk is copied to the device, which counts its
// newlines, derives and verifies the record count (frame_setup_kernel), frames every record (frame_parse_kernel),
// searches, and builds the output text.  Nothing is waited for here.  n_reads (host value, 0 = unknown): when
// the caller knows the record count it is only used as the upper bound the grids are sized for.
// utb_batch_frame_error() tells after the wait whether the chunk or one of its records was malformed,
// utb_batch_reads() how many records it held.
static int ensure_chunk_buffers(utb_batch *b) {
    const size_t nl_cap = (b->fastq ? 4 : 2) * b->max_reads + 2;  // lines per record
    if (b->d_nl && b->nl_cap < nl_cap) {                           // a FASTQ batch: grown once, by utb_batch_set_input
        void *q = nullptr;
        CK(cudaMalloc(&q, nl_cap * 4));
        cudaFree(b->d_nl);
        b->d_nl = (uint32_t *)q; b->nl_cap = nl_cap;
    }
    if (b->d_nl) return UTB_OK;
    void *p[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaError_t e = cudaMalloc(&p[0], nl_cap * 4);
    if (e == cudaSuccess) e = cudaMalloc(&p[1], (b->max_bytes / FR_BLOCK + 2) * 4);
    if (e == cudaSuccess) e = cudaMalloc(&p[2], 4);
    if (e == cudaSuccess) e = cudaMalloc(&p[3], 8);
    if (e == cudaSuccess) e = cudaMallocHost(&p[4], 4);
    if (e != cudaSuccess) { for (int i = 0; i < 4; ++i) cudaFree(p[i]); cudaFreeHost(p[4]); CK(e); }
    b->d_nl = (uint32_t *)p[0]; b->d_blk = (uint32_t *)p[1]; b->d_frame_err = (uint32_t *)p[2]; b->d_frame_info = (uint32_t *)p[3];
    b->h_frame_err = (uint32_t *)p[4];
    b->nl_cap = nl_cap;
    return UTB_OK;
}
static int ensure_shallow_buffers(utb_batch *b) {
    if (b->d_sel) return UTB_OK;
    // a kept hit uses up >= 8 text positions: a quarter of the lookup slots is room for every read's ids
    b->sel_cap = (size_t)b->max_groups * 32 * 2 / 4 + 64;
    CK(cudaMalloc(&b->d_sel_gap, b->sel_cap * 4));
    CK(cudaMalloc(&b->d_sel_cnt, (b->max_reads + 1) * 4));
    CK(cudaMalloc(&b->d_sel_off, (b->max_reads + 1) * 4));
    CK(cudaMalloc(&b->d_sel, b->sel_cap * 4));
    CK(cudaMalloc(&b->d_sel_total, 4));
    CK(cudaMemset(b->d_sel_total, 0, 4));
    CK(cudaMallocHost(&b->h_sel_cnt, (b->max_reads + 1) * 4));
    CK(cudaMallocHost(&b->h_sel, b->sel_cap * 4));
    CK(cudaMallocHost(&b->h_sel_total, 4));
    return UTB_OK;
}
// Everything a searcher's batch will need, allocated up front (utb_searcher_create) instead of inside its first search.
extern "C" int utb_batch_prepare(utb_batch *b, utb_batch_out out, int chunked) {
    if (!b) { utb_set_error("utb_batch_prepare: null batch"); return UTB_ERR_ARG; }
    CK(cudaSetDevice(b->db->device));
    int rc = out == UTB_OUT_SELECTIONS ? ensure_shallow_buffers(b) : out == UTB_OUT_TEXT ? ensure_text_buffers(b) : UTB_OK;
    if (!rc && chunked) rc = ensure_chunk_buffers(b);
    return rc;
}
// The input format of the batch's later submits (UTB_INPUT_*; min_qual for FASTQ); allocates what the format needs.
static int ensure_wrapped_buffers(utb_batch *b, int chunked) {
    if (!b->h_join) {
        void *h = nullptr, *d = nullptr;
        cudaError_t e = cudaMallocHost(&h, b->max_bytes + 64);
        if (e == cudaSuccess) e = cudaMalloc(&d, b->max_bytes + 128);   // pack_kernel's over-read, as for d_raw
        if (e == cudaSuccess) e = cudaMemset(d, 0, b->max_bytes + 128);
        if (e != cudaSuccess) { cudaFreeHost(h); cudaFree(d); CK(e); }
        b->h_join = (char *)h; b->d_join = (uint8_t *)d;
    }
    if (!chunked || b->d_wt) return UTB_OK;
    const size_t nt = b->max_bytes / 64 + 2;
    void *p[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaError_t e = cudaMalloc(&p[0], 6 * nt * 4);
    if (e == cudaSuccess) e = cudaMalloc(&p[1], (nt / SCAN_TILE + 2) * 4);
    if (e == cudaSuccess) e = cudaMalloc(&p[2], 8);
    if (e == cudaSuccess) e = cudaMalloc(&p[3], nt * 8);
    if (e != cudaSuccess) { for (int i = 0; i < 4; ++i) cudaFree(p[i]); CK(e); }
    b->d_wt = (uint32_t *)p[0]; b->d_wsums = (uint32_t *)p[1]; b->d_wtotal = (uint32_t *)p[2]; b->d_kmask = (uint64_t *)p[3];
    b->wt_cap = nt;
    return UTB_OK;
}
extern "C" int utb_batch_set_input(utb_batch *b, int format, uint32_t min_qual, int chunked) {
    if (!b || format < UTB_INPUT_FASTA || format > UTB_INPUT_FASTA_WRAPPED || (format != UTB_INPUT_FASTQ && min_qual) || min_qual > 222) {
        utb_set_error("utb_batch_set_input: bad argument"); return UTB_ERR_ARG;
    }
    const int fastq = format == UTB_INPUT_FASTQ;
    CK(cudaSetDevice(b->db->device));
    if (fastq && !b->h_qual_off) {                                 // both arrays or neither
        void *h = nullptr, *d = nullptr;
        cudaError_t e = cudaMallocHost(&h, b->max_reads * 8);
        if (e == cudaSuccess) e = cudaMalloc(&d, b->max_reads * 8);
        if (e != cudaSuccess) { cudaFreeHost(h); cudaFree(d); CK(e); }
        b->h_qual_off = (uint64_t *)h; b->d_qual_off = (uint64_t *)d;
    }
    if (format == UTB_INPUT_FASTA_WRAPPED) { int rw = ensure_wrapped_buffers(b, chunked); if (rw) return rw; }
    const int old_fastq = b->fastq;
    b->fastq = fastq;                                              // ensure_chunk_buffers sizes the newline index by it
    const int rc = chunked ? ensure_chunk_buffers(b) : UTB_OK;     // keeps the old index if the larger one cannot be had
    if (rc) { b->fastq = old_fastq; return rc; }
    b->min_qual = min_qual;
    b->wrapped = format == UTB_INPUT_FASTA_WRAPPED;
    return UTB_OK;
}
extern "C" uint64_t *utb_batch_qual_off(utb_batch *b) { return b->h_qual_off; }
extern "C" char *utb_batch_join(utb_batch *b) { return b->h_join; }
extern "C" int utb_batch_submit_chunk(utb_batch *b, const char *src, size_t n_bytes, size_t n_reads, int do_rc, utb_batch_out out) {
    if (!b || !n_bytes || out == UTB_OUT_RESULTS) { utb_set_error("utb_batch_submit_chunk: bad argument"); return UTB_ERR_ARG; }
    if (n_bytes > b->max_bytes || n_reads > b->max_reads || n_bytes >= 0xFFFFFFFFull) { utb_set_error("utb_batch_submit_chunk: batch over capacity"); return UTB_ERR_LIMIT; }
    CK(cudaSetDevice(b->db->device));
    { int ra = ensure_chunk_buffers(b); if (!ra && b->wrapped) ra = ensure_wrapped_buffers(b, 1); if (ra) return ra; }
    int rt = out == UTB_OUT_SELECTIONS ? ensure_shallow_buffers(b) : ensure_text_buffers(b);
    if (rt) return rt;
    // upper bounds the launches are sized for: every read owns ceil((len+1)/32) <= len/32 + 1 groups
    const size_t n_ub = n_reads ? n_reads : b->max_reads;
    uint64_t g_ub = n_bytes / 32 + n_ub + 1;
    if (g_ub > b->max_groups) g_ub = b->max_groups;
    if (g_ub * 32ull * (do_rc ? 2u : 1u) >= 0xFFFFFFFFull) { utb_set_error("utb_batch_submit_chunk: chunk too large for the 32-bit slot space"); return UTB_ERR_LIMIT; }
    b->n_reads = n_ub; b->n_groups = (uint32_t)g_ub; b->do_rc = do_rc ? 1 : 0;
    b->out = out; b->dims_dev = b->d_dims; b->framed_on_device = 1;
    b->d_pack = b->wrapped ? b->d_join : b->d_raw;
    *b->h_frame_err = FR_ERR_NONE;
    CK(cudaMemcpyAsync(b->d_raw, src ? src : b->h_bytes, n_bytes, cudaMemcpyHostToDevice, b->st));
    CK(cudaMemsetAsync(b->d_frame_err, 0xFF, 4, b->st));
    CK(cudaMemsetAsync(b->d_frame_info, 0, 8, b->st));
    const uint32_t fb = (uint32_t)((n_bytes + FR_BLOCK - 1) / FR_BLOCK), n = (uint32_t)n_ub, nt = (n + SCAN_TILE - 1) / SCAN_TILE;
    if (b->wrapped) {
        const uint32_t T = (uint32_t)((n_bytes + 63) / 64), tt = (T + SCAN_TILE - 1) / SCAN_TILE;
        uint32_t *last_ls = b->d_wt, *ls_in = last_ls + b->wt_cap, *hdr = ls_in + b->wt_cap, *rec0 = hdr + b->wt_cap;
        uint32_t *keep = rec0 + b->wt_cap, *join_off = keep + b->wt_cap;
        wrap_tile_kernel<<<fb, 256, 0, b->st>>>(b->d_raw, n_bytes, T, last_ls, hdr, b->d_frame_err);
        scan_sums_kernel<true><<<gs_grid(b, tt, 1, 8), 256, 0, b->st>>>(last_ls, T, nullptr, tt, b->d_wsums);
        scan_top_kernel<true><<<1, 1024, 0, b->st>>>(b->d_wsums, tt, b->d_wtotal + 1);
        scan_apply_kernel<true><<<gs_grid(b, tt, 1, 8), 256, 0, b->st>>>(last_ls, T, nullptr, tt, b->d_wsums, ls_in);
        scan_sums_kernel<false><<<gs_grid(b, tt, 1, 8), 256, 0, b->st>>>(hdr, T, nullptr, tt, b->d_wsums);
        scan_top_kernel<false><<<1, 1024, 0, b->st>>>(b->d_wsums, tt, b->d_frame_info);          // total headers
        scan_apply_kernel<false><<<gs_grid(b, tt, 1, 8), 256, 0, b->st>>>(hdr, T, nullptr, tt, b->d_wsums, rec0);
        frame_setup_kernel<1><<<1, 1, 0, b->st>>>(b->d_frame_info, (uint32_t)n_ub, b->d_dims, b->d_frame_err);
        wrap_keep_kernel<<<fb, 256, 0, b->st>>>(b->d_raw, n_bytes, T, ls_in, rec0, b->d_dims, b->d_kmask, keep, b->d_name_off, b->d_frame_err);
        scan_sums_kernel<false><<<gs_grid(b, tt, 1, 8), 256, 0, b->st>>>(keep, T, nullptr, tt, b->d_wsums);
        scan_top_kernel<false><<<1, 1024, 0, b->st>>>(b->d_wsums, tt, b->d_wtotal);              // total sequence bytes
        scan_apply_kernel<false><<<gs_grid(b, tt, 1, 8), 256, 0, b->st>>>(keep, T, nullptr, tt, b->d_wsums, join_off);
        wrap_join_kernel<<<fb, 256, 0, b->st>>>(b->d_raw, n_bytes, T, b->d_kmask, join_off, b->d_join);
        wrap_record_kernel<<<gs_grid(b, n, 256, 16), 256, 0, b->st>>>(b->d_raw, n_bytes, b->d_kmask, join_off, b->d_wtotal, n, b->d_dims,
                                                                      b->d_seq_off, b->d_seq_len, b->d_name_off, b->d_name_len, b->d_line_len, b->d_frame_err);
        b->launches += 14;
    } else {
        nl_count_kernel<<<fb, 256, 0, b->st>>>(b->d_raw, n_bytes, b->d_blk, b->d_frame_info + 1);
        scan_top_kernel<false><<<1, 1024, 0, b->st>>>(b->d_blk, fb, b->d_frame_info);       // block counts -> exclusive offsets, total newlines
        if (b->fastq) {
            frame_setup_kernel<4><<<1, 1, 0, b->st>>>(b->d_frame_info, (uint32_t)n_ub, b->d_dims, b->d_frame_err);
            nl_index_kernel<4><<<fb, 256, 0, b->st>>>(b->d_raw, n_bytes, b->d_blk, 0, b->d_dims, b->d_nl);
            frame_parse_fastq_kernel<<<gs_grid(b, n, 256, 16), 256, 0, b->st>>>(b->d_raw, b->d_nl, n, b->d_dims, b->d_seq_off, b->d_seq_len,
                                                                                b->d_qual_off, b->d_name_off, b->d_name_len, b->d_line_len, b->d_frame_err);
        } else {
            frame_setup_kernel<2><<<1, 1, 0, b->st>>>(b->d_frame_info, (uint32_t)n_ub, b->d_dims, b->d_frame_err);
            nl_index_kernel<2><<<fb, 256, 0, b->st>>>(b->d_raw, n_bytes, b->d_blk, 0, b->d_dims, b->d_nl);
            frame_parse_kernel<<<gs_grid(b, n, 256, 16), 256, 0, b->st>>>(b->d_raw, b->d_nl, n, b->d_dims, b->d_seq_off, b->d_seq_len, b->d_name_off,
                                                                          b->d_name_len, b->d_line_len, b->d_frame_err);
        }
        b->launches += 5;
    }
    // grp_off = exclusive scan of the per-read group counts; the total (dims[1]) stays on the device
    scan_sums_kernel<false><<<gs_grid(b, nt, 1, 8), 256, 0, b->st>>>(b->d_line_len, n, b->d_dims, nt, b->d_scan_sums);
    scan_top_kernel<false><<<1, 1024, 0, b->st>>>(b->d_scan_sums, nt, b->d_dims + 1);
    scan_apply_kernel<false><<<gs_grid(b, nt, 1, 8), 256, 0, b->st>>>(b->d_line_len, n, b->d_dims, nt, b->d_scan_sums, b->d_grp_off);
    b->launches += 3;
    CK(cudaGetLastError());
    if (b->fastq && b->min_qual) { int rm = launch_mask(b); if (rm) return rm; }
    CK(cudaMemcpyAsync(b->h_frame_err, b->d_frame_err, 4, cudaMemcpyDeviceToHost, b->st));
    return finish_submit(b);
}
// After the wait of a chunk submit: 0 if the chunk and every record of it were well formed, else 1 with the index
// of the first malformed record and its code (1 no header '>', 2 sequence begins '>', 4 line too long, 7 the
// chunk itself: odd line count, NUL byte, more records than the batch holds).
extern "C" int utb_batch_frame_error(const utb_batch *b, size_t *record, int *code) {
    if (!b || !b->framed_on_device || !b->h_frame_err || *b->h_frame_err == FR_ERR_NONE) return 0;
    if (record) *record = *b->h_frame_err >> 3;
    if (code) *code = (int)(*b->h_frame_err & 7u);
    return 1;
}
// records of the last batch (after the wait)
extern "C" size_t utb_batch_reads(const utb_batch *b) { return b ? b->n_reads : 0; }

extern "C" int utb_batch_wait(utb_batch *b, const utb_result **results) {
    if (!b) { utb_set_error("utb_batch_wait: null batch"); return UTB_ERR_ARG; }
    CK(cudaSetDevice(b->db->device));
    CK(cudaEventSynchronize(b->done));
    if (b->in_flight) {
        uint64_t l = 0, h = 0;
        for (int i = 0; i < COUNTER_SLOTS; ++i) { l += b->h_counters[i]; h += b->h_counters[COUNTER_SLOTS + i]; }
        if (l >= 4096) {                                            // steer the pre-filter: hit rate seen so far
            double r = (double)h / (double)l;
            b->db->ema_hit_rate = b->db->ema_hit_rate < 0 ? r : 0.5 * b->db->ema_hit_rate + 0.5 * r;
        }
    }
    if (b->in_flight && b->dims_dev) b->n_reads = b->h_dims[0];     // device-side framing: the record count arrives with the results
    b->in_flight = 0;
    if (results) *results = b->h_results;
    return UTB_OK;
}

// UTB_OUT_TEXT: blocks until the batch is done; its text (*len bytes) is still on the device.
extern "C" int utb_batch_wait_len(utb_batch *b, size_t *len, uint64_t *good_finds) {
    if (!b || !len) { utb_set_error("utb_batch_wait_len: null argument"); return UTB_ERR_ARG; }
    if (b->out != UTB_OUT_TEXT) { utb_set_error("utb_batch_wait_len: batch was not submitted with the text left on the device"); return UTB_ERR_ARG; }
    int rc = utb_batch_wait(b, nullptr);
    if (rc) return rc;
    *len = *b->h_text_len;
    if (*len > b->text_cap) { utb_set_error("device text overflow"); return UTB_ERR_LIMIT; }
    if (good_finds) { uint64_t g = 0; for (int i = 0; i < COUNTER_SLOTS; ++i) g += b->h_counters[2 * COUNTER_SLOTS + i]; *good_finds = g; }
    return UTB_OK;
}
// UTB_OUT_SELECTIONS (non-GG mode): blocks until the batch is done and the ids its reads selected are in page-locked host
// memory: sel_cnt[r] ids per read, back to back in sel; name_off / name_len: where the read names sit in the raw bytes.
extern "C" int utb_batch_wait_shallow(utb_batch *b, const uint32_t **sel_cnt, const uint32_t **sel, size_t *sel_total,
                                      const uint32_t **name_off, const uint32_t **name_len) {
    if (!b || !sel_cnt || !sel || !sel_total) { utb_set_error("utb_batch_wait_shallow: null argument"); return UTB_ERR_ARG; }
    if (b->out != UTB_OUT_SELECTIONS) { utb_set_error("utb_batch_wait_shallow: batch was not submitted in the non-GG mode"); return UTB_ERR_ARG; }
    int rc = utb_batch_wait(b, nullptr);
    if (rc) return rc;
    const size_t n = b->n_reads ? *b->h_sel_total : 0;
    if (n > b->sel_cap) { utb_set_error("selected-hit list overflow"); return UTB_ERR_LIMIT; }
    if (n) {
        CK(cudaMemcpyAsync(b->h_sel, b->d_sel, n * 4, cudaMemcpyDeviceToHost, b->st));
        CK(cudaStreamSynchronize(b->st));
    }
    *sel_cnt = b->h_sel_cnt; *sel = b->h_sel; *sel_total = n;
    if (name_off) *name_off = b->h_name_off;
    if (name_len) *name_len = b->h_name_len;
    return UTB_OK;
}
// ... and is copied from there straight to its place in the caller's page-locked output (no staging, no host
// memcpy); asynchronous on the batch's stream, i.e. ordered before the slot's next batch.  utb_batch_sync waits.
extern "C" int utb_batch_text_to(utb_batch *b, char *dst, size_t len) {
    if (!b || (!dst && len) || len > b->text_cap) { utb_set_error("utb_batch_text_to: bad argument"); return UTB_ERR_ARG; }
    CK(cudaSetDevice(b->db->device));
    if (len) CK(cudaMemcpyAsync(dst, b->d_text, len, cudaMemcpyDeviceToHost, b->st));
    return UTB_OK;
}
// ... or piece by piece through the batch's own page-locked staging (file sinks): bytes [off, off + *len) of the text,
// *len clipped to the staging size; blocks until they are there.
extern "C" int utb_batch_text_piece(utb_batch *b, size_t off, size_t *len, const char **piece) {
    if (!b || !len || !piece || off > b->text_cap) { utb_set_error("utb_batch_text_piece: bad argument"); return UTB_ERR_ARG; }
    CK(cudaSetDevice(b->db->device));
    if (*len > b->h_text_cap) *len = b->h_text_cap;
    if (off + *len > b->text_cap) { utb_set_error("utb_batch_text_piece: beyond the text"); return UTB_ERR_ARG; }
    if (*len) CK(cudaMemcpyAsync(b->h_text, b->d_text + off, *len, cudaMemcpyDeviceToHost, b->st));
    CK(cudaStreamSynchronize(b->st));
    *piece = b->h_text;
    return UTB_OK;
}
extern "C" int utb_batch_sync(utb_batch *b) {
    if (!b) return UTB_OK;
    CK(cudaSetDevice(b->db->device));
    CK(cudaStreamSynchronize(b->st));
    return UTB_OK;
}

extern "C" int utb_batch_counts(utb_batch *b, uint64_t *lookups, uint64_t *hits) {
    if (!b) { utb_set_error("utb_batch_counts: null batch"); return UTB_ERR_ARG; }
    uint64_t l = 0, h = 0;
    for (int i = 0; i < COUNTER_SLOTS; ++i) { l += b->h_counters[i]; h += b->h_counters[COUNTER_SLOTS + i]; }
    if (lookups) *lookups = l;
    if (hits) *hits = h;
    return UTB_OK;
}

// device-stage milliseconds of the LAST submit (valid after wait): pack, lookup, vote, total
extern "C" int utb_batch_last_ms(utb_batch *b, float ms[4]) {
    if (!b || !ms) { utb_set_error("utb_batch_last_ms: null argument"); return UTB_ERR_ARG; }
    CK(cudaSetDevice(b->db->device));
    for (int i = 0; i < 3; ++i) CK(cudaEventElapsedTime(&ms[i], b->ev[i], b->ev[i + 1]));
    CK(cudaEventElapsedTime(&ms[3], b->ev[0], b->ev[3]));
    return UTB_OK;
}
extern "C" uint64_t utb_batch_launches(const utb_batch *b) { return b ? b->launches : 0; }
// Two-phase detail of the LAST run (valid after wait): ms[0] filter kernel, ms[1] queue kernel (0/0 when the
// single lookup kernel ran); sectors[0] = lookups answered by the filter (one sector per position, both
// strands), sectors[1] = sectors the exact path touched for the survivors.
extern "C" int utb_batch_lookup_detail(utb_batch *b, float ms[2], uint64_t sectors[2]) {
    if (!b || !ms || !sectors) { utb_set_error("utb_batch_lookup_detail: null argument"); return UTB_ERR_ARG; }
    CK(cudaSetDevice(b->db->device));
    ms[0] = ms[1] = 0; sectors[0] = sectors[1] = 0;
    if (!b->used_sieve) {                                         // single lookup kernel: only the table sectors are known
        for (int i = 0; i < COUNTER_SLOTS; ++i) sectors[1] += b->h_counters[3 * COUNTER_SLOTS + i];
        return UTB_OK;
    }
    CK(cudaEventElapsedTime(&ms[0], b->ev[4], b->ev[5]));   // the kernel alone (the hits fill before it is part of the stage)
    CK(cudaEventElapsedTime(&ms[1], b->ev[5], b->ev[2]));
    for (int i = 0; i < COUNTER_SLOTS; ++i) { sectors[0] += b->h_counters[i]; sectors[1] += b->h_counters[3 * COUNTER_SLOTS + i]; }
    return UTB_OK;
}

extern "C" int utb_batch_rerun_device(utb_batch *b, int iters, float ms[4], uint64_t *launches) {
    if (!b || iters < 1) { utb_set_error("utb_batch_rerun_device: bad argument"); return UTB_ERR_ARG; }
    CK(cudaSetDevice(b->db->device));
    CK(cudaStreamSynchronize(b->st));
    float acc[4] = {0, 0, 0, 0};
    uint64_t l0 = b->launches;
    for (int it = 0; it < iters; ++it) {
        int rc = launch_stages(b, true);
        if (rc) return rc;
        CK(cudaMemcpyAsync(b->h_counters, b->d_counters, 4 * COUNTER_SLOTS * 8, cudaMemcpyDeviceToHost, b->st));
        CK(cudaStreamSynchronize(b->st));
        float t[4];
        rc = utb_batch_last_ms(b, t);
        if (rc) return rc;
        for (int i = 0; i < 4; ++i) acc[i] += t[i];
    }
    if (ms) for (int i = 0; i < 4; ++i) ms[i] = acc[i];
    if (launches) *launches = b->launches - l0;
    return UTB_OK;
}

// ---------------------------------------------------------------------------
// C ABI: stage-level entry points for parity tests
// ---------------------------------------------------------------------------
extern "C" int utb_lookup_words(utb_db *db, const uint64_t *words, size_t n, uint32_t *ix) {
    if (!db || (!words && n) || (!ix && n)) { utb_set_error("utb_lookup_words: null argument"); return UTB_ERR_ARG; }
    if (!n) return UTB_OK;
    CK(cudaSetDevice(db->device));
    uint64_t *dw = nullptr; uint32_t *di = nullptr;
    CK(cudaMalloc(&dw, n * 8));
    CK(cudaMalloc(&di, n * 4));
    CK(cudaMemcpy(dw, words, n * 8, cudaMemcpyHostToDevice));
    if (db->use_table) lookup_words_kernel<true><<<(unsigned)((n + 255) / 256), 256>>>(db->d, dw, n, di);
    else lookup_words_kernel<false><<<(unsigned)((n + 255) / 256), 256>>>(db->d, dw, n, di);
    CK(cudaGetLastError());
    CK(cudaMemcpy(ix, di, n * 4, cudaMemcpyDeviceToHost));
    cudaFree(dw); cudaFree(di);
    return UTB_OK;
}

extern "C" int utb_pack_sequence(utb_db *db, const char *seq, uint32_t len, uint64_t *fwd, uint64_t *rc, uint8_t *valid) {
    if (!db || !seq || !fwd || !rc || !valid) { utb_set_error("utb_pack_sequence: null argument"); return UTB_ERR_ARG; }
    if (len > UTB_MAXSEQ) { utb_set_error("sequence too long"); return UTB_ERR_LIMIT; }
    if (!len) return UTB_OK;
    CK(cudaSetDevice(db->device));
    // deliberately misaligned by 1 byte, as sequences are inside a FASTA chunk
    uint32_t n_groups = (uint32_t)utb_read_slots(len), n_pos = n_groups * 32;
    uint8_t *d_raw; uint64_t *d_off, *d_pk, *d_f, *d_r; uint32_t *d_len, *d_grp, *d_bad; uint8_t *d_v;
    CK(cudaMalloc(&d_raw, (size_t)len + 128)); CK(cudaMemset(d_raw, 0, (size_t)len + 128));
    CK(cudaMalloc(&d_off, 8)); CK(cudaMalloc(&d_len, 4)); CK(cudaMalloc(&d_grp, 8));
    CK(cudaMalloc(&d_pk, (size_t)(n_groups + PK_GUARD + 2) * 8)); CK(cudaMalloc(&d_bad, (size_t)(n_groups + PK_GUARD + 2) * 4));
    CK(cudaMalloc(&d_f, (size_t)n_pos * 8)); CK(cudaMalloc(&d_r, (size_t)n_pos * 8)); CK(cudaMalloc(&d_v, n_pos));
    uint64_t off = 1; uint32_t grp[2] = {0, n_groups};
    CK(cudaMemcpy(d_raw + 1, seq, len, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_off, &off, 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_len, &len, 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_grp, grp, 8, cudaMemcpyHostToDevice));
    pack_kernel<true, false><<<(n_groups + PK_GUARD + 255) / 256, 256>>>(d_raw, d_off, d_len, d_grp, 1, n_groups, nullptr, d_pk, d_bad, nullptr, nullptr);
    expand_windows_kernel<<<(n_pos + 255) / 256, 256>>>(d_pk, d_bad, n_pos, d_f, d_r, d_v);
    CK(cudaGetLastError());
    CK(cudaMemcpy(fwd, d_f, (size_t)len * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(rc, d_r, (size_t)len * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(valid, d_v, len, cudaMemcpyDeviceToHost));
    cudaFree(d_raw); cudaFree(d_off); cudaFree(d_len); cudaFree(d_grp); cudaFree(d_pk); cudaFree(d_bad);
    cudaFree(d_f); cudaFree(d_r); cudaFree(d_v);
    return UTB_OK;
}

extern "C" int utb_vote_hits(utb_db *db, const uint32_t *hits, const uint64_t *off, size_t n_reads, utb_result *results) {
    if (!db || !off || !results || (!hits && n_reads && off[n_reads])) { utb_set_error("utb_vote_hits: null argument"); return UTB_ERR_ARG; }
    if (!n_reads) return UTB_OK;
    CK(cudaSetDevice(db->device));
    size_t nh = off[n_reads];
    uint32_t *d_hits, *d_gl, *d_gc; uint64_t *d_off; utb_result *d_res; unsigned long long *d_cnt; vote_scratch vs;
    CK(cudaMalloc(&d_hits, (nh + 1) * 4)); CK(cudaMalloc(&d_off, (n_reads + 1) * 8));
    CK(cudaMalloc(&d_res, n_reads * sizeof(utb_result)));
    CK(cudaMalloc(&d_gl, n_reads * 4)); CK(cudaMalloc(&d_gc, 4)); CK(cudaMalloc(&d_cnt, 4 * COUNTER_SLOTS * 8));
    { int rv = vs_alloc(db, (size_t)nh / 2 + 1, &vs); if (rv) return rv; }
    CK(cudaMemset(d_gc, 0, 4)); CK(cudaMemset(d_cnt, 0, 4 * COUNTER_SLOTS * 8));
    if (nh) CK(cudaMemcpy(d_hits, hits, nh * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_off, off, (n_reads + 1) * 8, cudaMemcpyHostToDevice));
    VoteIn in; in.hits = d_hits; in.grp_off = nullptr; in.seq_len = nullptr; in.off = d_off; in.nstr = 1; in.hitmap = nullptr;
    vote_warp_kernel<<<(unsigned)((n_reads + VW_WARPS - 1) / VW_WARPS), VW_WARPS * 32>>>(db->d, in, (uint32_t)n_reads, nullptr, nullptr, nullptr, d_res, d_gl, d_gc, d_cnt);
    { int rv = launch_long_vote(db, in, d_res, d_gl, d_gc, &vs, d_cnt, 0); if (rv) return rv; }
    CK(cudaMemcpy(results, d_res, n_reads * sizeof(utb_result), cudaMemcpyDeviceToHost));
    cudaFree(d_hits); cudaFree(d_off); cudaFree(d_res); cudaFree(d_gl); cudaFree(d_gc); cudaFree(d_cnt);
    vs_free(&vs);
    return UTB_OK;
}

// Same vote through the representation the batch pipeline uses: per read a list of the labels that hit (misses
// and windowless slots are not in it), and the reads go thread kernel -> warp kernel -> block kernel by way of the
// device-side deferral lists.
extern "C" int utb_vote_hits_sparse(utb_db *db, const uint32_t *hits, const uint64_t *off, size_t n_reads, utb_result *results) {
    if (!db || !off || !results || (!hits && n_reads && off[n_reads])) { utb_set_error("utb_vote_hits_sparse: null argument"); return UTB_ERR_ARG; }
    if (!n_reads) return UTB_OK;
    CK(cudaSetDevice(db->device));
    uint64_t *poff = (uint64_t *)malloc((n_reads + 1) * 8);
    uint32_t *ph = (uint32_t *)malloc((off[n_reads] + 1) * 4);
    if (!poff || !ph) { free(poff); free(ph); utb_set_error("out of memory"); return UTB_ERR_NOMEM; }
    uint64_t tot = 0;
    for (size_t r = 0; r < n_reads; ++r) {
        poff[r] = tot;
        for (uint64_t i = off[r]; i < off[r + 1]; ++i) if (hits[i] < HIT_NOWIN) ph[tot++] = hits[i];
    }
    poff[n_reads] = tot;
    uint32_t *d_hits, *d_gl, *d_gc, *d_wl, *d_wc; uint64_t *d_off; utb_result *d_res; unsigned long long *d_cnt; vote_scratch vs;
    CK(cudaMalloc(&d_hits, (tot + 1) * 4)); CK(cudaMalloc(&d_off, (n_reads + 1) * 8));
    CK(cudaMalloc(&d_res, n_reads * sizeof(utb_result)));
    CK(cudaMalloc(&d_gl, n_reads * 4)); CK(cudaMalloc(&d_gc, 4)); CK(cudaMalloc(&d_wl, n_reads * 4)); CK(cudaMalloc(&d_wc, 4));
    CK(cudaMalloc(&d_cnt, 4 * COUNTER_SLOTS * 8));
    { int rv = vs_alloc(db, (size_t)tot / 2 + 1, &vs); if (rv) return rv; }
    CK(cudaMemset(d_gc, 0, 4)); CK(cudaMemset(d_wc, 0, 4)); CK(cudaMemset(d_cnt, 0, 4 * COUNTER_SLOTS * 8));
    if (tot) CK(cudaMemcpy(d_hits, ph, tot * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_off, poff, (n_reads + 1) * 8, cudaMemcpyHostToDevice));
    free(poff); free(ph);
    VoteIn in; in.hits = d_hits; in.off = d_off; in.nstr = 1;
    vote_thread_kernel<<<(unsigned)((n_reads + VT_THREADS - 1) / VT_THREADS), VT_THREADS>>>(db->d, in, (uint32_t)n_reads, nullptr, d_res, d_wl, d_wc, d_cnt);
    vote_warp_kernel<<<(unsigned)db->sm_count * 6, VW_WARPS * 32>>>(db->d, in, (uint32_t)n_reads, nullptr, d_wl, d_wc, d_res, d_gl, d_gc, d_cnt);
    { int rv = launch_long_vote(db, in, d_res, d_gl, d_gc, &vs, d_cnt, 0); if (rv) return rv; }
    CK(cudaMemcpy(results, d_res, n_reads * sizeof(utb_result), cudaMemcpyDeviceToHost));
    cudaFree(d_hits); cudaFree(d_off); cudaFree(d_res); cudaFree(d_gl); cudaFree(d_gc); cudaFree(d_wl); cudaFree(d_wc);
    cudaFree(d_cnt); vs_free(&vs);
    return UTB_OK;
}

// ---------------------------------------------------------------------------
// C ABI: roofline denominator
// ---------------------------------------------------------------------------
extern "C" int utb_measure_rand32(int device, uint64_t ws_bytes, uint64_t loads, int iters, double *gbs) {
    if (!gbs || ws_bytes < 4096 || iters < 1) { utb_set_error("utb_measure_rand32: bad argument"); return UTB_ERR_ARG; }
    int rc = check_device(device);
    if (rc) return rc;
    CK(cudaSetDevice(device));
    uint8_t *buf; unsigned long long *sink;
    CK(cudaMalloc(&buf, ws_bytes));
    CK(cudaMalloc(&sink, 8));
    CK(cudaMemset(buf, 1, ws_bytes));
    CK(cudaMemset(sink, 0, 8));
    const uint32_t per_thread = 64;
    uint64_t threads = (loads + per_thread - 1) / per_thread;
    uint32_t blocks = (uint32_t)((threads + 255) / 256);
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    double best = 0;
    for (int it = 0; it < iters + 1; ++it) {
        CK(cudaEventRecord(e0));
        rand32_kernel<<<blocks, 256>>>(buf, ws_bytes / 32, per_thread, 0x1234 + it, sink);
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        float ms;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        double g = (double)blocks * 256 * per_thread * 32.0 / (ms * 1e-3) / 1e9;
        if (it > 0 && g > best) best = g;                          // first pass is warm-up
    }
    *gbs = best;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(buf); cudaFree(sink);
    return UTB_OK;
}
