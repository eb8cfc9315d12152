// join.cu — hash join build + probe for sm_100a.
//
// Reference semantics reproduced (bit-exact on address indices and output row order):
//   build : PagesIndex.addPage (M/operator/PagesIndex.java:224-256) keeps every build row; the address
//           index of a row is its global row number.  BigintPagesHash.insertValue
//           (M/operator/join/BigintPagesHash.java:122-141) + ArrayPositionLinks.link
//           (M/operator/join/ArrayPositionLinks.java:45-50): rows with a NULL key are skipped; for
//           duplicate keys the LAST inserted row is the chain head and links to the previous head, so a
//           chain lists its rows in descending row order.
//   probe : JoinProbe.fillCache (M/operator/join/unspilled/JoinProbe.java:112-180) ->
//           BigintPagesHash.getAddressIndex (:184-220): chain head or -1, NULL probe keys -> -1.
//   expand: PageJoiner.joinCurrentPosition / outerJoinCurrentPosition (PageJoiner.java:203-242) and
//           LookupJoinPageBuilder.build (LookupJoinPageBuilder.java:119-160): output rows in probe order,
//           within one probe row in chain order; probe columns first, then build output columns.
//
// B200 design: the table is an open-addressing array of 16-byte slots {int64 key, int32 head} so that one
// probe touches exactly one 32-byte sector; the deterministic "head = highest row" of the sequential
// reference insert order is obtained with atomicMax, and duplicate chains are materialised by a radix sort
// of (slot,row) pairs only when duplicates exist.  Slot placement (mix(key) & mask, linear probing) is not
// observable, only key -> head is.
#include <algorithm>
#include <mutex>

#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "rowkeys.cuh"

namespace {

using tg::KeyCols;

constexpr unsigned long long EMPTY_KEY = 0x8000000000000000ULL;   // INT64_MIN is kept out of the table

struct __align__(16) JoinSlot {
    unsigned long long key;
    int head;
    int pad;
};

enum KeyKind { KEY_INT = 0, KEY_DOUBLE = 1 };

// Slot of a key and the probe sequence.  Slot placement is not observable (only key -> head is).
//   mode 0: mix(key) & mask with linear probing, like the reference (M/operator/join/PagesHash.java:35-51).
//   mode 1: line-local: the 8 keys that share key >> 3 prefer the 8 slots of one 128-byte line (slot = key & 7), the
//           LINES are scattered with the murmur3 finaliser; the probe sequence walks the 8 slots of the line (wrapping
//           inside it) and then does the same in the following line.  Dense / clustered key domains probed in key
//           order turn random sector reads into sequential line reads; random keys behave like mode 0.
//   mode 2: order-preserving lines: line = (key - kmin) >> shift, with shift chosen at build time so that a line expects
//           about four keys; same in-line walk as mode 1.  The table is then laid out in key order: a probe page that arrives in
//           key order (TPC-H clustering; every sender's run after a stable hash exchange) walks the table front to back, whatever
//           subset of the key domain this table holds - after a hash exchange over W ranks a table holds every W-th key or so
//           of its domain, which leaves mode 1 with one useful key per line.  Chosen when the build keys spread evenly enough
//           over [kmin, kmax] (rows that had to leave their home line are counted during the build; too many -> mode 1).
struct JoinGeom {
    unsigned long long mask;   // capacity - 1 (capacity is a power of two, at least one 8-slot line)
    unsigned long long kmin;   // mode 2
    int shift;                 // mode 2
    int mode;
};

__host__ __device__ __forceinline__ unsigned long long join_slot_of(unsigned long long k, const JoinGeom& g)
{
    if (g.mode == 2) return ((((k - g.kmin) >> g.shift) << 3) | (k & 7)) & g.mask;
    if (g.mode == 1) return ((tg::murmur3_mix(k >> 3) << 3) | (k & 7)) & g.mask;
    return tg::murmur3_mix(k) & g.mask;
}

__host__ __device__ __forceinline__ unsigned long long join_next_slot(unsigned long long pos, unsigned long long k, const JoinGeom& g)
{
    if (g.mode != 0) {
        unsigned long long in = (pos + 1) & 7;
        if (in != (k & 7)) return (pos & ~7ULL) | in;
        return ((((pos >> 3) + 1) << 3) | (k & 7)) & g.mask;
    }
    return (pos + 1) & g.mask;
}

// canonical 64-bit join key; returns false when the row can never match (NULL, or NaN under EQUAL)
__device__ __forceinline__ bool join_key(const ColRef& c, int kind, int64_t i, unsigned long long* out)
{
    if (!tg_valid(c.validity, i)) return false;
    int64_t v = tg_load_i64(c, i);
    if (kind == KEY_DOUBLE) {
        unsigned long long u = (unsigned long long)v;
        if ((u << 1) == 0) u = 0;                                            // -0.0 == +0.0
        if ((u & 0x7FFFFFFFFFFFFFFFULL) > 0x7FF0000000000000ULL) return false;  // NaN != NaN
        v = (int64_t)u;
    }
    *out = (unsigned long long)v;
    return true;
}

__global__ void join_table_init_kernel(int4* table, int64_t slots)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int4 empty = make_int4(0, (int)0x80000000, -1, 0);
    for (; i < slots; i += stride) table[i] = empty;
}

// one thread per build row: claim/find the key's slot, head = max(row).  *dup_flag is set when a key repeats.
// moved[0] += rows that left their home line, moved[1] += rows that went more than 8 lines away (layout quality of modes 1 / 2).
// give_up_lines > 0 (a TRIAL geometry): a row that would have to move further than that many lines is not inserted and counted in
// *gave_up, and once more than give_up_limit rows did so the whole pass stops - the host rejects the geometry, so the rest of the
// table is never needed.  (Without the bound a geometry that does not suit the keys - e.g. the dense lines over the random half of an
// order-key domain that a hash exchange leaves on a rank - clusters into chains thousands of lines long: 174 s for 75 M rows, measured.)
__global__ void __launch_bounds__(256) join_build_kernel(ColRef key, int kind, int64_t n, JoinSlot* __restrict__ table, JoinGeom geo,
                                                         int* __restrict__ special_head, int* __restrict__ dup_flag, unsigned int* __restrict__ moved,
                                                         int give_up_lines, unsigned int give_up_limit, unsigned int* __restrict__ gave_up)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned int left_home = 0, went_far = 0;
    for (; i < n; i += stride) {
        if (give_up_lines > 0 && *((volatile unsigned int*)gave_up) > give_up_limit) break;
        unsigned long long k;
        if (!join_key(key, kind, i, &k)) continue;
        if (k == EMPTY_KEY) {
            int old = atomicMax(special_head, (int)i);
            if (old >= 0) *dup_flag = 1;
            continue;
        }
        unsigned long long pos = join_slot_of(k, geo);
        const unsigned long long home = pos >> 3;
        bool placed = true;
        while (true) {
            unsigned long long cur = *((volatile unsigned long long*)&table[pos].key);
            if (cur == EMPTY_KEY) cur = atomicCAS(&table[pos].key, EMPTY_KEY, k);
            if (cur == EMPTY_KEY || cur == k) {
                int old = atomicMax(&table[pos].head, (int)i);
                if (old >= 0) *dup_flag = 1;
                break;
            }
            pos = join_next_slot(pos, k, geo);
            if (give_up_lines > 0 && (((pos >> 3) - home) & (geo.mask >> 3)) > (unsigned long long)give_up_lines) { placed = false; break; }
        }
        if (!placed) { atomicAdd(gave_up, 1u); continue; }
        if (geo.mode != 0 && (pos >> 3) != home) {
            left_home++;
            went_far += (((pos >> 3) - home) & (geo.mask >> 3)) > 8;
        }
    }
    if (geo.mode != 0) {
        for (int off = 16; off > 0; off >>= 1) {
            left_home += __shfl_xor_sync(0xffffffffu, left_home, off);
            went_far += __shfl_xor_sync(0xffffffffu, went_far, off);
        }
        if ((threadIdx.x & 31) == 0 && left_home) { atomicAdd(moved, left_home); atomicAdd(moved + 1, went_far); }
    }
}

// min / max of the non-NULL integer keys of the build side (mode 2 geometry)
__global__ void join_key_range_kernel(ColRef key, int64_t n, long long* __restrict__ minmax)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    long long lo = INT64_MAX, hi = INT64_MIN;
    for (; i < n; i += stride) {
        if (!tg_valid(key.validity, i)) continue;
        long long v = tg_load_i64(key, i);
        if ((unsigned long long)v == EMPTY_KEY) continue;
        lo = v < lo ? v : lo;
        hi = v > hi ? v : hi;
    }
    for (int off = 16; off > 0; off >>= 1) {
        long long a = __shfl_xor_sync(0xffffffffu, lo, off), b = __shfl_xor_sync(0xffffffffu, hi, off);
        lo = a < lo ? a : lo;
        hi = b > hi ? b : hi;
    }
    if ((threadIdx.x & 31) == 0 && lo <= hi) { atomicMin(minmax, lo); atomicMax(minmax + 1, hi); }
}

__device__ __forceinline__ int join_lookup(const JoinSlot* __restrict__ table, JoinGeom geo, unsigned long long k, int special_head)
{
    if (k == EMPTY_KEY) return special_head;
    unsigned long long pos = join_slot_of(k, geo);
    while (true) {
        int4 s = __ldg((const int4*)&table[pos]);
        unsigned long long sk = (unsigned long long)(unsigned int)s.x | ((unsigned long long)(unsigned int)s.y << 32);
        if (sk == k) return s.z;
        if (sk == EMPTY_KEY) return -1;
        pos = join_next_slot(pos, k, geo);
    }
}

// Index-only probe (the headline kernel).  ROWS independent lookups per thread are issued before any is
// consumed so that each thread keeps ROWS random 16-byte sector reads in flight; consecutive probe rows with
// the same key (TPC-H clustering) collapse in the coalescer / L1.
// Algorithmic bytes per probe row: 8 (key) + 12 (slot) + 4 (position) = 24 (SURVEY.md §8d).
template <int ROWS, bool INT64_NO_NULLS>
__global__ void __launch_bounds__(256) join_probe_kernel(ColRef key, int kind, int64_t n, const JoinSlot* __restrict__ table, JoinGeom geo,
                                                         int special_head, int* __restrict__ out)
{
    int64_t tile = (int64_t)blockDim.x * ROWS;
    int64_t tiles = (n + tile - 1) / tile;
    for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
        int64_t base = t * tile + threadIdx.x;
        unsigned long long k[ROWS];
        bool ok[ROWS];
        int4 s[ROWS];
        unsigned long long pos[ROWS];
#pragma unroll
        for (int j = 0; j < ROWS; j++) {
            int64_t i = base + (int64_t)j * blockDim.x;
            ok[j] = false;
            k[j] = 0;
            if (i < n) {
                if (INT64_NO_NULLS) { k[j] = (unsigned long long)__ldg((const long long*)key.data + i); ok[j] = true; }
                else ok[j] = join_key(key, kind, i, &k[j]);
            }
            pos[j] = join_slot_of(k[j], geo);
        }
#pragma unroll
        for (int j = 0; j < ROWS; j++) {
            if (ok[j] && k[j] != EMPTY_KEY) s[j] = __ldg((const int4*)&table[pos[j]]);
            else s[j] = make_int4(0, (int)0x80000000, -1, 0);
        }
        // each row walks its probe sequence on its own (measured alternative: lock-step rounds over the ROWS rows of a
        // thread were ~15 % slower on B200)
#pragma unroll
        for (int j = 0; j < ROWS; j++) {
            int64_t i = base + (int64_t)j * blockDim.x;
            if (i >= n) continue;
            int res = -1;
            if (ok[j]) {
                if (k[j] == EMPTY_KEY) res = special_head;
                else {
                    unsigned long long p = pos[j];
                    int4 cur = s[j];
                    while (true) {
                        unsigned long long sk = (unsigned long long)(unsigned int)cur.x | ((unsigned long long)(unsigned int)cur.y << 32);
                        if (sk == k[j]) { res = cur.z; break; }
                        if (sk == EMPTY_KEY) break;
                        p = join_next_slot(p, k[j], geo);
                        cur = __ldg((const int4*)&table[p]);
                    }
                }
            }
            out[i] = res;
        }
    }
}



struct GatherCols {
    int count;
    int by_slot;
    int elem[4];
    const void* src[4];
    void* dst[4];
};

// Match bitmap of the fused probe kernels: LSB first, bit i = probe row i matched - the Arrow validity layout, so a PROBE_OUTER join hands
// it to the build columns as it is.  Every fused kernel runs 256-thread CTAs over 1024-row tiles, where the j-th row set of a warp (rows
// tile * 1024 + j * 256 + 32 * warp + lane) is 32 consecutive rows: one ballot, one word written by lane 0.  Every lane of the warp must
// call it (a lane without a row votes false).  Returns the number of matches of the word on lane 0, 0 on the other lanes.
__device__ __forceinline__ unsigned int match_bits_word(unsigned int* __restrict__ bits, int64_t tile, int j, bool hit)
{
    const unsigned int w = __ballot_sync(0xffffffffu, hit);
    if ((threadIdx.x & 31) != 0) return 0;
    bits[tile * 32 + j * 8 + (threadIdx.x >> 5)] = w;
    return __popc(w);
}

// Fused probe + build-side gather for the common join shape (no duplicate chains, fixed-width non-null build
// columns): the chain head is looked up and the build payload of the matching row is fetched while the slot is
// still in flight in the same thread, so the positions never make a round trip through HBM before the gather and
// no count/scan pass is needed when every probe row matches (FK -> PK joins).  Misses are counted and marked in the
// match bitmap; the host compacts only when there are any.
template <bool INT64_NO_NULLS>
__global__ void __launch_bounds__(256) join_probe_gather_kernel(ColRef key, int kind, int64_t n, const JoinSlot* __restrict__ table, JoinGeom geo,
                                                                int special_head, GatherCols g, unsigned int* __restrict__ match_bits,
                                                                unsigned long long* __restrict__ match_count)
{
    // g.by_slot: payload arrays are indexed by table slot (special key at index mask + 1), else by build row id
    constexpr int ROWS = 4;      // 256 threads x 4 rows: the 1024-row tiles of match_bits_word
    int64_t tile = (int64_t)blockDim.x * ROWS;
    int64_t tiles = (n + tile - 1) / tile;
    unsigned int matched = 0;
    for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
        int64_t base = t * tile + threadIdx.x;
        unsigned long long k[ROWS];
        bool ok[ROWS];
        int4 s[ROWS];
        unsigned long long pos[ROWS];
        int res[ROWS];
        long long at[ROWS];      // index into the payload arrays
#pragma unroll
        for (int j = 0; j < ROWS; j++) {
            int64_t i = base + (int64_t)j * blockDim.x;
            ok[j] = false;
            k[j] = 0;
            if (i < n) {
                if (INT64_NO_NULLS) { k[j] = (unsigned long long)__ldg((const long long*)key.data + i); ok[j] = true; }
                else ok[j] = join_key(key, kind, i, &k[j]);
            }
            pos[j] = join_slot_of(k[j], geo);
        }
#pragma unroll
        for (int j = 0; j < ROWS; j++) {
            if (ok[j] && k[j] != EMPTY_KEY) s[j] = __ldg((const int4*)&table[pos[j]]);
            else s[j] = make_int4(0, (int)0x80000000, -1, 0);
        }
#pragma unroll
        for (int j = 0; j < ROWS; j++) {
            int r = -1;
            long long where = 0;
            if (ok[j]) {
                if (k[j] == EMPTY_KEY) { r = special_head; where = (long long)geo.mask + 1; }
                else {
                    unsigned long long p = pos[j];
                    int4 cur = s[j];
                    while (true) {
                        unsigned long long sk = (unsigned long long)(unsigned int)cur.x | ((unsigned long long)(unsigned int)cur.y << 32);
                        if (sk == k[j]) { r = cur.z; where = (long long)p; break; }
                        if (sk == EMPTY_KEY) break;
                        p = join_next_slot(p, k[j], geo);
                        cur = __ldg((const int4*)&table[p]);
                    }
                }
            }
            res[j] = r;
            at[j] = g.by_slot ? where : (long long)r;
        }
        // build payload: ROWS x columns independent random loads, then coalesced stores
        for (int c = 0; c < g.count; c++) {
            long long v[ROWS];
#pragma unroll
            for (int j = 0; j < ROWS; j++) {
                v[j] = 0;
                if (res[j] >= 0) {
                    switch (g.elem[c]) {
                        case 8: v[j] = __ldg((const long long*)g.src[c] + at[j]); break;
                        case 4: v[j] = __ldg((const int*)g.src[c] + at[j]); break;
                        case 2: v[j] = __ldg((const short*)g.src[c] + at[j]); break;
                        default: v[j] = __ldg((const signed char*)g.src[c] + at[j]); break;
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < ROWS; j++) {
                int64_t i = base + (int64_t)j * blockDim.x;
                if (i >= n) continue;
                switch (g.elem[c]) {
                    case 8: ((long long*)g.dst[c])[i] = v[j]; break;
                    case 4: ((int*)g.dst[c])[i] = (int)v[j]; break;
                    case 2: ((short*)g.dst[c])[i] = (short)v[j]; break;
                    default: ((signed char*)g.dst[c])[i] = (signed char)v[j]; break;
                }
            }
        }
        // rows past n have res = -1 and vote 0; every lane reaches the ballot
#pragma unroll
        for (int j = 0; j < ROWS; j++) matched += match_bits_word(match_bits, t, j, res[j] >= 0);
    }
    // one atomic per warp
    if ((threadIdx.x & 31) == 0 && matched) atomicAdd(match_count, (unsigned long long)matched);
}

// select predicate over row numbers: bit i of the match bitmap
struct MatchBit {
    const unsigned int* bits;
    __device__ __forceinline__ bool operator()(int32_t i) const { return (bits[i >> 5] >> (i & 31)) & 1u; }
};



// ---- generic join keys (DefaultPagesHash shape: several channels and/or variable width) ---------------------------
// The table is keyed by the 64-bit ROW HASH of the key columns (the reference's DefaultPagesHash also addresses by
// mix(rowHash), M/operator/join/DefaultPagesHash.java:105-122).  Exactness comes from two checks against the real key
// columns: at build time every row must carry the same key as the head of its slot (a 64-bit collision between
// different keys makes the build answer NOT_SUPPORTED so the caller keeps the Java operator), and at probe time a hit
// is kept only when the probe row's key equals the build row's key.
__global__ void join_fingerprint_kernel(KeyCols k, int64_t n, const uint8_t* __restrict__ attempt, long long* __restrict__ fp, uint8_t* __restrict__ is_null)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        bool ok = tg::row_joinable(k, i);
        fp[i] = ok ? (long long)tg::row_hash_attempt(k, i, attempt ? attempt[i] : 0) : 0;
        is_null[i] = ok ? 0 : 1;
    }
}

// build: a row whose key differs from the key of its slot's head row shares the slot's 64-bit hash with another key: it moves on to
// its next hash function (attempt + 1); the table is then rebuilt.  Rows of one key always agree with their head, so chains stay pure.
__global__ void join_verify_build_kernel(KeyCols k, const long long* __restrict__ fp, const uint8_t* __restrict__ fp_validity, int64_t n,
                                         const JoinSlot* __restrict__ table, JoinGeom geo, int special_head, uint8_t* __restrict__ attempt, int* __restrict__ moved)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        if (!tg_valid(fp_validity, i)) continue;
        int head = join_lookup(table, geo, (unsigned long long)fp[i], special_head);
        if (head != (int)i && head >= 0 && !tg::rows_equal_for_join(k, i, k, head)) {
            attempt[i] = (uint8_t)(attempt[i] + 1);
            atomicAdd(moved, 1);
        }
    }
}

// probe, attempt 0: a hit whose key differs is a miss when the build needed one hash function only, else it stays open (-2) for the
// next attempt
__global__ void join_verify_probe_kernel(KeyCols probe, KeyCols build, int64_t n, int more_attempts, int* __restrict__ jp)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        int b = jp[i];
        if (b >= 0 && !tg::rows_equal_for_join(probe, i, build, b)) jp[i] = more_attempts ? -2 : -1;
    }
}

// probe, attempt a >= 1 of the rows still open: look the a-th hash up; an empty slot or the last attempt closes the row as a miss
__global__ void join_probe_retry_kernel(KeyCols probe, KeyCols build, int64_t n, const JoinSlot* __restrict__ table, JoinGeom geo, int special_head, int attempt, int last,
                                        int* __restrict__ jp)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        if (jp[i] != -2) continue;
        int head = join_lookup(table, geo, (unsigned long long)tg::row_hash_attempt(probe, i, attempt), special_head);
        if (head >= 0 && tg::rows_equal_for_join(probe, i, build, head)) jp[i] = head;
        else if (head < 0 || last) jp[i] = -1;
    }
}

// ---- lean probe kernels for the headline shape (BIGINT key without NULLs, whole 1024-row tiles) -------------------
// Same algorithm as join_probe_kernel / join_probe_gather_kernel with the per-row bookkeeping stripped: the layout
// mode is a template parameter, slot indices are 32-bit, there are no bounds or validity checks (the ragged tail and
// every other key shape go through the generic kernels).  ncu showed the generic kernels spending ~215 thread
// instructions per probe row at 44-48 % issue utilisation, i.e. instruction-bound as much as latency-bound.
template <int MODE>
__device__ __forceinline__ unsigned int lean_slot(unsigned long long k, unsigned int mask, unsigned long long kmin, int shift)
{
    if (MODE == 2) return (((unsigned int)((k - kmin) >> shift) << 3) | ((unsigned int)k & 7u)) & mask;
    if (MODE == 1) return (((unsigned int)tg::murmur3_mix(k >> 3) << 3) | ((unsigned int)k & 7u)) & mask;
    return (unsigned int)tg::murmur3_mix(k) & mask;
}

template <int MODE>
__device__ __forceinline__ unsigned int lean_next(unsigned int pos, unsigned int k_low3, unsigned int mask)
{
    if (MODE != 0) {
        unsigned int in = (pos + 1) & 7u;
        return in != k_low3 ? ((pos & ~7u) | in) : (((pos & ~7u) + 8u + k_low3) & mask);
    }
    return (pos + 1) & mask;
}

// persistent-tile kernels: exactly as many CTAs as are co-resident, so that no partial second wave runs at low occupancy
template <class K>
static int lean_grid(tgpu_ctx* ctx, K kernel, int64_t tiles)
{
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, 0) != cudaSuccess || per_sm < 1) per_sm = 4;
    return (int)std::min<int64_t>(tiles, (int64_t)ctx->sm_count * per_sm);
}

// GATHER: the payload columns of g are written and, instead of positions, a match bitmap (see match_bits_word); else out = positions
template <int MODE, bool GATHER, int MINB = 1>
__global__ void __launch_bounds__(256, MINB) join_probe_lean_kernel(const long long* __restrict__ keys, int64_t tiles, const int4* __restrict__ table, unsigned int mask,
                                                              unsigned long long kmin, int shift, int special_head, int* __restrict__ out, GatherCols g,
                                                              unsigned int* __restrict__ match_bits, unsigned long long* __restrict__ match_count)
{
    // the word behind the match counter holds the layout choice of the page (0 = these 16-byte slots; join_probe_locality_kernel decides)
    if (GATHER && *(const volatile int*)(match_count + 1) != 0) return;
    unsigned int matched = 0;
    for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
        const int64_t base = t * 1024 + threadIdx.x;
        unsigned long long k[4];
        unsigned int pos[4];
        int4 s[4];
#pragma unroll
        for (int j = 0; j < 4; j++) k[j] = (unsigned long long)__ldg(keys + base + j * 256);
#pragma unroll
        for (int j = 0; j < 4; j++) pos[j] = lean_slot<MODE>(k[j], mask, kmin, shift);
#pragma unroll
        for (int j = 0; j < 4; j++) s[j] = __ldg(table + pos[j]);
        int res[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const unsigned int klo = (unsigned int)k[j], khi = (unsigned int)(k[j] >> 32);
            int r = -1;
            int4 cur = s[j];
            unsigned int p = pos[j];
            while (true) {
                if ((unsigned int)cur.x == klo && (unsigned int)cur.y == khi) { r = cur.z; break; }
                if (cur.x == 0 && cur.y == (int)0x80000000) break;                 // EMPTY_KEY
                p = lean_next<MODE>(p, klo & 7u, mask);
                cur = __ldg(table + p);
            }
            if (k[j] == EMPTY_KEY) { r = special_head; p = mask + 1u; }
            res[j] = r;
            pos[j] = p;
        }
        if (GATHER) {
#pragma unroll
            for (int c = 0; c < 4; c++) {      // static indices: the parameter struct stays in the constant bank
                if (c >= g.count) break;
                if (g.elem[c] == 8) {
                    long long v[4];
#pragma unroll
                    for (int j = 0; j < 4; j++) v[j] = res[j] >= 0 ? __ldg((const long long*)g.src[c] + (g.by_slot ? (long long)pos[j] : (long long)res[j])) : 0;
#pragma unroll
                    for (int j = 0; j < 4; j++) ((long long*)g.dst[c])[base + j * 256] = v[j];
                }
                else if (g.elem[c] == 4) {
                    int v[4];
#pragma unroll
                    for (int j = 0; j < 4; j++) v[j] = res[j] >= 0 ? __ldg((const int*)g.src[c] + (g.by_slot ? (long long)pos[j] : (long long)res[j])) : 0;
#pragma unroll
                    for (int j = 0; j < 4; j++) ((int*)g.dst[c])[base + j * 256] = v[j];
                }
                else {
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        long long at = g.by_slot ? (long long)pos[j] : (long long)res[j];
                        if (g.elem[c] == 2) ((short*)g.dst[c])[base + j * 256] = res[j] >= 0 ? ((const short*)g.src[c])[at] : (short)0;
                        else ((signed char*)g.dst[c])[base + j * 256] = res[j] >= 0 ? ((const signed char*)g.src[c])[at] : (signed char)0;
                    }
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (GATHER) matched += match_bits_word(match_bits, t, j, res[j] >= 0);
            else out[base + j * 256] = res[j];
        }
    }
    if (GATHER && (threadIdx.x & 31) == 0 && matched) atomicAdd(match_count, (unsigned long long)matched);
}

// launch of the lean probe kernel for the table's layout mode
template <bool GATHER>
static int launch_lean(tgpu_ctx* ctx, const JoinGeom& geo, const long long* keys, int64_t tiles, const int4* table, int special_head, int* out, const GatherCols& g,
                       unsigned int* match_bits, unsigned long long* matches)
{
    const unsigned int mask32 = (unsigned int)geo.mask;
    // 8 CTAs per SM (32 registers): full occupancy is worth more than the registers (measured 4.9 -> 3.4 ms at SF100)
    if (geo.mode == 2) {
        auto k = join_probe_lean_kernel<2, GATHER, 8>;
        TG_LAUNCH(ctx, k, lean_grid(ctx, k, tiles), 256, 0, keys, tiles, table, mask32, geo.kmin, geo.shift, special_head, out, g, match_bits, matches);
    }
    else if (geo.mode == 1) {
        auto k = join_probe_lean_kernel<1, GATHER, 8>;
        TG_LAUNCH(ctx, k, lean_grid(ctx, k, tiles), 256, 0, keys, tiles, table, mask32, 0ULL, 0, special_head, out, g, match_bits, matches);
    }
    else {
        auto k = join_probe_lean_kernel<0, GATHER, 8>;
        TG_LAUNCH(ctx, k, lean_grid(ctx, k, tiles), 256, 0, keys, tiles, table, mask32, 0ULL, 0, special_head, out, g, match_bits, matches);
    }
    return TGPU_OK;
}

// ---- wide slots: key, head and the build payload of the head row in ONE 32-byte sector ------------------------------------------
// A probe page without key locality (the survey's variant B, or any join whose probe side is not clustered on the join key) pays one
// random DRAM sector per array it touches for a row: the 16-byte slot, then one sector per slot-ordered payload column.  The wide table
// holds the same slots at a 32-byte stride with up to two payload cells (8 bytes each) behind key and head, so that a row costs ONE
// random sector whatever the number of payload columns - and one 256-bit load (LDG.E.256) instead of three dependent-address loads.
// On a key-ordered probe page the bytes are the same as slot table + slot-ordered payload arrays, read front to back.
// Built next to the 16-byte table (which the index-only probe, the duplicate chains and every generic kernel keep using).
struct __align__(32) WideSlot {
    unsigned long long key;
    int head;
    int pad;
    unsigned long long cell[2];
};

// LD: 0 = one 256-bit read-only load; 3 = the same with an explicit 64-byte L2 fetch size (LDG...LTC64B); 5 = two 128-bit loads
template <int LD>
__device__ __forceinline__ WideSlot wide_load(const WideSlot* p)
{
    WideSlot w;
    unsigned long long kh;
    if (LD == 3) asm("ld.global.nc.L2::64B.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(w.key), "=l"(kh), "=l"(w.cell[0]), "=l"(w.cell[1]) : "l"(p));
    else if (LD == 5) {
        asm("ld.global.nc.v2.u64 {%0,%1}, [%2];" : "=l"(w.key), "=l"(kh) : "l"(p));
        asm("ld.global.nc.v2.u64 {%0,%1}, [%2+16];" : "=l"(w.cell[0]), "=l"(w.cell[1]) : "l"(p));
    }
    else asm("ld.global.nc.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(w.key), "=l"(kh), "=l"(w.cell[0]), "=l"(w.cell[1]) : "l"(p));
    w.head = (int)(unsigned int)kh;
    w.pad = 0;
    return w;
}

__device__ __forceinline__ unsigned long long wide_cell_of(const void* src, int elem, int row)
{
    switch (elem) {
        case 8: return ((const unsigned long long*)src)[row];
        case 4: return ((const unsigned int*)src)[row];
        case 2: return ((const unsigned short*)src)[row];
        default: return ((const unsigned char*)src)[row];
    }
}

__global__ void join_wide_table_kernel(const JoinSlot* __restrict__ table, int64_t slots, int special_head, const void* __restrict__ src0, int elem0,
                                       const void* __restrict__ src1, int elem1, WideSlot* __restrict__ wide)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i <= slots; i += stride) {
        WideSlot w;
        w.key = i < slots ? table[i].key : EMPTY_KEY;
        w.head = i < slots ? table[i].head : special_head;
        w.pad = 0;
        w.cell[0] = w.head >= 0 && src0 ? wide_cell_of(src0, elem0, w.head) : 0ULL;
        w.cell[1] = w.head >= 0 && src1 ? wide_cell_of(src1, elem1, w.head) : 0ULL;
        wide[i] = w;
    }
}

// same contract as join_probe_lean_kernel<MODE, true>: whole 1024-row tiles of a BIGINT key without NULLs; ROWS rows of a thread are in
// flight together (a tile is 4 rows per thread, taken ROWS at a time)
template <int MODE, int ROWS, int MINB, int LD = 0>
__global__ void __launch_bounds__(256, MINB) join_probe_wide_kernel(const long long* __restrict__ keys, int64_t tiles, const WideSlot* __restrict__ wide, unsigned int mask,
                                                                  unsigned long long kmin, int shift, int special_head, GatherCols g, unsigned int* __restrict__ match_bits,
                                                                  unsigned long long* __restrict__ match_count, const int* __restrict__ layout_choice)
{
    if (layout_choice && *layout_choice == 0) return;      // the page goes through the 16-byte slots
    unsigned int matched = 0;
    for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
#pragma unroll
        for (int h = 0; h < 4; h += ROWS) {
            const int64_t base = t * 1024 + h * 256 + threadIdx.x;
            unsigned long long k[ROWS];
            unsigned int pos[ROWS];
            WideSlot w[ROWS];
#pragma unroll
            for (int j = 0; j < ROWS; j++) k[j] = (unsigned long long)__ldg(keys + base + j * 256);
#pragma unroll
            for (int j = 0; j < ROWS; j++) pos[j] = lean_slot<MODE>(k[j], mask, kmin, shift);
#pragma unroll
            for (int j = 0; j < ROWS; j++) w[j] = wide_load<LD>(wide + pos[j]);
#pragma unroll
            for (int j = 0; j < ROWS; j++) {
                unsigned int p = pos[j];
                int r = -1;
                while (true) {
                    if (w[j].key == k[j]) { r = w[j].head; break; }
                    if (w[j].key == EMPTY_KEY) break;
                    p = lean_next<MODE>(p, (unsigned int)k[j] & 7u, mask);
                    w[j] = wide_load<LD>(wide + p);
                }
                if (k[j] == EMPTY_KEY) {                       // INT64_MIN lives outside the table, in the slot behind the last one
                    r = special_head;
                    if (r >= 0) w[j] = wide_load<LD>(wide + (mask + 1u));
                }
                if (r < 0) { w[j].cell[0] = 0ULL; w[j].cell[1] = 0ULL; }
                w[j].head = r;
            }
#pragma unroll
            for (int c = 0; c < 2; c++) {
                if (c >= g.count) break;
#pragma unroll
                for (int j = 0; j < ROWS; j++) {
                    const unsigned long long v = w[j].cell[c];
                    switch (g.elem[c]) {
                        case 8: ((unsigned long long*)g.dst[c])[base + j * 256] = v; break;
                        case 4: ((unsigned int*)g.dst[c])[base + j * 256] = (unsigned int)v; break;
                        case 2: ((unsigned short*)g.dst[c])[base + j * 256] = (unsigned short)v; break;
                        default: ((unsigned char*)g.dst[c])[base + j * 256] = (unsigned char)v; break;
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < ROWS; j++) matched += match_bits_word(match_bits, t, h + j, w[j].head >= 0);
        }
    }
    if ((threadIdx.x & 31) == 0 && matched) atomicAdd(match_count, (unsigned long long)matched);
}

// Which layout a probe page should read.  A wide slot is 32 bytes, a 16-byte slot plus its slot-ordered payload cells 16 + (payload bytes):
// with less than 16 bytes of payload a probe page that arrives in key order reads fewer bytes from the narrow layout (whole lines are used either
// way), while a page without key locality pays a 32-byte sector per ARRAY it touches and is better off with the wide slot.  256 pairs of
// neighbouring rows, spread over the page, vote: a pair is local when its two slots lie within 8 lines of each other.
// choice: 0 = narrow, 1 = wide.  No host round trip: both probe kernels are launched and the one not chosen returns at once.
template <int MODE>
__global__ void __launch_bounds__(256) join_probe_locality_kernel(const long long* __restrict__ keys, int64_t tiles, unsigned int mask, unsigned long long kmin, int shift,
                                                                  int* __restrict__ layout_choice)
{
    const int64_t at = (tiles * (int64_t)threadIdx.x / 256) * 1024 + (threadIdx.x & 31) * 32;
    const unsigned int a = lean_slot<MODE>((unsigned long long)__ldg(keys + at), mask, kmin, shift);
    const unsigned int b = lean_slot<MODE>((unsigned long long)__ldg(keys + at + 1), mask, kmin, shift);
    const unsigned int d = a > b ? a - b : b - a;
    const int local = __syncthreads_count(d <= 64u);
    if (threadIdx.x == 0) *layout_choice = local * 2 >= 256 ? 0 : 1;
}

static int launch_locality(tgpu_ctx* ctx, const JoinGeom& geo, const long long* keys, int64_t tiles, int* layout_choice)
{
    const unsigned int mask32 = (unsigned int)geo.mask;
    if (geo.mode == 2) TG_LAUNCH(ctx, join_probe_locality_kernel<2>, 1, 256, 0, keys, tiles, mask32, geo.kmin, geo.shift, layout_choice);
    else if (geo.mode == 1) TG_LAUNCH(ctx, join_probe_locality_kernel<1>, 1, 256, 0, keys, tiles, mask32, 0ULL, 0, layout_choice);
    else TG_LAUNCH(ctx, join_probe_locality_kernel<0>, 1, 256, 0, keys, tiles, mask32, 0ULL, 0, layout_choice);
    return TGPU_OK;
}

template <int ROWS, int MINB, int LD = 0>
static int launch_wide_shape(tgpu_ctx* ctx, const JoinGeom& geo, const long long* keys, int64_t tiles, const WideSlot* wide, int special_head, const GatherCols& g,
                             unsigned int* match_bits, unsigned long long* matches, const int* layout_choice)
{
    const unsigned int mask32 = (unsigned int)geo.mask;
    if (geo.mode == 2) {
        auto k = join_probe_wide_kernel<2, ROWS, MINB, LD>;
        TG_LAUNCH(ctx, k, lean_grid(ctx, k, tiles), 256, 0, keys, tiles, wide, mask32, geo.kmin, geo.shift, special_head, g, match_bits, matches, layout_choice);
    }
    else if (geo.mode == 1) {
        auto k = join_probe_wide_kernel<1, ROWS, MINB, LD>;
        TG_LAUNCH(ctx, k, lean_grid(ctx, k, tiles), 256, 0, keys, tiles, wide, mask32, 0ULL, 0, special_head, g, match_bits, matches, layout_choice);
    }
    else {
        auto k = join_probe_wide_kernel<0, ROWS, MINB, LD>;
        TG_LAUNCH(ctx, k, lean_grid(ctx, k, tiles), 256, 0, keys, tiles, wide, mask32, 0ULL, 0, special_head, g, match_bits, matches, layout_choice);
    }
    return TGPU_OK;
}

// rows in flight per thread x CTAs per SM; TGPU_JOIN_WIDE_SHAPE=<rows><ctas> picks one of the built shapes (sweeps)
static int launch_wide(tgpu_ctx* ctx, const JoinGeom& geo, const long long* keys, int64_t tiles, const WideSlot* wide, int special_head, const GatherCols& g,
                       unsigned int* match_bits, unsigned long long* matches, const int* layout_choice)
{
    const char* e = getenv("TGPU_JOIN_WIDE_SHAPE");
    int shape = e ? atoi(e) : 28;
    const char* le = getenv("TGPU_JOIN_WIDE_LOAD");
    int ld = le ? atoi(le) : 3;       // measured on the shuffled SF100 probe: 0 -> 17.87 ms, 3 -> 17.37 ms, 5 -> 19.5 ms
    if (shape == 28 && ld == 3) return launch_wide_shape<2, 8, 3>(ctx, geo, keys, tiles, wide, special_head, g, match_bits, matches, layout_choice);
    if (shape == 28 && ld == 5) return launch_wide_shape<2, 8, 5>(ctx, geo, keys, tiles, wide, special_head, g, match_bits, matches, layout_choice);
    switch (shape) {
        case 18: return launch_wide_shape<1, 8>(ctx, geo, keys, tiles, wide, special_head, g, match_bits, matches, layout_choice);
        case 26: return launch_wide_shape<2, 6>(ctx, geo, keys, tiles, wide, special_head, g, match_bits, matches, layout_choice);
        case 45: return launch_wide_shape<4, 5>(ctx, geo, keys, tiles, wide, special_head, g, match_bits, matches, layout_choice);
        case 44: return launch_wide_shape<4, 4>(ctx, geo, keys, tiles, wide, special_head, g, match_bits, matches, layout_choice);
        default: return launch_wide_shape<2, 8>(ctx, geo, keys, tiles, wide, special_head, g, match_bits, matches, layout_choice);
    }
}

// ---- packed slots: key and the head row's payload in ONE 16-byte entry (one-column builds) -----------------------------------------
// The fused probe needs the head row id only to find the payload.  A build with exactly one fixed-width output column without NULLs and no
// duplicate keys (the FK -> PK shape of every join in the benchmark) therefore gets a table of {key, payload of the head row zero-extended
// to 8 bytes} in the slot geometry of the 16-byte table, with entry `capacity` holding the INT64_MIN key's payload under the key EMPTY_KEY.
// A probe row reads one 16-byte entry - the bytes of the JoinSlot alone - and neither the slot-ordered payload array nor the wide table is
// built for this shape.  The JoinSlot table stays: the index-only probe, the ragged tail and the generic kernels read it.
struct __align__(16) PackedSlot {
    unsigned long long key;
    unsigned long long cell;
};

__global__ void join_packed_table_kernel(const JoinSlot* __restrict__ table, int64_t slots, int special_head, const void* __restrict__ src, int elem,
                                         PackedSlot* __restrict__ packed)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i <= slots; i += stride) {
        const int head = i < slots ? table[i].head : special_head;
        PackedSlot s;
        s.key = i < slots ? table[i].key : EMPTY_KEY;
        s.cell = head >= 0 ? wide_cell_of(src, elem, head) : 0ULL;
        packed[i] = s;
    }
}

// same tile contract as join_probe_lean_kernel<MODE, true>; two rows of a thread are in flight together (a tile is 4 rows per thread,
// taken 2 at a time): 8 CTAs per SM at 32 registers without spills - with 4 rows the key and entry registers alone take 24 of the 32 and
// ptxas spills.  special: the key INT64_MIN has a build row.  A miss writes 0 and a 0 bit.  Row numbers are 32-bit (a page has at most
// 2^31 - 1 rows), and a row's home slot is recomputed from its key on the rare walk past it, so that only key and entry stay live.
template <int MODE>
__global__ void __launch_bounds__(256, 8) join_probe_packed_kernel(const long long* __restrict__ keys, int64_t tiles, const ulonglong2* __restrict__ packed,
                                                                   unsigned int mask, unsigned long long kmin, int shift, int special, void* __restrict__ dst, int elem,
                                                                   unsigned int* __restrict__ match_bits, unsigned long long* __restrict__ match_count)
{
    constexpr int ROWS = 2;
    unsigned int matched = 0;
    for (unsigned int t = blockIdx.x; t < (unsigned int)tiles; t += gridDim.x) {
#pragma unroll 1
        for (int h = 0; h < 4; h += ROWS) {
            const unsigned int base = t * 1024u + h * 256u + threadIdx.x;
            unsigned long long k[ROWS];
            ulonglong2 s[ROWS];
#pragma unroll
            for (int j = 0; j < ROWS; j++) k[j] = (unsigned long long)__ldg(keys + base + j * 256);
#pragma unroll
            for (int j = 0; j < ROWS; j++) s[j] = __ldg(packed + (k[j] == EMPTY_KEY ? mask + 1u : lean_slot<MODE>(k[j], mask, kmin, shift)));
#pragma unroll
            for (int j = 0; j < ROWS; j++) {
                if (s[j].x != k[j] && s[j].x != EMPTY_KEY) {            // the key left its home slot (INT64_MIN's entry always matches)
                    unsigned int p = lean_slot<MODE>(k[j], mask, kmin, shift);
                    do {
                        p = lean_next<MODE>(p, (unsigned int)k[j] & 7u, mask);
                        s[j] = __ldg(packed + p);
                    } while (s[j].x != k[j] && s[j].x != EMPTY_KEY);
                }
                const bool hit = s[j].x == k[j] && (k[j] != EMPTY_KEY || special);
                matched += match_bits_word(match_bits, t, h + j, hit);
                const unsigned long long v = hit ? s[j].y : 0ULL;
                const unsigned int i = base + j * 256;
                switch (elem) {
                    case 8: ((unsigned long long*)dst)[i] = v; break;
                    case 4: ((unsigned int*)dst)[i] = (unsigned int)v; break;
                    case 2: ((unsigned short*)dst)[i] = (unsigned short)v; break;
                    default: ((unsigned char*)dst)[i] = (unsigned char)v; break;
                }
            }
        }
    }
    if ((threadIdx.x & 31) == 0 && matched) atomicAdd(match_count, (unsigned long long)matched);
}

static int launch_packed(tgpu_ctx* ctx, const JoinGeom& geo, const long long* keys, int64_t tiles, const PackedSlot* packed, int special, void* dst, int elem,
                         unsigned int* match_bits, unsigned long long* matches)
{
    const unsigned int mask32 = (unsigned int)geo.mask;
    const ulonglong2* table = (const ulonglong2*)packed;
    if (geo.mode == 2) {
        auto k = join_probe_packed_kernel<2>;
        TG_LAUNCH(ctx, k, lean_grid(ctx, k, tiles), 256, 0, keys, tiles, table, mask32, geo.kmin, geo.shift, special, dst, elem, match_bits, matches);
    }
    else if (geo.mode == 1) {
        auto k = join_probe_packed_kernel<1>;
        TG_LAUNCH(ctx, k, lean_grid(ctx, k, tiles), 256, 0, keys, tiles, table, mask32, 0ULL, 0, special, dst, elem, match_bits, matches);
    }
    else {
        auto k = join_probe_packed_kernel<0>;
        TG_LAUNCH(ctx, k, lean_grid(ctx, k, tiles), 256, 0, keys, tiles, table, mask32, 0ULL, 0, special, dst, elem, match_bits, matches);
    }
    return TGPU_OK;
}

// build payload re-laid out in SLOT order (one pass at build time): the fused probe then reads the payload right next
// to where it found the key instead of chasing the row id into the (arbitrarily ordered) build pages
__global__ void join_payload_by_slot_kernel(const JoinSlot* __restrict__ table, int64_t slots, int special_head, const void* __restrict__ src, int elem,
                                            void* __restrict__ dst)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i <= slots; i += stride) {
        int head = i < slots ? table[i].head : special_head;
        if (head < 0) continue;
        switch (elem) {
            case 8: ((long long*)dst)[i] = ((const long long*)src)[head]; break;
            case 4: ((int*)dst)[i] = ((const int*)src)[head]; break;
            case 2: ((short*)dst)[i] = ((const short*)src)[head]; break;
            default: ((signed char*)dst)[i] = ((const signed char*)src)[head]; break;
        }
    }
}

// --- duplicate chains -------------------------------------------------------------------------------
// sort key = (slot << 32 | row) for rows that are in the table; rows with NULL keys sort last
__global__ void join_slot_of_row_kernel(ColRef key, int kind, int64_t n, const JoinSlot* __restrict__ table, JoinGeom geo,
                                        unsigned long long special_slot, unsigned long long* __restrict__ out)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        unsigned long long k;
        unsigned long long slot = 0xFFFFFFFFULL;
        if (join_key(key, kind, i, &k)) {
            if (k == EMPTY_KEY) slot = special_slot;
            else {
                unsigned long long pos = join_slot_of(k, geo);
                while (table[pos].key != k) pos = join_next_slot(pos, k, geo);
                slot = pos;
            }
        }
        out[i] = (slot << 32) | (unsigned long long)(unsigned int)i;
    }
}

// after the sort rows of one key are adjacent in ascending row order: next(row) = previous row of the key
__global__ void join_links_kernel(const unsigned long long* __restrict__ sorted, int64_t n, int* __restrict__ links)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        unsigned long long cur = sorted[i];
        unsigned int slot = (unsigned int)(cur >> 32);
        int row = (int)(unsigned int)cur;
        int next = -1;
        if (slot != 0xFFFFFFFFu && i > 0) {
            unsigned long long prev = sorted[i - 1];
            if ((unsigned int)(prev >> 32) == slot) next = (int)(unsigned int)prev;
        }
        links[row] = next;
    }
}

// --- expansion --------------------------------------------------------------------------------------
__global__ void join_count_kernel(const int* __restrict__ jp, int64_t n, const int* __restrict__ links, int single_match, int outer,
                                  int* __restrict__ counts)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        int p = jp[i];
        int c = 0;
        if (p >= 0) {
            c = 1;
            if (links && !single_match) {
                p = links[p];
                while (p >= 0) { c++; p = links[p]; }
            }
        }
        else if (outer) c = 1;
        counts[i] = c;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) counts[n] = 0;
}

__global__ void join_fill_kernel(const int* __restrict__ jp, int64_t n, const int* __restrict__ links, int single_match, int outer,
                                 const long long* __restrict__ offsets, int* __restrict__ out_probe, int* __restrict__ out_build)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        int p = jp[i];
        long long o = offsets[i];
        if (p >= 0) {
            out_probe[o] = (int)i;
            out_build[o] = p;
            if (links && !single_match) {
                p = links[p];
                while (p >= 0) { o++; out_probe[o] = (int)i; out_build[o] = p; p = links[p]; }
            }
        }
        else if (outer) {
            out_probe[o] = (int)i;
            out_build[o] = -1;
        }
    }
}

int key_kind_of(int type) { return type == TGPU_FLOAT64 ? KEY_DOUBLE : KEY_INT; }

}  // namespace

// ------------------------------------------------------------------------------------------------
// LookupSource
// ------------------------------------------------------------------------------------------------
struct tgpu_lookup {
    tgpu_ctx* ctx = nullptr;
    int refs = 1;
    int64_t positions = 0;              // build rows (incl. NULL-key rows: PagesIndex keeps them)
    int key_type = 0;
    DevBuf table;                       // JoinSlot[capacity]
    JoinGeom geo = {0, 0, 0, 0};        // capacity - 1, slot placement mode and its parameters
    int special_head = -1;
    bool has_dups = false;
    DevBuf links;                       // int32[positions], only when has_dups
    DevPage store;                      // key column first, then build output columns
    int32_t num_output = 0;
    std::vector<DevBuf> by_slot;        // build output columns in table-slot order (fused probe fast path)
    DevBuf wide;                        // WideSlot[capacity + 1]: slots with the payload of their head row (2 build output columns)
    DevBuf packed;                      // PackedSlot[capacity + 1]: key + payload of the head row (1 build output column; no by_slot, no wide then)
    bool generic = false;               // keyed by row hash + verification against build_keys
    int attempts = 1;                   // generic only: hash functions the build needed (> 1 iff two keys shared a 64-bit hash)
    std::vector<DevColumn> build_keys;  // generic only: the real key columns of the build side
    // OuterPositionTracker (M/operator/join/OuterLookupSource.java:168-196): one byte per build position, set by the
    // LOOKUP_OUTER / FULL_OUTER probes for every build row they emit, read by the LookupOuterOperator
    DevBuf visited;
    std::mutex visited_lock;
    int64_t null_key_rows = -1;         // build rows whose (first) key channel is NULL; -1 = not counted yet
    int64_t nan_key_rows = -1;          // DOUBLE / REAL key: build rows whose key is NaN (members of a semi-join's ChannelSet); -1 = not counted yet
};

namespace {


// row-hash column (+ validity: NULL / NaN keys can never match) of a set of key columns
int make_fingerprint(tgpu_ctx* ctx, const std::vector<const DevColumn*>& keys, int64_t n, DevColumn* out, const uint8_t* d_attempt = nullptr)
{
    KeyCols k;
    memset(&k, 0, sizeof(k));
    if (keys.size() > (size_t)tg::MAX_KEY_COLS) return tg_fail(ctx, TGPU_ERR_NOT_SUPPORTED, "more than %d join channels", tg::MAX_KEY_COLS);
    k.count = (int32_t)keys.size();
    for (size_t c = 0; c < keys.size(); c++) tg::key_cols_set(&k, (int)c, *keys[c]);
    DevColumn fp;
    fp.type = TGPU_INT64;
    fp.length = n;
    fp.own_data = std::make_shared<DevBuf>();
    TG_TRY(fp.own_data->alloc(ctx, (size_t)std::max<int64_t>(n, 1) * 8));
    fp.data = fp.own_data->p;
    DevBuf is_null;
    TG_TRY(is_null.alloc(ctx, (size_t)std::max<int64_t>(n, 1)));
    if (n > 0) {
        TG_LAUNCH(ctx, join_fingerprint_kernel, tg_grid(ctx, n, 256, 8), 256, 0, k, n, d_attempt, fp.own_data->as<long long>(), is_null.as<uint8_t>());
        tgpu_column bm;
        memset(&bm, 0, sizeof(bm));
        bm.type = TGPU_INT8;
        bm.flags = TGPU_COL_NULLS_BYTEMAP;
        bm.length = n;
        bm.data = is_null.p;
        bm.validity = is_null.as<uint8_t>();
        DevColumn packed;
        TG_TRY(tg_ingest_column(ctx, &bm, true, &packed));
        fp.own_validity = packed.own_validity;
        fp.validity = packed.validity;
    }
    *out = std::move(fp);
    return TGPU_OK;
}

KeyCols key_cols_of(const std::vector<DevColumn>& cols)
{
    KeyCols k;
    memset(&k, 0, sizeof(k));
    k.count = (int32_t)cols.size();
    for (size_t c = 0; c < cols.size(); c++) tg::key_cols_set(&k, (int)c, cols[c]);
    return k;
}

int lookup_positions(tgpu_ctx* ctx, const tgpu_lookup* lk, const DevColumn& key, int* d_out)
{
    int64_t n = key.length;
    if (n == 0) return TGPU_OK;
    if (key.type == TGPU_UTF8) return tg_fail(ctx, TGPU_ERR_NOT_SUPPORTED, "variable-width join keys are not supported on the GPU path");
    if (key_kind_of(key.type) != key_kind_of(lk->key_type) || key.elem_size() == 0)
        return tg_fail(ctx, TGPU_ERR_INVALID_ARGUMENT, "probe key type %d does not match build key type %d", key.type, lk->key_type);
    const JoinSlot* table = lk->table.as<JoinSlot>();
    bool fast = key.type == TGPU_INT64 && !key.validity;
    int kind = fast ? KEY_INT : key_kind_of(key.type);
    auto k4f = join_probe_kernel<4, true>;
    auto k4a = join_probe_kernel<4, false>;
    int64_t done = 0;
    TG_TIMED_BEGIN(ctx);
    if (fast && !getenv("TGPU_JOIN_GENERIC_KERNELS")) {
        // whole 1024-row tiles through the lean kernel, the ragged tail through the generic one
        int64_t tiles = n / 1024;
        if (tiles > 0) {
            GatherCols none;
            memset(&none, 0, sizeof(none));
            TG_TRY(launch_lean<false>(ctx, lk->geo, (const long long*)key.data, tiles, (const int4*)table, lk->special_head, d_out, none, nullptr, nullptr));
            done = tiles * 1024;
        }
    }
    if (done < n) {
        ColRef kr = tg_colref(key);
        if (done > 0) kr.data = (const char*)kr.data + done * 8;   // only the fast (INT64, no validity) shape gets here with done > 0
        int grid = tg_grid(ctx, n - done, 256 * 4, 8);
        if (fast) TG_LAUNCH(ctx, k4f, grid, 256, 0, kr, kind, n - done, table, lk->geo, lk->special_head, d_out + done);
        else TG_LAUNCH(ctx, k4a, grid, 256, 0, kr, kind, n - done, table, lk->geo, lk->special_head, d_out + done);
    }
    TG_TIMED_END(ctx);
    return TGPU_OK;
}

// join positions for a generic-key lookup: probe the row hashes, then keep only hits whose key columns really match
int lookup_positions_generic(tgpu_ctx* ctx, const tgpu_lookup* lk, const std::vector<const DevColumn*>& keys, int64_t n, int* d_out)
{
    if (keys.size() != lk->build_keys.size()) return tg_fail(ctx, TGPU_ERR_INVALID_ARGUMENT, "probe has %zu join channels, build has %zu", keys.size(), lk->build_keys.size());
    for (size_t c = 0; c < keys.size(); c++) {
        bool pu = keys[c]->type == TGPU_UTF8, bu = lk->build_keys[c].type == TGPU_UTF8, pd = keys[c]->type == TGPU_FLOAT64, bd = lk->build_keys[c].type == TGPU_FLOAT64;
        bool pr = keys[c]->type == TGPU_FLOAT32, br = lk->build_keys[c].type == TGPU_FLOAT32;
        if (pu != bu || pd != bd || pr != br) return tg_fail(ctx, TGPU_ERR_INVALID_ARGUMENT, "join channel %zu: probe type %d does not match build type %d", c, keys[c]->type, lk->build_keys[c].type);
    }
    if (n == 0) return TGPU_OK;
    DevColumn fp;
    TG_TRY(make_fingerprint(ctx, keys, n, &fp));
    TG_TRY(lookup_positions(ctx, lk, fp, d_out));
    KeyCols pk;
    memset(&pk, 0, sizeof(pk));
    pk.count = (int32_t)keys.size();
    for (size_t c = 0; c < keys.size(); c++) tg::key_cols_set(&pk, (int)c, *keys[c]);
    const KeyCols bk = key_cols_of(lk->build_keys);
    TG_LAUNCH(ctx, join_verify_probe_kernel, tg_grid(ctx, n, 256, 8), 256, 0, pk, bk, n, lk->attempts > 1 ? 1 : 0, d_out);
    for (int a = 1; a < lk->attempts; a++)
        TG_LAUNCH(ctx, join_probe_retry_kernel, tg_grid(ctx, n, 256, 8), 256, 0, pk, bk, n, lk->table.as<JoinSlot>(), lk->geo, lk->special_head, a,
                  a == lk->attempts - 1 ? 1 : 0, d_out);
    return TGPU_OK;
}

// LookupSource.appendTo -> positionVisited for every build row an outer-tracking probe emitted
__global__ void join_mark_visited_kernel(const int* __restrict__ build_idx, int64_t n, uint8_t* __restrict__ visited)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        int b = build_idx[i];
        if (b >= 0) visited[b] = 1;
    }
}

__global__ void join_unvisited_flags_kernel(const uint8_t* __restrict__ visited, int64_t n, uint8_t* __restrict__ flags)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) flags[i] = visited[i] ? 0 : 1;
}

// HashSemiJoinOperator.process :181-199: value and NULL byte of the appended BOOLEAN column
// float_kind: 0 = not a floating-point key, 1 = DOUBLE, 2 = REAL.  The ChannelSet compares with IDENTICAL (M/operator/FlatSet.java:54,374): a NaN
// probe key is in the set iff the set holds a NaN - which the EQUAL-semantics lookup cannot answer (NaN matches nothing there) - while -0.0 / +0.0
// are one member under both
__device__ __forceinline__ bool key_is_nan(const ColRef& key, int float_kind, int64_t i)
{
    if (float_kind == 1) return ((unsigned long long)tg_load_i64(key, i) & 0x7FFFFFFFFFFFFFFFULL) > 0x7FF0000000000000ULL;
    if (float_kind == 2) return ((unsigned int)tg_load_i64(key, i) & 0x7FFFFFFFu) > 0x7F800000u;
    return false;
}

__global__ void count_nan_keys_kernel(ColRef key, int float_kind, int64_t n, unsigned long long* __restrict__ out)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned int mine = 0;
    for (; i < n; i += stride) mine += tg_valid(key.validity, i) && key_is_nan(key, float_kind, i);
    for (int off = 16; off > 0; off >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, off);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(out, (unsigned long long)mine);
}

__global__ void semi_join_kernel(const int* __restrict__ positions, const uint8_t* __restrict__ key_validity, int64_t n, int set_empty, int set_has_null,
                                 signed char* __restrict__ value, uint8_t* __restrict__ is_null, ColRef key, int float_kind, int set_has_nan)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        bool probe_null = !tg_valid(key_validity, i);
        bool contains = positions[i] >= 0;
        if (float_kind && !probe_null && key_is_nan(key, float_kind, i)) contains = set_has_nan != 0;
        bool out_null, v;
        if (probe_null) { out_null = !set_empty; v = false; }
        else if (!contains && set_has_null) { out_null = true; v = false; }
        else { out_null = false; v = contains; }
        value[i] = v ? 1 : 0;
        is_null[i] = out_null ? 1 : 0;
    }
}

__global__ void count_nulls_kernel(const uint8_t* __restrict__ validity, int64_t n, unsigned long long* __restrict__ out)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned int c = 0;
    for (; i < n; i += stride) c += tg_valid(validity, i) ? 0 : 1;
    for (int off = 16; off > 0; off >>= 1) c += __shfl_xor_sync(0xffffffffu, c, off);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, (unsigned long long)c);
}

// DynamicFilterSourceOperator / JoinDomainBuilder: min, max, number of distinct keys and (while they fit) the keys themselves,
// read off the table (one occupied slot per distinct non-NULL key)
__global__ void join_key_domain_kernel(const JoinSlot* __restrict__ table, int64_t slots, int64_t max_values, long long* __restrict__ minmax /* [2] */,
                                       unsigned long long* __restrict__ count, long long* __restrict__ values)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < slots; i += stride) {
        long long k = table[i].key;
        if ((unsigned long long)k == EMPTY_KEY) continue;
        atomicMin(minmax, k);
        atomicMax(minmax + 1, k);
        unsigned long long at = atomicAdd(count, 1ULL);
        if ((long long)at < max_values) values[at] = k;
    }
}

// HashBuilderOperator: NEEDS_INPUT -> (finish) LOOKUP_SOURCE_BUILT -> CLOSED
struct JoinBuildOp : tgpu_op {
    std::vector<int32_t> key_channels, output_channels;
    std::vector<DevPage> chunks;     // key column + output columns of every input page
    std::vector<int32_t> col_types;  // types of [key, outputs...] as first seen (an empty build still needs them)
    int64_t rows = 0;
    bool finishing = false;
    tgpu_lookup* lookup = nullptr;

    explicit JoinBuildOp(tgpu_ctx* c) : tgpu_op(c) {}
    ~JoinBuildOp() override { if (lookup) tgpu_lookup_release(lookup); }

    bool needs_input() override { return !finishing; }

    int add_input(const tgpu_page* page) override
    {
        // HashBuilderOperator.addInput :253-277 -> PagesIndex.addPage :224-256
        if (col_types.empty()) {
            auto type_of = [&](int32_t ch) -> int32_t {
                if (ch < 0 || ch >= page->num_columns) return 0;
                const tgpu_column* c = &page->columns[ch];
                while ((c->type == TGPU_DICT32 || c->type == TGPU_RLE) && c->dictionary) c = c->dictionary;
                return c->type;
            };
            for (int32_t ch : key_channels) col_types.push_back(type_of(ch));
            for (int32_t ch : output_channels) col_types.push_back(type_of(ch));
        }
        if (page->num_rows == 0) return TGPU_OK;
        if (rows + page->num_rows > (int64_t)INT32_MAX)
            return tg_fail(ctx, TGPU_ERR_INSUFFICIENT_RESOURCES, "Size of pages index cannot exceed 2 billion entries");   // PagesIndex.java:247-250
        bool device = (page->flags & TGPU_PAGE_DEVICE) != 0;
        DevPage p;
        p.rows = page->num_rows;
        auto take = [&](int32_t ch) -> int {
            if (ch < 0 || ch >= page->num_columns) return tg_fail(ctx, TGPU_ERR_INVALID_ARGUMENT, "channel %d out of range", ch);
            DevColumn c;
            TG_TRY(tg_ingest_column(ctx, &page->columns[ch], device, &c));
            p.cols.push_back(std::move(c));
            return TGPU_OK;
        };
        for (int32_t ch : key_channels) TG_TRY(take(ch));
        for (int32_t ch : output_channels) TG_TRY(take(ch));
        if (!device) TG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        rows += p.rows;
        chunks.push_back(std::move(p));
        return TGPU_OK;
    }

    int concat(DevPage* out)
    {
        if (chunks.size() == 1) { *out = std::move(chunks[0]); chunks.clear(); return TGPU_OK; }
        DevPage r;
        r.rows = rows;
        size_t ncols = key_channels.size() + output_channels.size();
        r.cols.resize(ncols);
        for (size_t c = 0; c < ncols && !chunks.empty(); c++) {
            std::vector<const DevColumn*> parts;
            for (auto& ch : chunks) parts.push_back(&ch.cols[c]);
            TG_TRY(tg_concat_columns(ctx, parts, &r.cols[c]));
        }
        chunks.clear();
        *out = std::move(r);
        return TGPU_OK;
    }

    int finish() override
    {
        // HashBuilderOperator.finish :286-308 -> finishInput :310-333 -> PagesIndex.createLookupSourceSupplier :523-542
        if (finishing) return TGPU_OK;   // re-entrant
        std::unique_ptr<tgpu_lookup> lk(new tgpu_lookup());
        lk->ctx = ctx;
        lk->positions = rows;
        lk->num_output = (int32_t)output_channels.size();
        DevPage all;
        TG_TRY(concat(&all));
        const size_t nk = key_channels.size();
        if (rows == 0) {
            all.cols.resize(nk + output_channels.size());
            for (size_t c = 0; c < all.cols.size(); c++) all.cols[c].type = c < col_types.size() && col_types[c] ? col_types[c] : TGPU_INT64;
        }
        // one fixed-width channel -> the table is keyed by the value itself; anything else -> by the row hash + verification
        lk->generic = nk != 1 || all.cols[0].type == TGPU_UTF8 || all.cols[0].type == TGPU_INT128 || all.cols[0].type == TGPU_FLOAT32;      // (no 64-bit canonical key; REAL keys compare as floats in rowkeys.cuh)
        lk->store.rows = rows;
        if (lk->generic) {
            for (size_t c = 0; c < nk; c++) lk->build_keys.push_back(all.cols[c]);
            std::vector<const DevColumn*> kp;
            for (auto& c : lk->build_keys) kp.push_back(&c);
            DevColumn fp;
            TG_TRY(make_fingerprint(ctx, kp, rows, &fp));
            lk->store.cols.push_back(std::move(fp));
        }
        else lk->store.cols.push_back(all.cols[0]);
        for (size_t c = nk; c < all.cols.size(); c++) lk->store.cols.push_back(all.cols[c]);
        lk->key_type = lk->store.cols[0].type;
        int64_t cap = 0;
        auto build_table = [&]() -> int {
            // sizing: IncrementalLoadFactorHashArraySizeSupplier.getHashArraySize :40-47 (capacity is not observable)
            double lf = rows <= (1 << 16) ? 0.25 : rows <= (1 << 20) ? 0.5 : 0.75;
            int64_t need = (int64_t)((double)rows / lf) + 1;
            cap = 8;   // at least one 8-slot line
            while (cap < need) cap <<= 1;
            // line layouts (modes 1 / 2) want lines at most about half full (measured: exp_join_summary in profiles/), unless the keys
            // fill their lines evenly: candidates are tried in this order, each judged by the rows that had to leave their home line
            //   mode 2, base capacity  : "dense" - e.g. TPC-H order keys: every line of 32 key values holds exactly its 8 keys
            //   mode 2, 2 x capacity   : a line expects ~4 keys (random subsets of a dense domain: what a hash exchange leaves on a rank)
            //   mode 1, 2 x capacity   : scattered lines, any distribution
            const char* env_mode = getenv("TGPU_JOIN_HASH");
            const DevColumn& bkey = lk->store.cols[0];
            const bool int_key = !lk->generic && key_kind_of(bkey.type) == KEY_INT;
            int hash_mode = env_mode ? atoi(env_mode) : (int_key && rows > 0 ? 2 : 1);
            if (hash_mode == 2 && !(int_key && rows > 0)) hash_mode = 1;
            const char* env_shift = getenv("TGPU_JOIN_CAP_SHIFT");
            const int64_t base_cap = cap;
            unsigned long long span = 0, kmin = 0;
            if (hash_mode == 2) {
                long long* d_range = (long long*)(ctx->d_scratch + 24);
                long long init_range[2] = {INT64_MAX, INT64_MIN};
                TG_CUDA(ctx, cudaMemcpyAsync(d_range, init_range, sizeof(init_range), cudaMemcpyHostToDevice, ctx->stream));
                TG_LAUNCH(ctx, join_key_range_kernel, tg_grid(ctx, rows, 1024, 8), 256, 0, tg_colref(bkey), rows, d_range);
                long long h_range[2];
                TG_CUDA(ctx, cudaMemcpyAsync(h_range, d_range, sizeof(h_range), cudaMemcpyDeviceToHost, ctx->stream));
                TG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
                if (h_range[0] > h_range[1]) hash_mode = 1;      // no insertable key at all
                else {
                    span = (unsigned long long)h_range[1] - (unsigned long long)h_range[0];   // kmax - kmin, exact in 64 bits
                    kmin = (unsigned long long)h_range[0];
                }
            }
            int* d_flags = (int*)ctx->d_scratch;   // [0] special_head, [1] dup flag, [2] rows off their home line, [3] rows more than 8 lines off
            unsigned int* d_gave_up = (unsigned int*)(ctx->d_scratch + 22);   // rows a trial geometry could not place within its bound
            // attempt 0: dense mode 2; attempt 1: roomy mode 2; attempt 2: mode 1 (or whatever the environment pinned)
            for (int attempt = (hash_mode == 2 && !env_shift && !getenv("TGPU_JOIN_NO_DENSE")) ? 0 : 1; ; attempt++) {
                if (hash_mode == 2 && attempt >= 2) hash_mode = 1;
                const int cap_shift = env_shift ? atoi(env_shift) : (hash_mode == 0 ? 0 : (hash_mode == 2 && attempt == 0) ? 0 : 1);
                cap = base_cap << cap_shift;
                if (cap > (1LL << 31)) return tg_fail(ctx, TGPU_ERR_INSUFFICIENT_RESOURCES, "hash array too large");
                lk->geo.mask = (unsigned long long)cap - 1;
                lk->geo.kmin = 0;
                lk->geo.shift = 0;
                if (hash_mode == 2) {
                    // order-preserving lines: the key range [kmin, kmax] is cut into cap / 8 lines of 2^shift key values
                    const unsigned long long lines = (unsigned long long)cap >> 3;
                    int shift = 0;
                    while (shift < 63 && (span >> shift) >= lines) shift++;
                    if ((span >> shift) >= lines) { hash_mode = 1; attempt = 1; continue; }   // a span of 2^63 or more over very few lines
                    lk->geo.kmin = kmin;
                    lk->geo.shift = shift;
                }
                lk->geo.mode = hash_mode;
                TG_TRY(lk->table.alloc(ctx, (size_t)cap * sizeof(JoinSlot)));
                TG_LAUNCH(ctx, join_table_init_kernel, tg_grid(ctx, cap, 1024, 8), 256, 0, lk->table.as<int4>(), cap);
                int init[4] = {-1, 0, 0, 0};
                TG_CUDA(ctx, cudaMemcpyAsync(d_flags, init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
                TG_CUDA(ctx, cudaMemsetAsync(d_gave_up, 0, 8, ctx->stream));
                // mode 2 geometries are trials (the keys must suit them): bounded probing, early stop
                const int give_up_lines = hash_mode == 2 ? 16 : 0;
                const unsigned int give_up_limit = (unsigned int)std::min<int64_t>(rows / 1024, 1 << 20);
                if (rows > 0) {
                    TG_LAUNCH(ctx, join_build_kernel, tg_grid(ctx, rows, 256, 8), 256, 0, tg_colref(bkey), key_kind_of(bkey.type), rows,
                              lk->table.as<JoinSlot>(), lk->geo, d_flags, d_flags + 1, (unsigned int*)(d_flags + 2), give_up_lines, give_up_limit, d_gave_up);
                }
                if (hash_mode != 2) break;
                // mode 2 relies on the keys spreading evenly over their range; clustered domains pile up in a few lines.  Dense: at most
                // 1/64 of the rows off their home line; roomy: at most 1/8; and (nearly) no row further than 8 lines away, and every
                // row placed
                int64_t moved = 0, unplaced = 0;
                TG_TRY(tg_read_i64(ctx, d_flags + 2, &moved));
                TG_TRY(tg_read_i64(ctx, d_gave_up, &unplaced));
                const int64_t off_home = moved & 0xFFFFFFFFLL, far = (moved >> 32) & 0xFFFFFFFFLL;
                if ((unplaced & 0xFFFFFFFFLL) == 0 && off_home * (attempt == 0 ? 64 : 8) <= rows && far * 1024 <= rows) break;
            }
            int64_t packed = 0;
            TG_TRY(tg_read_i64(ctx, d_flags, &packed));
            lk->special_head = (int)(packed & 0xFFFFFFFFLL);
            lk->has_dups = (packed >> 32) != 0;
            return TGPU_OK;
        };
        if (!lk->generic) TG_TRY(build_table());
        else {
            // the fingerprint table: every row must sit in a slot whose head row carries ITS key.  Rows that share a 64-bit hash with a
            // different key move on to their next hash function and the table is rebuilt (never needed in practice; never a failure)
            DevBuf attempt;
            TG_TRY(attempt.alloc(ctx, (size_t)std::max<int64_t>(rows, 1)));
            TG_CUDA(ctx, cudaMemsetAsync(attempt.p, 0, (size_t)std::max<int64_t>(rows, 1), ctx->stream));
            for (int round = 0; ; round++) {
                if (round >= 8) return tg_fail(ctx, TGPU_ERR_INSUFFICIENT_RESOURCES, "join keys collide under 8 independent 64-bit hashes");
                if (round > 0) {
                    std::vector<const DevColumn*> kp;
                    for (auto& c : lk->build_keys) kp.push_back(&c);
                    DevColumn fp;
                    TG_TRY(make_fingerprint(ctx, kp, rows, &fp, attempt.as<uint8_t>()));
                    lk->store.cols[0] = std::move(fp);
                }
                TG_TRY(build_table());
                lk->attempts = round + 1;
                if (rows == 0) break;
                int* d_moved = (int*)(ctx->d_scratch + 16);
                TG_CUDA(ctx, cudaMemsetAsync(d_moved, 0, 8, ctx->stream));
                const DevColumn& fp = lk->store.cols[0];
                TG_LAUNCH(ctx, join_verify_build_kernel, tg_grid(ctx, rows, 256, 8), 256, 0, key_cols_of(lk->build_keys), (const long long*)fp.data, fp.validity, rows,
                          lk->table.as<JoinSlot>(), lk->geo, lk->special_head, attempt.as<uint8_t>(), d_moved);
                int64_t moved = 0;
                TG_TRY(tg_read_i64(ctx, d_moved, &moved));
                if ((moved & 0xFFFFFFFFLL) == 0) break;
            }
        }
        if (lk->has_dups) {
            // ArrayPositionLinks: chains in descending row order
            const DevColumn& key = lk->store.cols[0];
            DevBuf keys_in, keys_out, tmp;
            TG_TRY(keys_in.alloc(ctx, (size_t)rows * 8));
            TG_TRY(keys_out.alloc(ctx, (size_t)rows * 8));
            TG_LAUNCH(ctx, join_slot_of_row_kernel, tg_grid(ctx, rows, 256, 8), 256, 0, tg_colref(key), key_kind_of(key.type), rows,
                      lk->table.as<JoinSlot>(), lk->geo, (unsigned long long)cap, keys_in.as<unsigned long long>());
            size_t tmp_bytes = 0;
            cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, keys_in.as<unsigned long long>(), keys_out.as<unsigned long long>(), (int)rows, 0, 64, ctx->stream);
            TG_TRY(tmp.alloc(ctx, tmp_bytes));
            TG_CUDA(ctx, cub::DeviceRadixSort::SortKeys(tmp.p, tmp_bytes, keys_in.as<unsigned long long>(), keys_out.as<unsigned long long>(), (int)rows, 0, 64, ctx->stream));
            TG_TRY(lk->links.alloc(ctx, (size_t)rows * 4));
            TG_LAUNCH(ctx, join_links_kernel, tg_grid(ctx, rows, 256, 8), 256, 0, keys_out.as<unsigned long long>(), rows, lk->links.as<int>());
            TG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        }
        // slot-ordered copy of the build output columns for the fused probe
        bool slot_payload = !getenv("TGPU_JOIN_PAYLOAD_BY_ROW") && rows > 0 && lk->num_output > 0 && lk->num_output <= 4;
        for (int32_t b = 0; b < lk->num_output && slot_payload; b++)
            slot_payload = lk->store.cols[1 + b].elem_size() > 0 && lk->store.cols[1 + b].elem_size() <= 8 && !lk->store.cols[1 + b].validity;
        // one output column: key and payload share a 16-byte entry, which replaces both the slot-ordered payload and the wide table
        const bool packed = slot_payload && lk->num_output == 1 && !lk->has_dups && !lk->generic && cap + 1 < (1LL << 31);
        if (packed) {
            const DevColumn& c = lk->store.cols[1];
            TG_TRY(lk->packed.alloc(ctx, (size_t)(cap + 1) * sizeof(PackedSlot)));
            TG_LAUNCH(ctx, join_packed_table_kernel, tg_grid(ctx, cap + 1, 1024, 8), 256, 0, lk->table.as<JoinSlot>(), cap, lk->special_head, c.data, c.elem_size(),
                      lk->packed.as<PackedSlot>());
        }
        else if (slot_payload) {
            lk->by_slot.resize(lk->num_output);
            for (int32_t b = 0; b < lk->num_output; b++) {
                const DevColumn& c = lk->store.cols[1 + b];
                TG_TRY(lk->by_slot[b].alloc(ctx, (size_t)(cap + 1) * c.elem_size()));
                TG_LAUNCH(ctx, join_payload_by_slot_kernel, tg_grid(ctx, cap + 1, 1024, 8), 256, 0, lk->table.as<JoinSlot>(), cap, lk->special_head, c.data,
                          c.elem_size(), lk->by_slot[b].p);
            }
        }
        if (slot_payload && !packed && lk->num_output <= 2 && !lk->has_dups && !lk->generic && cap + 1 < (1LL << 31) && !getenv("TGPU_JOIN_NO_WIDE")) {
            TG_TRY(lk->wide.alloc(ctx, (size_t)(cap + 1) * sizeof(WideSlot)));
            const DevColumn& c0 = lk->store.cols[1];
            const DevColumn* c1 = lk->num_output > 1 ? &lk->store.cols[2] : nullptr;
            TG_LAUNCH(ctx, join_wide_table_kernel, tg_grid(ctx, cap + 1, 1024, 8), 256, 0, lk->table.as<JoinSlot>(), cap, lk->special_head, c0.data, c0.elem_size(),
                      c1 ? c1->data : (const void*)nullptr, c1 ? c1->elem_size() : 0, lk->wide.as<WideSlot>());
        }
        TG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        lookup = lk.release();
        finishing = true;
        return TGPU_OK;
    }

    int get_output(OwnedPage** out) override { *out = nullptr; return TGPU_OK; }
    // HashBuilderOperator.isFinished: after the lookup source was handed over and released
    bool is_finished() override { return finishing; }
    int64_t memory_bytes() override
    {
        int64_t b = 0;
        for (auto& c : chunks) b += c.memory_bytes();
        if (lookup) b += tgpu_lookup_memory_bytes(lookup);
        return b;
    }
};

// LookupJoinOperator
struct JoinProbeOp : tgpu_op {
    tgpu_lookup* lookup;
    int join_type = 0, single_match = 0;
    std::vector<int32_t> key_channels, output_channels;
    std::vector<OwnedPage*> pending;
    size_t next_out = 0;
    bool finishing = false;
    // fast path: addInput only enqueues the probe kernel; the match count is read (the one host synchronisation of the
    // step) when the output is asked for, so the caller can overlap other work - the next exchange - with the probe
    struct Deferred {
        bool active = false;
        DevPage in;
        std::shared_ptr<DevBuf> match_bits;     // bit i = probe row i matched (match_bits_word)
        std::vector<DevColumn> built;
        int64_t n = 0;
    } deferred;
    DevBuf match_counter;     // per operator: the count must survive until get_output
    // LookupJoinPageBuilder.build :144-150 hands probe blocks through as views.  With by_reference set, a HOST probe page
    // only has its join-key channel uploaded; pass-through output columns of the result then carry no device data
    // (data == NULL, tgpu_page_passthrough_channel names the input block) unless rows had to be dropped or repeated
    bool by_reference = false;

    JoinProbeOp(tgpu_ctx* c, tgpu_lookup* lk) : tgpu_op(c), lookup(lk) { lookup->refs++; }
    ~JoinProbeOp() override
    {
        for (size_t i = next_out; i < pending.size(); i++) delete pending[i];
        tgpu_lookup_release(lookup);
    }

    bool needs_input() override { return !finishing && !deferred.active && next_out >= pending.size(); }

    // fused probe + gather (see join_probe_gather_kernel); returns handled=false when the shape needs the general path
    int fast_path(DevPage& in, const DevColumn& key, int64_t n, bool* handled)
    {
        *handled = false;
        
        if (lookup->has_dups && !single_match) return TGPU_OK;
        if (lookup->num_output > 4 || key.type == TGPU_UTF8) return TGPU_OK;
        if (key_kind_of(key.type) != key_kind_of(lookup->key_type)) return TGPU_OK;   // reported by the general path
        for (int32_t b = 0; b < lookup->num_output; b++) {
            const DevColumn& c = lookup->store.cols[1 + b];
            if (c.elem_size() == 0 || c.elem_size() > 8 || c.validity) return TGPU_OK;      // (the fused gather moves 1 / 2 / 4 / 8-byte payloads)
        }
        // one 32-bit word per 32 rows of every (possibly partial) 1024-row tile: each word is written by a probe kernel
        auto bits = std::make_shared<DevBuf>();
        TG_TRY(bits->alloc(ctx, (size_t)((n + 1023) / 1024) * 128));
        unsigned int* d_bits = bits->as<unsigned int>();
        GatherCols g;
        memset(&g, 0, sizeof(g));
        g.count = lookup->num_output;
        std::vector<DevColumn> built(lookup->num_output);
        for (int32_t b = 0; b < lookup->num_output; b++) {
            const DevColumn& c = lookup->store.cols[1 + b];
            built[b].type = c.type;
            built[b].length = n;
            built[b].own_data = std::make_shared<DevBuf>();
            TG_TRY(built[b].own_data->alloc(ctx, (size_t)n * c.elem_size()));
            built[b].data = built[b].own_data->p;
            g.elem[b] = c.elem_size();
            g.src[b] = lookup->by_slot.empty() ? c.data : lookup->by_slot[b].p;
            g.dst[b] = built[b].own_data->p;
        }
        g.by_slot = lookup->by_slot.empty() ? 0 : 1;
        if (!match_counter.p) TG_TRY(match_counter.alloc(ctx, 16));       // [0] matches of the page, [1] (int) layout choice of the page
        unsigned long long* d_matches = match_counter.as<unsigned long long>();
        TG_CUDA(ctx, cudaMemsetAsync(d_matches, 0, 16, ctx->stream));     // no matches yet; layout choice 0 = the 16-byte slots
        auto k_fast = join_probe_gather_kernel<true>;
        auto k_any = join_probe_gather_kernel<false>;
        const JoinSlot* table = lookup->table.as<JoinSlot>();
        TG_TIMED_BEGIN(ctx);
        int64_t done = 0;
        bool fast = key.type == TGPU_INT64 && !key.validity;
        if (fast && !getenv("TGPU_JOIN_GENERIC_KERNELS")) {
            int64_t tiles = n / 1024;
            if (tiles > 0 && lookup->packed.p) {
                // one output column: the packed table, whatever the page's key locality
                TG_TRY(launch_packed(ctx, lookup->geo, (const long long*)key.data, tiles, lookup->packed.as<PackedSlot>(), lookup->special_head >= 0 ? 1 : 0, g.dst[0],
                                     g.elem[0], d_bits, d_matches));
                done = tiles * 1024;
            }
            else if (tiles > 0) {
                // TGPU_JOIN_WIDE = always | never | auto (default): auto lets the page's key locality decide whenever the wide layout is the
                // bigger one (payload cells < 16 bytes); with 16 bytes of payload the two layouts hold the same bytes and wide always wins
                const char* we = getenv("TGPU_JOIN_WIDE");
                int payload_bytes = 0;
                for (int c = 0; c < g.count; c++) payload_bytes += g.elem[c];
                const bool have_wide = lookup->wide.p && !getenv("TGPU_JOIN_NO_WIDE") && !(we && !strcmp(we, "never"));
                const bool always = have_wide && ((we && !strcmp(we, "always")) || payload_bytes >= 16 || !g.by_slot);
                if (always)
                    TG_TRY(launch_wide(ctx, lookup->geo, (const long long*)key.data, tiles, lookup->wide.as<WideSlot>(), lookup->special_head, g, d_bits, d_matches, nullptr));
                else if (have_wide) {
                    int* d_choice = (int*)(d_matches + 1);
                    TG_TRY(launch_locality(ctx, lookup->geo, (const long long*)key.data, tiles, d_choice));
                    TG_TRY(launch_lean<true>(ctx, lookup->geo, (const long long*)key.data, tiles, (const int4*)table, lookup->special_head, nullptr, g, d_bits, d_matches));
                    TG_TRY(launch_wide(ctx, lookup->geo, (const long long*)key.data, tiles, lookup->wide.as<WideSlot>(), lookup->special_head, g, d_bits, d_matches, d_choice));
                }
                else
                    TG_TRY(launch_lean<true>(ctx, lookup->geo, (const long long*)key.data, tiles, (const int4*)table, lookup->special_head, nullptr, g, d_bits, d_matches));
                done = tiles * 1024;
            }
        }
        if (done < n) {
            ColRef kr = tg_colref(key);
            GatherCols gt = g;
            if (done > 0) {
                kr.data = (const char*)kr.data + done * 8;
                for (int c = 0; c < gt.count; c++) gt.dst[c] = (char*)gt.dst[c] + done * gt.elem[c];
            }
            // done is a multiple of 1024: the tail's tiles start on a word of the bitmap
            int tgrid = tg_grid(ctx, n - done, 1024, 8);
            if (fast) TG_LAUNCH(ctx, k_fast, tgrid, 256, 0, kr, KEY_INT, n - done, table, lookup->geo, lookup->special_head, gt, d_bits + done / 32, d_matches);
            else TG_LAUNCH(ctx, k_any, tgrid, 256, 0, kr, key_kind_of(key.type), n - done, table, lookup->geo, lookup->special_head, gt, d_bits + done / 32, d_matches);
        }
        TG_TIMED_END(ctx);
        *handled = true;
        deferred.active = true;
        deferred.in = std::move(in);
        deferred.match_bits = bits;
        deferred.built = std::move(built);
        deferred.n = n;
        return TGPU_OK;
    }

    // second half of the fast path: read the match count and shape the output page
    // partial ingest of a host page: the join-key channel goes to the device, the others stay placeholders
    int ingest_keys_only(const tgpu_page* page, DevPage* out)
    {
        DevPage p;
        p.rows = page->num_rows;
        p.cols.resize(page->num_columns);
        for (int32_t c = 0; c < page->num_columns; c++) {
            if (page->columns[c].length != page->num_rows) return tg_fail(ctx, TGPU_ERR_INVALID_ARGUMENT, "column %d has %lld positions, page has %lld", c,
                                                                          (long long)page->columns[c].length, (long long)page->num_rows);
            bool is_key = c == key_channels[0];
            if (is_key) TG_TRY(tg_ingest_column(ctx, &page->columns[c], false, &p.cols[c]));
            else { p.cols[c].type = page->columns[c].type; p.cols[c].length = page->num_rows; }
        }
        TG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        *out = std::move(p);
        return TGPU_OK;
    }

    static bool absent(const DevColumn& c) { return c.data == nullptr && c.length > 0; }

    int upload_absent(const tgpu_page* page, DevPage* in)
    {
        bool any = false;
        for (int32_t c = 0; c < page->num_columns; c++) {
            if (!absent(in->cols[c])) continue;
            TG_TRY(tg_ingest_column(ctx, &page->columns[c], false, &in->cols[c]));
            any = true;
        }
        if (any) TG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        return TGPU_OK;
    }

    // `host_page`: the input of a by-reference probe (its pass-through channels were not uploaded), else nullptr
    int complete_fast(const tgpu_page* host_page = nullptr)
    {
        deferred.active = false;
        DevPage in = std::move(deferred.in);
        std::shared_ptr<DevBuf> bits = std::move(deferred.match_bits);
        std::vector<DevColumn> built = std::move(deferred.built);
        const int64_t n = deferred.n;
        const bool outer = join_type == TGPU_JOIN_PROBE_OUTER;     // (tracking join types never take the fast path)
        int64_t matches = 0;
        TG_TRY(tg_read_i64(ctx, match_counter.as<int64_t>(), &matches));
        DevPage outp;
        if (host_page && !(matches == n || outer) && matches > 0) TG_TRY(upload_absent(host_page, &in));   // rows are dropped: the gather needs them
        if (matches == n || outer) {
            // every probe row yields exactly one output row: probe blocks pass through
            // (LookupJoinPageBuilder.build :144-150 "outputProbeBlocksDirectly")
            outp.rows = n;
            for (int32_t ch : output_channels) outp.cols.push_back(in.cols[ch]);
            // PROBE_OUTER with misses: the match bitmap is the build columns' validity
            for (auto& c : built) {
                if (matches < n) { c.own_validity = bits; c.validity = bits->as<uint8_t>(); }
                outp.cols.push_back(std::move(c));
            }
        }
        else {
            if (matches == 0) return TGPU_OK;
            // compact the matched rows (stable): selection list from the match bitmap, then sequential-read gathers
            DevBuf sel, tmp;
            TG_TRY(sel.alloc(ctx, (size_t)n * 4));
            long long* d_count = (long long*)(ctx->d_scratch + 14);
            size_t tmp_bytes = 0;
            thrust::counting_iterator<int32_t> iota(0);
            const MatchBit matched{bits->as<unsigned int>()};
            cub::DeviceSelect::If(nullptr, tmp_bytes, iota, sel.as<int32_t>(), d_count, (int)n, matched, ctx->stream);
            TG_TRY(tmp.alloc(ctx, tmp_bytes));
            TG_CUDA(ctx, cub::DeviceSelect::If(tmp.p, tmp_bytes, iota, sel.as<int32_t>(), d_count, (int)n, matched, ctx->stream));
            outp.rows = matches;
            for (int32_t ch : output_channels) {
                DevColumn c;
                TG_TRY(tg_gather_column(ctx, in.cols[ch], sel.as<int32_t>(), matches, false, &c));
                outp.cols.push_back(std::move(c));
            }
            for (auto& b : built) {
                DevColumn c;
                TG_TRY(tg_gather_column(ctx, b, sel.as<int32_t>(), matches, false, &c));
                outp.cols.push_back(std::move(c));
            }
        }
        OwnedPage* o = tg_make_owned_page(std::move(outp));
        if (matches == n || outer) o->passthrough.assign(output_channels.begin(), output_channels.end());   // probe blocks passed through 1:1
        pending.push_back(o);
        return TGPU_OK;
    }

    int add_input(const tgpu_page* page) override
    {
        if (deferred.active) return tg_fail(ctx, TGPU_ERR_ILLEGAL_STATE, "addInput while the previous page's output has not been taken (needsInput() is false)");
        for (size_t i = next_out; i < pending.size(); i++) delete pending[i];
        pending.clear();
        next_out = 0;
        int64_t n = page->num_rows;
        if (n == 0) return TGPU_OK;
        if (n > (int64_t)INT32_MAX) return tg_fail(ctx, TGPU_ERR_INVALID_ARGUMENT, "page has more than 2^31-1 positions");
        DevPage in;
        const bool lazy = by_reference && !(page->flags & TGPU_PAGE_DEVICE) && !lookup->generic && key_channels.size() == 1;
        if (lazy) TG_TRY(ingest_keys_only(page, &in));
        else TG_TRY(tg_ingest_page(ctx, page, &in));
        if (key_channels[0] < 0 || key_channels[0] >= (int32_t)in.cols.size()) return tg_fail(ctx, TGPU_ERR_INVALID_ARGUMENT, "probe key channel out of range");
        for (int32_t ch : output_channels)
            if (ch < 0 || ch >= (int32_t)in.cols.size()) return tg_fail(ctx, TGPU_ERR_INVALID_ARGUMENT, "probe output channel out of range");
        for (int32_t ch : key_channels)
            if (ch < 0 || ch >= (int32_t)in.cols.size()) return tg_fail(ctx, TGPU_ERR_INVALID_ARGUMENT, "probe key channel out of range");
        const DevColumn& key = in.cols[key_channels[0]];
        if (!lookup->generic && key_channels.size() != 1) return tg_fail(ctx, TGPU_ERR_INVALID_ARGUMENT, "probe has %zu join channels, build has 1", key_channels.size());
        const bool tracking = join_type == TGPU_JOIN_LOOKUP_OUTER || join_type == TGPU_JOIN_FULL_OUTER;
        if (!lookup->generic && !tracking && !getenv("TGPU_JOIN_GENERAL_PATH")) {
            bool handled = false;
            TG_TRY(fast_path(in, key, n, &handled));
            if (handled) return lazy ? complete_fast(page) : TGPU_OK;   // host buffers are the caller's again after this call
        }
        if (lazy) TG_TRY(upload_absent(page, &in));
        // joinPositionCache (JoinProbe.java:112-180)
        auto jp = std::make_shared<DevBuf>();
        TG_TRY(jp->alloc(ctx, (size_t)(n + 1) * 4));
        if (lookup->generic) {
            std::vector<const DevColumn*> kp;
            for (int32_t ch : key_channels) kp.push_back(&in.cols[ch]);
            TG_TRY(lookup_positions_generic(ctx, lookup, kp, n, jp->as<int>()));
        }
        else TG_TRY(lookup_positions(ctx, lookup, key, jp->as<int>()));
        bool outer = join_type == TGPU_JOIN_PROBE_OUTER || join_type == TGPU_JOIN_FULL_OUTER;
        const int* links = lookup->has_dups ? lookup->links.as<int>() : nullptr;
        // match counts -> exclusive scan -> output offsets
        DevBuf counts, offsets, tmp;
        TG_TRY(counts.alloc(ctx, (size_t)(n + 1) * 4));
        TG_TRY(offsets.alloc(ctx, (size_t)(n + 1) * 8));
        int grid = tg_grid(ctx, n, 256 * 4, 8);
        TG_LAUNCH(ctx, join_count_kernel, grid, 256, 0, jp->as<int>(), n, links, single_match, outer ? 1 : 0, counts.as<int>());
        size_t tmp_bytes = 0;
        cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, counts.as<int>(), offsets.as<long long>(), n + 1, ctx->stream);
        TG_TRY(tmp.alloc(ctx, tmp_bytes));
        TG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, counts.as<int>(), offsets.as<long long>(), n + 1, ctx->stream));
        int64_t total = 0;
        TG_TRY(tg_read_i64(ctx, offsets.as<long long>() + n, &total));
        if (total == 0) return TGPU_OK;
        if (total > (int64_t)INT32_MAX) return tg_fail(ctx, TGPU_ERR_INSUFFICIENT_RESOURCES, "join output of one probe page exceeds 2^31-1 rows");

        DevPage outp;
        outp.rows = total;
        // every probe row produced exactly one row and there are no chains: probe rows map 1:1
        // (LookupJoinPageBuilder.build :144-150 "outputProbeBlocksDirectly")
        bool identity = (total == n) && (!links || single_match);
        const int* build_idx = nullptr;
        bool build_may_be_null = outer;
        DevBuf out_probe, out_build;
        if (identity) {
            for (int32_t ch : output_channels) outp.cols.push_back(in.cols[ch]);   // shares ownership, no copy
            build_idx = jp->as<int>();
        }
        else {
            TG_TRY(out_probe.alloc(ctx, (size_t)total * 4));
            TG_TRY(out_build.alloc(ctx, (size_t)total * 4));
            TG_LAUNCH(ctx, join_fill_kernel, grid, 256, 0, jp->as<int>(), n, links, single_match, outer ? 1 : 0, offsets.as<long long>(),
                      out_probe.as<int>(), out_build.as<int>());
            for (int32_t ch : output_channels) {
                DevColumn c;
                TG_TRY(tg_gather_column(ctx, in.cols[ch], out_probe.as<int>(), total, false, &c));
                outp.cols.push_back(std::move(c));
            }
            build_idx = out_build.as<int>();
        }
        for (int32_t b = 0; b < lookup->num_output; b++) {
            DevColumn c;
            TG_TRY(tg_gather_column(ctx, lookup->store.cols[1 + b], build_idx, total, build_may_be_null, &c));
            outp.cols.push_back(std::move(c));
        }
        if (tracking && lookup->visited.p)
            TG_LAUNCH(ctx, join_mark_visited_kernel, tg_grid(ctx, total, 1024, 8), 256, 0, build_idx, total, lookup->visited.as<uint8_t>());
        pending.push_back(tg_make_owned_page(std::move(outp)));
        if (tracking) TG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // the marks must be visible to the outer operator's context
        return TGPU_OK;
    }

    int get_output(OwnedPage** out) override
    {
        *out = nullptr;
        if (deferred.active) TG_TRY(complete_fast());
        if (next_out < pending.size()) *out = pending[next_out++];
        return TGPU_OK;
    }
    int finish() override { finishing = true; return TGPU_OK; }
    bool is_finished() override { return finishing && !deferred.active && next_out >= pending.size(); }
};

// LookupOuterOperator (M/operator/join/LookupOuterOperator.java:170-206): after every probe has finished, the build rows no
// probe emitted, in position order, with NULLs in the probe output channels.  A source operator.
struct JoinOuterOp : tgpu_op {
    tgpu_lookup* lookup;
    std::vector<int32_t> probe_types;
    bool done = false;
    OwnedPage* pending = nullptr;

    JoinOuterOp(tgpu_ctx* c, tgpu_lookup* lk) : tgpu_op(c), lookup(lk) { lookup->refs++; }
    ~JoinOuterOp() override { delete pending; tgpu_lookup_release(lookup); }

    bool needs_input() override { return false; }
    int add_input(const tgpu_page*) override { return tg_fail(ctx, TGPU_ERR_ILLEGAL_STATE, "LookupOuterOperator does not take input"); }

    int produce()
    {
        done = true;
        const int64_t n = lookup->positions;
        if (n == 0) return TGPU_OK;
        DevBuf flags, sel, tmp;
        TG_TRY(flags.alloc(ctx, (size_t)n));
        TG_TRY(sel.alloc(ctx, (size_t)n * 4));
        if (lookup->visited.p) TG_LAUNCH(ctx, join_unvisited_flags_kernel, tg_grid(ctx, n, 1024, 8), 256, 0, lookup->visited.as<uint8_t>(), n, flags.as<uint8_t>());
        else TG_CUDA(ctx, cudaMemsetAsync(flags.p, 1, (size_t)n, ctx->stream));     // no tracking probe ever ran: every row is unvisited
        long long* d_count = (long long*)(ctx->d_scratch + 14);
        size_t tmp_bytes = 0;
        thrust::counting_iterator<int32_t> iota(0);
        cub::DeviceSelect::Flagged(nullptr, tmp_bytes, iota, flags.as<uint8_t>(), sel.as<int32_t>(), d_count, (int)n, ctx->stream);
        TG_TRY(tmp.alloc(ctx, tmp_bytes));
        TG_CUDA(ctx, cub::DeviceSelect::Flagged(tmp.p, tmp_bytes, iota, flags.as<uint8_t>(), sel.as<int32_t>(), d_count, (int)n, ctx->stream));
        int64_t m = 0;
        TG_TRY(tg_read_i64(ctx, d_count, &m));
        if (m == 0) return TGPU_OK;
        DevPage outp;
        outp.rows = m;
        // probe channels: all NULL
        auto all_null = std::make_shared<DevBuf>();
        TG_TRY(all_null->alloc(ctx, (size_t)((m + 7) / 8)));
        TG_CUDA(ctx, cudaMemsetAsync(all_null->p, 0, (size_t)((m + 7) / 8), ctx->stream));
        for (int32_t t : probe_types) {
            DevColumn c;
            c.type = t;
            c.length = m;
            c.own_validity = all_null;
            c.validity = all_null->as<uint8_t>();
            size_t es = (size_t)(t == TGPU_UTF8 ? 1 : c.elem_size());
            c.own_data = std::make_shared<DevBuf>();
            TG_TRY(c.own_data->alloc(ctx, std::max<size_t>((size_t)m * es, 8)));
            TG_CUDA(ctx, cudaMemsetAsync(c.own_data->p, 0, std::max<size_t>((size_t)m * es, 8), ctx->stream));
            c.data = c.own_data->p;
            if (t == TGPU_UTF8) {
                c.own_offsets = std::make_shared<DevBuf>();
                TG_TRY(c.own_offsets->alloc(ctx, (size_t)(m + 1) * 4));
                TG_CUDA(ctx, cudaMemsetAsync(c.own_offsets->p, 0, (size_t)(m + 1) * 4, ctx->stream));
                c.offsets = c.own_offsets->as<int32_t>();
            }
            outp.cols.push_back(std::move(c));
        }
        for (int32_t b = 0; b < lookup->num_output; b++) {
            DevColumn c;
            TG_TRY(tg_gather_column(ctx, lookup->store.cols[1 + b], sel.as<int32_t>(), m, false, &c));
            outp.cols.push_back(std::move(c));
        }
        TG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        pending = tg_make_owned_page(std::move(outp));
        return TGPU_OK;
    }

    int get_output(OwnedPage** out) override
    {
        *out = nullptr;
        if (!done) TG_TRY(produce());
        *out = pending;
        pending = nullptr;
        return TGPU_OK;
    }
    int finish() override { return TGPU_OK; }
    bool is_finished() override { return done && !pending; }
};

// HashSemiJoinOperator (M/operator/HashSemiJoinOperator.java:155-201) over a lookup built by a HashBuilder on the filtering
// source's join channel (the ChannelSet of SetBuilderOperator): input page + one BOOLEAN column.
struct SemiJoinOp : tgpu_op {
    tgpu_lookup* lookup;
    int32_t probe_channel = 0;
    OwnedPage* pending = nullptr;
    bool finishing = false;

    SemiJoinOp(tgpu_ctx* c, tgpu_lookup* lk) : tgpu_op(c), lookup(lk) { lookup->refs++; }
    ~SemiJoinOp() override { delete pending; tgpu_lookup_release(lookup); }

    bool needs_input() override { return !finishing && !pending; }

    int add_input(const tgpu_page* page) override
    {
        if (pending) return tg_fail(ctx, TGPU_ERR_ILLEGAL_STATE, "addInput while the previous page's output has not been taken");
        int64_t n = page->num_rows;
        if (n == 0) return TGPU_OK;
        DevPage in;
        TG_TRY(tg_ingest_page(ctx, page, &in));
        if (probe_channel < 0 || probe_channel >= (int32_t)in.cols.size()) return tg_fail(ctx, TGPU_ERR_INVALID_ARGUMENT, "probe join channel out of range");
        const DevColumn& key = in.cols[probe_channel];
        const int float_kind = key.type == TGPU_FLOAT64 ? 1 : key.type == TGPU_FLOAT32 ? 2 : 0;
        DevBuf pos;
        TG_TRY(pos.alloc(ctx, (size_t)n * 4));
        if (lookup->generic) {
            std::vector<const DevColumn*> kp{&key};
            TG_TRY(lookup_positions_generic(ctx, lookup, kp, n, pos.as<int>()));
        }
        else TG_TRY(lookup_positions(ctx, lookup, key, pos.as<int>()));
        DevColumn out;
        out.type = TGPU_INT8;
        out.length = n;
        out.own_data = std::make_shared<DevBuf>();
        TG_TRY(out.own_data->alloc(ctx, (size_t)n));
        out.data = out.own_data->p;
        DevBuf is_null;
        TG_TRY(is_null.alloc(ctx, (size_t)n));
        TG_LAUNCH(ctx, semi_join_kernel, tg_grid(ctx, n, 1024, 8), 256, 0, pos.as<int>(), key.validity, n, lookup->positions == 0 ? 1 : 0,
                  lookup->null_key_rows > 0 ? 1 : 0, out.own_data->as<signed char>(), is_null.as<uint8_t>(), tg_colref(key), float_kind, lookup->nan_key_rows > 0 ? 1 : 0);
        tgpu_column bm;
        memset(&bm, 0, sizeof(bm));
        bm.type = TGPU_INT8;
        bm.flags = TGPU_COL_NULLS_BYTEMAP;
        bm.length = n;
        bm.data = is_null.p;
        bm.validity = is_null.as<uint8_t>();
        DevColumn packed;
        TG_TRY(tg_ingest_column(ctx, &bm, true, &packed));
        out.own_validity = packed.own_validity;
        out.validity = packed.validity;
        DevPage outp;
        outp.rows = n;
        outp.cols = in.cols;            // inputPage.appendColumn(...): the input blocks pass through
        outp.cols.push_back(std::move(out));
        TG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        pending = tg_make_owned_page(std::move(outp));
        for (int32_t c = 0; c + 1 < (int32_t)pending->page.cols.size(); c++) pending->passthrough.push_back(c);
        return TGPU_OK;
    }

    int get_output(OwnedPage** out) override
    {
        *out = pending;
        pending = nullptr;
        return TGPU_OK;
    }
    int finish() override { finishing = true; return TGPU_OK; }
    bool is_finished() override { return finishing && !pending; }
};

// rows of the build side whose join key is NULL (HashSemiJoin's containsNull; never matched, so always outer rows)
static int lookup_count_null_keys(tgpu_ctx* ctx, tgpu_lookup* lk)
{
    if (lk->null_key_rows >= 0) return TGPU_OK;
    lk->null_key_rows = 0;
    if (lk->positions == 0) return TGPU_OK;
    const DevColumn* key = lk->generic ? (lk->build_keys.empty() ? nullptr : &lk->build_keys[0]) : (lk->store.cols.empty() ? nullptr : &lk->store.cols[0]);
    if (!key || !key->validity) return TGPU_OK;
    DevBuf cnt;
    TG_TRY(cnt.alloc(ctx, 8));
    TG_CUDA(ctx, cudaMemsetAsync(cnt.p, 0, 8, ctx->stream));
    TG_LAUNCH(ctx, count_nulls_kernel, tg_grid(ctx, lk->positions, 1024, 8), 256, 0, key->validity, lk->positions, cnt.as<unsigned long long>());
    int64_t v = 0;
    TG_TRY(tg_read_i64(ctx, cnt.p, &v));
    lk->null_key_rows = v;
    return TGPU_OK;
}

static int lookup_count_nan_keys(tgpu_ctx* ctx, tgpu_lookup* lk)
{
    if (lk->nan_key_rows >= 0) return TGPU_OK;
    lk->nan_key_rows = 0;
    if (lk->positions == 0) return TGPU_OK;
    const DevColumn* key = lk->generic ? (lk->build_keys.empty() ? nullptr : &lk->build_keys[0]) : (lk->store.cols.empty() ? nullptr : &lk->store.cols[0]);
    const int float_kind = !key ? 0 : key->type == TGPU_FLOAT64 ? 1 : key->type == TGPU_FLOAT32 ? 2 : 0;
    if (!float_kind) return TGPU_OK;
    DevBuf cnt;
    TG_TRY(cnt.alloc(ctx, 8));
    TG_CUDA(ctx, cudaMemsetAsync(cnt.p, 0, 8, ctx->stream));
    TG_LAUNCH(ctx, count_nan_keys_kernel, tg_grid(ctx, lk->positions, 1024, 8), 256, 0, tg_colref(*key), float_kind, lk->positions, cnt.as<unsigned long long>());
    int64_t v = 0;
    TG_TRY(tg_read_i64(ctx, cnt.p, &v));
    lk->nan_key_rows = v;
    return TGPU_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" int tgpu_join_build_create(tgpu_ctx* ctx, const tgpu_join_build_spec* spec, tgpu_op** out)
{
    if (!ctx || !spec || !out) return TGPU_ERR_INVALID_ARGUMENT;
    if (spec->num_key_channels < 1 || spec->num_key_channels > tg::MAX_KEY_COLS)
        return tg_fail(ctx, TGPU_ERR_NOT_SUPPORTED, "GPU hash join supports 1..%d join channels (got %d)", tg::MAX_KEY_COLS, spec->num_key_channels);
    JoinBuildOp* op = new JoinBuildOp(ctx);
    op->key_channels.assign(spec->key_channels, spec->key_channels + spec->num_key_channels);
    op->output_channels.assign(spec->output_channels, spec->output_channels + spec->num_output_channels);
    *out = op;
    return TGPU_OK;
}

extern "C" int tgpu_join_build_get_lookup(tgpu_op* build, tgpu_lookup** out)
{
    JoinBuildOp* op = dynamic_cast<JoinBuildOp*>(build);
    if (!op || !out) return TGPU_ERR_INVALID_ARGUMENT;
    if (!op->lookup) return tg_fail(op->ctx, TGPU_ERR_ILLEGAL_STATE, "lookup source is not built yet: call finish() first");
    op->lookup->refs++;
    *out = op->lookup;
    return TGPU_OK;
}

extern "C" void tgpu_lookup_release(tgpu_lookup* lookup)
{
    if (!lookup) return;
    if (--lookup->refs == 0) {
        cudaSetDevice(lookup->ctx->device);
        delete lookup;
    }
}

extern "C" int64_t tgpu_lookup_position_count(const tgpu_lookup* lookup) { return lookup ? lookup->positions : 0; }

extern "C" int64_t tgpu_lookup_memory_bytes(const tgpu_lookup* lookup)
{
    if (!lookup) return 0;
    int64_t b = (int64_t)lookup->table.bytes + (int64_t)lookup->links.bytes + lookup->store.memory_bytes();
    for (auto& s : lookup->by_slot) b += (int64_t)s.bytes;
    b += (int64_t)lookup->wide.bytes + (int64_t)lookup->packed.bytes;
    return b;
}

extern "C" int tgpu_lookup_has_duplicates(const tgpu_lookup* lookup) { return lookup && lookup->has_dups ? 1 : 0; }

extern "C" int tgpu_join_probe_create(tgpu_ctx* ctx, const tgpu_join_probe_spec* spec, tgpu_lookup* lookup, tgpu_op** out)
{
    if (!ctx || !spec || !lookup || !out) return TGPU_ERR_INVALID_ARGUMENT;
    if (spec->num_key_channels < 1 || spec->num_key_channels > tg::MAX_KEY_COLS)
        return tg_fail(ctx, TGPU_ERR_NOT_SUPPORTED, "GPU hash join supports 1..%d join channels (got %d)", tg::MAX_KEY_COLS, spec->num_key_channels);
    if (spec->join_type < TGPU_JOIN_INNER || spec->join_type > TGPU_JOIN_FULL_OUTER) return tg_fail(ctx, TGPU_ERR_INVALID_ARGUMENT, "bad join type %d", spec->join_type);
    if (spec->join_type == TGPU_JOIN_LOOKUP_OUTER || spec->join_type == TGPU_JOIN_FULL_OUTER) {
        // OuterLookupSourceSupplier: the visited-positions array is shared by every probe of this lookup source
        TG_CUDA(ctx, cudaSetDevice(ctx->device));
        std::lock_guard<std::mutex> guard(lookup->visited_lock);
        if (!lookup->visited.p && lookup->positions > 0) {
            TG_TRY(lookup->visited.alloc(ctx, (size_t)lookup->positions));
            TG_CUDA(ctx, cudaMemsetAsync(lookup->visited.p, 0, (size_t)lookup->positions, ctx->stream));
            TG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        }
    }
    JoinProbeOp* op = new JoinProbeOp(ctx, lookup);
    op->join_type = spec->join_type;
    op->single_match = spec->output_single_match;
    op->key_channels.assign(spec->key_channels, spec->key_channels + spec->num_key_channels);
    op->output_channels.assign(spec->output_channels, spec->output_channels + spec->num_output_channels);
    *out = op;
    return TGPU_OK;
}

extern "C" int tgpu_join_outer_create(tgpu_ctx* ctx, tgpu_lookup* lookup, const int32_t* probe_output_types, int32_t num_probe_outputs, tgpu_op** out)
{
    if (!ctx || !lookup || !out || num_probe_outputs < 0 || (num_probe_outputs > 0 && !probe_output_types)) return TGPU_ERR_INVALID_ARGUMENT;
    JoinOuterOp* op = new JoinOuterOp(ctx, lookup);
    op->probe_types.assign(probe_output_types, probe_output_types + num_probe_outputs);
    *out = op;
    return TGPU_OK;
}

extern "C" int tgpu_semi_join_create(tgpu_ctx* ctx, tgpu_lookup* lookup, int32_t probe_join_channel, tgpu_op** out)
{
    if (!ctx || !lookup || !out) return TGPU_ERR_INVALID_ARGUMENT;
    TG_CUDA(ctx, cudaSetDevice(ctx->device));
    if (lookup->generic && lookup->build_keys.size() != 1) return tg_fail(ctx, TGPU_ERR_INVALID_ARGUMENT, "a semi-join set has one channel");
    TG_TRY(lookup_count_null_keys(ctx, lookup));
    TG_TRY(lookup_count_nan_keys(ctx, lookup));
    SemiJoinOp* op = new SemiJoinOp(ctx, lookup);
    op->probe_channel = probe_join_channel;
    *out = op;
    return TGPU_OK;
}

extern "C" int tgpu_lookup_key_domain(tgpu_ctx* ctx, tgpu_lookup* lookup, int64_t max_values, int64_t* min_out, int64_t* max_out, int64_t* distinct_out,
                                      int64_t* values_out, int32_t* has_null_out)
{
    if (!ctx || !lookup || !min_out || !max_out || !distinct_out || max_values < 0 || (max_values > 0 && !values_out)) return TGPU_ERR_INVALID_ARGUMENT;
    TG_CUDA(ctx, cudaSetDevice(ctx->device));
    if (lookup->generic || lookup->key_type == TGPU_FLOAT64 || lookup->key_type == TGPU_UTF8)
        return tg_fail(ctx, TGPU_ERR_NOT_SUPPORTED, "key domains are collected for single BIGINT-family join keys only");
    TG_TRY(lookup_count_null_keys(ctx, lookup));
    if (has_null_out) *has_null_out = lookup->null_key_rows > 0;
    const int64_t slots = (int64_t)lookup->geo.mask + 1;
    DevBuf state, vals;
    TG_TRY(state.alloc(ctx, 24));
    TG_TRY(vals.alloc(ctx, (size_t)std::max<int64_t>(max_values, 1) * 8));
    long long init[3] = {INT64_MAX, INT64_MIN, 0};
    TG_CUDA(ctx, cudaMemcpyAsync(state.p, init, 24, cudaMemcpyHostToDevice, ctx->stream));
    if (lookup->table.p && lookup->positions > 0)
        TG_LAUNCH(ctx, join_key_domain_kernel, tg_grid(ctx, slots, 1024, 8), 256, 0, lookup->table.as<JoinSlot>(), slots, max_values, state.as<long long>(),
                  (unsigned long long*)(state.as<long long>() + 2), vals.as<long long>());
    long long res[3];
    TG_CUDA(ctx, cudaMemcpyAsync(res, state.p, 24, cudaMemcpyDeviceToHost, ctx->stream));
    TG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    int64_t distinct = res[2];
    int64_t got = std::min<int64_t>(distinct, max_values);
    if (got > 0) {
        TG_CUDA(ctx, cudaMemcpyAsync(values_out, vals.p, (size_t)got * 8, cudaMemcpyDeviceToHost, ctx->stream));
        TG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    if (lookup->special_head >= 0) {       // the key INT64_MIN lives beside the table
        if (distinct < max_values) values_out[distinct] = INT64_MIN;
        distinct++;
        res[0] = INT64_MIN;
        if (res[1] < res[0]) res[1] = INT64_MIN;
    }
    if (distinct <= max_values && distinct > 0) std::sort(values_out, values_out + distinct);
    *min_out = res[0];
    *max_out = res[1];
    *distinct_out = distinct;
    return TGPU_OK;
}

extern "C" int tgpu_join_probe_set_passthrough_by_reference(tgpu_op* op, int32_t enable)
{
    JoinProbeOp* p = dynamic_cast<JoinProbeOp*>(op);
    if (!p) return TGPU_ERR_INVALID_ARGUMENT;
    p->by_reference = enable != 0;
    return TGPU_OK;
}

extern "C" int tgpu_lookup_get_join_positions(tgpu_ctx* ctx, const tgpu_lookup* lookup, const tgpu_page* keys_page, int32_t* out_positions)
{
    if (!ctx || !lookup || !keys_page || !out_positions) return TGPU_ERR_INVALID_ARGUMENT;
    TG_CUDA(ctx, cudaSetDevice(ctx->device));
    bool device = (keys_page->flags & TGPU_PAGE_DEVICE) != 0;
    int64_t n = keys_page->num_rows;
    if (lookup->generic) {
        DevPage kp;
        TG_TRY(tg_ingest_page(ctx, keys_page, &kp));
        std::vector<const DevColumn*> refs;
        for (auto& c : kp.cols) refs.push_back(&c);
        if (device) return lookup_positions_generic(ctx, lookup, refs, n, out_positions);
        DevBuf gout;
        TG_TRY(gout.alloc(ctx, (size_t)std::max<int64_t>(n, 1) * 4));
        TG_TRY(lookup_positions_generic(ctx, lookup, refs, n, gout.as<int>()));
        TG_CUDA(ctx, cudaMemcpyAsync(out_positions, gout.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
        TG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        return TGPU_OK;
    }
    if (keys_page->num_columns != 1) return tg_fail(ctx, TGPU_ERR_INVALID_ARGUMENT, "exactly one key column expected");
    DevColumn key;
    TG_TRY(tg_ingest_column(ctx, &keys_page->columns[0], device, &key));
    if (device) return lookup_positions(ctx, lookup, key, out_positions);
    DevBuf out;
    TG_TRY(out.alloc(ctx, (size_t)n * 4));
    TG_TRY(lookup_positions(ctx, lookup, key, out.as<int>()));
    TG_CUDA(ctx, cudaMemcpyAsync(out_positions, out.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    TG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return TGPU_OK;
}

extern "C" int tgpu_lookup_copy_position_links(tgpu_ctx* ctx, const tgpu_lookup* lookup, int32_t* out_links_host)
{
    if (!ctx || !lookup || !out_links_host) return TGPU_ERR_INVALID_ARGUMENT;
    if (!lookup->has_dups) {
        for (int64_t i = 0; i < lookup->positions; i++) out_links_host[i] = -1;
        return TGPU_OK;
    }
    TG_CUDA(ctx, cudaMemcpyAsync(out_links_host, lookup->links.p, (size_t)lookup->positions * 4, cudaMemcpyDeviceToHost, ctx->stream));
    TG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return TGPU_OK;
}
