// hap_b200/csrc/snappy_encode.cuh -- K5: second-stage compressor for one fragment of a Hap chunk.
//
// Replaces snappy_compress as the reference calls it from the chunk loop of hap_encode_texture
// (/root/reference/source/hap.c:448-476, call site :453).  The reference's loop is serial over chunks
// and Snappy is serial inside a chunk; here a chunk is cut into independent 32 KiB FRAGMENTS (a raw
// Snappy stream is varint(length) followed by elements, so fragment element streams concatenate
// into one legal chunk stream as long as copies never reach outside their fragment), two resident CTAs
// per SM striding over the fragments, and inside a fragment every 8-byte unit is handled on its own:
//   1. first-occurrence hash of every aligned word (shared-memory table, atomicMin => deterministic);
//   2. each word picks a source: the word one DXT block back when its whole block repeats the
//      previous block (block RLE, decodes as one periodic fill), else the first earlier occurrence
//      of the same word.  Choosing FIRST occurrences makes copies point at literal data, so the
//      decoder's dependency depth stays ~1 (see snappy_decode.cuh);
//   3. runs of words with one distance become copy elements (<= 64 bytes each), everything else
//      literal runs; element sizes are prefix-summed and every word writes its own bytes (for this
//      last step the words are re-dealt so that the lanes of a warp write neighbouring bytes).
// The output differs from Google's encoder byte-for-byte (the reference pins no Snappy bytes,
// SURVEY.md 8c); parity is: the reference's HapDecode reproduces the input exactly.
#pragma once
#include "hap_codes.h"
#include "hap_index.h"
#include "simt.h"

namespace hapb200 {

constexpr int kEncThreads = 512;
constexpr int kEncWarps = kEncThreads / 32;
constexpr int kEncCtasPerSm = 2;            // resident CTAs per SM the kernel is built for (registers and shared memory)
constexpr int kFragBytes = 32768;
constexpr int kFragCap = kFragBytes + 32;   // element stream of a fragment never exceeds n + 3
constexpr int kEncHashBits = 13;
constexpr uint32_t kFragStoredRaw = 0xFFFFFFFFu;  // fragment size marker: chunk must be stored raw
constexpr int kFragEntryPieces = (kFragCap + (1 << kIndexSubLog2) - 1) >> kIndexSubLog2;   // 128-byte pieces of a fragment's stream (hap_index.h)
constexpr int kFragEntryStride = 272;             // bytes reserved per fragment in the entries scratch (multiple of 16)
static_assert(kFragEntryPieces <= kFragEntryStride, "entries of one fragment fit their scratch slot");

// Shared memory of one fragment.  The unit of every decision is 8 BYTES (a DXT1 / RGTC1 block, half a DXT5 block).  Units are
// grouped in STRIPS of 4 consecutive units; thread t owns the two strips t and t + kEncThreads, i.e. units [4t, 4t+4) and
// [4t + kHalfUnits, 4t + kHalfUnits + 4), and keeps them (and every per-unit quantity) in registers.  Shared memory only
// carries what OTHER threads read: the data (random match verification), the hash table, the strip-boundary values of the
// per-unit arrays, and -- for the last step, which re-distributes the units over the threads -- positions and run starts.
// (Round 1 decided per 4-byte word: twice the elements in every step, and 4-byte matches that were demoted again because a
// copy element costs 3 bytes.  Matches that start at an odd word are lost; DXT payloads hardly have any.)
// Two CTAs share an SM, so that one CTA's barrier drains are filled by the other's work.  To fit two, the output step's
// arrays (positions, run starts and the element stream) overlay the hash table, which is dead by then.  (Overlaying the
// element stream on the input units instead, with the output step reading its literal bytes from global memory, was
// measured: K5 5.35 ms per 444 4K Hap Q frames against 5.64 with one 1024-thread CTA -- eight dependent L2 reads per
// thread in the output loop ate most of what the second CTA brings.)
#ifndef HAPB200_K5_ROUNDS
#define HAPB200_K5_ROUNDS 1
#endif
constexpr int kFragUnits = kFragBytes / 8;        // 4096
constexpr int kUnitStrip = 4;                     // units per strip
constexpr int kEncStrips = kFragUnits / (kUnitStrip * kEncThreads);   // strips per thread
constexpr int kHalfUnits = kUnitStrip * kEncThreads;                  // units of all threads' first strips (2048)
static_assert(kEncStrips == 2, "a thread owns two strips: the block scans carry the two halves of the fragment as one packed word");
struct EncodeSmem {
    uint2 data[kFragUnits + 2];                     // input units
    union {
        uint32_t table[1 << kEncHashBits];          // first occurrence of every hashed unit (steps 1 .. 2)
        struct {
            uint16_t b[kFragUnits];                 // run start per unit (step 5)
            uint16_t c[kFragUnits];                 // stream position per unit (step 5)
            alignas(16) uint32_t out[(kFragCap + 3) / 4 + 6];   // the element stream (step 5, copied out in 16-byte words)
        } h;
    } u;
    uint16_t da[kFragUnits];                        // candidate distances (ping) | one of the two holds the final distances,
    uint16_t db[kFragUnits];                        // candidate distances (pong) | the other then the run ends (stored at the run start)
    uint32_t warp_tot[kEncWarps];
    uint32_t entry[kFragEntryStride];               // fragment index: offset of the first element start in every 128 bytes of the stream
    uint32_t total;
};
// Two resident CTAs: 233,472 B of shared memory per SM, of which every CTA reserves 1 KiB for the system.
static_assert(sizeof(EncodeSmem) <= 233472 / kEncCtasPerSm - 1024, "two K5 CTAs fit one SM's shared memory");

__device__ __forceinline__ uint32_t enc_hash(uint2 u) { return ((u.x * 0x9E3779B1u) ^ (u.y * 0x85EBCA6Bu)) >> (32 - kEncHashBits); }
__device__ __forceinline__ bool same_unit(uint2 a, uint2 b) { return a.x == b.x && a.y == b.y; }

__device__ __forceinline__ uint32_t literal_header_bytes(uint32_t len) { return len <= 60 ? 1u : len <= 256 ? 2u : 3u; }

__device__ __forceinline__ void store_strip16(uint16_t *arr, uint32_t base, const uint32_t v[4])
{
    *reinterpret_cast<uint2 *>(arr + base) = make_uint2(v[0] | (v[1] << 16), v[2] | (v[3] << 16));
}

// Per-half max of two 16-bit values packed in one word (the block scans below carry both halves of a fragment at once).
__device__ __forceinline__ uint32_t enc_max_u16x2(uint32_t a, uint32_t b)
{
#ifdef HAPB200_EMU
    const uint32_t lo = (a & 0xFFFFu) > (b & 0xFFFFu) ? (a & 0xFFFFu) : (b & 0xFFFFu), hi = (a >> 16) > (b >> 16) ? (a >> 16) : (b >> 16);
    return lo | (hi << 16);
#else
    return __vmaxu2(a, b);
#endif
}

// Inclusive max / sum over the block of one PACKED value per thread (two 16-bit halves, scanned independently: a sum
// never carries out of the low half because every half-fragment total stays below 2^16); returns the exclusive prefix
// for this thread and the block total, both packed.  Two barriers.  The warp totals are scanned by every warp with
// shuffles (lane w holds the total of warp w) instead of a loop over shared memory.
__device__ __forceinline__ uint32_t enc_block_excl(uint32_t v, bool is_max, uint32_t *total, uint32_t *warp_tot)
{
    static_assert(kEncWarps <= 32 && (kEncWarps & (kEncWarps - 1)) == 0, "one warp total per lane");
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t o = __shfl_up_sync(HAP_FULL_MASK, incl, d);
        if (lane >= d) incl = is_max ? enc_max_u16x2(incl, o) : incl + o;
    }
    uint32_t prev = __shfl_up_sync(HAP_FULL_MASK, incl, 1);
    if (lane == 0) prev = 0;
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    uint32_t wi = lane < kEncWarps ? warp_tot[lane] : 0u;   // (0 is the identity of both operations)
#pragma unroll
    for (int d = 1; d < kEncWarps; d <<= 1) {
        uint32_t o = __shfl_up_sync(HAP_FULL_MASK, wi, d);
        if (lane >= d) wi = is_max ? enc_max_u16x2(wi, o) : wi + o;
    }
    const uint32_t tot = __shfl_sync(HAP_FULL_MASK, wi, kEncWarps - 1);
    uint32_t base = __shfl_sync(HAP_FULL_MASK, wi, warp > 0 ? warp - 1 : 0);
    if (warp == 0) base = 0;
    __syncthreads();
    *total = tot;
    return is_max ? enc_max_u16x2(base, prev) : base + prev;
}

// One fragment: U units (8 bytes each; U <= kFragUnits) already in S.data AND in the caller's registers d[8] (units
// 4t..4t+3, then kHalfUnits+4t..kHalfUnits+4t+3) -> element stream written to S.u.h.out as bytes; returns its size (all
// threads).
// period_units = DXT block size in units (1 or 2).
// FULL = the fragment has all kFragUnits units (31 of 32 fragments of a 1 MiB chunk): every per-unit bounds test
// folds away at compile time.
// Every decision below is a rule over unit indices (atomicMin, one Jacobi round of propagation, max and sum scans in unit
// order), so the stream does not depend on which thread owns which unit.
template <bool FULL>
__device__ __forceinline__ uint32_t compress_fragment(EncodeSmem &S, const uint2 d[8], uint32_t Udyn, uint32_t period_units)
{
    constexpr int kUnitsPerThread = kEncStrips * kUnitStrip;
    const uint32_t t = threadIdx.x;
    const uint32_t U = FULL ? (uint32_t)kFragUnits : Udyn;
    uint32_t i0[kEncStrips], nv[kEncStrips];       // first unit of each of my strips, and its valid units
#pragma unroll
    for (int h = 0; h < kEncStrips; h++) {
        i0[h] = h * kHalfUnits + t * kUnitStrip;
        nv[h] = FULL ? (uint32_t)kUnitStrip : (i0[h] >= U ? 0u : (U - i0[h] < (uint32_t)kUnitStrip ? U - i0[h] : (uint32_t)kUnitStrip));
    }

    // 1. first occurrence of every unit (the table was initialised by the caller, before the barrier)
    uint32_t hsh[kUnitsPerThread];
#pragma unroll
    for (int h = 0; h < kEncStrips; h++)
#pragma unroll
        for (int k = 0; k < kUnitStrip; k++) {
            hsh[h * kUnitStrip + k] = enc_hash(d[h * kUnitStrip + k]);
            if ((uint32_t)k < nv[h]) atomicMin(&S.u.table[hsh[h * kUnitStrip + k]], i0[h] + k);
        }
    __syncthreads();

    // 2. candidate distance per unit: first earlier occurrence, or one block back when the whole block repeats
    uint32_t dd[kUnitsPerThread];
#pragma unroll
    for (int h = 0; h < kEncStrips; h++) {
        const uint2 *dh = d + h * kUnitStrip;
        uint32_t *ddh = dd + h * kUnitStrip;
        const uint32_t s0 = i0[h];
#pragma unroll
        for (int k = 0; k < kUnitStrip; k++) {
            ddh[k] = 0;
            if ((uint32_t)k < nv[h]) {
                const uint32_t c = S.u.table[hsh[h * kUnitStrip + k]];
                if (c < s0 + k && same_unit(S.data[c], dh[k])) ddh[k] = s0 + k - c;
            }
        }
        if (period_units == 2) {
            // DXT5-sized blocks: units (2b, 2b+1); the block repeats when both units equal the block before
            const uint2 p0 = s0 >= 2 ? S.data[s0 - 2] : make_uint2(0, 0), p1 = s0 >= 2 ? S.data[s0 - 1] : make_uint2(0, 0);
            if (s0 >= 2 && nv[h] >= 2 && same_unit(p0, dh[0]) && same_unit(p1, dh[1])) { ddh[0] = 2; ddh[1] = 2; }
            if (nv[h] >= 4 && same_unit(dh[0], dh[2]) && same_unit(dh[1], dh[3])) { ddh[2] = 2; ddh[3] = 2; }
        } else {
            const uint2 p = s0 >= 1 ? S.data[s0 - 1] : make_uint2(0, 0);
            if (s0 >= 1 && nv[h] >= 1 && same_unit(p, dh[0])) ddh[0] = 1;
#pragma unroll
            for (int k = 1; k < kUnitStrip; k++)
                if ((uint32_t)k < nv[h] && same_unit(dh[k - 1], dh[k])) ddh[k] = 1;
        }
        store_strip16(S.da, s0, ddh);
    }
    __syncthreads();

    // 2b. propagation: a unit that is not yet part of a run adopts its left (else right) neighbour's distance when its own
    //     data also matches there.  First occurrences of neighbouring units often point at different earlier blocks; this
    //     re-aligns them and recovers most of what a greedy match extension finds.
    uint16_t *cur = S.da, *nxt = S.db;
    {
#pragma unroll 1
        for (int round = 0; round < HAPB200_K5_ROUNDS; round++) {
            uint32_t nd[kUnitsPerThread];
#pragma unroll
            for (int h = 0; h < kEncStrips; h++) {
                const uint32_t s0 = i0[h];
                const uint32_t lb = s0 > 0 ? cur[s0 - 1] : 0u;
                const uint32_t rb = s0 + kUnitStrip < U ? cur[s0 + kUnitStrip] : 0u;
#pragma unroll
                for (int k = 0; k < kUnitStrip; k++) {
                    const int u = h * kUnitStrip + k;
                    const uint32_t l = k > 0 ? dd[u - 1] : lb, r = k < kUnitStrip - 1 ? dd[u + 1] : rb;
                    const uint32_t cd = dd[u], i = s0 + k;
                    nd[u] = cd;
                    if ((uint32_t)k < nv[h] && !(cd != 0 && (cd == l || cd == r))) {
                        // one look-up decides: the left neighbour's distance if there is one, else the right one's
                        const uint32_t cand = l != 0 ? l : r;
                        if (cand != 0 && i >= cand && same_unit(S.data[i - cand], d[u])) nd[u] = cand;
                        else if (l != 0 && r != 0 && r != l && i >= r && same_unit(S.data[i - r], d[u])) nd[u] = r;
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < kUnitsPerThread; u++) dd[u] = nd[u];
#pragma unroll
            for (int h = 0; h < kEncStrips; h++) store_strip16(nxt, i0[h], dd + h * kUnitStrip);
            __syncthreads();
            uint16_t *tmp = cur; cur = nxt; nxt = tmp;
        }
    }
    // `cur` holds the final distances (read across strip boundaries below, and by the output step); the other buffer is
    // free: it takes the run ends.
    // (Measured on the emulator cases: with 8-byte units ONE round recovers what two did -- frame sizes equal on picture
    // content, +0.1 .. 0.5 % on the stitched random cases; none costs 5 .. 16 %.)
    const uint16_t *fin = cur;
    uint16_t *ends = nxt;
    // (a single matching unit is kept: an 8-byte copy costs 3 bytes)

    // 3. run start of every unit (max-scan of "i+1 where a run starts") and run ends (stored at the run start)
    uint32_t rs[kUnitsPerThread];
    {
        uint32_t last[kEncStrips];  // (index + 1) of the last run start inside each strip so far
        uint32_t loc[kUnitsPerThread];
#pragma unroll
        for (int h = 0; h < kEncStrips; h++) {
            const uint32_t s0 = i0[h];
            const uint32_t lb = s0 > 0 ? fin[s0 - 1] : 0u;
            last[h] = 0;
#pragma unroll
            for (int k = 0; k < kUnitStrip; k++) {
                const int u = h * kUnitStrip + k;
                const uint32_t prev = k > 0 ? dd[u - 1] : lb;
                if ((uint32_t)k < nv[h] && (s0 + k == 0 || dd[u] != prev)) last[h] = s0 + k + 1;
                loc[u] = last[h];
            }
        }
        uint32_t tot;
        const uint32_t ex = enc_block_excl(last[0] | (last[1] << 16), true, &tot, S.warp_tot);
        // strips of the second half follow every strip of the first half in unit order
        const uint32_t carry[kEncStrips] = {ex & 0xFFFFu, (tot & 0xFFFFu) > (ex >> 16) ? (tot & 0xFFFFu) : (ex >> 16)};
#pragma unroll
        for (int u = 0; u < kUnitsPerThread; u++) rs[u] = (loc[u] ? loc[u] : carry[u / kUnitStrip]) - 1;
#pragma unroll
        for (int h = 0; h < kEncStrips; h++) {
            const uint32_t s0 = i0[h];
            const uint32_t rb = s0 + kUnitStrip < U ? fin[s0 + kUnitStrip] : 0xFFFFFFFFu;
#pragma unroll
            for (int k = 0; k < kUnitStrip; k++) {
                const int u = h * kUnitStrip + k;
                const uint32_t nx = k < kUnitStrip - 1 ? dd[u + 1] : rb;
                if ((uint32_t)k < nv[h] && (s0 + k + 1 == U || nx != dd[u])) ends[rs[u]] = (uint16_t)(s0 + k);
            }
        }
    }
    __syncthreads();

    // 4. bytes each unit contributes and their exclusive prefix sum
    uint32_t pos[kUnitsPerThread];
    {
        uint32_t run[kEncStrips];
#pragma unroll
        for (int h = 0; h < kEncStrips; h++) {
            run[h] = 0;
#pragma unroll
            for (int k = 0; k < kUnitStrip; k++) {
                const int u = h * kUnitStrip + k;
                uint32_t c = 0;
                if ((uint32_t)k < nv[h]) {
                    const uint32_t i = i0[h] + k;
                    if (dd[u] == 0) {
                        c = 8;
                        if (i == rs[u]) c += literal_header_bytes(8u * (ends[i] - i + 1));
                    } else if (((i - rs[u]) & 7) == 0) {
                        c = 3;      // one copy element per 64 bytes of the run
                    }
                }
                pos[u] = run[h];
                run[h] += c;
            }
        }
        uint32_t tot;
        const uint32_t ex = enc_block_excl(run[0] | (run[1] << 16), false, &tot, S.warp_tot);
        const uint32_t base[kEncStrips] = {ex & 0xFFFFu, (tot & 0xFFFFu) + (ex >> 16)};
#pragma unroll
        for (int u = 0; u < kUnitsPerThread; u++) pos[u] += base[u / kUnitStrip];
        if (t == 0) S.total = (tot & 0xFFFFu) + (tot >> 16);
    }

    // 5. every unit writes its own bytes.  Ownership changes for this step: thread t takes units t, t + kEncThreads, ... so
    //    that the lanes of a warp write neighbouring bytes of the stream (with the strip layout they sit 32 bytes apart: bank
    //    conflicts on every store).  Positions and run starts travel through shared memory as 16-bit strips, the distances
    //    are the final ones of step 2b.
    //    Inside a literal run the stream is the input shifted by (p & 3) bytes, so a unit writes TWO aligned 32-bit words
    //    made of its own bytes and the next unit's first bytes; only the two ends of a run, headers and copy elements are
    //    written bytewise.
#pragma unroll
    for (int h = 0; h < kEncStrips; h++) {
        store_strip16(S.u.h.c, i0[h], pos + h * kUnitStrip);
        store_strip16(S.u.h.b, i0[h], rs + h * kUnitStrip);
    }
    __syncthreads();
    uint8_t *out = reinterpret_cast<uint8_t *>(S.u.h.out);
#pragma unroll 1
    for (int j = 0; j < kUnitsPerThread; j++) {
        const uint32_t i = t + (uint32_t)j * kEncThreads;
        if (!FULL && i >= U) continue;
        const uint32_t dist = fin[i], rs_i = S.u.h.b[i];
        uint32_t p = S.u.h.c[i];
        if (dist == 0) {
            const uint2 w = S.data[i];
            const uint32_t e = ends[rs_i];   // last unit of this literal run
            if (i == rs_i) {
                const uint32_t len = 8u * (e - i + 1);
                atomicMin(&S.entry[p >> kIndexSubLog2], p & ((1u << kIndexSubLog2) - 1u));   // an element starts here
                if (len <= 60) {
                    out[p++] = (uint8_t)((len - 1) << 2);
                } else if (len <= 256) {
                    out[p++] = (uint8_t)(60 << 2);
                    out[p++] = (uint8_t)(len - 1);
                } else {
                    out[p++] = (uint8_t)(61 << 2);
                    out[p++] = (uint8_t)(len - 1);
                    out[p++] = (uint8_t)((len - 1) >> 8);
                }
            }
            const uint32_t sh = p & 3u;
            if (sh == 0) {
                *reinterpret_cast<uint32_t *>(out + p) = w.x;
                *reinterpret_cast<uint32_t *>(out + p + 4) = w.y;
            } else {
                const uint32_t a1 = (p & ~3u) + 4u;   // the first aligned word behind p
                if (i == rs_i)
                    for (uint32_t q = 0; q < 4u - sh; q++) out[p + q] = (uint8_t)(w.x >> (8 * q));   // the run's first bytes
                *reinterpret_cast<uint32_t *>(out + a1) = __funnelshift_r(w.x, w.y, 8 * (4u - sh));
                if (i < e) {
                    *reinterpret_cast<uint32_t *>(out + a1 + 4) = __funnelshift_r(w.y, S.data[i + 1].x, 8 * (4u - sh));
                } else {
                    for (uint32_t q = 0; q < sh; q++) out[a1 + 4 + q] = (uint8_t)(w.y >> (8 * (4u - sh + q)));   // the run's last bytes
                }
            }
        } else if (((i - rs_i) & 7) == 0) {
            const uint32_t left = ends[rs_i] - i + 1;          // units left in the run
            const uint32_t len = 8u * (left < 8 ? left : 8);    // 8..64 bytes
            const uint32_t off = 8u * dist;
            atomicMin(&S.entry[p >> kIndexSubLog2], p & ((1u << kIndexSubLog2) - 1u));       // an element starts here
            out[p] = (uint8_t)(2u | ((len - 1) << 2));          // copy with 2-byte offset
            out[p + 1] = (uint8_t)off;
            out[p + 2] = (uint8_t)(off >> 8);
        }
    }
    __syncthreads();
    return S.total;
}

// Geometry of one texture section of a batch of identical frames (host fills it once per call).
struct SectionGeom {
    uint32_t bytes;            // texture bytes (hap.c: inputBufferBytes)
    uint32_t chunks;           // limited chunk count (hap.c:277-300)
    uint32_t chunk_bytes;      // bytes / chunks (hap.c:433)
    uint32_t frags_per_chunk;  // ceil(chunk_bytes / kFragBytes)
    uint32_t period_words;     // DXT block size in 4-byte words (2 or 4)
    uint32_t compress;         // 1 = HapCompressorSnappy requested and chunk_bytes % 8 == 0
    uint32_t inv_frags_per_chunk;  // floor(2^32 / frags_per_chunk), 0xFFFFFFFF for 1 (fast_divmod)
    uint32_t frag_base;        // index of this section's first fragment inside a frame
    uint32_t fmt_nibble;       // wire format id (hap.c:45-51)
    uint32_t top_hdr;          // 4 or 8 (hap.c:398-405, :425-428)
    uint32_t want_snappy;      // caller passed HapCompressorSnappy
    uint64_t in_offset;        // this texture's bytes of frame f start at dxt + in_offset + f * in_stride
    uint64_t in_stride;
};

struct FrameGeom {
    uint32_t sections;         // 1 or 2
    uint32_t outer_hdr;        // 0 (single texture), 4 or 8 (hap.c:563-576)
    uint32_t frags_per_frame;
    uint32_t inv_frags_per_frame;  // floor(2^32 / frags_per_frame), 0xFFFFFFFF for 1
    SectionGeom s[2];
};

// Where fragment `gfrag` of the batch lives and how long it is.
struct FragRef {
    const uint8_t *in;
    bool second;         // fragment of the frame's second texture
    uint32_t units;      // 8-byte units; 0: the section is not compressed (fragment stored raw)
};
// x / d and x % d with a multiplication: magic = floor(2^32 / d) (0xFFFFFFFF for d = 1), one correction step
__device__ __forceinline__ uint32_t fast_divmod(uint32_t x, uint32_t d, uint32_t magic, uint32_t &rem)
{
#ifdef HAPB200_EMU
    rem = x % d;
    (void)magic;
    return x / d;
#else
    uint32_t q = __umulhi(x, magic);
    uint32_t r = x - q * d;
    while (r >= d) { q++; r -= d; }
    rem = r;
    return q;
#endif
}
__device__ __forceinline__ FragRef locate_fragment(const uint8_t *dxt, const FrameGeom &G, uint32_t gfrag)
{
    uint32_t f;
    const uint32_t frame = fast_divmod(gfrag, G.frags_per_frame, G.inv_frags_per_frame, f);
    const bool second = G.sections == 2 && f >= G.s[1].frag_base;
    const uint32_t frag_base = second ? G.s[1].frag_base : G.s[0].frag_base, fpc = second ? G.s[1].frags_per_chunk : G.s[0].frags_per_chunk;
    const uint32_t inv_fpc = second ? G.s[1].inv_frags_per_chunk : G.s[0].inv_frags_per_chunk;
    const uint32_t chunk_bytes = second ? G.s[1].chunk_bytes : G.s[0].chunk_bytes, compress = second ? G.s[1].compress : G.s[0].compress;
    const uint64_t in_stride = second ? G.s[1].in_stride : G.s[0].in_stride, in_offset = second ? G.s[1].in_offset : G.s[0].in_offset;
    uint32_t j;
    const uint32_t chunk = fast_divmod(f - frag_base, fpc, inv_fpc, j);
    FragRef r;
    r.in = dxt + (uint64_t)frame * in_stride + in_offset + (uint64_t)chunk * chunk_bytes + (uint64_t)j * kFragBytes;
    const uint32_t left = chunk_bytes - j * kFragBytes;
    r.units = compress ? (left < (uint32_t)kFragBytes ? left : (uint32_t)kFragBytes) >> 3 : 0u;
    r.second = second;
    return r;
}

// A strip of 4 units of a fragment, from global memory: two 16-byte loads when possible
__device__ __forceinline__ void load_strip(const FragRef &fr, uint32_t i0, uint2 d[4])
{
    if ((((uintptr_t)fr.in) & 15) == 0 && i0 + kUnitStrip <= fr.units) {
        const uint4 *in4 = reinterpret_cast<const uint4 *>(fr.in) + (i0 >> 1);
        const uint4 a = in4[0], b = in4[1];
        d[0] = make_uint2(a.x, a.y); d[1] = make_uint2(a.z, a.w); d[2] = make_uint2(b.x, b.y); d[3] = make_uint2(b.z, b.w);
    } else {
#pragma unroll
        for (int k = 0; k < kUnitStrip; k++) {
            const uint32_t i = i0 + k;
            d[k] = make_uint2(0, 0);
            if (i < fr.units) {
                const uint8_t *b = fr.in + 8 * (size_t)i;
                d[k].x = b[0] | (b[1] << 8) | (b[2] << 16) | ((uint32_t)b[3] << 24);
                d[k].y = b[4] | (b[5] << 8) | (b[6] << 16) | ((uint32_t)b[7] << 24);
            }
        }
    }
}

// A fixed grid (kEncCtasPerSm resident CTAs per SM) strides over the nfrag = frames * frags_per_frame fragments of the
// batch.  The HBM latency of a fragment's input and the turn-over between fragments are covered by the other CTA on the
// same SM, which is at a different phase of its own fragment.
// dxt: base pointer of the texture bytes; scratch: [nfrag][kFragCap]; frag_size: [nfrag] (kFragStoredRaw when the
// fragment was not compressed); frag_entries: [nfrag][kFragEntryStride] or nullptr (fragment index, hap_index.h).
__global__ void __launch_bounds__(kEncThreads, kEncCtasPerSm) snappy_encode_fragments_kernel(
    const uint8_t *__restrict__ dxt, FrameGeom G, uint32_t nfrag, uint8_t *__restrict__ scratch, uint32_t *__restrict__ frag_size,
    uint8_t *__restrict__ frag_entries)
{
    HAP_DYN_SMEM(smem_raw);
    EncodeSmem &S = *reinterpret_cast<EncodeSmem *>(smem_raw);
    const int t = threadIdx.x;
    for (uint32_t gfrag = blockIdx.x; gfrag < nfrag; gfrag += gridDim.x) {
        const FragRef cur = locate_fragment(dxt, G, gfrag);
        if (cur.units == 0) {
            if (t == 0) frag_size[gfrag] = kFragStoredRaw;
            continue;
        }
        const uint32_t U = cur.units;
        uint2 d[kEncStrips * kUnitStrip];
#pragma unroll
        for (int h = 0; h < kEncStrips; h++) {
            const uint32_t i0 = h * kHalfUnits + (uint32_t)t * kUnitStrip;
            uint2 *dh = d + h * kUnitStrip;
            load_strip(cur, i0, dh);
            *reinterpret_cast<uint4 *>(&S.data[i0]) = make_uint4(dh[0].x, dh[0].y, dh[1].x, dh[1].y);
            *reinterpret_cast<uint4 *>(&S.data[i0 + 2]) = make_uint4(dh[2].x, dh[2].y, dh[3].x, dh[3].y);
        }
        {
            uint4 *tb = reinterpret_cast<uint4 *>(S.u.table);
            const uint4 ones = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
            for (int q = t; q < (1 << kEncHashBits) / 4; q += kEncThreads) tb[q] = ones;
            if (t < kFragEntryStride) S.entry[t] = kIndexNoEntry;
        }
        __syncthreads();
        const uint32_t period_units = (cur.second ? G.s[1].period_words : G.s[0].period_words) >> 1;   // 8-byte blocks: 1, 16-byte blocks: 2
        const uint32_t total = U == (uint32_t)kFragUnits ? compress_fragment<true>(S, d, U, period_units)
                                                         : compress_fragment<false>(S, d, U, period_units);
        uint8_t *o = scratch + (uint64_t)gfrag * kFragCap;
        const uint4 *o4s = reinterpret_cast<const uint4 *>(S.u.h.out);
        uint4 *o4 = reinterpret_cast<uint4 *>(o);       // (scratch slots are kFragCap = 32800 bytes apart: 16-byte aligned)
        for (uint32_t i = t; i < (total + 15) / 16; i += kEncThreads) o4[i] = o4s[i];
        if (frag_entries != nullptr && t < kFragEntryStride) frag_entries[(uint64_t)gfrag * kFragEntryStride + t] = (uint8_t)S.entry[t];
        if (t == 0) frag_size[gfrag] = total;
        __syncthreads();   // S.data and the tables (with the element stream) are rewritten by the next fragment
    }
}

}  // namespace hapb200
