// rice_vs.cuh -- Rice decode (K5), second generation: parallelism INSIDE a stream.
//
// rice::RiceDecoder::generateDecodedUnsignedInts (src/rice/rice_decoder.cpp:21-44) is a sequential
// parse: symbol n+1 starts where symbol n ended.  One lane per stream therefore gives a batch of
// 25 838 streams (BASELINE config 3) only 808 warps, each crawling along one dependent chain.
// Here the 2048 symbols of a stream are cut into S parts of 2048/S symbols ("virtual streams") that
// are decoded by S different lanes; what makes that possible is a table of the S-1 bit positions at
// which the parts begin, produced by a first, much cheaper pass:
//
//   k_rice_split_index<S>   S lanes per stream, each parsing ONLY the symbol boundaries of one
//                           contiguous 1/S of the stream's bits, speculatively: a lane that starts
//                           in the middle of the stream does not know where a symbol begins.  Rice
//                           codes resynchronise: the lane before it keeps parsing past its own end
//                           until it lands on a boundary the next lane also found; from there on
//                           the next lane's boundaries are the true ones.  A prefix sum of the
//                           per-lane symbol counts then names the lane (and, through sparse
//                           checkpoints, the bit) where symbol t*2048/S begins.
//   k_rice_decode_vc        one lane per virtual stream, decoding values.
//
// Both kernels parse from a three-word register window over a small ring in shared memory per lane, so
// that no shared-memory load sits on the symbol-to-symbol dependency chain.  The split index tops its
// lane's ring up itself with 16-byte cp.async copies (VsStream); the decoder's rings are topped up by the
// whole warp in 128-byte segments and bit-reversed in place (VsCoopStream).  The decoder stages its values
// in a shared tile and writes them as whole row segments (128-byte lines) instead of one 16-byte store per
// lane.
//
// Nothing is taken on trust: part l must end exactly where the table says part l+1 begins (part 0
// starts at bit 0, so by induction every part is the sequential parse); a stream that fails that
// check, cannot be split, or meets a symbol the fast paths do not handle is flagged, and the
// general lane-per-stream kernel (k_rice_decode, rice.cuh) decodes it again afterwards.  With S = 1
// the second kernel alone is the large-batch decoder.
#pragma once

#include "rice.cuh"

namespace selab200 {

constexpr uint32_t kNoSplit = 0xffffffffu;
constexpr int kVsWarps = 4;

struct RiceVsParams {
    const selab200_subframe_desc *descs;
    uint32_t n_sub, channels;
    const uint32_t *words;
    unsigned long long n_words;
    int32_t *out;      // [n_sub][2048]
    uint32_t *table;   // [n_sub][S-1]: bit position (from the stream's first bit) of symbol t*2048/S
    uint32_t *flags;   // [n_sub]: 1 = the general kernel must decode this stream
    int32_t *status;
};

__device__ __forceinline__ bool rice_desc_ok(const selab200_subframe_desc &d, uint32_t channels, unsigned long long n_words)
{
    return d.channel < channels && d.parent_channel < channels && d.subframe_type <= 1 && d.lpc_order <= kMaxOrder &&
           d.refl_rice_param < 32 && d.res_rice_param < 32 && d.samples == kFrame &&
           d.refl_offset + d.refl_words <= n_words && d.res_offset + d.res_words <= n_words &&
           !(d.subframe_type == 1 && d.parent_channel == d.channel);
}

// Position of the highest set bit, 0xffffffff for zero: the raw FLO, without the 31 - x of __clz.
__device__ __forceinline__ uint32_t bfind_u32(uint32_t x)
{
    uint32_t r;
    asm("bfind.u32 %0, %1;" : "=r"(r) : "r"(x));
    return r;
}

// convertUnsignedToSigned (src/rice/rice_decoder.cpp:46-52) in three instructions: the sign is bit 0 of u,
// sign-extended by a one-bit signed field extract.
__device__ __forceinline__ int32_t unzigzag3(uint32_t u)
{
    int32_t s;
    asm("bfe.s32 %0, %1, 0, 1;" : "=r"(s) : "r"(u));
    return (int32_t)(u >> 1) ^ s;
}

__device__ __forceinline__ uint32_t lds_u32(uint32_t saddr)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}

// ------------------------------------------------------------------ the lane's ring --
//
// RING words in one row of shared memory, word w of the stream (counted from its 16-byte aligned base) at
// byte ((4w + rot) & (4*RING - 1)) of the row; rot = 16 * lane spreads the lanes over the banks.  Rows are
// 4*RING-aligned in the shared window: addresses are formed with OR.
template <int RING>
struct VsRing {
    static constexpr uint32_t kMask = RING * 4 - 1;
    uint32_t row, rot;  // shared-space byte address of the row; rotation
    const uint4 *gvec;  // the stream from its 16-byte aligned base
    int total_bytes;    // bytes from gvec to the end of the stream; everything behind reads as zero
    __device__ __forceinline__ uint32_t word_addr(uint32_t w) const { return row | ((4 * w + rot) & kMask); }
    __device__ __forceinline__ uint32_t word(uint32_t w) const { return lds_u32(word_addr(w)); }
    __device__ __forceinline__ void issue(uint32_t fv) const // vector fv: words [4fv, 4fv+4)
    {
        const uint32_t off = 16 * fv;
        const uint32_t dst = row | ((off + rot) & kMask);
        if ((int)(off + 16) <= total_bytes) { // the common case: a whole vector of the stream
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(reinterpret_cast<const char *>(gvec) + off) : "memory");
        } else { // the ragged end, and zeros behind it
            const int rem = total_bytes - (int)off;
            const uint32_t sz = rem <= 0 ? 0u : (uint32_t)rem;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(reinterpret_cast<const char *>(gvec) + (sz ? off : 0u)), "r"(sz) : "memory");
        }
    }
};

__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// The streaming state of a lane: a window of three words in registers (r0 = word wb - 1 holds the current
// bit, r1, and r2 loaded one word ahead of its first use) over the ring.  ROUND symbols of at most 32 bits
// are parsed between two boundaries; at a boundary the ring is topped up as far as the words still needed
// allow, and the copies issued at the previous boundary are retired.
// A round reads at most ROUND + 2 words past r1.  With RING >= 2 * ROUND + 16 what landed a boundary ago
// always covers that; a smaller ring (half the shared memory, twice the warps per SM) covers it for
// ordinary streams and otherwise waits for the copies just issued (RING >= ROUND + 16 suffices then).
template <int RING, int ROUND>
struct VsStream {
    static_assert(RING >= ROUND + 16 && (RING & (RING - 1)) == 0, "ring too small for the round");
    VsRing<RING> rg;
    uint32_t pos;         // current bit, counted from the aligned base
    uint32_t r0, r1, r2;  // window
    uint32_t wa;          // running byte offset (rotated) of r2's word
    uint32_t fv, rv;      // next vector to request / first vector not yet landed
    uint32_t cv_next;     // vectors below cv_next have been requested by the previous boundary
    uint32_t ce;          // words below ce have landed

    __device__ __forceinline__ uint32_t wb() const { return (pos >> 5) + 1; }
    __device__ __forceinline__ void load_window()
    {
        const uint32_t w = wb();
        r0 = rg.word(w - 1);
        r1 = rg.word(w);
        r2 = rg.word(w + 1);
        wa = 4 * (w + 1) + rg.rot;
    }
    __device__ __forceinline__ void retire(uint32_t upto) // vectors below `upto` have landed
    {
        if (upto > rv) {
            rv = upto;
            ce = 4 * upto;
        }
    }
    // (Re)start at bit p.  Every earlier copy of this lane must have landed.
    __device__ __forceinline__ void prime(uint32_t p)
    {
        pos = p;
        const uint32_t w = wb();
        fv = rv = (w - 1) >> 2;
        const uint32_t first = (w + ROUND + 2) >> 2; // last vector the first round can touch
        while (fv <= first) {
            rg.issue(fv);
            fv++;
        }
        cp_async_commit();
        const uint32_t landed = fv;
        const uint32_t lim = (w + RING - 5) >> 2; // vector v overwrites words [4v - RING, 4v - RING + 3]; below w - 1 all is dead
        while (fv <= lim) {
            rg.issue(fv);
            fv++;
        }
        cp_async_commit();
        cp_async_wait<1>();
        ce = 4 * rv;
        retire(landed);
        cv_next = fv;
        load_window();
    }
    __device__ __forceinline__ void boundary()
    {
        const uint32_t w = wb();
        const uint32_t lim = (w + RING - 5) >> 2;
        while (fv <= lim) {
            rg.issue(fv);
            fv++;
        }
        cp_async_commit();
        cp_async_wait<1>(); // everything but the group just committed has landed
        retire(cv_next);
        cv_next = fv;
        if (RING < 2 * ROUND + 16 && ce < w + ROUND + 3) { // a dense stretch: the round may outrun what has landed
            cp_async_wait<0>();
            retire(fv);
        }
    }
    // one word further (the parser crossed a 32-bit boundary)
    __device__ __forceinline__ void advance()
    {
        r0 = r1;
        r1 = r2;
        wa += 4;
        r2 = lds_u32(rg.row | (wa & VsRing<RING>::kMask));
    }
};

// ------------------------------------------------------------------ the warp's rings, filled together --
//
// Per-lane cp.async top-ups as in VsStream cost a 16-byte request to 32 different lines per instruction: at
// scale the load/store unit replays of those requests, not the parse, bound a decoder built that way
// (measured: with the top-ups removed it ran 2.3x faster).  Here the 32 rings of a warp are topped up
// COOPERATIVELY in 128-byte segments: a ring is two segments of 32 words; a lane whose parser has left a
// segment puts its row on a list, and eight lanes copy one row's next segment (8 x 16 bytes = one whole
// line) -- four rows, four lines per instruction instead of 32 -- and, when it has landed, reverse it the
// same way.  The value parser wants the stream MSB first (a leading-zero count finds the terminator, the
// payload reads as a number): reversing each word once, in place, costs one BREV per word instead of one per
// symbol.  The copies bypass L1 (cp.async.cg): every line is fetched exactly once, and letting those lines
// allocate in the 16 KB of L1 the kernel leaves was the second wall (1.43 -> 1.19 ms at 413 k streams).  All
// calls are warp-convergent.
struct VsCoopMeta { // per warp, in shared memory
    // rows that want a segment, each entry written by the row's owner and read by the eight lanes that copy
    // it (and, a boundary later, reverse it): x, y = source address of the segment; z = bytes of stream left
    // from there (<= 0: zeros only); w = shared byte address of the segment's first word in the row's ring.
    // Two lists: the one being filled now and the one whose copies are landing.
    uint4 list[2][32];
};

// add / subtract on the FMA pipe (IMAD.IADD): the parser is bound by the ALU pipe (shifts, logic, compares)
__device__ __forceinline__ uint32_t fma_add(uint32_t a, uint32_t b)
{
    uint32_t d;
    asm("mad.lo.u32 %0, %1, 1, %2;" : "=r"(d) : "r"(a), "r"(b));
    return d;
}
__device__ __forceinline__ uint32_t fma_sub(uint32_t a, uint32_t b) // a - b
{
    uint32_t d;
    asm("mad.lo.u32 %0, %1, 0xffffffff, %2;" : "=r"(d) : "r"(b), "r"(a));
    return d;
}

template <int ROUND>
struct VsCoopStream {
    static constexpr int kRing = 64, kSeg = 32;     // words
    static constexpr uint32_t kMask = kRing * 4 - 1;
    static_assert(ROUND <= 16, "a round must not outrun one segment's slack");
    uint32_t row, rot;     // this lane's ring row (shared byte address, 256-aligned) and rotation
    uint32_t rows0;        // shared byte address of the warp's row 0
    unsigned char *sbase;  // the kernel's dynamic shared memory as a pointer, and its shared byte address
    uint32_t s0;
    VsCoopMeta *meta;
    unsigned long long gbase; // this lane's stream from its 16-byte aligned base
    int total_bytes;          // bytes from gbase to the end of the stream (zeros behind)
    uint32_t pos, r0, r1, r2, wa;
    uint32_t fs;           // next segment to request
    bool pending;          // the segment requested at the previous boundary is still on its way
    int cur, n_prev;       // (warp-uniform) the list being filled; rows on the other one, whose copies are landing
    uint32_t ce;           // words below ce are readable (landed and reversed)
    uint32_t seg_limit;    // no segment beyond this one is ever needed

    __device__ __forceinline__ uint32_t wb() const { return (pos >> 5) + 1; }
    __device__ __forceinline__ uint32_t word_addr(uint32_t w) const { return row | ((4 * w + rot) & kMask); }
    __device__ __forceinline__ uint32_t word(uint32_t w) const { return lds_u32(word_addr(w)); }
    __device__ __forceinline__ void load_window()
    {
        const uint32_t w = wb();
        r0 = word(w - 1);
        r1 = word(w);
        r2 = word(w + 1);
        wa = 4 * (w + 1) + rot;
    }
    __device__ __forceinline__ void advance()
    {
        r0 = r1;
        r1 = r2;
        wa = fma_add(wa, 4);
        r2 = lds_u32(row | (wa & kMask));
    }
    __device__ __forceinline__ void setup(unsigned char *smem, uint32_t rows0_, VsCoopMeta *m, const uint4 *gvec, int total_bytes)
    {
        const int lane = lane_id();
        sbase = smem;
        s0 = (uint32_t)__cvta_generic_to_shared(smem);
        rows0 = rows0_;
        row = rows0_ + (uint32_t)lane * (kRing * 4);
        rot = (16u * lane) & kMask;
        meta = m;
        gbase = (unsigned long long)reinterpret_cast<uintptr_t>(gvec);
        this->total_bytes = total_bytes;
        seg_limit = ((uint32_t)total_bytes >> 7) + 2;
    }
    // Copy one segment for every lane with `want` (its `fs`) through list `which`; returns how many rows.  Does not commit.
    __device__ __forceinline__ int fill(bool want, int which)
    {
        const int lane = lane_id();
        const uint32_t mask = __ballot_sync(kFull, want);
        if (mask == 0)
            return 0;
        uint4 *list = meta->list[which];
        if (want) {
            const uint32_t off = fs * 128u;
            const int rem = total_bytes - (int)off;
            const unsigned long long src = gbase + (rem > 0 ? off : 0u);
            list[__popc(mask & ((1u << lane) - 1u))] =
                make_uint4((uint32_t)src, (uint32_t)(src >> 32), (uint32_t)rem, row | ((off + rot) & kMask));
        }
        __syncwarp();
        const int n = __popc(mask);
        const uint32_t piece = 16u * (lane & 7);
        for (int it = 0; it * 4 < n; it++) { // four rows per instruction, eight lanes x 16 bytes each
            const int idx = it * 4 + (lane >> 3);
            if (idx < n) {
                const uint4 e = list[idx];
                const int rem = (int)e.z - (int)piece;
                const uint32_t sz = rem <= 0 ? 0u : rem < 16 ? (uint32_t)rem : 16u;
                const unsigned long long src = (((unsigned long long)e.y << 32) | e.x) + (sz ? piece : 0u);
                // the segment may wrap inside the row only at its end: it starts on a 128-byte boundary of the rotated row
                const uint32_t dst = (e.w & ~kMask) | ((e.w + piece) & kMask);
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz) : "memory");
            }
        }
        return n;
    }
    // The segments of list `which` have landed: the lanes that copied them reverse them, one 16-byte piece each
    // (all 32 lanes busy -- a lane reversing its own whole segment would leave the other 31 idle).  Convergent.
    __device__ __forceinline__ void reverse_list(int which, int n) const
    {
        const int lane = lane_id();
        const uint4 *list = meta->list[which];
        const uint32_t piece = 16u * (lane & 7);
        for (int it = 0; it * 4 < n; it++) {
            const int idx = it * 4 + (lane >> 3);
            if (idx < n) {
                const uint32_t w0 = list[idx].w;
                const uint32_t a = (w0 & ~kMask) | ((w0 + piece) & kMask);
                // (plain loads through the shared array: behind an inline-asm load ptxas lowers BREV to three instructions)
                uint4 *q = reinterpret_cast<uint4 *>(sbase + (a - s0));
                uint4 v = *q;
                v.x = __brev(v.x), v.y = __brev(v.y), v.z = __brev(v.z), v.w = __brev(v.w);
                *q = v;
            }
        }
        __syncwarp(); // reversed words visible to their owners; the list is free again
    }
    // (Re)start the lanes with `want` at bit p.  Convergent.
    __device__ __forceinline__ void prime(uint32_t p, bool want)
    {
        cp_async_wait<0>();
        __syncwarp();
        if (want) {
            pos = p;
            fs = (wb() - 1) >> 5;
        }
        const int n0 = fill(want, 0);
        if (want)
            fs++;
        const int n1 = fill(want, 1);
        if (want)
            fs++;
        cp_async_commit();
        cp_async_wait<0>();
        __syncwarp();
        reverse_list(0, n0);
        reverse_list(1, n1);
        if (want) {
            ce = kSeg * fs;
            load_window();
        }
        cur = 0;
        n_prev = 0;
        pending = false;
    }
    // Top-up for the lanes with `want`.  Convergent.
    __device__ __forceinline__ void boundary(bool want)
    {
        // segment fs goes where segment fs - 2 was: free once the parser (r0 = word wb - 1) has left it
        const uint32_t w = wb();
        const bool ready = want && kSeg * (fs - 1) <= w - 1 && fs <= seg_limit;
        const int n_cur = fill(ready, cur);
        cp_async_commit();
        cp_async_wait<1>(); // what the previous boundary requested has landed ...
        __syncwarp();       // ... for every lane of the warp
        reverse_list(cur ^ 1, n_prev);
        if (pending)
            ce = kSeg * fs; // (fs still counts the segment requested at the previous boundary, not this one's)
        pending = ready;
        if (ready)
            fs++;
        // A round reads at most ROUND + 2 words past r1.  A parser that entered its last landed segment late in
        // a dense stretch needs the segment requested just now: wait for it (rare).
        if (__any_sync(kFull, ready && ce < w + ROUND + 3)) {
            cp_async_wait<0>();
            __syncwarp();
            reverse_list(cur, n_cur);
            if (pending)
                ce = kSeg * fs;
            pending = false;
            n_prev = 0;
        } else {
            n_prev = n_cur;
        }
        cur ^= 1;
    }
};

// ------------------------------------------------------------------ split index --
//
// No payload is read here, so the words stay as they lie in memory (stream bit b = bit b%32 of word b/32):
// the terminator of a symbol is the lowest zero of the window, isolated with ~w & (w + 1); no bit reversal.

constexpr int kCpDense = 16;             // checkpoints at symbols 0, 4, .., 60 of a lane's own parse,
constexpr int kCpMax = kCpDense + 32;    // then at 64, 96, ..: boundary positions relative to the chunk start
__device__ __forceinline__ uint32_t cp_symbol(uint32_t i) { return i < kCpDense ? 4 * i : 64 + 32 * (i - kCpDense); }
__device__ __forceinline__ uint32_t cp_index(uint32_t j) { return j < 64 ? j >> 2 : kCpDense + ((j - 64) >> 5); }
__device__ __forceinline__ uint32_t cp_count(uint32_t n) { return n == 0 ? 0u : cp_index(n - 1) + 1; } // checkpoints among symbols 0..n-1

// Random access for the short walks (merge search, table look-up, the tail of a chunk, long symbols):
// RING consecutive words at a time, fetched on demand.  Every earlier copy of the lane must have landed.
template <int RING>
struct VsReader {
    VsRing<RING> rg;
    uint32_t base_w, end_w;
};
template <int RING>
__device__ __noinline__ uint32_t reader_next_boundary(VsReader<RING> *rd, uint32_t total_bits, uint32_t q, uint32_t kp1)
{
    while (q < total_bits) {
        const uint32_t w = q >> 5;
        if (w < rd->base_w || w + 1 >= rd->end_w) {
            const uint32_t fv0 = w >> 2;
            for (uint32_t i = 0; i < RING / 4; i++)
                rd->rg.issue(fv0 + i);
            cp_async_commit();
            cp_async_wait<0>();
            rd->base_w = 4 * fv0;
            rd->end_w = rd->base_w + RING;
        }
        const uint32_t win = __funnelshift_r(rd->rg.word(w), rd->rg.word(w + 1), q);
        const uint32_t c = bfind_u32(~win & (win + 1)); // trailing ones; 0xffffffff: 32 or more
        if (c < 32)
            return q + c + kp1;
        q += 32;
    }
    return total_bits + kp1; // ran off the end: the zero padding terminates the run
}

template <int LOG2S, int RING, int ROUND>
__global__ void __launch_bounds__(32 * kVsWarps) k_rice_split_index(RiceVsParams p)
{
    static_assert(ROUND % 4 == 0 && 64 % ROUND == 0, "geometry");
    constexpr int S = 1 << LOG2S;
    constexpr uint32_t kPart = kFrame >> LOG2S;
    extern __shared__ __align__(16) unsigned char split_smem[];
    const int lane = lane_id(), warp = warp_id();
    const uint32_t smem0 = (uint32_t)__cvta_generic_to_shared(split_smem);
    const uint32_t pad = (RING * 4 - (smem0 & (RING * 4 - 1))) & (RING * 4 - 1);
    uint16_t *cps = reinterpret_cast<uint16_t *>(split_smem + pad + kVsWarps * 32 * RING * 4) + (size_t)warp * kCpMax * 32;

    const uint32_t l = lane & (S - 1), gb = lane & ~(S - 1);
    const uint32_t st = ((blockIdx.x * kVsWarps + warp) * 32 + lane) >> LOG2S;
    const bool exists = st < p.n_sub;
    selab200_subframe_desc d;
    memset(&d, 0, sizeof d);
    if (exists)
        d = p.descs[st];
    // splittable: well-formed and every lane gets at least four words
    const bool ok = exists && rice_desc_ok(d, p.channels, p.n_words) && d.res_words >= 4u * S;
    const uintptr_t addr = reinterpret_cast<uintptr_t>(p.words + (ok ? d.res_offset : 0));
    const uint32_t skip = (uint32_t)(addr >> 2) & 3u;
    const uint32_t total = ok ? (uint32_t)d.res_words + skip : 0u; // words from the aligned base
    const uint32_t k = ok ? d.res_rice_param : 0u, kp1 = k + 1;

    using Stream = VsStream<RING, ROUND>;
    Stream s;
    s.rg.row = smem0 + pad + (uint32_t)(warp * 32 + lane) * (RING * 4);
    s.rg.rot = (16u * lane) & (RING * 4 - 1);
    s.rg.gvec = reinterpret_cast<const uint4 *>(addr & ~(uintptr_t)15);
    s.rg.total_bytes = (int)(total * 4);
    VsReader<RING> rd;
    rd.rg = s.rg;
    rd.base_w = rd.end_w = 0;

    // ---- phase 1: every lane parses the boundaries of its own chunk of bits ----
    const uint32_t total_bits = total * 32;
    const uint32_t cw = total >> LOG2S;                                // words per chunk (>= 4); the last lane takes the rest
    const uint32_t cstart = l == 0 ? skip * 32 : l * cw * 32;         // lane 0 starts at the stream's first bit: a true boundary
    const uint32_t cend = l == S - 1 ? total_bits : (l + 1) * cw * 32;
    bool fail = false;
    bool active = ok && cstart < cend;
    uint32_t j = 0; // symbols parsed by completed rounds (the same for every lane still active)
    if (active)
        s.prime(cstart);
    else
        s.pos = cstart;
    uint16_t *cpl = cps + lane;
    while (__ballot_sync(kFull, active)) {
        if (active) {
            if (j)
                s.boundary();
            const uint32_t pos_s = s.pos;
            const bool dense = j < 64;
            if (!dense && ((j - 64) & 31) == 0) {
                const uint32_t i = kCpDense + ((j - 64) >> 5), rel = pos_s - cstart;
                if (i < (uint32_t)kCpMax && rel < 0xffffu)
                    cpl[i * 32] = (uint16_t)rel;
                else
                    fail = true;
            }
            uint32_t mx = 0;
#pragma unroll
            for (int e = 0; e < ROUND; e++) {
                if (dense && (e & 3) == 0) { // uniform over the active lanes
                    const uint32_t rel = s.pos - cstart;
                    if (rel < 0xffffu)
                        cpl[((j + e) >> 2) * 32] = (uint16_t)rel;
                    else
                        fail = true;
                }
                const uint32_t win = __funnelshift_r(s.r0, s.r1, s.pos);
                const uint32_t ones = bfind_u32(~win & (win + 1)); // trailing ones (0xffffffff: the whole window)
                mx = max(mx, ones);
                const uint32_t pn = s.pos + ones + kp1;
                if ((s.pos ^ pn) >= 32u)
                    s.advance();
                s.pos = pn;
            }
            if (mx > 32u - kp1) {
                // a symbol longer than the window: redo the round with the on-demand reader, then restart the stream
                cp_async_wait<0>();
                rd.base_w = rd.end_w = 0;
                uint32_t q = pos_s;
                bool crossed = false;
#pragma unroll 1
                for (int e = 0; e < ROUND; e++) {
                    q = reader_next_boundary<RING>(&rd, total_bits, q, kp1);
                    crossed |= q >= cend;
                }
                if (crossed) {
                    s.prime(pos_s); // (the reader has overwritten the ring)
                    active = false;
                } else {
                    s.prime(q);
                    j += ROUND;
                }
            } else if (s.pos >= cend || j + ROUND >= (uint32_t)kFrame + 64) {
                s.pos = pos_s; // the chunk ends inside this round: the tail loop below finds where
                active = false;
            } else {
                j += ROUND;
            }
        }
    }
    // One boundary forward, keeping the streaming state valid (a top-up every ROUND symbols); a symbol longer
    // than the window goes through the on-demand reader and restarts the stream behind it.
    uint32_t since = 0;
    auto step = [&]() {
        const uint32_t win = __funnelshift_r(s.r0, s.r1, s.pos);
        const uint32_t ones = bfind_u32(~win & (win + 1));
        if (ones + kp1 > 32u) {
            cp_async_wait<0>();
            rd.base_w = rd.end_w = 0;
            const uint32_t q = reader_next_boundary<RING>(&rd, total_bits, s.pos, kp1);
            s.prime(q);
            since = 0;
        } else {
            const uint32_t pn = s.pos + ones + kp1;
            if ((s.pos ^ pn) >= 32u)
                s.advance();
            s.pos = pn;
            if (++since == ROUND) {
                s.boundary();
                since = 0;
            }
        }
    };
    // ---- the tail: the round in which the chunk ends, one symbol at a time, all lanes together ----
    uint32_t n = j, exitp = cstart;
    bool found = !(ok && cstart < cend);
    if (!found)
        s.load_window(); // back at the start of that round; the ring still holds it
    for (int e = 0; e <= ROUND && __ballot_sync(kFull, !found); e++) {
        if (!found) {
            if (s.pos >= cend) {
                found = true;
                exitp = s.pos;
            } else {
                if (n < 64 ? (n & 3) == 0 : ((n - 64) & 31) == 0) {
                    const uint32_t i = cp_index(n), rel = s.pos - cstart;
                    if (i < (uint32_t)kCpMax && rel < 0xffffu)
                        cpl[i * 32] = (uint16_t)rel;
                    else
                        fail = true;
                }
                step();
                n++;
            }
        }
    }
    if (!found) { // more symbols than a chunk may hold
        fail = true;
        exitp = s.pos;
    }
    const uint32_t ncp = cp_count(n);
    if (ncp > (uint32_t)kCpMax)
        fail = true;
    __syncwarp();

    // ---- phase 2: run on into the next lane's chunk until landing on one of its boundaries ----
    const uint32_t ncp_s = __shfl_down_sync(kFull, ncp, 1), n_s = __shfl_down_sync(kFull, n, 1);
    const uint32_t exit_s = __shfl_down_sync(kFull, exitp, 1), cstart_s = __shfl_down_sync(kFull, cstart, 1);
    uint32_t x = 0, m_next = 0; // overflow symbols of this lane; index (in the next lane's parse) of the merge boundary
    {
        bool done = !(ok && !fail && l < S - 1);
        uint32_t i = 0;
        const uint16_t *cn = cps + lane + 1;
        for (uint32_t guard = 0; __ballot_sync(kFull, !done); guard++) {
            if (!done) {
                const uint32_t rel = s.pos - cstart_s;
                if (rel >= 0xffffu || guard > 2048u) {
                    fail = true;
                    done = true;
                } else {
                    while (i < ncp_s && cn[i * 32] < rel)
                        i++;
                    if (i < ncp_s) {
                        if (cn[i * 32] == rel) {
                            m_next = cp_symbol(i);
                            done = true;
                        }
                    } else if (s.pos >= exit_s) { // behind the last checkpoint: only the next lane's exit is left to meet
                        if (s.pos == exit_s)
                            m_next = n_s;
                        else
                            fail = true;
                        done = true;
                    }
                    if (!done) {
                        step();
                        x++;
                    }
                }
            }
        }
    }
    // ---- phase 3: symbol index of every lane's first true boundary ----
    const uint32_t m_up = __shfl_up_sync(kFull, m_next, 1);
    const uint32_t m = l == 0 ? 0u : m_up; // this lane's parse is the true one from its symbol m on
    const uint32_t valid = n >= m ? n - m : 0u;
    if (n < m)
        fail = true;
    uint32_t incl = valid + x;
#pragma unroll
    for (int o = 1; o < S; o <<= 1) {
        const uint32_t t = __shfl_up_sync(kFull, incl, o, S);
        if ((int)l >= o)
            incl += t;
    }
    const uint32_t base = incl - (valid + x);
    const uint32_t fail_mask = __ballot_sync(kFull, fail || !ok);
    const bool group_bad = ((fail_mask >> gb) & ((S == 32) ? 0xffffffffu : ((1u << S) - 1u))) != 0;

    // ---- phase 4: lane l looks up where symbol l*2048/S begins ----
    const uint32_t target = l * kPart;
    uint32_t ls = 0;
#pragma unroll
    for (int ll = 1; ll < S; ll++) {
        const uint32_t b = __shfl_sync(kFull, base, gb + ll);
        if (b <= target)
            ls = ll;
    }
    const uint32_t b_s = __shfl_sync(kFull, base, gb + ls), valid_s = __shfl_sync(kFull, valid, gb + ls);
    const uint32_t m_s = __shfl_sync(kFull, m, gb + ls), exitp_s = __shfl_sync(kFull, exitp, gb + ls);
    const uint32_t cst_s = __shfl_sync(kFull, cstart, gb + ls), x_s = __shfl_sync(kFull, x, gb + ls);
    if (exists && l == 0)
        p.flags[st] = group_bad ? 1u : 0u;
    {
        const bool work = exists && l > 0 && !group_bad;
        const uint32_t rel = target - b_s;
        uint32_t q = 0, walk = 0;
        bool have = false;
        if (work) {
            if (rel < valid_s) {
                const uint32_t jj = m_s + rel, i = cp_index(jj);
                q = cst_s + cps[i * 32 + gb + ls];
                walk = jj - cp_symbol(i);
                have = true;
            } else {
                q = exitp_s;
                walk = rel - valid_s;
                have = walk < x_s; // else: a stream with too few symbols
            }
        }
        cp_async_wait<0>();
        if (have) {
            s.prime(q);
            since = 0;
        }
        for (uint32_t t = 0; __ballot_sync(kFull, have && t < walk); t++)
            if (have && t < walk)
                step();
        if (exists && l > 0)
            p.table[(size_t)st * (S - 1) + (l - 1)] = group_bad ? kNoSplit : have ? s.pos - skip * 32 : 0u; // 0: the decoder's end check fails
    }
}

template <int RING>
constexpr size_t split_smem_bytes()
{
    return RING * 4 + (size_t)kVsWarps * 32 * RING * 4 + (size_t)kVsWarps * kCpMax * 32 * 2;
}

// --------------------------------------------------------------- virtual streams --
//
// k_rice_decode_vc: one lane per virtual stream on the cooperative rings (VsCoopStream, 64 words per lane).
// Geometry (template parameters; the launch uses ROUND = 16, TILE = 32):
//   ROUND  symbols a lane decodes between two ring top-ups
//   TILE   symbols per lane staged in shared memory before they leave as 4*TILE-byte row segments

// General decode of `count` symbols from bit `pos`, ring words (reversed) only up to `ce` (exclusive).
// Out of line: runs for the rare round that holds a symbol longer than one 32-bit window.
// Returns false if it would need words the ring does not hold (the stream is then flagged).
template <int RING>
__device__ __noinline__ bool vs_slow_round(const VsRing<RING> rg, uint32_t ce, uint32_t *pos, uint32_t k, int32_t *dst, int count)
{
    uint32_t q = *pos;
    for (int e = 0; e < count; e++) {
        uint32_t ones = 0;
        while (true) {
            const uint32_t w = q >> 5;
            if (w + 2 > ce)
                return false;
            const uint32_t c = __clz(~__funnelshift_l(rg.word(w + 1), rg.word(w), q));
            ones += c;
            q += c;
            if (c < 32)
                break;
        }
        q += 1;
        const uint32_t w = q >> 5;
        if (w + 2 > ce)
            return false;
        const uint32_t win = __funnelshift_l(rg.word(w + 1), rg.word(w), q);
        const uint32_t pay = __funnelshift_rc(win, 0u, 32 - k);
        q += k;
        dst[e] = unzigzag((ones << k) | pay); // uint32 shift as in rice_decoder.cpp:37
    }
    if ((q >> 5) + 3 > ce)
        return false;
    *pos = q;
    return true;
}

template <int RING>
__device__ __noinline__ bool vc_slow_round(uint32_t row, uint32_t rot, uint32_t ce, uint32_t *pos, uint32_t k, int32_t *dst, int count)
{
    VsRing<RING> rg;
    rg.row = row;
    rg.rot = rot;
    rg.gvec = nullptr;
    rg.total_bytes = 0;
    return vs_slow_round<RING>(rg, ce, pos, k, dst, count);
}

template <int ROUND, int TILE>
__global__ void __launch_bounds__(32 * kVsWarps) k_rice_decode_vc(RiceVsParams p, int log2s)
{
    using Stream = VsCoopStream<ROUND>;
    constexpr int RING = Stream::kRing;
    static_assert(TILE % ROUND == 0 && TILE % 4 == 0 && ROUND % 4 == 0 && TILE <= 128, "tile geometry");
    constexpr int kTilePitch = TILE + 4;       // words: rows stay 16-byte aligned, banks rotate by 4 per row
    constexpr int kRowLanes = TILE / 4;        // lanes that move one row segment (16 bytes each)
    constexpr int kRowsPerIt = 32 / kRowLanes; // rows per store instruction
    extern __shared__ __align__(16) unsigned char vc_smem[];
    const int lane = lane_id(), warp = warp_id();
    const uint32_t smem0 = (uint32_t)__cvta_generic_to_shared(vc_smem);
    const uint32_t pad = (RING * 4 - (smem0 & (RING * 4 - 1))) & (RING * 4 - 1);
    int32_t *tile = reinterpret_cast<int32_t *>(vc_smem + pad + kVsWarps * 32 * RING * 4) + warp * 32 * kTilePitch;
    VsCoopMeta *meta = reinterpret_cast<VsCoopMeta *>(vc_smem + pad + kVsWarps * 32 * RING * 4 + kVsWarps * 32 * kTilePitch * 4) + warp;

    const uint32_t S = 1u << log2s, part = (uint32_t)kFrame >> log2s;
    const uint32_t v0 = (blockIdx.x * kVsWarps + warp) * 32;
    const uint32_t v = v0 + lane, st = v >> log2s, l = v & (S - 1);
    const bool exists = st < p.n_sub;
    selab200_subframe_desc d;
    memset(&d, 0, sizeof d);
    if (exists)
        d = p.descs[st];
    bool ok = exists && rice_desc_ok(d, p.channels, p.n_words);
    if (exists && !ok && l == 0)
        raise_status(p.status, SELAB200_ERR_BITSTREAM);
    const bool store_row = ok; // rows of flagged streams may hold garbage: the general kernel rewrites them
    uint32_t sb = 0, expect_end = kNoSplit;
    if (ok && S > 1) {
        const uint32_t *tb = p.table + (size_t)st * (S - 1);
        if (tb[0] == kNoSplit) {
            ok = false; // not split: the general kernel decodes it
        } else {
            if (l > 0)
                sb = tb[l - 1];
            if (l < S - 1)
                expect_end = tb[l];
        }
    }
    const uintptr_t addr = reinterpret_cast<uintptr_t>(p.words + (ok ? d.res_offset : 0));
    const uint32_t skip = (uint32_t)(addr >> 2) & 3u;
    const uint32_t total = ok && d.res_words ? (uint32_t)d.res_words + skip : 0u;
    Stream s;
    s.setup(vc_smem, smem0 + pad + (uint32_t)(warp * 32) * (RING * 4), meta, reinterpret_cast<const uint4 *>(addr & ~(uintptr_t)15), (int)(total * 4));
    const uint32_t k = ok ? d.res_rice_param : 0u, kp1 = k + 1, kk = 32 - k, kpow = 1u << k;
    const uint32_t row_mask = __ballot_sync(kFull, store_row);

    uint32_t p0 = sb + 32 * skip;
    if (p0 > total * 32 + 64)
        p0 = total * 32 + 64; // a nonsense table entry: parse zeros, fail the end check
    s.prime(p0, true);
    bool dead = false;

    int32_t *out_warp = p.out + (size_t)v0 * part;
    const uint32_t n_rounds = part / ROUND;
    const uint32_t c_pn = kp1 + 31;
#pragma unroll 1
    for (uint32_t r = 0; r < n_rounds; r++) {
        if (r)
            s.boundary(!dead);
        uint32_t pos_s = s.pos;
        int mn = 31; // lowest FLO result of the round; below k: a symbol longer than the window
        int32_t *trow = tile + lane * kTilePitch + (r % (TILE / ROUND)) * ROUND;
#pragma unroll
        for (int e4 = 0; e4 < ROUND; e4 += 4) {
            int32_t val[4];
#pragma unroll
            for (int e = 0; e < 4; e++) {
                const uint32_t win = __funnelshift_l(s.r1, s.r0, s.pos);
                const uint32_t f = bfind_u32(~win);           // 31 - ones; 0xffffffff: the window is all ones
                const uint32_t pn = fma_sub(s.pos + c_pn, f); // pos + ones + 1 + k (the adds run on the FMA pipe)
                mn = min(mn, (int)f);
                const uint32_t ones = fma_sub(31u, f);
                const uint32_t t = __funnelshift_lc(0u, win, fma_sub(32u, f));
                const uint32_t pay = __funnelshift_rc(t, 0u, kk);
                val[e] = unzigzag3(ones * kpow + pay);
                if ((s.pos ^ pn) >= 32u)
                    s.advance();
                s.pos = pn;
            }
            *reinterpret_cast<int4 *>(trow + e4) = make_int4(val[0], val[1], val[2], val[3]);
        }
        if (mn < (int)k && !dead) { // a symbol longer than the window: redo the round with the general parser
            if (vc_slow_round<RING>(s.row, s.rot, s.ce, &pos_s, k, trow, ROUND)) {
                s.pos = pos_s;
                s.load_window();
            } else {
                dead = true;
            }
        }
        if (dead)
            s.pos = pos_s; // parked: its ring is not topped up any more
        // ---- a full tile: TILE symbols per lane leave as row segments of 4*TILE bytes ----
        if (r % (TILE / ROUND) == TILE / ROUND - 1) {
            __syncwarp();
            int32_t *dst = out_warp + (size_t)(r / (TILE / ROUND)) * TILE + (lane % kRowLanes) * 4;
#pragma unroll
            for (int it = 0; it < 32 / kRowsPerIt; it++) {
                const int row = kRowsPerIt * it + lane / kRowLanes;
                if ((row_mask >> row) & 1u) {
                    const int4 q = *reinterpret_cast<const int4 *>(tile + row * kTilePitch + (lane % kRowLanes) * 4);
                    *reinterpret_cast<int4 *>(dst + (size_t)row * part) = q;
                }
            }
            __syncwarp();
        }
    }
    cp_async_wait<0>();
    if (exists && store_row) {
        bool bad = dead;
        if (ok) {
            if (expect_end != kNoSplit)
                bad |= s.pos - 32 * skip != expect_end;
            else
                bad |= s.pos > total * 32;
        }
        if (bad)
            p.flags[st] = 1u; // (several parts may say so: idempotent)
    }
}

template <int TILE>
constexpr size_t vc_smem_bytes()
{
    return 64 * 4 + (size_t)kVsWarps * 32 * 64 * 4 + (size_t)kVsWarps * 32 * (TILE + 4) * 4 + kVsWarps * sizeof(VsCoopMeta);
}

} // namespace selab200
