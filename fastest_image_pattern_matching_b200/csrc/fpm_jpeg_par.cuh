// fpm_jpeg_par.cuh -- Huffman decoding of a baseline JPEG scan ON THE DEVICE (the entropy-coded segment is the only H2D
// traffic of a JPEG ingest: 1.5 MB for the reference's 12 MP Src6.jpg instead of 24 MB of coefficients or 12 MB of pixels).
//
// A Huffman stream has no index, but it is self-synchronising: a decoder that starts at a wrong bit falls into step with
// the true symbol sequence after a few symbols.  The scan (0xFF00 stuffing and RST markers removed on the device by a
// stream compaction, jp_unstuff_*) is cut into sub-sequences of SUB bits, one thread each:
//   pass 0     every thread decodes its sub-sequence from its first bit as if a block started there and records its EXIT
//              state: the bit where its last symbol ended (inside the next sub-sequence), the block slot inside the MCU
//              and the coefficient index it was at, and how many blocks it completed;
//   pass 1..n  thread i restarts from the exit state of thread i-1 and decodes again; thread 0 is exact from the start, so
//              the exit states are a fixed point exactly when every thread started from the true state (induction over i).
//              Self-synchronisation makes that a handful of passes instead of one per sub-sequence; a thread whose entry
//              state did not change keeps its result;
//   then       an exclusive scan of the block counts gives every thread the index of its first block; a last pass decodes
//              once more and writes the coefficients of the luma blocks (DC as differences); a scan over the luma blocks in
//              scan order turns the DC differences into values.
// Every phase function is __host__ __device__: fpm_dbg_jpeg_luma_parallel(_batch) runs the same code thread by thread on the
// CPU and tests/test_ingest.py, tests/test_ingest_batch.py check it against the sequential decoder (fpm_jpeg.h) without a GPU.
// A batch of files is decoded by the same launches: every file has a descriptor (JpFile), a CTA finds its file by a binary
// search over the first-CTA prefix, and each file's sub-sequences / luma blocks start on a 4096 / JP_DC_TILE boundary of the
// shared state / DC arrays so that the tile scans run over the concatenation unchanged.
// Restart intervals are exact entry points: a decoder that reaches the (all-ones, < 8 bits) padding at the end of an interval,
// or runs over its end while it is out of step, restarts at the first bit of the next interval; the DC differences are then
// summed per interval.
#pragma once
#include "fpm_common.cuh"

#define JP_MAX_SLOTS 10            // blocks per MCU (JPEG limit)
#define JP_SUB_BITS 512            // sub-sequence length: a thread is a chain of dependent steps, so short sub-sequences (more
                                   // threads, a few more synchronisation passes) are faster: 83 us per pass at 1024 bits on a 1.5 MB scan
#define JP_SUB_WORDS (JP_SUB_BITS / 32)

struct JpTable {                   // one Huffman table: 9-bit direct lookup + canonical search for longer codes
    uint16_t fast[512];            // (length << 8) | symbol for codes of <= 9 bits, 0 otherwise
    uint32_t limit[18];            // limit[l]: first 16-bit window that is NOT a code of <= l bits (left-aligned), l = 1..16
    int32_t valoff[17];            // symbol index = valoff[l] + (window >> (16 - l))
    uint8_t sym[256];
};

struct JpScan {
    int nslots;                                // blocks per MCU
    int dc_tab[JP_MAX_SLOTS], ac_tab[JP_MAX_SLOTS];   // table index of each slot (into JpTable[8]: 0..3 DC, 4..7 AC)
    int luma_slots, luma_h, luma_v;            // the first luma_h * luma_v slots are luma blocks
    int mcux, mcuy, bw;                        // MCUs per row / column, luma blocks per row
    unsigned total_blocks;                     // blocks of the whole scan
    unsigned nbits;                            // length of the unstuffed scan in bits
    int nsub;                                  // sub-sequences
    // restart intervals (DRI): the RSTn markers are removed with the stuffing; rst[r] = first bit of interval r (byte aligned),
    // rst[nint] = nbits.  restart_blocks = blocks per interval (0: none, then rst is not read)
    unsigned restart_blocks;
    int nint;
    const unsigned* rst;
};

struct JpState {                   // where a decoder stands: next bit, slot in the MCU, next coefficient index; blocks completed
    unsigned p;
    unsigned slot_k;               // slot << 8 | k
    unsigned nblk;
    unsigned pad;
};

// where the bits come from: a plain byte array (host emulation, global memory) ...
struct JpBytes {
    const uint8_t* bits;
    FPM_HD unsigned peek32(unsigned p) const
    {
        const uint8_t* b = bits + (p >> 3);
        const unsigned hi = ((unsigned)b[0] << 24) | ((unsigned)b[1] << 16) | ((unsigned)b[2] << 8) | b[3];
        const unsigned lo = b[4];
        const unsigned s = p & 7;
        return s ? (hi << s) | (lo >> (8 - s)) : hi;
    }
};

// ... or the CTA's chunk in shared memory as big-endian 32-bit words, one pad word after the words of every sub-sequence:
// the 32 lanes of a warp sit at roughly the same offset of consecutive sub-sequences -- with a power-of-two distance the
// loads of a warp pile up on a few banks (1024-bit sub-sequences: ONE bank, 3x slower)
struct JpWords {
    const uint32_t* words;         // words[k + k / JP_SUB_WORDS] = big-endian word k of the CTA's chunk
    unsigned bit0;                 // absolute bit position of word 0
    FPM_HD unsigned peek32(unsigned p) const
    {
        const unsigned q = p - bit0, k = q >> 5, s = q & 31;
        const unsigned w0 = words[k + k / JP_SUB_WORDS], w1 = words[k + 1 + (k + 1) / JP_SUB_WORDS];
        return s ? (w0 << s) | (w1 >> (32 - s)) : w0;
    }
};

// one symbol of table t at window w (32 bits, left-aligned): code length and symbol; an invalid code (only met while a
// thread is still out of step) consumes one bit
FPM_HD void jp_symbol(const JpTable& t, unsigned w, int* len, int* sym)
{
    const unsigned f = t.fast[w >> 23];
    if (f) { *len = (int)(f >> 8); *sym = (int)(f & 255); return; }
    const unsigned w16 = w >> 16;
    for (int l = 10; l <= 16; l++)
        if (w16 < t.limit[l]) {
            const int idx = t.valoff[l] + (int)(w16 >> (16 - l));
            *len = l; *sym = t.sym[idx & 255];
            return;
        }
    *len = 1; *sym = 0;
}

__device__ __constant__ uint8_t jp_zigzag_dev[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                                     41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                                     30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
static const uint8_t jp_zigzag_host[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                           41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                           30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
FPM_HD int jp_zigzag(int k)
{
#ifdef __CUDA_ARCH__
    return jp_zigzag_dev[k];
#else
    return jp_zigzag_host[k];
#endif
}

// coefficient block of luma block number `slot` of MCU m
FPM_HD size_t jp_luma_block(const JpScan& sc, unsigned m, int slot)
{
    const unsigned my = m / sc.mcux, mx = m - my * sc.mcux;
    const int sy = slot / sc.luma_h, sx = slot - sy * sc.luma_h;
    return (size_t)(my * sc.luma_v + sy) * sc.bw + (mx * sc.luma_h + sx);
}

// Decode from state `in` up to bit p_end (symbols that START before p_end).  WRITE: blk0 = index of the block the run starts
// in; the AC coefficients of luma blocks go to coef, their DC DIFFERENCES to dcval[scan-order index of the luma block].
template <bool WRITE, class Src>
FPM_HD JpState jp_run(const Src& bits, const JpTable* __restrict__ tabs, const JpScan& sc, JpState in, unsigned p_end,
                      unsigned blk0, int16_t* __restrict__ coef, int* __restrict__ dcval)
{
    unsigned p = in.p, nblk = 0;
    int slot = (int)(in.slot_k >> 8), k = (int)(in.slot_k & 255);
    unsigned blk = blk0;
    // restart interval of p and where the next one starts
    int ri = 0;
    unsigned nxt = 0xffffffffu;
    if (sc.restart_blocks) {
        int lo = 0, hi = sc.nint;
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (sc.rst[mid] <= p) lo = mid; else hi = mid;
        }
        ri = lo;
        if (ri + 1 < sc.nint) nxt = sc.rst[ri + 1];
    }
    // where the current block's coefficients go (recomputed when a block ends, not per coefficient: the index arithmetic
    // divides)
    size_t cbase = 0, dcidx = 0;
    if (WRITE && slot < sc.luma_slots && blk < sc.total_blocks) {
        cbase = jp_luma_block(sc, blk / sc.nslots, slot) * 64;
        dcidx = (size_t)(blk / sc.nslots) * sc.luma_slots + slot;
    }
    while (p < p_end && (!WRITE || blk < sc.total_blocks)) {
        const unsigned w = bits.peek32(p);
        int len, sym;
        bool done = false;
        if (k == 0) {
            jp_symbol(tabs[sc.dc_tab[slot]], w, &len, &sym);
            const int s = sym & 15;
            if (WRITE && slot < sc.luma_slots) {
                int v = 0;
                if (s) {
                    v = (int)((w << len) >> (32 - s));
                    if (v < (1 << (s - 1))) v = v - (1 << s) + 1;
                }
                dcval[dcidx] = v;
            }
            p += len + s;
            k = 1;
        } else {
            jp_symbol(tabs[sc.ac_tab[slot]], w, &len, &sym);
            const int r = sym >> 4, s = sym & 15;
            p += len + s;
            if (s == 0) {
                if (r == 15) { k += 16; done = k >= 64; }
                else done = true;                                            // EOB
            } else {
                k += r;
                if (k < 64) {
                    if (WRITE && slot < sc.luma_slots) {
                        int v = (int)((w << len) >> (32 - s));
                        if (v < (1 << (s - 1))) v = v - (1 << s) + 1;
                        coef[cbase + jp_zigzag(k)] = (int16_t)v;
                    }
                    k++;
                }
                done = k >= 64;
            }
        }
        bool jump = false;
        if (nxt != 0xffffffffu) {
            if (p >= nxt) {
                jump = true;                                                 // over the end: only a thread out of step gets here
            } else if (done) {
                const unsigned rem = nxt - p;                                // the padding of an interval: < 8 bits, all ones
                jump = rem < 8 && (bits.peek32(p) >> (32 - rem)) == (1u << rem) - 1u;
            }
        }
        if (done) {
            k = 0;
            slot = slot + 1 == sc.nslots ? 0 : slot + 1;
            nblk++;
            blk++;
        }
        if (jump) {
            p = nxt; slot = 0; k = 0;
            ri++;
            nxt = ri + 1 < sc.nint ? sc.rst[ri + 1] : 0xffffffffu;
            if (WRITE) blk = (unsigned)ri * sc.restart_blocks;
        }
        if ((done || jump) && WRITE && slot < sc.luma_slots && blk < sc.total_blocks) {
            cbase = jp_luma_block(sc, blk / sc.nslots, slot) * 64;
            dcidx = (size_t)(blk / sc.nslots) * sc.luma_slots + slot;
        }
    }
    JpState out;
    out.p = p; out.slot_k = ((unsigned)slot << 8) | (unsigned)k; out.nblk = nblk; out.pad = 0;
    return out;
}

// ---- the passes, one call per thread ---------------------------------------------------------------------------------
// pass 0: cold start at the first bit of the sub-sequence
template <class Src>
FPM_HD void jp_pass_cold(int i, const Src& bits, const JpTable* tabs, const JpScan& sc, JpState* exit_state, JpState* entry_used)
{
    if (i >= sc.nsub) return;
    JpState in;
    in.p = (unsigned)i * JP_SUB_BITS; in.slot_k = 0; in.nblk = 0; in.pad = 0;
    const unsigned p_end = min((unsigned)(i + 1) * JP_SUB_BITS, sc.nbits);
    exit_state[i] = jp_run<false>(bits, tabs, sc, in, p_end, 0, nullptr, nullptr);
    entry_used[i] = in;
}

// synchronisation pass: start from the previous pass's exit state of the thread before; *changed is raised when an exit
// state moved.  prev and next are different arrays.
template <class Src>
FPM_HD void jp_pass_sync(int i, const Src& bits, const JpTable* tabs, const JpScan& sc, const JpState* prev, JpState* next,
                         JpState* entry_used, int* changed)
{
    if (i >= sc.nsub) return;
    if (i == 0) { next[0] = prev[0]; return; }
    const JpState in = prev[i - 1];
    const JpState used = entry_used[i];
    if (in.p == used.p && in.slot_k == used.slot_k) { next[i] = prev[i]; return; }      // same entry, same result
    const unsigned p_end = min((unsigned)(i + 1) * JP_SUB_BITS, sc.nbits);
    JpState out;
    if (in.p >= p_end) { out = in; out.nblk = 0; }                                        // nothing starts in this sub-sequence
    else out = jp_run<false>(bits, tabs, sc, in, p_end, 0, nullptr, nullptr);
    entry_used[i] = in;
    next[i] = out;
    const JpState old = prev[i];
    if (out.p != old.p || out.slot_k != old.slot_k || out.nblk != old.nblk) {
#ifdef __CUDA_ARCH__
        atomicOr(changed, 1);
#else
        *changed = 1;
#endif
    }
}

// final pass: blk_first[i] (+ blk_tile_off[i / 4096] when given) = blocks completed before sub-sequence i
template <class Src>
FPM_HD void jp_pass_write(int i, const Src& bits, const JpTable* tabs, const JpScan& sc, const JpState* state, const unsigned* blk_first,
                          const int* blk_tile_off, int16_t* coef, int* dcval)
{
    if (i >= sc.nsub) return;
    JpState in;
    if (i == 0) { in.p = 0; in.slot_k = 0; in.nblk = 0; in.pad = 0; }
    else in = state[i - 1];
    const unsigned p_end = min((unsigned)(i + 1) * JP_SUB_BITS, sc.nbits);
    if (in.p >= p_end) return;
    jp_run<true>(bits, tabs, sc, in, p_end, blk_first[i] + (blk_tile_off ? (unsigned)blk_tile_off[i / 4096] : 0u), coef, dcval);
}

// scan-order index (MCU order, slots inside the MCU) of the luma block at block row / column (row, col)
FPM_HD unsigned jp_luma_scan_index(const JpScan& sc, int row, int col)
{
    const int my = row / sc.luma_v, sy = row - my * sc.luma_v, mx = col / sc.luma_h, sx = col - mx * sc.luma_h;
    return (unsigned)(my * sc.mcux + mx) * sc.luma_slots + (unsigned)(sy * sc.luma_h + sx);
}

// ---- batches -----------------------------------------------------------------------------------------------------------
// last i in [0, n) with first[i] <= x (first non-decreasing, first[0] <= x): the file of a CTA or tile.  Files with no CTAs
// share their first[] value with the next file and are never picked.
FPM_HD int jp_file_of(const int* first, int n, int x)
{
    int lo = 0, hi = n;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (first[mid] <= x) lo = mid; else hi = mid;
    }
    return lo;
}

// Unstuffing as a stream compaction over the entropy-coded segments of all files.  Whether byte i is emitted depends on
// d[i-1], d[i], d[i+1] only (jp_unstuff_class); the output position of an emitted byte is an exclusive scan of the emit flags,
// the restart interval a RST marker opens a scan of the RST flags.  The scan ends at the first other marker (a min-reduction
// over the file) or at the position after the file's last byte; the thread that owns that position writes nbits / nint, the
// sentinel rst[nint] and the 16 zero bytes the decoder reads ahead.  The output equals the sequential jpeg_unstuff
// (fpm_host.cu) for every input, damaged and truncated files included.
#define JP_UNSTUFF_THREADS 256
#define JP_UNSTUFF_BYTES 16                                          // per thread
#define JP_UNSTUFF_TILE (JP_UNSTUFF_THREADS * JP_UNSTUFF_BYTES)      // per CTA; a tile never spans two files

struct JpUnstuff {                 // one file of a batch (offsets into the uploaded batch buffer / the output arrays)
    unsigned long long begin, end; // entropy-coded data: from the byte after SOS to the end of the file
    unsigned long long out;        // output slot, 4-aligned, align4(end - begin) + 16 bytes
    unsigned long long rst;        // first of the file's rst_cap entries of rst[]
    unsigned long long stop;       // in: end; out: the position where the scan ends
    int rst_cap;
    int restart;                   // DRI present: RSTn separates intervals; otherwise it ends the scan like any other marker
    unsigned nbits;                // out: unstuffed length in bits
    int nint;                      // out: restart intervals (RST markers before the stop + 1)
};
enum { JP_EMIT = 1, JP_RST = 2, JP_STOP = 4 };

FPM_HD int jp_unstuff_class(const uint8_t* d, const JpUnstuff& f, unsigned long long i)
{
    if (i >= f.end) return JP_STOP;                                      // the position after the last byte
    const unsigned b = d[i];
    if (b != 0xFF) return i > f.begin && d[i - 1] == 0xFF ? 0 : JP_EMIT; // an FF is never the second byte of a pair, so this
                                                                         // byte is the second byte of FF xx exactly when d[i-1] is FF
    if (i + 1 >= f.end) return 0;                                        // 0xFF as the last byte
    const unsigned c = d[i + 1];
    if (c == 0x00) return JP_EMIT;                                       // stuffed 0xFF
    if (c == 0xFF) return 0;                                             // fill byte
    if (f.restart && c >= 0xD0 && c <= 0xD7) return JP_RST;
    return JP_STOP;
}

// positions [a, b) of one thread's chunk: emitted bytes, RST markers, first stop (~0 if none)
FPM_HD void jp_unstuff_count(const uint8_t* d, const JpUnstuff& f, unsigned long long a, unsigned long long b, unsigned* emit,
                             unsigned* rst, unsigned long long* stop)
{
    unsigned e = 0, r = 0;
    unsigned long long s = ~0ull;
    for (unsigned long long i = a; i < b; i++) {
        const int c = jp_unstuff_class(d, f, i);
        e += c & JP_EMIT;
        r += (c >> 1) & 1;
        if ((c & JP_STOP) && s == ~0ull) s = i;
    }
    *emit = e; *rst = r; *stop = s;
}

// the same chunk again, f.stop final: o / r = bytes emitted / RST markers met before position a
FPM_HD void jp_unstuff_write(const uint8_t* d, JpUnstuff& f, unsigned long long a, unsigned long long b, unsigned o, unsigned r,
                             uint8_t* out, unsigned* rst)
{
    const unsigned long long stop = f.stop;
    uint8_t* dst = out + f.out;
    unsigned* rs = rst + f.rst;
    const unsigned cap = (unsigned)f.rst_cap;
    for (unsigned long long i = a; i < b && i <= stop; i++) {
        if (i == stop) {
            for (unsigned k = o; k < ((o + 3) & ~3u) + 16; k++) dst[k] = 0;
            if (cap > 0) rs[0] = 0;
            if (r + 1 < cap) rs[r + 1] = o * 8;                      // sentinel rst[nint] = nbits
            f.nbits = o * 8;
            f.nint = (int)r + 1;
            return;
        }
        const int c = jp_unstuff_class(d, f, i);
        if (c & JP_EMIT) dst[o++] = d[i];
        if (c & JP_RST) {
            r++;
            if (r < cap) rs[r] = o * 8;
        }
    }
}

// positions [a, b) of thread `t` of tile `tile` of the file (b <= end + 1: end itself is the position that may stop the scan)
FPM_HD void jp_unstuff_chunk(const JpUnstuff& f, int tile, int t, unsigned long long* a, unsigned long long* b)
{
    *a = f.begin + (unsigned long long)tile * JP_UNSTUFF_TILE + (unsigned long long)t * JP_UNSTUFF_BYTES;
    *b = *a + JP_UNSTUFF_BYTES < f.end + 1 ? *a + JP_UNSTUFF_BYTES : f.end + 1;
}

struct JpFile {                    // one file of a decode wave
    JpTable tabs[8];
    JpScan sc;                     // sc.rst points at the file's entries of the batch's rst array
    uint16_t quant[64];            // luma quantisation table, natural order
    unsigned long long bits;       // byte offset of the unstuffed scan (4-aligned)
    unsigned long long coef;       // first coefficient of luma block 0 in the wave's coefficient array
    unsigned long long frame;      // byte offset of the output frame
    int sub0;                      // first sub-sequence in the state arrays (a multiple of 4096)
    int luma0;                     // first luma block in the DC array (a multiple of JP_DC_TILE)
    int width, height;
    int device_huffman;            // 0: Huffman-decoded on the host, coef holds its coefficients with the DC values
    int pad;
};

#ifdef __CUDACC__
// A decoder thread is one long chain of dependent loads (window -> table -> next window): out of global memory that is
// ~1.4 us per symbol with one warp per SM sub-partition.  The CTA therefore stages its 128 sub-sequences (16 KB + the few
// bytes the last symbol may reach into the next one) and its file's eight tables (11 KB) in shared memory first.
#define JP_THREADS 128
#define JP_CHUNK_BYTES (JP_THREADS * JP_SUB_BITS / 8)

#define JP_CHUNK_WORDS (JP_CHUNK_BYTES / 4)
struct JpShared {
    JpTable tabs[8];
    JpScan sc;                                                  // indexed by the slot: not from the parameter bank
    uint32_t words[JP_CHUNK_WORDS + JP_CHUNK_WORDS / JP_SUB_WORDS + 8];
};

// chunk `cta` of the file's unstuffed scan
__device__ __forceinline__ JpWords jp_stage(JpShared& sh, const uint8_t* __restrict__ bits, const JpTable* __restrict__ tabs,
                                            const JpScan& sc, int cta)
{
    const size_t byte0 = (size_t)cta * JP_CHUNK_BYTES;
    const size_t total = (((size_t)sc.nbits + 7) / 8 + 16 + 3) & ~(size_t)3;     // data + the zero padding after it
    const uint32_t* gt = reinterpret_cast<const uint32_t*>(tabs);
    uint32_t* st = reinterpret_cast<uint32_t*>(sh.tabs);
    for (int i = threadIdx.x; i < (int)(sizeof(sh.tabs) / 4); i += JP_THREADS) st[i] = gt[i];
    if (threadIdx.x == 0) sh.sc = sc;
    const uint32_t* gb = reinterpret_cast<const uint32_t*>(bits + byte0);       // byte0 is a multiple of the chunk size
    for (int k = threadIdx.x; k < JP_CHUNK_WORDS + 4; k += JP_THREADS) {
        const uint32_t v = byte0 + 4 * (size_t)k + 4 <= total ? gb[k] : 0u;
        sh.words[k + k / JP_SUB_WORDS] = __byte_perm(v, 0, 0x0123);
    }
    __syncthreads();
    JpWords src;
    src.words = sh.words;
    src.bit0 = (unsigned)(byte0 * 8);
    return src;
}

// the decoder grids: cta_first[i] = first CTA of file i (n + 1 entries), blockIdx.x -> (file, CTA of the file)
__global__ void __launch_bounds__(JP_THREADS)
fpm_jpeg_cold_kernel(const JpFile* __restrict__ files, const int* __restrict__ cta_first, int n, const uint8_t* bits,
                     JpState* exit_state, JpState* entry_used)
{
    __shared__ JpShared sh;
    const int fi = jp_file_of(cta_first, n, blockIdx.x), cta = blockIdx.x - cta_first[fi];
    const JpFile& f = files[fi];
    const JpWords b = jp_stage(sh, bits + f.bits, f.tabs, f.sc, cta);
    jp_pass_cold(cta * JP_THREADS + threadIdx.x, b, sh.tabs, sh.sc, exit_state + f.sub0, entry_used + f.sub0);
}

// one changed-flag for the whole wave: the pass loop ends when no file moved
__global__ void __launch_bounds__(JP_THREADS)
fpm_jpeg_sync_kernel(const JpFile* __restrict__ files, const int* __restrict__ cta_first, int n, const uint8_t* bits,
                     const JpState* prev, JpState* next, JpState* entry_used, int* changed)
{
    __shared__ JpShared sh;
    const int fi = jp_file_of(cta_first, n, blockIdx.x), cta = blockIdx.x - cta_first[fi];
    const JpFile& f = files[fi];
    const int nsub = f.sc.nsub;
    prev += f.sub0; next += f.sub0; entry_used += f.sub0;
    // a CTA whose entry states did not move (its file has converged) has nothing to decode: skip the staging too
    const int i = cta * JP_THREADS + threadIdx.x;
    bool work = false;
    if (i > 0 && i < nsub) {
        const JpState in = prev[i - 1], used = entry_used[i];
        work = in.p != used.p || in.slot_k != used.slot_k;
    }
    if (!__syncthreads_or(work)) {
        if (i < nsub) next[i] = prev[i];
        return;
    }
    const JpWords b = jp_stage(sh, bits + f.bits, f.tabs, f.sc, cta);
    jp_pass_sync(i, b, sh.tabs, sh.sc, prev, next, entry_used, changed);
}

__global__ void __launch_bounds__(JP_THREADS)
fpm_jpeg_write_kernel(const JpFile* __restrict__ files, const int* __restrict__ cta_first, int n, const uint8_t* bits,
                      const JpState* state, const unsigned* blk_first, const int* blk_tile_off, int16_t* coef, int* dcval)
{
    __shared__ JpShared sh;
    const int fi = jp_file_of(cta_first, n, blockIdx.x), cta = blockIdx.x - cta_first[fi];
    const JpFile& f = files[fi];
    const JpWords b = jp_stage(sh, bits + f.bits, f.tabs, f.sc, cta);
    jp_pass_write(cta * JP_THREADS + threadIdx.x, b, sh.tabs, sh.sc, state + f.sub0, blk_first + f.sub0, blk_tile_off + f.sub0 / 4096,
                  coef + f.coef, dcval + f.luma0);
}

// Exclusive scan of the block counts: tiles of 4096 sub-sequences by one CTA each (blk_first[i] = blocks before i inside its
// tile, tile_sum = the tile's total), fpm_jpeg_offsets_kernel scans the totals of every file, the write pass adds its tile's
// offset.  A file's sub-sequences start on a tile boundary, so no tile mixes two files.
__global__ void __launch_bounds__(256)
fpm_jpeg_block_tile_kernel(const JpState* __restrict__ state, int n, unsigned* __restrict__ blk_first, int* __restrict__ tile_sum)
{
    __shared__ int s_warp[8];
    const int t = threadIdx.x, base = blockIdx.x * 4096 + t * 16;
    int v[16], sum = 0;
#pragma unroll
    for (int k = 0; k < 16; k++) { v[k] = sum; sum += base + k < n ? (int)state[base + k].nblk : 0; }     // exclusive inside the thread
    int inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, inc, o);
        if ((t & 31) >= o) inc += u;
    }
    if ((t & 31) == 31) s_warp[t >> 5] = inc;
    __syncthreads();
    int woff = 0;
    for (int w = 0; w < (t >> 5); w++) woff += s_warp[w];
    const int excl = woff + inc - sum;
#pragma unroll
    for (int k = 0; k < 16; k++)
        if (base + k < n) blk_first[base + k] = (unsigned)(v[k] + excl);
    if (t == 255) tile_sum[blockIdx.x] = woff + inc;
}

// DC differences -> DC values: an inclusive scan over the luma blocks in scan order.  Tiles of 4096 values are scanned in
// place by one CTA each (fpm_jpeg_dc_tile_kernel), the tile totals of every file by fpm_jpeg_offsets_kernel; the IDCT kernel
// adds the offset of a value's tile when it reads it.
#define JP_DC_TILE 4096
__global__ void __launch_bounds__(256)
fpm_jpeg_dc_tile_kernel(int n, int* __restrict__ dcval, int* __restrict__ tile_sum)
{
    __shared__ int s_warp[8];
    const int t = threadIdx.x, base = blockIdx.x * JP_DC_TILE + t * 16;
    int v[16], sum = 0;
#pragma unroll
    for (int k = 0; k < 16; k++) { v[k] = base + k < n ? dcval[base + k] : 0; sum += v[k]; v[k] = sum; }
    int inc = sum;                                                       // inclusive scan of the thread totals over the CTA
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, inc, o);
        if ((t & 31) >= o) inc += u;
    }
    if ((t & 31) == 31) s_warp[t >> 5] = inc;
    __syncthreads();
    int woff = 0;
    for (int w = 0; w < (t >> 5); w++) woff += s_warp[w];
    const int excl = woff + inc - sum;
#pragma unroll
    for (int k = 0; k < 16; k++)
        if (base + k < n) dcval[base + k] = v[k] + excl;
    if (t == 255) tile_sum[blockIdx.x] = woff + inc;
}

// exclusive scan in place of the tile totals v[seg[b] .. seg[b+1]) of file b, one CTA per file (a 12 MP image has 47 DC
// tiles, a 1.5 MB scan 370 unstuffing tiles)
template <class T>
__global__ void __launch_bounds__(1024)
fpm_jpeg_offsets_kernel(const int* __restrict__ seg, T* __restrict__ v)
{
    __shared__ T s_sum[1024];
    T* tile_sum = v + seg[blockIdx.x];
    const int ntiles = seg[blockIdx.x + 1] - seg[blockIdx.x];
    const int t = threadIdx.x, per = (ntiles + 1023) / 1024, a = min(ntiles, t * per), b = min(ntiles, a + per);
    T sum = 0;
    for (int i = a; i < b; i++) sum += tile_sum[i];
    s_sum[t] = sum;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        const T u = t >= o ? s_sum[t - o] : (T)0;
        __syncthreads();
        s_sum[t] += u;
        __syncthreads();
    }
    T run = s_sum[t] - sum;
    for (int i = a; i < b; i++) { const T u = tile_sum[i]; tile_sum[i] = run; run += u; }
}

// ---- unstuffing kernels: tile_first[i] = first tile of file i (n + 1 entries), a tile = JP_UNSTUFF_TILE positions ----------

// exclusive scan over the CTA of (emitted << 32 | rst), 256 threads
__device__ __forceinline__ unsigned long long jp_unstuff_block_scan(unsigned long long v, unsigned long long* total)
{
    __shared__ unsigned long long s_warp[JP_UNSTUFF_THREADS / 32];
    const int t = threadIdx.x;
    unsigned long long inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long u = __shfl_up_sync(0xffffffffu, inc, o);
        if ((t & 31) >= o) inc += u;
    }
    if ((t & 31) == 31) s_warp[t >> 5] = inc;
    __syncthreads();
    unsigned long long woff = 0, all = 0;
    for (int w = 0; w < JP_UNSTUFF_THREADS / 32; w++) {
        if (w < (t >> 5)) woff += s_warp[w];
        all += s_warp[w];
    }
    *total = all;
    return woff + inc - v;
}

__global__ void __launch_bounds__(JP_UNSTUFF_THREADS)
fpm_jpeg_unstuff_count_kernel(const uint8_t* __restrict__ d, JpUnstuff* files, const int* __restrict__ tile_first, int n,
                              unsigned long long* __restrict__ tile_sum)
{
    const int fi = jp_file_of(tile_first, n, blockIdx.x);
    JpUnstuff& f = files[fi];
    unsigned long long a, b, s = ~0ull;
    jp_unstuff_chunk(f, blockIdx.x - tile_first[fi], threadIdx.x, &a, &b);
    unsigned e = 0, r = 0;
    if (a < b) jp_unstuff_count(d, f, a, b, &e, &r, &s);
    if (s != ~0ull) atomicMin(&f.stop, s);
    unsigned long long total;
    jp_unstuff_block_scan(((unsigned long long)e << 32) | r, &total);
    if (threadIdx.x == 0) tile_sum[blockIdx.x] = total;
}

__global__ void __launch_bounds__(JP_UNSTUFF_THREADS)
fpm_jpeg_unstuff_write_kernel(const uint8_t* __restrict__ d, JpUnstuff* files, const int* __restrict__ tile_first, int n,
                              const unsigned long long* __restrict__ tile_off, uint8_t* __restrict__ out, unsigned* __restrict__ rst)
{
    const int fi = jp_file_of(tile_first, n, blockIdx.x);
    JpUnstuff& f = files[fi];
    unsigned long long a, b, s;
    jp_unstuff_chunk(f, blockIdx.x - tile_first[fi], threadIdx.x, &a, &b);
    unsigned e = 0, r = 0;
    if (a < b) jp_unstuff_count(d, f, a, b, &e, &r, &s);
    unsigned long long total;
    const unsigned long long x = jp_unstuff_block_scan(((unsigned long long)e << 32) | r, &total) + tile_off[blockIdx.x];
    if (a < b && a <= f.stop) jp_unstuff_write(d, f, a, b, (unsigned)(x >> 32), (unsigned)x, out, rst);
}
#endif
