/*
 * xm_tile.h -- what one CTA does with one tile of a SAM stream.
 *
 *   scan_tile      secondary stream: stage window, byte-class masks, line
 *                  index, per-line parse, record ranks by decoupled
 *                  look-back, compact per-record arrays (SCompact).
 *   classify_tile  primary stream: the same front end, then joins each record
 *                  with its secondary-stream entry by record index, decides
 *                  the category (single reads or adjacent-QNAME pairs),
 *                  histograms it, scans the six bins' byte counts (second
 *                  look-back chain) and copies the emitted lines to their
 *                  final place in the six outputs: clean primary lines that
 *                  are neighbours in the input and in a bin are merged into
 *                  runs and copied from the staged window 512 bytes per warp
 *                  step; everything else (secondary-stream lines, lines that
 *                  need re-tokenising, lines outside the window) goes through
 *                  a short list of single items.
 *
 * A line belongs to the tile that holds its first byte.  The window staged in
 * shared memory extends HALO bytes to both sides so that the last owned line
 * and the line before the first owned one are normally inside it.  Lines that
 * are not take the exact byte-wise path through global memory: the last owned
 * line when it ends past the window, and the halo line when it starts before
 * it -- its start is found by walking back from the window, it is parsed from
 * global memory, its QNAME is compared with the first owned line's through
 * global memory (prev_name_equal) and a pair unit that begins with it is copied
 * from there.  A tile that one line covers owns no line.
 *
 * Byte classes.  Two exact masks are built per tile: W (byte < 0x21 or
 * >= 0x80: every separator, control and non-ASCII byte) and T (tab).  Line
 * terminators are taken to be W & ~T.  That is exact for clean SAM; a tile in
 * which some W & ~T byte is not '\n' (spaces, CR, controls, non-ASCII) is
 * "dirty": its masks are rebuilt from an exact newline mask and every line of
 * it takes the exact byte-wise parser.
 *
 * The code is written as barrier-separated phases so that one source builds
 * both the CUDA kernels (each phase runs once per thread) and the CPU
 * emulation used by the tests (each phase loops over the emulated threads).
 */
#pragma once
#include "xm_parse.h"

#if !defined(__CUDACC__)
#include <string.h>
#endif

namespace xm {

/* ---- shared-memory layout --------------------------------------------- */
template <class C>
struct TileMem {
    uint8_t *win;            /* staged bytes (+48 slack) */
    uint32_t *tbm, *nlm;     /* NW words each: tabs, line-terminator candidates (W & ~T) */
    uint16_t *trk;           /* NW: tabs in the window before each mask word */
    uint16_t *lstart;        /* LCAP+2 window offsets of the owned lines; [nlines] = first line after the tile */
    uint16_t *lpre;          /* THREADS+1: owned line starts in the mask words before each thread's words */
    uint4 *qx;               /* LCAP+1 (qs, qlen, h1, h2) of each line for the run-head test while the masks are live; [0] is the halo line */
    /* these overlay the masks, which are dead once the lines are parsed */
    uint4 *shl;              /* LCAP+1 per-line records shared with the next line's owner; [0] is the halo line */
    uint32_t *p_dst, *p_src, *p_meta;   /* LCAP: the line's primary-stream copy item */
    uint32_t *s_dst, *s_src, *s_meta;   /* LCAP: its secondary-stream copy item */
    uint16_t *rare;          /* LCAP: lines that own an item the run copier does not handle */
    /* run table, overlays shl (dead once the items are built) */
    uint32_t *run_sb, *run_dst, *run_cb;   /* LCAP+1 each */
    uint32_t *scr;           /* 160 words of scratch for block collectives and the halo line */
    unsigned long long *scr64;   /* 24 */
    uint32_t *hist;          /* 36 */
};

/* scratch slots */
enum { SCR_WT0 = 0, SCR_WT1 = 32, SCR_BINS = 64 /* [16 warps][8] */, SCR_FAKE = 192, SCR_ADJ, SCR_NRARE, SCR_SPARE,
       SCR_HALO_QLEN, SCR_HALO_H1, SCR_HALO_H2, SCR_HALO_FLAGS, SCR_HALO_OUTLEN, SCR_HALO_AS, SCR_HALO_XS, SCR_HALO_VALID, SCR_WORDS = 208 };
enum { S64_TOT = 0 /* 0..7 */, S64_TSUM = 8 /* 8..15 */, S64_HALO_START = 16, S64_HALO_QS, S64_BASE, S64_PSTOP, S64_BLANK_OFF, S64_MBAR, S64_WORDS = 24 };

template <class C>
struct TileLayout {
    static constexpr size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }
    static constexpr size_t win_bytes = align16((size_t)C::WIN + 48);
    static constexpr size_t mw = align16((size_t)C::NW * 4), mt = align16((size_t)C::NW * 2);
    static constexpr size_t masks_bytes = 2 * mw + mt;
    static constexpr size_t shl_bytes = (size_t)(C::LCAP + 1) * 16, it = align16((size_t)C::LCAP * 4), rr = align16((size_t)C::LCAP * 2);
    static constexpr size_t post_bytes = shl_bytes + 6 * it + rr;
    static constexpr size_t union_bytes = masks_bytes > post_bytes ? masks_bytes : post_bytes;
    static constexpr size_t o_union = win_bytes;
    static constexpr size_t o_lstart = o_union + union_bytes;
    static constexpr size_t o_lpre = o_lstart + align16((size_t)(C::LCAP + 2) * 2);
    static constexpr size_t o_qx = o_lpre + align16((size_t)(C::THREADS + 1) * 2);
    static constexpr size_t o_scr = o_qx + (size_t)(C::LCAP + 1) * 16;
    static constexpr size_t o_scr64 = o_scr + SCR_WORDS * 4;
    static constexpr size_t o_hist = o_scr64 + S64_WORDS * 8;
    static constexpr size_t total = o_hist + align16(36 * 4);
};

template <class C>
XM_HD TileMem<C> carve(void *base)
{
    using Lo = TileLayout<C>;
    uint8_t *b = (uint8_t *)base;
    TileMem<C> m;
    m.win = b;
    uint8_t *u = b + Lo::o_union;
    m.tbm = (uint32_t *)u;
    m.nlm = (uint32_t *)(u + Lo::mw);
    m.trk = (uint16_t *)(u + 2 * Lo::mw);
    m.shl = (uint4 *)u;
    m.p_dst = (uint32_t *)(u + Lo::shl_bytes);
    m.p_src = (uint32_t *)(u + Lo::shl_bytes + Lo::it);
    m.p_meta = (uint32_t *)(u + Lo::shl_bytes + 2 * Lo::it);
    m.s_dst = (uint32_t *)(u + Lo::shl_bytes + 3 * Lo::it);
    m.s_src = (uint32_t *)(u + Lo::shl_bytes + 4 * Lo::it);
    m.s_meta = (uint32_t *)(u + Lo::shl_bytes + 5 * Lo::it);
    m.rare = (uint16_t *)(u + Lo::shl_bytes + 6 * Lo::it);
    m.run_sb = (uint32_t *)u;
    m.run_dst = m.run_sb + (C::LCAP + 1);
    m.run_cb = m.run_dst + (C::LCAP + 1);
    m.lstart = (uint16_t *)(b + Lo::o_lstart);
    m.lpre = (uint16_t *)(b + Lo::o_lpre);
    m.qx = (uint4 *)(b + Lo::o_qx);
    m.scr = (uint32_t *)(b + Lo::o_scr);
    m.scr64 = (unsigned long long *)(b + Lo::o_scr64);
    m.hist = (uint32_t *)(b + Lo::o_hist);
    return m;
}

/* ---- per-thread state that lives across phases -------------------------- */
template <class C>
struct ThreadState {
    LineRec L;
    uint32_t rank;       /* position among the records this tile yields; ~0u = not yielded */
    uint32_t ymeta;      /* bin (3 bits, NO_BIN = nothing emitted) | Y_* bits */
    uint32_t ybytes;     /* bytes the record (or pair unit) emits into its bin */
    uint32_t yoff;       /* where, relative to the tile's first byte in that bin */
    uint32_t sraw;       /* raw input bytes of the line if it was yielded */
    uint32_t sin, sout;  /* block-collective operand / result */
};
enum : uint32_t { Y_ASSERT = 0x100, Y_PREV_DIRTY = 0x200 };
constexpr uint32_t NOT_YIELDED = 0xffffffffu;
constexpr uint16_t LSTART_FAR = 0xffffu;

template <class C>
struct TileCtx {
    TileMem<C> m;
    ThreadState<C> *emu;     /* CPU emulation only: the THREADS thread states */
};

/* copy items: meta = len (24 bits) | bin << 24 | kind << 27 | two_lines << 29 */
enum { IT_NONE = 0, IT_P_COPY = 1, IT_P_NORM = 2, IT_P_FAR = 3, IT_S = 1 };
constexpr uint32_t IT_LEN_MASK = (1u << 24) - 1u;
XM_HD uint32_t it_pack(uint32_t len, uint32_t bin, uint32_t kind, bool two) { return (len & IT_LEN_MASK) | (bin << 24) | (kind << 27) | ((uint32_t)two << 29); }
XM_HD uint32_t it_kind(uint32_t m) { return (m >> 27) & 3u; }
XM_HD uint32_t it_bin(uint32_t m) { return (m >> 24) & 7u; }
constexpr uint32_t RUN_CB_BITS = 22;      /* a tile's run bytes: every window line at most twice, < 4 MiB */

/* word shared with the next line's owner: outlen (24) | state (3) << 24 | evalerr (3) << 27 | dirty << 30 | evalstream << 31 */
XM_HD uint32_t shl_pack(uint32_t outlen, int state, int evalerr, int evalstream, bool dirty)
{
    return (outlen & META_LEN_MASK) | ((uint32_t)state << 24) | ((uint32_t)evalerr << 27) | ((uint32_t)dirty << 30) | ((uint32_t)evalstream << 31);
}

/* ---- execution-model macros ---------------------------------------------- */
#if XM_DEVICE_PASS
#define XM_THREADS_BEGIN { const int tid = (int)threadIdx.x; ThreadState<C> &th = th_; (void)tid; (void)th;
#define XM_THREADS_END }
#define XM_BARRIER() __syncthreads()
/* one barrier each; consecutive collectives must alternate the scratch bank (0 / 1) */
#define XM_BLOCK_SCAN(bank, total) do { th_.sout = dev_block_scan(th_.sin, T.m.scr + ((bank) ? SCR_WT1 : SCR_WT0), total); } while (0)
#define XM_BLOCK_MIN(bank, result) do { result = dev_block_min(th_.sin, T.m.scr + ((bank) ? SCR_WT1 : SCR_WT0)); } while (0)
#define XM_SCAN_BINS() do { th_.yoff = dev_scan_bins(th_.ymeta & 7u, th_.ybytes, th_.sraw, T.m.scr + SCR_BINS); } while (0)
#define XM_HIST_ADD(key) dev_hist_add(T.m.hist, key)
#define XM_SMEM_INC(p, result) do { result = atomicAdd((p), 1u); } while (0)
#else
#define XM_THREADS_BEGIN for (int tid = 0; tid < C::THREADS; ++tid) { ThreadState<C> &th = T.emu[tid]; (void)th;
#define XM_THREADS_END }
#define XM_BARRIER() ((void)0)
#define XM_BLOCK_SCAN(bank, total) do { uint32_t run_ = 0; for (int t_ = 0; t_ < C::THREADS; ++t_) { T.emu[t_].sout = run_; run_ += T.emu[t_].sin; } total = run_; } while (0)
#define XM_BLOCK_MIN(bank, result) do { uint32_t m_ = 0xffffffffu; for (int t_ = 0; t_ < C::THREADS; ++t_) m_ = T.emu[t_].sin < m_ ? T.emu[t_].sin : m_; result = m_; } while (0)
#define XM_SCAN_BINS() do { for (int b_ = 0; b_ < C2_SLOTS; ++b_) tsum[b_] = 0; for (int t_ = 0; t_ < C::THREADS; ++t_) { const uint32_t b_ = T.emu[t_].ymeta & 7u; if (b_ != NO_BIN) { T.emu[t_].yoff = (uint32_t)tsum[b_]; tsum[b_] += T.emu[t_].ybytes; } tsum[6] += T.emu[t_].sraw; } } while (0)
#define XM_HIST_ADD(key) do { if ((key) < 36) T.m.hist[(key)]++; } while (0)
#define XM_SMEM_INC(p, result) do { result = (*(p))++; } while (0)
#endif

/* the warp that runs the serial look-back sections */
#define XM_LB_WARP(C) (threadIdx.x < 32)

/* phase timing (profiling builds only): thread 0 adds the cycles since the previous mark to Globals::phase[k] */
#if XM_DEVICE_PASS && defined(XM_PHASE_TIMING)
#define XM_MARK(fr, k) do { if (threadIdx.x == 0) { const long long t_ = clock64(); atomicAdd(&(fr).g->phase[(fr).pbase + (k)], (unsigned long long)(t_ - (fr).tmark)); (fr).tmark = t_; } } while (0)
#define XM_MARK_INIT(fr, gp, base) do { (fr).g = (gp); (fr).pbase = (base); (fr).tmark = clock64(); } while (0)
#else
#define XM_MARK(fr, k) ((void)0)
#define XM_MARK_INIT(fr, gp, base) ((void)0)
#endif

#if defined(__CUDACC__)
/* device collectives, window staging, look-back and the copy engines: xm_kernels.cu */
__device__ uint32_t dev_block_scan(uint32_t v, uint32_t *wt, uint32_t &total);
__device__ uint32_t dev_block_min(uint32_t v, uint32_t *wt);
__device__ uint32_t dev_scan_bins(uint32_t bin, uint32_t bytes, uint32_t raw, uint32_t *wt);
__device__ void dev_bin_totals(const uint32_t *wt, unsigned long long *tot /* smem [8] */);
__device__ void dev_hist_add(uint32_t *hist, uint32_t key);
__device__ void dev_stage_window(uint8_t *win, const uint8_t *src, uint32_t bytes, unsigned long long *mbar);
__device__ void dev_publish1(unsigned long long *desc, uint32_t tile, unsigned long long agg_count, bool agg_stop);
__device__ void dev_resolve1(unsigned long long *desc, uint32_t tile, unsigned long long agg_count, bool agg_stop,
                             unsigned long long *out /* [0] exclusive count, [1] exclusive stop */);
__device__ void dev_publish2(unsigned long long *chain, uint32_t tile, const unsigned long long *tot /* smem [C2_SLOTS] */);
__device__ void dev_resolve2(unsigned long long *chain, uint32_t tile, unsigned long long *tot_to_base /* in: totals; out: exclusive bases */,
                             unsigned long long *dbg /* profiling builds: two counters, else nullptr */);
__device__ void dev_warp_copy(uint8_t *dst, const uint8_t *src_smem, const uint8_t *src_glob, uint32_t len);
__device__ void dev_copy_piece(uint8_t *dst, const uint8_t *win, uint32_t src_off, uint32_t len);
#endif

XM_HD void atomic_add64(unsigned long long *p, unsigned long long v)
{
#if XM_DEVICE_PASS
    atomicAdd(p, v);
#else
    *p += v;
#endif
}

/* ---- window geometry of a tile ------------------------------------------- */
struct Geo {
    uint64_t tstart, g0;
    uint32_t hoff, wbytes, nbits;
    int virt;
    bool at_eof;
};
template <class C>
XM_HD Geo tile_geo(const StreamBuf &B, uint32_t tile)
{
    Geo g;
    g.tstart = (uint64_t)tile * C::TILE;
    g.g0 = g.tstart >= (uint64_t)C::HALO ? g.tstart - C::HALO : 0;
    g.hoff = (uint32_t)(g.tstart - g.g0);
    uint64_t wend = g.g0 + C::WIN;
    if (wend >= B.len) { wend = B.len; g.at_eof = true; } else g.at_eof = false;
    g.wbytes = (uint32_t)(wend - g.g0);
    /* an unterminated last line gets a virtual newline one past the data */
    g.virt = (g.at_eof && B.len > 0 && B.p[B.len - 1] != '\n') ? (int)g.wbytes : -1;
    g.nbits = g.wbytes + (g.virt >= 0 ? 1u : 0u);
    return g;
}

/* global offset where the line ending just before window position s0 starts */
XM_HD uint64_t prev_line_start(const uint32_t *nlm, const uint8_t *glob, uint64_t g0, int s0)
{
    const int q = s0 - 1;              /* the newline that ends the previous line; look for the one before it */
    if (q > 0) {
        int w = (q - 1) >> 5;
        uint32_t m = nlm[w] & (0xffffffffu >> (31 - ((q - 1) & 31)));
        for (;;) {
            if (m) return g0 + (uint64_t)((w << 5) + 32 - clz32(m));
            if (--w < 0) break;
            m = nlm[w];
        }
    }
    uint64_t p = g0;                   /* not inside the window: walk back through global memory */
    while (p > 0 && glob[p - 1] != '\n') --p;
    return p;
}

/* the primary QNAME [pq, pq + qlen) equals the first token of the secondary line that starts at sstart */
XM_HD bool qname_equals_secondary(const Reader &rd, uint64_t pq, uint32_t qlen, const StreamBuf &S, uint64_t sstart)
{
    uint64_t q = sstart;
    while (q < S.len && S.p[q] != '\n' && is_ascii_space(S.p[q])) ++q;
    if (q + qlen > S.len) return false;
    for (uint32_t k = 0; k < qlen; ++k)
        if (S.p[q + k] != rd.at(pq + k)) return false;
    return q + qlen == S.len || is_ascii_space(S.p[q + qlen]);
}

template <class C>
struct Front {
    Geo geo;
    uint32_t nlines;       /* owned lines considered (0 on overflow) */
    uint32_t n_eff;        /* owned lines before the first blank one */
    uint32_t count;        /* records the tile yields (valid when `ranked`) */
    bool stop;             /* a blank line ends the stream inside this tile */
    bool overflow;
    bool dirty;            /* the tile's terminator candidates are not all '\n': every line takes the exact parser */
    bool early;            /* the tile's record count was published on chain 1 before the parse finished */
    bool ranked;           /* th.rank is already set */
    Globals *g;            /* phase timing only */
    int pbase;
    long long tmark;
};

/* bits of mask word w that lie in the byte range this tile owns */
template <class C>
XM_HD uint32_t own_mask(const Geo &geo, int w)
{
    uint32_t hi = geo.hoff + (uint32_t)C::TILE;
    if (hi > geo.wbytes) hi = geo.wbytes;
    const uint32_t base = (uint32_t)w << 5;
    if (base < geo.hoff || base >= hi) return 0u;       /* hoff is a multiple of 32 */
    return hi - base < 32u ? (1u << (hi - base)) - 1u : 0xffffffffu;
}
/* line starts (bit p: a line starts at window position p) of mask word w that this tile owns */
template <class C>
XM_HD uint32_t line_starts(const TileMem<C> &m, const Geo &geo, int w)
{
    const uint32_t own = own_mask<C>(geo, w);
    if (!own) return 0u;
    return ((m.nlm[w] << 1) | (w ? m.nlm[w - 1] >> 31 : (geo.g0 == 0 ? 1u : 0u))) & own;   /* the stream's first byte starts a line */
}

/* ---- emulated look-back for the CPU build: tiles run in order ------------- */
#if !XM_DEVICE_PASS
inline void emu_lookback1(unsigned long long *desc, uint32_t tile, unsigned long long agg_count, bool agg_stop, unsigned long long *out)
{
    unsigned long long ec = 0;
    bool es = false;
    if (tile > 0) { ec = desc[tile - 1] & C1_COUNT; es = (desc[tile - 1] & C1_STOP) != 0; }
    out[0] = ec; out[1] = es;
    desc[tile] = C1_INC | ((es || agg_stop) ? C1_STOP : 0) | (es ? ec : ec + agg_count);
}
inline void emu_lookback2(unsigned long long *chain, uint32_t tile, unsigned long long *tot)
{
    for (int b = 0; b < 6; ++b) {
        const unsigned long long ex = tile ? chain[(size_t)(tile - 1) * C2_SLOTS + b] & C2_VAL : 0;
        chain[(size_t)tile * C2_SLOTS + b] = C2_INC | (ex + tot[b]);
        tot[b] = ex;
    }
}
#endif

/* names_equal for a previous QNAME that may start before the window (the halo line of a tile whose first owned line
 * is preceded by a line longer than the halo): names_equal's word-wise path takes both names to start inside it */
XM_HD bool prev_name_equal(const Reader &rd, uint64_t prev_qs, uint32_t prev_qlen, uint64_t qs, uint32_t qlen)
{
    if (prev_qs >= rd.g0) return names_equal(rd, prev_qs, prev_qlen, qs, qlen);
    const Reader rg{rd.win, rd.glob, 0, 0u, rd.len};      /* every byte from global memory */
    return names_equal(rg, prev_qs, prev_qlen, qs, qlen);
}

/* is line i (QNAME in th.L) the first of its run of equal QNAMEs?  prev = (qs, qlen, h1, h2) of the line before */
XM_HD bool run_head(const Reader &rd, const LineRec &L, const uint4 prev, uint64_t prev_qs_global)
{
    if (prev.y != L.qlen || prev.z != L.h1 || prev.w != L.h2) return true;
    return !prev_name_equal(rd, prev_qs_global, prev.y, rd.g0 + L.qs, L.qlen);
}

/* ---- front end shared by both kernels: stage, mask, index, parse --------- */
/*
 * skip: getReadPairs' skip_repeated_reads.  The tile's record count goes onto look-back chain 1 as soon as it
 * is known: straight after the line index when the tile has no blank lines (no two touching W bytes) and does
 * not skip, after the QNAME half of the parse when it skips, after the whole parse otherwise (fr.early false).
 */
template <class C>
XM_HD void front_end(TileCtx<C> &T, ThreadState<C> &th_, const StreamBuf &B, int score_src, uint32_t debug,
                     bool need_prev, unsigned long long *chain1, uint32_t tile, bool skip, Front<C> &fr)
{
    (void)th_;
    const Geo geo = fr.geo;
    XM_THREADS_BEGIN
        if (tid == 0) { T.m.scr[SCR_FAKE] = 0; T.m.scr[SCR_ADJ] = 0; T.m.scr[SCR_NRARE] = 0; }
    XM_THREADS_END
    /* stage the window: one bulk copy on the device */
#if XM_DEVICE_PASS
    dev_stage_window(T.m.win, B.p + geo.g0, (geo.wbytes + 15u) & ~15u, T.m.scr64 + S64_MBAR);
#else
    memcpy(T.m.win, B.p + geo.g0, (geo.wbytes + 15u) & ~15u);
#endif
    XM_MARK(fr, 0);
    bool exact = (debug & DBG_FORCE_GENERIC) != 0;      /* exact newline mask: the tile is dirty (or forced) */
    uint32_t tot = 0, total_lines = 0;
    bool adj = false;
    for (int attempt = 0;; ++attempt) {
        /* byte-class masks of each thread's WPT consecutive 32-byte words, with the counts the index needs */
        XM_THREADS_BEGIN
            uint32_t cnt = 0, tabs = 0, aj = 0, cW, cN;
            const int wb = tid * C::WPT;
            if (wb == 0) cW = cN = geo.g0 == 0 ? 1u : 0u;       /* the stream's start acts as a terminator */
            else if ((uint32_t)(32 * wb - 1) < geo.wbytes) {
                const uint32_t c = T.m.win[32 * wb - 1];
                cW = is_w_byte(c) ? 1u : 0u;
                cN = exact ? (c == '\n' ? 1u : 0u) : (cW && c != '\t' ? 1u : 0u);
            } else cW = cN = 0u;
#pragma unroll 1
            for (int j = 0; j < C::WPT; ++j) {
                const int w = wb + j;
                if (w >= C::NW) break;
                const uint32_t off = 32u * (uint32_t)w;
                uint32_t W = 0, Tm = 0, N = 0;
                if (off < geo.wbytes) {
                    const uint4 va = *(const uint4 *)(T.m.win + off), vb = *(const uint4 *)(T.m.win + off + 16u);
                    uint32_t Wa, Ta, Wb, Tb;
                    masks16(va, Wa, Ta);
                    masks16(vb, Wb, Tb);
                    W = Wa | (Wb << 16);
                    Tm = Ta | (Tb << 16);
                    if (exact) N = newlines16(va) | (newlines16(vb) << 16);
                    const uint32_t valid = geo.wbytes - off;
                    if (valid < 32u) { const uint32_t k = (1u << valid) - 1u; W &= k; Tm &= k; N &= k; }
                }
                if (geo.virt >= 0 && (uint32_t)w == (geo.wbytes >> 5)) { W |= 1u << (geo.wbytes & 31u); N |= 1u << (geo.wbytes & 31u); }
                if (exact) Tm = W & ~N;          /* every other W byte is filed under "tab": the line index stays exact */
                else N = W & ~Tm;
                aj |= W & ((W << 1) | cW);
                tabs += (uint32_t)popc32(Tm);
                cnt += (uint32_t)popc32(((N << 1) | cN) & own_mask<C>(geo, w));
                T.m.tbm[w] = Tm;
                T.m.nlm[w] = N;
                cW = W >> 31; cN = N >> 31;
            }
            th.sin = cnt | (tabs << 16);
            if (aj) T.m.scr[SCR_ADJ] = 1;
        XM_THREADS_END
        XM_BLOCK_SCAN(attempt & 1, tot);
        XM_MARK(fr, 1);
        total_lines = tot & 0xffffu;
        XM_THREADS_BEGIN
            T.m.lpre[tid] = (uint16_t)(th.sout & 0xffffu);
            if (tid == 0) T.m.lpre[C::THREADS] = (uint16_t)total_lines;
            uint32_t tabs = th.sout >> 16;
            for (int j = 0; j < C::WPT; ++j) {
                const int w = tid * C::WPT + j;
                if (w >= C::NW) break;
                T.m.trk[w] = (uint16_t)tabs;
                tabs += (uint32_t)popc32(T.m.tbm[w]);
            }
        XM_THREADS_END
        XM_BARRIER();
        XM_MARK(fr, 2);
        /* the start of owned line i, found through the per-thread counts; every terminator candidate that bounds
         * an owned line is checked to be a real '\n' on the way */
        XM_THREADS_BEGIN
            uint32_t fake = 0;
            for (uint32_t i = (uint32_t)tid; i < total_lines && i <= (uint32_t)C::LCAP; i += (uint32_t)C::LCAP) {
                int lo = 0, hi = C::THREADS - 1;            /* the thread whose words hold line i */
                while (hi > lo) {
                    const int mid = (lo + hi + 1) >> 1;
                    if ((uint32_t)T.m.lpre[mid] <= i) lo = mid; else hi = mid - 1;
                }
                uint32_t r = i - (uint32_t)T.m.lpre[lo];
                int w = lo * C::WPT;
                uint32_t sw = line_starts<C>(T.m, geo, w);
                for (;;) {
                    const uint32_t c = (uint32_t)popc32(sw);
                    if (r < c) break;
                    r -= c;
                    sw = line_starts<C>(T.m, geo, ++w);
                }
                for (; r; --r) sw &= sw - 1;
                const uint32_t p = ((uint32_t)w << 5) + (uint32_t)ffs32(sw) - 1u;
                T.m.lstart[i] = (uint16_t)p;
                if (p > 0 && T.m.win[p - 1] != '\n') fake = 1;
            }
            if (tid == C::THREADS - 1 && total_lines <= (uint32_t)C::LCAP) {
                /* the last owned line ends at the first terminator at or after the tile's last byte */
                const int nwords = (int)((geo.nbits + 31u) >> 5);
                uint32_t q = geo.hoff + (uint32_t)C::TILE - 1u;
                if (q > geo.nbits - 1u) q = geo.nbits - 1u;
                uint16_t sent = LSTART_FAR;
                for (int w = (int)(q >> 5); w < nwords; ++w) {
                    uint32_t m = T.m.nlm[w];
                    if (w == (int)(q >> 5)) m &= 0xffffffffu << (q & 31u);
                    if (m) { sent = (uint16_t)(((uint32_t)w << 5) + (uint32_t)ffs32(m)); break; }
                }
                T.m.lstart[total_lines] = sent;
                if (sent != LSTART_FAR && (uint32_t)sent - 1u < geo.wbytes && T.m.win[sent - 1] != '\n') fake = 1;
            }
            if (fake && !exact) T.m.scr[SCR_FAKE] = 1;
        XM_THREADS_END
        XM_BARRIER();
        adj = T.m.scr[SCR_ADJ] != 0;
        XM_MARK(fr, 3);
        if (exact || !T.m.scr[SCR_FAKE]) break;
        exact = true;
    }
    const bool dirty = exact;
    fr.dirty = dirty;
    fr.nlines = total_lines;
    fr.overflow = false;
    if (total_lines > (uint32_t)C::LCAP) {
        if (C::TILE / 2 <= C::LCAP) fr.nlines = (uint32_t)C::LCAP;   /* the stop is among the first TILE/2 lines */
        else { fr.overflow = true; fr.nlines = 0; }
    }
    fr.stop = false;
    fr.n_eff = fr.nlines;
    fr.ranked = false;
    fr.count = 0;
    /* a blank line needs two touching W bytes (or a separator opening the stream): without them the tile yields
     * all its owned lines (or, skipping, the run heads among them) and can say so before the parse is over */
    fr.early = !adj && !dirty;
    if (fr.early && !skip) {
        fr.count = fr.nlines;
#if XM_DEVICE_PASS
        if (threadIdx.x == 0) dev_publish1(chain1, tile, fr.nlines, false);
#else
        unsigned long long o_[2];
        emu_lookback1(chain1, tile, fr.nlines, false, o_);
        T.m.scr64[S64_BASE] = o_[0]; T.m.scr64[S64_PSTOP] = o_[1];
#endif
    }

    /* Parse the owned lines.  In a clean tile with fewer than THREADS/2 lines two threads share a line: thread i
     * does the checks and the QNAME (fast_head), thread THREADS/2+i the aux tokens (fast_tail) and leaves its
     * result in qx[THREADS/2+1+i] (so at most THREADS/2-1 lines).  The last thread owns no line: it parses the line before the first owned one
     * when the walk needs it. */
    constexpr int HALF = C::THREADS / 2;
    const bool pair = fr.early && fr.nlines < (uint32_t)HALF;     /* thread THREADS-1 serves the halo line, not line HALF-1's aux half */
    const bool split = pair && skip;
    if (skip && !split) fr.early = false;
    XM_THREADS_BEGIN
        const WinMasks M_{T.m.win, T.m.tbm, T.m.nlm, T.m.trk, geo.wbytes, adj};
        Reader rd_{T.m.win, B.p, geo.g0, geo.wbytes, B.len};
        th.rank = NOT_YIELDED;
        th.sraw = 0;
        th.yoff = 0;                    /* 1 = the aux half of the line is done by the partner thread */
        th.sin = 0xffffffffu;
        const bool mine = (uint32_t)tid < fr.nlines;
        bool halo = false, farline = false, clean = false, tjob = false, split_line = false;
        int s = 0, e = 0;
        uint64_t gs = 0;
        FastCtx fc;
        fc.r0 = 0; fc.ntab = 0;
        if (tid == C::THREADS - 1) {
            T.m.scr[SCR_HALO_VALID] = 0;
            if (need_prev && fr.nlines > 0 && geo.g0 + T.m.lstart[0] > 0) {
                halo = true;
                const int s0 = (int)T.m.lstart[0];
                gs = prev_line_start(T.m.nlm, B.p, geo.g0, s0);
                if (!dirty && gs > geo.g0 && T.m.win[gs - geo.g0 - 1] != '\n') {
                    /* the candidate before the halo line is not a newline: find its real start byte-wise.  The line
                     * holds that candidate (a space, a CR ...), so the mask-driven parse does not apply to it. */
                    --gs;
                    while (gs > 0 && rd_.at(gs - 1) != '\n') --gs;
                    split_line = true;
                }
                farline = gs < geo.g0;
                if (farline) { rd_.wbytes = 0; rd_.g0 = gs; }       /* read it all from global memory */
                s = (int)(gs - geo.g0);
                e = s0 - 1;
            }
        }
        if (mine) {
            s = (int)T.m.lstart[tid];
            const uint16_t nx = T.m.lstart[tid + 1];
            e = (int)nx - 1;
            farline = nx == LSTART_FAR;
            gs = geo.g0 + (uint64_t)s;
        }
        if (mine || halo) {
            if (!dirty && !farline && !split_line) clean = fast_head(M_, s, e, th.L, fc);
            if (!clean) {               /* out of line: keep its operands off this thread's registers' stack */
                const Reader rg_ = rd_;
                LineRec G;
                generic_parse(rg_, gs, score_src, G);
                th.L = G;
            }
            tjob = clean && !(pair && mine);
            if (clean && pair && mine) th.yoff = 1;
        } else if (pair && tid >= HALF && (uint32_t)(tid - HALF) < fr.nlines) {
            s = (int)T.m.lstart[tid - HALF];
            const uint16_t nx = T.m.lstart[tid - HALF + 1];
            e = (int)nx - 1;
            /* the conditions under which fast_head accepts the line in a tile without touching W bytes */
            if (nx != LSTART_FAR && (uint32_t)e < geo.wbytes && e > s && T.m.win[e] == '\n' && !(s == 0 && (M_.wsm(0) & 1u))) {
                fc.r0 = tabs_before(M_, s);
                fc.ntab = tabs_before(M_, e) - fc.r0;
                tjob = true;
            }
        }
        if (tjob) {
            LineRec X;
            X.flags = 0; X.as = SCORE_ABSENT; X.xs = SCORE_ABSENT;
            fast_tail(M_, s, e, score_src, fc, X);
            if (mine || halo) { th.L.flags = X.flags; th.L.as = X.as; th.L.xs = X.xs; }
            else T.m.qx[tid + 1] = make_uint4(X.flags, (uint32_t)X.as, (uint32_t)X.xs, 1u);
        }
        if (mine) {
            if (th.L.flags & F_BLANK) th.sin = (uint32_t)tid;
            if (split) T.m.qx[tid + 1] = make_uint4(th.L.qs, th.L.qlen, th.L.h1, th.L.h2);
        }
        if (halo) {
            const LineRec &H = th.L;
            T.m.scr64[S64_HALO_START] = gs;
            T.m.scr64[S64_HALO_QS] = rd_.g0 + H.qs;
            T.m.scr[SCR_HALO_QLEN] = H.qlen; T.m.scr[SCR_HALO_H1] = H.h1; T.m.scr[SCR_HALO_H2] = H.h2;
            T.m.scr[SCR_HALO_FLAGS] = H.flags; T.m.scr[SCR_HALO_OUTLEN] = H.outlen;
            T.m.scr[SCR_HALO_AS] = (uint32_t)H.as; T.m.scr[SCR_HALO_XS] = (uint32_t)H.xs;
            T.m.scr[SCR_HALO_VALID] = 1;
        }
    XM_THREADS_END
    if (split) {
        /* run heads (getReadPairs skip mode, xm.py:110-114) from the QNAMEs alone; then the rest of each line */
        XM_BARRIER();
        XM_MARK(fr, 4);
        XM_THREADS_BEGIN
            uint32_t head = 0;
            if ((uint32_t)tid < fr.nlines) {
                const Reader rd_{T.m.win, B.p, geo.g0, geo.wbytes, B.len};
                if (tid == 0) {
                    head = 1;
                    if (T.m.scr[SCR_HALO_VALID])
                        head = run_head(rd_, th.L, make_uint4(0, T.m.scr[SCR_HALO_QLEN], T.m.scr[SCR_HALO_H1], T.m.scr[SCR_HALO_H2]), T.m.scr64[S64_HALO_QS]);
                } else {
                    const uint4 pv = T.m.qx[tid];
                    head = run_head(rd_, th.L, pv, geo.g0 + pv.x);
                }
            }
            th.sin = head;
        XM_THREADS_END
        uint32_t cnt_;
        XM_BLOCK_SCAN(0, cnt_);
        XM_MARK(fr, 5);
        fr.count = cnt_;
        fr.ranked = true;
#if XM_DEVICE_PASS
        if (threadIdx.x == 0) dev_publish1(chain1, tile, cnt_, false);
#else
        {
            unsigned long long o_[2];
            emu_lookback1(chain1, tile, cnt_, false, o_);
            T.m.scr64[S64_BASE] = o_[0]; T.m.scr64[S64_PSTOP] = o_[1];
        }
#endif
        XM_THREADS_BEGIN
            if ((uint32_t)tid < fr.nlines) {
                if (th.sin) th.rank = th.sout;
            }
        XM_THREADS_END
    } else if (adj || dirty) {
        uint32_t fb_;
        XM_BLOCK_MIN(0, fb_);
        fr.stop = fb_ < fr.nlines;
        fr.n_eff = fr.stop ? fb_ : fr.nlines;
    }
    if (pair) {
        if (!split) XM_BARRIER();       /* (the split walk has passed a barrier since the aux halves were written) */
        XM_THREADS_BEGIN
            if ((uint32_t)tid < fr.nlines && th.yoff) {
                const uint4 r = T.m.qx[HALF + 1 + tid];
                th.L.flags = r.x; th.L.as = (int32_t)r.y; th.L.xs = (int32_t)r.z;
            }
        XM_THREADS_END
    }
    /* where the stream stops, if it does so here (needed after the masks are gone) */
    XM_THREADS_BEGIN
        if (tid == 0) T.m.scr64[S64_BLANK_OFF] = fr.stop ? geo.g0 + (uint64_t)T.m.lstart[fr.n_eff] : B.len;
    XM_THREADS_END
    XM_BARRIER();      /* every thread is done with the masks: the per-line arrays may overlay them now */
    XM_MARK(fr, 6);
}

/* Ranks among the records the tile yields: every line before the stop, or only
 * the first line of each run of equal QNAMEs (getReadPairs skip mode,
 * xm.py:110-114).  Expects shl[i+1] = (qs, qlen, h1, h2) of line i.  Returns the count. */
template <class C>
XM_HD uint32_t rank_lines(TileCtx<C> &T, ThreadState<C> &th_, const StreamBuf &B, const Front<C> &fr, bool skip)
{
    (void)th_;
    if (fr.ranked) return fr.count;
    if (!skip) {
        XM_THREADS_BEGIN
            if ((uint32_t)tid < fr.n_eff) th.rank = (uint32_t)tid;
        XM_THREADS_END
        return fr.n_eff;
    }
    XM_THREADS_BEGIN
        const uint32_t i = (uint32_t)tid;
        uint32_t head = 0;
        if (i < fr.n_eff) {
            const Reader rd_{T.m.win, B.p, fr.geo.g0, fr.geo.wbytes, B.len};
            if (i == 0) {
                head = 1;
                if (T.m.scr[SCR_HALO_VALID])
                    head = run_head(rd_, th.L, make_uint4(0, T.m.scr[SCR_HALO_QLEN], T.m.scr[SCR_HALO_H1], T.m.scr[SCR_HALO_H2]), T.m.scr64[S64_HALO_QS]);
            } else {
                const uint4 pv = T.m.shl[i];
                head = run_head(rd_, th.L, pv, fr.geo.g0 + pv.x);
            }
        }
        th.sin = head;
    XM_THREADS_END
    uint32_t tot;
    XM_BLOCK_SCAN(1, tot);
    XM_THREADS_BEGIN
        if ((uint32_t)tid < fr.n_eff && th.sin) th.rank = th.sout;
    XM_THREADS_END
    return tot;
}

/* record base of a tile through look-back chain 1 (count + stop flag); `early`: the count is already published */
#if XM_DEVICE_PASS
#define XM_LOOKBACK1(chain, tile, count, stop, early, base, pstop) do { \
        if (XM_LB_WARP(C)) { \
            if (!(early) && (threadIdx.x & 31) == 0) dev_publish1((chain), (tile), (count), (stop)); \
            dev_resolve1((chain), (tile), (count), (stop), T.m.scr64 + S64_BASE); \
        } \
        __syncthreads(); \
        base = T.m.scr64[S64_BASE]; pstop = T.m.scr64[S64_PSTOP]; } while (0)
#else
#define XM_LOOKBACK1(chain, tile, count, stop, early, base, pstop) do { \
        if (!(early)) { unsigned long long o_[2]; emu_lookback1((chain), (tile), (count), (stop), o_); T.m.scr64[S64_BASE] = o_[0]; T.m.scr64[S64_PSTOP] = o_[1]; } \
        base = T.m.scr64[S64_BASE]; pstop = T.m.scr64[S64_PSTOP]; } while (0)
#endif

/* =========================================================================
 * Secondary-stream scan.
 * ========================================================================= */
template <class C>
XM_HD void scan_tile(TileCtx<C> &T, const ScanArgs &a, uint32_t tile)
{
#if XM_DEVICE_PASS
    ThreadState<C> th_;
#else
    ThreadState<C> &th_ = T.emu[0];
#endif
    Front<C> fr;
    fr.geo = tile_geo<C>(a.S, tile);
    XM_MARK_INIT(fr, a.g, 0);
    front_end<C>(T, th_, a.S, a.score_src, a.debug, a.skip != 0, a.chain1, tile, a.skip != 0, fr);

    if (a.skip && !fr.ranked) {
        XM_THREADS_BEGIN
            if ((uint32_t)tid < fr.n_eff) T.m.shl[tid + 1] = make_uint4(th.L.qs, th.L.qlen, th.L.h1, th.L.h2);
        XM_THREADS_END
        XM_BARRIER();
    }
    const uint32_t count = rank_lines<C>(T, th_, a.S, fr, a.skip != 0);

    unsigned long long base, pstop;
    XM_LOOKBACK1(a.chain1, tile, count, fr.stop, fr.early, base, pstop);
    XM_MARK(fr, 7);

    XM_THREADS_BEGIN
        if (!pstop) {
            if (th.rank != NOT_YIELDED) {
                const unsigned long long gi = base + th.rank;
                if (gi < a.sc_cap) {
                    const LineRec &L = th.L;
                    a.sc.start[gi] = fr.geo.g0 + L.s;
                    a.sc.rec[gi] = make_uint4((uint32_t)L.as, (uint32_t)L.xs, L.h1, L.h2);
                    a.sc.meta[gi] = (L.outlen & META_LEN_MASK) | ((L.flags & 0x3fu) << META_LEN_BITS);
                }
            }
            if (tid == 0 && (fr.stop || tile + 1 == a.ntiles)) {
                const unsigned long long n = base + count;
                a.g->n_stream[a.stream_id] = n;
                a.g->end_off[a.stream_id] = T.m.scr64[S64_BLANK_OFF];
                if (a.sc.start && n <= a.sc_cap) a.sc.start[n] = T.m.scr64[S64_BLANK_OFF];
            }
        }
        if (tid == 0 && fr.overflow) a.g->overflow = 1;
    XM_THREADS_END
}

/* =========================================================================
 * Primary-stream classify + emit.
 * ========================================================================= */
XM_HD void report_error(Globals *g, unsigned long long rec, int code, int stream, int prev = 0)
{
    const unsigned long long w = (rec << 8) | ((unsigned long long)code << 2) | ((unsigned long long)prev << 1) | (unsigned long long)stream;
#if XM_DEVICE_PASS
    atomicMin(&g->err, w);
#else
    if (w < g->err) g->err = w;
#endif
}

/* first tag-evaluation failure of a record, in the reference's call order AS1, XS1, AS2, XS2 (xm.py:323-326) */
XM_HD void eval_error(uint32_t pflags, uint32_t sflags, int &code, int &stream)
{
    code = 0; stream = 0;
    if (pflags & F_AS_DUP) code = EC_DUP; else if (pflags & F_AS_NUM) code = EC_NUM_AS;
    else if (pflags & F_XS_DUP) code = EC_DUP; else if (pflags & F_XS_NUM) code = EC_NUM_XS;
    if (code) return;
    if (sflags & F_AS_DUP) code = EC_DUP; else if (sflags & F_AS_NUM) code = EC_NUM_AS;
    else if (sflags & F_XS_DUP) code = EC_DUP; else if (sflags & F_XS_NUM) code = EC_NUM_XS;
    if (code) stream = 1;
}

/* byte-wise writer for lines whose output differs from their raw bytes:
 * tokens joined by single tabs + '\n' (xm.py:334).  gs may point at the
 * line's first byte or its first token. */
XM_COLD void write_normalised(const Reader &rd, uint64_t gs, int nlines, uint8_t *dst)
{
    uint64_t p = gs;
    for (int l = 0; l < nlines; ++l) {
        bool in_tok = false, first = true;
        for (;; ++p) {
            bool end = p >= rd.len;
            const uint32_t c = end ? (uint32_t)'\n' : rd.at(p);
            if (c == '\n') end = true;
            const bool ws = end || c == '\r' || (c < 0x80 && is_ascii_space((uint8_t)c));
            if (ws) {
                in_tok = false;
                if (end) break;
            } else {
                if (!in_tok) { if (!first) *dst++ = '\t'; first = false; in_tok = true; }
                *dst++ = (uint8_t)c;
            }
        }
        *dst++ = '\n';
        ++p;
    }
}

template <class C>
XM_HD void classify_tile(TileCtx<C> &T, const ClassifyArgs &a, uint32_t tile)
{
#if XM_DEVICE_PASS
    ThreadState<C> th_;
#else
    ThreadState<C> &th_ = T.emu[0];
    unsigned long long tsum[C2_SLOTS];
#endif
    const bool paired = a.mode != MODE_SE;
    Front<C> fr;
    fr.geo = tile_geo<C>(a.P, tile);
    XM_MARK_INIT(fr, a.g, 12);
    front_end<C>(T, th_, a.P, a.score_src, a.debug, paired || a.skip, a.chain1, tile, a.skip != 0, fr);

    XM_THREADS_BEGIN
        if (tid < 36) T.m.hist[tid] = 0;
        if ((uint32_t)tid < fr.n_eff) T.m.shl[tid + 1] = make_uint4(th.L.qs, th.L.qlen, th.L.h1, th.L.h2);
    XM_THREADS_END
    XM_BARRIER();
    const uint32_t count = rank_lines<C>(T, th_, a.P, fr, a.skip != 0);

    unsigned long long base, pstop;
    XM_MARK(fr, 7);
    XM_LOOKBACK1(a.chain1, tile, count, fr.stop, fr.early, base, pstop);
    XM_MARK(fr, 8);
    /* records at or beyond ncap are not yielded: the other stream ended first, or an error re-run cut here */
    unsigned long long ncap = a.g->n_stream[1];
    if (a.limit < ncap) ncap = a.limit;
    if (a.sc_cap < ncap) ncap = a.sc_cap;      /* the secondary stream held more records than the compact arrays: nothing past them is read */
    if (pstop) ncap = 0;

    /* per-record decision.  Paired walks publish it for the next line's owner. */
    XM_THREADS_BEGIN
        th.ymeta = NO_BIN; th.ybytes = 0; th.yoff = 0;
        uint32_t key = 36;
        if (th.rank != NOT_YIELDED) {
            const unsigned long long gi = base + th.rank;
            const LineRec &L = th.L;
            if (gi == a.limit) a.g->limit_off = fr.geo.g0 + L.s;
            if (gi >= ncap) th.rank = NOT_YIELDED;
            else {
                if (a.p_start && gi < a.p_start_cap) a.p_start[gi] = fr.geo.g0 + L.s;
                const uint4 sr = a.sc.rec[gi];
                const uint32_t smeta = a.sc.meta[gi];
                const uint32_t sflags = smeta >> META_LEN_BITS;
                int ec = 0;
                /* text the device does not tokenise like the reference comes first: nothing derived from it can be trusted */
                if ((L.flags | sflags) & F_TEXT) ec = EC_TEXT;
                else if (sr.z != L.h1 || sr.w != L.h2) ec = EC_ASSERT;     /* xm.py:106 */
                else {
                    /* equal hashes are not yet equal names: the reference compares the strings */
                    const Reader rd_{T.m.win, a.P.p, fr.geo.g0, fr.geo.wbytes, a.P.len};
                    if (!qname_equals_secondary(rd_, fr.geo.g0 + L.qs, L.qlen, a.S, a.sc.start[gi])) ec = EC_ASSERT;
                }
                if (ec) report_error(a.g, gi, ec, (ec == EC_TEXT && !(L.flags & F_TEXT)) ? 1 : 0);
                int ev, evs;
                eval_error(L.flags, sflags, ev, evs);
                const int st = mapping_state(L.as, L.xs, (int32_t)sr.x, (int32_t)sr.y, a.thr);
                th.sraw = L.rawbytes;
                if (!paired) {
                    if (!ec && !(a.halo && gi == 0)) {
                        if (ev) report_error(a.g, gi, ev, evs);
                        else {
                            key = (uint32_t)st;
                            const uint32_t slen = smeta & META_LEN_MASK;
                            uint32_t bytes = (st == PS || st == PM || st == UA) ? L.outlen : (st == UR ? L.outlen + slen : slen);
                            if (!((a.enabled >> st) & 1u)) bytes = 0;
                            th.ymeta = (uint32_t)st;
                            th.ybytes = bytes;
                        }
                    }
                } else {
                    th.yoff = shl_pack(L.outlen, st, ev, evs, (L.flags & F_DIRTY) != 0);   /* parked until published */
                    if (ec) th.ymeta |= Y_ASSERT;
                }
            }
        }
        if (!paired) XM_HIST_ADD(key);
    XM_THREADS_END

    if (paired) {
        XM_THREADS_BEGIN
            if ((uint32_t)tid < fr.n_eff) {
                const bool y = th.rank != NOT_YIELDED;
                T.m.shl[tid + 1] = make_uint4(th.L.qs, y ? th.L.qlen : 0xffffffffu, th.L.h1, y ? th.yoff : 0u);
            }
            if (tid == 0) {
                /* the line before the first owned one is record base-1 */
                uint4 h = make_uint4(0, 0xffffffffu, 0, 0);
                if (!a.skip && T.m.scr[SCR_HALO_VALID] && base > 0 && base - 1 < ncap) {
                    const unsigned long long gi = base - 1;
                    const uint4 sr = a.sc.rec[gi];
                    int ev, evs;
                    eval_error(T.m.scr[SCR_HALO_FLAGS], a.sc.meta[gi] >> META_LEN_BITS, ev, evs);
                    const int st = mapping_state((int32_t)T.m.scr[SCR_HALO_AS], (int32_t)T.m.scr[SCR_HALO_XS], (int32_t)sr.x, (int32_t)sr.y, a.thr);
                    h = make_uint4(0, T.m.scr[SCR_HALO_QLEN], T.m.scr[SCR_HALO_H1],
                                   shl_pack(T.m.scr[SCR_HALO_OUTLEN], st, ev, evs, (T.m.scr[SCR_HALO_FLAGS] & F_DIRTY) != 0));
                }
                T.m.shl[0] = h;
            }
        XM_THREADS_END
        XM_BARRIER();
        XM_THREADS_BEGIN
            const uint32_t i = (uint32_t)tid;
            const bool own_ec = (th.ymeta & Y_ASSERT) != 0;
            th.yoff = 0;
            th.ymeta = NO_BIN;
            uint32_t key = 36;
            /* with skip_repeated the yielded records are run heads: adjacent ones never share a QNAME */
            if (!a.skip && th.rank != NOT_YIELDED && base + th.rank > 0) {
                const unsigned long long gi = base + th.rank;
                const LineRec &L = th.L;
                const uint4 pv = T.m.shl[i];
                /* a unit fires when the previous yielded primary QNAME equals this one (xm.py:402) */
                bool fire = pv.y == L.qlen && pv.z == L.h1;
                if (fire) {
                    const Reader rd_{T.m.win, a.P.p, fr.geo.g0, fr.geo.wbytes, a.P.len};
                    const uint64_t pq = (i == 0) ? T.m.scr64[S64_HALO_QS] : fr.geo.g0 + pv.x;
                    fire = prev_name_equal(rd_, pq, pv.y, fr.geo.g0 + L.qs, L.qlen);
                }
                if (fire && !own_ec) {                      /* the assert fires before the unit is looked at */
                    const int pst = (int)((pv.w >> 24) & 7u), pev = (int)((pv.w >> 27) & 7u), pevs = (int)(pv.w >> 31);
                    const uint32_t smeta = a.sc.meta[gi], pmeta = a.sc.meta[gi - 1];
                    const uint4 sr = a.sc.rec[gi];
                    int ev, evs;
                    eval_error(L.flags, smeta >> META_LEN_BITS, ev, evs);
                    if (pev) report_error(a.g, gi, pev, pevs, 1);       /* xm.py:408-411 come first */
                    else if (ev) report_error(a.g, gi, ev, evs);
                    else {
                        const int st = mapping_state(L.as, L.xs, (int32_t)sr.x, (int32_t)sr.y, a.thr);
                        key = (uint32_t)(pst * 6 + st);
                        const int bin = a.mode == MODE_PE_CONSERVATIVE ? pair_bin_conservative(pst, st) : pair_bin_liberal(pst, st);
                        const uint32_t plen = (pv.w & META_LEN_MASK) + L.outlen;
                        const uint32_t slen = (pmeta & META_LEN_MASK) + (smeta & META_LEN_MASK);
                        uint32_t bytes = (bin == PS || bin == PM || bin == UA) ? plen : (bin == UR ? plen + slen : slen);
                        if (!((a.enabled >> bin) & 1u)) bytes = 0;
                        th.ymeta = (uint32_t)bin | (((pv.w >> 30) & 1u) ? Y_PREV_DIRTY : 0u);
                        th.ybytes = bytes;
                    }
                }
            }
            XM_HIST_ADD(key);
        XM_THREADS_END
    }

    XM_MARK(fr, 9);
    /* byte offsets inside each bin: warp scans over the six bins, then the second look-back chain */
    XM_SCAN_BINS();
    /* publish the tile's bytes per bin now; the bases are looked up once everything that can do without them is done */
#if XM_DEVICE_PASS
    __syncthreads();
    if (XM_LB_WARP(C)) {
        dev_bin_totals(T.m.scr + SCR_BINS, T.m.scr64 + S64_TSUM);
        dev_publish2(a.chain2, tile, T.m.scr64 + S64_TSUM);
    }
#else
    for (int b = 0; b < C2_SLOTS; ++b) T.m.scr64[S64_TSUM + b] = tsum[b];
#endif

    XM_MARK(fr, 10);
    /* copy items: at most two per owning line (its primary-stream part, its secondary-stream part) */
    const uint32_t nown = fr.n_eff;
    XM_THREADS_BEGIN
        const uint32_t i = (uint32_t)tid;
        if (i < nown) {
            uint32_t pm = 0, pd = 0, ps = 0, sm = 0, sd = 0, ss = 0;
            const uint32_t bin = th.ymeta & 7u;
            if (th.rank != NOT_YIELDED && bin != NO_BIN && th.ybytes) {
                const LineRec &L = th.L;
                const bool pside = bin == PS || bin == PM || bin == UA || bin == UR;
                const bool sside = bin == SS || bin == SM || bin == UR;
                uint32_t plen = 0;
                bool rare = sside;
                if (pside) {
                    uint32_t prevlen = 0;
                    bool dirty = (L.flags & F_DIRTY) != 0;
                    if (paired) { prevlen = T.m.shl[i].w & META_LEN_MASK; dirty = dirty || (th.ymeta & Y_PREV_DIRTY); }
                    plen = prevlen + L.outlen;
                    pd = th.yoff;
                    if (!dirty) {
                        ps = L.s - prevlen;                 /* clean neighbours are contiguous in the input */
                        const long long so = (long long)(int32_t)ps;
                        const bool inwin = so >= 0 && (unsigned long long)so + plen <= fr.geo.wbytes;
                        pm = it_pack(plen, bin, inwin ? IT_P_COPY : IT_P_FAR, false);
                        rare = rare || !inwin;
                    } else {
                        if (!paired) ps = L.qs;
                        else ps = (i == 0) ? (uint32_t)(T.m.scr64[S64_HALO_QS] - fr.geo.g0) : T.m.shl[i].x;
                        pm = it_pack(plen, bin, IT_P_NORM, paired);
                        rare = true;
                    }
                }
                if (sside) {
                    sd = th.yoff + plen;
                    ss = th.rank;
                    sm = it_pack(th.ybytes - plen, bin, IT_S, paired);
                }
                if (rare) {
                    uint32_t k;
                    XM_SMEM_INC(&T.m.scr[SCR_NRARE], k);
                    T.m.rare[k] = (uint16_t)i;
                }
            }
            T.m.p_dst[i] = pd; T.m.p_src[i] = ps; T.m.p_meta[i] = pm;
            T.m.s_dst[i] = sd; T.m.s_src[i] = ss; T.m.s_meta[i] = sm;
        }
    XM_THREADS_END
    XM_BARRIER();

    /* runs: an in-window copy item joins its predecessor's run when both sit in the same bin and follow each
     * other directly in the input and in the output.  The predecessor is the previous line, or the one before
     * it when the previous line emits no primary-stream bytes (first mates in a paired walk). */
    XM_THREADS_BEGIN
        const uint32_t i = (uint32_t)tid;
        uint32_t v = 0;
        if (i < nown) {
            const uint32_t pm = T.m.p_meta[i];
            if (it_kind(pm) == IT_P_COPY) {
                bool merge = false;
                int j = (int)i - 1;
                if (j >= 0 && it_kind(T.m.p_meta[j]) == IT_NONE) --j;
                if (j >= 0) {
                    const uint32_t qm = T.m.p_meta[j];
                    const uint32_t ql = qm & IT_LEN_MASK;
                    merge = it_kind(qm) == IT_P_COPY && it_bin(qm) == it_bin(pm) && T.m.p_src[j] + ql == T.m.p_src[i] && T.m.p_dst[j] + ql == T.m.p_dst[i];
                }
                v = (pm & IT_LEN_MASK) | (merge ? 0u : 1u << RUN_CB_BITS);
            }
        }
        th.sin = v;
    XM_THREADS_END
    XM_MARK(fr, 11);
    uint32_t rtot;
    XM_BLOCK_SCAN(0, rtot);
    const uint32_t nruns = rtot >> RUN_CB_BITS;
    XM_THREADS_BEGIN
        if (th.sin >> RUN_CB_BITS) {
            const uint32_t r = th.sout >> RUN_CB_BITS;
            T.m.run_sb[r] = T.m.p_src[tid] | (it_bin(T.m.p_meta[tid]) << 16);
            T.m.run_dst[r] = T.m.p_dst[tid];
            T.m.run_cb[r] = th.sout & ((1u << RUN_CB_BITS) - 1u);
        }
        if (tid == 0) T.m.run_cb[nruns] = rtot & ((1u << RUN_CB_BITS) - 1u);
    XM_THREADS_END
    XM_BARRIER();
    XM_MARK(fr, 12);
    /* exclusive byte bases of the tile in the six bins: second look-back chain */
    unsigned long long tot[C2_SLOTS];
#if XM_DEVICE_PASS
    if (XM_LB_WARP(C)) {
        if ((threadIdx.x & 31) < C2_SLOTS) T.m.scr64[S64_TOT + (threadIdx.x & 31)] = T.m.scr64[S64_TSUM + (threadIdx.x & 31)];
        __syncwarp();
#if defined(XM_PHASE_TIMING)
        dev_resolve2(a.chain2, tile, T.m.scr64 + S64_TOT, a.g->phase + 30);
#else
        dev_resolve2(a.chain2, tile, T.m.scr64 + S64_TOT, nullptr);
#endif
    }
    __syncthreads();
    for (int b = 0; b < C2_SLOTS; ++b) tot[b] = T.m.scr64[S64_TOT + b];
#else
    for (int b = 0; b < C2_SLOTS; ++b) tot[b] = T.m.scr64[S64_TSUM + b];
    emu_lookback2(a.chain2, tile, tot);
#endif
    XM_MARK(fr, 13);
    /* copy the runs: each warp takes an equal share of the tile's run bytes, cutting runs where its share ends.
     * Runs that do not fit their output are dropped (the host rejects the call). */
    {
        const uint32_t rbytes = rtot & ((1u << RUN_CB_BITS) - 1u);
#if XM_DEVICE_PASS
        const uint32_t nwarps = (uint32_t)(C::THREADS / 32), warp = threadIdx.x >> 5;
        const uint32_t per = ((rbytes + nwarps - 1) / nwarps + 15u) & ~15u;
        uint32_t lo = warp * per;
        const uint32_t hi = lo + per < rbytes ? lo + per : rbytes;
        if (lo < hi) {
            uint32_t r = 0, rh = nruns - 1;                 /* the run that holds byte lo */
            while (rh > r) {
                const uint32_t mid = (r + rh + 1) >> 1;
                if (T.m.run_cb[mid] <= lo) r = mid; else rh = mid - 1;
            }
            while (lo < hi) {
                const uint32_t rb = T.m.run_cb[r], re = T.m.run_cb[r + 1];
                const uint32_t pe = re < hi ? re : hi;
                const uint32_t sb = T.m.run_sb[r];
                const unsigned long long doff = tot[sb >> 16] + T.m.run_dst[r];
                if (doff + (re - rb) <= a.out_cap[sb >> 16])
                    dev_copy_piece(a.out[sb >> 16] + doff + (lo - rb), T.m.win, (sb & 0xffffu) + (lo - rb), pe - lo);
                lo = pe;
                ++r;
            }
        }
#else
        (void)rbytes;
        for (uint32_t r = 0; r < nruns; ++r) {
            const uint32_t sb = T.m.run_sb[r], len = T.m.run_cb[r + 1] - T.m.run_cb[r];
            const unsigned long long doff = tot[sb >> 16] + T.m.run_dst[r];
            if (doff + len <= a.out_cap[sb >> 16]) memcpy(a.out[sb >> 16] + doff, T.m.win + (sb & 0xffffu), len);
        }
#endif
    }
    XM_MARK(fr, 14);
    /* and the single items: one warp each */
    {
        const uint32_t nrare = T.m.scr[SCR_NRARE];
#if XM_DEVICE_PASS
        const int lane = (int)(threadIdx.x & 31);
        for (uint32_t k = threadIdx.x >> 5; k < nrare; k += (uint32_t)(C::THREADS / 32)) {
#else
        const int lane = 0;
        for (uint32_t k = 0; k < nrare; ++k) {
#endif
            const uint32_t i = T.m.rare[k];
            const uint32_t pm = T.m.p_meta[i], sm = T.m.s_meta[i];
            if (it_kind(pm) == IT_P_NORM || it_kind(pm) == IT_P_FAR) {
                const uint32_t len = pm & IT_LEN_MASK;
                const int bin = (int)it_bin(pm);
                const unsigned long long doff = tot[bin] + T.m.p_dst[i];
                if (doff + len <= a.out_cap[bin]) {
                    uint8_t *dst = a.out[bin] + doff;
                    const long long so = (long long)(int32_t)T.m.p_src[i];
                    if (it_kind(pm) == IT_P_FAR) {
#if XM_DEVICE_PASS
                        dev_warp_copy(dst, nullptr, a.P.p + fr.geo.g0 + so, len);
#else
                        memcpy(dst, a.P.p + fr.geo.g0 + so, len);
#endif
                    } else if (lane == 0) {
                        const Reader rd_{T.m.win, a.P.p, fr.geo.g0, fr.geo.wbytes, a.P.len};
                        write_normalised(rd_, fr.geo.g0 + so, ((pm >> 29) & 1u) ? 2 : 1, dst);
                    }
                }
            }
            if (it_kind(sm) == IT_S) {
                const uint32_t len = sm & IT_LEN_MASK;
                const int bin = (int)it_bin(sm);
                const int nl = ((sm >> 29) & 1u) ? 2 : 1;
                const unsigned long long doff = tot[bin] + T.m.s_dst[i];
                if (doff + len <= a.out_cap[bin]) {
                    uint8_t *dst = a.out[bin] + doff;
                    const unsigned long long gi = base + T.m.s_src[i];
                    const unsigned long long g_first = nl == 2 ? gi - 1 : gi;
                    const uint32_t fl = (a.sc.meta[gi] | a.sc.meta[g_first]) >> META_LEN_BITS;
                    const uint64_t ss = a.sc.start[g_first];
                    if (!(fl & F_DIRTY)) {
#if XM_DEVICE_PASS
                        dev_warp_copy(dst, nullptr, a.S.p + ss, len);
#else
                        memcpy(dst, a.S.p + ss, len);
#endif
                    } else if (lane == 0) {
                        const Reader rs_{nullptr, a.S.p, 0, 0, a.S.len};
                        write_normalised(rs_, ss, nl, dst);
                    }
                }
            }
        }
    }

    /* category histogram and stream totals */
    XM_BARRIER();
    XM_MARK(fr, 15);
    XM_THREADS_BEGIN
        if (tid < 36 && T.m.hist[tid]) atomic_add64(&a.g->counts[tid], (unsigned long long)T.m.hist[tid]);
        if (tid == 0) {
            const unsigned long long *ts = T.m.scr64 + S64_TSUM;
            if (ts[6]) atomic_add64(&a.g->bytes_in[0], ts[6]);
            for (int b = 0; b < 6; ++b)
                if (ts[b] >> 32) report_error(a.g, base, EC_TEXT, 1);   /* a tile's offsets inside a bin are 32-bit */
            const bool last = tile + 1 == a.ntiles;
            if (!pstop && (fr.stop || last)) {
                a.g->n_stream[0] = base + count;
                a.g->end_off[0] = T.m.scr64[S64_BLANK_OFF];
            }
            if (last) for (int b = 0; b < 6; ++b) a.g->out_len[b] = tot[b] + ts[b];
            if (fr.overflow) a.g->overflow = 1;
        }
    XM_THREADS_END
}

}  // namespace xm
