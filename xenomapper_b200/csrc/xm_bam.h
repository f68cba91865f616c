/*
 * xm_bam.h -- BAM input for the read-binning walk (BASELINE configs[4]).
 *
 * The reference pipes each BAM file through an external `samtools view`
 * (xm.py:48-64) and walks the SAM text it prints.  Here the BGZF blocks are
 * inflated on the host (zlib, one block per task over a pool of threads), the
 * host follows the block_size chain to find where each alignment record
 * starts, and the GPU turns the binary records into the SAM text lines
 * `samtools view` would print -- in device memory, where the walk's kernels
 * pick them up.  Three small kernels:
 *
 *   k_bam_len      one thread per record: length of its SAM line, validation
 *   k_bam_scan_blocks  exclusive scan of the lengths inside each CTA's 1024
 *                  records; the CTA totals are scanned on the host
 *   k_bam_render   one warp per record: QNAME, SEQ (4-bit codes) and QUAL
 *                  (+33) by all lanes, coalesced; the numeric fields, CIGAR
 *                  and the aux tags by lane 0
 *
 * Text rendering follows the SAM/BAM specification (sections 1.4, 4.2): the
 * aux integer types c C s S i I all print as `i`, B arrays as
 * `B:<type>,v,v...`, float aux values (`f`, `B:f`) with the C library's "%g"
 * (xm_fmtg.h reproduces it digit for digit for every 32-bit float).
 */
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>
#include <zlib.h>

#include "xm_fmtg.h"

#include <atomic>
#include <string>
#include <thread>
#include <vector>

namespace xm {

/* ---- host: BGZF + BAM structure ------------------------------------------- */
struct BgzfBlock {
    uint64_t in_off, out_off;
    uint32_t in_len, out_len, hdr_len;
};

inline uint32_t rd_u16(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }
inline uint32_t rd_u32(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }

/* the block table of a BGZF file; false on a malformed container */
inline bool bgzf_scan(const uint8_t *p, uint64_t n, std::vector<BgzfBlock> &blocks, uint64_t &total, std::string &err)
{
    uint64_t off = 0;
    total = 0;
    while (off < n) {
        if (n - off < 28 || p[off] != 31 || p[off + 1] != 139 || p[off + 2] != 8 || !(p[off + 3] & 4)) { err = "not a BGZF block at byte " + std::to_string(off); return false; }
        const uint32_t xlen = rd_u16(p + off + 10);
        if (12 + (uint64_t)xlen > n - off) { err = "truncated BGZF header"; return false; }
        uint32_t bsize = 0;
        for (uint32_t x = 0; x + 4 <= xlen;) {
            const uint8_t *sf = p + off + 12 + x;
            const uint32_t slen = rd_u16(sf + 2);
            if (sf[0] == 'B' && sf[1] == 'C' && slen == 2) bsize = rd_u16(sf + 4) + 1;
            x += 4 + slen;
        }
        if (!bsize || bsize > n - off || bsize < 12 + xlen + 8) { err = "bad BGZF block size at byte " + std::to_string(off); return false; }
        BgzfBlock b;
        b.in_off = off; b.in_len = bsize; b.hdr_len = 12 + xlen;
        b.out_len = rd_u32(p + off + bsize - 4);
        b.out_off = total;
        if (b.out_len > 65536) { err = "BGZF block inflates to more than 64 KiB"; return false; }
        total += b.out_len;
        blocks.push_back(b);
        off += bsize;
    }
    return true;
}

inline bool bgzf_inflate_block(const uint8_t *p, const BgzfBlock &b, uint8_t *dst)
{
    if (!b.out_len) return true;
    z_stream z;
    memset(&z, 0, sizeof z);
    if (inflateInit2(&z, -15) != Z_OK) return false;
    z.next_in = const_cast<Bytef *>(p + b.in_off + b.hdr_len);
    z.avail_in = b.in_len - b.hdr_len - 8;
    z.next_out = dst + b.out_off;
    z.avail_out = b.out_len;
    const int rc = inflate(&z, Z_FINISH);
    const bool ok = rc == Z_STREAM_END && z.avail_out == 0;
    inflateEnd(&z);
    if (!ok) return false;
    return (uint32_t)crc32(crc32(0L, Z_NULL, 0), dst + b.out_off, b.out_len) == rd_u32(p + b.in_off + b.in_len - 8);
}

/* inflate blocks [first, last) into dst (laid out by out_off) on `threads` host threads */
inline bool bgzf_inflate(const uint8_t *p, const std::vector<BgzfBlock> &blocks, size_t first, size_t last, uint8_t *dst, int threads, std::string &err)
{
    std::atomic<size_t> next(first);
    std::atomic<bool> bad(false);
    auto work = [&]() {
        for (;;) {
            const size_t k = next.fetch_add(1);
            if (k >= last || bad.load()) return;
            if (!bgzf_inflate_block(p, blocks[k], dst)) bad.store(true);
        }
    };
    const size_t nb = last - first;
    int nt = threads < 1 ? 1 : threads;
    if ((size_t)nt > nb) nt = (int)(nb ? nb : 1);
    std::vector<std::thread> pool;
    for (int t = 1; t < nt; ++t) pool.emplace_back(work);
    work();
    for (auto &t : pool) t.join();
    if (bad.load()) { err = "BGZF block does not inflate (corrupt data or CRC mismatch)"; return false; }
    return true;
}

struct BamIndex {
    std::string text;                   /* header text (l_text bytes, trailing NULs dropped) */
    std::vector<uint32_t> ref_off;      /* [n_ref + 1] into ref_names */
    std::string ref_names;
    uint64_t first_record = 0;          /* offset of the first record's block_size in the inflated stream */
    std::vector<uint64_t> rec;          /* offset of every record */
};

/* header fields and the record chain of an inflated BAM stream; header_only stops before the records */
inline bool bam_index(const uint8_t *d, uint64_t n, BamIndex &ix, bool header_only, std::string &err)
{
    if (n < 12 || memcmp(d, "BAM\1", 4) != 0) { err = "not a BAM file (bad magic)"; return false; }
    uint64_t o = 4;
    const uint32_t l_text = rd_u32(d + o); o += 4;
    if (o + l_text + 4 > n) { err = "truncated BAM header"; return false; }
    ix.text.assign((const char *)d + o, l_text);
    while (!ix.text.empty() && ix.text.back() == '\0') ix.text.pop_back();
    o += l_text;
    const uint32_t n_ref = rd_u32(d + o); o += 4;
    ix.ref_off.assign(1, 0);
    for (uint32_t r = 0; r < n_ref; ++r) {
        if (o + 4 > n) { err = "truncated BAM reference list"; return false; }
        const uint32_t l_name = rd_u32(d + o); o += 4;
        if (o + l_name + 4 > n || l_name == 0) { err = "truncated BAM reference list"; return false; }
        ix.ref_names.append((const char *)d + o, l_name - 1);
        ix.ref_off.push_back((uint32_t)ix.ref_names.size());
        o += l_name + 4;
    }
    ix.first_record = o;
    if (header_only) return true;
    ix.rec.reserve((size_t)((n - o) / 300 + 16));
    while (o < n) {
        if (o + 4 > n) { err = "truncated BAM record"; return false; }
        const uint32_t bs = rd_u32(d + o);
        if (bs < 32 || o + 4 + bs > n) { err = "truncated or corrupt BAM record at inflated byte " + std::to_string(o); return false; }
        ix.rec.push_back(o);
        o += 4 + (uint64_t)bs;
    }
    return true;
}

/* ---- device: record -> SAM text -------------------------------------------- */
struct BamDev {
    const uint8_t *data;          /* inflated stream */
    const uint64_t *rec;          /* [n] record offsets */
    uint64_t n;
    const uint32_t *ref_off;      /* [n_ref + 1] */
    const uint8_t *ref_names;
    uint32_t n_ref;
};
constexpr unsigned long long BAM_NO_ERROR = ~0ull;
enum { BAM_E_CORRUPT = 2 };

#if defined(__CUDACC__)
__device__ __forceinline__ uint32_t ld_u16(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }
__device__ __forceinline__ uint32_t ld_u32(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }

/* two sinks for the one renderer: a counter and a byte writer */
struct LenSink {
    uint32_t n = 0;
    __device__ void ch(uint8_t) { ++n; }
    __device__ void skip(uint32_t k) { n += k; }
    __device__ uint32_t pos() const { return n; }
};
struct BufSink {
    uint8_t *base, *p;
    __device__ void ch(uint8_t c) { *p++ = c; }
    __device__ void skip(uint32_t k) { p += k; }      /* bytes the other lanes write */
    __device__ uint32_t pos() const { return (uint32_t)(p - base); }
};

template <class S>
__device__ void put_uint(S &s, unsigned long long v)
{
    char tmp[20];
    int k = 0;
    do { tmp[k++] = (char)('0' + (int)(v % 10ull)); v /= 10ull; } while (v);
    while (k) s.ch((uint8_t)tmp[--k]);
}
template <class S>
__device__ void put_int(S &s, long long v)
{
    if (v < 0) { s.ch('-'); put_uint(s, (unsigned long long)(-v)); }
    else put_uint(s, (unsigned long long)v);
}
template <class S>
__device__ void put_ref(S &s, const BamDev &B, int32_t id)
{
    if (id < 0 || (uint32_t)id >= B.n_ref) { s.ch('*'); return; }
    for (uint32_t k = B.ref_off[id]; k < B.ref_off[id + 1]; ++k) s.ch(B.ref_names[k]);
}

/* a float aux value as samtools prints it: "%g" (xm_fmtg.h) */
template <class S>
__device__ void put_float(S &s, const uint8_t *p)
{
    const uint32_t bits = ld_u32(p);
    float f;
    memcpy(&f, &bits, 4);
    char tmp[16];
    const int n = fmt_g(f, tmp);
    for (int k = 0; k < n; ++k) s.ch((uint8_t)tmp[k]);
}

/* size in bytes of an integer aux value of type t (0: not an integer type) */
__device__ __forceinline__ int aux_size(uint8_t t)
{
    return (t == 'c' || t == 'C') ? 1 : (t == 's' || t == 'S') ? 2 : (t == 'i' || t == 'I') ? 4 : 0;
}
__device__ __forceinline__ long long aux_int(uint8_t t, const uint8_t *p)
{
    switch (t) {
    case 'c': return (int8_t)p[0];
    case 'C': return p[0];
    case 's': return (int16_t)ld_u16(p);
    case 'S': return ld_u16(p);
    case 'i': return (int32_t)ld_u32(p);
    default: return ld_u32(p);
    }
}

/*
 * The SAM line of the record at r (its block_size field), without the bulk
 * fields: QNAME, SEQ and QUAL are only measured (`skip`) so that the caller
 * can have all lanes write them.  Returns 0 or a BAM_E_* code; seq_at and
 * qual_at receive the offsets of SEQ and QUAL inside the line (QNAME opens it).
 */
template <class S>
__device__ int bam_line(S &s, const BamDev &B, const uint8_t *r, uint32_t &l_qname, uint32_t &l_seq_out, uint32_t &seq_at, uint32_t &qual_at, bool &qual_star)
{
    const uint32_t bs = ld_u32(r);
    const uint8_t *end = r + 4 + bs;
    const int32_t ref = (int32_t)ld_u32(r + 4), pos = (int32_t)ld_u32(r + 8);
    const uint32_t l_rn = r[12], mapq = r[13], n_cig = ld_u16(r + 16), flag = ld_u16(r + 18), l_seq = ld_u32(r + 20);
    const int32_t nref = (int32_t)ld_u32(r + 24), npos = (int32_t)ld_u32(r + 28), tlen = (int32_t)ld_u32(r + 32);
    const uint8_t *name = r + 36, *cig = name + l_rn, *seq = cig + 4ull * n_cig, *qual = seq + ((l_seq + 1) >> 1), *aux = qual + l_seq;
    if (aux > end || l_seq > (1u << 28)) return BAM_E_CORRUPT;
    /* QNAME: l_read_name counts the NUL */
    l_qname = l_rn > 1 ? l_rn - 1 : 0;
    if (l_qname) s.skip(l_qname); else s.ch('*');
    s.ch('\t'); put_uint(s, flag);
    s.ch('\t'); put_ref(s, B, ref);
    s.ch('\t'); put_int(s, (long long)pos + 1);
    s.ch('\t'); put_uint(s, mapq);
    s.ch('\t');
    if (!n_cig) s.ch('*');
    else
        for (uint32_t k = 0; k < n_cig; ++k) {
            const uint32_t v = ld_u32(cig + 4 * k);
            put_uint(s, v >> 4);
            const uint32_t op = v & 15u;
            s.ch(op < 9 ? (uint8_t)"MIDNSHP=X"[op] : (uint8_t)'?');
        }
    s.ch('\t');
    if (nref < 0) s.ch('*');
    else if (nref == ref) s.ch('=');
    else put_ref(s, B, nref);
    s.ch('\t'); put_int(s, (long long)npos + 1);
    s.ch('\t'); put_int(s, tlen);
    s.ch('\t');
    l_seq_out = l_seq;
    seq_at = s.pos(); qual_at = seq_at + l_seq + 1;
    qual_star = l_seq == 0 || qual[0] == 0xff;
    if (!l_seq) { s.ch('*'); s.ch('\t'); s.ch('*'); }
    else {
        s.skip(l_seq);
        s.ch('\t');
        if (qual_star) s.ch('*'); else s.skip(l_seq);
    }
    /* aux */
    const uint8_t *p = aux;
    while (p + 3 <= end) {
        const uint8_t t = p[2];
        s.ch('\t'); s.ch(p[0]); s.ch(p[1]); s.ch(':');
        p += 3;
        if (t == 'A') { if (p + 1 > end) return BAM_E_CORRUPT; s.ch('A'); s.ch(':'); s.ch(p[0]); p += 1; }
        else if (t == 'Z' || t == 'H') {
            s.ch(t); s.ch(':');
            while (p < end && *p) s.ch(*p++);
            if (p >= end) return BAM_E_CORRUPT;
            ++p;
        } else if (t == 'B') {
            if (p + 5 > end) return BAM_E_CORRUPT;
            const uint8_t st = p[0];
            const uint32_t cnt = ld_u32(p + 1);
            p += 5;
            s.ch('B'); s.ch(':'); s.ch(st);
            const int sz = st == 'f' ? 4 : aux_size(st);
            if (!sz || (unsigned long long)(end - p) < (unsigned long long)sz * cnt) return BAM_E_CORRUPT;
            if (st == 'f') for (uint32_t k = 0; k < cnt; ++k) { s.ch(','); put_float(s, p); p += 4; }
            else for (uint32_t k = 0; k < cnt; ++k) { s.ch(','); put_int(s, aux_int(st, p)); p += sz; }
        } else if (t == 'f') {
            if (p + 4 > end) return BAM_E_CORRUPT;
            s.ch('f'); s.ch(':'); put_float(s, p);
            p += 4;
        } else {
            const int sz = aux_size(t);
            if (!sz || p + sz > end) return BAM_E_CORRUPT;
            s.ch('i'); s.ch(':'); put_int(s, aux_int(t, p));
            p += sz;
        }
    }
    if (p != end) return BAM_E_CORRUPT;
    s.ch('\n');
    return 0;
}

__global__ void k_bam_len(const BamDev B, uint32_t *len, unsigned long long *err)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B.n) return;
    LenSink s;
    uint32_t a, b, c, d;
    bool q;
    const int e = bam_line(s, B, B.data + B.rec[i], a, b, c, d, q);
    if (e) atomicMin(err, (i << 8) | (unsigned long long)e);
    len[i] = e ? 0u : s.n;
}

/* exclusive scan of len[] inside each CTA's 1024 records; CTA totals to block_sum[] */
__global__ void k_bam_scan_blocks(const uint32_t *len, uint64_t n, uint32_t *local_off, unsigned long long *block_sum)
{
    __shared__ uint32_t wsum[32];
    const uint64_t i = (uint64_t)blockIdx.x * 1024 + threadIdx.x;
    const uint32_t v = i < n ? len[i] : 0u;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    if (warp == 0) {
        uint32_t t = wsum[lane], s2 = t;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, s2, o); if (lane >= o) s2 += y; }
        wsum[lane] = s2 - t;
        if (lane == 31) block_sum[blockIdx.x] = s2;
    }
    __syncthreads();
    if (i < n) local_off[i] = wsum[warp] + x - v;
}

/* one warp per record: records [i0, i0 + cnt) of B; local_off[] and block_base[] are indexed by record and by group of
 * 1024 records counted from i0's group (block_base[0] may be "negative": part of that group was rendered before) */
__global__ void k_bam_render(const BamDev B, uint64_t i0, uint64_t cnt, const uint32_t *local_off, const unsigned long long *block_base, uint8_t *out)
{
    const uint64_t w = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= cnt) return;
    const uint64_t i = i0 + w;
    const uint8_t *r = B.data + B.rec[i];
    uint8_t *dst = out + (block_base[(i >> 10) - (i0 >> 10)] + local_off[i]);
    /* lane 0 writes everything but the three bulk fields and tells the others where those go */
    uint32_t l_qname = 0, l_seq = 0, seq_at = 0, qual_at = 0;
    bool qstar = false;
    if (lane == 0) {
        BufSink s{dst, dst};
        bam_line(s, B, r, l_qname, l_seq, seq_at, qual_at, qstar);
    }
    l_qname = __shfl_sync(0xffffffffu, l_qname, 0);
    l_seq = __shfl_sync(0xffffffffu, l_seq, 0);
    seq_at = __shfl_sync(0xffffffffu, seq_at, 0);
    qual_at = __shfl_sync(0xffffffffu, qual_at, 0);
    qstar = __shfl_sync(0xffffffffu, (int)qstar, 0) != 0;
    const uint32_t l_rn = r[12], n_cig = ld_u16(r + 16);
    const uint8_t *name = r + 36, *seq = name + l_rn + 4ull * n_cig, *qual = seq + ((l_seq + 1) >> 1);
    for (uint32_t k = lane; k < l_qname; k += 32) dst[k] = name[k];
    if (l_seq) {
        uint8_t *ds = dst + seq_at, *dq = dst + qual_at;
        for (uint32_t k = lane; k < l_seq; k += 32) {
            const uint32_t b = seq[k >> 1];
            ds[k] = (uint8_t)"=ACMGRSVTWYHKDBN"[(k & 1) ? (b & 15u) : (b >> 4)];
        }
        if (!qstar) for (uint32_t k = lane; k < l_seq; k += 32) dq[k] = (uint8_t)(qual[k] + 33u);
    }
}
#endif  /* __CUDACC__ */

}  // namespace xm
