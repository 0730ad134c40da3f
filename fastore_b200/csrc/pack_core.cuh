// pack_core.cuh -- per-thread bit packing of one stored mate (and of a title / meta fields).
//
// Replaces IFastqPacker::StoreNextRecord / StoreDna / StoreQuality / StoreHeader and the
// BitMemoryWriter they append to (FastqPacker.cpp:113-287; BitMemory.h:216-433).  The reference
// pushes symbol after symbol into a sequential MSB-first bit writer.  Here the bit offset of every
// record in every stream is known beforehand (layout.cuh), so one thread packs one stored mate
// independently: K1 turns four quality symbols at a time into 4 / 12 / 24 output bits with word-wide
// arithmetic and derives the DNA stream from the bit planes of the signature search, streaming
// 32-bit words into the record's slot; K4 shifts whole segments to the record's bit phase.  Only
// the first and last word of a segment, which are shared with the neighbouring segments, need a
// merge; everything in between is a plain store.
//
// FSB_HD code: also compiled for the host by tests/emul/ (CPU-tier check against the oracle).
#pragma once

#include "core.cuh"

namespace fsb {

// ---- word-level helpers with host equivalents ----------------------------------------------------------
FSB_HD void or_word(uint32_t* p, uint32_t v)
{
#if defined(__CUDA_ARCH__)
    atomicOr(p, v);
#else
    *p |= v;
#endif
}

// ---- K1 output: one thread streams one segment into its record's slot ------------------------------------
// The segment is `nbits` bits at bit offset `off` of `words` (bit 0 = most significant bit of word
// 0; words are kept in big-endian *bit* order and byte-swapped when they leave for memory).  The
// producer pushes its stream as consecutive 32-bit words; every output word but the first is a
// plain store.  Word 0 may be shared with the segment in front of it (mate B follows mate A at a
// bit boundary), so it is held back and written by seg_finish, which the caller runs for the mates
// A first and -- after a __syncwarp -- for the mates B, merging into what A has stored.  No
// zero-initialisation and no atomics are needed; bits past the end of a segment are unspecified
// (K4 masks them).
struct SegEmit
{
    uint32_t* w;         // word holding the segment's first bit
    uint32_t phi;        // bit phase of the segment in that word
    uint32_t last;       // index of the last word with bits of the segment
    uint32_t idx;        // next output word
    uint32_t prev;       // previous stream word
    uint32_t v0;         // output word 0
    bool any;            // the segment is not empty
};
FSB_HD SegEmit seg_open(uint32_t* words, uint32_t off, uint32_t nbits)
{
    SegEmit e;
    e.w = words + (off >> 5);
    e.phi = off & 31u;
    e.any = nbits != 0;
    e.last = e.any ? (e.phi + nbits - 1u) >> 5 : 0u;
    e.idx = 0; e.prev = 0; e.v0 = 0;
    return e;
}
FSB_HD void seg_push(SegEmit& e, uint32_t x)                  // next 32 bits of the stream
{
    const uint32_t v = funnel_r(x, e.prev, e.phi);           // stream bits [32 idx - phi, 32 idx - phi + 32)
    e.prev = x;
    if (e.idx == 0) e.v0 = v;
    else if (e.idx <= e.last) e.w[e.idx] = v;
    e.idx++;
}
// the same for a word the caller knows to be neither word 0 nor (GUARD = false) past the segment's end
template <bool GUARD>
FSB_HD void seg_push_inner(SegEmit& e, uint32_t x)
{
    const uint32_t v = funnel_r(x, e.prev, e.phi);
    e.prev = x;
    if (!GUARD || e.idx <= e.last) e.w[e.idx] = v;
    e.idx++;
}
FSB_HD void seg_close(SegEmit& e) { if (e.idx <= e.last) seg_push(e, 0u); }     // the bits of the last stream word that spilled over
FSB_HD void seg_finish(const SegEmit& e, bool merge)
{
    if (!e.any) return;
    if (merge && e.phi) e.w[0] = (e.w[0] & ~(0xFFFFFFFFu >> e.phi)) | e.v0;     // the bits in front belong to mate A
    else e.w[0] = e.v0;
}

// small right-aligned values (meta fields): OR `nbits` (1..32) bits of v at bit offset off
FSB_HD void or_bits(uint32_t* words, uint32_t off, uint32_t v, uint32_t nbits)
{
    const uint32_t w = off >> 5, rel = off & 31u;
    const int32_t sh = 32 - (int32_t)rel - (int32_t)nbits;
    if (sh >= 0) or_word(words + w, v << sh);
    else
    {
        or_word(words + w, v >> (-sh));
        or_word(words + w + 1, v << (32 + sh));
    }
}

// ---- input: the stored symbols of one mate, four at a time ----------------------------------------------
// `w` is a word pointer, `addr` the byte offset of the mate's first source byte from it.  Stored
// order is the source order, or the reverse of it for a reversed read (FastqRecord::ComputeRC,
// FastqRecord.h:80-111: the quality is reversed alongside).  next() returns stored symbols
// 4j .. 4j+3 with the first one in the most significant byte; one PRMT does the unaligned
// extraction and the byte order for both directions.
struct SymReader
{
    const uint32_t* p;
    int32_t step;
    uint32_t sel;
    uint32_t carry;
};
FSB_HD SymReader reader_open(const uint32_t* w, uint32_t addr, uint32_t len, bool rev)
{
    SymReader r;
    if (!rev)
    {
        const uint32_t o = addr & 3u;
        r.p = w + (addr >> 2);
        r.step = 1;
        r.sel = ((o + 3u) & 7u) | (((o + 2u) & 7u) << 4) | (((o + 1u) & 7u) << 8) | (o << 12);      // result byte 3-t = pool[o + t]
    }
    else
    {
        const uint32_t e = addr + len, o = e & 3u;
        r.p = w + (e >> 2);
        r.step = -1;
        r.sel = ((4u + o) & 7u) | (((5u + o) & 7u) << 4) | (((6u + o) & 7u) << 8) | (((7u + o) & 7u) << 12);   // result byte t = pool[(4 + o + t) & 7]
    }
    r.carry = *r.p;
    return r;
}
FSB_HD uint32_t reader_next(SymReader& r)
{
    r.p += r.step;
    const uint32_t n = *r.p;
    const uint32_t x = byte_perm(r.carry, n, r.sel);
    r.carry = n;
    return x;
}

// ---- symbol coding --------------------------------------------------------------------------------------
// one 3-bit value per byte -> 12 bits, first symbol on top
FSB_HD uint32_t gather4x3(uint32_t v)
{
    const uint32_t y = (v & 0x00070007u) | ((v & 0x07000700u) >> 5);      // per half: [s_even s_odd] in 6 bits
    return (y & 0x3Fu) | ((y >> 10) & 0xFC0u);
}
// one bit per byte (bit 0) -> 4 bits, first symbol on top
FSB_HD uint32_t gather4x1(uint32_t f) { return (f * 0x10204080u) >> 28; }
// one 6-bit value per byte -> 24 bits, first symbol on top.  K1 is bound by the integer ALU pipe, so the
// two merge steps are written as multiply-adds (they issue on the other pipe): the odd bytes move down
// two bits as the high half of a product with 2^30, the upper 12-bit pair moves down four bits by
// subtracting 61440 times itself.
FSB_HD uint32_t mul_hi_add(uint32_t a, uint32_t b, uint32_t c)        // high word of a * b, plus c
{
#if defined(__CUDA_ARCH__)
    uint32_t r;
    asm("mad.hi.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
#else
    return (uint32_t)(((uint64_t)a * b) >> 32) + c;
#endif
}
FSB_HD uint32_t gather4x6(uint32_t x)
{
    const uint32_t c = mul_hi_add(x & 0x3F003F00u, 0x40000000u, x & 0x003F003Fu);      // [s0 s1] at bit 16, [s2 s3] at bit 0
    return (c >> 16) * 0xFFFF1000u + c;                                                  // c - 61440 * (c >> 16)
}
// StoreQuality (FastqPacker.cpp:205-269): four quality bytes -> four values of P.qua_bits bits.
template <int Q>
FSB_HD uint32_t quality4(uint32_t b, uint32_t off4 /* offset * 0x01010101 */, uint32_t thr4 /* threshold * 0x01010101 */)
{
    if (Q == 6) return gather4x6((b | 0x80808080u) - off4);             // (q - offset) & 63: the borrow guard bit 7 is masked off
    if (Q == 1)
    {   // c >= binaryThreshold on the unsigned difference: a "negative" difference is large.  The 1-bit mode takes every byte
        // from the offset up, so c needs all eight bits: per byte (q - offset) mod 256, no borrow between bytes
        const uint32_t c = ((b | 0x80808080u) - (off4 & 0x7F7F7F7Fu)) ^ ((b ^ ~off4) & 0x80808080u);
        const uint32_t ge = ((((c | 0x80808080u) - thr4) | c) >> 7) & 0x01010101u;
        return gather4x1(ge);
    }
    const uint32_t d = ((b | 0x80808080u) - off4) ^ 0x80808080u;        // per byte (q - offset) mod 256 for q < 128 (the table reads its low six bits)
    // quaToIdx_8bin (FastqPacker.cpp:41-64) of c & 63: [0,1]->0 [2,9]->1 [10,19]->2 [20,24]->3 [25,29]->4 [30,34]->5 [35,39]->6 >=40->7
    const uint32_t y = (d & 0x3F3F3F3Fu) | 0x80808080u;
    uint32_t v = 0;
    v += ((y - 0x02020202u) >> 7) & 0x01010101u;
    v += ((y - 0x0A0A0A0Au) >> 7) & 0x01010101u;
    v += ((y - 0x14141414u) >> 7) & 0x01010101u;
    v += ((y - 0x19191919u) >> 7) & 0x01010101u;
    v += ((y - 0x1E1E1E1Eu) >> 7) & 0x01010101u;
    v += ((y - 0x23232323u) >> 7) & 0x01010101u;
    v += ((y - 0x28282828u) >> 7) & 0x01010101u;
    return gather4x3(v);
}

// ---- K4: move one prepacked segment to its final bit position ------------------------------------------------
// `nbits` bits starting at bit `sbit` of src[] (MSB-first: bit 0 = most significant bit of src[0]) go
// to bit offset `off` of `words`.  Interior words are plain stores; the first and the last word --
// shared with the neighbouring segments -- are ORed into the zero-initialised buffer.  May read one
// word past the segment's last source word.
FSB_HD void shift_copy(const uint32_t* src, uint32_t sbit, uint32_t nbits, uint32_t* words, uint32_t off)
{
    if (nbits == 0) return;
    const uint32_t phi = off & 31u;
    uint32_t* w = words + (off >> 5);
    const uint32_t end = phi + nbits;
    const uint32_t last = (end - 1u) >> 5;                       // index of the last output word
    const uint32_t tailbits = end - 32u * last;                  // 1..32 valid bits in it
    const uint32_t lastmask = tailbits >= 32u ? 0xFFFFFFFFu : ~(0xFFFFFFFFu >> tailbits);
    // output word j holds the source bits [S + 32 j, S + 32 j + 32), S = sbit - phi >= -31
    const int32_t S = (int32_t)sbit - (int32_t)phi;
    const int32_t q = S >> 5;                                     // floor: -1 when the first word starts with bits of the neighbour
    const uint32_t r = (uint32_t)S & 31u;
    const uint32_t* p = src + q + 1;                              // output word j = (p[j - 1] : p[j]) << r
    uint32_t a = q >= 0 ? src[q] : 0u;
    uint32_t b = p[0];
    uint32_t v = funnel_l(b, a, r) & (0xFFFFFFFFu >> phi);
    a = b;
    if (last == 0) { or_word(w, v & lastmask); return; }
    or_word(w, v);
    uint32_t j = 1;
    for (; j + 4u <= last; j += 4)                                // words strictly inside the segment
    {
        const uint32_t x0 = p[j], x1 = p[j + 1], x2 = p[j + 2], x3 = p[j + 3];
        w[j] = funnel_l(x0, a, r); w[j + 1] = funnel_l(x1, x0, r); w[j + 2] = funnel_l(x2, x1, r); w[j + 3] = funnel_l(x3, x2, r);
        a = x3;
    }
    for (; j < last; ++j) { b = p[j]; w[j] = funnel_l(b, a, r); a = b; }
    b = p[last];
    or_word(w + last, funnel_l(b, a, r) & lastmask);
}

// ---- K4: the same for a 16-byte aligned source whose segment starts at bit 0 (vector loads) ------------------------
// `src` (16-byte aligned) holds `nbits` bits starting at bit 0 of src[0], MSB-first; they go to bit
// offset `off` of `words`.  Interior words are plain stores, the first and the last word -- shared
// with the neighbouring segments -- are ORed into the zero-initialised buffer.  Reads whole groups
// of four source words (up to 3 words past the segment; the caller's buffer covers them).
FSB_HD void load4(const uint32_t* p, uint32_t (&x)[4])
{
#if defined(__CUDA_ARCH__)
    const uint4 q = *reinterpret_cast<const uint4*>(p);
    x[0] = q.x; x[1] = q.y; x[2] = q.z; x[3] = q.w;
#else
    for (int u = 0; u < 4; ++u) x[u] = p[u];
#endif
}
FSB_HD void shift_copy_aligned(const uint32_t* src, uint32_t nbits, uint32_t* words, uint32_t off)
{
    if (nbits == 0) return;
    const uint32_t phi = off & 31u;
    uint32_t* w = words + (off >> 5);
    const uint32_t end = phi + nbits;
    const uint32_t last = (end - 1u) >> 5;                       // index of the last output word
    const uint32_t tailbits = end - 32u * last;                  // 1..32 valid bits in it
    const uint32_t lastmask = tailbits >= 32u ? 0xFFFFFFFFu : ~(0xFFFFFFFFu >> tailbits);
    uint32_t prev = 0, j = 0, x[4];
    if (last >= 4u)
    {   // first group: output word 0 is shared with the previous segment
        load4(src, x);
        or_word(w, funnel_r(x[0], 0u, phi));
        w[1] = funnel_r(x[1], x[0], phi); w[2] = funnel_r(x[2], x[1], phi); w[3] = funnel_r(x[3], x[2], phi);
        prev = x[3];
        for (j = 4; j + 4u <= last; j += 4)                       // groups whose four output words all lie strictly inside the segment
        {
            load4(src + j, x);
            w[j] = funnel_r(x[0], prev, phi); w[j + 1] = funnel_r(x[1], x[0], phi);
            w[j + 2] = funnel_r(x[2], x[1], phi); w[j + 3] = funnel_r(x[3], x[2], phi);
            prev = x[3];
        }
    }
    // last group: output words j .. last (1 to 4 of them; bits past the segment in the source are masked off)
    load4(src + j, x);
#pragma unroll
    for (uint32_t u = 0; u < 4; ++u)
    {
        const uint32_t jj = j + u;
        if (jj <= last)
        {
            const uint32_t v = funnel_r(x[u], prev, phi);       // stream bits [32 jj - phi, 32 jj - phi + 32)
            prev = x[u];
            if (jj == last) or_word(w + jj, v & lastmask);
            else if (jj == 0) or_word(w, v);
            else w[jj] = v;
        }
    }
}

// ---- quality stream of one stored mate (StoreQuality, FastqPacker.cpp:205-269) -------------------------------
// 32 symbols -> Q stream words per round; rounds are taken R at a time so that a step yields whole
// 16-byte vectors (12, 12 or 4 words), which go straight to the mate's quality region `dst` (16-byte
// aligned, in the record's slot in global memory): every lane stores its own vectors, no staging.
// Symbols past `len` inside the last round code to unspecified bits; rounds past the mate's end
// yield zero words; vectors past the stream's end are not written.
FSB_HD void store4(uint32_t* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d)
{
#if defined(__CUDA_ARCH__)
    *reinterpret_cast<uint4*>(p) = make_uint4(a, b, c, d);
#else
    p[0] = a; p[1] = b; p[2] = c; p[3] = d;
#endif
}
template <int Q>
FSB_HD void pack_quality_to(SymReader rd, uint32_t len, const DeviceParams& P, uint32_t* dst)
{
    constexpr int R = (Q == 6) ? 2 : 4;                          // rounds per step
    const uint32_t off4 = P.qua_offset * 0x01010101u, thr4 = P.qua_threshold * 0x01010101u;
    const uint32_t nwords = (len * Q + 31u) >> 5;
    uint32_t done = 0;                                           // symbols / words handled so far
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (uint32_t w0 = 0; w0 < nwords; w0 += R * Q, done += 32u * R)
    {
        uint32_t v[R * Q];
#pragma unroll
        for (int r = 0; r < R; ++r)
        {
            if (r == 0 || done + 32u * r < len)
            {
                uint32_t t[8];
#pragma unroll
#ifdef FSB_EXP_NOCOMPUTE
                for (int u = 0; u < 8; ++u) t[u] = u;
                (void)off4; (void)thr4;
#else
                for (int u = 0; u < 8; ++u) t[u] = quality4<Q>(reader_next(rd), off4, thr4);
#endif
                if constexpr (Q == 6)
                {   // 24 bits per group of four symbols: whole bytes, so the words are byte permutations
                    v[Q * r + 0] = byte_perm(t[1], t[0], 0x6542u);       // t0[23:0] t1[23:16]
                    v[Q * r + 1] = byte_perm(t[2], t[1], 0x5421u);       // t1[15:0] t2[23:8]
                    v[Q * r + 2] = byte_perm(t[3], t[2], 0x4210u);       // t2[7:0]  t3[23:0]
                    v[Q * r + 3] = byte_perm(t[5], t[4], 0x6542u);
                    v[Q * r + 4] = byte_perm(t[6], t[5], 0x5421u);
                    v[Q * r + 5] = byte_perm(t[7], t[6], 0x4210u);
                }
                else if constexpr (Q == 3)
                {
                    v[Q * r + 0] = (t[0] << 20) | (t[1] << 8) | (t[2] >> 4);
                    v[Q * r + 1] = (t[2] << 28) | (t[3] << 16) | (t[4] << 4) | (t[5] >> 8);
                    v[Q * r + 2] = (t[5] << 24) | (t[6] << 12) | t[7];
                }
                else
                    v[Q * r] = (t[0] << 28) | (t[1] << 24) | (t[2] << 20) | (t[3] << 16) | (t[4] << 12) | (t[5] << 8) | (t[6] << 4) | t[7];
            }
            else
            {
#pragma unroll
                for (int u = 0; u < Q; ++u) v[Q * r + u] = 0;
            }
        }
#pragma unroll
        for (int g = 0; g < R * Q / 4; ++g)
#ifndef FSB_EXP_NOSTORE
            if (w0 + 4u * g < nwords) store4(dst + w0 + 4 * g, v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
#else
            if (w0 + 4u * g < nwords && v[4 * g] == 0x12345u) store4(dst + w0 + 4 * g, v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
#endif
    }
}

// ---- DNA stream of one stored mate straight from K1's bit planes -----------------------------------------------
// K1 already holds the read as bit planes (sig_core.cuh: hi, lo, N; position p = bit p&31 of word
// p>>5).  The stored symbol stream is derived from them without touching the text again:
//   1. stored orientation, MSB-first planes: forward = bit-reversed words; reverse-complement
//      (FastqRecord::ComputeRC, FastqRecord.h:80-111) = complemented planes shifted so that base L-1
//      comes first.  'N' positions are cleared in hi/lo (N codes as 100b, FastqPacker.cpp:24-30);
//   2. the k signature symbols at [cut_pos, cut_pos + cut_len) are cut out of every plane;
//   3. hi and lo are interleaved into the 2-bit stream (perfect shuffle); a mate with 'N' expands
//      that to 3 bits per symbol with the N plane on top.
template <int NW> struct MsbPlanes { uint32_t h[NW + 1], l[NW + 1], n[NW + 1]; };

template <int NW> FSB_HD BV<NW> bv_shl_any(BV<NW> x, uint32_t s)          // r[p] = x[p - s], any s < 32 NW
{
    x = bv_shl(x, s & 31u);
    const uint32_t ws = s >> 5;
#pragma unroll
    for (int st = 1; st < NW; st <<= 1)
        if (ws & (uint32_t)st)
        {
#pragma unroll
            for (int j = NW - 1; j >= 0; --j) x.w[j] = j >= st ? x.w[j - st] : 0u;
        }
    return x;
}
FSB_HD uint32_t brev32(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __brev(x);
#else
    x = ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
    x = ((x >> 2) & 0x33333333u) | ((x & 0x33333333u) << 2);
    x = ((x >> 4) & 0x0F0F0F0Fu) | ((x & 0x0F0F0F0Fu) << 4);
    return bswap32(x);
#endif
}

template <int NW>
FSB_HD void stored_planes(const BV<NW>& H, const BV<NW>& Lo, const BV<NW>& Nm, uint32_t L, bool rev, MsbPlanes<NW>& o)
{
    if (!rev)
    {
#pragma unroll
        for (int j = 0; j < NW; ++j)
        {
            o.h[j] = brev32(H.w[j] & ~Nm.w[j]); o.l[j] = brev32(Lo.w[j] & ~Nm.w[j]); o.n[j] = brev32(Nm.w[j]);
        }
    }
    else
    {
        BV<NW> hc, lc;
#pragma unroll
        for (int j = 0; j < NW; ++j) { hc.w[j] = ~(H.w[j] | Nm.w[j]); lc.w[j] = ~(Lo.w[j] | Nm.w[j]); }       // 3 - code, 'N' stays clear
        const uint32_t sh = 32u * NW - L;
        // only positions below L may survive the shift: the planes hold text past the read there
        const BV<NW> valid = bv_range<NW>(0, (int32_t)L);
        const BV<NW> hs = bv_shl_any(bv_and(hc, valid), sh), ls = bv_shl_any(bv_and(lc, valid), sh), ns = bv_shl_any(Nm, sh);
#pragma unroll
        for (int j = 0; j < NW; ++j) { o.h[j] = hs.w[NW - 1 - j]; o.l[j] = ls.w[NW - 1 - j]; o.n[j] = ns.w[NW - 1 - j]; }
    }
    o.h[NW] = 0; o.l[NW] = 0; o.n[NW] = 0;
}

// remove cut_len (< 32) stream positions at cut_pos from MSB-first plane words
template <int NW>
FSB_HD void cut_planes(MsbPlanes<NW>& o, uint32_t cut_pos, uint32_t cut_len)
{
#pragma unroll
    for (int j = 0; j < NW; ++j)
    {
        const int32_t keep = (int32_t)cut_pos - 32 * j;            // leading positions of this word that precede the cut
        const uint32_t m = keep <= 0 ? 0u : (keep >= 32 ? 0xFFFFFFFFu : ~(0xFFFFFFFFu >> keep));
        o.h[j] = (o.h[j] & m) | (funnel_l(o.h[j + 1], o.h[j], cut_len) & ~m);
        o.l[j] = (o.l[j] & m) | (funnel_l(o.l[j + 1], o.l[j], cut_len) & ~m);
        o.n[j] = (o.n[j] & m) | (funnel_l(o.n[j + 1], o.n[j], cut_len) & ~m);
    }
}

// Bit-spreading tables: entry b of the first holds the bits of byte b at stride 2 (bit i -> bit 2i),
// entry 256 + b at stride 3 (bit i -> bit 3i).  The kernels keep a copy in shared memory; one
// lookup per plane byte replaces a shift-and-mask network per symbol group.
struct SpreadLut
{
    uint32_t v[512];
    constexpr SpreadLut() : v()
    {
        for (uint32_t b = 0; b < 256; ++b)
        {
            uint32_t s2 = 0, s3 = 0;
            for (uint32_t i = 0; i < 8; ++i)
                if (b & (1u << i)) { s2 |= 1u << (2 * i); s3 |= 1u << (3 * i); }
            v[b] = s2; v[256 + b] = s3;
        }
    }
};
// LUT accessors: a plain pointer (host emulation) or a 32-bit shared-memory address (K1)
struct LutPtr
{
    const uint32_t* t;
    FSB_HD uint32_t at(uint32_t tab, uint32_t byte) const { return t[tab + byte]; }
};
#if defined(__CUDACC__)
struct LutShared
{
    uint32_t base;           // shared-window address of the table
    __device__ __forceinline__ uint32_t at(uint32_t tab, uint32_t byte) const
    {
        uint32_t addr, v;
        asm("mad.lo.u32 %0, %1, 4, %2;" : "=r"(addr) : "r"(byte), "r"(base + 4u * tab));
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
        return v;
    }
};
#endif
FSB_HD uint32_t byte_of(uint32_t x, int b)                         // byte b of x, zero extended (pool bytes 4..7 are zero)
{
    return byte_perm(x, 0u, b == 0 ? 0x4440u : b == 1 ? 0x4441u : b == 2 ? 0x4442u : 0x4443u);
}

// the whole DNA segment of one stored mate.  The loop over the plane words stays rolled (see
// ascii_to_planes): each round codes word 0 of the planes, then the planes move down one word.  Mates
// with and without 'N' run the same round -- a warp nearly always holds both kinds: they differ in the
// table they look up (bits spread to stride 2 or 3; the N plane of a plain mate is empty and adds
// nothing) and in how the four symbol groups of a round (16 or 24 bits each) make up stream words.
template <int NW, class LUT>
FSB_HD void pack_dna_planes(const BV<NW>& H, const BV<NW>& Lo, const BV<NW>& Nm, uint32_t L, bool rev, bool plain,
                            uint32_t cut_pos, uint32_t cut_len, const LUT& lut, SegEmit& e)
{
    MsbPlanes<NW> o;
    stored_planes<NW>(H, Lo, Nm, L, rev, o);
    if (cut_len) cut_planes<NW>(o, cut_pos, cut_len);
    const uint32_t tab = plain ? 0u : 256u;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int j = 0; j < NW; ++j)
    {
        uint32_t t[4];                                               // symbols 8b .. 8b+7 of the round, first group in t[0]
#pragma unroll
        for (int b = 0; b < 4; ++b)
            t[b] = 4u * lut.at(tab, byte_of(o.n[0], 3 - b)) + 2u * lut.at(tab, byte_of(o.h[0], 3 - b)) + lut.at(tab, byte_of(o.l[0], 3 - b));
        // 2 bits per symbol: two words of two 16-bit groups; 3 bits: three words out of four 24-bit groups
        seg_push(e, plain ? (t[0] << 16) + t[1] : byte_perm(t[1], t[0], 0x6542u));          // t0[23:0] t1[23:16]
        seg_push(e, plain ? (t[2] << 16) + t[3] : byte_perm(t[2], t[1], 0x5421u));          // t1[15:0] t2[23:8]
        if (!plain) seg_push(e, byte_perm(t[3], t[2], 0x4210u));                            // t2[7:0]  t3[23:0]
#pragma unroll
        for (int i = 0; i + 1 < NW; ++i) { o.h[i] = o.h[i + 1]; o.l[i] = o.l[i + 1]; o.n[i] = o.n[i + 1]; }
    }
    seg_close(e);
}

// one 7-bit value per byte -> 28 bits, first symbol on top
FSB_HD uint32_t gather4x7(uint32_t x)
{
    const uint32_t c = ((x & 0x7F007F00u) >> 1) | (x & 0x007F007Fu);
    return ((c & 0x3FFF0000u) >> 2) | (c & 0x00003FFFu);
}
// Four characters per step; `hold` keeps the n < 32 stream bits not yet pushed, left aligned.
// The title is packed in two parts that start at word boundaries of the stream, so that the two lanes of a pair
// can take one each: part 0 = the length byte and the first eight characters (64 bits), part 1 = the rest.
// `region` is the word the title starts in (bit 0); both parts finish their own word 0.
FSB_HD void pack_head_part(const uint32_t* w, uint32_t addr, uint32_t H, uint32_t part, uint32_t* region)
{
    const uint32_t head_bits = 8u + 7u * (H ? H - 1u : 0u);
    const uint32_t groups_total = H > 1u ? (H + 2u) >> 2 : 0u;  // ceil((H - 1) / 4); characters past the title code to unspecified bits
    const uint32_t groups = part ? (groups_total > 2u ? groups_total - 2u : 0u) : (groups_total < 2u ? groups_total : 2u);
    const uint32_t nbits = part ? (head_bits > 64u ? head_bits - 64u : 0u) : (head_bits < 64u ? head_bits : 64u);
    if (nbits == 0) return;
    SegEmit e = seg_open(region, part ? 64u : 0u, nbits);
    uint32_t hold = part ? 0u : (H & 0xFFu) << 24, n = part ? 0u : 8u;
    if (groups)
    {
        SymReader rd = reader_open(w, addr + (part ? 9u : 1u), 4u * groups, false);
        for (uint32_t g = 0; g < groups; ++g)
        {
            const uint32_t c = gather4x7(reader_next(rd)) << 4;   // 28 bits, left aligned
            const uint32_t word = hold | (c >> n);
            if (n >= 4u) { seg_push(e, word); hold = c << (32u - n); n -= 4u; }
            else { hold = word; n += 28u; }
        }
    }
    if (n) seg_push(e, hold);
    seg_close(e);
    seg_finish(e, false);
}
FSB_HD void pack_head(const uint32_t* w, uint32_t addr, uint32_t H, uint32_t* region)
{
    pack_head_part(w, addr, H, 0u, region);
    pack_head_part(w, addr, H, 1u, region);
}

// ---- per-record framing (StoreRecords SE :734-759 / PE :815-859, StoreNextRecord :113-153) --------------
struct ReadBits { uint32_t meta, dna, qua, head; };

FSB_HD ReadBits read_bit_lengths(const DeviceParams& P, bool nbin, uint32_t info, uint32_t L1, uint32_t L2, uint32_t H,
                                 uint32_t bmin, uint32_t bmax)
{
    ReadBits b;
    const bool pe = P.paired != 0;
    const uint32_t bpl = (bmin != bmax) ? bit_length_u32(bmax - bmin) : 0;
    b.meta = (pe ? 2 * bpl : bpl) + (nbin ? 0u : (pe ? 10u : 9u)) + 1u + (pe ? 1u : 0u);
    const uint32_t bitsA = (info & FSB_INFO_PLAIN_A) ? 2u : 3u, bitsB = (info & FSB_INFO_PLAIN_B) ? 2u : 3u;
    b.dna = (L1 - (nbin ? 0u : P.k)) * bitsA + (pe ? L2 * bitsB : 0u);
    b.qua = (L1 + (pe ? L2 : 0u)) * P.qua_bits;
    b.head = P.has_headers ? 8u + 7u * (H ? H - 1u : 0u) : 0u;
    return b;
}

// the record's meta fields, most significant first, as one right-aligned value (at most 28 bits)
FSB_HD uint32_t meta_fields(const DeviceParams& P, bool nbin, uint32_t info, uint32_t lenA, uint32_t lenB, uint32_t bmin, uint32_t bmax, uint32_t& nbits)
{
    const bool pe = P.paired != 0;
    uint32_t v = 0, n = 0;
    if (bmin != bmax)
    {
        const uint32_t bpl = bit_length_u32(bmax - bmin), m = (1u << bpl) - 1u;
        v = (lenA - bmin) & m; n = bpl;                                               // rec->seqLen - minLen
        if (pe) { v = (v << bpl) | ((lenB - bmin) & m); n += bpl; }
    }
    if (!nbin)
    {
        if (pe) { v = (v << 1) | ((info & FSB_INFO_SWAPPED) ? 1u : 0u); n += 1; }
        v = (v << 1) | ((info & FSB_INFO_REVERSE) ? 1u : 0u); n += 1;
        v = (v << 8) | (info & 0xFFu); n += 8;
    }
    v = (v << 1) | ((info & FSB_INFO_PLAIN_A) ? 1u : 0u); n += 1;
    if (pe) { v = (v << 1) | ((info & FSB_INFO_PLAIN_B) ? 1u : 0u); n += 1; }
    nbits = n;
    return v;
}

} // namespace fsb
