// stage_core.cuh -- the byte check of FSB_OPT_VALIDATE (validate_text_kernel, stage.cuh): which bytes of an aligned
// 16-byte piece belong to a span, and whether the sequence symbols, quality bytes and title characters among them are
// inside the input contract, four bytes at a time.
//
// FSB_HD code: tests/emul/ runs the kernel's per-mate check on the host against a byte-by-byte statement of the
// contract (CPU tier).
#pragma once

#include <algorithm>

#include "core.cuh"

namespace fsb {

// 0xFF for every byte of a 4-byte word whose offset word_base + b lies in [lo, hi)
FSB_HD uint32_t bytes_in_range_mask(int32_t lo, int32_t hi, int32_t word_base)
{
    uint32_t ma, mb;
#if defined(__CUDA_ARCH__)
    const int32_t a = min(max(lo - word_base, 0), 4), b = min(max(hi - word_base, 0), 4);      // bytes [a, b) of the word
    asm("shl.b32 %0, %1, %2;" : "=r"(ma) : "r"(0xFFFFFFFFu), "r"(8u * (uint32_t)a));          // shl.b32 clamps counts above 31 (result 0)
    asm("shl.b32 %0, %1, %2;" : "=r"(mb) : "r"(0xFFFFFFFFu), "r"(8u * (uint32_t)b));
#else
    const int32_t a = std::min(std::max(lo - word_base, 0), 4), b = std::min(std::max(hi - word_base, 0), 4);
    ma = a < 4 ? 0xFFFFFFFFu << (8 * a) : 0u;                                                 // the same clamped shift
    mb = b < 4 ? 0xFFFFFFFFu << (8 * b) : 0u;
#endif
    return ma & ~mb;
}
// All four bytes at once.  A valid base is one of A 0x41, C 0x43, G 0x47, T 0x54, N 0x4E: bits 7..5 are 010, and with
// c = bits 3..1 (the code K1's bit planes are built from: A 000, C 001, T 010, G 011, N 111; 100, 101, 110 do not
// occur) bit 4 is set for T only and bit 0 is clear for T and N only.  Bit k of every byte is looked at in place
// (w >> k keeps it at bit 0 of the byte; the other bits of the byte are masked off at the end).
FSB_HD bool dna_word_ok(uint32_t w, uint32_t m)
{
    w = (w & m) | (0x41414141u & ~m);                                 // bytes outside the span count as 'A'
    const uint32_t s1 = w >> 1, s2 = w >> 2, s3 = w >> 3, s4 = w >> 4, s5 = w >> 5;
    const uint32_t isT = ~s3 & s2 & ~s1, isN = s3 & s2 & s1;
    const uint32_t bad_code = s3 & ~(s2 & s1);
    const uint32_t bad_b4 = s4 ^ isT, bad_b0 = w ^ ~(isT | isN);
    const uint32_t low = (bad_code | bad_b4 | bad_b0) & 0x01010101u;
    const uint32_t high = (s5 ^ 0x02020202u) & 0x07070707u;
    return (low | high) == 0;
}
// offset * 0x01010101 for qua_word_ok.  The check is only defined for offsets 0..127, which fsb_create enforces.
FSB_HD uint32_t quality_off4(uint32_t qua_offset) { return (qua_offset & 0x7Fu) * 0x01010101u; }
// q - offset in [0, 64) for the 6- and 3-bit modes (need_range), q >= offset for the 1-bit mode; off4 = offset * 0x01010101, offset <= 127.
// Per byte t = (q | 128) - offset never borrows from its neighbour.  For q < 128 that is q - offset + 128: in range <=> bit 7 set and
// bit 6 clear; for q >= 128 it is q - offset itself: in range <=> bits 7 and 6 clear.
FSB_HD bool qua_word_ok(uint32_t w, uint32_t m, uint32_t off4, bool need_range)
{
    w = (w & m) | (off4 & ~m);                                        // bytes outside the span count as quality 0
    const uint32_t t = (w | 0x80808080u) - off4;
    const uint32_t h = w & 0x80808080u;
    const uint32_t bad = need_range ? ((t ^ ~h) | (t << 1)) : (~t & ~w);
    return (bad & 0x80808080u) == 0;
}

// one aligned 16-byte piece (words w[0..3], in memory order) of a span: `lo`/`hi` = the span's byte range counted from the
// aligned address a0
template <int KIND>     // 0 sequence, 1 quality, 2 title characters
FSB_HD bool piece_ok(const uint32_t (&w)[4], int32_t piece, int32_t lo, int32_t hi, uint32_t off4, bool need_range)
{
    const bool inner = piece * 16 >= lo && piece * 16 + 16 <= hi;     // every byte of the piece belongs to the span (all but the first and last piece)
    bool ok = true;
#pragma unroll
    for (int j = 0; j < 4; ++j)
    {
        const uint32_t msk = inner ? 0xFFFFFFFFu : bytes_in_range_mask(lo, hi, piece * 16 + 4 * j);
        if (KIND == 0) ok = ok && dna_word_ok(w[j], msk);
        else if (KIND == 1) ok = ok && qua_word_ok(w[j], msk, off4, need_range);
        else ok = ok && ((w[j] & msk & 0x80808080u) == 0);
    }
    return ok;
}

struct CheckSpan { uintptr_t a0; int32_t lo, hi; };
FSB_HD CheckSpan check_span(const uint8_t* p0, uint32_t len)
{
    CheckSpan s;
    s.a0 = reinterpret_cast<uintptr_t>(p0) & ~(uintptr_t)15;          // the text buffers are padded: aligned pieces stay inside
    s.lo = (int32_t)(reinterpret_cast<uintptr_t>(p0) - s.a0);
    s.hi = len ? s.lo + (int32_t)len : 0;                             // hi = 0: nothing to check
    return s;
}

} // namespace fsb
