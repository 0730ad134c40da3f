// stage.cuh -- device-side check of the staged record tables and the batch statistics the host
// needs to size buffers and pick kernel instantiations.
//
// The reference only ASSERTs its input contract (FastqRecord.h:87,192; FastqParser.cpp:130): read
// length 1..255, equal mate lengths in a pair, views inside the chunk.  Violations would make the
// kernels read outside the staged text, so fsb_stage rejects them (FSB_ERR_INPUT).
#pragma once

#include <cuda_runtime.h>

#include "core.cuh"
#include "stage_core.cuh"

namespace fsb {

struct StageStats
{
    unsigned long long bases;        // sum of sequence lengths, both mates
    unsigned long long heads;        // sum of head_len (mate 1)
    unsigned long long first_bad;    // lowest record index violating the contract (~0 if none)
    uint32_t min_len, max_len;       // over all mates
    uint32_t max_head;
    uint32_t n_bad;
    unsigned long long first_bad_text;   // lowest record index with a symbol / quality / title byte outside the contract (~0 if none)
    uint32_t n_bad_text, pad;
};

// chunk_sums[2 c] / [2 c + 1]: bases (both mates) and kept title bytes of chunk c -- they bound the chunk's output, which lets
// fsb_run give every sub-batch of whole chunks its own region of the output streams.
__global__ void __launch_bounds__(256) stage_stats_kernel(BatchView B, DeviceParams P, const uint64_t* __restrict__ text_size0,
                                                          const uint64_t* __restrict__ text_size1, StageStats* __restrict__ st,
                                                          unsigned long long* __restrict__ chunk_sums)
{
    __shared__ unsigned long long sh_bases, sh_heads;
    __shared__ uint32_t sh_min, sh_max, sh_hmax;
    if (threadIdx.x == 0) { sh_bases = 0; sh_heads = 0; sh_min = 0xFFFFFFFFu; sh_max = 0; sh_hmax = 0; }
    __syncthreads();
    uint64_t bases = 0, heads = 0;
    uint32_t mn = 0xFFFFFFFFu, mx = 0, hmx = 0;
    const unsigned lane = threadIdx.x & 31;
    for (uint64_t i0 = (uint64_t)blockIdx.x * blockDim.x; i0 < B.n_records; i0 += (uint64_t)gridDim.x * blockDim.x)     // block uniform
    {
        const uint64_t i = i0 + threadIdx.x;
        const bool live = i < B.n_records;
        uint32_t ch = 0xFFFFFFFFu, rb = 0, rh = 0;
        if (live)
        {
            ch = find_chunk(B, i);
            const fsb_record a = B.rec[0][i];
            const uint64_t ts0 = text_size0[ch];
            bool ok = a.seq_len >= 1 && a.seq_len <= 255 && (uint64_t)a.seq_off + a.seq_len <= ts0 && (uint64_t)a.qua_off + a.seq_len <= ts0 &&
                      (uint64_t)a.head_off + a.head_len <= ts0;
            rb = a.seq_len; rh = a.head_len;
            mn = min(mn, (uint32_t)a.seq_len); mx = max(mx, (uint32_t)a.seq_len); hmx = max(hmx, (uint32_t)a.head_len);
            if (P.paired)
            {
                const fsb_record b = B.rec[1][i];
                const uint64_t ts1 = text_size1[ch];
                ok = ok && b.seq_len == a.seq_len && (uint64_t)b.seq_off + b.seq_len <= ts1 && (uint64_t)b.qua_off + b.seq_len <= ts1;
                rb += b.seq_len;
            }
            if (!ok) { atomicAdd(&st->n_bad, 1u); atomicMin(&st->first_bad, (unsigned long long)i); }
        }
        bases += rb; heads += rh;
        // per-chunk sums: the lanes of a warp nearly always share the chunk, one lane per (warp, chunk) adds
        const unsigned peers = __match_any_sync(0xFFFFFFFFu, ch);
        const uint32_t sb = __reduce_add_sync(peers, rb), sh = __reduce_add_sync(peers, rh);
        if (live && (unsigned)(__ffs(peers) - 1) == lane)
        {
            atomicAdd(&chunk_sums[2 * ch], (unsigned long long)sb);
            atomicAdd(&chunk_sums[2 * ch + 1], (unsigned long long)sh);
        }
    }
    atomicAdd(&sh_bases, (unsigned long long)bases); atomicAdd(&sh_heads, (unsigned long long)heads);
    atomicMin(&sh_min, mn); atomicMax(&sh_max, mx); atomicMax(&sh_hmax, hmx);
    __syncthreads();
    if (threadIdx.x == 0)
    {
        atomicAdd(&st->bases, sh_bases); atomicAdd(&st->heads, sh_heads);
        atomicMin(&st->min_len, sh_min); atomicMax(&st->max_len, sh_max); atomicMax(&st->max_head, sh_hmax);
    }
}

// ---- FSB_OPT_VALIDATE: the bytes behind the record table ---------------------------------------------------------
// The reference leaves symbols outside ACGTN undefined (out-of-table look-ups in ComputeRC / StoreDna,
// FastqRecord.h:95-96, FastqPacker.cpp:24-30) and indexes its 64-entry quality table with (q - offset)
// unchecked (FastqPacker.cpp:250); K1 would code such bytes as something, silently.  This kernel rejects them
// before the pipeline runs: sequence bytes must be one of A C G T N, quality bytes must lie in
// [offset, offset + 64) for the 6- and 3-bit modes and be >= offset for the 1-bit mode, kept title characters
// must be 7-bit (StoreHeader packs 7 bits per character, FastqPacker.cpp:272-287) -- the same rules the host
// parser applies (csrc/host/fastq_parser.cpp).  It is a streaming pass over the staged text with 16-byte loads
// (a half warp per mate: lane j checks the j-th aligned 16-byte piece of the sequence, of the quality and of the
// title), part of fsb_stage, not of the timed fsb_run path.
// The checks of one piece live in stage_core.cuh; here the piece arrives as one 16-byte load.
template <int KIND>
__device__ __forceinline__ bool piece_ok(const uint4& q, int32_t piece, int32_t lo, int32_t hi, uint32_t off4, bool need_range)
{
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
    return piece_ok<KIND>(w, piece, lo, hi, off4, need_range);
}

// A half warp per mate: lane j checks the j-th aligned 16-byte piece of the sequence, of the quality and of the title (the
// three loads are issued together; reads longer than ~240 bases take a second round).  The chunk tables sit in shared
// memory, and the next mate's record is fetched while the current one is checked.
__global__ void __launch_bounds__(256) validate_text_kernel(BatchView B, DeviceParams P, const uint64_t* __restrict__ text_size0,
                                                            const uint64_t* __restrict__ text_size1, StageStats* __restrict__ st)
{
    constexpr uint32_t kMaxChunks = 256;
    __shared__ uint64_t s_first[kMaxChunks + 1], s_base[2][kMaxChunks], s_size[2][kMaxChunks];
    for (uint32_t c = threadIdx.x; c <= B.n_chunks && c <= kMaxChunks; c += blockDim.x)
    {
        s_first[c] = B.chunk_first_rec[c];
        if (c < B.n_chunks)
        {
            s_base[0][c] = B.chunk_text_base[0][c]; s_size[0][c] = text_size0[c];
            s_base[1][c] = P.paired ? B.chunk_text_base[1][c] : 0ull; s_size[1][c] = P.paired ? text_size1[c] : 0ull;
        }
    }
    __syncthreads();
    const uint32_t half = threadIdx.x >> 4;                                              // 16 half warps per block
    const int32_t l16 = (int32_t)(threadIdx.x & 15u);
    const uint64_t n_mates = P.paired ? 2 * B.n_records : B.n_records;
    const bool need_range = P.qua_bits != 1;                                            // 1-bit mode: only q >= offset (the threshold compare takes any value)
    const uint32_t off4 = quality_off4(P.qua_offset);
    const uint64_t stride = (uint64_t)gridDim.x * 16u;
    uint64_t g = (uint64_t)blockIdx.x * 16u + half;
    auto load_rec = [&](uint64_t gg) -> uint4
    {
        if (gg >= n_mates) return make_uint4(0, 0, 0, 0);
        const uint64_t i = P.paired ? (gg >> 1) : gg;
        return *reinterpret_cast<const uint4*>(((P.paired && (gg & 1u)) ? B.rec[1] : B.rec[0]) + i);
    };
    uint4 rw = load_rec(g);
    for (; g < n_mates; g += stride)
    {
        const uint4 cur = rw;
        rw = load_rec(g + stride);                                                       // in flight during the checks
        const uint64_t i = P.paired ? (g >> 1) : g;
        const uint32_t m = P.paired ? (uint32_t)(g & 1u) : 0u;
        uint32_t lo_c = 0, hi_c = B.n_chunks;                                            // chunk of the record: first[lo] <= i < first[hi]
        while (hi_c - lo_c > 1) { const uint32_t mid = (lo_c + hi_c) >> 1; if (s_first[mid] <= i) lo_c = mid; else hi_c = mid; }
        const uint32_t head_off = cur.x, seq_off = cur.y, qua_off = cur.z, L = cur.w & 0xFFFFu, head_len = (cur.w >> 16) & 0xFFu;
        const uint64_t ts = s_size[m][lo_c];
        // records whose views leave the chunk are reported by stage_stats_kernel; never follow them
        if (L < 1 || L > 255 || (uint64_t)seq_off + L > ts || (uint64_t)qua_off + L > ts || (uint64_t)head_off + head_len > ts) continue;
        const uint8_t* text = B.text[m] + s_base[m][lo_c];
        const uint32_t H = (m == 0 && P.has_headers) ? head_len : 0u;
        const CheckSpan sq = check_span(text + seq_off, L), qu = check_span(text + qua_off, L), hd = check_span(text + head_off + 1u, H > 1u ? H - 1u : 0u);
        // first round: pieces 0..15 of the three spans, the loads side by side
        const bool in_s = l16 * 16 < sq.hi, in_q = l16 * 16 < qu.hi, in_h = l16 * 16 < hd.hi;
        uint4 vs = make_uint4(0, 0, 0, 0), vq = vs, vh = vs;
        if (in_s) vs = *reinterpret_cast<const uint4*>(sq.a0 + 16u * (uint32_t)l16);
        if (in_q) vq = *reinterpret_cast<const uint4*>(qu.a0 + 16u * (uint32_t)l16);
        if (in_h) vh = *reinterpret_cast<const uint4*>(hd.a0 + 16u * (uint32_t)l16);
        bool ok = true;
        if (in_s) ok = piece_ok<0>(vs, l16, sq.lo, sq.hi, off4, need_range);
        if (in_q) ok = ok && piece_ok<1>(vq, l16, qu.lo, qu.hi, off4, need_range);
        if (in_h) ok = ok && piece_ok<2>(vh, l16, hd.lo, hd.hi, off4, need_range);
        // the 17th piece of spans of more than 240 bytes
        for (int32_t piece = l16 + 16; piece * 16 < sq.hi; piece += 16) ok = ok && piece_ok<0>(*reinterpret_cast<const uint4*>(sq.a0 + 16u * (uint32_t)piece), piece, sq.lo, sq.hi, off4, need_range);
        for (int32_t piece = l16 + 16; piece * 16 < qu.hi; piece += 16) ok = ok && piece_ok<1>(*reinterpret_cast<const uint4*>(qu.a0 + 16u * (uint32_t)piece), piece, qu.lo, qu.hi, off4, need_range);
        for (int32_t piece = l16 + 16; piece * 16 < hd.hi; piece += 16) ok = ok && piece_ok<2>(*reinterpret_cast<const uint4*>(hd.a0 + 16u * (uint32_t)piece), piece, hd.lo, hd.hi, off4, need_range);
        const unsigned half_mask = 0xFFFFu << (16u * (half & 1u));                        // the 16 lanes of this mate
        const bool bad = __any_sync(half_mask, !ok);
        if (bad && l16 == 0) { atomicAdd(&st->n_bad_text, 1u); atomicMin(&st->first_bad_text, (unsigned long long)i); }
    }
}

} // namespace fsb
