// layout_fused.cuh -- the layout of a batch whose reads all have one length, as one scan (sm_100a).
//
// Replaces, for such batches, the kernels of layout.cuh and the placement kernel of place.cuh: three
// streaming launches turn the sorted (key, card) pairs into everything K4 needs -- every record's bit
// position inside its K4 tile for the four streams, the tiles' first bits, the per-record bin info --
// plus the bin descriptors and the per-chunk summary.  The arithmetic is layout_core.cuh's scan.
//
// Mapping: a thread owns one K4 tile (32 consecutive sorted records) and walks over it sequentially; a block
// of 128 threads owns 4096 records.  A warp first copies its 32 runs into shared memory with coalesced loads (a
// thread's own 128 + 256 contiguous bytes, loaded by the thread, would touch 32 lines per warp instruction), and
// lay_apply stages loc / binfo in shared memory for eight records a round so that the warp writes whole sectors.
//   lay_reduce   every block's LayState                              -> tile_states[block]
//   lay_scan_groups / lay_scan_finish   exclusive scan over the block states (in place; [nblocks] = the whole batch)
//   lay_apply    thread prefix = block prefix (+) threads in front; absolute walk that writes loc / binfo / tbase,
//                clears the stream words two K4 tiles share, and emits the descriptor of every bin at its last record
//   chunk_summary_fused   per chunk: first bin, stream offsets and sizes, raw sizes (block per chunk)
#pragma once

#include <cuda_runtime.h>

#include "layout_core.cuh"
#include "layout.cuh"
#include "place.cuh"

namespace fsb {

constexpr uint32_t kLayThreads = 128;
constexpr uint32_t kLayPerThread = kPlaceTile;                      // a thread walks over one K4 tile
constexpr uint32_t kLayBlock = kLayThreads * kLayPerThread;         // 4096 records per block
static_assert(kLayPerThread == 32, "a warp stages its runs as 32 x 32 records");

// ---- moving a LayState between lanes ---------------------------------------------------------------------------
constexpr int kLayWords = (int)(sizeof(LayState) / 4);
static_assert(sizeof(LayState) % 4 == 0, "LayState moves as 32-bit words");
__device__ __forceinline__ LayState lay_shfl_up(const LayState& s, unsigned d)
{
    LayState r;
    const uint32_t* in = reinterpret_cast<const uint32_t*>(&s);
    uint32_t* out = reinterpret_cast<uint32_t*>(&r);
#pragma unroll
    for (int w = 0; w < kLayWords; ++w) out[w] = __shfl_up_sync(0xFFFFFFFFu, in[w], d);
    return r;
}
// inclusive scan over the lanes of a warp (lane order = record order)
__device__ __forceinline__ LayState lay_warp_scan(LayState s)
{
    const unsigned lane = threadIdx.x & 31;
#pragma unroll
    for (unsigned d = 1; d < 32; d <<= 1)
    {
        const LayState o = lay_shfl_up(s, d);
        if (lane >= d) s = lay_combine(o, s);
    }
    return s;
}
// Exclusive prefix of `mine` over the threads of the block (thread order = record order); `total` = the block's state.
__device__ __forceinline__ LayState lay_block_scan(const LayState& mine, LayState& total, LayState* sm /* kLayThreads / 32 entries */)
{
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const LayState inc = lay_warp_scan(mine);
    if (lane == 31) sm[warp] = inc;
    __syncthreads();
    LayState before = lay_identity();                               // the warps in front of this one
    total = lay_identity();
#pragma unroll
    for (unsigned w = 0; w < kLayThreads / 32; ++w)
    {
        if (w == warp) before = total;
        total = lay_combine(total, sm[w]);
    }
    LayState excl = lay_shfl_up(inc, 1);                            // the lanes in front inside the warp
    if (lane == 0) excl = lay_identity();
    __syncthreads();
    return lay_combine(before, excl);
}

// A thread's run of sorted records.
struct LayRun
{
    uint64_t i0;             // first record
    uint32_t cnt;            // records (0 .. 32)
};
__device__ __forceinline__ LayRun lay_run(uint64_t n)
{
    LayRun r;
    r.i0 = ((uint64_t)blockIdx.x * kLayThreads + threadIdx.x) * kLayPerThread;
    r.cnt = r.i0 < n ? (uint32_t)min((uint64_t)kLayPerThread, n - r.i0) : 0u;
    return r;
}

// A warp's 32 runs in shared memory, one row per thread.  Rows of 33 entries: a thread walking its row and the
// warp filling the rows with coalesced loads both hit 32 different banks.
constexpr uint32_t kLayRow = kLayPerThread + 1;
struct LayWarpIn
{
    uint32_t keys[32][kLayRow];
    unsigned long long cards[32][kLayRow];
};
// loc[0..3] and binfo of one round of kLayRound records per thread, before the warp writes them out together
constexpr uint32_t kLayRound = 8;
constexpr uint32_t kLayOutWords = 5 * 32 * kLayRound;
constexpr size_t kLayReduceSmem = (kLayThreads / 32) * sizeof(LayWarpIn);
constexpr size_t kLayApplySmem = (kLayThreads / 32) * (sizeof(LayWarpIn) + kLayOutWords * 4);
static_assert(sizeof(LayWarpIn) % 16 == 0, "the out staging behind the runs takes 16-byte vectors");

// the records [wb, wb + 32 * kLayPerThread) of the warp (those below n) into its rows, with 16-byte loads
__device__ __forceinline__ void lay_stage(const SortedView& S, uint64_t n, uint64_t wb, LayWarpIn& w)
{
    const unsigned lane = threadIdx.x & 31;
    if (wb + 32 * kLayPerThread <= n)
    {
        const uint4* k4 = reinterpret_cast<const uint4*>(S.skeys + wb);
        const ulonglong2* c2 = reinterpret_cast<const ulonglong2*>(S.cards + wb);
#pragma unroll
        for (uint32_t it = 0; it < kLayPerThread / 4; ++it)
        {
            const uint32_t v = it * 32 + lane;
            const uint4 q = k4[v];
            uint32_t* o = &w.keys[v / 8][4 * (v % 8)];
            o[0] = q.x; o[1] = q.y; o[2] = q.z; o[3] = q.w;
        }
#pragma unroll
        for (uint32_t it = 0; it < kLayPerThread / 2; ++it)
        {
            const uint32_t v = it * 32 + lane;
            const ulonglong2 q = c2[v];
            unsigned long long* o = &w.cards[v / 16][2 * (v % 16)];
            o[0] = q.x; o[1] = q.y;
        }
    }
    else
    {
        for (uint32_t r = lane; r < 32 * kLayPerThread && wb + r < n; r += 32)
        {
            w.keys[r / kLayPerThread][r % kLayPerThread] = S.skeys[wb + r];
            w.cards[r / kLayPerThread][r % kLayPerThread] = S.cards[wb + r];
        }
    }
    __syncwarp();
}
// the key in front of the thread's run (only the last run of a batch is partial, so the run in front is whole); 0 for an empty
// run, whose lane 0 would otherwise read behind the end of the keys
__device__ __forceinline__ uint32_t lay_prev_key(const SortedView& S, const LayWarpIn& w, const LayRun& run)
{
    const unsigned lane = threadIdx.x & 31;
    if (!run.cnt) return 0u;
    return lane ? w.keys[lane - 1][kLayPerThread - 1] : (run.i0 ? S.skeys[run.i0 - 1] : 0u);
}
// the state of a thread's run, walked from its row
__device__ __forceinline__ LayState lay_run_state(const DeviceParams& P, const LayWarpIn& w, uint32_t prev, const LayRun& run, uint32_t uniform_len)
{
    const unsigned lane = threadIdx.x & 31;
    LayState st = lay_identity();
#pragma unroll 4
    for (uint32_t j = 0; j < run.cnt; ++j)
    {
        const uint32_t key = w.keys[lane][j];
        lay_push(st, lay_record(P, run.i0 + j == 0, key, prev, w.cards[lane][j], uniform_len));
        prev = key;
    }
    return st;
}

__global__ void __launch_bounds__(kLayThreads) lay_reduce_kernel(uint64_t n, DeviceParams P, SortedView S, uint32_t uniform_len, LayState* __restrict__ tile_states)
{
    extern __shared__ uint4 lay_smem_raw[];
    __shared__ LayState sm[kLayThreads / 32];
    LayWarpIn& w = reinterpret_cast<LayWarpIn*>(lay_smem_raw)[threadIdx.x >> 5];
    const LayRun run = lay_run(n);
    lay_stage(S, n, run.i0 - (uint64_t)(threadIdx.x & 31) * kLayPerThread, w);
    const LayState mine = lay_run_state(P, w, lay_prev_key(S, w, run), run, uniform_len);
    LayState total;
    lay_block_scan(mine, total, sm);
    if (threadIdx.x == 0) tile_states[blockIdx.x] = total;
}

// states[j] <- combination of states[0 .. j)  (j = 0 .. count; entry [count] is the whole batch), in two launches over groups
// of kLayScanThreads states: a group scans itself and leaves its total in group_totals[group]; then every state takes the
// groups in front of its own (a few dozen at most: a batch of 2^28 records has 2^16 block states, i.e. 256 groups).
constexpr uint32_t kLayScanThreads = 256;
__global__ void __launch_bounds__(kLayScanThreads) lay_scan_groups_kernel(LayState* __restrict__ states, uint32_t count, LayState* __restrict__ group_totals)
{
    __shared__ LayState sm[kLayScanThreads / 32];
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t j = blockIdx.x * kLayScanThreads + threadIdx.x;
    const LayState mine = j < count ? states[j] : lay_identity();
    const LayState inc = lay_warp_scan(mine);
    if (lane == 31) sm[warp] = inc;
    __syncthreads();
    LayState before = lay_identity();                               // the warps in front of this one
    for (unsigned w = 0; w < warp; ++w) before = lay_combine(before, sm[w]);
    LayState excl = lay_shfl_up(inc, 1);
    if (lane == 0) excl = lay_identity();
    const LayState pre = lay_combine(before, excl);
    if (j < count) states[j] = pre;
    if (threadIdx.x == kLayScanThreads - 1) group_totals[blockIdx.x] = lay_combine(pre, mine);
}
__global__ void __launch_bounds__(kLayScanThreads) lay_scan_finish_kernel(LayState* __restrict__ states, uint32_t count, const LayState* __restrict__ group_totals)
{
    __shared__ LayState front_sm;
    if (threadIdx.x == 0)
    {
        LayState f = lay_identity();
        for (uint32_t g = 0; g < blockIdx.x; ++g) f = lay_combine(f, group_totals[g]);
        front_sm = f;
        if (blockIdx.x == gridDim.x - 1) states[count] = lay_combine(f, group_totals[blockIdx.x]);
    }
    __syncthreads();
    const uint32_t j = blockIdx.x * kLayScanThreads + threadIdx.x;
    if (blockIdx.x && j < count) states[j] = lay_combine(front_sm, states[j]);
}

// first bin and first stream bytes of every chunk that holds records; entry [n_chunks] = bins and stream bytes of the whole batch
struct ChunkStart
{
    unsigned long long first_bin;
    unsigned long long off[4];
};

struct LayOut
{
    Placement pm;            // loc[4], binfo, tbase (place.cuh)
    OutStreams O;            // the streams: words shared by two K4 tiles are cleared here
    fsb_bin_descriptor* desc;
    ChunkStart* chunk_start; // [n_chunks + 1]
    uint32_t* nb_out;        // number of bins
};

__global__ void __launch_bounds__(kLayThreads) lay_apply_kernel(uint64_t n, uint32_t n_chunks, DeviceParams P, SortedView S, uint32_t uniform_len,
                                                                const LayState* __restrict__ tile_prefix, LayOut out)
{
    extern __shared__ uint4 lay_smem_raw[];
    __shared__ LayState sm[kLayThreads / 32];
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    LayWarpIn& w = reinterpret_cast<LayWarpIn*>(lay_smem_raw)[warp];
    // per array (loc[0..3], binfo) and thread: two 16-byte halves of a round, swapped in every other group of four
    // threads so that neither the threads' stores nor the warp's loads meet twice in a bank
    uint4* ost = reinterpret_cast<uint4*>(reinterpret_cast<LayWarpIn*>(lay_smem_raw) + kLayThreads / 32) + warp * (kLayOutWords / 4);
    const LayRun run = lay_run(n);
    const uint64_t wb = run.i0 - (uint64_t)lane * kLayPerThread;   // the warp's first record
    lay_stage(S, n, wb, w);
    uint32_t prev = lay_prev_key(S, w, run);
    const LayState mine = lay_run_state(P, w, prev, run, uniform_len);
    LayState total;
    const LayState excl = lay_combine(tile_prefix[blockIdx.x], lay_block_scan(mine, total, sm));
    LayCursor cur = lay_cursor(excl);
    const uint64_t tile = run.i0 / kPlaceTile;                      // the thread's K4 tile
    const uint32_t key_mask = (1u << P.key_bits) - 1u;
    const bool has_head = P.has_headers != 0;
    // the key behind the run
    const uint32_t key_after = lane < 31 ? w.keys[lane + 1][0] : (run.i0 + kLayPerThread < n ? S.skeys[run.i0 + kLayPerThread] : 0u);
    unsigned long long b0[4] = {0, 0, 0, 0};                        // first bit of the tile in every stream
    uint32_t base_bits_lo[4] = {0, 0, 0, 0};
    for (uint32_t rnd = 0; rnd < kLayPerThread / kLayRound; ++rnd)
    {
        uint32_t loc[4][kLayRound], binfo[kLayRound];
#pragma unroll
        for (uint32_t u = 0; u < kLayRound; ++u)
        {
            const uint32_t j = rnd * kLayRound + u;
#pragma unroll
            for (int k = 0; k < 4; ++k) loc[k][u] = 0;
            binfo[u] = 0;
            if (j < run.cnt)
            {
                const uint64_t i = run.i0 + j;
                const uint32_t key = w.keys[lane][j];
                // the key behind this record; the last record of the batch closes its bin whatever follows
                const uint32_t next = i + 1 >= n ? ~key : (j + 1 < kLayPerThread ? w.keys[lane][j + 1] : key_after);
                const LayRec r = lay_record(P, i == 0, key, prev, w.cards[lane][j], uniform_len);
                uint64_t at[4];
                lay_step(cur, r, at);
                if (r.chunk_start)
                {
                    ChunkStart cs;
                    cs.first_bin = cur.nb - 1u;
#pragma unroll
                    for (int k = 0; k < 4; ++k) cs.off[k] = cur.ls[k] >> 3;
                    out.chunk_start[key >> P.key_bits] = cs;
                }
                if (j == 0)
                {   // the tile starts at its first record, or at the first byte of the bin that record opens (bin header and all)
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                    {
                        const bool has = !(k == 3 && !has_head);
                        b0[k] = has ? (r.start ? cur.ls[k] : at[k]) : 0ull;
                        out.pm.tbase[4 * tile + k] = b0[k];
                        if (b0[k] & 31u) out.O.w[k][b0[k] >> 5] = 0;  // write_out ORs into the word it shares with the tile in front
                        base_bits_lo[k] = (uint32_t)(b0[k] & 127u);   // staging_bit: bits from the 16-byte group the tile starts in
                    }
                }
#pragma unroll
                for (int k = 0; k < 4; ++k)
                {
                    const bool has = !(k == 3 && !has_head);
                    loc[k][u] = has ? (uint32_t)(at[k] - b0[k]) + base_bits_lo[k] : 0u;
                }
                binfo[u] = (uniform_len & 0xFFu) | ((uniform_len & 0xFFu) << 8) | (r.start ? 0x10000u : 0u) | (r.nbin ? 0x20000u : 0u);
                if (next != key) out.desc[cur.nb - 1u] = lay_descriptor(cur, key & key_mask);   // last record of its bin
                prev = key;
            }
        }
        const uint32_t sw = (lane >> 2) & 1u;
#pragma unroll
        for (int k = 0; k < 4; ++k)
        {
            ost[(k * 32 + lane) * 2 + sw] = make_uint4(loc[k][0], loc[k][1], loc[k][2], loc[k][3]);
            ost[(k * 32 + lane) * 2 + (sw ^ 1u)] = make_uint4(loc[k][4], loc[k][5], loc[k][6], loc[k][7]);
        }
        ost[(4 * 32 + lane) * 2 + sw] = make_uint4(binfo[0], binfo[1], binfo[2], binfo[3]);
        ost[(4 * 32 + lane) * 2 + (sw ^ 1u)] = make_uint4(binfo[4], binfo[5], binfo[6], binfo[7]);
        __syncwarp();
        // the warp writes the round out: two lanes per thread, 32 contiguous bytes per thread and array
#pragma unroll
        for (uint32_t it = 0; it < 2; ++it)
        {
            const uint32_t t = it * 16 + (lane >> 1), h = lane & 1u;
            const uint64_t g = wb + (uint64_t)t * kLayPerThread + rnd * kLayRound + 4 * h;
            if (g < n)
            {
#pragma unroll
                for (int a = 0; a < 5; ++a)
                {
                    const uint4 q = ost[(a * 32 + t) * 2 + (h ^ ((t >> 2) & 1u))];
                    uint32_t* dst = a < 4 ? out.pm.loc[a] : out.pm.binfo;
                    if (g + 4 <= n) *reinterpret_cast<uint4*>(dst + g) = q;
                    else
                    {
                        dst[g] = q.x;
                        if (g + 1 < n) dst[g + 1] = q.y;
                        if (g + 2 < n) dst[g + 2] = q.z;
                    }
                }
            }
        }
        __syncwarp();
    }
    if (run.cnt && run.i0 + run.cnt == n)
    {   // end of the batch: the end of the last tile, the totals
        const uint64_t tiles = (n + kPlaceTile - 1) / kPlaceTile;
        ChunkStart cs;
        cs.first_bin = cur.nb;
#pragma unroll
        for (int k = 0; k < 4; ++k)
        {
            const bool has = !(k == 3 && !has_head);
            const unsigned long long e = has ? roundup8(cur.pos[k]) : 0ull;
            out.pm.tbase[4 * tiles + k] = e;
            if (e & 31u) out.O.w[k][e >> 5] = 0;
            cs.off[k] = roundup8(cur.pos[k]) >> 3;
        }
        out.chunk_start[n_chunks] = cs;
        *out.nb_out = cur.nb;
    }
}

// ChunkSummary (layout.cuh) of every chunk from the chunk starts: a chunk without records takes the start of the next chunk
// that has some (or the end of the batch), so its sizes come out as zero.
__global__ void __launch_bounds__(128) chunk_summary_fused_kernel(BatchView Bv, const ChunkStart* __restrict__ cs, const fsb_bin_descriptor* __restrict__ desc,
                                                                  ChunkSummary* __restrict__ out)
{
    const uint32_t c = blockIdx.x;                 // one block per chunk
    auto start_of = [&](uint32_t ch) { while (ch < Bv.n_chunks && Bv.chunk_first_rec[ch] == Bv.chunk_first_rec[ch + 1]) ++ch; return cs[ch]; };
    const ChunkStart s0 = start_of(c), s1 = start_of(c + 1);
    __shared__ unsigned long long raw[2];
    if (threadIdx.x == 0) { raw[0] = 0; raw[1] = 0; }
    __syncthreads();
    unsigned long long a = 0, h = 0;
    for (uint64_t b = s0.first_bin + threadIdx.x; b < s1.first_bin; b += blockDim.x) { a += desc[b].raw_dna_size; h += desc[b].raw_head_size; }
    atomicAdd(&raw[0], a); atomicAdd(&raw[1], h);
    __syncthreads();
    if (threadIdx.x == 0)
    {
        ChunkSummary s;
        s.first_bin = s0.first_bin; s.n_bins = s1.first_bin - s0.first_bin;
        for (int k = 0; k < 4; ++k) { s.off[k] = s0.off[k]; s.size[k] = s1.off[k] - s0.off[k]; }
        s.raw_dna = raw[0]; s.raw_head = raw[1];
        out[c] = s;
    }
}

// block states and group totals the layout of n records takes in `states`
inline uint64_t lay_states_count(uint64_t n)
{
    const uint64_t nlay = (n + kLayBlock - 1) / kLayBlock;
    return nlay + 1 + (nlay + kLayScanThreads - 1) / kLayScanThreads;
}

// The five launches of the layout of n >= 1 sorted records whose reads all have `uniform_len` bases, in B.n_chunks chunks.
inline cudaError_t lay_fused_launch(uint64_t n, const DeviceParams& P, const SortedView& S, uint32_t uniform_len, const BatchView& B, LayState* states,
                                    const LayOut& out, ChunkSummary* summary, cudaStream_t st)
{
    const unsigned nlay = (unsigned)((n + kLayBlock - 1) / kLayBlock);
    if (cudaError_t e = cudaFuncSetAttribute(lay_reduce_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLayReduceSmem)) return e;
    if (cudaError_t e = cudaFuncSetAttribute(lay_apply_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLayApplySmem)) return e;
    lay_reduce_kernel<<<nlay, kLayThreads, kLayReduceSmem, st>>>(n, P, S, uniform_len, states);
    const unsigned ngroups = (nlay + kLayScanThreads - 1) / kLayScanThreads;
    lay_scan_groups_kernel<<<ngroups, kLayScanThreads, 0, st>>>(states, nlay, states + nlay + 1);
    lay_scan_finish_kernel<<<ngroups, kLayScanThreads, 0, st>>>(states, nlay, states + nlay + 1);
    lay_apply_kernel<<<nlay, kLayThreads, kLayApplySmem, st>>>(n, B.n_chunks, P, S, uniform_len, states, out);
    chunk_summary_fused_kernel<<<B.n_chunks, 128, 0, st>>>(B, out.chunk_start, out.desc, summary);
    return cudaSuccess;
}

} // namespace fsb
