// scan_sort.cuh -- device-wide exclusive scan and stable LSD radix sort, hand-written for sm_100a.
//
// These are the "histogram, prefix-sum and scatter" pieces of the path: the reference builds
// std::map<uint32, FastqRecordsPtrBin> by push_back in parse order (FastqCategorizer.cpp:247,357),
// i.e. a *stable* grouping of records by signature.  On the device that is a stable sort of
// (key = chunk:signature, value = record index): per-block digit histograms in shared memory,
// a device-wide exclusive scan over the digit-major count table, and a rank-and-scatter pass that
// keeps equal keys in input order.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace fsb {

constexpr int kScanThreads = 256;
constexpr int kScanItems = 16;                       // items per thread
constexpr int kScanTile = kScanThreads * kScanItems; // 4096 items per block

// ---- block-wide exclusive scan of one value per thread (256 threads) ----------------------------
template <typename T>
__device__ __forceinline__ T warp_inclusive_scan(T v)
{
    const unsigned lane = threadIdx.x & 31;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1)
    {
        T o = __shfl_up_sync(0xFFFFFFFFu, v, d);
        if (lane >= (unsigned)d) v += o;
    }
    return v;
}

// returns the exclusive prefix of `v` over the block; `total` receives the block sum (all threads)
template <typename T, int THREADS>
__device__ __forceinline__ T block_exclusive_scan(T v, T& total, T* smem /* THREADS/32 + 1 entries */)
{
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const T inc = warp_inclusive_scan(v);
    if (lane == 31) smem[warp] = inc;
    __syncthreads();
    if (warp == 0)
    {
        T w = (lane < THREADS / 32) ? smem[lane] : T(0);
        T winc = warp_inclusive_scan(w);
        if (lane < THREADS / 32) smem[lane] = winc - w;     // exclusive warp offsets
        if (lane == THREADS / 32 - 1) smem[THREADS / 32] = winc;
    }
    __syncthreads();
    const T res = smem[warp] + inc - v;
    total = smem[THREADS / 32];
    __syncthreads();
    return res;
}

// ---- three-phase device-wide exclusive scan ------------------------------------------------------
// phase A: per-tile sums; phase B: one block scans the tile sums; phase C: per-tile scan + offset.
// IN may be narrower than OUT (u32 counts -> u64 bit offsets).  out[n] (one past the end) receives
// the grand total, so callers can read segment ends without a special case.
template <typename IN, typename OUT>
__global__ void __launch_bounds__(kScanThreads) scan_tile_sums(const IN* __restrict__ in, uint64_t n, OUT* __restrict__ tile_sums)
{
    __shared__ OUT sm[kScanThreads / 32 + 1];
    const uint64_t base = (uint64_t)blockIdx.x * kScanTile;
    OUT s = 0;
#pragma unroll
    for (int i = 0; i < kScanItems; ++i)
    {
        const uint64_t idx = base + (uint64_t)i * kScanThreads + threadIdx.x;
        if (idx < n) s += (OUT)in[idx];
    }
    OUT total;
    block_exclusive_scan<OUT, kScanThreads>(s, total, sm);
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

template <typename OUT>
__global__ void __launch_bounds__(1024) scan_small(OUT* __restrict__ data, uint64_t n)
{
    // single block, in-place exclusive scan of `n` values (tile sums); data[n] <- total
    __shared__ OUT sm[1024 / 32 + 1];
    OUT carry = 0;
    for (uint64_t base = 0; base < n; base += 1024)
    {
        const uint64_t idx = base + threadIdx.x;
        const OUT v = idx < n ? data[idx] : OUT(0);
        OUT total;
        const OUT ex = block_exclusive_scan<OUT, 1024>(v, total, sm);
        if (idx < n) data[idx] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) data[n] = carry;
}

template <typename T> __device__ __forceinline__ void load_items(const T* __restrict__ src, uint64_t base, uint64_t n, T (&v)[kScanItems]);
template <typename T> __device__ __forceinline__ void store_items(T* __restrict__ dst, uint64_t base, uint64_t n, const T (&v)[kScanItems]);

template <typename IN, typename OUT>
__global__ void __launch_bounds__(kScanThreads) scan_apply(const IN* __restrict__ in, uint64_t n, const OUT* __restrict__ tile_offsets,
                                                            OUT* __restrict__ out)
{
    __shared__ OUT sm[kScanThreads / 32 + 1];
    const uint64_t base = (uint64_t)blockIdx.x * kScanTile + (uint64_t)threadIdx.x * kScanItems;
    IN v[kScanItems];
    load_items<IN>(in, base, n, v);
    OUT s = 0;
#pragma unroll
    for (int i = 0; i < kScanItems; ++i) s += (OUT)v[i];
    OUT total;
    OUT ex = block_exclusive_scan<OUT, kScanThreads>(s, total, sm) + tile_offsets[blockIdx.x];
    OUT o[kScanItems];
#pragma unroll
    for (int i = 0; i < kScanItems; ++i) { o[i] = ex; ex += (OUT)v[i]; }
    store_items<OUT>(out, base, n, o);
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == kScanThreads - 1) out[n] = tile_offsets[gridDim.x];
}

inline uint64_t scan_num_tiles(uint64_t n) { return (n + kScanTile - 1) / kScanTile; }

// ---- the same scan over four arrays of equal length in one set of launches (blockIdx.y = array) ----------
template <typename T> struct Ptr4 { T* p[4]; };
template <typename T> __device__ __forceinline__ T* pick4(const Ptr4<T>& a, unsigned k) { return k == 0 ? a.p[0] : (k == 1 ? a.p[1] : (k == 2 ? a.p[2] : a.p[3])); }

template <typename IN, typename OUT>
__global__ void __launch_bounds__(kScanThreads) scan4_tile_sums(Ptr4<const IN> in, uint64_t n, OUT* __restrict__ tile_sums, uint64_t tiles_stride)
{
    __shared__ OUT sm[kScanThreads / 32 + 1];
    const IN* __restrict__ src = pick4(in, blockIdx.y);
    const uint64_t base = (uint64_t)blockIdx.x * kScanTile;
    OUT s = 0;
#pragma unroll
    for (int i = 0; i < kScanItems; ++i)
    {
        const uint64_t idx = base + (uint64_t)i * kScanThreads + threadIdx.x;
        if (idx < n) s += (OUT)src[idx];
    }
    OUT total;
    block_exclusive_scan<OUT, kScanThreads>(s, total, sm);
    if (threadIdx.x == 0) tile_sums[blockIdx.y * tiles_stride + blockIdx.x] = total;
}

template <typename OUT>
__global__ void __launch_bounds__(1024) scan4_small(OUT* __restrict__ data, uint64_t n, uint64_t tiles_stride)
{
    __shared__ OUT sm[1024 / 32 + 1];
    OUT* d = data + blockIdx.x * tiles_stride;                   // one block per array
    OUT carry = 0;
    for (uint64_t base = 0; base < n; base += 1024)
    {
        const uint64_t idx = base + threadIdx.x;
        const OUT v = idx < n ? d[idx] : OUT(0);
        OUT total;
        const OUT ex = block_exclusive_scan<OUT, 1024>(v, total, sm);
        if (idx < n) d[idx] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) d[n] = carry;
}

// a thread's kScanItems consecutive items, with 16-byte accesses where the tile is complete and the arrays are aligned
template <typename T>
__device__ __forceinline__ void load_items(const T* __restrict__ src, uint64_t base, uint64_t n, T (&v)[kScanItems])
{
    constexpr int PER = 16 / (int)sizeof(T);
    if (base + kScanItems <= n && (reinterpret_cast<uintptr_t>(src + base) & 15u) == 0)
    {
        const uint4* p = reinterpret_cast<const uint4*>(src + base);
#pragma unroll
        for (int i = 0; i < kScanItems / PER; ++i)
        {
            const uint4 q = p[i];
            if constexpr (sizeof(T) == 4) { v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w; }
            else { v[2 * i] = ((T)q.y << 32) | q.x; v[2 * i + 1] = ((T)q.w << 32) | q.z; }
        }
    }
    else
    {
#pragma unroll
        for (int i = 0; i < kScanItems; ++i) v[i] = base + i < n ? src[base + i] : T(0);
    }
}
template <typename T>
__device__ __forceinline__ void store_items(T* __restrict__ dst, uint64_t base, uint64_t n, const T (&v)[kScanItems])
{
    constexpr int PER = 16 / (int)sizeof(T);
    if (base + kScanItems <= n && (reinterpret_cast<uintptr_t>(dst + base) & 15u) == 0)
    {
        uint4* p = reinterpret_cast<uint4*>(dst + base);
#pragma unroll
        for (int i = 0; i < kScanItems / PER; ++i)
        {
            uint4 q;
            if constexpr (sizeof(T) == 4) { q.x = v[4 * i]; q.y = v[4 * i + 1]; q.z = v[4 * i + 2]; q.w = v[4 * i + 3]; }
            else { q.x = (uint32_t)v[2 * i]; q.y = (uint32_t)(v[2 * i] >> 32); q.z = (uint32_t)v[2 * i + 1]; q.w = (uint32_t)(v[2 * i + 1] >> 32); }
            p[i] = q;
        }
    }
    else
    {
#pragma unroll
        for (int i = 0; i < kScanItems; ++i) if (base + i < n) dst[base + i] = v[i];
    }
}

template <typename IN, typename OUT>
__global__ void __launch_bounds__(kScanThreads) scan4_apply(Ptr4<const IN> in, uint64_t n, const OUT* __restrict__ tile_offsets, uint64_t tiles_stride,
                                                             Ptr4<OUT> out)
{
    __shared__ OUT sm[kScanThreads / 32 + 1];
    const IN* __restrict__ src = pick4(in, blockIdx.y);
    OUT* __restrict__ dst = pick4(out, blockIdx.y);
    const OUT* toff = tile_offsets + blockIdx.y * tiles_stride;
    const uint64_t base = (uint64_t)blockIdx.x * kScanTile + (uint64_t)threadIdx.x * kScanItems;
    IN v[kScanItems];
    load_items<IN>(src, base, n, v);
    OUT s = 0;
#pragma unroll
    for (int i = 0; i < kScanItems; ++i) s += (OUT)v[i];
    OUT total;
    OUT ex = block_exclusive_scan<OUT, kScanThreads>(s, total, sm) + toff[blockIdx.x];
    OUT o[kScanItems];
#pragma unroll
    for (int i = 0; i < kScanItems; ++i) { o[i] = ex; ex += (OUT)v[i]; }
    store_items<OUT>(dst, base, n, o);
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == kScanThreads - 1) dst[n] = toff[gridDim.x];
}

// out[k] must hold n + 1 entries; tmp must hold 4 * (scan_num_tiles(n) + 1) entries.  3 launches.
template <typename IN, typename OUT>
inline int exclusive_scan4(Ptr4<const IN> in, uint64_t n, Ptr4<OUT> out, OUT* tmp, cudaStream_t st)
{
    if (n == 0)
    {
        for (int k = 0; k < 4; ++k) cudaMemsetAsync(out.p[k], 0, sizeof(OUT), st);
        return 0;
    }
    const uint64_t tiles = scan_num_tiles(n), stride = tiles + 1;
    scan4_tile_sums<IN, OUT><<<dim3((unsigned)tiles, 4), kScanThreads, 0, st>>>(in, n, tmp, stride);
    scan4_small<OUT><<<4, 1024, 0, st>>>(tmp, tiles, stride);
    scan4_apply<IN, OUT><<<dim3((unsigned)tiles, 4), kScanThreads, 0, st>>>(in, n, tmp, stride, out);
    return 3;
}

// out must hold n + 1 entries; tmp must hold scan_num_tiles(n) + 1 entries.  3 launches.
template <typename IN, typename OUT>
inline int exclusive_scan(const IN* in, uint64_t n, OUT* out, OUT* tmp, cudaStream_t st)
{
    if (n == 0)
    {
        cudaMemsetAsync(out, 0, sizeof(OUT), st);
        return 0;
    }
    const uint64_t tiles = scan_num_tiles(n);
    scan_tile_sums<IN, OUT><<<(unsigned)tiles, kScanThreads, 0, st>>>(in, n, tmp);
    scan_small<OUT><<<1, 1024, 0, st>>>(tmp, tiles);
    scan_apply<IN, OUT><<<(unsigned)tiles, kScanThreads, 0, st>>>(in, n, tmp, out);
    return 3;
}

// ---- stable LSD radix sort over chunk segments, digits of up to 9 bits -----------------------------------
// The keys are chunk : signature, and the records of a batch already arrive chunk by chunk.  Only the
// signature needs sorting: every sort tile lies inside one chunk (the host lays the tiles out, SortTile),
// and the count table is chunk-major -- [chunk][digit][tile of the chunk] -- so that one exclusive scan over
// the whole table yields global destinations in (chunk, digit, tile) order.  The chunk bits never enter a
// digit: 2k + 1 signature bits take two passes for k = 8 (8 + 9 bits) where chunk : signature took three.
// (The first pass takes the bits that are left over: the low signature bits are uniform, and a narrow first
// digit keeps the runs a block writes per digit long; the later digits are skewed anyway.)
constexpr int kSortThreads = 256;
constexpr int kSortStrips = 16;                          // 32-key strips per warp
constexpr int kSortTile = kSortThreads * kSortStrips;    // up to 4096 keys per block
constexpr int kMaxRadix = 512;

struct SortTile
{
    uint32_t first;          // first key of the tile (index inside the sub-batch)
    uint32_t count;          // keys in the tile (1 .. kSortTile)
    uint32_t cblk;           // tiles of all earlier chunks of the sub-batch
    uint32_t blk, nblk;      // index of the tile inside its chunk, tiles of that chunk
    uint32_t pad[3];
};
__device__ __forceinline__ uint64_t sort_count_index(const SortTile& t, uint32_t radix, uint32_t digit)
{
    return (uint64_t)radix * t.cblk + (uint64_t)digit * t.nblk + t.blk;
}

// A tile's keys or cards as 16-byte vectors: [0, head) and [head + nvec * PER, count) are read one by one, the
// vectors in between start at a 16-byte boundary (the tiles of a chunk start wherever the chunk's records do).
template <typename T>
struct TileSplit
{
    static constexpr uint32_t PER = 16u / sizeof(T);
    uint32_t head, nvec;
    __device__ __forceinline__ TileSplit(const T* src, uint32_t count)
    {
        head = min(count, (uint32_t)((16u - (reinterpret_cast<uintptr_t>(src) & 15u)) & 15u) / (uint32_t)sizeof(T));
        nvec = (count - head) / PER;
    }
};

constexpr int kSortWarps = kSortThreads / 32;

__global__ void __launch_bounds__(kSortThreads) sort_histogram(const uint32_t* __restrict__ keys, const SortTile* __restrict__ tiles, int shift, uint32_t mask,
                                                                uint32_t radix, uint32_t* __restrict__ counts)
{
    __shared__ uint32_t hist[kSortWarps][kMaxRadix];                // one sub-histogram per warp: 16 KB
    const unsigned warp = threadIdx.x >> 5;
    for (uint32_t d = threadIdx.x; d < radix; d += kSortThreads)
#pragma unroll
        for (int w = 0; w < kSortWarps; ++w) hist[w][d] = 0;
    __syncthreads();
    const SortTile t = tiles[blockIdx.x];
    const uint32_t* src = keys + t.first;
    const TileSplit<uint32_t> sp(src, t.count);
    uint32_t* h = hist[warp];
    const uint4* v = reinterpret_cast<const uint4*>(src + sp.head);
#pragma unroll 4
    for (uint32_t i = threadIdx.x; i < sp.nvec; i += kSortThreads)
    {
        const uint4 q = v[i];
        atomicAdd(&h[(q.x >> shift) & mask], 1u);
        atomicAdd(&h[(q.y >> shift) & mask], 1u);
        atomicAdd(&h[(q.z >> shift) & mask], 1u);
        atomicAdd(&h[(q.w >> shift) & mask], 1u);
    }
    if (threadIdx.x < sp.head) atomicAdd(&h[(src[threadIdx.x] >> shift) & mask], 1u);
    const uint32_t tail = sp.head + sp.nvec * 4u + threadIdx.x;
    if (tail < t.count) atomicAdd(&h[(src[tail] >> shift) & mask], 1u);
    __syncthreads();
    for (uint32_t d = threadIdx.x; d < radix; d += kSortThreads)
    {
        uint32_t c = 0;
#pragma unroll
        for (int w = 0; w < kSortWarps; ++w) c += hist[w][d];
        counts[sort_count_index(t, radix, d)] = c;
    }
}

// Copies a tile's keys or cards into shared memory with 16-byte loads.  `buf` has PER - 1 spare entries: the tile starts at
// buf + (its misalignment), so that the vectors land on 16-byte boundaries in shared memory too.  Returns the tile's start.
template <typename T>
__device__ __forceinline__ T* sort_stage(const T* __restrict__ src, uint32_t count, T* buf)
{
    const TileSplit<T> sp(src, count);
    T* dst = buf + (sp.head ? TileSplit<T>::PER - sp.head : 0u);
    const uint4* v = reinterpret_cast<const uint4*>(src + sp.head);
    uint4* o = reinterpret_cast<uint4*>(dst + sp.head);
    for (uint32_t i = threadIdx.x; i < sp.nvec; i += kSortThreads) o[i] = v[i];
    if (threadIdx.x < sp.head) dst[threadIdx.x] = src[threadIdx.x];
    const uint32_t tail = sp.head + sp.nvec * TileSplit<T>::PER + threadIdx.x;
    if (tail < count) dst[tail] = src[tail];
    return dst;
}

// Shared memory of sort_scatter (dynamic: more than the 48 KB a static array may take).
struct SortScatterSmem
{
    unsigned long long cards[kSortTile + 2];   // the tile's cards, then the same cards in (digit, rank) order
    uint32_t keys[kSortTile + 4];              // the same for the keys
    uint32_t warp_hist[kSortWarps][kMaxRadix]; // per warp and digit: keys, then the tile-local slot of the warp's first key
    uint32_t gbase[kMaxRadix];                 // per digit: global destination of tile-local slot 0
    uint32_t scan[kSortWarps + 1];
};

// offsets: exclusive scan of counts (same layout).  The 64-bit values are the records' cards (core.cuh).
// The tile is ranked in shared memory (stable: warp-major, input order inside a warp's strips) and reordered there into
// (digit, rank) order, so that consecutive threads store consecutive keys of one digit's run.
// next_counts (may be null): the count table of the NEXT pass, zeroed by the caller -- a key's destination tells the tile it
// will sit in, so the next pass needs no histogram kernel of its own (one L2 reduction per key, spread over tiles x digits counters).
__global__ void __launch_bounds__(kSortThreads) sort_scatter(const uint32_t* __restrict__ keys_in, const unsigned long long* __restrict__ vals_in,
                                                              const SortTile* __restrict__ tiles, int shift, uint32_t mask, uint32_t radix,
                                                              const uint32_t* __restrict__ offsets, uint32_t* __restrict__ keys_out,
                                                              unsigned long long* __restrict__ vals_out,
                                                              uint32_t* __restrict__ next_counts, int next_shift, uint32_t next_mask, uint32_t next_radix)
{
    extern __shared__ uint4 sort_smem_raw[];
    SortScatterSmem& sm = *reinterpret_cast<SortScatterSmem*>(sort_smem_raw);
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t d = threadIdx.x; d < radix; d += kSortThreads)
#pragma unroll
        for (int w = 0; w < kSortWarps; ++w) sm.warp_hist[w][d] = 0;
    const SortTile t = tiles[blockIdx.x];
    uint32_t* keys_s = sort_stage(keys_in + t.first, t.count, sm.keys);
    unsigned long long* cards_s = sort_stage(vals_in + t.first, t.count, sm.cards);
    __syncthreads();

    // each warp owns a contiguous run of kSortStrips * 32 keys (keeps the order stable)
    const uint32_t wlocal = warp * (kSortStrips * 32);
    uint32_t key[kSortStrips];
    uint32_t rank[kSortStrips];
#pragma unroll
    for (int i = 0; i < kSortStrips; ++i)
    {
        const uint32_t local = wlocal + (uint32_t)i * 32 + lane;
        const bool in = local < t.count;
        key[i] = in ? keys_s[local] : 0xFFFFFFFFu;
        const uint32_t d = in ? ((key[i] >> shift) & mask) : 0xFFFFFFFFu;
        const unsigned peers = __match_any_sync(0xFFFFFFFFu, d);
        const uint32_t before = in ? sm.warp_hist[warp][d] : 0;
        rank[i] = before + __popc(peers & ((1u << lane) - 1));
        __syncwarp();
        if (in && (__ffs(peers) - 1) == (int)lane) sm.warp_hist[warp][d] = before + __popc(peers);
        __syncwarp();
    }
    __syncthreads();
    // per digit (two per thread, radix <= 2 * kSortThreads): tile-local start of its run, global base, per-warp slots
    uint32_t c2[2] = {0, 0};
#pragma unroll
    for (int e = 0; e < 2; ++e)
    {
        const uint32_t d = 2u * threadIdx.x + (uint32_t)e;
        if (d < radix)
#pragma unroll
            for (int w = 0; w < kSortWarps; ++w) c2[e] += sm.warp_hist[w][d];
    }
    uint32_t total;
    uint32_t run = block_exclusive_scan<uint32_t, kSortThreads>(c2[0] + c2[1], total, sm.scan);
#pragma unroll
    for (int e = 0; e < 2; ++e)
    {
        const uint32_t d = 2u * threadIdx.x + (uint32_t)e;
        if (d < radix)
        {
            sm.gbase[d] = offsets[sort_count_index(t, radix, d)] - run;
#pragma unroll
            for (int w = 0; w < kSortWarps; ++w)
            {
                const uint32_t c = sm.warp_hist[w][d];
                sm.warp_hist[w][d] = run;
                run += c;
            }
        }
    }
    __syncthreads();
    // reorder: the keys (read into registers above), then the cards (read before the barrier, written after it)
    unsigned long long card[kSortStrips];
#pragma unroll
    for (int i = 0; i < kSortStrips; ++i)
    {
        const uint32_t local = wlocal + (uint32_t)i * 32 + lane;
        if (local < t.count)
        {
            rank[i] += sm.warp_hist[warp][(key[i] >> shift) & mask];
            sm.keys[rank[i]] = key[i];
        }
        card[i] = local < t.count ? cards_s[local] : 0ull;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < kSortStrips; ++i)
        if (wlocal + (uint32_t)i * 32 + lane < t.count) sm.cards[rank[i]] = card[i];
    __syncthreads();
    // the chunk's keys stay inside the chunk: destination - first key of the chunk = place inside the chunk
    const uint32_t chunk_first = t.first - t.blk * (uint32_t)kSortTile;
    for (uint32_t s = threadIdx.x; s < t.count; s += kSortThreads)
    {
        const uint32_t k = sm.keys[s];
        const uint32_t dst = sm.gbase[(k >> shift) & mask] + s;
        keys_out[dst] = k;
        vals_out[dst] = sm.cards[s];
        if (next_counts)
        {
            const uint32_t nt = (dst - chunk_first) / (uint32_t)kSortTile;
            atomicAdd(&next_counts[(uint64_t)next_radix * t.cblk + (uint64_t)((k >> next_shift) & next_mask) * t.nblk + nt], 1u);
        }
    }
}

// digit widths of the passes, least significant first: as few passes of at most 9 bits as cover `bits`, evenly wide, the narrower ones first
inline int sort_plan(int bits, int (&width)[8])
{
    const int passes = (bits + 8) / 9;
    const int base = bits / passes, rem = bits % passes;
    for (int p = 0; p < passes; ++p) width[p] = base + (p >= passes - rem ? 1 : 0);
    return passes;
}

} // namespace fsb
