// tests/gpu_harness/sort_layout.cu -- TEST INFRASTRUCTURE: the scans, the radix sort of one sub-batch and the one-scan layout,
// each launched through the same host function run_sub uses (scan_sort.cuh, layout_fused.cuh), on arrays from the caller.
// tests/test_sort_layout_kernels.py builds it and compares every result with a plain reference.
//
// Every device array is allocated at exactly the size its data takes, so that a memory checker sees any access behind the
// end, and every output array is first filled with 0xA5 bytes, so that a store the kernels miss shows up as the pattern.
// Entry points return 0 or the first CUDA error.
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../fastore_b200/csrc/layout_fused.cuh"
#include "../../fastore_b200/csrc/scan_sort.cuh"

using namespace fsb;

namespace {

struct Dev
{
    std::vector<void*> ptrs;
    cudaError_t err = cudaSuccess;
    ~Dev() { for (void* p : ptrs) cudaFree(p); }
    template <typename T> T* alloc(size_t count)
    {
        if (count == 0 || err) return nullptr;
        void* p = nullptr;
        err = cudaMalloc(&p, count * sizeof(T));
        if (err) return nullptr;
        ptrs.push_back(p);
        err = cudaMemset(p, 0xA5, count * sizeof(T));
        return static_cast<T*>(p);
    }
    template <typename T> T* upload(const T* src, size_t count)
    {
        T* p = alloc<T>(count);
        if (p && !err) err = cudaMemcpy(p, src, count * sizeof(T), cudaMemcpyHostToDevice);
        return p;
    }
    template <typename T> void download(T* dst, const T* src, size_t count)
    {
        if (count && !err) err = cudaMemcpy(dst, src, count * sizeof(T), cudaMemcpyDeviceToHost);
    }
    int finish()
    {
        if (!err) err = cudaGetLastError();
        if (!err) err = cudaDeviceSynchronize();
        return (int)err;
    }
};

template <typename IN, typename OUT>
int scan1(const IN* in, uint64_t n, OUT* out)
{
    Dev d;
    const IN* din = d.upload(in, n);
    OUT* dout = d.alloc<OUT>(n + 1);
    OUT* tmp = d.alloc<OUT>(scan_num_tiles(n) + 1);
    if (d.err) return (int)d.err;
    exclusive_scan<IN, OUT>(din, n, dout, tmp, 0);
    if (int rc = d.finish()) return rc;
    d.download(out, dout, n + 1);
    return (int)d.err;
}

// in: four arrays of n, back to back; out: four arrays of n + 1
template <typename IN, typename OUT>
int scan4(const IN* in, uint64_t n, OUT* out)
{
    Dev d;
    Ptr4<const IN> din;
    Ptr4<OUT> dout;
    for (int k = 0; k < 4; ++k) { din.p[k] = d.upload(in + k * n, n); dout.p[k] = d.alloc<OUT>(n + 1); }
    OUT* tmp = d.alloc<OUT>(4 * (scan_num_tiles(n) + 1));
    if (d.err) return (int)d.err;
    exclusive_scan4<IN, OUT>(din, n, dout, tmp, 0);
    if (int rc = d.finish()) return rc;
    for (int k = 0; k < 4; ++k) d.download(out + k * (n + 1), dout.p[k], n + 1);
    return (int)d.err;
}

} // namespace

extern "C" int h_scan_u32_u32(const uint32_t* in, uint64_t n, uint32_t* out) { return scan1<uint32_t, uint32_t>(in, n, out); }
extern "C" int h_scan_u32_u64(const uint32_t* in, uint64_t n, uint64_t* out) { return scan1<uint32_t, uint64_t>(in, n, out); }
extern "C" int h_scan4_u32_u64(const uint32_t* in, uint64_t n, uint64_t* out) { return scan4<uint32_t, uint64_t>(in, n, out); }
extern "C" int h_scan4_u64_u64(const uint64_t* in, uint64_t n, uint64_t* out) { return scan4<uint64_t, uint64_t>(in, n, out); }

// The sort of one sub-batch of n records in n_chunks chunks (chunk_first: n_chunks + 1 record indices from 0 to n), every pass
// counted by sort_histogram, or by the scatter of the pass in front when fused_hist is set.  n_tiles receives the sort tiles.
extern "C" int h_sort(const uint32_t* keys, const uint64_t* cards, uint64_t n, const uint64_t* chunk_first, uint32_t n_chunks, int key_bits, int fused_hist,
                      uint32_t* keys_out, uint64_t* cards_out, uint64_t* n_tiles)
{
    std::vector<SortTile> tiles;
    std::vector<uint32_t> ctiles;
    sort_tiles_build(chunk_first, n_chunks, tiles, ctiles);
    *n_tiles = tiles.size();
    if (n == 0) return 0;
    int width[8];
    const int passes = sort_plan(key_bits, width);
    uint32_t radix = 0;
    for (int p = 0; p < passes; ++p) radix = std::max(radix, 1u << width[p]);
    const uint64_t ncounts = (uint64_t)radix * tiles.size();
    Dev d;
    uint32_t* k[2] = {d.upload(keys, n), d.alloc<uint32_t>(n)};
    unsigned long long* c[2] = {d.upload(reinterpret_cast<const unsigned long long*>(cards), n), d.alloc<unsigned long long>(n)};
    const SortTile* dt = d.upload(tiles.data(), tiles.size());
    uint32_t* counts = d.alloc<uint32_t>(ncounts);
    uint32_t* counts_scan = d.alloc<uint32_t>(ncounts + 1);
    uint32_t* tmp = d.alloc<uint32_t>(scan_num_tiles(ncounts) + 1);
    if (d.err) return (int)d.err;
    int cur = 0;
    uint64_t launches = 0;
    if (cudaError_t e = sort_passes(k, c, dt, (uint32_t)tiles.size(), key_bits, false, fused_hist != 0, counts, counts_scan, tmp, 0, cur, launches)) return (int)e;
    if (int rc = d.finish()) return rc;
    d.download(keys_out, k[cur], n);
    d.download(reinterpret_cast<unsigned long long*>(cards_out), c[cur], n);
    return (int)d.err;
}

// The layout of n >= 1 sorted records (keys, cards) whose reads all have uniform_len bases, in n_chunks chunks.  Outputs, each
// prefilled with 0xA5 bytes on the device:
//   loc          4 x n            binfo      n                     tbase     4 x (ceil(n / 32) + 1)
//   desc         the batch's bins (keys that differ from the one in front, counted here)
//   chunk_start  5 x (n_chunks + 1) words of 64 bits               nb        1
//   summary      n_chunks ChunkSummary (12 words of 64 bits each)
//   streams      stream_words[k] words of stream k, back to back
extern "C" int h_layout(const fsb_params* p, const uint32_t* keys, const uint64_t* cards, uint64_t n, uint32_t uniform_len, const uint64_t* chunk_first,
                        uint32_t n_chunks, const uint64_t* stream_words, uint32_t* loc, uint32_t* binfo, uint64_t* tbase, fsb_bin_descriptor* desc,
                        uint64_t* chunk_start, uint32_t* nb, uint64_t* summary, uint32_t* streams)
{
    if (n == 0) return (int)cudaErrorInvalidValue;
    const DeviceParams P = make_device_params(*p);
    uint64_t nbins = 0;
    for (uint64_t i = 0; i < n; ++i) nbins += (i == 0 || keys[i] != keys[i - 1]) ? 1 : 0;
    const uint64_t tiles = (n + kPlaceTile - 1) / kPlaceTile;
    Dev d;
    const SortedView S{d.upload(keys, n), d.upload(reinterpret_cast<const unsigned long long*>(cards), n)};
    BatchView B{};
    B.chunk_first_rec = d.upload(chunk_first, n_chunks + 1);
    B.n_chunks = n_chunks;
    B.n_records = n;
    LayOut out{};
    for (int k = 0; k < 4; ++k) { out.pm.loc[k] = d.alloc<uint32_t>(n); out.O.w[k] = d.alloc<uint32_t>(stream_words[k]); }
    out.pm.binfo = d.alloc<uint32_t>(n);
    out.pm.tbase = d.alloc<unsigned long long>(4 * (tiles + 1));
    out.desc = d.alloc<fsb_bin_descriptor>(nbins);
    out.chunk_start = d.alloc<ChunkStart>(n_chunks + 1);
    out.nb_out = d.alloc<uint32_t>(1);
    ChunkSummary* dsum = d.alloc<ChunkSummary>(n_chunks);
    LayState* states = d.alloc<LayState>(lay_states_count(n));
    if (d.err) return (int)d.err;
    if (cudaError_t e = lay_fused_launch(n, P, S, uniform_len, B, states, out, dsum, 0)) return (int)e;
    if (int rc = d.finish()) return rc;
    for (int k = 0; k < 4; ++k) d.download(loc + k * n, out.pm.loc[k], n);
    d.download(binfo, out.pm.binfo, n);
    d.download(reinterpret_cast<unsigned long long*>(tbase), out.pm.tbase, 4 * (tiles + 1));
    d.download(desc, out.desc, nbins);
    d.download(reinterpret_cast<ChunkStart*>(chunk_start), out.chunk_start, n_chunks + 1);
    d.download(nb, out.nb_out, 1);
    d.download(reinterpret_cast<ChunkSummary*>(summary), dsum, n_chunks);
    uint64_t off = 0;
    for (int k = 0; k < 4; ++k) { d.download(streams + off, out.O.w[k], stream_words[k]); off += stream_words[k]; }
    return (int)d.err;
}
