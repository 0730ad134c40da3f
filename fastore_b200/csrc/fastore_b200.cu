// fastore_b200.cu -- the C ABI of include/fastore_b200.h: context, staging, the kernel pipeline
// (K1 ingest -> stable radix sort -> layout scans -> K4 place) and result fetch.
//
// Host-side structure mirrors what the reference does per chunk in its -t1 loop
// (BinModule.cpp:124-167): Categorize(reads, bins); PackToBins(bins, block).  Several chunks may be
// processed by one pass of the pipeline ("batch"): bins are keyed by (chunk, signature), so every
// chunk still yields exactly its own BinaryBinBlock, byte for byte.
//
// fsb_run can split the staged batch into sub-batches of whole chunks that go through the pipeline on
// two streams ("lanes", each with its own intermediates): K1 of one sub-batch is bound by the integer
// pipe, sort / layout / K4 of the other by latency and HBM, so they share the SMs well.
//
// fsb_bin_chunks (host buffers in, host blocks out) cuts its chunk list into sub-batches and runs
// them as a three-stage pipeline over two sets of device buffers: host->device copy of sub-batch
// g+1, kernels of g and device->host copy of g-1 overlap on three streams, the way the reference's
// reader thread, encoder threads and writer overlap (BinModule.cpp:58-90).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <mutex>
#include <new>
#include <string>
#include <unordered_map>
#include <vector>

#include <sys/mman.h>

#include <cuda_runtime.h>

#include "../../include/fastore_b200.h"
#include "scan_sort.cuh"
#include "stage.cuh"
#include "ingest.cuh"
#include "layout.cuh"
#include "place.cuh"
#include "layout_fused.cuh"
#include "parse.cuh"
#include "rebin_sig.cuh"

using namespace fsb;

namespace {

thread_local std::string g_create_error;

struct DevBuf
{
    void* p = nullptr;
    size_t cap = 0;
    // `zero_on`: clear the buffer on that stream when it is (re)allocated -- for buffers whose padding may be over-read by
    // aligned vector loads (the clear is ordered before whatever the caller enqueues on the stream next)
    cudaError_t ensure(size_t bytes, const cudaStream_t* zero_on = nullptr)
    {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        const size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) { cap = want; if (zero_on) e = cudaMemsetAsync(p, 0, want, *zero_on); }
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// Page-locked host memory.  On the B200 hosts cudaHostAlloc pins at 2.4 GB/s under the driver's lock, while pages the process
// has already touched are registered at 45 GB/s and touching them costs 7 GB/s (profiles/r02n_pinning.json): a one-shot tool
// that pins a few GB feels the difference.  So large buffers are anonymous mappings (transparent huge pages where the kernel
// grants them), touched here and then registered; small ones and FSB_PIN=alloc take cudaHostAlloc.
struct PinRegistry
{
    std::mutex mu;
    std::unordered_map<void*, size_t> mapped;        // registered mappings: pointer -> mapped bytes
};
PinRegistry& pin_registry() { static PinRegistry* r = new PinRegistry; return *r; }      // (never destroyed: frees may come late in exit)

void* pinned_alloc(size_t bytes)
{
    static const bool use_register = []() { const char* e = std::getenv("FSB_PIN"); return !(e && std::strcmp(e, "alloc") == 0); }();
    constexpr size_t kHuge = 2u << 20;
    if (use_register && bytes >= (8u << 20))
    {
        const size_t len = (bytes + kHuge - 1) / kHuge * kHuge;
        void* m = mmap(nullptr, len + kHuge, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
        if (m != MAP_FAILED)
        {
            // a 2 MB aligned window inside the mapping; what lies in front of it and behind it is given back
            uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(m) + kHuge - 1) / kHuge * kHuge);
            if (base != m) munmap(m, (size_t)(base - reinterpret_cast<uint8_t*>(m)));
            const size_t tail = (size_t)(reinterpret_cast<uint8_t*>(m) + len + kHuge - (base + len));
            if (tail) munmap(base + len, tail);
            madvise(base, len, MADV_HUGEPAGE);
            for (size_t o = 0; o < len; o += 4096) base[o] = 0;                           // fault the pages in outside the driver
            if (cudaHostRegister(base, len, cudaHostRegisterPortable | cudaHostRegisterMapped) == cudaSuccess)
            {
                PinRegistry& r = pin_registry();
                std::lock_guard<std::mutex> l(r.mu);
                r.mapped[base] = len;
                return base;
            }
            cudaGetLastError();
            munmap(base, len);
        }
    }
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable | cudaHostAllocMapped) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void pinned_free(void* p)
{
    if (!p) return;
    size_t len = 0;
    {
        PinRegistry& r = pin_registry();
        std::lock_guard<std::mutex> l(r.mu);
        auto it = r.mapped.find(p);
        if (it != r.mapped.end()) { len = it->second; r.mapped.erase(it); }
    }
    if (len) { cudaHostUnregister(p); munmap(p, len); }
    else cudaFreeHost(p);
}

struct PinBuf
{
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        pinned_free(p);
        p = nullptr; cap = 0;
        const size_t want = bytes + bytes / 8 + 256;
        p = pinned_alloc(want);
        if (!p) return cudaErrorMemoryAllocation;
        cap = want;
        return cudaSuccess;
    }
    void release() { pinned_free(p); p = nullptr; cap = 0; }
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// FSB_TRACE=1: the host-side timeline of fsb_bin_chunks on stderr (ms since the call began)
struct CallTrace
{
    bool on;
    std::chrono::steady_clock::time_point t0;
    CallTrace() : on(std::getenv("FSB_TRACE") != nullptr), t0(std::chrono::steady_clock::now()) {}
    void mark(const char* what, uint32_t g) const
    {
        if (!on) return;
        const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        std::fprintf(stderr, "[fsb %9.3f ms] %-28s sub-batch %u\n", ms, what, g);
    }
};

// Small tables and results move between page-locked host memory and the device through a kernel, not through cudaMemcpyAsync
// (mapped memory: under unified addressing the device reads and writes the host buffer directly).  The copy engines work
// through their transfers in the order of submission: a 100-byte copy submitted while the next sub-batch's 540 MB of text are
// on their way waits 10 ms for them, a small result behind a sub-batch's 280 MB of output 5 ms -- and the host side of the
// pipeline waits for exactly these small things (check statistics, line counts of the device-side parse).
__global__ void words_copy_kernel(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst, uint32_t n_words)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += gridDim.x * blockDim.x) dst[i] = src[i];
}
__global__ void words_fill_kernel(uint32_t* __restrict__ dst, uint32_t value, uint32_t n_words)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += gridDim.x * blockDim.x) dst[i] = value;
}
inline unsigned words_grid(size_t n_words) { return (unsigned)std::max<size_t>(1, std::min<size_t>(64, (n_words + 1023) / 1024)); }
inline cudaError_t small_to_host(void* host_pinned, const void* dev, size_t bytes, cudaStream_t st)
{
    if (bytes == 0) return cudaSuccess;
    void* mapped = nullptr;
    cudaError_t e = cudaHostGetDevicePointer(&mapped, host_pinned, 0);
    if (e != cudaSuccess) return e;
    const size_t n = (bytes + 3) / 4;
    words_copy_kernel<<<words_grid(n), 256, 0, st>>>(reinterpret_cast<const uint32_t*>(dev), reinterpret_cast<uint32_t*>(mapped), (uint32_t)n);
    return cudaGetLastError();
}
inline cudaError_t small_fill(void* dev, uint32_t value, size_t bytes, cudaStream_t st)
{
    if (bytes == 0) return cudaSuccess;
    const size_t n = (bytes + 3) / 4;
    words_fill_kernel<<<words_grid(n), 256, 0, st>>>(reinterpret_cast<uint32_t*>(dev), value, (uint32_t)n);
    return cudaGetLastError();
}

constexpr size_t kTextPad = 64;           // slack around every chunk text: aligned vector loads may over-read
constexpr uint32_t kMaxChunksPerBatch = 256;
constexpr int kMaxPendingProfiles = 256;

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

} // namespace

// A run of whole chunks of a staged batch that goes through the kernel pipeline on its own (fsb_run may split a batch
// into several to overlap them on two streams).  Record, bin and output offsets are relative to the batch.
struct Sub
{
    uint32_t c0 = 0, c1 = 0;                     // chunks [c0, c1)
    uint64_t r0 = 0, r1 = 0;                     // records [r0, r1)
    uint64_t nb_max = 0, bin_off = 0;            // bound of the number of bins; first entry in the batch's descriptor array
    uint64_t tile_off = 0, n_tiles = 0;          // its sort tiles in the batch's tile table
    uint64_t ctile_off = 0;                      // its table "sort tiles in front of every chunk" (chunks + 1 entries)
    size_t out_off[4] = {0, 0, 0, 0}, out_cap[4] = {0, 0, 0, 0};   // its region of the batch's output streams (bytes, 64-byte aligned)
    size_t meta_first = 0;                       // index of its relative first-record table in the device chunk tables
};

// One staged group of chunks: its inputs and its results on the device.
struct Batch
{
    bool staged = false, ran = false;
    uint32_t n_chunks = 0;
    uint32_t chunk0 = 0;                         // index of the first chunk in the caller's list: rejections name the caller's chunk
    uint64_t n_records = 0;
    std::vector<uint64_t> chunk_first_rec;       // n_chunks + 1
    std::vector<uint64_t> chunk_text_base[2], chunk_text_size[2];
    cudaStream_t st_check = nullptr;             // the stream the staging kernels of this batch run on
    std::vector<uint64_t> meta_host;             // host copy of the chunk tables (must outlive its async copy)
    uint64_t total_bases = 0, total_head = 0, nb_max = 0, algorithmic_in = 0, h2d_bytes = 0;
    uint32_t min_len = 0, max_len = 0, max_head = 0;
    SlotGeom geom{};
    std::vector<Sub> subs;
    size_t out_total[4] = {0, 0, 0, 0};          // sum of the sub-batches' regions

    std::vector<SortTile> tiles_host;            // sort tiles of all sub-batches (must outlive its async copy)
    std::vector<uint32_t> ctiles_host;           // per sub-batch: sort tiles in front of every chunk
    DevBuf d_chunk_tiles;
    // ---- device-side parse (chunks handed over without record tables; parse.cuh) ------------------------------------------
    bool device_parse = false;
    int parse_state = 0;                         // 0: nothing pending (tables from the host, or parse finished); 1: line ends counted; 2: records built
    std::vector<ParseSeg> segs_host;             // one segment per (chunk, mate)
    PinBuf h_up;                                 // page-locked arena the small tables go up from (upload_small)
    size_t up_used = 0;
    std::vector<uint8_t> seg_open_end;           // 1: the segment's text does not end with a line end (its last line is one more line)
    std::vector<uint64_t> chunk_cap;             // record candidates per chunk (table capacity)
    std::vector<uint64_t> chunk_n;               // records per chunk (what the parse found, or what the caller's tables hold)
    uint64_t total_tiles = 0;
    uint32_t split = 1;
    bool profile_check = false;
    DevBuf d_segs, d_tile_count, d_tile_prefix, d_end_mask, d_line_start, d_parse_res, d_seg_ends, d_rec_tmp, d_parse_scan_tmp;
    PinBuf h_seg_ends, h_parse_res;
    cudaEvent_t ev_parse = nullptr;
    DevBuf d_text[2], d_rec[2], d_chunk_meta, d_stage_stats, d_chunk_sums, d_sort_tiles;
    PinBuf h_stage_stats, h_chunk_sums;
    DevBuf d_out[4], d_desc, d_summary, d_sig, d_info;
    cudaEvent_t ev_h2d = nullptr, ev_chk = nullptr, ev_run = nullptr, ev_d2h = nullptr;
};

// Pinned host memory holding the results of one (sub-)batch until the next call on the context.
struct HostOut
{
    PinBuf out[4], desc, summary, sig, info, rec[2];
    uint64_t d2h_bytes = 0;
};

struct fsb_ctx
{
    fsb_params params{};
    DeviceParams dp{};
    int device = 0;
    cudaStream_t stream = nullptr;               // kernels
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr, s_chk[3] = {nullptr, nullptr, nullptr};   // copy streams and one input-check stream per buffer set of the pipelined fsb_bin_chunks (created on first use)
    bool own_stream = false;
    std::string err;
    bool per_read = false, profile = false, validate = true;
    const CallTrace* trace = nullptr;            // FSB_TRACE: the timeline of the fsb_bin_chunks call in progress
    uint64_t sub_batch_records = 400000;         // fsb_bin_chunks cuts its chunk list into sub-batches of at least this many records

    Batch batch[3];                              // [0] is the batch of fsb_stage / fsb_run / fsb_fetch; fsb_bin_chunks cycles through all three
    std::vector<HostOut*> host;                  // [g] results of sub-batch g ([0] for the resident interface)

    // the pipeline's intermediates; lane 0 runs on `stream`, lane 1 (second stream) only when fsb_run splits a batch
    struct Lane
    {
        cudaStream_t st = nullptr;
        bool own = false;
        cudaEvent_t ev_done = nullptr;
        DevBuf d_keys[2], d_cards[2], d_slots, d_counts, d_counts_scan, d_scan_tmp;
        DevBuf d_flags, d_flags_excl, d_bin_of, d_bin_start, d_bin_min, d_bin_max, d_raw_dna, d_raw_head, d_tbase;
        DevBuf d_bits[4], d_P[4], d_bytes[4], d_BO[4];
        DevBuf d_lay_states, d_chunk_start, d_nb;     // the one-scan layout (layout_fused.cuh)
        template <class F> void each(F f)
        {
            DevBuf* all[] = {&d_keys[0], &d_keys[1], &d_cards[0], &d_cards[1], &d_slots, &d_counts, &d_counts_scan, &d_scan_tmp, &d_flags, &d_flags_excl,
                             &d_bin_of, &d_bin_start, &d_bin_min, &d_bin_max, &d_raw_dna, &d_raw_head, &d_tbase, &d_bits[0], &d_bits[1], &d_bits[2], &d_bits[3],
                             &d_P[0], &d_P[1], &d_P[2], &d_P[3], &d_bytes[0], &d_bytes[1], &d_bytes[2], &d_bytes[3], &d_BO[0], &d_BO[1], &d_BO[2], &d_BO[3],
                             &d_lay_states, &d_chunk_start, &d_nb};
            for (DevBuf* d : all) f(*d);
        }
    } lane[2];
    cudaEvent_t ev_fork = nullptr;
    uint32_t run_split = 1;                      // sub-batches fsb_run cuts a staged batch into (FSB_OPT_RUN_SPLIT)
    uint32_t k1_batches_per_warp = 32, k4_tiles_per_block = 64;   // block granularity of K1 / K4 when sub-batches share the GPU (0: persistent)
    bool block_grids_always = false;             // use that granularity for unsplit runs too (measurement only)
    bool fused_layout = true;                    // batches of one read length take the one-scan layout (FSB_OPT_FUSED_LAYOUT, measurement only)
    bool fused_hist = false;                     // K1 / every scatter pass count the digits of the next radix pass (FSB_OPT_FUSED_HIST).  Measured SLOWER than the
                                                 // histogram kernels (sort 0.79 vs 0.44 ms per 10M pairs, r02l): 10M scattered L2 reductions cost more than re-reading the keys
    bool keep_records = false;                   // device-side parse inside fsb_bin_chunks: copy the record tables back too (FSB_OPT_KEEP_RECORDS)
    struct RecRef { const fsb_record* host[2]; uint64_t n; };
    std::vector<RecRef> rec_index;               // per chunk of the last fsb_bin_chunks call (device-side parse + keep_records)
    bool keep_comments = true;                   // device-side parse: keep the title's comment (FSB_OPT_KEEP_COMMENTS; 0 = the reference's -C)

    // ---- profiling -----------------------------------------------------------------------------
    std::vector<cudaEvent_t> events;             // kMaxPendingProfiles * (FSB_STAGE_COUNT + 1)
    int pending_profiles = 0;
    std::vector<uint8_t> pending_first;          // per pending profile: it is the first sub-batch of its run
    float stage_ms[FSB_STAGE_COUNT] = {0, 0, 0, 0};
    uint32_t stage_runs = 0;
    cudaEvent_t ev_check[2] = {nullptr, nullptr};   // around the input-check kernels of fsb_stage (FSB_OPT_PROFILE)
    bool check_pending = false;
    float check_ms = 0;

    fsb_stats stats{};
};

namespace {

int fail(fsb_ctx* c, int code, const std::string& msg)
{
    if (c) c->err = msg; else g_create_error = msg;
    return code;
}

#define CUDA_TRY(ctx, expr)                                                                              \
    do {                                                                                                 \
        cudaError_t e__ = (expr);                                                                        \
        if (e__ != cudaSuccess)                                                                          \
            return fail(ctx, e__ == cudaErrorMemoryAllocation ? FSB_ERR_NOMEM : FSB_ERR_CUDA,            \
                        std::string(#expr) + ": " + cudaGetErrorString(e__));                            \
    } while (0)

BatchView batch_view(const Batch& b)
{
    BatchView B{};
    const uint64_t* meta = b.d_chunk_meta.as<uint64_t>();
    B.text[0] = b.d_text[0].as<uint8_t>(); B.text[1] = b.d_text[1].as<uint8_t>();
    B.rec[0] = b.d_rec[0].as<fsb_record>(); B.rec[1] = b.d_rec[1].as<fsb_record>();
    B.chunk_first_rec = meta;
    B.chunk_text_base[0] = meta + (b.n_chunks + 1);
    B.chunk_text_base[1] = meta + (b.n_chunks + 1) + b.n_chunks;
    B.n_chunks = b.n_chunks; B.n_records = b.n_records;
    return B;
}
// the same for one sub-batch: records and chunks counted from its own start
BatchView sub_view(const Batch& b, const Sub& s)
{
    BatchView B = batch_view(b);
    const uint64_t* meta = b.d_chunk_meta.as<uint64_t>();
    B.rec[0] += s.r0; if (B.rec[1]) B.rec[1] += s.r0;
    B.chunk_first_rec = meta + s.meta_first;
    B.chunk_text_base[0] += s.c0; B.chunk_text_base[1] += s.c0;
    B.n_chunks = s.c1 - s.c0; B.n_records = s.r1 - s.r0;
    return B;
}

template <int NW, int Q>
cudaError_t launch_ingest_q(const BatchView& B, const DeviceParams& P, const SlotGeom& G, uint32_t max_head, uint32_t R, uint32_t* keys, unsigned long long* cards,
                            uint32_t* slots, uint32_t* sig, uint32_t* info, const SortSeed& seed, cudaStream_t st)
{
    IngestPlan pl = make_ingest_plan<NW>(P, G, max_head);
    pl.batches_per_warp = R;
    cudaError_t e = cudaFuncSetAttribute(ingest_kernel<NW, Q>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.total_bytes);
    if (e != cudaSuccess) return e;
    const uint64_t n_mates = P.paired ? 2 * B.n_records : B.n_records;
    // persistent warps: as many blocks as fit on the device at once, each warp strides over the warp batches
    int dev = 0, sms = 0, per_sm = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ingest_kernel<NW, Q>, (int)(pl.warps * 32), pl.total_bytes)) != cudaSuccess) return e;
    const uint64_t need = (n_mates + pl.warps * 32 - 1) / (pl.warps * 32);
    // persistent: as many blocks as fit on the device at once; otherwise every block owns R warp batches per warp
    const unsigned blocks = R ? (unsigned)std::max<uint64_t>(1, (need + R - 1) / R)
                              : (unsigned)std::max<uint64_t>(1, std::min<uint64_t>(need, (uint64_t)sms * (uint64_t)std::max(per_sm, 1)));
    ingest_kernel<NW, Q><<<blocks, pl.warps * 32, pl.total_bytes, st>>>(B, P, G, pl, keys, cards, slots, sig, info, seed);
    return cudaGetLastError();
}
template <int NW>
cudaError_t launch_ingest(const BatchView& B, const DeviceParams& P, const SlotGeom& G, uint32_t max_head, uint32_t R, uint32_t* keys, unsigned long long* cards,
                          uint32_t* slots, uint32_t* sig, uint32_t* info, const SortSeed& seed, cudaStream_t st)
{
    if (P.qua_bits == 6) return launch_ingest_q<NW, 6>(B, P, G, max_head, R, keys, cards, slots, sig, info, seed, st);
    if (P.qua_bits == 3) return launch_ingest_q<NW, 3>(B, P, G, max_head, R, keys, cards, slots, sig, info, seed, st);
    return launch_ingest_q<NW, 1>(B, P, G, max_head, R, keys, cards, slots, sig, info, seed, st);
}

cudaError_t launch_place(const PlaceArgs& pa, const Placement& pm, uint32_t max_len, uint32_t max_head, uint32_t R, bool tables_ready, cudaStream_t st, int* launches)
{
    const uint64_t n = pa.B.n_records;
    PlacePlan pl = make_place_plan(pa.P, pa.G, max_len, max_head);
    pl.tiles_per_block = R;
    const uint64_t tiles = (n + pl.T - 1) / pl.T;
    // placement tables (tile ranges, every record's position inside its tile) and the zeroing of the words two tiles share --
    // unless the one-scan layout has produced them already
    if (!tables_ready) { placement_kernel<<<(unsigned)((tiles * pl.T + 255) / 256), 256, 0, st>>>(pa, pm, tiles); *launches += 1; }
    cudaError_t e = cudaFuncSetAttribute(place_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.total_bytes);
    if (e != cudaSuccess) return e;
    // persistent blocks: as many as fit on the device at once
    int dev = 0, sms = 0, per_sm = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, place_kernel, (int)pl.threads, pl.total_bytes)) != cudaSuccess) return e;
    const unsigned blocks = R ? (unsigned)std::max<uint64_t>(1, (tiles + R - 1) / R)
                              : (unsigned)std::max<uint64_t>(1, std::min<uint64_t>(tiles, (uint64_t)sms * (uint64_t)std::max(per_sm, 1)));
    place_kernel<<<blocks, pl.threads, pl.total_bytes, st>>>(pa, pl, pm, tiles);
    *launches += 1;
    return cudaGetLastError();
}


int resolve_profiles(fsb_ctx* c)
{
    if (c->pending_profiles == 0) return FSB_OK;
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    for (int r = 0; r < c->pending_profiles; ++r)
    {
        cudaEvent_t* ev = &c->events[(size_t)r * (FSB_STAGE_COUNT + 1)];
        for (int s = 0; s < FSB_STAGE_COUNT; ++s)
        {
            float ms = 0;
            CUDA_TRY(c, cudaEventElapsedTime(&ms, ev[s], ev[s + 1]));
            c->stage_ms[s] += ms;
        }
        if (c->pending_first[r]) c->stage_runs++;                 // a batch with more than 32 chunks runs as several sub-batches: one run
    }
    c->pending_profiles = 0;
    return FSB_OK;
}

// A shared intermediate may be in use by kernels of the previous sub-batch: wait for them before it is reallocated.
cudaError_t ensure_shared(cudaStream_t st, DevBuf& b, size_t bytes)
{
    if (bytes <= b.cap) return cudaSuccess;
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return e;
    return b.ensure(bytes);
}

HostOut* host_out(fsb_ctx* c, size_t g)
{
    while (c->host.size() <= g) c->host.push_back(new (std::nothrow) HostOut());
    return c->host[g];
}

// `bytes` of host data to device memory on `st` without the copy engine: through the batch's page-locked arena and a kernel.
// The arena is rewound by stage_enqueue; it grows (after waiting for `st`, so that nothing reads the old one) if it runs out.
int upload_small(fsb_ctx* c, Batch& b, void* dev, const void* src, size_t bytes, cudaStream_t st)
{
    if (bytes == 0) return FSB_OK;
    const size_t need = align_up(bytes, 16);
    if (b.up_used + need > b.h_up.cap)
    {
        CUDA_TRY(c, cudaStreamSynchronize(st));
        b.up_used = 0;
        CUDA_TRY(c, b.h_up.ensure(std::max<size_t>(2 * need, (size_t)1 << 20)));
    }
    uint8_t* slot = b.h_up.as<uint8_t>() + b.up_used;
    std::memcpy(slot, src, bytes);
    b.up_used += need;
    void* mapped = nullptr;
    CUDA_TRY(c, cudaHostGetDevicePointer(&mapped, slot, 0));
    const size_t n = (bytes + 3) / 4;
    words_copy_kernel<<<words_grid(n), 256, 0, st>>>(reinterpret_cast<const uint32_t*>(mapped), reinterpret_cast<uint32_t*>(dev), (uint32_t)n);
    CUDA_TRY(c, cudaGetLastError());
    c->stats.kernel_launches++;
    return FSB_OK;
}

// ------------------------------------------------------------------------------------------------
// Stage, last enqueue step: the records per chunk are known (b.chunk_n: from the caller's tables or from the device-side
// parse).  Chunk tables, sub-batches and sort tiles go up, then the device-side check of the record tables (offsets
// inside the chunk, lengths, PE mate-length equality - the things the reference only ASSERTs: FastqRecord.h:87,
// FastqParser.cpp:130) together with the batch statistics that size the buffers, the byte-level check, and the copy of
// the results back.  Everything goes to `st`; b.ev_chk fires when the results are on the host.
int stage_finalize(fsb_ctx* c, Batch& b, cudaStream_t st)
{
    const uint32_t n_chunks = b.n_chunks;
    b.chunk_first_rec.assign(n_chunks + 1, 0);
    uint64_t n = 0;
    for (uint32_t ci = 0; ci < n_chunks; ++ci) { b.chunk_first_rec[ci] = n; n += b.chunk_n[ci]; }
    b.chunk_first_rec[n_chunks] = n;
    if (n > kMaxBatchRecords) return fail(c, FSB_ERR_PARAM, "fsb_stage: more than 2^28-1 records in one batch");
    b.n_records = n;

    // ---- sub-batches: runs of whole chunks with about n / split records each --------------------------------------
    b.subs.clear();
    {
        // (K1 keeps the chunk tables of up to 32 chunks in registers; a batch of more chunks is cut so that every sub-batch qualifies)
        const uint32_t S = std::max<uint32_t>(1, std::min<uint32_t>(std::max<uint32_t>(b.split, (n_chunks + 31u) / 32u), n_chunks));
        uint32_t c0 = 0;
        for (uint32_t j = 0; j < S && c0 < n_chunks; ++j)
        {
            const uint64_t goal = n * (uint64_t)(j + 1) / S;                 // records the first j + 1 sub-batches should hold together
            uint32_t c1 = n_chunks;
            if (j + 1 < S)
            {
                const uint32_t last = n_chunks - (S - 1 - j);               // leave a chunk for every later sub-batch
                c1 = c0 + 1;
                while (c1 < last && b.chunk_first_rec[c1] < goal) ++c1;
            }
            Sub sb;
            sb.c0 = c0; sb.c1 = c1; sb.r0 = b.chunk_first_rec[c0]; sb.r1 = b.chunk_first_rec[c1];
            b.subs.push_back(sb);
            c0 = c1;
        }
    }
    uint64_t h2d = 0;
    // chunk tables: [first_rec (n_chunks+1)] [text_base0] [text_base1] [text_size0] [text_size1]  (n_chunks each), then per sub-batch
    // its own first-record table counted from the sub-batch's first record (chunks + 1 entries)
    std::vector<uint64_t>& meta = b.meta_host;
    meta.clear();
    meta.insert(meta.end(), b.chunk_first_rec.begin(), b.chunk_first_rec.end());
    meta.insert(meta.end(), b.chunk_text_base[0].begin(), b.chunk_text_base[0].end());
    meta.insert(meta.end(), b.chunk_text_base[1].begin(), b.chunk_text_base[1].end());
    for (int m = 0; m < 2; ++m)
        for (uint32_t ci = 0; ci < n_chunks; ++ci) meta.push_back(b.chunk_text_size[m][ci]);
    for (Sub& sb : b.subs)
    {
        sb.meta_first = meta.size();
        for (uint32_t ci = sb.c0; ci <= sb.c1; ++ci) meta.push_back(b.chunk_first_rec[ci] - sb.r0);
    }
    CUDA_TRY(c, b.d_chunk_meta.ensure(meta.size() * sizeof(uint64_t)));
    if (int rc = upload_small(c, b, b.d_chunk_meta.p, meta.data(), meta.size() * sizeof(uint64_t), st)) return rc;
    h2d += meta.size() * sizeof(uint64_t);
    // sort tiles: every tile lies inside one chunk (scan_sort.cuh)
    b.tiles_host.clear(); b.ctiles_host.clear();
    for (Sub& sb : b.subs)
    {
        sb.tile_off = b.tiles_host.size();
        sb.ctile_off = b.ctiles_host.size();
        uint32_t cblk = 0;
        for (uint32_t ci = sb.c0; ci < sb.c1; ++ci)
        {
            b.ctiles_host.push_back(cblk);
            const uint64_t first = b.chunk_first_rec[ci] - sb.r0, cnt = b.chunk_first_rec[ci + 1] - b.chunk_first_rec[ci];
            const uint32_t nblk = (uint32_t)((cnt + kSortTile - 1) / kSortTile);
            for (uint32_t k = 0; k < nblk; ++k)
            {
                SortTile t{};
                t.first = (uint32_t)(first + (uint64_t)k * kSortTile);
                t.count = (uint32_t)std::min<uint64_t>(kSortTile, cnt - (uint64_t)k * kSortTile);
                t.cblk = cblk; t.blk = k; t.nblk = nblk;
                b.tiles_host.push_back(t);
            }
            cblk += nblk;
        }
        b.ctiles_host.push_back(cblk);
        sb.n_tiles = b.tiles_host.size() - sb.tile_off;
    }
    CUDA_TRY(c, b.d_chunk_tiles.ensure((b.ctiles_host.size() + 1) * 4));
    if (int rc = upload_small(c, b, b.d_chunk_tiles.p, b.ctiles_host.data(), b.ctiles_host.size() * 4, st)) return rc;
    CUDA_TRY(c, b.d_sort_tiles.ensure((b.tiles_host.size() + 1) * sizeof(SortTile)));
    if (int rc = upload_small(c, b, b.d_sort_tiles.p, b.tiles_host.data(), b.tiles_host.size() * sizeof(SortTile), st)) return rc;
    h2d += b.tiles_host.size() * sizeof(SortTile);

    CUDA_TRY(c, b.d_stage_stats.ensure(sizeof(StageStats)));
    CUDA_TRY(c, b.h_stage_stats.ensure(2 * sizeof(StageStats)));
    CUDA_TRY(c, b.d_chunk_sums.ensure((size_t)n_chunks * 2 * sizeof(uint64_t)));
    CUDA_TRY(c, b.h_chunk_sums.ensure((size_t)n_chunks * 2 * sizeof(uint64_t)));
    StageStats init{};
    init.first_bad = ~0ull; init.first_bad_text = ~0ull; init.min_len = 0xFFFFFFFFu;
    if (int rc = upload_small(c, b, b.d_stage_stats.p, &init, sizeof(StageStats), st)) return rc;
    CUDA_TRY(c, small_fill(b.d_chunk_sums.p, 0u, (size_t)n_chunks * 2 * sizeof(uint64_t), st));
    if (n)
    {
        const BatchView B = batch_view(b);
        const uint64_t* m64 = b.d_chunk_meta.as<uint64_t>();
        const unsigned blocks = (unsigned)std::min<uint64_t>((n + 255) / 256, 148ull * 8);
        if (b.profile_check)
        {
            for (cudaEvent_t& e : c->ev_check) if (!e) CUDA_TRY(c, cudaEventCreate(&e));
            CUDA_TRY(c, cudaEventRecord(c->ev_check[0], st));
        }
        stage_stats_kernel<<<blocks, 256, 0, st>>>(B, c->dp, m64 + (3 * (size_t)n_chunks + 1), m64 + (4 * (size_t)n_chunks + 1), b.d_stage_stats.as<StageStats>(),
                                                    b.d_chunk_sums.as<unsigned long long>());
        c->stats.kernel_launches++;
        if (c->validate)
        {   // FSB_OPT_VALIDATE: symbols, quality range and title characters behind the table (stage.cuh)
            const uint64_t n_mates = c->dp.paired ? 2 * n : n;
            const unsigned vblocks = (unsigned)std::min<uint64_t>((n_mates + 15) / 16, 148ull * 16);
            validate_text_kernel<<<vblocks, 256, 0, st>>>(B, c->dp, m64 + (3 * (size_t)n_chunks + 1), m64 + (4 * (size_t)n_chunks + 1), b.d_stage_stats.as<StageStats>());
            c->stats.kernel_launches++;
        }
        if (b.profile_check) { CUDA_TRY(c, cudaEventRecord(c->ev_check[1], st)); c->check_pending = true; }
    }
    CUDA_TRY(c, small_to_host(b.h_stage_stats.p, b.d_stage_stats.p, sizeof(StageStats), st));
    CUDA_TRY(c, small_to_host(b.h_chunk_sums.p, b.d_chunk_sums.p, (size_t)n_chunks * 2 * sizeof(uint64_t), st));
    CUDA_TRY(c, cudaEventRecord(b.ev_chk, st));
    b.h2d_bytes += h2d;
    c->stats.h2d_bytes += h2d;
    b.parse_state = 0;
    return FSB_OK;
}

// Device-side parse, step 1 (parse.cuh): line ends per tile of every (chunk, mate) text, their scan, the line ends per segment back
// to the host.  b.ev_parse fires when they are there.
int parse_enqueue_count(fsb_ctx* c, Batch& b, const fsb_chunk* chunks, cudaStream_t st)
{
    const int nfiles = c->dp.paired ? 2 : 1;
    b.segs_host.clear(); b.seg_open_end.clear();
    uint64_t tiles = 0;
    for (uint32_t ci = 0; ci < b.n_chunks; ++ci)
        for (int m = 0; m < nfiles; ++m)
        {
            ParseSeg sg{};
            sg.text_base = b.chunk_text_base[m][ci]; sg.size = chunks[ci].text_size[m]; sg.tile0 = tiles; sg.mate = (uint32_t)m; sg.chunk = ci;
            tiles += (sg.size + kParseTile - 1) / kParseTile;
            b.segs_host.push_back(sg);
            const uint8_t last = sg.size ? chunks[ci].text[m][sg.size - 1] : (uint8_t)'\n';
            b.seg_open_end.push_back((sg.size && last != '\n' && last != '\r') ? 1 : 0);
        }
    b.total_tiles = tiles;
    const size_t n_segs = b.segs_host.size();
    ParseSeg guard{};                                                  // one past the last segment: ends the tile search
    guard.tile0 = tiles;
    b.segs_host.push_back(guard);
    CUDA_TRY(c, b.d_segs.ensure((n_segs + 1) * sizeof(ParseSeg)));
    if (int rc = upload_small(c, b, b.d_segs.p, b.segs_host.data(), (n_segs + 1) * sizeof(ParseSeg), st)) return rc;
    CUDA_TRY(c, b.d_tile_count.ensure((tiles + 2) * 4));
    CUDA_TRY(c, b.d_end_mask.ensure((tiles + 1) * kParseTileVecs * sizeof(uint16_t)));
    CUDA_TRY(c, b.d_tile_prefix.ensure((tiles + 2) * 4));
    CUDA_TRY(c, b.d_parse_scan_tmp.ensure((scan_num_tiles(tiles + 1) + 2) * 4));
    CUDA_TRY(c, b.d_seg_ends.ensure((n_segs + 1) * 4));
    CUDA_TRY(c, b.h_seg_ends.ensure((n_segs + 1) * 4));
    if (tiles)
    {
        parse_count_kernel<<<(unsigned)tiles, kParseThreads, 0, st>>>(b.d_text[0].as<uint8_t>(), b.d_text[1].as<uint8_t>(), b.d_segs.as<ParseSeg>(), (uint32_t)n_segs,
                                                                       b.d_tile_count.as<uint32_t>(), b.d_end_mask.as<uint16_t>());
        c->stats.kernel_launches++;
    }
    c->stats.kernel_launches += exclusive_scan<uint32_t, uint32_t>(b.d_tile_count.as<uint32_t>(), tiles, b.d_tile_prefix.as<uint32_t>(), b.d_parse_scan_tmp.as<uint32_t>(), st);
    parse_seg_ends_kernel<<<(unsigned)((n_segs + 127) / 128), 128, 0, st>>>(b.d_segs.as<ParseSeg>(), (uint32_t)n_segs, b.d_tile_prefix.as<uint32_t>(), b.d_seg_ends.as<uint32_t>());
    c->stats.kernel_launches++;
    CUDA_TRY(c, small_to_host(b.h_seg_ends.p, b.d_seg_ends.p, n_segs * 4, st));
    CUDA_TRY(c, cudaEventRecord(b.ev_parse, st));
    b.parse_state = 1;
    return FSB_OK;
}

// Device-side parse, steps 2 and 3, and then the common last step: called until b.parse_state is 0 again.  Blocks on the small
// results of the step before (they size what comes next).
int stage_advance(fsb_ctx* c, Batch& b, cudaStream_t st)
{
    const int nfiles = c->dp.paired ? 2 : 1;
    const size_t n_segs = b.segs_host.size() - 1;
    if (b.parse_state == 1)
    {
        CUDA_TRY(c, cudaEventSynchronize(b.ev_parse));
        if (c->trace) c->trace->mark("  line ends counted", 0);
        const uint32_t* ends = b.h_seg_ends.as<uint32_t>();
        uint64_t lines = 0;
        b.chunk_cap.assign(b.n_chunks, 0);
        for (size_t k = 0; k < n_segs; ++k)
        {
            ParseSeg& sg = b.segs_host[k];
            sg.n_ends = ends[k];
            sg.n_lines = ends[k] + b.seg_open_end[k];
            sg.cap = (sg.n_lines + 3u) / 4u;
            sg.line0 = lines;
            lines += (uint64_t)sg.n_ends + 2;
            b.chunk_cap[sg.chunk] = std::max<uint64_t>(b.chunk_cap[sg.chunk], sg.cap);
        }
        uint64_t cap_total = 0;
        std::vector<uint64_t> cap_first(b.n_chunks + 1, 0);
        for (uint32_t ci = 0; ci < b.n_chunks; ++ci) { cap_first[ci] = cap_total; cap_total += b.chunk_cap[ci]; }
        cap_first[b.n_chunks] = cap_total;
        if (cap_total > kMaxBatchRecords) return fail(c, FSB_ERR_PARAM, "fsb_stage: more than 2^28-1 records in one batch");
        uint32_t cap_max = 0;
        for (size_t k = 0; k < n_segs; ++k) { b.segs_host[k].rec0 = cap_first[b.segs_host[k].chunk]; cap_max = std::max(cap_max, b.segs_host[k].cap); }
        if (int rc = upload_small(c, b, b.d_segs.p, b.segs_host.data(), (n_segs + 1) * sizeof(ParseSeg), st)) return rc;
        CUDA_TRY(c, b.d_line_start.ensure((lines + 2) * 4));
        for (int m = 0; m < nfiles; ++m) CUDA_TRY(c, b.d_rec[m].ensure((cap_total + 1) * sizeof(fsb_record)));
        CUDA_TRY(c, b.d_parse_res.ensure((n_segs + 1) * sizeof(ParseResult)));
        CUDA_TRY(c, b.h_parse_res.ensure((n_segs + 1) * sizeof(ParseResult)));
        CUDA_TRY(c, small_fill(b.d_parse_res.p, 0xFFFFFFFFu, (n_segs + 1) * sizeof(ParseResult), st));
        if (b.total_tiles)
        {
            parse_lines_kernel<<<(unsigned)b.total_tiles, kParseThreads, 0, st>>>(b.d_end_mask.as<uint16_t>(), b.d_segs.as<ParseSeg>(), (uint32_t)n_segs,
                                                                                   b.d_tile_prefix.as<uint32_t>(), b.d_line_start.as<uint32_t>());
            c->stats.kernel_launches++;
        }
        if (cap_max)
        {
            parse_records_kernel<<<dim3((cap_max + 255u) / 256u, (unsigned)n_segs), 256, 0, st>>>(b.d_text[0].as<uint8_t>(), b.d_text[1].as<uint8_t>(), b.d_segs.as<ParseSeg>(),
                b.d_line_start.as<uint32_t>(), c->dp.has_headers, c->keep_comments ? 1u : 0u, b.d_rec[0].as<fsb_record>(), b.d_rec[1].as<fsb_record>(), b.d_parse_res.as<ParseResult>());
            c->stats.kernel_launches++;
        }
        CUDA_TRY(c, small_to_host(b.h_parse_res.p, b.d_parse_res.p, n_segs * sizeof(ParseResult), st));
        CUDA_TRY(c, cudaEventRecord(b.ev_parse, st));
        b.parse_state = 2;
        return FSB_OK;
    }
    if (b.parse_state == 2)
    {
        CUDA_TRY(c, cudaEventSynchronize(b.ev_parse));
        if (c->trace) c->trace->mark("  records parsed", 0);
        const ParseResult* res = b.h_parse_res.as<ParseResult>();
        // records of a chunk: where the first of its (one or two) parsers stops -- FastqRecordsParserPE::ParseFrom runs both in step (FastqParser.cpp:527)
        b.chunk_n.assign(b.n_chunks, ~0ull);
        for (size_t k = 0; k < n_segs; ++k)
        {
            const ParseSeg& sg = b.segs_host[k];
            const uint64_t n_seg = std::min<uint64_t>(sg.cap, res[k].first_bad == ~0ull ? (uint64_t)sg.cap : (res[k].first_bad >> 8));
            b.chunk_n[sg.chunk] = std::min(b.chunk_n[sg.chunk], n_seg);
        }
        for (size_t k = 0; k < n_segs; ++k)
        {
            const ParseSeg& sg = b.segs_host[k];
            if (res[k].first_invalid < b.chunk_n[sg.chunk])
                return fail(c, FSB_ERR_INPUT, "fsb_stage: record " + std::to_string(res[k].first_invalid) + " of chunk " + std::to_string(b.chunk0 + sg.chunk) +
                                                  " is outside the input contract (read length 1..255, title at most 255 bytes)");
        }
        // the tables were written at capacity positions: close the gaps a chunk with fewer records than candidates leaves behind
        uint64_t dense = 0, at = 0;
        for (uint32_t ci = 0; ci < b.n_chunks; ++ci)
        {
            const uint64_t nc = b.chunk_n[ci];
            if (dense != at && nc)
            {
                CUDA_TRY(c, b.d_rec_tmp.ensure(nc * sizeof(fsb_record)));
                for (int m = 0; m < nfiles; ++m)
                {
                    CUDA_TRY(c, cudaMemcpyAsync(b.d_rec_tmp.p, b.d_rec[m].as<fsb_record>() + at, nc * sizeof(fsb_record), cudaMemcpyDeviceToDevice, st));
                    CUDA_TRY(c, cudaMemcpyAsync(b.d_rec[m].as<fsb_record>() + dense, b.d_rec_tmp.p, nc * sizeof(fsb_record), cudaMemcpyDeviceToDevice, st));
                }
            }
            dense += nc; at += b.chunk_cap[ci];
        }
        return stage_finalize(c, b, st);
    }
    return FSB_OK;
}

// Stage, first enqueue step: the host->device copies of a group of chunks on `st`.  With record tables from the caller the
// rest follows at once (stage_finalize on `st_check`, which waits for the copies); chunks handed over as text alone
// (records == NULL) are parsed on the device first (parse_enqueue_count here, then stage_advance until b.parse_state is 0).
// The batch's input buffers must not be in use.  `split` = sub-batches of whole chunks the kernels will run as.  The pipeline
// keeps its copy stream free of kernels, so that the next sub-batch's text follows at once.
int stage_enqueue(fsb_ctx* c, Batch& b, const fsb_chunk* chunks, uint32_t n_chunks, uint32_t chunk0, cudaStream_t st, cudaStream_t st_check, uint32_t split, bool profile = false)
{
    b.staged = false; b.ran = false; b.parse_state = 0; b.up_used = 0;
    b.split = split; b.profile_check = profile;
    const int nfiles = c->dp.paired ? 2 : 1;
    const uint32_t max_chunks = (uint32_t)std::min<uint64_t>(kMaxChunksPerBatch, 1ull << (32 - c->dp.key_bits));
    if (n_chunks == 0) return fail(c, FSB_ERR_PARAM, "fsb_stage: no chunks");
    if (n_chunks > max_chunks) return fail(c, FSB_ERR_PARAM, "fsb_stage: too many chunks in one batch for this signature length (max " + std::to_string(max_chunks) + ")");

    b.n_chunks = n_chunks;
    b.chunk0 = chunk0;
    b.device_parse = chunks[0].records[0] == nullptr && chunks[0].text[0] != nullptr;
    size_t text_bytes[2] = {kTextPad, kTextPad};
    for (int m = 0; m < 2; ++m) { b.chunk_text_base[m].assign(n_chunks, 0); b.chunk_text_size[m].assign(n_chunks, 0); }
    b.chunk_n.assign(n_chunks, 0);
    uint64_t n = 0;
    for (uint32_t ci = 0; ci < n_chunks; ++ci)
    {
        const fsb_chunk& ch = chunks[ci];
        for (int m = 0; m < nfiles; ++m)
        {
            if (b.device_parse ? (ch.records[m] != nullptr || (ch.text_size[m] && !ch.text[m])) : (ch.n_records && (!ch.text[m] || !ch.records[m])))
                return fail(c, FSB_ERR_PARAM, b.device_parse ? "fsb_stage: chunks without record tables (device-side parse) and chunks with them cannot be mixed" : "fsb_stage: null text/records");
            if (ch.text_size[m] >= 0xFFFFFFFFull) return fail(c, FSB_ERR_INPUT, "fsb_stage: chunk text must be < 4 GiB (32-bit record offsets)");
            b.chunk_text_base[m][ci] = text_bytes[m];
            b.chunk_text_size[m][ci] = ch.text_size[m];
            text_bytes[m] = align_up(text_bytes[m] + ch.text_size[m] + kTextPad, 256);
        }
        if (!b.device_parse) { b.chunk_n[ci] = ch.n_records; n += ch.n_records; }
    }
    if (n > kMaxBatchRecords) return fail(c, FSB_ERR_PARAM, "fsb_stage: more than 2^28-1 records in one batch");

    uint64_t h2d = 0;
    for (int m = 0; m < nfiles; ++m)
    {
        CUDA_TRY(c, b.d_text[m].ensure(text_bytes[m] + kTextPad, &st));      // padding between chunks is over-read by aligned window copies: keep it defined
        if (!b.device_parse) CUDA_TRY(c, b.d_rec[m].ensure((n + 1) * sizeof(fsb_record)));
        uint64_t first = 0;
        for (uint32_t ci = 0; ci < n_chunks; ++ci)
        {
            const fsb_chunk& ch = chunks[ci];
            if (ch.text_size[m])
                CUDA_TRY(c, cudaMemcpyAsync(b.d_text[m].as<uint8_t>() + b.chunk_text_base[m][ci], ch.text[m], ch.text_size[m], cudaMemcpyHostToDevice, st));
            h2d += ch.text_size[m];
            if (!b.device_parse && ch.n_records)
            {
                CUDA_TRY(c, cudaMemcpyAsync(b.d_rec[m].as<fsb_record>() + first, ch.records[m], ch.n_records * sizeof(fsb_record), cudaMemcpyHostToDevice, st));
                h2d += ch.n_records * sizeof(fsb_record);
                first += ch.n_records;
            }
        }
    }
    b.h2d_bytes = h2d;
    c->stats.h2d_bytes += h2d;
    if (st_check != st)
    {
        CUDA_TRY(c, cudaEventRecord(b.ev_h2d, st));
        CUDA_TRY(c, cudaStreamWaitEvent(st_check, b.ev_h2d, 0));
    }
    b.st_check = st_check;
    if (b.device_parse) return parse_enqueue_count(c, b, chunks, st_check);
    return stage_finalize(c, b, st_check);
}

// Stage, step 2 (after everything stage_enqueue put on its stream has completed): reject contract
// violations, then size the result buffers of the batch (which must not be in use) and the lanes'
// intermediates.
int stage_complete(fsb_ctx* c, Batch& b)
{
    const StageStats stats = *b.h_stage_stats.as<StageStats>();
    const uint64_t n = b.n_records;
    const uint32_t n_chunks = b.n_chunks;
    if (stats.n_bad)
    {
        // never run the kernels on tables that point outside the staged text
        uint32_t ci = 0;
        while (ci + 1 < n_chunks && b.chunk_first_rec[ci + 1] <= stats.first_bad) ++ci;
        return fail(c, FSB_ERR_INPUT, "fsb_stage: record " + std::to_string(stats.first_bad - b.chunk_first_rec[ci]) + " of chunk " + std::to_string(b.chunk0 + ci) +
                                          " violates the input contract (length 1..255, offsets inside the chunk, equal PE mate lengths); " +
                                          std::to_string(stats.n_bad) + " such record(s)");
    }
    if (stats.n_bad_text)
    {
        uint32_t ci = 0;
        while (ci + 1 < n_chunks && b.chunk_first_rec[ci + 1] <= stats.first_bad_text) ++ci;
        return fail(c, FSB_ERR_INPUT, "fsb_stage: record " + std::to_string(stats.first_bad_text - b.chunk_first_rec[ci]) + " of chunk " + std::to_string(b.chunk0 + ci) +
                                          " holds a byte outside the input contract (sequence symbols A C G T N, quality in [offset, offset + 64), 7-bit title characters); " +
                                          std::to_string(stats.n_bad_text) + " such mate(s)");
    }
    const uint64_t bases = stats.bases, heads = stats.heads;
    b.total_bases = bases; b.total_head = heads;
    b.min_len = n ? stats.min_len : 0; b.max_len = stats.max_len; b.max_head = stats.max_head;
    b.geom = make_slot_geom(c->dp, b.max_len, b.max_head);

    // ---- the sub-batches' regions of the results (exact stream sizes are only known on the device after the layout scans) ----
    const uint64_t* sums = b.h_chunk_sums.as<uint64_t>();
    uint64_t bin_off = 0;
    size_t off[4] = {0, 0, 0, 0};
    for (Sub& sb : b.subs)
    {
        const uint64_t ns = sb.r1 - sb.r0;
        uint64_t sb_bases = 0, sb_heads = 0;
        for (uint32_t ci = sb.c0; ci < sb.c1; ++ci) { sb_bases += sums[2 * ci]; sb_heads += sums[2 * ci + 1]; }
        sb.nb_max = std::min<uint64_t>(ns, (uint64_t)(sb.c1 - sb.c0) * ((uint64_t)c->dp.nbin + 1));
        sb.bin_off = bin_off; bin_off += sb.nb_max + 1;
        const uint64_t pad_bytes = sb.nb_max + 64;                          // < 1 byte of padding per bin and stream
        sb.out_cap[0] = align_up((28 * ns + 17 * sb.nb_max) / 8 + pad_bytes, 64);
        sb.out_cap[1] = align_up(3 * sb_bases / 8 + pad_bytes, 64);
        sb.out_cap[2] = align_up((uint64_t)c->dp.qua_bits * sb_bases / 8 + pad_bytes, 64);
        sb.out_cap[3] = align_up(c->dp.has_headers ? (8 * ns + 7 * sb_heads) / 8 + pad_bytes : 64, 64);
        for (int s = 0; s < 4; ++s) { sb.out_off[s] = off[s]; off[s] += sb.out_cap[s]; }
    }
    for (int s = 0; s < 4; ++s) b.out_total[s] = off[s];
    b.nb_max = bin_off;

    // ---- the lanes' intermediates (grow-only): lane l runs the sub-batches l, l + 2, .. ---------------------------------
    const size_t n_lanes = std::min<size_t>(2, b.subs.size());
    for (size_t l = 0; l < n_lanes; ++l)
    {
        fsb_ctx::Lane& L = c->lane[l];
        if (!L.st)
        {
            CUDA_TRY(c, cudaStreamCreateWithFlags(&L.st, cudaStreamNonBlocking));
            L.own = true;
            CUDA_TRY(c, cudaEventCreateWithFlags(&L.ev_done, cudaEventDisableTiming));
        }
        uint64_t ln = 0, lnbm = 0, ltiles = 0;
        for (size_t j = l; j < b.subs.size(); j += 2)
        {
            ln = std::max(ln, b.subs[j].r1 - b.subs[j].r0); lnbm = std::max(lnbm, b.subs[j].nb_max); ltiles = std::max(ltiles, b.subs[j].n_tiles);
        }
        const uint64_t ncounts = (uint64_t)kMaxRadix * std::max<uint64_t>(ltiles, 1);
        for (int i = 0; i < 2; ++i)
        {
            CUDA_TRY(c, ensure_shared(L.st, L.d_keys[i], (ln + 1) * 4));
            CUDA_TRY(c, ensure_shared(L.st, L.d_cards[i], (ln + 1) * 8));
        }
        CUDA_TRY(c, ensure_shared(L.st, L.d_slots, (ln + 1) * (size_t)b.geom.words * 4));
        CUDA_TRY(c, ensure_shared(L.st, L.d_counts, (ncounts + 1) * 4));
        CUDA_TRY(c, ensure_shared(L.st, L.d_counts_scan, (ncounts + 1) * 4));
        const uint64_t max_scan_n = std::max<uint64_t>(std::max<uint64_t>(ln, ncounts), lnbm) + 1;
        CUDA_TRY(c, ensure_shared(L.st, L.d_scan_tmp, 4 * (scan_num_tiles(max_scan_n) + 2) * 8));
        uint32_t lchunks = 0;
        for (size_t j = l; j < b.subs.size(); j += 2) lchunks = std::max(lchunks, b.subs[j].c1 - b.subs[j].c0);
        CUDA_TRY(c, ensure_shared(L.st, L.d_lay_states, ((ln + kLayBlock - 1) / kLayBlock + 2 + ((ln + kLayBlock - 1) / kLayBlock) / kLayScanThreads + 2) * sizeof(LayState)));      // block states, the total, the scan's group totals
        CUDA_TRY(c, ensure_shared(L.st, L.d_chunk_start, ((size_t)lchunks + 2) * sizeof(ChunkStart)));
        CUDA_TRY(c, ensure_shared(L.st, L.d_nb, 64));
        CUDA_TRY(c, ensure_shared(L.st, L.d_flags, (ln + 4) * 4));
        CUDA_TRY(c, ensure_shared(L.st, L.d_tbase, ((ln + kPlaceTile - 1) / kPlaceTile + 2) * 4 * 8));
        CUDA_TRY(c, ensure_shared(L.st, L.d_flags_excl, (ln + 2) * 4));
        CUDA_TRY(c, ensure_shared(L.st, L.d_bin_of, (ln + 1) * 4));
        CUDA_TRY(c, ensure_shared(L.st, L.d_bin_start, (lnbm + 2) * 4));
        CUDA_TRY(c, ensure_shared(L.st, L.d_bin_min, (lnbm + 1) * 4));
        CUDA_TRY(c, ensure_shared(L.st, L.d_bin_max, (lnbm + 1) * 4));
        CUDA_TRY(c, ensure_shared(L.st, L.d_raw_dna, (lnbm + 1) * 8));
        CUDA_TRY(c, ensure_shared(L.st, L.d_raw_head, (lnbm + 1) * 8));
        for (int s = 0; s < 4; ++s)
        {
            CUDA_TRY(c, ensure_shared(L.st, L.d_bits[s], (ln + 4) * 4));
            CUDA_TRY(c, ensure_shared(L.st, L.d_P[s], (ln + 2) * 8));
            CUDA_TRY(c, ensure_shared(L.st, L.d_bytes[s], (lnbm + 1) * 8));
            CUDA_TRY(c, ensure_shared(L.st, L.d_BO[s], (lnbm + 2) * 8));
        }
    }
    // ---- results of this batch ---------------------------------------------------------------------------
    CUDA_TRY(c, b.d_desc.ensure((b.nb_max + 1) * sizeof(fsb_bin_descriptor)));
    CUDA_TRY(c, b.d_summary.ensure((size_t)n_chunks * sizeof(ChunkSummary)));
    if (c->per_read)
    {
        CUDA_TRY(c, b.d_info.ensure((n + 1) * 4));
        CUDA_TRY(c, b.d_sig.ensure((n + 1) * 4));
    }
    for (int s = 0; s < 4; ++s) CUDA_TRY(c, b.d_out[s].ensure(b.out_total[s] + 64));

    // SURVEY 8(d) algorithmic input bytes: every sequence, quality and kept header byte once
    b.algorithmic_in = 2 * bases + (c->dp.has_headers ? heads : 0);
    b.staged = true;
    return FSB_OK;
}

// ------------------------------------------------------------------------------------------------
// The kernels of one sub-batch on one lane: K1 ingest -> sort -> layout -> K4 place.  `ev` (FSB_STAGE_COUNT + 1
// events, or null) brackets the stages; `R1` / `R4`: block granularity of K1 / K4 (0 = persistent grids).
int run_sub(fsb_ctx* c, Batch& b, const Sub& sb, fsb_ctx::Lane& L, cudaEvent_t* ev, uint32_t R1, uint32_t R4)
{
    cudaStream_t st = L.st;
    const uint64_t n = sb.r1 - sb.r0;
    const DeviceParams& P = c->dp;
    uint64_t launches = 0;
    if (ev) CUDA_TRY(c, cudaEventRecord(ev[0], st));

    const BatchView B = sub_view(b, sb);
    const uint32_t sub_chunks = sb.c1 - sb.c0;
    const unsigned tpb = 256;
    const unsigned grid_n = (unsigned)std::max<uint64_t>(1, (n + tpb - 1) / tpb);

    // digit plan of the sort; K1 counts the first pass's digits while it writes the keys (scan_sort.cuh, ingest.cuh: SortSeed)
    int width[8];
    const int passes = sort_plan((int)c->dp.key_bits, width);
    const bool seeded = c->fused_hist && n && sub_chunks <= 32u;
    SortSeed seed{nullptr, nullptr, 0, 0, (uint32_t)kSortTile};
    if (seeded)
    {
        seed.counts = L.d_counts.as<uint32_t>();
        seed.chunk_tiles = b.d_chunk_tiles.as<uint32_t>() + sb.ctile_off;
        seed.radix = 1u << width[0]; seed.mask = seed.radix - 1u;
        CUDA_TRY(c, cudaMemsetAsync(L.d_counts.p, 0, (size_t)seed.radix * sb.n_tiles * 4, st));
    }
    // ---- K1: ingest (signature + prepacked slots) -----------------------------------------------------------
    if (n)
    {
        uint32_t* keys = L.d_keys[0].as<uint32_t>();
        unsigned long long* cards = L.d_cards[0].as<unsigned long long>();
        uint32_t* slots = L.d_slots.as<uint32_t>();
        uint32_t* sig = c->per_read ? b.d_sig.as<uint32_t>() + sb.r0 : nullptr;
        uint32_t* info = c->per_read ? b.d_info.as<uint32_t>() + sb.r0 : nullptr;
        const SlotGeom& G = b.geom;
        cudaError_t e = cudaSuccess;
        switch ((b.max_len + 31) / 32)              // words of 32 bases per mate
        {
        case 0: case 1: e = launch_ingest<1>(B, P, G, b.max_head, R1, keys, cards, slots, sig, info, seed, st); break;
        case 2: e = launch_ingest<2>(B, P, G, b.max_head, R1, keys, cards, slots, sig, info, seed, st); break;
        case 3: e = launch_ingest<3>(B, P, G, b.max_head, R1, keys, cards, slots, sig, info, seed, st); break;
        case 4: e = launch_ingest<4>(B, P, G, b.max_head, R1, keys, cards, slots, sig, info, seed, st); break;
        case 5: e = launch_ingest<5>(B, P, G, b.max_head, R1, keys, cards, slots, sig, info, seed, st); break;
        case 6: e = launch_ingest<6>(B, P, G, b.max_head, R1, keys, cards, slots, sig, info, seed, st); break;
        case 7: e = launch_ingest<7>(B, P, G, b.max_head, R1, keys, cards, slots, sig, info, seed, st); break;
        default: e = launch_ingest<8>(B, P, G, b.max_head, R1, keys, cards, slots, sig, info, seed, st); break;
        }
        CUDA_TRY(c, e);
        launches++;
    }
    if (ev) CUDA_TRY(c, cudaEventRecord(ev[1], st));

    // ---- K2/K3: stable radix sort of the signatures inside every chunk segment (card as value) -------------------
    int cur = 0;
    if (n)
    {
        const SortTile* tiles = b.d_sort_tiles.as<SortTile>() + sb.tile_off;
        const uint32_t nblocks = (uint32_t)sb.n_tiles;
        int shift = 0;
        bool counted = seeded;                                       // the pass's digit counts are in d_counts already
        for (int pass = 0; pass < passes; ++pass)
        {
            const uint32_t radix = 1u << width[pass], mask = radix - 1u;
            const uint64_t ncounts = (uint64_t)radix * nblocks;
            if (!counted)
            {
                sort_histogram<<<nblocks, kSortThreads, 0, st>>>(L.d_keys[cur].as<uint32_t>(), tiles, shift, mask, radix, L.d_counts.as<uint32_t>());
                launches++;
            }
            launches += exclusive_scan<uint32_t, uint32_t>(L.d_counts.as<uint32_t>(), ncounts, L.d_counts_scan.as<uint32_t>(), L.d_scan_tmp.as<uint32_t>(), st);
            // the scatter counts the digits of the next pass: a key's destination is the tile it will be read from
            const bool count_next = c->fused_hist && pass + 1 < passes;
            const uint32_t next_radix = count_next ? (1u << width[pass + 1]) : 0u;
            if (count_next) CUDA_TRY(c, cudaMemsetAsync(L.d_counts.p, 0, (size_t)next_radix * nblocks * 4, st));
            CUDA_TRY(c, cudaFuncSetAttribute(sort_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SortScatterSmem)));
            sort_scatter<<<nblocks, kSortThreads, sizeof(SortScatterSmem), st>>>(L.d_keys[cur].as<uint32_t>(), L.d_cards[cur].as<unsigned long long>(), tiles, shift, mask, radix,
                                                            L.d_counts_scan.as<uint32_t>(), L.d_keys[cur ^ 1].as<uint32_t>(), L.d_cards[cur ^ 1].as<unsigned long long>(),
                                                            count_next ? L.d_counts.as<uint32_t>() : nullptr, shift + width[pass], next_radix ? next_radix - 1u : 0u, next_radix);
            counted = count_next;
            shift += width[pass];
            launches++;
            cur ^= 1;
        }
    }
    const uint32_t* sorted_keys = L.d_keys[cur].as<uint32_t>();
    const unsigned long long* sorted_cards = L.d_cards[cur].as<unsigned long long>();
    if (ev) CUDA_TRY(c, cudaEventRecord(ev[2], st));

    // ---- layout --------------------------------------------------------------------------------------
    SortedView S{sorted_keys, sorted_cards};
    BinArrays A{L.d_bin_of.as<uint32_t>(), L.d_bin_start.as<uint32_t>(), L.d_bin_min.as<uint32_t>(), L.d_bin_max.as<uint32_t>(),
                L.d_raw_dna.as<unsigned long long>(), L.d_raw_head.as<unsigned long long>()};
    StreamScans SC{{L.d_P[0].as<uint64_t>(), L.d_P[1].as<uint64_t>(), L.d_P[2].as<uint64_t>(), L.d_P[3].as<uint64_t>()}};
    BinOffsets BO{{L.d_BO[0].as<uint64_t>(), L.d_BO[1].as<uint64_t>(), L.d_BO[2].as<uint64_t>(), L.d_BO[3].as<uint64_t>()}};
    const bool fused = c->fused_layout && n && b.min_len == b.max_len;      // one read length: the layout is a single scan (layout_core.cuh)
    const uint32_t* nb_ptr = fused ? L.d_nb.as<uint32_t>() : L.d_flags_excl.as<uint32_t>() + n;
    fsb_bin_descriptor* desc = b.d_desc.as<fsb_bin_descriptor>() + sb.bin_off;
    OutStreams O{{reinterpret_cast<uint32_t*>(b.d_out[0].as<uint8_t>() + sb.out_off[0]), reinterpret_cast<uint32_t*>(b.d_out[1].as<uint8_t>() + sb.out_off[1]),
                  reinterpret_cast<uint32_t*>(b.d_out[2].as<uint8_t>() + sb.out_off[2]), reinterpret_cast<uint32_t*>(b.d_out[3].as<uint8_t>() + sb.out_off[3])}};
    // the placement tables take the arrays of the per-read bit lengths and the bin flags
    Placement pm{{L.d_bits[0].as<uint32_t>(), L.d_bits[1].as<uint32_t>(), L.d_bits[2].as<uint32_t>(), L.d_bits[3].as<uint32_t>()},
                 L.d_flags.as<uint32_t>(), L.d_tbase.as<unsigned long long>()};
    if (fused)
    {
        const unsigned nlay = (unsigned)((n + kLayBlock - 1) / kLayBlock);
        LayState* states = L.d_lay_states.as<LayState>();
        ChunkStart* cstart = L.d_chunk_start.as<ChunkStart>();
        CUDA_TRY(c, cudaFuncSetAttribute(lay_reduce_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLayReduceSmem));
        CUDA_TRY(c, cudaFuncSetAttribute(lay_apply_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLayApplySmem));
        lay_reduce_kernel<<<nlay, kLayThreads, kLayReduceSmem, st>>>(n, P, S, b.min_len, states);
        const unsigned ngroups = (nlay + kLayScanThreads - 1) / kLayScanThreads;
        lay_scan_groups_kernel<<<ngroups, kLayScanThreads, 0, st>>>(states, nlay, states + nlay + 1);
        lay_scan_finish_kernel<<<ngroups, kLayScanThreads, 0, st>>>(states, nlay, states + nlay + 1);
        lay_apply_kernel<<<nlay, kLayThreads, kLayApplySmem, st>>>(n, sub_chunks, P, S, b.min_len, states, LayOut{pm, O, desc, cstart, L.d_nb.as<uint32_t>()});
        chunk_summary_fused_kernel<<<sub_chunks, 128, 0, st>>>(B, cstart, desc, b.d_summary.as<ChunkSummary>() + sb.c0);
        launches += 5;
    }
    else
    {
        const uint64_t nbm = sb.nb_max;
        CUDA_TRY(c, cudaMemsetAsync(L.d_bin_min.p, 0xFF, (nbm + 1) * 4, st));
        CUDA_TRY(c, cudaMemsetAsync(L.d_bin_max.p, 0, (nbm + 1) * 4, st));
        CUDA_TRY(c, cudaMemsetAsync(L.d_raw_dna.p, 0, (nbm + 1) * 8, st));
        CUDA_TRY(c, cudaMemsetAsync(L.d_raw_head.p, 0, (nbm + 1) * 8, st));
        if (n)
        {
            bin_flags_kernel<<<grid_n, tpb, 0, st>>>(sorted_keys, n, L.d_flags.as<uint32_t>());
            launches++;
        }
        launches += exclusive_scan<uint32_t, uint32_t>(L.d_flags.as<uint32_t>(), n, L.d_flags_excl.as<uint32_t>(), L.d_scan_tmp.as<uint32_t>(), st);
        if (n)
        {
            bin_stats_kernel<<<grid_n, tpb, 0, st>>>(n, P, S, L.d_flags.as<uint32_t>(), L.d_flags_excl.as<uint32_t>(), A);
            read_bits_kernel<<<grid_n, tpb, 0, st>>>(n, P, S, A, L.d_bits[0].as<uint32_t>(), L.d_bits[1].as<uint32_t>(), L.d_bits[2].as<uint32_t>(),
                                                      L.d_bits[3].as<uint32_t>());
            launches += 2;
        }
        {
            Ptr4<const uint32_t> in4{{L.d_bits[0].as<uint32_t>(), L.d_bits[1].as<uint32_t>(), L.d_bits[2].as<uint32_t>(), L.d_bits[3].as<uint32_t>()}};
            Ptr4<uint64_t> out4{{L.d_P[0].as<uint64_t>(), L.d_P[1].as<uint64_t>(), L.d_P[2].as<uint64_t>(), L.d_P[3].as<uint64_t>()}};
            launches += exclusive_scan4<uint32_t, uint64_t>(in4, n, out4, L.d_scan_tmp.as<uint64_t>(), st);
        }
        if (nbm)
        {
            const unsigned grid_b = (unsigned)((nbm + tpb - 1) / tpb);
            bin_sizes_kernel<<<grid_b, tpb, 0, st>>>(P, n, nb_ptr, nbm, sorted_keys, A, SC, L.d_bytes[0].as<uint64_t>(), L.d_bytes[1].as<uint64_t>(),
                                                      L.d_bytes[2].as<uint64_t>(), L.d_bytes[3].as<uint64_t>(), desc);
            launches++;
        }
        {
            Ptr4<const uint64_t> in4{{L.d_bytes[0].as<uint64_t>(), L.d_bytes[1].as<uint64_t>(), L.d_bytes[2].as<uint64_t>(), L.d_bytes[3].as<uint64_t>()}};
            Ptr4<uint64_t> out4{{L.d_BO[0].as<uint64_t>(), L.d_BO[1].as<uint64_t>(), L.d_BO[2].as<uint64_t>(), L.d_BO[3].as<uint64_t>()}};
            launches += exclusive_scan4<uint64_t, uint64_t>(in4, nbm, out4, L.d_scan_tmp.as<uint64_t>(), st);
        }
        chunk_summary_kernel<<<sub_chunks, 128, 0, st>>>(B, nb_ptr, A.bin_of, BO, desc, b.d_summary.as<ChunkSummary>() + sb.c0);
        launches++;
    }
    if (ev) CUDA_TRY(c, cudaEventRecord(ev[3], st));

    // ---- K4: place ------------------------------------------------------------------------------------
    if (n)
    {
        PlaceArgs pa{B, P, b.geom, S, A, SC, BO, O, L.d_slots.as<uint32_t>(), nb_ptr};
        int place_launches = 0;
        CUDA_TRY(c, launch_place(pa, pm, b.max_len, b.max_head, R4, fused, st, &place_launches));
        launches += place_launches;
    }
    if (ev) CUDA_TRY(c, cudaEventRecord(ev[4], st));
    CUDA_TRY(c, cudaGetLastError());
    c->stats.kernel_launches += launches;
    c->stats.records += n;
    return FSB_OK;
}

// The kernels of one batch.  A batch staged as one sub-batch runs on the context's stream with persistent K1 / K4 grids.
// Several sub-batches alternate between the two lanes (sub-batch j on lane j mod 2): lane 1's stream forks from the
// context's stream and joins it again, so callers still see one stream; K1 and K4 then run with block-sized work units
// and the hardware interleaves the blocks of whatever kernels the two lanes have in flight.
int run_enqueue(fsb_ctx* c, Batch& b, bool profile)
{
    // FSB_OPT_PROFILE times the stages of an unsplit run: sub-batches that exist only because a batch holds more than 32 chunks
    // then follow each other on one stream, each with its own events
    const bool timed = profile && b.split <= 1;
    const bool split = b.subs.size() > 1 && !timed;
    if (timed)
    {
        if (c->pending_profiles + (int)b.subs.size() > kMaxPendingProfiles) { int rc = resolve_profiles(c); if (rc != FSB_OK) return rc; }
        const size_t need = (size_t)(c->pending_profiles + b.subs.size()) * (FSB_STAGE_COUNT + 1);
        while (c->events.size() < need) { cudaEvent_t e; CUDA_TRY(c, cudaEventCreate(&e)); c->events.push_back(e); }
        c->pending_first.resize(kMaxPendingProfiles + b.subs.size(), 0);
    }
    if (split)
    {
        CUDA_TRY(c, cudaEventRecord(c->ev_fork, c->stream));
        CUDA_TRY(c, cudaStreamWaitEvent(c->lane[1].st, c->ev_fork, 0));
    }
    for (size_t j = 0; j < b.subs.size(); ++j)
    {
        const bool blocks = split || c->block_grids_always;
        cudaEvent_t* ev = nullptr;
        if (timed)
        {
            ev = &c->events[(size_t)c->pending_profiles * (FSB_STAGE_COUNT + 1)];
            c->pending_first[c->pending_profiles] = j == 0;
        }
        const int rc = run_sub(c, b, b.subs[j], c->lane[split ? (j & 1) : 0], ev, blocks ? c->k1_batches_per_warp : 0u, blocks ? c->k4_tiles_per_block : 0u);
        if (rc != FSB_OK) return rc;
        if (timed) c->pending_profiles++;
    }
    if (split)
    {
        CUDA_TRY(c, cudaEventRecord(c->lane[1].ev_done, c->lane[1].st));
        CUDA_TRY(c, cudaStreamWaitEvent(c->stream, c->lane[1].ev_done, 0));
    }
    b.ran = true;
    return FSB_OK;
}

// ------------------------------------------------------------------------------------------------
// Results, step 1: the per-chunk summary (sizes are only known on the device).
int summary_enqueue(fsb_ctx* c, Batch& b, HostOut& h, cudaStream_t st)
{
    CUDA_TRY(c, h.summary.ensure((size_t)b.n_chunks * sizeof(ChunkSummary)));
    CUDA_TRY(c, small_to_host(h.summary.p, b.d_summary.p, (size_t)b.n_chunks * sizeof(ChunkSummary), st));
    return FSB_OK;
}
// Results, step 2 (summary on the host): enqueue the copies of the streams and descriptors, sub-batch by sub-batch
// (every sub-batch owns a region of the batch's streams and of its descriptor array; the host buffers mirror them).
int fetch_enqueue(fsb_ctx* c, Batch& b, HostOut& h, cudaStream_t st)
{
    const uint64_t n = b.n_records;
    uint64_t d2h = (size_t)b.n_chunks * sizeof(ChunkSummary);
    const ChunkSummary* sum = h.summary.as<ChunkSummary>();
    for (int s = 0; s < 4; ++s) CUDA_TRY(c, h.out[s].ensure(b.out_total[s] + 64));
    CUDA_TRY(c, h.desc.ensure((b.nb_max + 1) * sizeof(fsb_bin_descriptor)));
    for (const Sub& sb : b.subs)
    {
        const ChunkSummary& last = sum[sb.c1 - 1];
        const uint64_t nb = last.first_bin + last.n_bins;
        if (nb > sb.nb_max) return fail(c, FSB_ERR_STATE, "internal error: bin count exceeds its bound");
        for (int s = 0; s < 4; ++s)
        {
            const uint64_t total = last.off[s] + last.size[s];
            if (total > sb.out_cap[s]) return fail(c, FSB_ERR_STATE, "internal error: stream size exceeds its bound");
            if (total) CUDA_TRY(c, cudaMemcpyAsync(h.out[s].as<uint8_t>() + sb.out_off[s], b.d_out[s].as<uint8_t>() + sb.out_off[s], total, cudaMemcpyDeviceToHost, st));
            d2h += total;
        }
        if (nb) CUDA_TRY(c, cudaMemcpyAsync(h.desc.as<fsb_bin_descriptor>() + sb.bin_off, b.d_desc.as<fsb_bin_descriptor>() + sb.bin_off, nb * sizeof(fsb_bin_descriptor),
                                            cudaMemcpyDeviceToHost, st));
        d2h += nb * sizeof(fsb_bin_descriptor);
    }
    if (c->keep_records && b.device_parse)
    {
        for (int m = 0; m < (c->dp.paired ? 2 : 1); ++m)
        {
            CUDA_TRY(c, h.rec[m].ensure((n + 1) * sizeof(fsb_record)));
            if (n) CUDA_TRY(c, cudaMemcpyAsync(h.rec[m].p, b.d_rec[m].p, n * sizeof(fsb_record), cudaMemcpyDeviceToHost, st));
            d2h += n * sizeof(fsb_record);
        }
    }
    if (c->per_read)
    {
        CUDA_TRY(c, h.sig.ensure((n + 1) * 4));
        CUDA_TRY(c, h.info.ensure((n + 1) * 4));
        if (n)
        {
            CUDA_TRY(c, cudaMemcpyAsync(h.sig.p, b.d_sig.p, n * 4, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(c, cudaMemcpyAsync(h.info.p, b.d_info.p, n * 4, cudaMemcpyDeviceToHost, st));
        }
        d2h += 8 * n;
    }
    h.d2h_bytes = d2h;
    c->stats.d2h_bytes += d2h;
    return FSB_OK;
}
// Results, step 3 (copies complete): describe every chunk's block.
void fill_blocks(fsb_ctx* c, const Batch& b, const HostOut& h, fsb_block* blocks)
{
    const ChunkSummary* sum = h.summary.as<ChunkSummary>();
    uint64_t alg_out = 0;
    for (const Sub& sb : b.subs)
        for (uint32_t ci = sb.c0; ci < sb.c1; ++ci)
        {
            const ChunkSummary& s = sum[ci];                     // offsets and bin indices count from the sub-batch's regions
            fsb_block& o = blocks[ci];
            std::memset(&o, 0, sizeof(o));
            o.meta = h.out[0].as<uint8_t>() + sb.out_off[0] + s.off[0]; o.meta_size = s.size[0];
            o.dna = h.out[1].as<uint8_t>() + sb.out_off[1] + s.off[1];  o.dna_size = s.size[1];
            o.qua = h.out[2].as<uint8_t>() + sb.out_off[2] + s.off[2];  o.qua_size = s.size[2];
            o.head = h.out[3].as<uint8_t>() + sb.out_off[3] + s.off[3]; o.head_size = s.size[3];
            o.raw_dna_size = s.raw_dna; o.raw_head_size = s.raw_head;
            o.bins = h.desc.as<fsb_bin_descriptor>() + sb.bin_off + s.first_bin;
            o.n_bins = s.n_bins;
            o.n_records = b.chunk_first_rec[ci + 1] - b.chunk_first_rec[ci];
            if (c->per_read)
            {
                o.read_signature = h.sig.as<uint32_t>() + b.chunk_first_rec[ci];
                o.read_info = h.info.as<uint32_t>() + b.chunk_first_rec[ci];
            }
            alg_out += s.size[0] + s.size[1] + s.size[2] + s.size[3];
        }
    c->stats.algorithmic_bytes += b.algorithmic_in + alg_out;
}

} // namespace

extern "C" int fsb_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    int ok = 0;
    for (int i = 0; i < n; ++i)
    {
        cudaDeviceProp p;
        if (cudaGetDeviceProperties(&p, i) == cudaSuccess && p.major == 10) ok++;
    }
    return ok;
}

extern "C" const char* fsb_last_error(const fsb_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

extern "C" int fsb_create(const fsb_params* p, int device, void* cuda_stream, fsb_ctx** out)
{
    if (!p || !out) return fail(nullptr, FSB_ERR_PARAM, "fsb_create: null argument");
    *out = nullptr;
    // MinimizerParameters (Params.h:22-96): k <= 15 because TotalMinimizersCount() is 1 << 2k in an int (:55-58);
    // k >= 3 because the AAA/AAC test shifts by 2k-6 (FastqCategorizer.cpp:56)
    if (p->signature_len < 3 || p->signature_len > 15) return fail(nullptr, FSB_ERR_PARAM, "signature_len must be in [3, 15]");
    if (p->signature_mask_cutoff_bits >= 2 * p->signature_len) return fail(nullptr, FSB_ERR_PARAM, "signature_mask_cutoff_bits too large");
    if (std::memcmp(p->dna_symbol_order, "ACGTN", 5) != 0) return fail(nullptr, FSB_ERR_PARAM, "only dna_symbol_order \"ACGTN\" is supported");
    if (p->quality_method > FSB_QUA_QVZ) return fail(nullptr, FSB_ERR_PARAM, "quality_method must be 0..3");
    if (p->quality_method == FSB_QUA_BINARY && p->binary_threshold >= 64) return fail(nullptr, FSB_ERR_PARAM, "binary_threshold must be < 64");
    // the byte check and the quality coding work on q - offset per byte with bit 7 as a borrow guard (stage_core.cuh, pack_core.cuh)
    if (p->quality_offset > 127) return fail(nullptr, FSB_ERR_PARAM, "quality_offset must be in [0, 127]");

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(nullptr, FSB_ERR_CUDA, "no CUDA device available (this library has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(nullptr, FSB_ERR_PARAM, "device index out of range");
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10)
        return fail(nullptr, FSB_ERR_CUDA, "device is not sm_100 (kernels are built for sm_100a only)");

    fsb_ctx* c = new (std::nothrow) fsb_ctx();
    if (!c) return fail(nullptr, FSB_ERR_NOMEM, "out of host memory");
    c->params = *p;
    c->device = device;
    c->dp = make_device_params(*p);

    if (cudaSetDevice(device) != cudaSuccess) { delete c; return fail(nullptr, FSB_ERR_CUDA, "cudaSetDevice failed"); }
    if (cuda_stream) { c->stream = (cudaStream_t)cuda_stream; c->own_stream = false; }
    else
    {
        if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return fail(nullptr, FSB_ERR_CUDA, "cudaStreamCreate failed"); }
        c->own_stream = true;
    }
    c->lane[0].st = c->stream; c->lane[0].own = false;
    if (cudaEventCreateWithFlags(&c->lane[0].ev_done, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) != cudaSuccess)
    {
        fsb_destroy(c);
        return fail(nullptr, FSB_ERR_CUDA, "cudaEventCreate failed");
    }
    // tuning knobs for experiments (the defaults are what the measurements in DESIGN.md chose)
    if (const char* e = std::getenv("FSB_RUN_SPLIT")) c->run_split = (uint32_t)std::max(1, std::atoi(e));
    if (const char* e = std::getenv("FSB_K1_R")) c->k1_batches_per_warp = (uint32_t)std::max(0, std::atoi(e));
    if (const char* e = std::getenv("FSB_K4_R")) c->k4_tiles_per_block = (uint32_t)std::max(0, std::atoi(e));
    for (Batch& b : c->batch)
    {
        if (cudaEventCreateWithFlags(&b.ev_h2d, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&b.ev_chk, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&b.ev_run, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&b.ev_parse, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&b.ev_d2h, cudaEventDisableTiming) != cudaSuccess)
        {
            fsb_destroy(c);
            return fail(nullptr, FSB_ERR_CUDA, "cudaEventCreate failed");
        }
    }
    *out = c;
    return FSB_OK;
}

extern "C" void fsb_destroy(fsb_ctx* c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    if (c->s_h2d) { cudaStreamSynchronize(c->s_h2d); cudaStreamDestroy(c->s_h2d); }
    if (c->s_d2h) { cudaStreamSynchronize(c->s_d2h); cudaStreamDestroy(c->s_d2h); }
    for (cudaStream_t& q : c->s_chk) if (q) { cudaStreamSynchronize(q); cudaStreamDestroy(q); q = nullptr; }
    for (auto& e : c->events) cudaEventDestroy(e);
    for (cudaEvent_t e : c->ev_check) if (e) cudaEventDestroy(e);
    for (Batch& b : c->batch)
    {
        DevBuf* dev[] = {&b.d_text[0], &b.d_text[1], &b.d_rec[0], &b.d_rec[1], &b.d_chunk_meta, &b.d_stage_stats, &b.d_chunk_sums, &b.d_sort_tiles, &b.d_chunk_tiles, &b.d_out[0], &b.d_out[1], &b.d_out[2], &b.d_out[3],
                         &b.d_desc, &b.d_summary, &b.d_sig, &b.d_info};
        for (DevBuf* d : dev) d->release();
        b.h_stage_stats.release(); b.h_chunk_sums.release(); b.h_up.release();
        if (b.ev_h2d) cudaEventDestroy(b.ev_h2d);
        if (b.ev_chk) cudaEventDestroy(b.ev_chk);
        if (b.ev_parse) cudaEventDestroy(b.ev_parse);
        b.d_segs.release(); b.d_tile_count.release(); b.d_end_mask.release(); b.d_tile_prefix.release(); b.d_line_start.release(); b.d_parse_res.release(); b.d_seg_ends.release(); b.d_rec_tmp.release(); b.d_parse_scan_tmp.release();
        b.h_seg_ends.release(); b.h_parse_res.release();
        if (b.ev_run) cudaEventDestroy(b.ev_run);
        if (b.ev_d2h) cudaEventDestroy(b.ev_d2h);
    }
    for (fsb_ctx::Lane& L : c->lane)
    {
        if (L.st && L.own) cudaStreamSynchronize(L.st);
        L.each([](DevBuf& d) { d.release(); });
        if (L.ev_done) cudaEventDestroy(L.ev_done);
        if (L.st && L.own) cudaStreamDestroy(L.st);
    }
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    for (HostOut* h : c->host)
    {
        if (!h) continue;
        PinBuf* pin[] = {&h->out[0], &h->out[1], &h->out[2], &h->out[3], &h->desc, &h->summary, &h->sig, &h->info, &h->rec[0], &h->rec[1]};
        for (PinBuf* q : pin) q->release();
        delete h;
    }
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete c;
}

extern "C" int fsb_set_option(fsb_ctx* c, int option, int64_t value)
{
    if (!c) return FSB_ERR_PARAM;
    switch (option)
    {
    case FSB_OPT_PER_READ: c->per_read = value != 0; return FSB_OK;
    case FSB_OPT_PROFILE: c->profile = value != 0; return FSB_OK;
    case FSB_OPT_VALIDATE: c->validate = value != 0; return FSB_OK;
    case FSB_OPT_SUBBATCH_RECORDS: c->sub_batch_records = value > 0 ? (uint64_t)value : 1; return FSB_OK;
    case FSB_OPT_RUN_SPLIT: c->run_split = value > 0 ? (uint32_t)std::min<int64_t>(value, 64) : 1; return FSB_OK;
    case FSB_OPT_K1_BLOCK_BATCHES: c->k1_batches_per_warp = (uint32_t)std::max<int64_t>(0, std::min<int64_t>(value, 1 << 20)); return FSB_OK;
    case FSB_OPT_K4_BLOCK_TILES: c->k4_tiles_per_block = (uint32_t)std::max<int64_t>(0, std::min<int64_t>(value, 1 << 20)); return FSB_OK;
    case FSB_OPT_BLOCK_GRIDS_ALWAYS: c->block_grids_always = value != 0; return FSB_OK;
    case FSB_OPT_FUSED_LAYOUT: c->fused_layout = value != 0; return FSB_OK;
    case FSB_OPT_KEEP_COMMENTS: c->keep_comments = value != 0; return FSB_OK;
    case FSB_OPT_KEEP_RECORDS: c->keep_records = value != 0; return FSB_OK;
    case FSB_OPT_FUSED_HIST: c->fused_hist = value != 0; return FSB_OK;
    }
    return fail(c, FSB_ERR_PARAM, "unknown option");
}

extern "C" void* fsb_host_alloc(size_t bytes)
{
    return pinned_alloc(bytes);
}
extern "C" void fsb_host_free(void* p) { pinned_free(p); }

extern "C" int fsb_sync(fsb_ctx* c)
{
    if (!c) return FSB_ERR_PARAM;
    CUDA_TRY(c, cudaSetDevice(c->device));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return FSB_OK;
}

extern "C" int fsb_get_stats(const fsb_ctx* c, fsb_stats* out)
{
    if (!c || !out) return FSB_ERR_PARAM;
    *out = c->stats;
    return FSB_OK;
}

extern "C" int fsb_stage_times(fsb_ctx* c, float* ms, uint32_t n_stages, uint32_t* n_runs)
{
    if (!c || !ms) return FSB_ERR_PARAM;
    CUDA_TRY(c, cudaSetDevice(c->device));
    int rc = resolve_profiles(c);
    if (rc != FSB_OK) return rc;
    if (c->check_pending)
    {
        CUDA_TRY(c, cudaEventSynchronize(c->ev_check[1]));
        float t = 0;
        CUDA_TRY(c, cudaEventElapsedTime(&t, c->ev_check[0], c->ev_check[1]));
        c->check_ms += t;
        c->check_pending = false;
    }
    for (uint32_t s = 0; s < n_stages; ++s) ms[s] = s < FSB_STAGE_COUNT ? c->stage_ms[s] : (s == FSB_STAGE_CHECK ? c->check_ms : 0.f);
    c->check_ms = 0;
    if (n_runs) *n_runs = c->stage_runs;
    for (int s = 0; s < FSB_STAGE_COUNT; ++s) c->stage_ms[s] = 0;
    c->stage_runs = 0;
    return FSB_OK;
}

// ---- the resident interface: one batch, everything on the context's stream ---------------------------------
extern "C" int fsb_stage(fsb_ctx* c, const fsb_chunk* chunks, uint32_t n_chunks)
{
    if (!c || (!chunks && n_chunks)) return FSB_ERR_PARAM;
    CUDA_TRY(c, cudaSetDevice(c->device));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));               // nothing may still be using the batch's buffers
    Batch& b = c->batch[0];
    int rc = stage_enqueue(c, b, chunks, n_chunks, 0, c->stream, c->stream, c->run_split, c->profile);
    while (rc == FSB_OK && b.parse_state) rc = stage_advance(c, b, c->stream);      // device-side parse: two more steps, each sized by the one before
    if (rc != FSB_OK) return rc;
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));               // pageable user buffers must outlive the copies; the statistics are back
    return stage_complete(c, b);
}

extern "C" int fsb_run(fsb_ctx* c)
{
    if (!c) return FSB_ERR_PARAM;
    if (!c->batch[0].staged) return fail(c, FSB_ERR_STATE, "fsb_run: nothing staged");
    CUDA_TRY(c, cudaSetDevice(c->device));
    return run_enqueue(c, c->batch[0], c->profile);
}

extern "C" int fsb_fetch(fsb_ctx* c, fsb_block* blocks, uint32_t n_blocks)
{
    if (!c || !blocks) return FSB_ERR_PARAM;
    Batch& b = c->batch[0];
    if (!b.ran) return fail(c, FSB_ERR_STATE, "fsb_fetch: fsb_run has not been called on the staged batch");
    if (n_blocks != b.n_chunks) return fail(c, FSB_ERR_PARAM, "fsb_fetch: n_blocks must equal the number of staged chunks");
    CUDA_TRY(c, cudaSetDevice(c->device));
    HostOut* h = host_out(c, 0);
    if (!h) return fail(c, FSB_ERR_NOMEM, "out of host memory");
    int rc = summary_enqueue(c, b, *h, c->stream);
    if (rc != FSB_OK) return rc;
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    rc = fetch_enqueue(c, b, *h, c->stream);
    if (rc != FSB_OK) return rc;
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    fill_blocks(c, b, *h, blocks);
    return FSB_OK;
}

extern "C" int fsb_get_records(fsb_ctx* c, uint32_t chunk, int mate, fsb_record* dst, uint64_t capacity, uint64_t* n_records)
{
    if (!c || !n_records || mate < 0 || mate > 1 || (mate == 1 && !c->dp.paired)) return FSB_ERR_PARAM;
    *n_records = 0;
    if (chunk < c->rec_index.size() && c->rec_index[chunk].host[mate])
    {   // tables copied back by the last fsb_bin_chunks call
        const fsb_ctx::RecRef& rr = c->rec_index[chunk];
        *n_records = rr.n;
        if (rr.n > capacity || (rr.n && !dst)) return fail(c, FSB_ERR_PARAM, "fsb_get_records: destination too small");
        if (rr.n) std::memcpy(dst, rr.host[mate], rr.n * sizeof(fsb_record));
        return FSB_OK;
    }
    Batch& b = c->batch[0];
    if (!b.staged || !b.device_parse || chunk >= b.n_chunks) return fail(c, FSB_ERR_STATE, "fsb_get_records: no device-side parse result for this chunk");
    const uint64_t first = b.chunk_first_rec[chunk], n = b.chunk_first_rec[chunk + 1] - first;
    *n_records = n;
    if (n > capacity || (n && !dst)) return fail(c, FSB_ERR_PARAM, "fsb_get_records: destination too small");
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (n) CUDA_TRY(c, cudaMemcpy(dst, b.d_rec[mate].as<fsb_record>() + first, n * sizeof(fsb_record), cudaMemcpyDeviceToHost));
    return FSB_OK;
}

// ---- fastore_rebin's signature scan (SURVEY 8f-3) ---------------------------------------------------------------------------
namespace {
template <int NW>
void launch_new_minimizer(const uint8_t* text, const fsb_record* rec, uint64_t n, const DeviceParams& P, uint32_t cur, uint32_t* sig, uint32_t* info, cudaStream_t st)
{
    find_new_minimizer_kernel<NW><<<(unsigned)((n + 127) / 128), 128, 0, st>>>(text, rec, n, P, cur, sig, info);
}
} // namespace

extern "C" int fsb_find_new_minimizers(fsb_ctx* c, const uint8_t* text, uint64_t text_size, const fsb_record* records, uint64_t n_records,
                                       uint32_t cur_signature, uint32_t signature_parity, uint32_t* signature, uint32_t* info)
{
    if (!c || (n_records && (!text || !records || !signature || !info))) return FSB_ERR_PARAM;
    if (signature_parity < 2 || (signature_parity & (signature_parity - 1)) != 0 || signature_parity > c->dp.nbin)
        return fail(c, FSB_ERR_PARAM, "fsb_find_new_minimizers: signature_parity must be a power of two in [2, 4^k]");
    if (text_size >= 0xFFFFFFFFull) return fail(c, FSB_ERR_INPUT, "fsb_find_new_minimizers: text must be < 4 GiB (32-bit record offsets)");
    if (n_records == 0) return FSB_OK;
    uint32_t max_len = 0;
    for (uint64_t i = 0; i < n_records; ++i)
    {
        const fsb_record& r = records[i];
        if (r.seq_len < 1 || r.seq_len > 255 || (uint64_t)r.seq_off + r.seq_len > text_size)
            return fail(c, FSB_ERR_INPUT, "fsb_find_new_minimizers: record " + std::to_string(i) + " violates the input contract (length 1..255, offsets inside the text)");
        max_len = std::max<uint32_t>(max_len, r.seq_len);
    }
    CUDA_TRY(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    CUDA_TRY(c, cudaStreamSynchronize(st));
    fsb_ctx::Lane& L = c->lane[0];                                   // scratch: the lane's key arrays take the results
    DevBuf d_text, d_rec;
    CUDA_TRY(c, d_text.ensure(text_size + 2 * kTextPad, &st));
    int rc = FSB_OK;
    auto done = [&](int code) { d_text.release(); d_rec.release(); return code; };
    if (d_rec.ensure(n_records * sizeof(fsb_record)) != cudaSuccess) return done(fail(c, FSB_ERR_NOMEM, "out of device memory"));
    if (ensure_shared(st, L.d_keys[0], (n_records + 1) * 4) != cudaSuccess || ensure_shared(st, L.d_keys[1], (n_records + 1) * 4) != cudaSuccess)
        return done(fail(c, FSB_ERR_NOMEM, "out of device memory"));
    DeviceParams P = c->dp;
    uint32_t lg = 0;
    while ((1u << lg) < signature_parity) ++lg;
    P.cutoff_bits = std::max(P.cutoff_bits, lg);                     // m % divisor == 0: the low log2(divisor) bits are zero
    cudaMemcpyAsync(d_text.as<uint8_t>(), text, text_size, cudaMemcpyHostToDevice, st);
    cudaMemcpyAsync(d_rec.p, records, n_records * sizeof(fsb_record), cudaMemcpyHostToDevice, st);
    uint32_t* d_sig = L.d_keys[0].as<uint32_t>();
    uint32_t* d_info = L.d_keys[1].as<uint32_t>();
    switch ((max_len + 31) / 32)
    {
    case 0: case 1: launch_new_minimizer<1>(d_text.as<uint8_t>(), d_rec.as<fsb_record>(), n_records, P, cur_signature, d_sig, d_info, st); break;
    case 2: launch_new_minimizer<2>(d_text.as<uint8_t>(), d_rec.as<fsb_record>(), n_records, P, cur_signature, d_sig, d_info, st); break;
    case 3: launch_new_minimizer<3>(d_text.as<uint8_t>(), d_rec.as<fsb_record>(), n_records, P, cur_signature, d_sig, d_info, st); break;
    case 4: launch_new_minimizer<4>(d_text.as<uint8_t>(), d_rec.as<fsb_record>(), n_records, P, cur_signature, d_sig, d_info, st); break;
    case 5: launch_new_minimizer<5>(d_text.as<uint8_t>(), d_rec.as<fsb_record>(), n_records, P, cur_signature, d_sig, d_info, st); break;
    case 6: launch_new_minimizer<6>(d_text.as<uint8_t>(), d_rec.as<fsb_record>(), n_records, P, cur_signature, d_sig, d_info, st); break;
    case 7: launch_new_minimizer<7>(d_text.as<uint8_t>(), d_rec.as<fsb_record>(), n_records, P, cur_signature, d_sig, d_info, st); break;
    default: launch_new_minimizer<8>(d_text.as<uint8_t>(), d_rec.as<fsb_record>(), n_records, P, cur_signature, d_sig, d_info, st); break;
    }
    c->stats.kernel_launches++;
    cudaMemcpyAsync(signature, d_sig, n_records * 4, cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(info, d_info, n_records * 4, cudaMemcpyDeviceToHost, st);
    const cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = fail(c, FSB_ERR_CUDA, std::string("fsb_find_new_minimizers: ") + cudaGetErrorString(e));
    return done(rc);
}

// ---- host buffers in, host blocks out ----------------------------------------------------------------------------
// The chunk list is cut into sub-batches of at least sub_batch_records records (whole chunks) which
// run as a pipeline over three sets of device buffers:
//     s_h2d   : copies in of g+1, g+2 ... back to back (a set is reused once the kernels that read it are done)
//     s_chk[] : input check (and device-side parse) of every sub-batch as soon as its copy has landed; one stream per buffer set,
//               because the parse of sub-batch g is enqueued in steps, and on a shared stream its later steps would sit behind
//               the wait for the text of g+1 that stage_enqueue(g+1) has already put there
//     stream  : kernels of g (the host has seen g's check results, and that copy out g-3 has released the result buffers)
//     s_d2h   : copy out g-1
// Two sub-batches are always staged ahead, so the copy stream -- the PCIe link is what bounds this call -- never waits for
// the host.  The host only blocks on small things: the check results of a sub-batch (they size the buffers and carry the
// input validation) and its chunk summary (the stream sizes).
extern "C" int fsb_bin_chunks(fsb_ctx* c, const fsb_chunk* chunks, uint32_t n_chunks, fsb_block* blocks)
{
    if (!c || !blocks || (!chunks && n_chunks)) return FSB_ERR_PARAM;
    if (n_chunks == 0) return fail(c, FSB_ERR_PARAM, "fsb_bin_chunks: no chunks");
    CUDA_TRY(c, cudaSetDevice(c->device));

    // sub-batches: [first[g], first[g + 1])
    const uint32_t max_chunks = (uint32_t)std::min<uint64_t>(kMaxChunksPerBatch, 1ull << (32 - c->dp.key_bits));
    std::vector<uint32_t> first{0};
    {
        uint64_t recs = 0;
        for (uint32_t ci = 0; ci < n_chunks; ++ci)
        {
            const uint64_t est = chunks[ci].records[0] ? chunks[ci].n_records : chunks[ci].text_size[0] / 8u;       // at most a record per 8 bytes
            if (ci > first.back() && (recs >= c->sub_batch_records || ci - first.back() >= max_chunks || recs + est > kMaxBatchRecords))
            {
                first.push_back(ci);
                recs = 0;
            }
            // (chunks to be parsed on the device: about one record per 250 bytes of text)
            recs += chunks[ci].records[0] ? chunks[ci].n_records : chunks[ci].text_size[0] / 250u;
        }
        first.push_back(n_chunks);
    }
    const uint32_t G = (uint32_t)first.size() - 1;
    const CallTrace trace;
    struct TraceScope { fsb_ctx* c; ~TraceScope() { c->trace = nullptr; } } trace_scope{c};
    c->trace = &trace;
    if (!c->s_h2d) CUDA_TRY(c, cudaStreamCreateWithFlags(&c->s_h2d, cudaStreamNonBlocking));
    if (!c->s_d2h) CUDA_TRY(c, cudaStreamCreateWithFlags(&c->s_d2h, cudaStreamNonBlocking));
    for (cudaStream_t& q : c->s_chk) if (!q) CUDA_TRY(c, cudaStreamCreateWithFlags(&q, cudaStreamNonBlocking));
    constexpr uint32_t kSets = 3, kAhead = 2;
    auto set_of = [&](uint32_t g) -> Batch& { return c->batch[g % kSets]; };
    for (uint32_t g = 0; g < G; ++g) if (!host_out(c, g)) return fail(c, FSB_ERR_NOMEM, "out of host memory");
    trace.mark("host sets ready", G);
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));               // earlier work on the context (resident interface) is done
    CUDA_TRY(c, cudaStreamSynchronize(c->s_d2h));

    int rc = FSB_OK;
    auto drain = [&]() { cudaStreamSynchronize(c->s_h2d); for (cudaStream_t q : c->s_chk) cudaStreamSynchronize(q); cudaStreamSynchronize(c->stream); cudaStreamSynchronize(c->s_d2h); };
    // copy out of sub-batch g: its summary is on the host once ev_run has fired
    auto finish = [&](uint32_t g) -> int
    {
        Batch& b = set_of(g);
        CUDA_TRY(c, cudaEventSynchronize(b.ev_run));
        CUDA_TRY(c, cudaStreamWaitEvent(c->s_d2h, b.ev_run, 0));
        int r = fetch_enqueue(c, b, *c->host[g], c->s_d2h);
        if (r != FSB_OK) return r;
        CUDA_TRY(c, cudaEventRecord(b.ev_d2h, c->s_d2h));
        // the batch object is reused three sub-batches later: describe the blocks now (the pointers are final,
        // the bytes arrive before the call returns)
        fill_blocks(c, b, *c->host[g], blocks + first[g]);
        if (c->keep_records && b.device_parse)
            for (uint32_t ci = 0; ci < b.n_chunks; ++ci)
            {
                fsb_ctx::RecRef& rr = c->rec_index[first[g] + ci];
                rr.n = b.chunk_first_rec[ci + 1] - b.chunk_first_rec[ci];
                for (int m = 0; m < 2; ++m) rr.host[m] = c->host[g]->rec[m].p ? c->host[g]->rec[m].as<fsb_record>() + b.chunk_first_rec[ci] : nullptr;
            }
        return FSB_OK;
    };
    c->rec_index.assign(c->keep_records ? n_chunks : 0, fsb_ctx::RecRef{{nullptr, nullptr}, 0});

    for (uint32_t g = 0; g < std::min(G, kAhead) && rc == FSB_OK; ++g)
        rc = stage_enqueue(c, set_of(g), chunks + first[g], first[g + 1] - first[g], first[g], c->s_h2d, c->s_chk[g % kSets], 1);
    trace.mark("first copies enqueued", 0);
    for (uint32_t g = 0; g < G && rc == FSB_OK; ++g)
    {
        Batch& b = set_of(g);
        while (rc == FSB_OK && b.parse_state) rc = stage_advance(c, b, c->s_chk[g % kSets]);     // device-side parse: the steps behind the copy
        if (rc != FSB_OK) break;
        trace.mark("parsed", g);
        if (cudaEventSynchronize(b.ev_chk) != cudaSuccess) { rc = fail(c, FSB_ERR_CUDA, "copy to the device failed"); break; }    // text on the device, check results on the host
        trace.mark("text on the device, checked", g);
        if (g >= kSets && cudaEventSynchronize(b.ev_d2h) != cudaSuccess) { rc = fail(c, FSB_ERR_CUDA, "copy from the device failed"); break; }   // result buffers of g-3 are free
        if ((rc = stage_complete(c, b)) != FSB_OK) break;
        if ((rc = run_enqueue(c, b, false)) != FSB_OK) break;
        if ((rc = summary_enqueue(c, b, *c->host[g], c->stream)) != FSB_OK) break;
        if (cudaEventRecord(b.ev_run, c->stream) != cudaSuccess) { rc = fail(c, FSB_ERR_CUDA, "cudaEventRecord failed"); break; }
        trace.mark("kernels enqueued", g);
        // The next copies in first (set g+2 = set g-1: its kernels were waited for one iteration ago, its results are guarded by
        // ev_d2h), then this sub-batch's results: finish() blocks for the half millisecond the kernels take and the copy out
        // starts the moment they end -- the host has nothing else to do until the text of g+1 has arrived.
        if (g + kAhead < G)
        {
            if ((rc = stage_enqueue(c, set_of(g + kAhead), chunks + first[g + kAhead], first[g + kAhead + 1] - first[g + kAhead], first[g + kAhead], c->s_h2d, c->s_chk[(g + kAhead) % kSets], 1)) != FSB_OK) break;
        }
        if ((rc = finish(g)) != FSB_OK) break;
        trace.mark("copy out enqueued", g);
    }
    drain();
    trace.mark("drained", G);
    if (rc == FSB_OK && cudaGetLastError() != cudaSuccess) rc = fail(c, FSB_ERR_CUDA, "CUDA error in the pipeline");
    c->batch[0].staged = c->batch[0].ran = false;                // the resident interface starts from a fresh fsb_stage
    return rc;
}
