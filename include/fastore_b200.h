/*
 * fastore_b200.h -- C ABI of the B200-native fastore_bin categorise + scatter path.
 *
 * This is the drop-in boundary.  One call takes parsed FASTQ chunks (the chunk text as cut by the
 * host chunk cutter plus a compact record table produced by the host parser) and returns, per
 * chunk, what the reference produces with
 *
 *     FastqCategorizerSE/PE::Categorize(records, bins)      (FastqCategorizer.h:68-69, .cpp:169-363)
 *     FastqRecordsPackerSE/PE::PackToBins(bins, binBlock)   (FastqPacker.h:127-128, .cpp:417-491)
 *
 * i.e. the content of one BinaryBinBlock (BinBlockData.h:62-180): four MSB-first bit streams
 * (meta / dna / qua / head), byte-aligned per bin, bins in ascending signature order with the
 * N-bin last, in-bin order = chunk parse order, plus one BinaryBinDescriptor per bin.
 * The block is consumed unchanged by BinFileWriter::WriteNextBlock (BinFile.cpp:85-222).
 *
 * Plain C, plain pointers and sizes.  No CUDA or torch types cross this boundary (the optional
 * stream handle is an opaque void*).  There is no CPU fallback: every entry point that computes
 * fails with FSB_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef FASTORE_B200_H
#define FASTORE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FSB_VERSION 1

/* status codes (reference: `throw Exception(msg)`, Exception.h:20-40; no exceptions cross the ABI) */
enum {
    FSB_OK = 0,
    FSB_ERR_PARAM = 1,      /* invalid parameter / unsupported configuration */
    FSB_ERR_INPUT = 2,      /* record table violates the contract (symbols, lengths, offsets) */
    FSB_ERR_CUDA = 3,       /* CUDA runtime failure or no usable device */
    FSB_ERR_NOMEM = 4,      /* host or device allocation failure */
    FSB_ERR_STATE = 5       /* call sequence error (e.g. fetch before run) */
};

/* quality modes: QualityCompressionParams::CompressionMethod (Quality.h:29-35) */
enum { FSB_QUA_NONE = 0, FSB_QUA_BINARY = 1, FSB_QUA_8BIN = 2, FSB_QUA_QVZ = 3 };

/* per-read flags: FastqRecord::RecordFlags (FastqRecord.h:34-38), stored in read_info bits 16.. */
#define FSB_INFO_POS_MASK     0x0000FFFFu   /* minimPos in the stored orientation            */
#define FSB_INFO_REVERSE      0x00010000u   /* FlagReadIsReverse                             */
#define FSB_INFO_SWAPPED      0x00020000u   /* FlagIsPairSwapped (PE only)                   */
#define FSB_INFO_PLAIN_A      0x00040000u   /* stored mate A has no 'N' (isDnaPlain)         */
#define FSB_INFO_PLAIN_B      0x00080000u   /* stored mate B has no 'N' (PE only)            */

/*
 * Binning parameters: the subset of BinModuleConfig (Params.h:167-193) the path reads.
 *   signature_len              MinimizerParameters::signatureLen      (-p, 3..15)
 *   skip_zone_len              MinimizerParameters::skipZoneLen       (-s)
 *   signature_mask_cutoff_bits MinimizerParameters::signatureMaskCutoffBits (no CLI flag, 0)
 *   paired_end                 ArchiveType::readType == READ_PE       (-z)
 *   quality_method             QualityCompressionParams::method       (-q0..3)
 *   quality_offset             ArchiveType::qualityOffset             (33, or 64 with -I)
 *   binary_threshold           QualityCompressionParams::binaryThreshold (-w, default 20)
 *   reads_have_headers         ArchiveType::readsHaveHeaders          (-H)
 *   dna_symbol_order           MinimizerParameters::dnaSymbolOrder    (only "ACGTN" is accepted)
 */
typedef struct fsb_params {
    uint8_t signature_len;
    uint8_t skip_zone_len;
    uint8_t signature_mask_cutoff_bits;
    uint8_t paired_end;
    uint8_t quality_method;
    uint8_t quality_offset;
    uint8_t binary_threshold;
    uint8_t reads_have_headers;
    char    dna_symbol_order[5];
    uint8_t reserved[3];
} fsb_params;

/*
 * One parsed FASTQ record = what SingleFastqRecordParser::ReadNextRecord (FastqParser.cpp:118-165)
 * leaves in a FastqRecord (FastqRecord.h:41-49), as byte offsets into the chunk text instead of
 * pointers.  head_off points at the '@'; head_len is 0 when headers are not kept.
 */
typedef struct fsb_record {
    uint32_t head_off;
    uint32_t seq_off;
    uint32_t qua_off;
    uint16_t seq_len;
    uint8_t  head_len;
    uint8_t  reserved;
} fsb_record;

/*
 * One input chunk (FastqChunk / FastqChunkCollectionSE,PE: FastqRecord.h:336-391).
 *
 * Device-side parse: a chunk handed over with records[0] == NULL (and records[1] == NULL) is parsed by the library on the
 * GPU -- SingleFastqRecordParser::ReadNextRecord's rules (FastqParser.cpp:118-165: LF / CR LF / CR line ends, parsing stops
 * silently at the first malformed record; PE keeps min(n1, n2) pairs, :527) -- and n_records is ignored on input; the record
 * count comes back in fsb_block.n_records and the tables can be read with fsb_get_records.  All chunks of one call are
 * handed over the same way.
 * SE uses index 0 only.  PE: text[0]/records[0] are mate 1, text[1]/records[1] mate 2, record i
 * of both tables forms pair i; the two mates of a pair must have equal length (the reference
 * ASSERTs this, FastqRecord.h:87,192) and only mate 1's header is kept (FastqPacker.cpp:854).
 */
typedef struct fsb_chunk {
    const uint8_t*    text[2];
    uint64_t          text_size[2];
    const fsb_record* records[2];
    uint64_t          n_records;
} fsb_chunk;

/* BinaryBinDescriptor (BinBlockData.h:27-55) + the bin's signature (the map key). */
typedef struct fsb_bin_descriptor {
    uint64_t signature;      /* 0 .. 4^k ; 4^k is the N-bin */
    uint64_t meta_size;
    uint64_t dna_size;
    uint64_t qua_size;
    uint64_t head_size;
    uint64_t records_count;
    uint64_t raw_dna_size;
    uint64_t raw_head_size;
} fsb_bin_descriptor;

/*
 * One output block = BinaryBinBlock with blockType == MultiSignatureType (BinBlockData.h:62-180).
 * All pointers are library-owned pinned host memory, valid until the next fsb_fetch /
 * fsb_bin_chunks / fsb_destroy on the same context.  read_signature / read_info are per record in
 * chunk parse order (signature, minimPos | flags); they are NULL unless per-read output was
 * enabled with fsb_set_option(ctx, FSB_OPT_PER_READ, 1).
 */
typedef struct fsb_block {
    const uint8_t* meta;
    const uint8_t* dna;
    const uint8_t* qua;
    const uint8_t* head;
    uint64_t meta_size;
    uint64_t dna_size;
    uint64_t qua_size;
    uint64_t head_size;
    uint64_t raw_dna_size;
    uint64_t raw_head_size;
    const fsb_bin_descriptor* bins;   /* ascending signature, N-bin last */
    uint64_t n_bins;
    uint64_t n_records;
    const uint32_t* read_signature;
    const uint32_t* read_info;
} fsb_block;

typedef struct fsb_ctx fsb_ctx;

/* options for fsb_set_option */
enum {
    FSB_OPT_PER_READ = 1,    /* also return per-read signature/info arrays (parity Mode B)        */
    FSB_OPT_PROFILE = 2,     /* record CUDA events around every pipeline stage of fsb_run (runs with FSB_OPT_RUN_SPLIT 1 only: overlapped
                                sub-batches have no per-stage duration; a batch of more than 32 chunks is then run as sub-batches one after
                                the other and their stage times add up) */
    FSB_OPT_VALIDATE = 3,    /* device-side check of the bytes behind the record table in fsb_stage / fsb_bin_chunks: sequence
                                symbols A C G T N, quality in [offset, offset + 64) (>= offset in the 1-bit mode), 7-bit title
                                characters; default 1.  The record table itself (lengths, offsets, mate lengths) is always checked. */
    FSB_OPT_SUBBATCH_RECORDS = 4, /* fsb_bin_chunks pipelines sub-batches of at least this many records (default 400000) */
    FSB_OPT_RUN_SPLIT = 5,        /* fsb_run cuts the staged batch into this many sub-batches of whole chunks and overlaps them on
                                     two streams (takes effect at the next fsb_stage; 1 = one pass on the context's stream) */
    /* tuning knobs behind the measurements in DESIGN.md (may change between versions) */
    FSB_OPT_K1_BLOCK_BATCHES = 6, /* warp batches per warp of a K1 block when sub-batches share the GPU (0: persistent grid) */
    FSB_OPT_K4_BLOCK_TILES = 7,   /* tiles per K4 block in that mode (0: persistent grid) */
    FSB_OPT_BLOCK_GRIDS_ALWAYS = 8, /* use those block sizes for unsplit runs as well */
    FSB_OPT_FUSED_LAYOUT = 9,     /* 1 (default): batches whose reads all have one length take the one-scan layout; 0: always the general kernels */
    FSB_OPT_FUSED_HIST = 12,      /* 1: K1 and every scatter pass count the digits of the next radix pass; 0 (default): histogram kernels -- the fused
                                     form measured slower on B200 (one scattered L2 reduction per record and pass) */
    FSB_OPT_KEEP_RECORDS = 11,    /* device-side parse inside fsb_bin_chunks: also copy the record tables to the host (fsb_get_records) */
    FSB_OPT_KEEP_COMMENTS = 10    /* device-side parse (chunks without record tables): 1 (default) keeps the whole title, 0 cuts it at the first
                                     space like the reference's -C (HeadersCompressionParams::preserveComments, FastqParser.cpp:148-155) */
};

/* pipeline stages reported by fsb_stage_times (order of execution inside fsb_run) */
enum {
    FSB_STAGE_INGEST = 0,    /* K1: signature on both strands + prepacked per-record slots        */
    FSB_STAGE_SORT = 1,      /* K2/K3: histogram + scan + stable rank (radix passes)              */
    FSB_STAGE_LAYOUT = 2,    /* bin boundaries, per-bin length stats, bit-offset scans            */
    FSB_STAGE_PLACE = 3,     /* K4: gather the slots and shift them into the four streams         */
    FSB_STAGE_COUNT = 4,
    FSB_STAGE_CHECK = 4      /* not part of fsb_run: the input-check kernels of the last fsb_stage calls (record table +
                                FSB_OPT_VALIDATE byte check); reported as ms[4] when fsb_stage_times is asked for 5 values */
};

typedef struct fsb_stats {
    uint64_t kernel_launches;      /* kernels of this library launched since creation              */
    uint64_t h2d_bytes;            /* bytes copied host->device since creation                     */
    uint64_t d2h_bytes;            /* bytes copied device->host since creation                     */
    uint64_t records;              /* records binned since creation                                */
    uint64_t algorithmic_bytes;    /* SURVEY 8(d): input bytes consumed + output bytes produced    */
} fsb_stats;

/*
 * Limits of one call (FSB_ERR_PARAM / FSB_ERR_INPUT beyond them): a chunk text is shorter than 4 GiB (32-bit record
 * offsets, as in fsb_record); one batch -- the chunk list of fsb_stage, or one internal sub-batch of fsb_bin_chunks,
 * which splits longer lists itself -- holds at most 256 chunks (fewer for signature_len > 11: 2^(31 - 2 * signature_len))
 * and at most 2^28 - 1 records; reads are 1..255 bases (FastqRecord.h:45-48) and titles at most 255 bytes.
 *
 * Create a context bound to one GPU.  `cuda_stream` may be NULL (the context creates its own
 * stream) or a cudaStream_t the caller owns; all work of the context is enqueued on that stream.
 * One context per GPU worker; calls on one context must be serialised by the caller, different
 * contexts are independent (reference: one BinEncoder operator per thread, BinOperator.cpp:71).
 */
int  fsb_create(const fsb_params* params, int device, void* cuda_stream, fsb_ctx** out_ctx);
void fsb_destroy(fsb_ctx* ctx);

/* Message of the last error on this context; with ctx == NULL, of the last failed fsb_create. */
const char* fsb_last_error(const fsb_ctx* ctx);

int fsb_set_option(fsb_ctx* ctx, int option, int64_t value);

/*
 * Categorise + pack `n_chunks` chunks held in host memory: host->device copies, kernels,
 * device->host copies, synchronous; internally the chunks run as a pipeline of sub-batches so that
 * the copies in both directions overlap the kernels.  blocks[i] describes chunk i.  This is the call that replaces
 * the Categorize + PackToBins pair at BinModule.cpp:130-133 / :379-382 and
 * BinOperator.cpp:97+205 / :375+472.
 */
int fsb_bin_chunks(fsb_ctx* ctx, const fsb_chunk* chunks, uint32_t n_chunks, fsb_block* blocks);

/*
 * The same work split into its three phases, for callers that keep input resident or overlap
 * transfers with compute:
 *   fsb_stage  enqueue host->device copies of the chunks (text + record tables);
 *   fsb_run    enqueue the kernels over the staged chunks (may be repeated on the same staging);
 *   fsb_fetch  enqueue device->host copies of the result, wait, fill `blocks`.
 * fsb_sync waits for everything enqueued on the context's stream.
 */
int fsb_stage(fsb_ctx* ctx, const fsb_chunk* chunks, uint32_t n_chunks);
int fsb_run(fsb_ctx* ctx);
int fsb_fetch(fsb_ctx* ctx, fsb_block* blocks, uint32_t n_blocks);
int fsb_sync(fsb_ctx* ctx);

/*
 * Device-side parse only: the record table the library built for chunk `chunk` (index in the last fsb_bin_chunks / fsb_stage
 * call) and mate `mate`, copied to `dst` (capacity in records; the count is returned in *n_records, FSB_ERR_PARAM if it does
 * not fit).  For callers that need the tables on the host as well, e.g. for the title statistics of the bin-file footer.
 * Valid until the next staging call on the context (fsb_bin_chunks: needs FSB_OPT_KEEP_RECORDS, which makes the call copy the
 * tables back while the batches are in flight).
 */
int fsb_get_records(fsb_ctx* ctx, uint32_t chunk, int mate, fsb_record* dst, uint64_t capacity, uint64_t* n_records);

/*
 * fastore_rebin's signature scan (SURVEY.md 8f-3): DnaRebalancer::FindNewMinimizer (fastore_rebin/DnaRebalancer.cpp:570-616) for a
 * table of reads.  For every read: the smallest valid signature on either strand that differs from `cur_signature` and is a
 * multiple of `signature_parity` (a power of two, fastore_rebin -p), with the context's signature_len / skip_zone_len; ties go
 * to the forward strand.  signature[i] = 4^k when there is none (or the read has >= len/3 N); info[i] = position in the chosen
 * orientation | FSB_INFO_REVERSE.  records: seq_off / seq_len into `text` (the other fields are ignored).  Host buffers in and
 * out, synchronous.  The variant that admits only signatures present in the input bin file (BinBalanceParameters::
 * validBinSignatures filled from the file, RebinModule.cpp:62-68) is not covered.
 */
int fsb_find_new_minimizers(fsb_ctx* ctx, const uint8_t* text, uint64_t text_size, const fsb_record* records, uint64_t n_records,
                            uint32_t cur_signature, uint32_t signature_parity, uint32_t* signature, uint32_t* info);

/* Accumulated per-stage device time in milliseconds since the last call (needs FSB_OPT_PROFILE); n_runs counts fsb_run calls. */
int fsb_stage_times(fsb_ctx* ctx, float* ms, uint32_t n_stages, uint32_t* n_runs);

int fsb_get_stats(const fsb_ctx* ctx, fsb_stats* out);

/* Page-locked host memory for chunk text / record tables (optional; pageable memory also works, at a fifth of the copy
 * speed).  Buffers of 8 MB and more are anonymous mappings, touched and then registered with the driver -- on the B200 hosts
 * that pins 2.5 times faster than cudaHostAlloc (DESIGN.md section 9); free them with fsb_host_free only.
 * Environment: FSB_PIN=alloc takes cudaHostAlloc for every size; FSB_TRACE=1 prints the host-side timeline of every
 * fsb_bin_chunks call on stderr. */
void* fsb_host_alloc(size_t bytes);
void  fsb_host_free(void* p);

/* Number of usable sm_100 devices (0 when there is none; never falls back to the CPU). */
int fsb_device_count(void);

#ifdef __cplusplus
}
#endif
#endif /* FASTORE_B200_H */
