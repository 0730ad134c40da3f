// tests/emul/emul.cpp -- TEST INFRASTRUCTURE: runs the per-thread routines of the CUDA kernels
// (fastore_b200/csrc/*_core.cuh, plain integer code marked FSB_HD) on the CPU, one "thread" after
// the other, over a whole chunk.  The CPU-only test tier compares the result with the oracle so
// that kernel logic is checked before GPU time is spent.  Built only by tests/ (g++, no CUDA);
// nothing in the product loads it.
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../fastore_b200/csrc/sig_core.cuh"

using namespace fsb;

namespace {

// What the kernel's staging does for one mate: 16-byte pieces of the aligned window around the
// sequence land in a shared-memory slot; the thread then reads 4-byte words from it.
template <int NW>
void stage_slot(const uint8_t* text, uint64_t text_size, uint32_t seq_off, uint32_t L, uint32_t* slot /* (2NW+1)*4 words */)
{
    const int64_t a0 = (int64_t)(seq_off & ~15u);
    const uint32_t npieces = ((seq_off & 15u) + L + 15u) >> 4;
    uint8_t* dst = reinterpret_cast<uint8_t*>(slot);
    std::memset(dst, 0xAB, (2 * NW + 1) * 16);                    // stale shared memory
    for (uint32_t j = 0; j < npieces && j < 2 * NW + 1; ++j)
        for (int b = 0; b < 16; ++b)
        {
            const int64_t src = a0 + 16 * j + b;
            dst[16 * j + b] = (src >= 0 && (uint64_t)src < text_size) ? text[src] : 0x5A;   // device pad bytes
        }
}

template <int NW>
void mate_scan(const uint8_t* text, uint64_t text_size, const fsb_record& r, const DeviceParams& P, StrandMin& f, StrandMin& rv, uint32_t& nN)
{
    uint32_t slot[(2 * NW + 1) * 4 + 4];
    stage_slot<NW>(text, text_size, r.seq_off, r.seq_len, slot);
    const uint32_t a = r.seq_off & 15u;
    BV<NW> H, Lo, Nm;
    mate_minimizers<NW>(slot + (a >> 2), 8 * (a & 3u), r.seq_len, P, f, rv, nN, H, Lo, Nm);
}

template <int NW>
void run_signatures(const DeviceParams& P, const fsb_chunk* ch, uint32_t* sig_out, uint32_t* info_out)
{
    for (uint64_t i = 0; i < ch->n_records; ++i)
    {
        StrandMin f1, r2;
        uint32_t n1;
        mate_scan<NW>(ch->text[0], ch->text_size[0], ch->records[0][i], P, f1, r2, n1);
        if (!P.paired) select_se(f1, r2, n1, P, sig_out[i], info_out[i]);
        else
        {
            StrandMin f2, r1;
            uint32_t n2;
            mate_scan<NW>(ch->text[1], ch->text_size[1], ch->records[1][i], P, f2, r1, n2);
            select_pe(f1, f2, r1, r2, n1, n2, P, sig_out[i], info_out[i]);
        }
    }
}

} // namespace

extern "C" int emul_signatures(const fsb_params* p, const fsb_chunk* ch, uint32_t* sig_out, uint32_t* info_out)
{
    const DeviceParams P = make_device_params(*p);
    uint32_t maxL = 1;
    for (int m = 0; m < (P.paired ? 2 : 1); ++m)
        for (uint64_t i = 0; i < ch->n_records; ++i) if (ch->records[m][i].seq_len > maxL) maxL = ch->records[m][i].seq_len;
    switch ((maxL + 31) / 32)
    {
    case 1: run_signatures<1>(P, ch, sig_out, info_out); break;
    case 2: run_signatures<2>(P, ch, sig_out, info_out); break;
    case 3: run_signatures<3>(P, ch, sig_out, info_out); break;
    case 4: run_signatures<4>(P, ch, sig_out, info_out); break;
    case 5: run_signatures<5>(P, ch, sig_out, info_out); break;
    case 6: run_signatures<6>(P, ch, sig_out, info_out); break;
    case 7: run_signatures<7>(P, ch, sig_out, info_out); break;
    case 8: run_signatures<8>(P, ch, sig_out, info_out); break;
    default: return FSB_ERR_INPUT;
    }
    return FSB_OK;
}

// ================================================================================================
// pack: host-side layout (plain loops restating layout.cuh) + the per-thread routines of
// pack_core.cuh in the order the kernels use them: K1 codes every stored mate into the record's
// slot, K4 shifts the slot's segments to their final bit positions in flat word buffers.
#include <algorithm>
#include <numeric>

#include "../../fastore_b200/csrc/pack_core.cuh"

namespace {

struct Slot
{
    std::vector<uint32_t> w;     // 16-byte guard + aligned window + slack
    uint32_t addr;               // byte offset of the first source byte
    void fill(const uint8_t* text, uint64_t text_size, uint32_t off, uint32_t len)
    {
        const int64_t a0 = (int64_t)(off & ~15u);
        const uint32_t npieces = ((off & 15u) + len + 15u) >> 4;
        w.assign((npieces + 4) * 4, 0xCDCDCDCDu);
        uint8_t* dst = reinterpret_cast<uint8_t*>(w.data()) + 16;
        for (uint32_t j = 0; j < npieces * 16; ++j)
        {
            const int64_t src = a0 + j;
            dst[j] = (src >= 0 && (uint64_t)src < text_size) ? text[src] : 0x5A;
        }
        addr = 16 + (off & 15u);
    }
};

// What K1 (ingest.cuh) does for one stored mate: code its DNA bits into the title + DNA region of the
// record's slot and its quality bits into the mate's quality region.
// `roleB`: the mate is stored second, its DNA starts where mate A's ends.
template <int NW>
void prepack_mate(const DeviceParams& P, const SlotGeom& G, const Slot& seq, const Slot& qua, uint32_t len, bool rev, bool plain, uint32_t cut_pos, uint32_t cut_len,
                  uint32_t* slot, uint32_t dna_off, bool roleB)
{
    // K1 derives the DNA from the bit planes it built for the signature search
    BV<NW> H, Lo, Nm;
    mate_planes<NW>(seq.w.data() + (seq.addr >> 2), 8u * (seq.addr & 3u), len, H, Lo, Nm);
    SegEmit ed = seg_open(slot + G.qw, dna_off, (len - cut_len) * (plain ? 2u : 3u));
    static const SpreadLut tables;
    pack_dna_planes<NW>(H, Lo, Nm, len, rev, plain, cut_pos, cut_len, LutPtr{tables.v}, ed);
    seg_finish(ed, true);
    // the quality goes straight to the mate's quality region
    const SymReader rq = reader_open(qua.w.data(), qua.addr, len, rev);
    uint32_t* dst = slot + (roleB ? G.wqa : 0u);
    switch (P.qua_bits)
    {
    case 6: pack_quality_to<6>(rq, len, P, dst); break;
    case 3: pack_quality_to<3>(rq, len, P, dst); break;
    default: pack_quality_to<1>(rq, len, P, dst); break;
    }
}

template <int NW>
int run_pack(const DeviceParams& P, const fsb_chunk* ch, const uint32_t* sig, const uint32_t* info, uint8_t* out[4], uint64_t out_size[4])
{
    const uint64_t n = ch->n_records;
    const bool pe = P.paired != 0;
    std::vector<uint32_t> order(n);
    std::iota(order.begin(), order.end(), 0u);
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return sig[a] < sig[b]; });
    // bins
    std::vector<uint64_t> bin_start;
    for (uint64_t i = 0; i < n; ++i) if (i == 0 || sig[order[i]] != sig[order[i - 1]]) bin_start.push_back(i);
    bin_start.push_back(n);
    const uint64_t nb = bin_start.size() - 1;
    // per-record bit offsets
    std::vector<uint64_t> off[4];
    for (auto& v : off) v.resize(n);
    std::vector<uint32_t> bmin(nb), bmax(nb);
    uint64_t pos[4] = {0, 0, 0, 0};          // running byte-aligned stream positions, in bits
    for (uint64_t b = 0; b < nb; ++b)
    {
        uint32_t mn = 0xFFFFFFFFu, mx = 0;
        for (uint64_t i = bin_start[b]; i < bin_start[b + 1]; ++i)
        {
            const uint32_t L = ch->records[0][order[i]].seq_len;
            mn = std::min(mn, L); mx = std::max(mx, L);
        }
        bmin[b] = mn; bmax[b] = mx;
        pos[0] += 17;
        for (uint64_t i = bin_start[b]; i < bin_start[b + 1]; ++i)
        {
            const uint32_t r = order[i];
            const fsb_record& ra = ch->records[0][r];
            const uint32_t L2 = pe ? ch->records[1][r].seq_len : 0;
            const ReadBits rb = read_bit_lengths(P, sig[r] == P.nbin, info[r], ra.seq_len, L2, P.has_headers ? ra.head_len : 0, mn, mx);
            const uint32_t bits[4] = {rb.meta, rb.dna, rb.qua, rb.head};
            for (int s = 0; s < 4; ++s) { off[s][i] = pos[s]; pos[s] += bits[s]; }
        }
        for (int s = 0; s < 4; ++s) pos[s] = (pos[s] + 7) & ~7ull;
    }
    std::vector<uint32_t> words[4];
    for (int s = 0; s < 4; ++s) { words[s].assign(pos[s] / 32 + 4, 0u); out_size[s] = pos[s] / 8; }

    uint32_t maxH = 0;
    for (uint64_t i = 0; i < n; ++i) maxH = std::max<uint32_t>(maxH, ch->records[0][i].head_len);
    const SlotGeom G = make_slot_geom(P, 32 * NW < 255 ? 32 * NW : 255, P.has_headers ? maxH : 0);
    std::vector<uint32_t> slot(G.words + 8);
    Slot seqA, quaA, seqB, quaB, head;
    for (uint64_t b = 0; b < nb; ++b)
    {
        for (uint64_t i = bin_start[b]; i < bin_start[b + 1]; ++i)
        {
            const uint32_t r = order[i], inf = info[r];
            const bool nbin = sig[r] == P.nbin;
            const bool rev = (inf & FSB_INFO_REVERSE) != 0, swp = (inf & FSB_INFO_SWAPPED) != 0;
            const bool a_is_m2 = pe && (rev != swp);
            const int ma = a_is_m2 ? 1 : 0, mb = a_is_m2 ? 0 : 1;
            const fsb_record& ra = ch->records[ma][r];
            seqA.fill(ch->text[ma], ch->text_size[ma], ra.seq_off, ra.seq_len);
            quaA.fill(ch->text[ma], ch->text_size[ma], ra.qua_off, ra.seq_len);
            const uint32_t sfx = nbin ? 0u : P.k, mpos = inf & FSB_INFO_POS_MASK;
            const bool plainA = (inf & FSB_INFO_PLAIN_A) != 0, plainB = (inf & FSB_INFO_PLAIN_B) != 0;
            // ---- K1: the record's slot (title first: the DNA segments merge into the word the title ends in) ----
            std::fill(slot.begin(), slot.end(), 0xDEADBEEFu);      // the slot staging is never cleared
            const fsb_record& r1 = ch->records[0][r];
            const uint32_t H = P.has_headers ? r1.head_len : 0u;
            const uint32_t head_bits = P.has_headers ? 8u + 7u * (H ? H - 1u : 0u) : 0u;
            if (P.has_headers)
            {
                head.fill(ch->text[0], ch->text_size[0], r1.head_off, r1.head_len);
                pack_head(head.w.data(), head.addr, r1.head_len, slot.data() + G.qw);
            }
            uint32_t lenB = 0;
            prepack_mate<NW>(P, G, seqA, quaA, ra.seq_len, rev, plainA, nbin ? 0u : mpos, sfx, slot.data(), head_bits, false);
            if (pe)
            {
                const fsb_record& rbm = ch->records[mb][r];
                lenB = rbm.seq_len;
                seqB.fill(ch->text[mb], ch->text_size[mb], rbm.seq_off, rbm.seq_len);
                quaB.fill(ch->text[mb], ch->text_size[mb], rbm.qua_off, rbm.seq_len);
                prepack_mate<NW>(P, G, seqB, quaB, rbm.seq_len, rev, plainB, 0, 0, slot.data(), head_bits + (ra.seq_len - sfx) * (plainA ? 2u : 3u), true);
            }
            // the card must survive the trip through the sort
            const uint64_t card = card_make(r, inf, ra.seq_len, lenB, H);
            if (card_rec(card) != r || card_info(card) != inf || card_lenA(card) != ra.seq_len || card_lenB(card) != lenB || card_head(card) != H) return FSB_ERR_STATE;
            // ---- K4: place the slot's segments ----
            const ReadBits rb = read_bit_lengths(P, nbin, inf, ra.seq_len, lenB, H, bmin[b], bmax[b]);
            if (i == bin_start[b])
            {   // PackToBin header (FastqPacker.cpp:581-583): minLen, maxLen, hasReadGroups = 0
                or_bits(words[0].data(), (uint32_t)(off[0][i] - 17), ((bmin[b] & 0xFFu) << 9) | ((bmax[b] & 0xFFu) << 1), 17);
            }
            uint32_t mbits;
            const uint32_t mv = meta_fields(P, nbin, inf, ra.seq_len, lenB, bmin[b], bmax[b], mbits);
            if (mbits != rb.meta) return FSB_ERR_STATE;
            or_bits(words[0].data(), (uint32_t)off[0][i], mv, mbits);
            const uint32_t qa = ra.seq_len * P.qua_bits;
            shift_copy_aligned(slot.data(), qa, words[2].data(), (uint32_t)off[2][i]);
            shift_copy_aligned(slot.data() + G.wqa, rb.qua - qa, words[2].data(), (uint32_t)off[2][i] + qa);
            shift_copy(slot.data() + G.qw, rb.head, rb.dna, words[1].data(), (uint32_t)off[1][i]);
            if (P.has_headers) shift_copy_aligned(slot.data() + G.qw, rb.head, words[3].data(), (uint32_t)off[3][i]);
        }
    }
    for (int s = 0; s < 4; ++s)
        for (uint64_t j = 0; j < out_size[s]; ++j) out[s][j] = (uint8_t)(words[s][j >> 2] >> (24 - 8 * (j & 3)));
    return FSB_OK;
}

} // namespace

// out[s] must have room for the oracle's stream size + 64 bytes
extern "C" int emul_pack(const fsb_params* p, const fsb_chunk* ch, uint8_t* meta, uint8_t* dna, uint8_t* qua, uint8_t* head, uint64_t* sizes)
{
    const DeviceParams P = make_device_params(*p);
    const uint64_t n = ch->n_records;
    std::vector<uint32_t> sig(n), info(n);
    int rc = emul_signatures(p, ch, sig.data(), info.data());
    if (rc != FSB_OK) return rc;
    uint32_t maxL = 1;
    for (int m = 0; m < (P.paired ? 2 : 1); ++m)
        for (uint64_t i = 0; i < n; ++i) maxL = std::max<uint32_t>(maxL, ch->records[m][i].seq_len);
    uint8_t* out[4] = {meta, dna, qua, head};
    switch ((maxL + 31) / 32)
    {
    case 1: return run_pack<1>(P, ch, sig.data(), info.data(), out, sizes);
    case 2: return run_pack<2>(P, ch, sig.data(), info.data(), out, sizes);
    case 3: return run_pack<3>(P, ch, sig.data(), info.data(), out, sizes);
    case 4: return run_pack<4>(P, ch, sig.data(), info.data(), out, sizes);
    case 5: return run_pack<5>(P, ch, sig.data(), info.data(), out, sizes);
    case 6: return run_pack<6>(P, ch, sig.data(), info.data(), out, sizes);
    case 7: return run_pack<7>(P, ch, sig.data(), info.data(), out, sizes);
    case 8: return run_pack<8>(P, ch, sig.data(), info.data(), out, sizes);
    }
    return FSB_ERR_INPUT;
}

// ================================================================================================
// layout as one scan (layout_core.cuh): the three phases of layout_fused.cuh -- per-thread run states, block
// states, exclusive scan over the blocks, absolute walk -- with a free choice of records per thread and threads
// per block, against the plain sequential walk over the sorted records.  Returns the number of mismatches
// (positions, bin descriptors, bin count), or a negative value when the chunk's reads differ in length.
#include "../../fastore_b200/csrc/layout_core.cuh"

namespace {

// A chunk's records sorted as the device sorts a batch: by chunk : signature, stably; records from `split` on form a second chunk.
// Returns the reads' common length, 0 when they differ or there are none, or -2 when the signatures fail.
long sorted_case(const fsb_params* p, const fsb_chunk* ch, uint64_t split, std::vector<uint32_t>& keys, std::vector<uint64_t>& cards)
{
    const DeviceParams P = make_device_params(*p);
    const uint64_t n = ch->n_records;
    keys.clear();
    cards.clear();
    if (n == 0) return 0;
    std::vector<uint32_t> sig(n), info(n);
    if (emul_signatures(p, ch, sig.data(), info.data()) != FSB_OK) return -2;
    const bool pe = P.paired != 0;
    uint32_t ulen = ch->records[0][0].seq_len;
    for (int m = 0; m < (pe ? 2 : 1); ++m)
        for (uint64_t i = 0; i < n; ++i) if (ch->records[m][i].seq_len != ulen) ulen = 0;
    std::vector<uint32_t> order(n);
    std::iota(order.begin(), order.end(), 0u);
    auto key_of = [&](uint32_t r) { return ((r < split ? 0u : 1u) << P.key_bits) | sig[r]; };
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return key_of(a) < key_of(b); });
    keys.resize(n);
    cards.resize(n);
    for (uint64_t i = 0; i < n; ++i)
    {
        const uint32_t r = order[i];
        keys[i] = key_of(r);
        cards[i] = card_make(r, info[r], ch->records[0][r].seq_len, pe ? ch->records[1][r].seq_len : 0, P.has_headers ? ch->records[0][r].head_len : 0);
    }
    return ulen;
}

// The plain walk over sorted records (the way run_pack above lays a chunk out): every record's first bit per stream, every bin's descriptor.
void plain_walk(const DeviceParams& P, const uint32_t* keys, const uint64_t* cards, uint64_t n, uint32_t ulen, std::vector<uint64_t> (&want_at)[4],
                std::vector<fsb_bin_descriptor>& want_desc)
{
    for (auto& v : want_at) v.resize(n);
    uint64_t pos[4] = {0, 0, 0, 0}, start[4] = {0, 0, 0, 0};
    fsb_bin_descriptor d{};
    for (uint64_t i = 0; i < n; ++i)
    {
        const bool st = i == 0 || keys[i] != keys[i - 1];
        if (st)
        {
            for (int s = 0; s < 4; ++s) { pos[s] = (pos[s] + 7) & ~7ull; start[s] = pos[s]; }
            pos[0] += 17;
            d = fsb_bin_descriptor{};
            d.signature = keys[i] & ((1u << P.key_bits) - 1u);
        }
        const uint64_t c = cards[i];
        const bool nbin = d.signature == P.nbin;
        const ReadBits rb = read_bit_lengths(P, nbin, card_info(c), card_lenA(c), card_lenB(c), card_head(c), ulen, ulen);
        const uint32_t bits[4] = {rb.meta, rb.dna, rb.qua, rb.head};
        for (int s = 0; s < 4; ++s) { want_at[s][i] = pos[s]; pos[s] += bits[s]; }
        d.records_count++; d.raw_dna_size += card_lenA(c) + card_lenB(c); d.raw_head_size += P.has_headers ? card_head(c) : 0;
        if (i + 1 == n || keys[i + 1] != keys[i])
        {
            d.meta_size = (((pos[0] + 7) & ~7ull) - start[0]) >> 3; d.dna_size = (((pos[1] + 7) & ~7ull) - start[1]) >> 3;
            d.qua_size = (((pos[2] + 7) & ~7ull) - start[2]) >> 3; d.head_size = (((pos[3] + 7) & ~7ull) - start[3]) >> 3;
            want_desc.push_back(d);
        }
    }
}

} // namespace

// sorted_case for the tests: keys / cards must hold ch->n_records entries
extern "C" long emul_sorted_case(const fsb_params* p, const fsb_chunk* ch, uint64_t split, uint32_t* keys_out, uint64_t* cards_out)
{
    std::vector<uint32_t> keys;
    std::vector<uint64_t> cards;
    const long ulen = sorted_case(p, ch, split, keys, cards);
    std::copy(keys.begin(), keys.end(), keys_out);
    std::copy(cards.begin(), cards.end(), cards_out);
    return ulen;
}

// plain_walk for the tests: at[4 * n]; desc must have room for every bin; returns the number of bins
extern "C" uint64_t emul_plain_walk(const fsb_params* p, const uint32_t* keys, const uint64_t* cards, uint64_t n, uint32_t ulen, uint64_t* at, fsb_bin_descriptor* desc)
{
    std::vector<uint64_t> want_at[4];
    std::vector<fsb_bin_descriptor> want_desc;
    plain_walk(make_device_params(*p), keys, cards, n, ulen, want_at, want_desc);
    for (int s = 0; s < 4; ++s) std::copy(want_at[s].begin(), want_at[s].end(), at + s * n);
    std::copy(want_desc.begin(), want_desc.end(), desc);
    return want_desc.size();
}

extern "C" long emul_layout_fused(const fsb_params* p, const fsb_chunk* ch, uint32_t per_thread, uint32_t threads)
{
    const DeviceParams P = make_device_params(*p);
    const uint64_t n = ch->n_records;
    if (n == 0) return 0;
    // sorted keys and cards (one chunk: chunk bits 0; a second pseudo-chunk is made of the upper half to exercise chunk starts)
    std::vector<uint32_t> keys;
    std::vector<uint64_t> cards;
    const long sc = sorted_case(p, ch, n / 2, keys, cards);
    if (sc < 0) return sc;
    if (sc == 0) return -1;
    const uint32_t ulen = (uint32_t)sc;
    std::vector<uint64_t> want_at[4];
    std::vector<fsb_bin_descriptor> want_desc;
    plain_walk(P, keys.data(), cards.data(), n, ulen, want_at, want_desc);
    // ---- the three phases ------------------------------------------------------------------------------------------
    const uint64_t per_block = (uint64_t)per_thread * threads;
    const uint64_t nblocks = (n + per_block - 1) / per_block;
    auto run_state = [&](uint64_t i0, uint64_t cnt) {
        LayState st = lay_identity();
        for (uint64_t j = 0; j < cnt; ++j)
            lay_push(st, lay_record(P, i0 + j == 0, keys[i0 + j], i0 + j ? keys[i0 + j - 1] : 0u, cards[i0 + j], ulen));
        return st;
    };
    auto thread_run = [&](uint64_t blk, uint32_t t, uint64_t& i0, uint64_t& cnt) {
        i0 = (blk * threads + t) * per_thread;
        cnt = i0 < n ? std::min<uint64_t>(per_thread, n - i0) : 0;
    };
    std::vector<LayState> block_state(nblocks + 1);
    for (uint64_t blk = 0; blk < nblocks; ++blk)                        // lay_reduce
    {
        LayState tot = lay_identity();
        for (uint32_t t = 0; t < threads; ++t) { uint64_t i0, cnt; thread_run(blk, t, i0, cnt); tot = lay_combine(tot, run_state(i0, cnt)); }
        block_state[blk] = tot;
    }
    {                                                                   // lay_scan (exclusive, in place)
        LayState carry = lay_identity();
        for (uint64_t blk = 0; blk < nblocks; ++blk) { const LayState mine = block_state[blk]; block_state[blk] = carry; carry = lay_combine(carry, mine); }
        block_state[nblocks] = carry;
    }
    long bad = 0;
    std::vector<fsb_bin_descriptor> got_desc(want_desc.size() + 1);
    uint32_t nb_total = 0;
    for (uint64_t blk = 0; blk < nblocks; ++blk)                        // lay_apply
    {
        LayState before = block_state[blk];
        for (uint32_t t = 0; t < threads; ++t)
        {
            uint64_t i0, cnt;
            thread_run(blk, t, i0, cnt);
            LayCursor cur = lay_cursor(before);
            for (uint64_t j = 0; j < cnt; ++j)
            {
                const uint64_t i = i0 + j;
                const LayRec r = lay_record(P, i == 0, keys[i], i ? keys[i - 1] : 0u, cards[i], ulen);
                uint64_t at[4];
                lay_step(cur, r, at);
                for (int s = 0; s < 4; ++s) if (at[s] != want_at[s][i]) bad++;
                if (i + 1 == n || keys[i + 1] != keys[i])
                {
                    if (cur.nb == 0 || cur.nb > want_desc.size()) { bad++; continue; }
                    got_desc[cur.nb - 1] = lay_descriptor(cur, keys[i] & ((1u << P.key_bits) - 1u));
                }
                if (i + 1 == n) nb_total = cur.nb;
            }
            before = lay_combine(before, run_state(i0, cnt));
        }
    }
    if (nb_total != want_desc.size()) bad++;
    if (block_state[nblocks].nstarts != want_desc.size()) bad++;
    for (size_t b = 0; b < want_desc.size(); ++b) if (std::memcmp(&got_desc[b], &want_desc[b], sizeof(fsb_bin_descriptor)) != 0) bad++;
    return bad;
}

// What lay_apply (layout_fused.cuh) must hand K4 for n sorted records whose reads all have `ulen` bases, in n_chunks chunks, as a
// plain walk record after record: no LayState, no scan.  Outputs as tests/gpu_harness/sort_layout.cu's h_layout returns them:
//   loc[k][i]    record i's first bit in stream k minus b0 plus (b0 & 127), b0 = the first bit of its 32-record tile: the tile's first
//                record, or the first byte of the bin that record opens (0 for the title stream when titles are dropped)
//   binfo[i]     ulen | ulen << 8 | opens its bin << 16 | N-bin << 17
//   tbase        [tile][k] = b0, and [tiles][k] = the end of stream k rounded up to a byte
//   desc, nb     the bins; chunk_start[5 * c] = the first bin and the first byte of every stream of chunk c (chunks that hold records
//                only), then the same for the end of the batch
//   cleared      the stream words K4 shares between two tiles, which the layout zeroes, as k << 60 | word; returns their number
extern "C" uint64_t emul_layout_tables(const fsb_params* p, const uint32_t* keys, const uint64_t* cards, uint64_t n, uint32_t ulen, uint32_t n_chunks,
                                       uint32_t* loc, uint32_t* binfo, uint64_t* tbase, fsb_bin_descriptor* desc, uint64_t* chunk_start, uint32_t* nb,
                                       uint64_t* cleared)
{
    const DeviceParams P = make_device_params(*p);
    const uint32_t key_mask = (1u << P.key_bits) - 1u;
    uint64_t pos[4] = {0, 0, 0, 0}, start[4] = {0, 0, 0, 0}, b0[4] = {0, 0, 0, 0};
    uint64_t n_cleared = 0;
    auto clear = [&](int k, uint64_t bit) { if (bit & 31u) cleared[n_cleared++] = ((uint64_t)k << 60) | (bit >> 5); };
    uint32_t bins = 0;
    fsb_bin_descriptor d{};
    for (uint64_t i = 0; i < n; ++i)
    {
        const uint32_t key = keys[i];
        const bool opens = i == 0 || key != keys[i - 1];
        const bool nbin = (key & key_mask) == P.nbin;
        if (opens)
        {
            for (int k = 0; k < 4; ++k) { pos[k] = roundup8(pos[k]); start[k] = pos[k]; }
            pos[0] += 17;                                              // minLen, maxLen, hasReadGroups
            bins++;
            d = fsb_bin_descriptor{};
            d.signature = key & key_mask;
            if (i == 0 || (key >> P.key_bits) != (keys[i - 1] >> P.key_bits))
            {
                uint64_t* cs = chunk_start + 5 * (key >> P.key_bits);
                cs[0] = bins - 1;
                for (int k = 0; k < 4; ++k) cs[1 + k] = start[k] >> 3;
            }
        }
        const uint64_t c = cards[i];
        const ReadBits rb = read_bit_lengths(P, nbin, card_info(c), card_lenA(c), card_lenB(c), card_head(c), ulen, ulen);
        const uint32_t bits[4] = {rb.meta, rb.dna, rb.qua, rb.head};
        for (int k = 0; k < 4; ++k)
        {
            const bool has = k < 3 || P.has_headers;
            if (i % 32 == 0)
            {
                b0[k] = has ? (opens ? start[k] : pos[k]) : 0;
                tbase[4 * (i / 32) + k] = b0[k];
                clear(k, b0[k]);
            }
            loc[k * n + i] = has ? (uint32_t)(pos[k] - b0[k] + (b0[k] & 127u)) : 0u;
            pos[k] += bits[k];
        }
        binfo[i] = (ulen & 0xFFu) | ((ulen & 0xFFu) << 8) | (opens ? 0x10000u : 0u) | (nbin ? 0x20000u : 0u);
        d.records_count++;
        d.raw_dna_size += card_lenA(c) + card_lenB(c);
        d.raw_head_size += P.has_headers ? card_head(c) : 0u;
        if (i + 1 == n || keys[i + 1] != key)
        {
            d.meta_size = (roundup8(pos[0]) - start[0]) >> 3; d.dna_size = (roundup8(pos[1]) - start[1]) >> 3;
            d.qua_size = (roundup8(pos[2]) - start[2]) >> 3; d.head_size = (roundup8(pos[3]) - start[3]) >> 3;
            desc[bins - 1] = d;
        }
    }
    const uint64_t tiles = (n + 31) / 32;
    uint64_t* cs = chunk_start + 5 * (uint64_t)n_chunks;
    cs[0] = bins;
    for (int k = 0; k < 4; ++k)
    {
        const bool has = k < 3 || P.has_headers;
        tbase[4 * tiles + k] = has ? roundup8(pos[k]) : 0;
        clear(k, tbase[4 * tiles + k]);
        cs[1 + k] = roundup8(pos[k]) >> 3;
    }
    *nb = bins;
    return n_cleared;
}

// ================================================================================================
// fastore_rebin's scan (sig_core.cuh: plane_new_minimizer) "thread" by "thread" over a record table.
template <int NW>
static void run_new_minimizers(const DeviceParams& P, const uint8_t* text, uint64_t text_size, const fsb_record* rec, uint64_t n, uint32_t cur, uint32_t* sig, uint32_t* info)
{
    for (uint64_t i = 0; i < n; ++i)
    {
        uint32_t slot[(2 * NW + 1) * 4 + 4];
        stage_slot<NW>(text, text_size, rec[i].seq_off, rec[i].seq_len, slot);
        const uint32_t a = rec[i].seq_off & 15u;
        BV<NW> H, Lo, Nm;
        mate_planes<NW>(slot + (a >> 2), 8 * (a & 3u), rec[i].seq_len, H, Lo, Nm);
        plane_new_minimizer<NW>(H, Lo, Nm, rec[i].seq_len, P, cur, sig[i], info[i]);
    }
}

extern "C" int emul_new_minimizers(const fsb_params* p, const uint8_t* text, uint64_t text_size, const fsb_record* rec, uint64_t n, uint32_t cur, uint32_t divisor,
                                   uint32_t* sig, uint32_t* info)
{
    DeviceParams P = make_device_params(*p);
    uint32_t lg = 0;
    while ((1u << lg) < divisor) ++lg;
    P.cutoff_bits = std::max(P.cutoff_bits, lg);
    uint32_t maxL = 1;
    for (uint64_t i = 0; i < n; ++i) maxL = std::max<uint32_t>(maxL, rec[i].seq_len);
    switch ((maxL + 31) / 32)
    {
    case 1: run_new_minimizers<1>(P, text, text_size, rec, n, cur, sig, info); break;
    case 2: run_new_minimizers<2>(P, text, text_size, rec, n, cur, sig, info); break;
    case 3: run_new_minimizers<3>(P, text, text_size, rec, n, cur, sig, info); break;
    case 4: run_new_minimizers<4>(P, text, text_size, rec, n, cur, sig, info); break;
    case 5: run_new_minimizers<5>(P, text, text_size, rec, n, cur, sig, info); break;
    case 6: run_new_minimizers<6>(P, text, text_size, rec, n, cur, sig, info); break;
    case 7: run_new_minimizers<7>(P, text, text_size, rec, n, cur, sig, info); break;
    case 8: run_new_minimizers<8>(P, text, text_size, rec, n, cur, sig, info); break;
    default: return FSB_ERR_INPUT;
    }
    return FSB_OK;
}

// ---- device-side parse: the line-end mask of every 16-byte vector of a text (parse_core.cuh) -------------------------
#include "../../fastore_b200/csrc/parse_core.cuh"

extern "C" void emul_line_end_masks(const uint8_t* text, uint64_t size, uint16_t* masks /* ceil(size / 16) */)
{
    for (uint64_t off = 0; off < size; off += 16)
    {
        uint8_t v[16] = {0};
        const uint32_t valid = (uint32_t)std::min<uint64_t>(16, size - off);
        std::memcpy(v, text + off, valid);
        uint32_t w[4];
        std::memcpy(w, v, 16);
        const uint32_t next = off + 16 < size ? text[off + 16] : 0u;           // parse_load: the byte behind the vector, 0 at the end of the text
        masks[off / 16] = (uint16_t)fsb::line_end_mask(w, next, valid);
    }
}

// The whole device-side parse of one text, pass by pass as the kernels do it (parse.cuh): masks -> line starts -> candidates.
// Returns the number of records in front of the first rejected candidate; *first_invalid = first record outside the device
// contract among them (~0: none).
extern "C" uint64_t emul_parse_text(const uint8_t* text, uint64_t size, int keep_headers, int keep_comments, fsb_record* out, uint64_t capacity,
                                    uint32_t* stop_reason, uint64_t* first_invalid)
{
    std::vector<uint16_t> masks((size + 15) / 16 + 1, 0);
    emul_line_end_masks(text, size, masks.data());
    std::vector<uint32_t> ls{0};
    for (uint64_t v = 0; v * 16 < size; ++v)
        for (uint32_t b = 0; b < 16; ++b)
            if (masks[v] >> b & 1u) ls.push_back((uint32_t)(v * 16 + b + 1));
    const uint32_t n_ends = (uint32_t)ls.size() - 1;
    const uint8_t last = size ? text[size - 1] : (uint8_t)'\n';
    const uint32_t n_lines = n_ends + ((size && last != '\n' && last != '\r') ? 1u : 0u);
    const uint32_t cap = (n_lines + 3u) / 4u;
    *stop_reason = 0; *first_invalid = ~0ull;
    uint64_t n = 0;
    for (uint32_t r = 0; r < cap; ++r)
    {
        fsb_record o{};
        bool invalid = false;
        const uint32_t reason = fsb::parse_candidate(text, (uint32_t)size, ls.data(), n_ends, n_lines, r, keep_headers != 0, keep_comments != 0, o, invalid);
        if (reason != fsb::kStopNone) { *stop_reason = reason; break; }
        if (invalid && *first_invalid == ~0ull) *first_invalid = r;
        if (n < capacity) out[n] = o;
        ++n;
    }
    return n;
}

// ---- FSB_OPT_VALIDATE: validate_text_kernel's per-mate byte check (stage_core.cuh) -------------------------------------
// `spans` holds n triples (offset into buf, length, kind: 0 sequence, 1 quality, 2 title characters).  buf is copied to a
// 16-byte aligned buffer with 64 zero bytes behind it, so the aligned pieces stay inside as they do in the padded device
// text.  Each span is checked the way one half warp checks a mate: lanes 0..15 take pieces 0..15, then each lane its
// pieces 16, 32, ... (the 17th piece of spans over 240 bytes).  ok[i] = 1 when span i passes.
#include "../../fastore_b200/csrc/stage_core.cuh"

extern "C" void emul_check_spans(const uint8_t* buf, uint64_t size, const int32_t* spans, uint64_t n, uint32_t qua_offset, int need_range, uint8_t* ok)
{
    struct alignas(16) Piece { uint8_t b[16]; };
    std::vector<Piece> text((size + 64 + 15) / 16);
    std::memset(text.data(), 0, text.size() * sizeof(Piece));
    std::memcpy(text.data(), buf, size);
    const uint8_t* base = text.data()->b;
    const uint32_t off4 = fsb::quality_off4(qua_offset);
    for (uint64_t i = 0; i < n; ++i)
    {
        const int32_t kind = spans[3 * i + 2];
        const CheckSpan s = check_span(base + spans[3 * i], (uint32_t)spans[3 * i + 1]);
        auto piece = [&](int32_t p) {
            uint32_t w[4];
            std::memcpy(w, reinterpret_cast<const uint8_t*>(s.a0) + 16 * p, 16);
            return kind == 0 ? piece_ok<0>(w, p, s.lo, s.hi, off4, need_range != 0)
                 : kind == 1 ? piece_ok<1>(w, p, s.lo, s.hi, off4, need_range != 0)
                             : piece_ok<2>(w, p, s.lo, s.hi, off4, need_range != 0);
        };
        bool all = true;
        for (int32_t l16 = 0; l16 < 16; ++l16)
        {
            bool lane = true;
            if (l16 * 16 < s.hi) lane = piece(l16);
            for (int32_t p = l16 + 16; p * 16 < s.hi; p += 16) lane = lane && piece(p);
            all = all && lane;
        }
        ok[i] = all ? 1 : 0;
    }
}

// quality4<Q> (pack_core.cuh) on single words, with off4 / thr4 formed as pack_quality_to forms them
extern "C" void emul_quality4(int q_bits, const uint32_t* words, uint64_t n, uint32_t qua_offset, uint32_t threshold, uint32_t* out)
{
    const uint32_t off4 = qua_offset * 0x01010101u, thr4 = threshold * 0x01010101u;
    for (uint64_t i = 0; i < n; ++i)
        out[i] = q_bits == 6 ? quality4<6>(words[i], off4, thr4) : q_bits == 3 ? quality4<3>(words[i], off4, thr4) : quality4<1>(words[i], off4, thr4);
}
