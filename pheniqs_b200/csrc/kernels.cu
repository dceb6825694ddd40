/*  kernels.cu — hand-written sm_100a kernels of the barcode classification path.

    pamld_kernel   PamlDecoder::classify (pamld.cpp:37-123) with Barcode::compensated_decoding_probability
                   (barcode.h:131-164), Decoder::classify (decoder.h:68-76) and Classifier::classify
                   (classifier.h:78-86) for a batch of reads against every barcode of one decoder.
    mdd_kernel     MdDecoder::classify (mdd.cpp:37-86) with Sequence::distance_from /
                   ObservedSequence::masked_distance_from (sequence.h:90-98, 321-332).
    count_kernel   the bookkeeping NaiveMolecularDecoder / passthrough classifiers do (naive.h:40-45).
    pamld_long_kernel, pamld_long_tie_kernel, mdd_long_kernel
                   the same for decoders of 33-64 nucleotides, over the split form of LongBarcodeEntry (kernels.cuh).

    Design (DESIGN.md has the long form). One lane owns one read; the barcode table streams
    through shared memory in 16 KB chunks moved by TMA bulk copies (cp.async.bulk + mbarrier),
    so every barcode word is a warp-uniform broadcast read. Bases are two 32-position bit
    planes, so the mismatch mask of a (read, barcode) pair is two LOP3s:

        m = (o_lo ^ e_lo) | (o_hi ^ e_hi) | n_mask

    PAMLD never evaluates pow() per pair. With B = 10^-0.1 the reference's

        P(r|b) = B ^ sum_j s(e_j, o_j, q_j)

    factors into a per-read constant P0 = prod_j B^s(match) times prod_{j in m} w_j with
    w_j = B^(q_j - tq[q_j]) (1 for N / q = 0 positions), and the product over the mismatch set
    is looked up four positions at a time in a per-lane table of the 16 subset products held in
    shared memory ([entry][lane] layout: conflict free). The exact scans do all probability
    arithmetic in f64; the prefilter scans (pamld_fast_kernel, pamld_fast_grid_kernel) walk the
    same pairs in f32 first, decide the reads whose maximum stands alone by 2^20 and leave the
    others to the exact scans through an index list. The first-maximum selection of the
    reference (strict >) is done on the high words of the f64 products; whenever the runner-up
    is within 2^-19 of the winner (structural ties, which the reference resolves by the
    rounding of its position-ordered Kahan sums) the read is queued with its possible winners
    and pamld_tie_kernel re-evaluates those in the reference's exact operation order.
*/
#include "kernels.cuh"
#include <cstdio>

namespace phq {

namespace {

constexpr int WARP_SIZE = 32;
constexpr int MAX_WARPS = 12;
constexpr int STAGE_ENTRIES = 1024;             /* barcodes per staged chunk: 16 KB */
constexpr int SHARED_ACCUMULATOR_ROWS = 1025;   /* per-CTA accumulators live in shared memory up to N + 1 = 1025 rows */
constexpr unsigned FULL_MASK = 0xffffffffu;

/* ------------------------------------------------------------------ shared memory plan (host and device agree) */
struct SharedPlan {
    int stage_capacity;         /* entries per stage buffer */
    int stage_buffers;          /* 1 when the whole table fits one chunk, else 2 */
    int accumulator_rows;       /* N + 1 when accumulators are staged in shared memory, else 0 */
    unsigned off_stage, off_phred, off_ratio32, off_hard, off_acc_f64, off_acc_u32, off_misc, off_mbarrier, off_tables;
    unsigned fixed_bytes;       /* everything except the per-warp tables */
};
__host__ __device__ inline unsigned align_up(unsigned v, unsigned a) { return (v + a - 1) / a * a; }
__host__ __device__ inline SharedPlan make_plan(int barcode_cardinality, bool phred_tables, int blob_entries = 0, bool ratio32 = false) {
    SharedPlan p;
    p.stage_capacity = barcode_cardinality < STAGE_ENTRIES ? barcode_cardinality : STAGE_ENTRIES;
    p.stage_buffers = barcode_cardinality <= STAGE_ENTRIES ? 1 : 2;
    if(blob_entries > 0) {      /* the combinatorial scan stages its grid blob instead of the barcode table */
        p.stage_capacity = blob_entries;
        p.stage_buffers = 1;
    }
    p.accumulator_rows = (barcode_cardinality + 1 <= SHARED_ACCUMULATOR_ROWS) ? barcode_cardinality + 1 : 0;
    unsigned at = 0;
    p.off_stage = at;       at += align_up(unsigned(p.stage_capacity) * unsigned(p.stage_buffers) * 16u, 128u);
    p.off_phred = at;       at += phred_tables ? 256u * 8u : 0u;
    p.off_ratio32 = at;     at += ratio32 ? 512u * 16u : 0u;     /* position table of the prefilter scans (PositionEntry) */
    p.off_hard = at;        at += ratio32 ? 32u * 256u : 0u;     /* per-warp staging of the hard list (HardList): 64 reads per warp */
    p.off_acc_f64 = at;     at += align_up(unsigned(p.accumulator_rows) * ACC_F64_COLUMNS * 8u, 16u);
    p.off_acc_u32 = at;     at += align_up(unsigned(p.accumulator_rows) * ACC_U64_COLUMNS * 4u, 16u);
    p.off_misc = at;        at += 16u;          /* totals count, pf_count; diagnostics exact, band */
    p.off_mbarrier = at;    at += 16u;
    /* The per-warp table blocks follow, 4 KB aligned IN THE SHARED WINDOW (lookup addresses are formed with one
       LOP3); dynamic shared memory does not start at window offset 0, so the kernel aligns at run time and the
       host reserves 4 KB of slack. */
    p.off_tables = align_up(at, 256u);
    p.fixed_bytes = p.off_tables + 4096u;
    return p;
}

/* ------------------------------------------------------------------ PTX helpers: mbarrier + TMA bulk copy */
__device__ __forceinline__ uint32_t shared_address(const void* p) { return static_cast< uint32_t >(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbarrier_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(shared_address(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbarrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbarrier_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(shared_address(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbarrier_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" :: "r"(shared_address(bar)), "r"(parity) : "memory");
}
/* 1-D TMA bulk copy global -> shared, completion counted in bytes on the mbarrier */
__device__ __forceinline__ void tma_bulk_load(void* destination, const void* source, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(shared_address(destination)), "l"(source), "r"(bytes), "r"(shared_address(bar)) : "memory");
}

/* streaming loads / stores: tiles and results are touched once */
__device__ __forceinline__ uint32_t load_stream(const uint32_t* p) { return __ldcs(p); }
__device__ __forceinline__ uint32_t load_stream(const uint16_t* p) { return static_cast< uint32_t >(__ldcs(reinterpret_cast< const unsigned short* >(p))); }
__device__ __forceinline__ void store_result(const TileArguments& A, long long r, int32_t index, int32_t distance, double confidence, uint32_t qcfail) {
    if(A.compact != nullptr) {
        /* Read::flush: float(1.0 - confidence) (read.h:189) */
        int2 v;
        v.x = static_cast< int >(static_cast< uint32_t >(index) | (static_cast< uint32_t >(distance) << 24) | (qcfail << 30));
        v.y = __float_as_int(static_cast< float >(1.0 - confidence));
        __stcs(reinterpret_cast< int2* >(A.compact) + r, v);
    } else if(A.results != nullptr) {
        int4 v;
        v.x = index;
        v.y = distance;
        v.z = __double2loint(confidence);
        v.w = __double2hiint(confidence);
        __stcs(reinterpret_cast< int4* >(A.results) + r, v);
    }
}

/*  The four Phred bytes of quality word g (positions 4g .. 4g+3) of read r, whatever form they travelled
    in. Codebook forms are decoded with byte permutes: a 2-bit index word selects among the 4 bytes of one
    codebook register with a single PRMT, a 4-bit index word among 16 bytes with two and a byte-wise blend. */
__device__ __forceinline__ uint32_t quality_word(const TileArguments& A, long long r, int g) {
    if(A.quality_bits == 8) { return load_stream(A.quality + g * A.pitch + r); }
    /* index 0 is a real quality in a codebook: positions past the observation must still read as Phred 0 */
    const int valid = A.nucleotides - 4 * g;
    const uint32_t keep = valid >= 4 ? 0xffffffffu : (valid <= 0 ? 0u : ((1u << (8 * valid)) - 1u));
    if(A.quality_bits == 2) {
        const uint32_t packed = load_stream(A.quality + (g >> 2) * A.pitch + r);
        const uint32_t c = (packed >> (8 * (g & 3))) & 0xffu;
        const uint32_t selector = (c & 0x3u) | ((c & 0xcu) << 2) | ((c & 0x30u) << 4) | ((c & 0xc0u) << 6);
        return __byte_perm(A.codebook[0], 0u, selector) & keep;
    }
    if(A.quality_bits == 4) {
        const uint32_t packed = load_stream(A.quality + (g >> 1) * A.pitch + r);
        const uint32_t c = (packed >> (16 * (g & 1))) & 0xffffu;
        const uint32_t low = __byte_perm(A.codebook[0], A.codebook[1], c & 0x7777u);
        const uint32_t high = __byte_perm(A.codebook[2], A.codebook[3], c & 0x7777u);
        /* bit 3 of every index chooses the upper half of the codebook: one flag bit per byte, widened to a byte mask */
        const uint32_t flag = ((c & 0x8u) >> 3) | ((c & 0x80u) << 1) | ((c & 0x800u) << 5) | ((c & 0x8000u) << 9);
        const uint32_t mask = flag * 0xffu;
        return (low ^ ((low ^ high) & mask)) & keep;
    }
    return 0u;
}

/*  The row of the 128-entry Phred tables a quality byte scores with. The reference's tables end at 127 and a byte
    above (a FASTQ decoded at too high an offset, a BAM record without qualities) indexes past them; such a byte
    carries no information and scores 0, as q = 0 does (DESIGN.md §5). The high quality filter still compares
    the raw byte. */
__device__ __forceinline__ uint32_t phred_quality(uint32_t q) { return q > 127u ? 0u : q; }

/* ------------------------------------------------------------------ per-CTA accumulators
   AccumulatingOption (selector.h:32-60). Staged in shared memory (u32 counters, f64 sums) when the
   table is small, flushed with one global atomic per non-zero cell; straight to global otherwise. */
/*  The per-CTA tables in shared memory hold every (total, pass-filter) column pair SPLIT: a read that passes
    the filter is added to the pass-filter column only, one that fails to the total column only, and the
    epilogue flushes total = failed + passed. One shared atomic per read and pair instead of two. */
struct Accumulator {
    uint32_t* shared_u32;
    double* shared_f64;
    unsigned long long* global_u64;
    double* global_f64;
    __device__ __forceinline__ void add(int row, int column, uint32_t value) const {
        if(shared_u32 != nullptr) { atomicAdd(&shared_u32[row * ACC_U64_COLUMNS + column], value); }
        else { atomicAdd(&global_u64[static_cast< long long >(row) * ACC_U64_COLUMNS + column], static_cast< unsigned long long >(value)); }
    }
    /* total += value, and pass_filter += value when the read passes */
    __device__ __forceinline__ void add_pair(int row, int total, int pass_filter, uint32_t value, bool passes) const {
        if(shared_u32 != nullptr) { atomicAdd(&shared_u32[row * ACC_U64_COLUMNS + (passes ? pass_filter : total)], value); }
        else {
            atomicAdd(&global_u64[static_cast< long long >(row) * ACC_U64_COLUMNS + total], static_cast< unsigned long long >(value));
            if(passes) { atomicAdd(&global_u64[static_cast< long long >(row) * ACC_U64_COLUMNS + pass_filter], static_cast< unsigned long long >(value)); }
        }
    }
    /*  Confidences (0 < value <= 1) are summed per CTA in 2^-46 fixed point: shared memory has native 32-bit integer
        atomics only (a f64 atomicAdd there is a compare-and-swap loop), so the cell — the 8 bytes of the double it
        stands for — is a low and a high word, the carry of the low word travelling with the high word's add. Exact
        to 1.4e-14 per read and independent of the order of the adds; a launch covers at most 2^24 reads, far from
        the 2^18 x 2^14 the high word holds. flush_accumulators converts back. */
    __device__ __forceinline__ void add_pair(int row, int total, int pass_filter, double value, bool passes) const {
        if(shared_f64 != nullptr) {
            const unsigned long long fixed = static_cast< unsigned long long >(value * 70368744177664.0 + 0.5);
            uint32_t* const cell = reinterpret_cast< uint32_t* >(&shared_f64[row * ACC_F64_COLUMNS + (passes ? pass_filter : total)]);
            const uint32_t low = static_cast< uint32_t >(fixed);
            const uint32_t before = atomicAdd(cell, low);
            atomicAdd(cell + 1, static_cast< uint32_t >(fixed >> 32) + (before + low < before ? 1u : 0u));
        }
        else {
            atomicAdd(&global_f64[static_cast< long long >(row) * ACC_F64_COLUMNS + total], value);
            if(passes) { atomicAdd(&global_f64[static_cast< long long >(row) * ACC_F64_COLUMNS + pass_filter], value); }
        }
    }
};

/* per-position factors of the prefilter scans: B ^ s(match) in f64 (it goes into P0) and B ^ (s(mismatch) - s(match)) in f32 */
struct __align__(16) PositionEntry {
    double factor;
    float ratio;
    uint32_t pad;
};

struct BlockState {
    SharedPlan plan;
    BarcodeEntry* stage;
    double* phred;
    uint32_t* misc;             /* [0] count [1] pf_count [2] exact path [3] band */
    uint64_t* mbarrier;
    Accumulator accumulator;
};

__device__ __forceinline__ BlockState block_prologue(unsigned char* smem, const DecoderParams& P, bool phred_tables, int blob_entries = 0, bool ratio32 = false) {
    BlockState s;
    s.plan = make_plan(P.barcode_cardinality, phred_tables, blob_entries, ratio32);
    s.stage = reinterpret_cast< BarcodeEntry* >(smem + s.plan.off_stage);
    s.phred = reinterpret_cast< double* >(smem + s.plan.off_phred);
    s.misc = reinterpret_cast< uint32_t* >(smem + s.plan.off_misc);
    s.mbarrier = reinterpret_cast< uint64_t* >(smem + s.plan.off_mbarrier);
    s.accumulator.global_u64 = P.acc_u64;
    s.accumulator.global_f64 = P.acc_f64;
    s.accumulator.shared_u32 = s.plan.accumulator_rows ? reinterpret_cast< uint32_t* >(smem + s.plan.off_acc_u32) : nullptr;
    s.accumulator.shared_f64 = s.plan.accumulator_rows ? reinterpret_cast< double* >(smem + s.plan.off_acc_f64) : nullptr;

    const int tid = threadIdx.x;
    if(phred_tables) {
        for(int i = tid; i < 256; i += blockDim.x) { s.phred[i] = P.phred[i]; }
    }
    if(ratio32) {
        /* what one position contributes, by Phred byte (0..255; a byte above 127 carries no information and scores as
           q = 0: phred_quality) and, from entry 256 on, for a base that is not A / C / G / T: one 16-byte load
           per position */
        PositionEntry* const position = reinterpret_cast< PositionEntry* >(smem + s.plan.off_ratio32);
        for(int i = tid; i < 512; i += blockDim.x) {
            const int q = static_cast< int >(phred_quality(static_cast< uint32_t >(i & 255)));
            PositionEntry e;
            e.pad = 0u;
            if(i < 256) {
                e.factor = P.phred[PHRED_MATCH_FACTOR + q];
                e.ratio = P.phred32[q];
            } else {
                e.factor = q != 0 ? P.phred[PHRED_UNIFORM_FACTOR] : 1.0;
                e.ratio = 1.0f;
            }
            position[i] = e;
        }
    }
    for(int i = tid; i < s.plan.accumulator_rows * ACC_U64_COLUMNS; i += blockDim.x) { s.accumulator.shared_u32[i] = 0; }
    for(int i = tid; i < s.plan.accumulator_rows * ACC_F64_COLUMNS; i += blockDim.x) { s.accumulator.shared_f64[i] = 0.0; }
    if(tid < 4) { s.misc[tid] = 0; }
    if(tid == 0) {
        mbarrier_init(&s.mbarrier[0], 1);
        mbarrier_init(&s.mbarrier[1], 1);
        fence_mbarrier_init();
    }
    __syncthreads();
    return s;
}

/* per-CTA accumulator tables -> global, one atomic per non-zero cell (call after a __syncthreads) */
__device__ __forceinline__ void flush_accumulators(const Accumulator& accumulator, int rows, const DecoderParams& P) {
    const int tid = threadIdx.x;
    for(int i = tid; i < rows * ACC_U64_COLUMNS; i += blockDim.x) {
        const int column = i % ACC_U64_COLUMNS;
        unsigned long long v = accumulator.shared_u32[i];
        /* split pairs (Accumulator): the total column also receives what went to its pass-filter column */
        if(column == ACC_COUNT) { v += accumulator.shared_u32[i - ACC_COUNT + ACC_PF_COUNT]; }
        if(column == ACC_DISTANCE) { v += accumulator.shared_u32[i - ACC_DISTANCE + ACC_PF_DISTANCE]; }
        if(v) { atomicAdd(&P.acc_u64[i], v); }
    }
    for(int i = tid; i < rows * ACC_F64_COLUMNS; i += blockDim.x) {
        /* 2^-46 fixed point cells (Accumulator::add_pair) back to f64 */
        unsigned long long fixed = reinterpret_cast< const unsigned long long* >(accumulator.shared_f64)[i];
        if(i % ACC_F64_COLUMNS == ACC_CONFIDENCE) { fixed += reinterpret_cast< const unsigned long long* >(accumulator.shared_f64)[i - ACC_CONFIDENCE + ACC_PF_CONFIDENCE]; }
        if(fixed != 0ull) { atomicAdd(&P.acc_f64[i], static_cast< double >(fixed) * 1.4210854715202004e-14); }
    }
}

__device__ __forceinline__ void block_epilogue(const BlockState& s, const DecoderParams& P) {
    __syncthreads();
    const int tid = threadIdx.x;
    flush_accumulators(s.accumulator, s.plan.accumulator_rows, P);
    if(tid < 2 && P.totals != nullptr && s.misc[tid]) { atomicAdd(&P.totals[tid], static_cast< unsigned long long >(s.misc[tid])); }
    if(tid >= 2 && tid < 4 && P.diagnostics != nullptr && s.misc[tid]) { atomicAdd(&P.diagnostics[tid - 2], static_cast< unsigned long long >(s.misc[tid])); }
}

/* the barcode table as a sequence of TMA-staged chunks; `iteration` counts chunks over the whole CTA lifetime */
struct BarcodeStream {
    const BlockState& s;
    const DecoderParams& P;
    const BarcodeEntry* source;         /* 16-byte entries: the barcode table, or its f32 form (FastEntry) */
    int chunk_cardinality;
    __device__ __forceinline__ BarcodeStream(const BlockState& s, const DecoderParams& P, const void* table = nullptr) : s(s), P(P) {
        source = table != nullptr ? static_cast< const BarcodeEntry* >(table) : P.barcodes;
        chunk_cardinality = (P.barcode_cardinality + s.plan.stage_capacity - 1) / s.plan.stage_capacity;
    }
    __device__ __forceinline__ int count(int chunk) const {
        const int remaining = P.barcode_cardinality - chunk * s.plan.stage_capacity;
        return remaining < s.plan.stage_capacity ? remaining : s.plan.stage_capacity;
    }
    /* one elected thread: arm the barrier of the buffer with the byte count and start the bulk copy */
    __device__ __forceinline__ void issue(unsigned iteration) const {
        const int chunk = iteration % chunk_cardinality;
        const int buffer = (s.plan.stage_buffers == 1) ? 0 : (iteration & 1u);
        const uint32_t bytes = static_cast< uint32_t >(count(chunk)) * 16u;
        mbarrier_expect_tx(&s.mbarrier[buffer], bytes);
        tma_bulk_load(s.stage + static_cast< size_t >(buffer) * s.plan.stage_capacity,
                      source + static_cast< size_t >(chunk) * s.plan.stage_capacity, bytes, &s.mbarrier[buffer]);
    }
    __device__ __forceinline__ const BarcodeEntry* wait(unsigned iteration) const {
        const int buffer = (s.plan.stage_buffers == 1) ? 0 : (iteration & 1u);
        const uint32_t use = (s.plan.stage_buffers == 1) ? iteration : (iteration >> 1);
        mbarrier_wait(&s.mbarrier[buffer], use & 1u);
        return s.stage + static_cast< size_t >(buffer) * s.plan.stage_capacity;
    }
};

/* ------------------------------------------------------------------ PAMLD hot loop pieces */

/* m = (o_lo ^ e_lo) | (o_hi ^ e_hi) | n_mask as two LOP3 (truth table 0xBE = (a ^ b) | c) */
__device__ __forceinline__ uint32_t mismatch_mask(uint32_t o_lo, uint32_t o_hi, uint32_t nmask, uint32_t e_lo, uint32_t e_hi) {
    uint32_t t, m;
    asm("lop3.b32 %0, %1, %2, %3, 0xBE;" : "=r"(t) : "r"(o_hi), "r"(e_hi), "r"(nmask));
    asm("lop3.b32 %0, %1, %2, %3, 0xBE;" : "=r"(m) : "r"(o_lo), "r"(e_lo), "r"(t));
    return m;
}
/*  Subset product of group g for mismatch mask m. The lane's table block is 4 KB aligned per group with
    entry e at byte e * 256 + lane * 8, so the address is (nibble g of m, moved to bits 8..11) | base:
    one shift and one LOP3 (truth table 0xEA = (a & b) | c), the group offset rides in the immediate. */
template < int g >
__device__ __forceinline__ double table_lookup(uint32_t base, uint32_t m) {
    const uint32_t moved = (g < 2) ? (m << (8 - 4 * g)) : (m >> (4 * g - 8));
    uint32_t address;
    asm("lop3.b32 %0, %1, 0xF00, %2, 0xEA;" : "=r"(address) : "r"(moved), "r"(base));
    double value;
    /* volatile: must stay behind the table stores of this tile (the compiler cannot see through the address) */
    asm volatile("ld.shared.f64 %0, [%1 + %2];" : "=d"(value) : "r"(address), "n"(g * 4096));
    return value;
}
template < int G >
__device__ __forceinline__ double subset_product(uint32_t base, uint32_t m) {
    /* ((T0 * T1) * T2) * ... : a fixed order, so equal mismatch sets give bit-equal products */
    double t = table_lookup< 0 >(base, m);
    if(G > 1) { t *= table_lookup< (G > 1 ? 1 : 0) >(base, m); }
    if(G > 2) { t *= table_lookup< (G > 2 ? 2 : 0) >(base, m); }
    if(G > 3) { t *= table_lookup< (G > 3 ? 3 : 0) >(base, m); }
    if(G > 4) { t *= table_lookup< (G > 4 ? 4 : 0) >(base, m); }
    if(G > 5) { t *= table_lookup< (G > 5 ? 5 : 0) >(base, m); }
    if(G > 6) { t *= table_lookup< (G > 6 ? 6 : 0) >(base, m); }
    if(G > 7) { t *= table_lookup< (G > 7 ? 7 : 0) >(base, m); }
    return t;
}

/*  Running selection state of one read. `best` is the first maximum seen so far (compared on the high
    words of the f64 products, strict >, earlier index wins), `rest` the sum of everything else, `second`
    the largest high word among the values that lost a comparison (tie detection). */
struct Selection {
    double best;
    double rest;
    int index;
    int second;
};
/* the larger of (a, ia) and (b, ib) with a the earlier one; the loser is returned in `low` */
__device__ __forceinline__ void duel(double a, int ia, double b, int ib, double& high, int& ihigh, double& low) {
    const bool later = __double2hiint(b) > __double2hiint(a);
    high = later ? b : a;
    ihigh = later ? ib : ia;
    low = later ? a : b;
}
__device__ __forceinline__ void select_one(Selection& s, double p, int i) {
    double high, low; int ihigh;
    duel(s.best, s.index, p, i, high, ihigh, low);
    s.best = high; s.index = ihigh;
    s.rest += low;
    s.second = max(s.second, __double2hiint(low));
}
/* four candidates reduced as a tree, then one merge with the running state: one serial step per four pairs */
__device__ __forceinline__ void select_four(Selection& s, double p0, double p1, double p2, double p3, int i) {
    double a, b, c, la, lb, lc, low; int ia, ib, ic, ihigh;
    duel(p0, i, p1, i + 1, a, ia, la);
    duel(p2, i + 2, p3, i + 3, b, ib, lb);
    duel(a, ia, b, ib, c, ic, lc);
    const double losers = (la + lb) + lc;
    const int second = max(max(__double2hiint(la), __double2hiint(lb)), __double2hiint(lc));
    double high;
    duel(s.best, s.index, c, ic, high, ihigh, low);
    s.best = high; s.index = ihigh;
    s.rest += losers + low;
    s.second = max(max(s.second, second), __double2hiint(low));
}

/*  The barcodes that can still tie with the running maximum. Two products tie in the reference when they are equal up
    to the rounding of its Kahan sums, i.e. their high words differ by at most one; so every barcode whose high word
    reaches (high word of the running maximum) - 1 when it is scanned is pushed, and a value that exceeds everything
    before it by more than that empties the list first. Whatever ties with the FINAL maximum is then in the list (the
    running maximum never exceeds the final one); stale entries are harmless, the tie pass evaluates what is listed and
    a barcode that is not a candidate loses. More than TIE_CANDIDATES pushes since the last reset = overflow: the tie
    pass scans the table itself. Used where the test is cheap: the exact path of the whitelist scan (per surviving
    candidate) and, as bit masks over the distinct words, the separable form of the combinatorial scan. */
template < int CAPACITY >
struct CandidateListOf {
    static constexpr int capacity = CAPACITY;
    uint32_t count;
    uint32_t entry[CAPACITY];
    __device__ __forceinline__ void reset() { count = 0u; }
    __device__ __forceinline__ void push(uint32_t index) {
        if(count < static_cast< uint32_t >(CAPACITY)) { entry[count] = index; }
        ++count;
    }
};
typedef CandidateListOf< TIE_CANDIDATES > CandidateList;
typedef CandidateListOf< TIE_POOLED_CANDIDATES > LongCandidateList;        /* local memory; only touched by the rare pushes */
template < class LIST >
__device__ __forceinline__ void capture_one(LIST& list, int& running, double p, int i) {
    const int h = __double2hiint(p);
    if(h >= running - 1) {
        if(h > running + 1) { list.reset(); }
        list.push(static_cast< uint32_t >(i));
        running = max(running, h);
    }
}
/*  The pair loops do not name single barcodes (a push per near tie costs a branch that some lane of nearly every
    block takes) but keep ONE bit per run of blocks of four: set when the largest high word of a block reaches (high word
    of the running maximum) - 1, the mask restarting when a block exceeds everything before it by more than that. Two
    compares and two selects per block, no branch; the tie pass evaluates the barcodes of the flagged runs. */
__device__ __forceinline__ void note_block(uint32_t& near_blocks, int running_high, int top, int index, int shift) {
    const uint32_t bit = 1u << (((index >> 2) >> shift) & 31);
    near_blocks = top > running_high + 1 ? bit : (top >= running_high - 1 ? (near_blocks | bit) : near_blocks);
}
__device__ __forceinline__ int top_high(double p0, double p1, double p2, double p3) {
    return max(max(__double2hiint(p0), __double2hiint(p1)), max(__double2hiint(p2), __double2hiint(p3)));
}
/* the CandidateList a pair loop hands to queue_ties: its block mask */
__device__ __forceinline__ CandidateList block_candidates(uint32_t near_blocks, int shift, bool grid_entries) {
    CandidateList list;
    list.count = TIE_BLOCKS;
    #pragma unroll
    for(int c = 0; c < TIE_CANDIDATES; ++c) { list.entry[c] = 0u; }
    list.entry[0] = near_blocks;
    list.entry[1] = static_cast< uint32_t >(shift);
    list.entry[2] = grid_entries ? 1u : 0u;
    return list;
}

/*  Selection over the word probabilities of one part of a separable codec: the maximum (first on equality),
    the largest of the others and the sum of the others. */
struct PartSelection {
    double best;
    double second;
    double rest;
    int index;
    uint32_t near;          /* words (first 32) that can still tie with the running maximum, as CandidateList does it */
};
__device__ __forceinline__ void select_part(PartSelection& s, double value, int i) {
    const int hv = __double2hiint(value), hb = __double2hiint(s.best);
    const uint32_t bit = 1u << (i & 31);
    s.near = hv > hb + 1 ? bit : (hv >= hb - 1 ? (s.near | bit) : s.near);
    const bool higher = value > s.best;
    const double low = higher ? s.best : value;
    s.index = higher ? i : s.index;
    s.best = higher ? value : s.best;
    s.second = fmax(s.second, low);
    s.rest += low;
}

/* ------------------------------------------------------------------ the observation of one read
   Everything a PAMLD scan needs from the tile planes. The scan kernels request the next tile's observation
   before they start on the current one, so the DRAM latency of the planes is hidden behind a whole tile of
   work even at the low occupancy the shared memory tables allow. */
template < int G >
struct ObservedRead {
    uint32_t o_lo, o_hi, nmask, qcfail;
    uint32_t raw[G];            /* quality plane words as they travelled (Phred bytes or codebook indices) */
};
template < int G >
__device__ __forceinline__ ObservedRead< G > fetch_read(const TileArguments& A, long long r) {
    ObservedRead< G > o;
    o.o_lo = 0; o.o_hi = 0; o.nmask = 0; o.qcfail = 0;
    #pragma unroll
    for(int g = 0; g < G; ++g) { o.raw[g] = 0; }
    if(r < A.n_reads) {
        const uint32_t w0 = load_stream(A.bases + r);
        o.o_lo = w0 & 0xffffu;
        o.o_hi = w0 >> 16;
        o.nmask = load_stream(A.nmask + r);
        if(G > 4) {
            const uint32_t w1 = load_stream(A.bases + A.pitch + r);
            o.o_lo |= w1 << 16;
            o.o_hi |= w1 & 0xffff0000u;
            o.nmask |= load_stream(A.nmask + A.pitch + r) << 16;
        }
        const int rows = (A.nucleotides * A.quality_bits + 31) >> 5;
        #pragma unroll
        for(int g = 0; g < G; ++g) { if(g < rows) { o.raw[g] = load_stream(A.quality + g * A.pitch + r); } }
        o.qcfail = A.qcfail[r];
    }
    return o;
}
/*  The scans work on reads 0 .. n_reads of the launch or, when the launch carries an index list (the reads an earlier
    kernel left to this one), on reads index_list[0 .. *index_count). Item -> read, or n_reads (which fetch_read
    answers with an empty observation) past the end. */
__device__ __forceinline__ long long item_cardinality_of(const TileArguments& A) {
    return A.index_list != nullptr ? static_cast< long long >(*A.index_count) : A.n_reads;
}
__device__ __forceinline__ long long read_of_item(const TileArguments& A, long long item, long long item_cardinality) {
    if(item >= item_cardinality) { return A.n_reads; }
    return A.index_list != nullptr ? static_cast< long long >(A.index_list[item]) : item;
}
/* the four Phred bytes of quality word g from the raw words (see quality_word) */
template < int G >
__device__ __forceinline__ uint32_t decode_quality(const TileArguments& A, const uint32_t (&raw)[G], int g) {
    if(A.quality_bits == 8) { return raw[g]; }
    const int valid = A.nucleotides - 4 * g;
    const uint32_t keep = valid >= 4 ? 0xffffffffu : (valid <= 0 ? 0u : ((1u << (8 * valid)) - 1u));
    if(A.quality_bits == 2) {
        const uint32_t c = (raw[g >> 2] >> (8 * (g & 3))) & 0xffu;
        const uint32_t selector = (c & 0x3u) | ((c & 0xcu) << 2) | ((c & 0x30u) << 4) | ((c & 0xc0u) << 6);
        return __byte_perm(A.codebook[0], 0u, selector) & keep;
    }
    const uint32_t c = (raw[g >> 1] >> (16 * (g & 1))) & 0xffffu;
    const uint32_t low = __byte_perm(A.codebook[0], A.codebook[1], c & 0x7777u);
    const uint32_t high = __byte_perm(A.codebook[2], A.codebook[3], c & 0x7777u);
    const uint32_t flag = ((c & 0x8u) >> 3) | ((c & 0x80u) << 1) | ((c & 0x800u) << 5) | ((c & 0x8000u) << 9);
    return (low ^ ((low ^ high) & (flag * 0xffu))) & keep;
}

/* ------------------------------------------------------------------ PAMLD decision
   pamld.cpp:87-122 followed by Decoder::classify (decoder.h:68-76) and Classifier::classify
   (classifier.h:78-86) for one read whose winner is known. `t` is the winner's subset product and
   `others` the sum of the prior adjusted products of all other barcodes, both relative to the per-read
   constant `base_probability` (P0), which is divided out of confidence = p / sigma_p (pamld.cpp:92). */
struct Verdict {
    int decoded;
    int distance;
    double confidence;
    uint32_t qcfail;
};
constexpr double WHITELIST_BAND = 4.76837158203125e-07;      /* = WHITELIST_TOLERANCE of pamld_whitelist_kernel */
/* the branches of pamld.cpp:96-122 and the accumulator updates, once P(r|b) and the confidence of the winner are known.
   GUARDED: the caller has already kept the confidence away from its threshold (the prefilter scans' 2^-38 guard is
   wider than the diagnostic's band), so only the other threshold is watched */
template < bool GUARDED = false >
__device__ __forceinline__ Verdict pamld_apply_counted(const DecoderParams& P, const Accumulator& accumulator, uint32_t* band_counter,
                                                       int best_index, int distance, int high_quality_distance, double conditional_probability,
                                                       double confidence, bool uniform, uint32_t qcfail) {
    Verdict v;
    v.confidence = confidence;
    v.distance = distance;
    v.decoded = best_index + 1;
    v.qcfail = qcfail;
    const int best_row = best_index + 1;

    /* diagnostic: reads whose decision sits within the accuracy of this path of a threshold. 1e-12 for the exact and
       prefilter scans; the pruned whitelist scan can move a confidence by up to 2^-21 (1 - confidence) */
    bool band = false;
    if(!GUARDED) {
        const double confidence_band = P.whitelist != nullptr ? fmax(1e-12, WHITELIST_BAND * (1.0 - v.confidence)) : 1e-12;
        band = fabs(v.confidence - P.confidence_threshold) <= confidence_band;
    }
    if(!uniform) { band = band || fabs(conditional_probability - P.random_barcode_probability) <= 1e-12 * P.random_barcode_probability; }
    if(band) { atomicAdd(band_counter, 1u); }

    if(conditional_probability > P.random_barcode_probability) {
        if(v.confidence > P.confidence_threshold) {
            if(P.high_quality_distance_threshold > 0 && high_quality_distance >= P.high_quality_distance_threshold) { v.qcfail = 1; }
            accumulator.add_pair(best_row, ACC_CONFIDENCE, ACC_PF_CONFIDENCE, v.confidence, !v.qcfail);
        } else {
            accumulator.add(best_row, ACC_LOW_CONFIDENCE, 1u);
            v.qcfail = 1;
        }
    } else {
        accumulator.add(best_row, ACC_LOW_CONDITIONAL, 1u);
        v.qcfail = 1;
        v.decoded = 0;
        v.distance = 0;
        v.confidence = 0.0;
    }
    if(v.decoded > 0 && v.distance > 0) {
        accumulator.add_pair(v.decoded, ACC_DISTANCE, ACC_PF_DISTANCE, static_cast< uint32_t >(v.distance), !v.qcfail);
    }
    accumulator.add_pair(v.decoded, ACC_COUNT, ACC_PF_COUNT, 1u, !v.qcfail);
    return v;
}
/* the same for a mismatch mask m of the winner over at most 32 positions */
template < bool GUARDED = false >
__device__ __forceinline__ Verdict pamld_apply(const DecoderParams& P, const Accumulator& accumulator, uint32_t* band_counter,
                                               int best_index, uint32_t m, double conditional_probability, double confidence,
                                               bool uniform, uint32_t high_quality_mask, uint32_t qcfail) {
    return pamld_apply_counted< GUARDED >(P, accumulator, band_counter, best_index, __popc(m), __popc(m & high_quality_mask), conditional_probability,
                                          confidence, uniform, qcfail);
}
__device__ __forceinline__ Verdict pamld_decide_counted(const DecoderParams& P, const Accumulator& accumulator, uint32_t* band_counter,
                                                        int best_index, int distance, int high_quality_distance, double t, double prior, double others,
                                                        double base_probability, bool uniform, uint32_t qcfail) {
    /* when every position scores UNIFORM_BASE_QUALITY all barcodes share sigma = L x U and the
       reference's P(r|b) is the host libm constant */
    if(uniform) { base_probability = P.uniform_observation_probability; }
    const double conditional_probability = base_probability * t;
    const double p = t * prior;
    const double sigma_p = p + (others + P.adjusted_noise_probability / base_probability);
    return pamld_apply_counted(P, accumulator, band_counter, best_index, distance, high_quality_distance, conditional_probability, p / sigma_p, uniform, qcfail);
}
__device__ __forceinline__ Verdict pamld_decide(const DecoderParams& P, const Accumulator& accumulator, uint32_t* band_counter,
                                                int best_index, uint32_t m, double t, double prior, double others,
                                                double base_probability, bool uniform, uint32_t high_quality_mask, uint32_t qcfail) {
    return pamld_decide_counted(P, accumulator, band_counter, best_index, __popc(m), __popc(m & high_quality_mask), t, prior, others,
                                base_probability, uniform, qcfail);
}

/* per-position factors of an observation: what one base contributes to P0 and to a mismatch product */
struct PositionFactor {
    double factor;          /* B ^ s(match)    : match_factor[q], B^U for an ambiguous base, 1 for q = 0 */
    double ratio;           /* B ^ (s(mismatch) - s(match)) : mismatch_ratio[q], 1 for ambiguous / q = 0 */
    bool uniform;           /* scores UNIFORM_BASE_QUALITY */
};
__device__ __forceinline__ PositionFactor position_factor(const double* __restrict__ phred_shared, double uniform_factor, uint32_t q, bool ambiguous) {
    PositionFactor f;
    q = phred_quality(q);
    f.factor = phred_shared[PHRED_MATCH_FACTOR + q];
    f.ratio = phred_shared[PHRED_MISMATCH_RATIO + q];
    f.uniform = ambiguous && q != 0u;
    if(f.uniform) { f.factor = uniform_factor; }
    if(ambiguous) { f.ratio = 1.0; }
    return f;
}

/* queue the lanes with `tied` set for the tie pass: one TieRecord each (one atomic per warp) */
template < int G, class LIST >
__device__ __forceinline__ void queue_ties(const DecoderParams& P, bool tied, int lane, const Selection& selection, double base_probability,
                                           uint32_t high_quality_mask, bool uniform, uint32_t o_lo, uint32_t o_hi, uint32_t nmask, long long r,
                                           const uint32_t (&quality)[G], const LIST& candidates) {
    const unsigned queued = __ballot_sync(FULL_MASK, tied);
    if(queued) {
        unsigned slot = 0;
        if(lane == 0) { slot = atomicAdd(P.tie_count, static_cast< unsigned >(__popc(queued))); }
        slot = __shfl_sync(FULL_MASK, slot, 0);
        if(tied) {
            const unsigned at = slot + __popc(queued & ((1u << lane) - 1u));
            TieRecord record;
            record.best = selection.best;
            record.rest = selection.rest;
            record.base_probability = base_probability;
            record.high_quality_mask = high_quality_mask;
            record.uniform = uniform ? 1u : 0u;
            record.o_lo = o_lo;
            record.o_hi = o_hi;
            record.nmask = nmask;
            record.read = static_cast< uint32_t >(r);
            #pragma unroll
            for(int g = 0; g < 8; ++g) { record.quality[g] = g < G ? quality[g < G ? g : 0] : 0u; }
            #pragma unroll
            for(int c = 0; c < TIE_CANDIDATES; ++c) { record.candidate[c] = c < LIST::capacity ? candidates.entry[c < LIST::capacity ? c : 0] : 0u; }
            record.candidate_count = candidates.count;
            if(candidates.count > static_cast< uint32_t >(TIE_CANDIDATES) && candidates.count != TIE_BLOCKS && candidates.count != TIE_MASKS) {
                record.candidate_count = TIE_RESCAN;
                if(candidates.count <= static_cast< uint32_t >(LIST::capacity) && P.tie_pool != nullptr) {
                    /* more than a record holds: the list goes to the pool */
                    const uint32_t first = atomicAdd(P.tie_count + 3, candidates.count);
                    if(first + candidates.count <= P.tie_pool_capacity) {
                        for(uint32_t c = 0; c < candidates.count; ++c) { P.tie_pool[first + c] = candidates.entry[c < static_cast< uint32_t >(LIST::capacity) ? c : 0]; }
                        record.candidate_count = TIE_POOLED | candidates.count;
                        record.candidate[0] = first;
                    }
                }
            }
            P.tie_record[at] = record;
        }
    }
}

/* ------------------------------------------------------------------ PAMLD scan kernel */
/* warps per CTA of the generic scan: as many as the per-warp tables (G x 4 KB) and the register file allow; short
   barcodes leave room for more warps, which is what hides the latency of the dependent lookup -> multiply chains */
__host__ __device__ constexpr int pamld_warps(int G) { return G <= 2 ? 20 : (G == 3 ? 16 : MAX_WARPS); }

template < int G >
__global__ void __launch_bounds__(pamld_warps(G) * WARP_SIZE, 1)
pamld_kernel(const DecoderParams P, const TileArguments A) {
    extern __shared__ __align__(256) unsigned char smem[];
    const BlockState S = block_prologue(smem, P, true);
    const BarcodeStream stream(S, P);
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    /* per-lane subset product tables: entry (g, subset) of this lane at [(g * 16 + subset) * 32 + lane] */
    const uint32_t window = shared_address(smem);
    const uint32_t aligned_tables = ((window + S.plan.off_tables + 4095u) & ~4095u) - window;
    double* const table = reinterpret_cast< double* >(smem + aligned_tables) + static_cast< size_t >(warp) * (G * 16 * WARP_SIZE) + lane;
    const uint32_t table_base = shared_address(table);
    const double uniform_factor = P.phred[PHRED_UNIFORM_FACTOR];
    const int L = P.nucleotide_cardinality;

    const long long items = item_cardinality_of(A);
    const long long tile_cardinality = (items + blockDim.x - 1) / blockDim.x;
    const long long my_tiles = tile_cardinality > blockIdx.x ? (tile_cardinality - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const unsigned long long total_iterations = static_cast< unsigned long long >(my_tiles) * stream.chunk_cardinality;
    unsigned iteration = 0;
    if(tid == 0 && total_iterations > 0) { stream.issue(0); }
    const bool resident = stream.chunk_cardinality == 1;     /* whole table staged once */
    const BarcodeEntry* resident_stage = nullptr;
    if(resident && total_iterations > 0) { resident_stage = stream.wait(0); }

    /* the observation of the next tile and the read number of the one after it are requested a tile ahead: in index-list
       mode the planes cannot be requested before the list entry has arrived */
    long long upcoming_read = read_of_item(A, static_cast< long long >(blockIdx.x) * blockDim.x + tid, items);
    long long following_read = read_of_item(A, (static_cast< long long >(blockIdx.x) + gridDim.x) * blockDim.x + tid, items);
    ObservedRead< G > upcoming = fetch_read< G >(A, upcoming_read);
    for(long long tile = blockIdx.x; tile < tile_cardinality; tile += gridDim.x) {
        const long long r = upcoming_read;
        const bool valid = r < A.n_reads;

        /* ---- this lane's read (requested one tile ago); request the next one */
        const ObservedRead< G > observed = upcoming;
        upcoming_read = following_read;
        following_read = read_of_item(A, (tile + 2 * static_cast< long long >(gridDim.x)) * blockDim.x + tid, items);
        upcoming = fetch_read< G >(A, upcoming_read);
        const uint32_t o_lo = observed.o_lo, o_hi = observed.o_hi, nmask = observed.nmask;
        uint32_t qcfail = observed.qcfail;
        uint32_t quality[G];
        #pragma unroll
        for(int g = 0; g < G; ++g) { quality[g] = decode_quality< G >(A, observed.raw, g); }

        /* ---- per-read constant P0, subset product tables, high quality mask */
        double base_probability = 1.0;
        uint32_t high_quality_mask = 0;
        int uniform_positions = 0;
        #pragma unroll
        for(int g = 0; g < G; ++g) {
            double w[4];
            #pragma unroll
            for(int k = 0; k < 4; ++k) {
                const int j = g * 4 + k;
                const uint32_t q = (quality[g] >> (8 * k)) & 0xffu;
                if(static_cast< int >(q) >= P.high_quality_threshold) { high_quality_mask |= 1u << j; }
                const PositionFactor f = position_factor(S.phred, uniform_factor, q, (nmask >> j) & 1u);
                uniform_positions += f.uniform ? 1 : 0;
                base_probability *= f.factor;
                w[k] = f.ratio;
            }
            double* const t = table + g * 16 * WARP_SIZE;
            const double w01 = w[0] * w[1];
            const double w02 = w[0] * w[2];
            const double w12 = w[1] * w[2];
            const double w012 = w01 * w[2];
            t[0 * WARP_SIZE] = 1.0;
            t[1 * WARP_SIZE] = w[0];
            t[2 * WARP_SIZE] = w[1];
            t[3 * WARP_SIZE] = w01;
            t[4 * WARP_SIZE] = w[2];
            t[5 * WARP_SIZE] = w02;
            t[6 * WARP_SIZE] = w12;
            t[7 * WARP_SIZE] = w012;
            t[8 * WARP_SIZE] = w[3];
            t[9 * WARP_SIZE] = w[0] * w[3];
            t[10 * WARP_SIZE] = w[1] * w[3];
            t[11 * WARP_SIZE] = w01 * w[3];
            t[12 * WARP_SIZE] = w[2] * w[3];
            t[13 * WARP_SIZE] = w02 * w[3];
            t[14 * WARP_SIZE] = w12 * w[3];
            t[15 * WARP_SIZE] = w012 * w[3];
        }
        high_quality_mask &= (L >= 32) ? 0xffffffffu : ((1u << L) - 1u);
        __syncwarp();

        /* ---- score every barcode. The reference Kahan-sums p over the barcodes (pamld.cpp:68-72); here the
           running maximum is kept out of the sum (`rest` only ever receives the loser of a comparison), so no
           small term is absorbed by a dominant one and best + rest is accurate to an ulp without
           compensation. The first maximum (strict >, pamld.cpp:73) is tracked on the high words. */
        Selection selection;
        selection.best = 0.0; selection.rest = 0.0; selection.index = 0; selection.second = 0;
        uint32_t near_blocks = 0u;              /* runs of barcodes that can hold the winner of a tie (note_block) */
        for(int chunk = 0; chunk < stream.chunk_cardinality; ++chunk) {
            const BarcodeEntry* stage;
            if(resident) {
                stage = resident_stage;
            } else {
                if(tid == 0 && iteration + 1 < total_iterations) { stream.issue(iteration + 1); }
                stage = stream.wait(iteration);
            }
            const int count = stream.count(chunk);
            const int first = chunk * S.plan.stage_capacity;
            int i = 0;
            #pragma unroll 2
            for(; i + 4 <= count; i += 4) {
                double p[4];
                #pragma unroll
                for(int u = 0; u < 4; ++u) {
                    const uint4 raw = *reinterpret_cast< const uint4* >(stage + i + u);
                    const uint32_t m = mismatch_mask(o_lo, o_hi, nmask, raw.x, raw.y);
                    p[u] = subset_product< G >(table_base, m) * __hiloint2double(raw.w, raw.z);
                }
                note_block(near_blocks, __double2hiint(selection.best), top_high(p[0], p[1], p[2], p[3]), first + i, P.tie_block_shift);
                select_four(selection, p[0], p[1], p[2], p[3], first + i);
            }
            for(; i < count; ++i) {
                const uint4 raw = *reinterpret_cast< const uint4* >(stage + i);
                const uint32_t m = mismatch_mask(o_lo, o_hi, nmask, raw.x, raw.y);
                const double p = subset_product< G >(table_base, m) * __hiloint2double(raw.w, raw.z);
                note_block(near_blocks, __double2hiint(selection.best), __double2hiint(p), first + i, P.tie_block_shift);
                select_one(selection, p, first + i);
            }
            if(!resident) {
                __syncthreads();
                ++iteration;
            }
        }

        /* ---- structural ties (runner-up within 2^-19 of the winner) are resolved by the reference through the
           rounding of its Kahan sums; pamld_tie_kernel reproduces that. Such reads are only queued here. */
        const bool tied = valid && (selection.second + 1 >= __double2hiint(selection.best));
        queue_ties< G, CandidateList >(P, tied, lane, selection, base_probability, high_quality_mask, uniform_positions == L, o_lo, o_hi, nmask, r, quality,
                                       block_candidates(near_blocks, P.tie_block_shift, false));

        /* ---- decision for this lane's read */
        const bool decided = valid && !tied;
        if(decided) {
            const BarcodeEntry e = P.barcodes[selection.index];
            const uint32_t m = mismatch_mask(o_lo, o_hi, nmask, e.lo, e.hi);
            const double t = subset_product< G >(table_base, m);
            const Verdict v = pamld_decide(P, S.accumulator, &S.misc[3], selection.index, m, t, e.prior, selection.rest, base_probability,
                                           uniform_positions == L, high_quality_mask, qcfail);
            qcfail = v.qcfail;
            A.qcfail[r] = static_cast< uint8_t >(v.qcfail);
            store_result(A, r, v.decoded, v.distance, v.confidence, v.qcfail);
        }
        if(P.totals != nullptr) {
            const unsigned live = __ballot_sync(FULL_MASK, decided);
            const unsigned pass = __ballot_sync(FULL_MASK, decided && !qcfail);
            if(lane == 0) {
                atomicAdd(&S.misc[0], static_cast< uint32_t >(__popc(live)));
                atomicAdd(&S.misc[1], static_cast< uint32_t >(__popc(pass)));
            }
        }
        __syncwarp();
    }
    block_epilogue(S, P);
}

/* ------------------------------------------------------------------ long barcodes (33-64 nucleotides)
   The observation and the barcodes travel in split form (LongBarcodeEntry): word 0 = positions [0, split), word 1 =
   positions [split, L), split = 4 H with H = ceil(L / 8) groups of four positions per word. */
constexpr int LONG_STAGE_ENTRIES = 256;          /* long barcodes per staged chunk: 8 KB */
constexpr int LONG_MAX_WARPS = 16;
/* the staging area of the long kernels in 16-byte units, as make_plan's blob_entries: one chunk, or two when the table streams */
__host__ __device__ inline int long_stage_blob(int barcode_cardinality) {
    return barcode_cardinality <= LONG_STAGE_ENTRIES ? 2 * barcode_cardinality : 4 * LONG_STAGE_ENTRIES;
}

struct LongObservation {
    uint32_t lo[2], hi[2], nmask[2];    /* split form */
    uint32_t qcfail;
};
/* the planes of read r in split form; positions past L are cleared */
__device__ __forceinline__ LongObservation fetch_long_observation(const TileArguments& A, long long r, int split) {
    LongObservation o;
    uint64_t lo = 0, hi = 0, n = 0;
    const int words = (A.nucleotides + 15) >> 4;
    #pragma unroll
    for(int w = 0; w < PHQ_MAX_NUCLEOTIDES / 16; ++w) {
        if(w < words) {
            const uint32_t b = load_stream(A.bases + w * A.pitch + r);
            lo |= static_cast< uint64_t >(b & 0xffffu) << (16 * w);
            hi |= static_cast< uint64_t >(b >> 16) << (16 * w);
            n |= static_cast< uint64_t >(load_stream(A.nmask + w * A.pitch + r)) << (16 * w);
        }
    }
    const uint64_t observed = A.nucleotides >= 64 ? ~0ull : ((1ull << A.nucleotides) - 1ull);
    const uint64_t first = (1ull << split) - 1ull;
    lo &= observed; hi &= observed; n &= observed;
    o.lo[0] = static_cast< uint32_t >(lo & first); o.lo[1] = static_cast< uint32_t >(lo >> split);
    o.hi[0] = static_cast< uint32_t >(hi & first); o.hi[1] = static_cast< uint32_t >(hi >> split);
    o.nmask[0] = static_cast< uint32_t >(n & first); o.nmask[1] = static_cast< uint32_t >(n >> split);
    o.qcfail = A.qcfail[r];
    return o;
}

/* the long barcode table as TMA-staged chunks of 32-byte entries (BarcodeStream for LongBarcodeEntry) */
struct LongBarcodeStream {
    const BlockState& s;
    const DecoderParams& P;
    LongBarcodeEntry* stage;
    int capacity;
    int buffers;
    int chunk_cardinality;
    __device__ __forceinline__ LongBarcodeStream(const BlockState& s, const DecoderParams& P) : s(s), P(P) {
        stage = reinterpret_cast< LongBarcodeEntry* >(s.stage);
        capacity = P.barcode_cardinality < LONG_STAGE_ENTRIES ? P.barcode_cardinality : LONG_STAGE_ENTRIES;
        buffers = P.barcode_cardinality <= LONG_STAGE_ENTRIES ? 1 : 2;
        chunk_cardinality = (P.barcode_cardinality + capacity - 1) / capacity;
    }
    __device__ __forceinline__ int count(int chunk) const {
        const int remaining = P.barcode_cardinality - chunk * capacity;
        return remaining < capacity ? remaining : capacity;
    }
    __device__ __forceinline__ void issue(unsigned iteration) const {
        const int chunk = iteration % chunk_cardinality;
        const int buffer = buffers == 1 ? 0 : (iteration & 1u);
        const uint32_t bytes = static_cast< uint32_t >(count(chunk)) * 32u;
        mbarrier_expect_tx(&s.mbarrier[buffer], bytes);
        tma_bulk_load(stage + static_cast< size_t >(buffer) * capacity, P.long_barcodes + static_cast< size_t >(chunk) * capacity, bytes, &s.mbarrier[buffer]);
    }
    __device__ __forceinline__ const LongBarcodeEntry* wait(unsigned iteration) const {
        const int buffer = buffers == 1 ? 0 : (iteration & 1u);
        const uint32_t use = buffers == 1 ? iteration : (iteration >> 1);
        mbarrier_wait(&s.mbarrier[buffer], use & 1u);
        return stage + static_cast< size_t >(buffer) * capacity;
    }
};

/*  PAMLD scan for 33-64 nucleotides. A LANE PAIR owns one read: lane 2k + h holds the subset product tables of word h
    of the split form (H groups, H x 4 KB per warp, as pamld_kernel< H > holds them for a whole read), so a warp keeps
    16 reads and the shared memory a warp needs stays that of a 32-nucleotide scan. For every barcode each lane forms
    the product over its word, the pair swaps the halves with one shuffle and both lanes hold p = (t0 * t1) * prior
    bit for bit, so both run the same selection; the even lane queues ties and takes the decision. */
template < int H >
__global__ void __launch_bounds__(LONG_MAX_WARPS * WARP_SIZE, 1)
pamld_long_kernel(const DecoderParams P, const TileArguments A) {
    extern __shared__ __align__(256) unsigned char smem[];
    const BlockState S = block_prologue(smem, P, true, long_stage_blob(P.barcode_cardinality));
    const LongBarcodeStream stream(S, P);
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int half = lane & 1;
    const uint32_t window = shared_address(smem);
    const uint32_t aligned_tables = ((window + S.plan.off_tables + 4095u) & ~4095u) - window;
    double* const table = reinterpret_cast< double* >(smem + aligned_tables) + static_cast< size_t >(warp) * (H * 16 * WARP_SIZE) + lane;
    const uint32_t table_base = shared_address(table);
    const double uniform_factor = P.phred[PHRED_UNIFORM_FACTOR];
    const int L = P.nucleotide_cardinality;
    const int G = (L + 3) >> 2;
    /* positions of this lane's word that the observation has */
    const int own_positions = half == 0 ? 4 * H : L - 4 * H;
    const uint32_t own_mask = own_positions >= 32 ? 0xffffffffu : ((1u << own_positions) - 1u);

    const long long items = A.n_reads;
    const int pairs = blockDim.x >> 1;
    const long long tile_cardinality = (items + pairs - 1) / pairs;
    const long long my_tiles = tile_cardinality > blockIdx.x ? (tile_cardinality - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const unsigned long long total_iterations = static_cast< unsigned long long >(my_tiles) * stream.chunk_cardinality;
    unsigned iteration = 0;
    if(tid == 0 && total_iterations > 0) { stream.issue(0); }
    const bool resident = stream.chunk_cardinality == 1;
    const LongBarcodeEntry* resident_stage = nullptr;
    if(resident && total_iterations > 0) { resident_stage = stream.wait(0); }

    for(long long tile = blockIdx.x; tile < tile_cardinality; tile += gridDim.x) {
        const long long item = tile * pairs + (tid >> 1);
        const bool valid = item < items;
        const long long r = valid ? item : A.n_reads;
        uint32_t o_lo = 0, o_hi = 0, nmask = 0, qcfail = 0;
        uint32_t quality[H];
        #pragma unroll
        for(int g = 0; g < H; ++g) { quality[g] = 0; }
        if(valid) {
            const LongObservation o = fetch_long_observation(A, r, 4 * H);
            o_lo = half ? o.lo[1] : o.lo[0]; o_hi = half ? o.hi[1] : o.hi[0]; nmask = half ? o.nmask[1] : o.nmask[0]; qcfail = o.qcfail;
            #pragma unroll
            for(int g = 0; g < H; ++g) {
                const int group = half * H + g;
                if(group < G) { quality[g] = quality_word(A, r, group); }
            }
        }

        /* ---- this lane's factor of P0, its subset product tables and high quality positions */
        double own_probability = 1.0;
        uint32_t own_high_quality = 0;
        int own_uniform = 0;
        #pragma unroll
        for(int g = 0; g < H; ++g) {
            double w[4];
            #pragma unroll
            for(int k = 0; k < 4; ++k) {
                const int j = g * 4 + k;
                const uint32_t q = (quality[g] >> (8 * k)) & 0xffu;
                if(static_cast< int >(q) >= P.high_quality_threshold) { own_high_quality |= 1u << j; }
                const PositionFactor f = position_factor(S.phred, uniform_factor, q, (nmask >> j) & 1u);
                own_uniform += f.uniform ? 1 : 0;
                own_probability *= f.factor;
                w[k] = f.ratio;
            }
            double* const t = table + g * 16 * WARP_SIZE;
            const double w01 = w[0] * w[1];
            const double w02 = w[0] * w[2];
            const double w12 = w[1] * w[2];
            const double w012 = w01 * w[2];
            t[0 * WARP_SIZE] = 1.0;
            t[1 * WARP_SIZE] = w[0];
            t[2 * WARP_SIZE] = w[1];
            t[3 * WARP_SIZE] = w01;
            t[4 * WARP_SIZE] = w[2];
            t[5 * WARP_SIZE] = w02;
            t[6 * WARP_SIZE] = w12;
            t[7 * WARP_SIZE] = w012;
            t[8 * WARP_SIZE] = w[3];
            t[9 * WARP_SIZE] = w[0] * w[3];
            t[10 * WARP_SIZE] = w[1] * w[3];
            t[11 * WARP_SIZE] = w01 * w[3];
            t[12 * WARP_SIZE] = w[2] * w[3];
            t[13 * WARP_SIZE] = w02 * w[3];
            t[14 * WARP_SIZE] = w12 * w[3];
            t[15 * WARP_SIZE] = w012 * w[3];
        }
        own_high_quality &= own_mask;
        const double other_probability = __shfl_xor_sync(FULL_MASK, own_probability, 1);
        const double base_probability = own_probability * other_probability;
        const int uniform_positions = own_uniform + __shfl_xor_sync(FULL_MASK, own_uniform, 1);
        __syncwarp();

        /* ---- score every barcode (pamld_kernel's selection, on the products both lanes of the pair hold) */
        Selection selection;
        selection.best = 0.0; selection.rest = 0.0; selection.index = 0; selection.second = 0;
        uint32_t near_blocks = 0u;
        for(int chunk = 0; chunk < stream.chunk_cardinality; ++chunk) {
            const LongBarcodeEntry* stage;
            if(resident) {
                stage = resident_stage;
            } else {
                if(tid == 0 && iteration + 1 < total_iterations) { stream.issue(iteration + 1); }
                stage = stream.wait(iteration);
            }
            const int count = stream.count(chunk);
            const int first = chunk * stream.capacity;
            int i = 0;
            #pragma unroll 2
            for(; i + 4 <= count; i += 4) {
                double p[4];
                #pragma unroll
                for(int u = 0; u < 4; ++u) {
                    const uint2 planes = reinterpret_cast< const uint2* >(stage + i + u)[half];
                    const double own = subset_product< H >(table_base, mismatch_mask(o_lo, o_hi, nmask, planes.x, planes.y));
                    const double other = __shfl_xor_sync(FULL_MASK, own, 1);
                    p[u] = (own * other) * stage[i + u].prior;       /* a product does not depend on the order of its factors */
                }
                note_block(near_blocks, __double2hiint(selection.best), top_high(p[0], p[1], p[2], p[3]), first + i, P.tie_block_shift);
                select_four(selection, p[0], p[1], p[2], p[3], first + i);
            }
            for(; i < count; ++i) {
                const uint2 planes = reinterpret_cast< const uint2* >(stage + i)[half];
                const double own = subset_product< H >(table_base, mismatch_mask(o_lo, o_hi, nmask, planes.x, planes.y));
                const double other = __shfl_xor_sync(FULL_MASK, own, 1);
                const double p = (own * other) * stage[i].prior;
                note_block(near_blocks, __double2hiint(selection.best), __double2hiint(p), first + i, P.tie_block_shift);
                select_one(selection, p, first + i);
            }
            if(!resident) {
                __syncthreads();
                ++iteration;
            }
        }

        /* ---- ties go to pamld_long_tie_kernel, which reads the observation from the tile again: the record keeps the
           scan's sums, P0 and the flagged runs of barcodes */
        const bool tied = valid && (selection.second + 1 >= __double2hiint(selection.best));
        const bool queued = tied && half == 0;
        const unsigned queue = __ballot_sync(FULL_MASK, queued);
        if(queue) {
            unsigned slot = 0;
            if(lane == 0) { slot = atomicAdd(P.tie_count, static_cast< unsigned >(__popc(queue))); }
            slot = __shfl_sync(FULL_MASK, slot, 0);
            if(queued) {
                TieRecord record;
                memset(&record, 0, sizeof(record));
                record.best = selection.best;
                record.rest = selection.rest;
                record.base_probability = base_probability;
                record.uniform = uniform_positions == L ? 1u : 0u;
                record.read = static_cast< uint32_t >(r);
                record.candidate_count = TIE_BLOCKS;
                record.candidate[0] = near_blocks;
                record.candidate[1] = static_cast< uint32_t >(P.tie_block_shift);
                P.tie_record[slot + __popc(queue & ((1u << lane) - 1u))] = record;
            }
        }

        /* ---- the decision: both lanes form their half of the winner's product and mismatch counts */
        const LongBarcodeEntry& winner = P.long_barcodes[selection.index];
        const uint2 planes = reinterpret_cast< const uint2* >(&winner)[half];
        const uint32_t m = mismatch_mask(o_lo, o_hi, nmask, planes.x, planes.y);
        const double own_t = subset_product< H >(table_base, m);
        const double other_t = __shfl_xor_sync(FULL_MASK, own_t, 1);
        const int distance = __popc(m) + __shfl_xor_sync(FULL_MASK, __popc(m), 1);
        const int high_quality_distance = __popc(m & own_high_quality) + __shfl_xor_sync(FULL_MASK, __popc(m & own_high_quality), 1);
        const bool decided = valid && !tied && half == 0;
        if(decided) {
            const Verdict v = pamld_decide_counted(P, S.accumulator, &S.misc[3], selection.index, distance, high_quality_distance, own_t * other_t, winner.prior,
                                                   selection.rest, base_probability, uniform_positions == L, qcfail);
            qcfail = v.qcfail;
            A.qcfail[r] = static_cast< uint8_t >(v.qcfail);
            store_result(A, r, v.decoded, v.distance, v.confidence, v.qcfail);
        }
        if(P.totals != nullptr) {
            const unsigned live = __ballot_sync(FULL_MASK, decided);
            const unsigned pass = __ballot_sync(FULL_MASK, decided && !qcfail);
            if(lane == 0) {
                atomicAdd(&S.misc[0], static_cast< uint32_t >(__popc(live)));
                atomicAdd(&S.misc[1], static_cast< uint32_t >(__popc(pass)));
            }
        }
        __syncwarp();
    }
    block_epilogue(S, P);
}

/* ------------------------------------------------------------------ PAMLD scan kernel for combinatorial codecs
   Multi-segment codecs are usually combinatorial: C1's 96 dual-index barcodes are 12 distinct i7 words
   x 8 distinct i5 words. P(r|b) factors over segments, so with A = the first segment and B = the rest

       p_b = SA[word_A(b)] * SB[word_B(b)] * prior_b

   The kernel computes SB for every distinct B word once per read into a per-lane column in shared memory,
   then walks the barcodes grouped by A word: SA is formed once per A word (uniform loop) and each barcode
   costs ONE conflict-free LDS.64 (its SB entry), two DMUL and the selection step, instead of four lookups,
   a mismatch mask and address arithmetic. The scan order is (A word, index); exact ties are queued for
   pamld_tie_kernel like in the generic kernel, so the first-maximum rule is not affected. */
struct __align__(16) GridHeader { uint32_t lo, hi, first, count; };                 /* a distinct A word and its run of entries */
struct __align__(16) GridWord { uint32_t lo, hi, pad0, pad1; };                     /* a distinct B word */
struct __align__(16) GridEntry { uint32_t suffix_offset; uint32_t index; double prior; };   /* a barcode: SB row (bytes), original index */

/*  Subset tables of the combinatorial scan use groups of W positions (2^W entries of 256 bytes per group and
    warp). The scan itself does one SB lookup per barcode, so the tables are only read ~44 times per read:
    W = 2 halves their footprint (8 KB per warp at 16 nucleotides) and doubles the resident warps. */
template < int W, int table_group, int local >
__device__ __forceinline__ double group_lookup(uint32_t base, uint32_t m) {
    constexpr int shift = 8 - W * local;        /* bits W*local.. of m land on bits 8.. of the address */
    const uint32_t moved = (shift >= 0) ? (m << (shift >= 0 ? shift : 0)) : (m >> (shift >= 0 ? 0 : -shift));
    uint32_t address;
    asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(address) : "r"(moved), "n"(((1 << W) - 1) << 8), "r"(base));
    double value;
    asm volatile("ld.shared.f64 %0, [%1 + %2];" : "=d"(value) : "r"(address), "n"(table_group * (256 << W)));
    return value;
}
/* product over the GROUPS groups of a part whose first table group is `first`; m = the part's mismatch bits from bit 0 */
template < int W, int first, int GROUPS, int k >
struct PartProduct {
    static __device__ __forceinline__ double of(uint32_t base, uint32_t m, double t) {
        return PartProduct< W, first, GROUPS, k + 1 >::of(base, m, t * group_lookup< W, first + k, k >(base, m));
    }
};
template < int W, int first, int GROUPS >
struct PartProduct< W, first, GROUPS, GROUPS > {
    static __device__ __forceinline__ double of(uint32_t, uint32_t, double t) { return t; }
};
template < int W, int first, int GROUPS >
__device__ __forceinline__ double part_product(uint32_t base, uint32_t m) {
    return PartProduct< W, first, GROUPS, 1 >::of(base, m, group_lookup< W, first, 0 >(base, m));
}
__device__ __forceinline__ double column_load(uint32_t address) {
    double value;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(value) : "r"(address));
    return value;
}

constexpr int GRID_MAX_WARPS = 20;
constexpr int GRID_GROUP_WIDTH = 2;

/*  KBP > 0 selects the dense form: the codec fills (most of) the grid of A words x B words, the B word
    probabilities stay in KBP registers and the barcodes of an A word are its KBP consecutive entries (absent
    combinations have prior 0), so the scan loop has no per-lane shared memory traffic at all. UNIFORM
    additionally drops the prior from the loop when every combination is present with the same prior. */
template < int LA, int LB, int W, int KBP, bool UNIFORM >
__global__ void __launch_bounds__(GRID_MAX_WARPS * WARP_SIZE, 1)
pamld_grid_kernel(const DecoderParams P, const TileArguments A) {
    constexpr int L = LA + LB;
    constexpr int G = (L + 3) / 4;              /* quality words */
    constexpr int GA = (LA + W - 1) / W;        /* table groups of W positions per part */
    constexpr int GB = (LB + W - 1) / W;
    constexpr int GROUP_BYTES = 256 << W;
    constexpr uint32_t MASK_A = (1u << LA) - 1u;
    constexpr uint32_t MASK_B = (1u << LB) - 1u;
    extern __shared__ __align__(256) unsigned char smem[];
    const BlockState S = block_prologue(smem, P, true, P.grid_a + P.grid_b + P.grid_entries);
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int warp_cardinality = blockDim.x >> 5;
    const int KA = P.grid_a;
    const int KB = P.grid_b;

    /* the grid blob (headers, B words, entries) is staged once per CTA by one TMA bulk copy */
    const GridHeader* const header = reinterpret_cast< const GridHeader* >(smem + S.plan.off_stage);
    const GridWord* const word = reinterpret_cast< const GridWord* >(header + KA);
    const GridEntry* const entry = reinterpret_cast< const GridEntry* >(word + KB);
    if(tid == 0) {
        const uint32_t bytes = static_cast< uint32_t >(KA + KB + P.grid_entries) * 16u;
        mbarrier_expect_tx(&S.mbarrier[0], bytes);
        tma_bulk_load(smem + S.plan.off_stage, P.grid, bytes, &S.mbarrier[0]);
    }
    mbarrier_wait(&S.mbarrier[0], 0);

    /* per warp: (GA + GB) table groups of 2^W entries x 256 bytes, then KB rows of 256 bytes for the B word products */
    const uint32_t window = shared_address(smem);
    const uint32_t aligned_tables = ((window + S.plan.off_tables + 4095u) & ~4095u) - window;
    const size_t warp_bytes = static_cast< size_t >(GA + GB) * GROUP_BYTES;
    double* const table = reinterpret_cast< double* >(smem + aligned_tables + warp * warp_bytes) + lane;
    const uint32_t table_base = shared_address(table);
    double* const suffix = reinterpret_cast< double* >(smem + aligned_tables + warp_cardinality * warp_bytes + static_cast< size_t >(warp) * KB * 256) + lane;
    const uint32_t suffix_base = shared_address(suffix);
    const double uniform_factor = P.phred[PHRED_UNIFORM_FACTOR];

    const long long items = item_cardinality_of(A);
    const long long tile_cardinality = (items + blockDim.x - 1) / blockDim.x;
    long long upcoming_read = read_of_item(A, static_cast< long long >(blockIdx.x) * blockDim.x + tid, items);
    long long following_read = read_of_item(A, (static_cast< long long >(blockIdx.x) + gridDim.x) * blockDim.x + tid, items);
    ObservedRead< G > upcoming = fetch_read< G >(A, upcoming_read);
    for(long long tile = blockIdx.x; tile < tile_cardinality; tile += gridDim.x) {
        const long long r = upcoming_read;
        const bool valid = r < A.n_reads;

        /* this lane's read (requested one tile ago); request the next one (and the read number of the one after it) */
        const ObservedRead< G > observed = upcoming;
        upcoming_read = following_read;
        following_read = read_of_item(A, (tile + 2 * static_cast< long long >(gridDim.x)) * blockDim.x + tid, items);
        upcoming = fetch_read< G >(A, upcoming_read);
        const uint32_t o_lo = observed.o_lo, o_hi = observed.o_hi, nmask = observed.nmask;
        uint32_t qcfail = observed.qcfail;
        uint32_t quality[G];
        #pragma unroll
        for(int g = 0; g < G; ++g) { quality[g] = decode_quality< G >(A, observed.raw, g); }

        /* ---- per-position factors; P0 in position order; subset tables per part */
        double base_probability = 1.0;
        uint32_t high_quality_mask = 0;
        int uniform_positions = 0;
        double w[(GA + GB) * W];
        #pragma unroll
        for(int k = 0; k < (GA + GB) * W; ++k) { w[k] = 1.0; }
        #pragma unroll
        for(int j = 0; j < L; ++j) {
            const uint32_t q = (quality[j >> 2] >> (8 * (j & 3))) & 0xffu;
            if(static_cast< int >(q) >= P.high_quality_threshold) { high_quality_mask |= 1u << j; }
            const PositionFactor f = position_factor(S.phred, uniform_factor, q, (nmask >> j) & 1u);
            uniform_positions += f.uniform ? 1 : 0;
            base_probability *= f.factor;
            w[j < LA ? j : GA * W + (j - LA)] = f.ratio;
        }
        #pragma unroll
        for(int g = 0; g < GA + GB; ++g) {
            const double* const v = w + g * W;
            double* const t = table + g * (GROUP_BYTES / 8);
            if(W == 2) {
                t[0 * WARP_SIZE] = 1.0;
                t[1 * WARP_SIZE] = v[0];
                t[2 * WARP_SIZE] = v[1];
                t[3 * WARP_SIZE] = v[0] * v[1];
            } else {
                const double w01 = v[0] * v[1];
                const double w02 = v[0] * v[2];
                const double w12 = v[1] * v[2];
                const double w012 = w01 * v[2];
                t[0 * WARP_SIZE] = 1.0;
                t[1 * WARP_SIZE] = v[0];
                t[2 * WARP_SIZE] = v[1];
                t[3 * WARP_SIZE] = w01;
                t[4 * WARP_SIZE] = v[2];
                t[5 * WARP_SIZE] = w02;
                t[6 * WARP_SIZE] = w12;
                t[7 * WARP_SIZE] = w012;
                t[8 * WARP_SIZE] = v[W - 1];
                t[9 * WARP_SIZE] = v[0] * v[W - 1];
                t[10 * WARP_SIZE] = v[1] * v[W - 1];
                t[11 * WARP_SIZE] = w01 * v[W - 1];
                t[12 * WARP_SIZE] = v[2] * v[W - 1];
                t[13 * WARP_SIZE] = w02 * v[W - 1];
                t[14 * WARP_SIZE] = w12 * v[W - 1];
                t[15 * WARP_SIZE] = w012 * v[W - 1];
            }
        }
        __syncwarp();

        const uint32_t a_lo = o_lo & MASK_A, a_hi = o_hi & MASK_A, a_n = nmask & MASK_A;
        const uint32_t b_lo = (o_lo >> LA) & MASK_B, b_hi = (o_hi >> LA) & MASK_B, b_n = (nmask >> LA) & MASK_B;

        Selection selection;
        selection.best = 0.0; selection.rest = 0.0; selection.index = 0; selection.second = 0;
        CandidateList candidates;       /* what the queue step hands to the tie pass: the separable form its two word masks, the pair loops their block mask */
        candidates.reset();
        #pragma unroll
        for(int c = 0; c < TIE_CANDIDATES; ++c) { candidates.entry[c] = 0u; }
        uint32_t near_blocks = 0u;      /* the pair loops flag runs of grid entries instead (note_block) */
        if constexpr(UNIFORM) {
            /* ---- full grid under one prior: p(a, k) = SA[a] * SB[k] * prior is separable, so the maximum is
               (argmax SA, argmax SB), the runner-up is one of (best A, second B) / (second A, best B), and the
               sum of everything else follows from the two parts' sums. KA + KB word products per read instead
               of KA * KB pair products; the values are the same single roundings the pair loop would form. */
            PartSelection part_b;
            part_b.best = 0.0; part_b.second = 0.0; part_b.rest = 0.0; part_b.index = 0; part_b.near = 0u;
            #pragma unroll 4
            for(int k = 0; k < KB; ++k) {
                const uint2 raw = *reinterpret_cast< const uint2* >(word + k);
                const uint32_t m = mismatch_mask(b_lo, b_hi, b_n, raw.x, raw.y);
                select_part(part_b, part_product< W, GA, GB >(table_base, m), k);
            }
            PartSelection part_a;
            part_a.best = 0.0; part_a.second = 0.0; part_a.rest = 0.0; part_a.index = 0; part_a.near = 0u;
            #pragma unroll 4
            for(int a = 0; a < KA; ++a) {
                const uint2 h = *reinterpret_cast< const uint2* >(header + a);
                const uint32_t m = mismatch_mask(a_lo, a_hi, a_n, h.x, h.y);
                select_part(part_a, part_product< W, 0, GA >(table_base, m), a);
            }
            const double prior = entry[0].prior;
            const double best = part_a.best * part_b.best;
            const double runner_up = fmax(part_a.best * part_b.second, part_a.second * part_b.best);
            /* tie detection on the products before the common prior, like the pair loops */
            selection.second = (__double2hiint(runner_up) + 1 >= __double2hiint(best)) ? 0x7ff00000 : 0;
            selection.index = part_a.index * KB + part_b.index;
            selection.rest = (part_a.best * part_b.rest + part_a.rest * (part_b.best + part_b.rest)) * prior;
            selection.best = best * prior;
            if(selection.second != 0) {
                /* whatever ties with the maximum pairs a word that ties with the best A word and one that ties with the best B word */
                if(KA > 32 || KB > 32) { candidates.count = TIE_CANDIDATES + 1; }
                else {
                    /* the two masks travel as they are (TIE_MASKS): the tie pass walks their cross product */
                    candidates.count = TIE_MASKS;
                    candidates.entry[0] = part_a.near;
                    candidates.entry[1] = part_b.near;
                    candidates.entry[2] = static_cast< uint32_t >(KB);
                }
            }
        } else if constexpr(KBP > 0) {
            /* ---- dense grid: B word probabilities in registers */
            double sb[KBP];
            #pragma unroll
            for(int k = 0; k < KBP; ++k) {
                const uint2 raw = *reinterpret_cast< const uint2* >(word + k);
                const uint32_t m = mismatch_mask(b_lo, b_hi, b_n, raw.x, raw.y);
                sb[k] = part_product< W, GA, GB >(table_base, m);
            }
            for(int a = 0; a < KA; ++a) {
                const uint2 h = *reinterpret_cast< const uint2* >(header + a);
                const uint32_t m = mismatch_mask(a_lo, a_hi, a_n, h.x, h.y);
                const double prefix = part_product< W, 0, GA >(table_base, m);
                const GridEntry* const run = entry + a * KBP;
                #pragma unroll
                for(int k = 0; k < KBP; k += 4) {
                    double p[4];
                    #pragma unroll
                    for(int u = 0; u < 4; ++u) {
                        p[u] = (prefix * sb[k + u]) * run[k + u].prior;
                    }
                    note_block(near_blocks, __double2hiint(selection.best), top_high(p[0], p[1], p[2], p[3]), a * KBP + k, P.tie_block_shift);
                    select_four(selection, p[0], p[1], p[2], p[3], a * KBP + k);
                }
            }
        } else {
            /* ---- SB: the product of every distinct B word, into this lane's column */
            #pragma unroll 2
            for(int k = 0; k < KB; ++k) {
                const uint2 raw = *reinterpret_cast< const uint2* >(word + k);
                const uint32_t m = mismatch_mask(b_lo, b_hi, b_n, raw.x, raw.y);
                suffix[k * WARP_SIZE] = part_product< W, GA, GB >(table_base, m);
            }
            __syncwarp();

            /* ---- barcodes grouped by A word */
            for(int a = 0; a < KA; ++a) {
                const uint4 h = *reinterpret_cast< const uint4* >(header + a);
                const uint32_t m = mismatch_mask(a_lo, a_hi, a_n, h.x, h.y);
                const double prefix = part_product< W, 0, GA >(table_base, m);
                const int last = static_cast< int >(h.z + h.w);
                #pragma unroll 2
                for(int i = static_cast< int >(h.z); i < last; i += 4) {        /* runs are padded to a multiple of four with prior 0 */
                    double p[4];
                    #pragma unroll
                    for(int u = 0; u < 4; ++u) {
                        const uint4 raw = *reinterpret_cast< const uint4* >(entry + i + u);
                        p[u] = (prefix * column_load(suffix_base + raw.x)) * __hiloint2double(raw.w, raw.z);
                    }
                    note_block(near_blocks, __double2hiint(selection.best), top_high(p[0], p[1], p[2], p[3]), i, P.tie_block_shift);
                    select_four(selection, p[0], p[1], p[2], p[3], i);
                }
            }
        }

        /* ---- ties are queued; everything else is decided here */
        const bool tied = valid && (selection.second + 1 >= __double2hiint(selection.best));
        if constexpr(!UNIFORM) { candidates = block_candidates(near_blocks, P.tie_block_shift, true); }
        queue_ties< G, CandidateList >(P, tied, lane, selection, base_probability, high_quality_mask, uniform_positions == L, o_lo, o_hi, nmask, r, quality, candidates);
        const bool decided = valid && !tied;
        if(decided) {
            const int winner = static_cast< int >(entry[selection.index].index);
            const BarcodeEntry e = P.barcodes[winner];
            const uint32_t m = mismatch_mask(o_lo, o_hi, nmask, e.lo, e.hi);
            const double t = part_product< W, 0, GA >(table_base, m & MASK_A) * part_product< W, GA, GB >(table_base, (m >> LA) & MASK_B);
            const Verdict v = pamld_decide(P, S.accumulator, &S.misc[3], winner, m, t, e.prior, selection.rest, base_probability,
                                           uniform_positions == L, high_quality_mask, qcfail);
            qcfail = v.qcfail;
            A.qcfail[r] = static_cast< uint8_t >(v.qcfail);
            store_result(A, r, v.decoded, v.distance, v.confidence, v.qcfail);
        }
        if(P.totals != nullptr) {
            const unsigned live = __ballot_sync(FULL_MASK, decided);
            const unsigned pass = __ballot_sync(FULL_MASK, decided && !qcfail);
            if(lane == 0) {
                atomicAdd(&S.misc[0], static_cast< uint32_t >(__popc(live)));
                atomicAdd(&S.misc[1], static_cast< uint32_t >(__popc(pass)));
            }
        }
        __syncwarp();
    }
    block_epilogue(S, P);
}

/* ------------------------------------------------------------------ PAMLD prefilter scans (f32)
   The exact scans above spend their time on (read, barcode) pairs that cannot matter: for most reads one barcode
   carries all but a vanishing part of sigma_p. The prefilter scans walk the same pairs in f32 — subset tables of
   four positions in f32 ([entry][lane] rows of 128 bytes: ONE shared-memory wavefront per lookup instead of two, half
   the footprint, so more resident warps), FMUL / FMNMX instead of DMUL and two-register selects — and keep, per read,
   the largest product, its barcode and the sum of all the others (blocks of four summed in f32, blocks added in f64).

   A read is EASY when the others sum to at most 2^-20 of the largest product: the maximum is then unique by six orders
   of magnitude (f32 rounding, 2^-22 relative over a product chain, cannot reorder it; ties and near ties are never
   easy), and everything the decision needs from the winner is recomputed exactly in f64 — its mismatch product from
   the f64 ratios, P0 in position order, the prior from the barcode table — so P(r|b) > rbp and the f64 noise term are
   what the exact scan forms. The only f32 quantity left in sigma_p is the sum of the others: a term with c mismatched
   positions carries at most 2c + 1 roundings of 2^-24 and the block sums two more, so the error probability
   1 - confidence of an easy read is within 6e-7 relative of the exact scan's in the worst case (typical: 1e-7) and the
   confidence itself within 6e-7 x 2^-20 < 1e-12. Reads whose confidence lands within 2^-38 of the confidence
   threshold are not easy either. Everything else — about one read in fifteen on the synthetic workloads: noise reads,
   reads with a confidently called mismatch, all-N reads, products too small for f32 — is HARD: its index is appended
   to a list and the exact scan (pamld_kernel / pamld_grid_kernel in index-list mode) followed by the tie pass decides
   it exactly as before. */
constexpr double FAST_EASY_RATIO = 9.5367431640625e-07;             /* 2^-20 */
constexpr float FAST_MINIMUM_BEST = 8.6736173798840355e-19f;        /* 2^-60: below it f32 products of the others may underflow */
constexpr double FAST_THRESHOLD_GUARD = 3.637978807091713e-12;      /* 2^-38 */
constexpr int FAST_BLOCK_SELECTION = 32;                            /* codecs from this size on keep the index per block of four (fast_select_block) */
constexpr int FAST_GROUP_FLOATS = 16 * WARP_SIZE;                   /* one table group: 16 subsets x 32 lanes, 2 KB */
/* warps per CTA (one CTA per SM): what the per-warp tables and the registers allow — 64 registers at 32 warps, which the
   scan under one prior fits up to 8 nt; its prior multiply per pair costs the other form the registers for that */
__host__ __device__ constexpr int fast_warps(int G, bool uniform) {
    return G <= 2 ? (uniform ? 32 : 24) : (G == 3 ? (uniform ? 24 : 20) : (G == 4 ? 20 : 16));       /* 20 nt at 19-20 warps measured 3 % slower than at 16 */
}

/* subset product of table group TABLE_GROUP for the nibble at bits 4 * LOCAL of m: entry e of the lane at
   base + TABLE_GROUP * 2048 + e * 128; the warp's block is 2 KB aligned in the shared window, so (nibble << 7) | base */
template < int TABLE_GROUP, int LOCAL, int SHIFTED >
__device__ __forceinline__ float fast_lookup(uint32_t base, uint32_t m) {
    /* the nibble sits at bit SHIFTED + 4 * LOCAL of m (the scan can hand the mask over already shifted left) and belongs at bit 7 */
    constexpr int left = 7 - SHIFTED - 4 * LOCAL;
    const uint32_t moved = left == 0 ? m : (left > 0 ? (m << (left > 0 ? left : 0)) : (m >> (left < 0 ? -left : 0)));
    uint32_t address;
    asm("lop3.b32 %0, %1, 0x780, %2, 0xEA;" : "=r"(address) : "r"(moved), "r"(base));
    float value;
    asm volatile("ld.shared.f32 %0, [%1 + %2];" : "=f"(value) : "r"(address), "n"(TABLE_GROUP * FAST_GROUP_FLOATS * 4));
    return value;
}
/* product over GROUPS consecutive table groups starting at FIRST; m holds the part's mismatch bits from bit SHIFTED */
template < int FIRST, int GROUPS, int SHIFTED, int k >
struct FastProduct {
    static __device__ __forceinline__ float of(uint32_t base, uint32_t m, float t) {
        return FastProduct< FIRST, GROUPS, SHIFTED, k + 1 >::of(base, m, t * fast_lookup< FIRST + k, k, SHIFTED >(base, m));
    }
};
template < int FIRST, int GROUPS, int SHIFTED >
struct FastProduct< FIRST, GROUPS, SHIFTED, GROUPS > {
    static __device__ __forceinline__ float of(uint32_t, uint32_t, float t) { return t; }
};
template < int FIRST, int GROUPS, int SHIFTED = 0 >
__device__ __forceinline__ float fast_product(uint32_t base, uint32_t m) {
    return FastProduct< FIRST, GROUPS, SHIFTED, 1 >::of(base, m, fast_lookup< FIRST, 0, SHIFTED >(base, m));
}
/*  Shift the planes of FastEntry (and of the observation) travel with. Tried: 7, so that the first lookup needs no shift — but
    the second then needs a RIGHT shift (SHF, ALU pipe) where it had a left shift (IMAD.SHL, FMA pipe), and the ALU pipe
    is what binds this loop (LOP3, FMNMX, FSETP, SEL): no gain, so the planes travel unshifted. */
__host__ __device__ constexpr int fast_preshift(int) { return 0; }
/* the 2^COUNT subset products of COUNT (1..4) positions into the lane's column of one table group */
template < int COUNT >
__device__ __forceinline__ void fast_store_group(float* t, const float* w) {
    const float w0 = w[0];
    const float w1 = COUNT > 1 ? w[COUNT > 1 ? 1 : 0] : 1.0f;
    const float w2 = COUNT > 2 ? w[COUNT > 2 ? 2 : 0] : 1.0f;
    const float w3 = COUNT > 3 ? w[COUNT > 3 ? 3 : 0] : 1.0f;
    const float w01 = w0 * w1;
    t[1 * WARP_SIZE] = w0;                  /* entry 0, the empty subset, is 1 for every read: the kernels store it once */
    if(COUNT > 1) {
        t[2 * WARP_SIZE] = w1;
        t[3 * WARP_SIZE] = w01;
    }
    if(COUNT > 2) {
        const float w02 = w0 * w2, w12 = w1 * w2, w012 = w01 * w2;
        t[4 * WARP_SIZE] = w2;
        t[5 * WARP_SIZE] = w02;
        t[6 * WARP_SIZE] = w12;
        t[7 * WARP_SIZE] = w012;
        if(COUNT > 3) {
            t[8 * WARP_SIZE] = w3;
            t[9 * WARP_SIZE] = w0 * w3;
            t[10 * WARP_SIZE] = w1 * w3;
            t[11 * WARP_SIZE] = w01 * w3;
            t[12 * WARP_SIZE] = w2 * w3;
            t[13 * WARP_SIZE] = w02 * w3;
            t[14 * WARP_SIZE] = w12 * w3;
            t[15 * WARP_SIZE] = w012 * w3;
        }
    }
}
/*  One table group of a read: the f32 mismatch ratios of its COUNT positions (from `first` on) out of the CTA's position
    table — one LDS.128 per position, indexed by the Phred byte and the no-call bit —, their match factors multiplied
    into P0 (f64, position order: the same bits the exact scans form), and the 2^COUNT subset products stored. Group by
    group, so only four ratios are live at a time. */
template < int G, int COUNT >
__device__ __forceinline__ void fast_group(uint32_t position_table, const uint32_t (&quality)[G], uint32_t nmask, int first, double& base_probability, float* t) {
    float w[COUNT];
    #pragma unroll
    for(int k = 0; k < COUNT; ++k) {
        const int j = first + k;
        const uint32_t q = __byte_perm(quality[j >> 2], 0u, 0x4440 + (j & 3));
        const uint32_t ambiguity = (j <= 8) ? (nmask << (j <= 8 ? 8 - j : 0)) : (nmask >> (j <= 8 ? 0 : j - 8));
        uint32_t index;
        asm("lop3.b32 %0, %1, 0x100, %2, 0xEA;" : "=r"(index) : "r"(ambiguity), "r"(q));      /* (ambiguity & 0x100) | q */
        uint32_t factor_lo, factor_hi, ratio, pad;
        asm("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(factor_lo), "=r"(factor_hi), "=r"(ratio), "=r"(pad) : "r"(position_table + index * 16u));
        w[k] = __uint_as_float(ratio);
        base_probability *= __hiloint2double(static_cast< int >(factor_hi), static_cast< int >(factor_lo));
    }
    fast_store_group< COUNT >(t, w);
}
template < int G >
__device__ __forceinline__ void fast_group_of(int count, uint32_t position_table, const uint32_t (&quality)[G], uint32_t nmask, int first, double& base_probability, float* t) {
    if(count >= 4) { fast_group< G, 4 >(position_table, quality, nmask, first, base_probability, t); }
    else if(count == 3) { fast_group< G, 3 >(position_table, quality, nmask, first, base_probability, t); }
    else if(count == 2) { fast_group< G, 2 >(position_table, quality, nmask, first, base_probability, t); }
    else { fast_group< G, 1 >(position_table, quality, nmask, first, base_probability, t); }
}
/* the winner's mismatch product in f64 over the mismatched, unambiguous positions, in position order: a loop over the
   set bits (most winners have none, a few have one or two) */
template < int G, int POSITIONS >
__device__ __forceinline__ double exact_product(const double* __restrict__ ratio64, const uint32_t (&quality)[G], uint32_t counted) {
    double t = 1.0;
    while(counted != 0u) {
        const int j = __ffs(static_cast< int >(counted)) - 1;
        counted &= counted - 1u;
        uint32_t word = quality[0];
        #pragma unroll
        for(int g = 1; g < G; ++g) { if((j >> 2) == g) { word = quality[g]; } }
        const uint32_t q = phred_quality((word >> (8 * (j & 3))) & 0xffu);
        t *= ratio64[q];
    }
    return t;
}
template < int G, int POSITIONS >
__device__ __forceinline__ uint32_t quality_mask(const uint32_t (&quality)[G], int threshold) {
    uint32_t mask = 0;
    #pragma unroll
    for(int j = 0; j < POSITIONS; ++j) {
        if(static_cast< int >((quality[j >> 2] >> (8 * (j & 3))) & 0xffu) >= threshold) { mask |= 1u << j; }
    }
    return mask;
}

/* running selection of a prefilter scan: the maximum, its index, and the f64 sum of everything else */
struct FastSelection {
    float best;
    int index;
    double rest;
};
__device__ __forceinline__ void fast_duel(float a, int ia, float b, int ib, float& high, int& ihigh, float& low) {
    const bool later = b > a;
    high = fmaxf(a, b);
    low = fminf(a, b);
    ihigh = later ? ib : ia;
}
__device__ __forceinline__ void fast_select_one(FastSelection& s, float p, int i) {
    float high, low; int ihigh;
    fast_duel(s.best, s.index, p, i, high, ihigh, low);
    s.best = high; s.index = ihigh;
    s.rest += static_cast< double >(low);
}
__device__ __forceinline__ void fast_select_four(FastSelection& s, float p0, float p1, float p2, float p3, int i) {
    float a, b, c, la, lb, lc, high, low; int ia, ib, ic, ihigh;
    fast_duel(p0, i, p1, i + 1, a, ia, la);
    fast_duel(p2, i + 2, p3, i + 3, b, ib, lb);
    fast_duel(a, ia, b, ib, c, ic, lc);
    fast_duel(s.best, s.index, c, ic, high, ihigh, low);
    s.best = high; s.index = ihigh;
    s.rest += static_cast< double >(((la + lb) + lc) + low);
}

/*  The same selection with the index kept per BLOCK of four: the block's maximum and sum cost three FMNMX and three
    FADD, and only the duel between the block and the running best carries an index (and the sums: the loser's whole
    sum goes to the rest, the leader's is held back). 13 instructions per block instead of 21, 8 of them on the ALU pipe
    instead of 16 — the pipe that binds these loops. The scan recomputes the four products of the leading block once
    per read to name the winner and to add the other three (fast_block_winner). */
struct FastBlockSelection {
    float best;             /* the largest product so far */
    float best_sum;         /* the sum of the block it sits in */
    int index;              /* that block's first barcode */
    double rest;            /* the sum of all other blocks */
};
__device__ __forceinline__ void fast_select_block(FastBlockSelection& s, float block_max, float block_sum, int i) {
    const bool later = block_max > s.best;
    const float loser = later ? s.best_sum : block_sum;
    s.best_sum = later ? block_sum : s.best_sum;
    s.index = later ? i : s.index;
    s.best = fmaxf(s.best, block_max);
    s.rest += static_cast< double >(loser);
}

/*  The hard list of a prefilter scan. Every tile leaves a few reads per warp (about 7 % of them); appending those with
    one global atomic per warp and tile means half a million atomics per launch on ONE address and a round trip to L2
    in every tile. So each warp stages its hard reads in 256 bytes of shared memory and moves them out 32 at a time:
    one atomic and one full 128-byte line per 32 reads. */
struct HardList {
    int* staged;            /* this warp's 64 slots in shared memory */
    unsigned held;          /* slots in use (warp uniform) */
    int* list;
    unsigned* count;
    __device__ __forceinline__ void append(bool flag, long long r, int lane) {
        const unsigned lanes = __ballot_sync(FULL_MASK, flag);
        if(lanes == 0u) { return; }
        if(flag) { staged[held + __popc(lanes & ((1u << lane) - 1u))] = static_cast< int >(r); }
        held += static_cast< unsigned >(__popc(lanes));
        __syncwarp();
        if(held >= 32u) {
            unsigned first = 0;
            if(lane == 0) { first = atomicAdd(count, 32u); }
            first = __shfl_sync(FULL_MASK, first, 0);
            list[first + lane] = staged[lane];
            const int moved = (static_cast< unsigned >(lane) + 32u < held) ? staged[32 + lane] : 0;
            __syncwarp();
            staged[lane] = moved;
            held -= 32u;
            __syncwarp();
        }
    }
    __device__ __forceinline__ void flush(int lane) {
        if(held == 0u) { return; }
        unsigned first = 0;
        if(lane == 0) { first = atomicAdd(count, held); }
        first = __shfl_sync(FULL_MASK, first, 0);
        if(static_cast< unsigned >(lane) < held) { list[first + lane] = staged[lane]; }
        held = 0u;
    }
};

/*  What both prefilter scans do once the winner of an easy read is known: the exact f64 evaluation of the winner, the
    guard around the confidence threshold, then the decision and the stores. Returns false when the read turns out
    hard after all. */
template < int G, int POSITIONS >
__device__ __forceinline__ bool fast_decide(const DecoderParams& P, const TileArguments& A, const BlockState& S, long long r, int winner,
                                            uint32_t o_lo, uint32_t o_hi, uint32_t nmask, const uint32_t (&quality)[G], double others,
                                            double base_probability, uint32_t& qcfail) {
    const BarcodeEntry e = P.barcodes[winner];
    const uint32_t m = mismatch_mask(o_lo, o_hi, nmask, e.lo, e.hi);
    const double t = exact_product< G, POSITIONS >(S.phred + PHRED_MISMATCH_RATIO, quality, m & ~nmask);
    const double p = t * e.prior;
    const double sigma_p = p + (others + P.adjusted_noise_probability / base_probability);
    const double confidence = p / sigma_p;
    if(fabs(confidence - P.confidence_threshold) <= FAST_THRESHOLD_GUARD) { return false; }
    uint32_t high_quality_mask = 0;
    if(P.high_quality_distance_threshold > 0) {
        high_quality_mask = quality_mask< G, POSITIONS >(quality, P.high_quality_threshold);
        high_quality_mask &= (P.nucleotide_cardinality >= 32) ? 0xffffffffu : ((1u << P.nucleotide_cardinality) - 1u);
    }
    const Verdict v = pamld_apply< true >(P, S.accumulator, &S.misc[3], winner, m, base_probability * t, confidence, false, high_quality_mask, qcfail);
    qcfail = v.qcfail;
    A.qcfail[r] = static_cast< uint8_t >(v.qcfail);
    store_result(A, r, v.decoded, v.distance, v.confidence, v.qcfail);
    return true;
}

template < int G, bool UNIFORM >
__global__ void __launch_bounds__(fast_warps(G, UNIFORM) * WARP_SIZE, 1)
pamld_fast_kernel(const DecoderParams P, const TileArguments A) {
    extern __shared__ __align__(256) unsigned char smem[];
    const BlockState S = block_prologue(smem, P, true, 0, true);
    const BarcodeStream stream(S, P, P.fast_barcodes);
    const uint32_t position_table = shared_address(smem + S.plan.off_ratio32);
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const uint32_t window = shared_address(smem);
    const uint32_t aligned_tables = ((window + S.plan.off_tables + 2047u) & ~2047u) - window;
    float* const table = reinterpret_cast< float* >(smem + aligned_tables) + static_cast< size_t >(warp) * (G * FAST_GROUP_FLOATS) + lane;
    const uint32_t table_base = shared_address(table);
    const int L = P.nucleotide_cardinality;
    const uint32_t all_positions = (L >= 32) ? 0xffffffffu : ((1u << L) - 1u);
    HardList hard;
    hard.staged = reinterpret_cast< int* >(smem + S.plan.off_hard) + warp * 64;
    hard.held = 0u;
    hard.list = P.hard_list;
    hard.count = P.tie_count + 2;
    const bool by_block = P.barcode_cardinality >= FAST_BLOCK_SELECTION;
    #pragma unroll
    for(int g = 0; g < G; ++g) { table[g * FAST_GROUP_FLOATS] = 1.0f; }         /* the empty subset of every group */

    const long long tile_cardinality = (A.n_reads + blockDim.x - 1) / blockDim.x;
    const long long my_tiles = tile_cardinality > blockIdx.x ? (tile_cardinality - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const unsigned long long total_iterations = static_cast< unsigned long long >(my_tiles) * stream.chunk_cardinality;
    unsigned iteration = 0;
    if(tid == 0 && total_iterations > 0) { stream.issue(0); }
    const bool resident = stream.chunk_cardinality == 1;
    const BarcodeEntry* resident_stage = nullptr;
    if(resident && total_iterations > 0) { resident_stage = stream.wait(0); }

    uint32_t decided_reads = 0u, passing_reads = 0u;
    ObservedRead< G > upcoming = fetch_read< G >(A, static_cast< long long >(blockIdx.x) * blockDim.x + tid);
    for(long long tile = blockIdx.x; tile < tile_cardinality; tile += gridDim.x) {
        const long long r = tile * blockDim.x + tid;
        const bool valid = r < A.n_reads;
        const ObservedRead< G > observed = upcoming;
        upcoming = fetch_read< G >(A, (tile + gridDim.x) * blockDim.x + tid);
        const uint32_t o_lo = observed.o_lo, o_hi = observed.o_hi, nmask = observed.nmask;
        uint32_t qcfail = observed.qcfail;
        uint32_t quality[G];
        #pragma unroll
        for(int g = 0; g < G; ++g) { quality[g] = decode_quality< G >(A, observed.raw, g); }

        /* ---- f32 ratios, P0, subset tables */
        double base_probability = 1.0;
        #pragma unroll
        for(int g = 0; g < G; ++g) { fast_group< G, 4 >(position_table, quality, nmask, 4 * g, base_probability, table + g * FAST_GROUP_FLOATS); }
        __syncwarp();

        /* ---- every barcode, in f32 (observation and FastEntry planes shifted left by PRE) */
        constexpr int PRE = fast_preshift(G);
        const uint32_t s_lo = o_lo << PRE, s_hi = o_hi << PRE, s_n = nmask << PRE;
        FastSelection selection;
        selection.best = 0.0f; selection.index = 0; selection.rest = 0.0;
        if(by_block) {
            /* codecs of 32 barcodes or more: the index travels per block of four (fast_select_block) */
            FastBlockSelection leader;
            leader.best = 0.0f; leader.best_sum = 0.0f; leader.index = 0; leader.rest = 0.0;
            for(int chunk = 0; chunk < stream.chunk_cardinality; ++chunk) {
                const BarcodeEntry* stage;
                if(resident) {
                    stage = resident_stage;
                } else {
                    if(tid == 0 && iteration + 1 < total_iterations) { stream.issue(iteration + 1); }
                    stage = stream.wait(iteration);
                }
                const int count = stream.count(chunk);
                const int first = chunk * S.plan.stage_capacity;
                int i = 0;
                #pragma unroll 2
                for(; i + 4 <= count; i += 4) {
                    float p[4];
                    #pragma unroll
                    for(int u = 0; u < 4; ++u) {
                        const uint4 raw = *reinterpret_cast< const uint4* >(stage + i + u);
                        const uint32_t m = mismatch_mask(s_lo, s_hi, s_n, raw.x, raw.y);
                        p[u] = fast_product< 0, G, PRE >(table_base, m);
                        if(!UNIFORM) { p[u] *= __uint_as_float(raw.z); }
                    }
                    fast_select_block(leader, fmaxf(fmaxf(p[0], p[1]), fmaxf(p[2], p[3])), (p[0] + p[1]) + (p[2] + p[3]), first + i);
                }
                for(; i < count; ++i) {          /* the last barcodes of a codec that is not a multiple of four: blocks of one */
                    const uint4 raw = *reinterpret_cast< const uint4* >(stage + i);
                    const uint32_t m = mismatch_mask(s_lo, s_hi, s_n, raw.x, raw.y);
                    float p = fast_product< 0, G, PRE >(table_base, m);
                    if(!UNIFORM) { p *= __uint_as_float(raw.z); }
                    fast_select_block(leader, p, p, first + i);
                }
                if(!resident) {
                    __syncthreads();
                    ++iteration;
                }
            }
            /* the leading block once more: which of its four it was, and the other three into the rest */
            selection.index = leader.index;
            selection.rest = leader.rest;
            if(leader.index < (P.barcode_cardinality & ~3)) {
                float p[4];
                #pragma unroll
                for(int u = 0; u < 4; ++u) {
                    const uint4 raw = __ldg(reinterpret_cast< const uint4* >(P.fast_barcodes + leader.index + u));
                    const uint32_t m = mismatch_mask(s_lo, s_hi, s_n, raw.x, raw.y);
                    p[u] = fast_product< 0, G, PRE >(table_base, m);
                    if(!UNIFORM) { p[u] *= __uint_as_float(raw.z); }
                }
                fast_select_four(selection, p[0], p[1], p[2], p[3], leader.index);
            } else {
                selection.best = leader.best;
            }
        } else {
        for(int chunk = 0; chunk < stream.chunk_cardinality; ++chunk) {
            const BarcodeEntry* stage;
            if(resident) {
                stage = resident_stage;
            } else {
                if(tid == 0 && iteration + 1 < total_iterations) { stream.issue(iteration + 1); }
                stage = stream.wait(iteration);
            }
            const int count = stream.count(chunk);
            const int first = chunk * S.plan.stage_capacity;
            int i = 0;
            #pragma unroll 2
            for(; i + 4 <= count; i += 4) {
                float p[4];
                #pragma unroll
                for(int u = 0; u < 4; ++u) {
                    const uint4 raw = *reinterpret_cast< const uint4* >(stage + i + u);
                    const uint32_t m = mismatch_mask(s_lo, s_hi, s_n, raw.x, raw.y);
                    p[u] = fast_product< 0, G, PRE >(table_base, m);
                    if(!UNIFORM) { p[u] *= __uint_as_float(raw.z); }
                }
                fast_select_four(selection, p[0], p[1], p[2], p[3], first + i);
            }
            for(; i < count; ++i) {
                const uint4 raw = *reinterpret_cast< const uint4* >(stage + i);
                const uint32_t m = mismatch_mask(s_lo, s_hi, s_n, raw.x, raw.y);
                float p = fast_product< 0, G, PRE >(table_base, m);
                if(!UNIFORM) { p *= __uint_as_float(raw.z); }
                fast_select_one(selection, p, first + i);
            }
            if(!resident) {
                __syncthreads();
                ++iteration;
            }
        }
        }

        if(UNIFORM) {
            /* one prior for every barcode: it multiplies the maximum and the sum of the others once per read */
            selection.best *= P.fast_uniform_prior;
            selection.rest *= static_cast< double >(P.fast_uniform_prior);
        }
        /* ---- easy reads are decided here, the others are left to the exact scan */
        bool decided = valid && selection.rest <= FAST_EASY_RATIO * static_cast< double >(selection.best)
                    && selection.best >= FAST_MINIMUM_BEST && (nmask & all_positions) != all_positions;
        if(decided) {
            decided = fast_decide< G, 4 * G >(P, A, S, r, selection.index, o_lo, o_hi, nmask, quality, selection.rest, base_probability, qcfail);
        }
        hard.append(valid && !decided, r, lane);
        decided_reads += decided ? 1u : 0u;                 /* the chain's totals: counted per thread, added once per warp below */
        passing_reads += (decided && !qcfail) ? 1u : 0u;
        __syncwarp();
    }
    hard.flush(lane);
    if(P.totals != nullptr) {
        decided_reads = __reduce_add_sync(FULL_MASK, decided_reads);
        passing_reads = __reduce_add_sync(FULL_MASK, passing_reads);
        if(lane == 0) {
            atomicAdd(&S.misc[0], decided_reads);
            atomicAdd(&S.misc[1], passing_reads);
        }
    }
    block_epilogue(S, P);
}

/*  The separable form of the combinatorial scan (full KA x KB grid under one prior; pamld_grid_kernel, UNIFORM) as a
    prefilter: KA + KB word products in f32, then sum of the others = SA* restB + restA (SB* + restB). */
struct FastPart {
    float best;
    int index;
    double rest;
};
__device__ __forceinline__ void fast_select_part(FastPart& s, float value, int i) {
    const bool later = value > s.best;
    const float low = fminf(s.best, value);
    s.best = fmaxf(s.best, value);
    s.index = later ? i : s.index;
    s.rest += static_cast< double >(low);
}
constexpr int FAST_GRID_WARPS = 24;
/* the dense form keeps the B word products in registers: fewer warps, no spills */
__host__ __device__ constexpr int fast_grid_warps(int KBP) { return KBP > 0 ? 20 : FAST_GRID_WARPS; }

template < int LA, int LB, int KBP >
__global__ void __launch_bounds__(fast_grid_warps(KBP) * WARP_SIZE, 1)
pamld_fast_grid_kernel(const DecoderParams P, const TileArguments A) {
    constexpr int L = LA + LB;
    constexpr int G = (L + 3) / 4;
    constexpr int GA = (LA + 3) / 4;            /* table groups of up to four positions per part */
    constexpr int GB = (LB + 3) / 4;
    constexpr uint32_t MASK_A = (1u << LA) - 1u;
    constexpr uint32_t MASK_B = (1u << LB) - 1u;
    extern __shared__ __align__(256) unsigned char smem[];
    const BlockState S = block_prologue(smem, P, true, P.grid_a + P.grid_b + P.grid_entries, true);
    const uint32_t position_table = shared_address(smem + S.plan.off_ratio32);
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int KA = P.grid_a;
    const int KB = P.grid_b;
    const GridHeader* const header = reinterpret_cast< const GridHeader* >(smem + S.plan.off_stage);
    const GridWord* const word = reinterpret_cast< const GridWord* >(header + KA);
    const GridEntry* const entry = reinterpret_cast< const GridEntry* >(word + KB);
    if(tid == 0) {
        const uint32_t bytes = static_cast< uint32_t >(KA + KB + P.grid_entries) * 16u;
        mbarrier_expect_tx(&S.mbarrier[0], bytes);
        tma_bulk_load(smem + S.plan.off_stage, P.grid, bytes, &S.mbarrier[0]);
    }
    mbarrier_wait(&S.mbarrier[0], 0);
    const uint32_t window = shared_address(smem);
    const uint32_t aligned_tables = ((window + S.plan.off_tables + 2047u) & ~2047u) - window;
    float* const table = reinterpret_cast< float* >(smem + aligned_tables) + static_cast< size_t >(warp) * ((GA + GB) * FAST_GROUP_FLOATS) + lane;
    const uint32_t table_base = shared_address(table);
    constexpr uint32_t all_positions = (L >= 32) ? 0xffffffffu : ((1u << L) - 1u);
    HardList hard;
    hard.staged = reinterpret_cast< int* >(smem + S.plan.off_hard) + warp * 64;
    hard.held = 0u;
    hard.list = P.hard_list;
    hard.count = P.tie_count + 2;
    const float prior32 = static_cast< float >(entry[0].prior);
    #pragma unroll
    for(int g = 0; g < GA + GB; ++g) { table[g * FAST_GROUP_FLOATS] = 1.0f; }   /* the empty subset of every group */
    /* dense form: the priors of the grid entries in f32, behind the per-warp tables */
    float* const dense_prior = reinterpret_cast< float* >(smem + aligned_tables + static_cast< size_t >(blockDim.x >> 5) * ((GA + GB) * FAST_GROUP_FLOATS * sizeof(float)));
    if(KBP > 0) {
        for(int i = tid; i < P.grid_entries; i += blockDim.x) { dense_prior[i] = static_cast< float >(entry[i].prior); }
        __syncthreads();
    }

    const long long tile_cardinality = (A.n_reads + blockDim.x - 1) / blockDim.x;
    uint32_t decided_reads = 0u, passing_reads = 0u;
    ObservedRead< G > upcoming = fetch_read< G >(A, static_cast< long long >(blockIdx.x) * blockDim.x + tid);
    for(long long tile = blockIdx.x; tile < tile_cardinality; tile += gridDim.x) {
        const long long r = tile * blockDim.x + tid;
        const bool valid = r < A.n_reads;
        const ObservedRead< G > observed = upcoming;
        upcoming = fetch_read< G >(A, (tile + gridDim.x) * blockDim.x + tid);
        const uint32_t o_lo = observed.o_lo, o_hi = observed.o_hi, nmask = observed.nmask;
        uint32_t qcfail = observed.qcfail;
        uint32_t quality[G];
        #pragma unroll
        for(int g = 0; g < G; ++g) { quality[g] = decode_quality< G >(A, observed.raw, g); }

        double base_probability = 1.0;          /* position order: the A part, then the B part */
        #pragma unroll
        for(int g = 0; g < GA; ++g) { fast_group_of< G >(LA - 4 * g, position_table, quality, nmask, 4 * g, base_probability, table + g * FAST_GROUP_FLOATS); }
        #pragma unroll
        for(int g = 0; g < GB; ++g) { fast_group_of< G >(LB - 4 * g, position_table, quality, nmask, LA + 4 * g, base_probability, table + (GA + g) * FAST_GROUP_FLOATS); }
        __syncwarp();

        const uint32_t a_lo = o_lo & MASK_A, a_hi = o_hi & MASK_A, a_n = nmask & MASK_A;
        const uint32_t b_lo = (o_lo >> LA) & MASK_B, b_hi = (o_hi >> LA) & MASK_B, b_n = (nmask >> LA) & MASK_B;
        float best;
        double others;
        int winner_entry;
        if constexpr(KBP == 0) {
            /* separable: the full grid under one prior */
            FastPart part_b;
            part_b.best = 0.0f; part_b.index = 0; part_b.rest = 0.0;
            #pragma unroll 4
            for(int k = 0; k < KB; ++k) {
                const uint2 raw = *reinterpret_cast< const uint2* >(word + k);
                const uint32_t m = mismatch_mask(b_lo, b_hi, b_n, raw.x, raw.y);
                fast_select_part(part_b, fast_product< GA, GB >(table_base, m), k);
            }
            FastPart part_a;
            part_a.best = 0.0f; part_a.index = 0; part_a.rest = 0.0;
            #pragma unroll 4
            for(int a = 0; a < KA; ++a) {
                const uint2 h = *reinterpret_cast< const uint2* >(header + a);
                const uint32_t m = mismatch_mask(a_lo, a_hi, a_n, h.x, h.y);
                fast_select_part(part_a, fast_product< 0, GA >(table_base, m), a);
            }
            best = (part_a.best * part_b.best) * prior32;
            others = (static_cast< double >(part_a.best) * part_b.rest + part_a.rest * (static_cast< double >(part_b.best) + part_b.rest)) * static_cast< double >(prior32);
            winner_entry = part_a.index * KB + part_b.index;
        } else {
            /* dense: any priors (after prior estimation), holes in the grid as prior 0. The B word products stay in
               registers; a pair costs one FMUL by the A word product, one by its f32 prior and the selection step */
            float sb[KBP];
            #pragma unroll
            for(int k = 0; k < KBP; ++k) {
                const uint2 raw = *reinterpret_cast< const uint2* >(word + k);
                const uint32_t m = mismatch_mask(b_lo, b_hi, b_n, raw.x, raw.y);
                sb[k] = fast_product< GA, GB >(table_base, m);
            }
            /* the index travels per block of four entries (fast_select_block); the leading block is formed once more below */
            FastBlockSelection leader;
            leader.best = 0.0f; leader.best_sum = 0.0f; leader.index = 0; leader.rest = 0.0;
            for(int a = 0; a < KA; ++a) {
                const uint2 h = *reinterpret_cast< const uint2* >(header + a);
                const uint32_t m = mismatch_mask(a_lo, a_hi, a_n, h.x, h.y);
                const float sa = fast_product< 0, GA >(table_base, m);
                #pragma unroll
                for(int k = 0; k < KBP; k += 4) {
                    const float4 prior = *reinterpret_cast< const float4* >(dense_prior + a * KBP + k);
                    const float p0 = (sa * sb[k]) * prior.x, p1 = (sa * sb[k + 1]) * prior.y, p2 = (sa * sb[k + 2]) * prior.z, p3 = (sa * sb[k + 3]) * prior.w;
                    fast_select_block(leader, fmaxf(fmaxf(p0, p1), fmaxf(p2, p3)), (p0 + p1) + (p2 + p3), a * KBP + k);
                }
            }
            FastSelection selection;
            selection.best = 0.0f; selection.index = leader.index; selection.rest = leader.rest;
            {
                const int a = leader.index / KBP, k = leader.index % KBP;
                const uint2 h = *reinterpret_cast< const uint2* >(header + a);
                const float sa = fast_product< 0, GA >(table_base, mismatch_mask(a_lo, a_hi, a_n, h.x, h.y));
                const float4 prior = *reinterpret_cast< const float4* >(dense_prior + leader.index);
                float p[4];
                #pragma unroll
                for(int u = 0; u < 4; ++u) {
                    const uint2 raw = *reinterpret_cast< const uint2* >(word + k + u);
                    p[u] = sa * fast_product< GA, GB >(table_base, mismatch_mask(b_lo, b_hi, b_n, raw.x, raw.y));
                }
                fast_select_four(selection, p[0] * prior.x, p[1] * prior.y, p[2] * prior.z, p[3] * prior.w, leader.index);
            }
            best = selection.best;
            others = selection.rest;
            winner_entry = selection.index;
        }

        bool decided = valid && others <= FAST_EASY_RATIO * static_cast< double >(best) && best >= FAST_MINIMUM_BEST && (nmask & all_positions) != all_positions;
        if(decided) {
            const int winner = static_cast< int >(entry[winner_entry].index);
            decided = fast_decide< G, L >(P, A, S, r, winner, o_lo, o_hi, nmask, quality, others, base_probability, qcfail);
        }
        hard.append(valid && !decided, r, lane);
        decided_reads += decided ? 1u : 0u;                 /* the chain's totals: counted per thread, added once per warp below */
        passing_reads += (decided && !qcfail) ? 1u : 0u;
        __syncwarp();
    }
    hard.flush(lane);
    if(P.totals != nullptr) {
        decided_reads = __reduce_add_sync(FULL_MASK, decided_reads);
        passing_reads = __reduce_add_sync(FULL_MASK, passing_reads);
        if(lane == 0) {
            atomicAdd(&S.misc[0], decided_reads);
            atomicAdd(&S.misc[1], passing_reads);
        }
    }
    block_epilogue(S, P);
}

/* ------------------------------------------------------------------ PAMLD scan for large whitelists
   A cellular whitelist (C5: 737,280 x 16 nt) is three to four orders of magnitude larger than a sample codec,
   and almost every (read, barcode) pair contributes nothing that survives rounding: a barcode with c
   mismatches at confidently called positions has p_b <= prior_max * (product of the c largest mismatch
   ratios of the read). The kernel therefore splits the scan:

     fast path   128 barcodes per step and lane, bit sliced. The table holds, per group of 128 barcodes,
                 position and base, the four words of barcodes that have that base there (equality planes). A
                 lane loads the 16 planes its read selects (one LDS.128 each; 5 distinct addresses per request:
                 conflict free), adds the 16 words of each block with a carry-save adder tree of 26 LOP3 (vertical
                 counters) whose carry-in bits hold the lane's current limit, and the carry out of the tree is the
                 word of barcodes with at most `limit` counted mismatches. 170 instructions per 32 x 128 pairs.
     exact path  the surviving (read, barcode) pairs are pooled over the warp in two steps without divergent
                 loops (non-empty pass words by ballot; 32 words at a time expanded into candidate keys) and
                 evaluated 32 at a time, one per lane, exactly like pamld_kernel does (mismatch mask, subset
                 products, prior); then every read folds its own candidates in, in barcode order (first-maximum
                 selection, tie detection). Pooling makes the cost follow the number of candidates.

   `limit` is the largest count c whose bound can still matter: bound[c] >= min(best / 2,
   tolerance * (noise term + rest) / N). Everything below best / 2 cannot be the maximum or a tie; the N
   barcodes together cannot add more than `tolerance` (2^-21) of the part of sigma_p that is not the winner, so
   confidence and 1 - confidence move by less than 4.8e-7 relative even if every barcode sat exactly at its bound
   (half of the 1e-6 the path allows; the mass actually dropped is one to two orders below that, because only a
   few percent of the barcodes are one mismatch beyond the limit).
   The bound only ever tightens (best and rest grow), so a stale limit is conservative. Positions that do not
   discriminate (N, quality 0, ratios >= 1 i.e. Phred < 3, positions past the barcode) are not counted: they
   select the all-ones plane, and ratios above 1 are folded into the bound.

   Every warp is its own pipeline: it owns 32 reads at a time (taken from a global counter, so slow reads do
   not hold a CTA back), streams the planes through a private three-stage ring of TMA bulk copies (one 1,280 byte
   group per stage, completion on the warp's own mbarriers) and never meets a CTA-wide barrier. Which positions a
   read counts is its own choice (see the per-read set-up): leaving its weakest positions out is always valid and
   often sends fewer barcodes to the exact path. */
constexpr int WHITELIST_STAGES = 3;
constexpr int WHITELIST_QUEUE = 128;            /* candidates a warp can hold back (a power of two); evaluated 32 at a time */
constexpr int WHITELIST_WORDS = 128;            /* non-empty pass words a warp can hold back (a power of two, at least 31 + 2 x 32); expanded up to 32 at a time */
constexpr int WHITELIST_MAX_WARPS = 15;
constexpr double WHITELIST_TOLERANCE = 4.76837158203125e-07;       /* 2^-21: half of the 1e-6 the path allows, as a worst case bound */

/* per-warp shared memory of pamld_whitelist_kernel */
constexpr unsigned WL_OFF_TABLE = 0;                                                    /* 32 entries x 256 B: subset products of 8 groups of 2 positions, lane skewed */
constexpr unsigned WL_OFF_RING = 8192;                                                  /* WHITELIST_STAGES groups of equality planes */
constexpr unsigned WL_OFF_VALUE = WL_OFF_RING + WHITELIST_STAGES * WHITELIST_CHUNK_BYTES;  /* f64 [32]: products of the batch being folded */
constexpr unsigned WL_OFF_KEY = WL_OFF_VALUE + 32 * 8;                                  /* u32 [queue]: owner lane << 27 | barcode index */
constexpr unsigned WL_OFF_WORD = WL_OFF_KEY + WHITELIST_QUEUE * 4;                      /* uint2 [words]: pass word, lane | block << 5 */
constexpr unsigned WL_OFF_OWN = WL_OFF_WORD + WHITELIST_WORDS * 8;                      /* u32 [32]: batch slots that belong to every lane's read */
constexpr unsigned WL_OFF_OBSERVATION = WL_OFF_OWN + 32 * 4;                            /* u32 [3][32]: low plane, high plane, no-call mask of every lane's read */
constexpr unsigned WL_OFF_MBARRIER = WL_OFF_OBSERVATION + 3 * 32 * 4;                   /* u64 [WHITELIST_STAGES] */
constexpr unsigned WL_WARP_BYTES = (WL_OFF_MBARRIER + WHITELIST_STAGES * 8 + 255u) / 256u * 256u;
constexpr unsigned WL_FIXED_BYTES = 256u * 8u + 256u;                                   /* Phred tables, counters */
static_assert(WHITELIST_CHUNK == 128 && WHITELIST_BLOCKS == 4, "the fast path is written out for groups of four blocks");
static_assert(WHITELIST_CHUNK_BYTES % 16 == 0, "TMA bulk copies move multiples of 16 bytes");
static_assert((WHITELIST_QUEUE & (WHITELIST_QUEUE - 1)) == 0 && WHITELIST_QUEUE >= 64, "queue positions are masked");

/*  P(Binomial(H, 3/4) <= l): the chance that a random barcode mismatches a read in at most l of H counted positions;
    [H][l], H and l in 0..16. Only used to choose which positions a read counts (a performance heuristic). */
__constant__ float WHITELIST_PASS_PROBABILITY[17][17] = {
    { 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f },
    { 2.500000e-01f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f },
    { 6.250000e-02f, 4.375000e-01f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f },
    { 1.562500e-02f, 1.562500e-01f, 5.781250e-01f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f },
    { 3.906250e-03f, 5.078125e-02f, 2.617188e-01f, 6.835938e-01f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f },
    { 9.765625e-04f, 1.562500e-02f, 1.035156e-01f, 3.671875e-01f, 7.626953e-01f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f },
    { 2.441406e-04f, 4.638672e-03f, 3.759766e-02f, 1.694336e-01f, 4.660645e-01f, 8.220215e-01f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f },
    { 6.103516e-05f, 1.342773e-03f, 1.287842e-02f, 7.055664e-02f, 2.435913e-01f, 5.550537e-01f, 8.665161e-01f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f },
    { 1.525879e-05f, 3.814697e-04f, 4.226685e-03f, 2.729797e-02f, 1.138153e-01f, 3.214569e-01f, 6.329193e-01f, 8.998871e-01f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f },
    { 3.814697e-06f, 1.068115e-04f, 1.342773e-03f, 9.994507e-03f, 4.892731e-02f, 1.657257e-01f, 3.993225e-01f, 6.996613e-01f, 9.249153e-01f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f },
    { 9.536743e-07f, 2.956390e-05f, 4.158020e-04f, 3.505707e-03f, 1.972771e-02f, 7.812691e-02f, 2.241249e-01f, 4.744072e-01f, 7.559748e-01f, 9.436865e-01f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f },
    { 2.384186e-07f, 8.106232e-06f, 1.261234e-04f, 1.188278e-03f, 7.561207e-03f, 3.432751e-02f, 1.146264e-01f, 2.866955e-01f, 5.447991e-01f, 8.029027e-01f, 9.577649e-01f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f },
    { 5.960464e-08f, 2.205372e-06f, 3.761053e-05f, 3.916621e-04f, 2.781510e-03f, 1.425278e-02f, 5.440223e-02f, 1.576437e-01f, 3.512214e-01f, 6.093250e-01f, 8.416182e-01f, 9.683236e-01f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f },
    { 1.490116e-08f, 5.960464e-07f, 1.105666e-05f, 1.261234e-04f, 9.891242e-04f, 5.649328e-03f, 2.429014e-02f, 8.021259e-02f, 2.060381e-01f, 4.157473e-01f, 6.673983e-01f, 8.732946e-01f, 9.762427e-01f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f },
    { 3.725290e-09f, 1.601875e-07f, 3.211200e-06f, 3.982335e-05f, 3.418736e-04f, 2.154175e-03f, 1.030953e-02f, 3.827076e-02f, 1.116690e-01f, 2.584654e-01f, 4.786600e-01f, 7.188724e-01f, 8.990316e-01f, 9.821821e-01f, 1.000000e+00f, 1.000000e+00f, 1.000000e+00f },
    { 9.313226e-10f, 4.284084e-08f, 9.229407e-07f, 1.236424e-05f, 1.153359e-04f, 7.949490e-04f, 4.193014e-03f, 1.729984e-02f, 5.662031e-02f, 1.483681e-01f, 3.135141e-01f, 5.387131e-01f, 7.639122e-01f, 9.198192e-01f, 9.866365e-01f, 1.000000e+00f, 1.000000e+00f },
    { 2.328306e-10f, 1.140870e-08f, 2.628658e-07f, 3.783265e-06f, 3.810716e-05f, 2.852392e-04f, 1.644465e-03f, 7.469720e-03f, 2.712996e-02f, 7.955725e-02f, 1.896546e-01f, 3.698138e-01f, 5.950129e-01f, 8.028890e-01f, 9.365236e-01f, 9.899774e-01f, 1.000000e+00f },
};

__device__ __forceinline__ void full_add(uint32_t a, uint32_t b, uint32_t c, uint32_t& sum, uint32_t& carry) {
    asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(sum) : "r"(a), "r"(b), "r"(c));        /* a ^ b ^ c */
    asm("lop3.b32 %0, %1, %2, %3, 0xE8;" : "=r"(carry) : "r"(a), "r"(b), "r"(c));      /* majority */
}
__device__ __forceinline__ uint32_t majority(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t carry;
    asm("lop3.b32 %0, %1, %2, %3, 0xE8;" : "=r"(carry) : "r"(a), "r"(b), "r"(c));
    return carry;
}
/*  Bit k of the result is set when (number of the 16 words with bit k set) + bias >= 16, bias = b0 + 2 b1 + 4 b2
    + 8 b3 given as all-zero / all-one words: a carry-save adder tree over vertical counters, 15 adders, 26 LOP3
    (the low sum bit of every weight is never formed). */
__device__ __forceinline__ uint32_t count_reaches_sixteen(const uint32_t (&e)[16], uint32_t b0, uint32_t b1, uint32_t b2, uint32_t b3) {
    uint32_t s0, s1, s2, s3, s4, t0, t1, c0, c1, c2, c3, c4, c5, c6;
    full_add(e[0], e[1], e[2], s0, c0);
    full_add(e[3], e[4], e[5], s1, c1);
    full_add(e[6], e[7], e[8], s2, c2);
    full_add(e[9], e[10], e[11], s3, c3);
    full_add(e[12], e[13], e[14], s4, c4);
    full_add(s0, s1, s2, t0, c5);
    full_add(s3, s4, e[15], t1, c6);
    const uint32_t c7 = majority(t0, t1, b0);
    uint32_t u0, u1, u2, d0, d1, d2;
    full_add(c0, c1, c2, u0, d0);
    full_add(c3, c4, c5, u1, d1);
    full_add(c6, c7, b1, u2, d2);
    const uint32_t d3 = majority(u0, u1, u2);
    uint32_t v0, f0;
    full_add(d0, d1, d2, v0, f0);
    const uint32_t f1 = majority(v0, d3, b2);
    return majority(f0, f1, b3);
}

/*  Product of the mismatch ratios of `owner`'s read over the mismatch set m: eight groups of two positions, entry
    e = 4 * group + subset of owner o at table + e * 256 + ((o + e) & 31) * 8, so that the entries of one read
    spread over the banks (pooled candidates often share a read) and one entry of all reads is conflict free.
    Fixed association (((T0 T1) T2) ...) T7: equal mismatch sets give bit-equal products. */
__device__ __forceinline__ double whitelist_product(uint32_t table, uint32_t owner, uint32_t m) {
    double t = 1.0;
    #pragma unroll
    for(int g = 0; g < 8; ++g) {
        const uint32_t e = 4u * g + ((m >> (2 * g)) & 3u);
        double value;
        asm volatile("ld.shared.f64 %0, [%1];" : "=d"(value) : "r"(table + e * 256u + ((owner + e) & 31u) * 8u));
        t = g == 0 ? value : t * value;
    }
    return t;
}

__global__ void __launch_bounds__(WHITELIST_MAX_WARPS * WARP_SIZE, 1)
pamld_whitelist_kernel(const DecoderParams P, const TileArguments A, unsigned* const work_counter) {
    extern __shared__ __align__(256) unsigned char smem[];
    double* const phred = reinterpret_cast< double* >(smem);
    uint32_t* const misc = reinterpret_cast< uint32_t* >(smem + 256 * 8);
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    unsigned char* const mine = smem + WL_FIXED_BYTES + static_cast< size_t >(warp) * WL_WARP_BYTES;
    double* const value = reinterpret_cast< double* >(mine + WL_OFF_VALUE);
    uint32_t* const queue_key = reinterpret_cast< uint32_t* >(mine + WL_OFF_KEY);
    uint2* const queue_word = reinterpret_cast< uint2* >(mine + WL_OFF_WORD);
    uint32_t* const own = reinterpret_cast< uint32_t* >(mine + WL_OFF_OWN);
    uint32_t* const observation = reinterpret_cast< uint32_t* >(mine + WL_OFF_OBSERVATION);
    uint64_t* const mbarrier = reinterpret_cast< uint64_t* >(mine + WL_OFF_MBARRIER);
    const uint32_t table = shared_address(mine + WL_OFF_TABLE);
    const uint32_t ring = shared_address(mine + WL_OFF_RING);

    for(int i = tid; i < 256; i += blockDim.x) { phred[i] = P.phred[i]; }
    if(tid < 4) { misc[tid] = 0; }
    if(lane == 0) {
        for(int s = 0; s < WHITELIST_STAGES; ++s) { mbarrier_init(&mbarrier[s], 1); }
        fence_mbarrier_init();
    }
    __syncthreads();
    Accumulator accumulator;
    accumulator.shared_u32 = nullptr; accumulator.shared_f64 = nullptr;
    accumulator.global_u64 = P.acc_u64; accumulator.global_f64 = P.acc_f64;

    const double uniform_factor = P.phred[PHRED_UNIFORM_FACTOR];
    const int L = P.nucleotide_cardinality;
    const int group_cardinality = P.whitelist_chunks;
    const double tolerance_per_barcode = WHITELIST_TOLERANCE / static_cast< double >(P.barcode_cardinality);
    const long long unit_cardinality = (A.n_reads + 31) / 32;
    /* the ring: groups are copied and consumed in one running order; the stage and the mbarrier phase of the next
       group to consume and of the next one to copy are carried along */
    unsigned consume_stage = 0, consume_phase = 0, copy_stage = 0;

    while(true) {
        /* ---- the next 32 reads */
        unsigned unit = 0;
        if(lane == 0) { unit = atomicAdd(work_counter, 1u); }
        unit = __shfl_sync(FULL_MASK, unit, 0);
        if(unit >= unit_cardinality) { break; }
        const long long r = static_cast< long long >(unit) * 32 + lane;
        const bool valid = r < A.n_reads;
        /* start the table stream before the per-read work */
        auto issue = [&](int group) {           /* every lane keeps copy_stage; lane 0 starts the copy */
            if(lane == 0) {
                mbarrier_expect_tx(&mbarrier[copy_stage], WHITELIST_CHUNK_BYTES);
                tma_bulk_load(mine + WL_OFF_RING + copy_stage * WHITELIST_CHUNK_BYTES, P.whitelist + static_cast< size_t >(group) * WHITELIST_CHUNK_BYTES, WHITELIST_CHUNK_BYTES, &mbarrier[copy_stage]);
            }
            copy_stage = copy_stage + 1 == WHITELIST_STAGES ? 0u : copy_stage + 1;
        };
        __syncwarp();
        for(int g = 0; g < WHITELIST_STAGES - 1 && g < group_cardinality; ++g) { issue(g); }

        const ObservedRead< 4 > observed = fetch_read< 4 >(A, r);
        const uint32_t o_lo = observed.o_lo, o_hi = observed.o_hi, nmask = observed.nmask;
        uint32_t qcfail = observed.qcfail;
        uint32_t quality[4];
        #pragma unroll
        for(int g = 0; g < 4; ++g) { quality[g] = decode_quality< 4 >(A, observed.raw, g); }
        observation[lane] = o_lo;
        observation[32 + lane] = o_hi;
        observation[64 + lane] = nmask;

        /* ---- per-read constant P0, subset product table, high quality mask; the plane every position selects */
        double base_probability = 1.0;
        uint32_t high_quality_mask = 0;
        int uniform_positions = 0;
        uint32_t plane_address[WHITELIST_POSITIONS];    /* shared address of the lane's plane of position j in stage 0, block 0 */
        double counted_ratio[WHITELIST_POSITIONS];      /* the ratio of a counted position, 2 (above every ratio that counts) otherwise */
        double loose = 1.0;                             /* product of the ratios above 1 */
        #pragma unroll
        for(int g = 0; g < 8; ++g) {
            double w[2];
            #pragma unroll
            for(int k = 0; k < 2; ++k) {
                const int j = g * 2 + k;
                const uint32_t q = (quality[j >> 2] >> (8 * (j & 3))) & 0xffu;
                if(static_cast< int >(q) >= P.high_quality_threshold) { high_quality_mask |= 1u << j; }
                const bool ambiguous = (nmask >> j) & 1u;
                const PositionFactor f = position_factor(phred, uniform_factor, q, ambiguous);
                uniform_positions += f.uniform ? 1 : 0;
                base_probability *= f.factor;
                w[k] = f.ratio;
                const bool counted = valid && !ambiguous && j < L && f.ratio < 1.0;
                counted_ratio[j] = counted ? f.ratio : 2.0;
                if(f.ratio > 1.0) { loose *= f.ratio; }
            }
            const double both = w[0] * w[1];
            #pragma unroll
            for(int e = 0; e < 4; ++e) {
                const uint32_t entry = 4u * g + e;
                const double v = e == 0 ? 1.0 : (e == 1 ? w[0] : (e == 2 ? w[1] : both));
                asm volatile("st.shared.f64 [%0], %1;" :: "r"(table + entry * 256u + ((static_cast< uint32_t >(lane) + entry) & 31u) * 8u), "d"(v) : "memory");
            }
        }
        high_quality_mask &= (L >= 32) ? 0xffffffffu : ((1u << L) - 1u);

        /* ---- which positions to count, and bound[c]: no barcode with c counted mismatches has a prior adjusted
           product above it. The candidate positions (ratio < 1) in descending order of their ratio, by rank (ties by
           position). Leaving the k weakest of them out is always valid (a mismatch there multiplies by less than 1)
           and often better: a Phred 12 position tells the counter little but loosens the bound by a factor 15, so
           the read would pass many more barcodes to the exact path. k is chosen to minimise the chance that a
           random barcode passes once the threshold has settled at its noise floor. The factor 1 + 2^-20 covers the
           rounding of the products on either side. */
        double bound[WHITELIST_POSITIONS + 1];
        int counted_positions = 0;
        const double noise_term = P.adjusted_noise_probability / base_probability;
        {
            double sorted[WHITELIST_POSITIONS];
            int rank_of[WHITELIST_POSITIONS];
            #pragma unroll
            for(int j = 0; j < WHITELIST_POSITIONS; ++j) { sorted[j] = 0.0; }
            int candidates = 0;
            #pragma unroll
            for(int j = 0; j < WHITELIST_POSITIONS; ++j) {
                rank_of[j] = -1;
                if(counted_ratio[j] < 1.0) {
                    int rank = 0;
                    #pragma unroll
                    for(int i = 0; i < WHITELIST_POSITIONS; ++i) {
                        if(counted_ratio[i] < 1.0 && (counted_ratio[i] > counted_ratio[j] || (counted_ratio[i] == counted_ratio[j] && i < j))) { ++rank; }
                    }
                    sorted[rank] = counted_ratio[j];
                    rank_of[j] = rank;
                    ++candidates;
                }
            }
            const double ceiling = P.prior_maximum * loose * (1.0 + 9.5367431640625e-07);
            const double floor_threshold = tolerance_per_barcode * noise_term;
            int skipped = 0;
            float lowest = 2.0f;
            for(int k = 0; k <= candidates; ++k) {
                double running = ceiling;
                int c = 0;
                while(c < candidates - k && running * sorted[k + c] >= floor_threshold) { running *= sorted[k + c]; ++c; }
                const float chance = WHITELIST_PASS_PROBABILITY[candidates - k][c];
                if(chance < lowest) { lowest = chance; skipped = k; }
            }
            counted_positions = candidates - skipped;
            double running = ceiling;
            bound[0] = running;
            for(int c = 1; c <= WHITELIST_POSITIONS; ++c) {
                running *= (skipped + c - 1 < WHITELIST_POSITIONS) ? sorted[skipped + c - 1] : 0.0;     /* 0 beyond the counted positions: such counts do not occur */
                bound[c] = running;
            }
            #pragma unroll
            for(int j = 0; j < WHITELIST_POSITIONS; ++j) {
                const uint32_t code = ((o_lo >> j) & 1u) | (((o_hi >> j) & 1u) << 1);
                plane_address[j] = ring + (static_cast< uint32_t >(j * WHITELIST_PLANES) + (rank_of[j] >= skipped ? code : 4u)) * 16u;
            }
        }
        int limit = counted_positions;
        double limit_bound = bound[limit];
        double threshold = 0.0;                     /* min(best / 2, tolerance share of the rest of sigma_p): only ever grows */
        const uint32_t valid_mask = valid ? 0xffffffffu : 0u;
        uint32_t b0, b1, b2, b3, take_all;
        auto set_limit = [&]() {
            b0 = 0u - (static_cast< uint32_t >(limit) & 1u);
            b1 = 0u - ((static_cast< uint32_t >(limit) >> 1) & 1u);
            b2 = 0u - ((static_cast< uint32_t >(limit) >> 2) & 1u);
            b3 = 0u - ((static_cast< uint32_t >(limit) >> 3) & 1u);
            take_all = 0u - ((static_cast< uint32_t >(limit) >> 4) & 1u);
        };
        set_limit();
        __syncwarp();

        Selection selection;
        selection.best = 0.0; selection.rest = 0.0; selection.index = 0; selection.second = 0;
        LongCandidateList candidates;           /* the barcodes that can tie with the maximum, for the tie pass */
        candidates.reset();
        unsigned head = 0, tail = 0;            /* candidates evaluated / appended so far (warp uniform) */

        /*  Evaluate candidates [head, head + n) of the queue, one per lane (the barcode word and prior come from the
            table in L2: one 16-byte load per lane and batch), then every read's lane folds its own in, in the order
            they were appended (= barcode order); match.any finds the slots that share a read. All loops run a warp
            uniform number of trips with predicated bodies, so the lanes stay converged. */
        auto process = [&](unsigned n) {
            __syncwarp();
            const bool active = static_cast< unsigned >(lane) < n;
            uint32_t owner = 32u + lane;
            if(active) {
                const uint32_t key = queue_key[(head + lane) & (WHITELIST_QUEUE - 1)];
                owner = key >> 27;
                const uint4 raw = *reinterpret_cast< const uint4* >(P.barcodes + (key & 0x7ffffffu));
                const uint32_t m = mismatch_mask(observation[owner], observation[32 + owner], observation[64 + owner], raw.x, raw.y);
                value[lane] = whitelist_product(table, owner, m) * __hiloint2double(raw.w, raw.z);
            }
            own[lane] = 0u;
            __syncwarp();
            const unsigned peers = __match_any_sync(FULL_MASK, owner);
            if(active) { own[owner] = peers; }
            __syncwarp();
            unsigned pending = own[lane];
            const unsigned trips = __reduce_max_sync(FULL_MASK, static_cast< unsigned >(__popc(pending)));
            const bool mine = pending != 0u;
            double half_best = 0.5 * selection.best;
            for(unsigned trip = 0; trip < trips; ++trip) {
                if(pending != 0u) {
                    const int e = __ffs(static_cast< int >(pending)) - 1;
                    pending &= pending - 1u;
                    const double p = value[e];
                    if(p < half_best) {
                        /* below half the maximum: neither the winner nor a tie, it only adds to the rest */
                        selection.rest += p;
                    } else {
                        const int barcode = static_cast< int >(queue_key[(head + e) & (WHITELIST_QUEUE - 1)] & 0x7ffffffu);
                        int running = __double2hiint(selection.best);
                        capture_one(candidates, running, p, barcode);       /* whatever can tie with the maximum is at least half of it */
                        select_one(selection, p, barcode);
                        half_best = 0.5 * selection.best;
                    }
                }
            }
            if(mine) {
                /* the threshold follows the maximum and the rest once per batch: it only grows, so the older one was conservative */
                threshold = fmin(half_best, tolerance_per_barcode * (noise_term + selection.rest));
                while(limit > 0 && limit_bound < threshold) { --limit; limit_bound = bound[limit]; }
            }
            head += n;
            __syncwarp();
        };

        /*  Second level of the compaction. The fast path leaves a 32 x 128 bit matrix per group with a handful of
            bits set; its non-empty words are appended to `queue_word` with one ballot per block (no loop at all),
            and 32 words at a time are expanded here into candidate keys: one word per lane, positions by a prefix
            sum, a warp uniform number of trips (a word rarely holds more than two candidates). Words are queued in
            (block, lane) order and bits expanded in order, so every read's candidates stay in barcode order. */
        unsigned word_head = 0, word_tail = 0;
        auto expand = [&](unsigned n) {         /* expands as many of the next n <= 32 words as the candidate queue has room for (at least one) */
            while(tail - head >= 32u) { process(32u); }
            __syncwarp();
            uint32_t bits = 0u, tag = 0u;
            if(static_cast< unsigned >(lane) < n) {
                const uint2 entry = queue_word[(word_head + lane) & (WHITELIST_WORDS - 1)];
                bits = entry.x; tag = entry.y;
            }
            const int pending = __popc(bits);
            int inclusive = pending;
            #pragma unroll
            for(int step = 1; step < 32; step <<= 1) {
                const int other = __shfl_up_sync(FULL_MASK, inclusive, step);
                if(lane >= step) { inclusive += other; }
            }
            /* fewer than 32 candidates are waiting, so the first word always fits: space >= queue - 31 >= 32 */
            const int space = WHITELIST_QUEUE - static_cast< int >(tail - head);
            const unsigned fitting = __ballot_sync(FULL_MASK, static_cast< unsigned >(lane) < n && inclusive <= space);
            const unsigned words = static_cast< unsigned >(__popc(fitting));      /* inclusive is monotonic: a prefix of the lanes */
            const bool mine_fits = (fitting >> lane) & 1u;
            const int total = __shfl_sync(FULL_MASK, inclusive, static_cast< int >(words) - 1);
            const int offset = inclusive - pending;
            const int trips = __reduce_max_sync(FULL_MASK, mine_fits ? pending : 0);
            for(int j = 0; j < trips; ++j) {
                if(mine_fits && bits != 0u) {
                    const int k = __ffs(static_cast< int >(bits)) - 1;
                    bits &= bits - 1u;
                    queue_key[(tail + offset + j) & (WHITELIST_QUEUE - 1)] = ((tag & 31u) << 27) | ((tag >> 5) * 32u + k);
                }
            }
            tail += static_cast< unsigned >(total);
            word_head += words;
        };

        for(int group = 0; group < group_cardinality; ++group) {
            /* keep the ring full: the stage freed by the previous group receives group + stages - 1 */
            if(group + WHITELIST_STAGES - 1 < group_cardinality) { issue(group + WHITELIST_STAGES - 1); }
            mbarrier_wait(&mbarrier[consume_stage], consume_phase);

            /* ---- fast path: one 16-byte load per position covers the four blocks of the group */
            uint32_t pass[4];
            {
                const uint32_t stage_offset = consume_stage * WHITELIST_CHUNK_BYTES;
                uint32_t e0[WHITELIST_POSITIONS], e1[WHITELIST_POSITIONS], e2[WHITELIST_POSITIONS], e3[WHITELIST_POSITIONS];
                #pragma unroll
                for(int j = 0; j < WHITELIST_POSITIONS; ++j) {
                    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(e0[j]), "=r"(e1[j]), "=r"(e2[j]), "=r"(e3[j]) : "r"(plane_address[j] + stage_offset));
                }
                pass[0] = (count_reaches_sixteen(e0, b0, b1, b2, b3) | take_all) & valid_mask;
                pass[1] = (count_reaches_sixteen(e1, b0, b1, b2, b3) | take_all) & valid_mask;
                pass[2] = (count_reaches_sixteen(e2, b0, b1, b2, b3) | take_all) & valid_mask;
                pass[3] = (count_reaches_sixteen(e3, b0, b1, b2, b3) | take_all) & valid_mask;
            }
            consume_stage = consume_stage + 1 == WHITELIST_STAGES ? 0u : consume_stage + 1;
            consume_phase ^= consume_stage == 0 ? 1u : 0u;

            /* ---- first level of the compaction: the non-empty pass words, one ballot per block */
            const int previous = limit;
            #pragma unroll
            for(int u = 0; u < 4; ++u) {
                const bool some = pass[u] != 0u;
                const unsigned lanes = __ballot_sync(FULL_MASK, some);
                if(lanes != 0u) {
                    if(some) {
                        queue_word[(word_tail + static_cast< unsigned >(__popc(lanes & ((1u << lane) - 1u)))) & (WHITELIST_WORDS - 1)] =
                            make_uint2(pass[u], static_cast< uint32_t >(lane) | (static_cast< uint32_t >(group * 4 + u) << 5));
                    }
                    word_tail += static_cast< unsigned >(__popc(lanes));
                }
                if(u == 1 || u == 3) {          /* the word queue holds 31 + two blocks' worth */
                    #pragma unroll 1
                    while(word_tail - word_head >= 32u) { expand(32u); }
                }
            }
            if(limit != previous) { set_limit(); }
            __syncwarp();       /* the stage is free for the copy the next trip issues */
        }
        /* ---- what is left in the queues */
        {
            const int previous = limit;
            #pragma unroll 1
            while(word_tail != word_head) { expand(word_tail - word_head < 32u ? word_tail - word_head : 32u); }
            #pragma unroll 1
            while(tail != head) { process(tail - head < 32u ? tail - head : 32u); }
            if(limit != previous) { set_limit(); }
        }

        /* ---- structural ties are queued for pamld_tie_kernel, everything else is decided here (as pamld_kernel) */
        const bool tied = valid && (selection.second + 1 >= __double2hiint(selection.best));
        queue_ties< 4, LongCandidateList >(P, tied, lane, selection, base_probability, high_quality_mask, uniform_positions == L, o_lo, o_hi, nmask, r, quality, candidates);
        const bool decided = valid && !tied;
        if(decided) {
            const BarcodeEntry e = P.barcodes[selection.index];
            const uint32_t m = mismatch_mask(o_lo, o_hi, nmask, e.lo, e.hi);
            const double t = whitelist_product(table, static_cast< uint32_t >(lane), m);
            const Verdict v = pamld_decide(P, accumulator, &misc[3], selection.index, m, t, e.prior, selection.rest, base_probability,
                                           uniform_positions == L, high_quality_mask, qcfail);
            qcfail = v.qcfail;
            A.qcfail[r] = static_cast< uint8_t >(v.qcfail);
            store_result(A, r, v.decoded, v.distance, v.confidence, v.qcfail);
        }
        if(P.totals != nullptr) {
            const unsigned live = __ballot_sync(FULL_MASK, decided);
            const unsigned passing = __ballot_sync(FULL_MASK, decided && !qcfail);
            if(lane == 0) {
                atomicAdd(&misc[0], static_cast< uint32_t >(__popc(live)));
                atomicAdd(&misc[1], static_cast< uint32_t >(__popc(passing)));
            }
        }
        __syncwarp();
    }
    __syncthreads();
    if(tid < 2 && P.totals != nullptr && misc[tid]) { atomicAdd(&P.totals[tid], static_cast< unsigned long long >(misc[tid])); }
    if(tid >= 2 && tid < 4 && P.diagnostics != nullptr && misc[tid]) { atomicAdd(&P.diagnostics[tid - 2], static_cast< unsigned long long >(misc[tid])); }
}

/* ------------------------------------------------------------------ PAMLD tie kernel
   Structural ties (equal multisets of mismatch qualities under equal priors) are common for noise reads
   (~2 % of the synthetic workloads). The reference resolves them by the rounding of its position ordered
   Kahan sums (barcode.h:147-162) and then keeps the first maximum (pamld.cpp:73), so the queued reads are
   re-decoded in exactly that operation order: every barcode that can be the winner (within 2^-18 of the scan's
   maximum; the scan names them) has its sigma_q evaluated bit for bit as the reference does; among equal priors the
   smaller sigma wins and equal sigmas keep the lower index, which is what strict > over p = pow(B, sigma) * prior
   yields. pow() is only consulted across different priors or for small sigma (see beats). */
struct Candidate {
    double prior;
    double sigma;
    int index;              /* -1 = none */
};

/*  pow(B, sigma) as the reference's libm forms it. The reference compares p = pow(B, sigma) * prior with strict >, so
    two candidates whose sigma_q differ in the last bits can still have EQUAL p (then the first keeps the read), and
    candidates with different priors are ordered by the rounded products. glibc's pow is correctly rounded except
    within 2^-68 (relative) of a rounding boundary, so the correctly rounded value is computed here: B^sigma =
    2^k exp(r), r = sigma ln B - k ln 2 in double-double arithmetic (ln of the DOUBLE B = pow(10.0, -0.1) the
    reference raises, to 160 bits), exp by its Taylor series to degree 24, rounded once. Only the tie pass calls it,
    and only where the comparison needs it (see beats); B itself is checked against the constant it was derived for. */
struct DoubleDouble { double hi, lo; };
__device__ __forceinline__ DoubleDouble two_sum(double a, double b) {
    DoubleDouble r;
    r.hi = __dadd_rn(a, b);
    const double bb = __dsub_rn(r.hi, a);
    r.lo = __dadd_rn(__dsub_rn(a, __dsub_rn(r.hi, bb)), __dsub_rn(b, bb));
    return r;
}
__device__ __forceinline__ DoubleDouble quick_two_sum(double a, double b) {
    DoubleDouble r;
    r.hi = __dadd_rn(a, b);
    r.lo = __dsub_rn(b, __dsub_rn(r.hi, a));
    return r;
}
__device__ __forceinline__ DoubleDouble two_product(double a, double b) {
    DoubleDouble r;
    r.hi = __dmul_rn(a, b);
    r.lo = __fma_rn(a, b, -r.hi);
    return r;
}
__device__ __forceinline__ DoubleDouble dd_add(DoubleDouble a, DoubleDouble b) {
    DoubleDouble s = two_sum(a.hi, b.hi);
    const DoubleDouble t = two_sum(a.lo, b.lo);
    s.lo = __dadd_rn(s.lo, t.hi);
    s = quick_two_sum(s.hi, s.lo);
    s.lo = __dadd_rn(s.lo, t.lo);
    return quick_two_sum(s.hi, s.lo);
}
__device__ __forceinline__ DoubleDouble dd_multiply(DoubleDouble a, DoubleDouble b) {
    DoubleDouble p = two_product(a.hi, b.hi);
    p.lo = __dadd_rn(p.lo, __dadd_rn(__dmul_rn(a.hi, b.lo), __dmul_rn(a.lo, b.hi)));
    return quick_two_sum(p.hi, p.lo);
}
__constant__ double INVERSE_FACTORIAL[25][2] = {
    { 0x1.0000000000000p+0, 0x0.0p+0 },
    { 0x1.0000000000000p+0, 0x0.0p+0 },
    { 0x1.0000000000000p-1, 0x0.0p+0 },
    { 0x1.5555555555555p-3, 0x1.5555555555555p-57 },
    { 0x1.5555555555555p-5, 0x1.5555555555555p-59 },
    { 0x1.1111111111111p-7, 0x1.1111111111111p-63 },
    { 0x1.6c16c16c16c17p-10, -0x1.f49f49f49f49fp-65 },
    { 0x1.a01a01a01a01ap-13, 0x1.a01a01a01a01ap-73 },
    { 0x1.a01a01a01a01ap-16, 0x1.a01a01a01a01ap-76 },
    { 0x1.71de3a556c734p-19, -0x1.c154f8ddc6c00p-73 },
    { 0x1.27e4fb7789f5cp-22, 0x1.cbbc05b4fa99ap-76 },
    { 0x1.ae64567f544e4p-26, -0x1.c062e06d1f209p-80 },
    { 0x1.1eed8eff8d898p-29, -0x1.2aec959e14c06p-83 },
    { 0x1.6124613a86d09p-33, 0x1.f28e0cc748ebep-87 },
    { 0x1.93974a8c07c9dp-37, 0x1.05d6f8a2efd1fp-92 },
    { 0x1.ae7f3e733b81fp-41, 0x1.1d8656b0ee8cbp-97 },
    { 0x1.ae7f3e733b81fp-45, 0x1.1d8656b0ee8cbp-101 },
    { 0x1.952c77030ad4ap-49, 0x1.ac981465ddc6cp-103 },
    { 0x1.6827863b97d97p-53, 0x1.eec01221a8b0bp-107 },
    { 0x1.2f49b46814157p-57, 0x1.2650f61dbdcb4p-112 },
    { 0x1.e542ba4020225p-62, 0x1.ea72b4afe3c2fp-120 },
    { 0x1.71b8ef6dcf572p-66, -0x1.d043ae40c4647p-120 },
    { 0x1.0ce396db7f853p-70, -0x1.aebcdbd20331cp-124 },
    { 0x1.761b41316381ap-75, -0x1.3423c7d91404fp-130 },
    { 0x1.f2cf01972f578p-80, -0x1.9ada5fcc1ab14p-135 },
};
constexpr double REFERENCE_BASE = 0x1.96b230bcdc434p-1;            /* pow(10.0, -0.1), phred.h:34 */
__device__ __noinline__ double reference_power(double base, double sigma) {
    if(base != REFERENCE_BASE || !(sigma >= 0.0) || sigma > 3000.0) { return pow(base, sigma); }      /* another libm's B, or a subnormal result */
    /* y = sigma ln B */
    DoubleDouble y = two_product(sigma, -0x1.d791c5f888823p-3);
    y.lo = __dadd_rn(y.lo, __dmul_rn(sigma, 0x1.28d13257a2671p-60));
    y = quick_two_sum(y.hi, y.lo);
    /* r = y - k ln 2 */
    const double k = rint(__dmul_rn(y.hi, 0x1.71547652b82fep+0));
    DoubleDouble t = two_product(k, -0x1.62e42fefa39efp-1);
    t.lo = __dadd_rn(t.lo, __dmul_rn(k, -0x1.abc9e3b39803fp-56));
    t = quick_two_sum(t.hi, t.lo);
    DoubleDouble r = dd_add(y, t);
    r.lo = __dadd_rn(r.lo, __dmul_rn(k, -0x1.7b57a079a1934p-111));
    r = quick_two_sum(r.hi, r.lo);
    /* exp(r), |r| <= 0.35: Horner over the Taylor coefficients */
    DoubleDouble e;
    e.hi = INVERSE_FACTORIAL[24][0]; e.lo = INVERSE_FACTORIAL[24][1];
    #pragma unroll 1
    for(int n = 23; n >= 0; --n) {
        DoubleDouble c;
        c.hi = INVERSE_FACTORIAL[n][0]; c.lo = INVERSE_FACTORIAL[n][1];
        e = dd_add(dd_multiply(e, r), c);
    }
    return scalbn(e.hi, static_cast< int >(k));
}
__device__ __forceinline__ bool beats(const Candidate& a, const Candidate& b, double base) {
    if(a.index < 0) { return false; }
    if(b.index < 0) { return true; }
    if(a.prior == b.prior) {
        if(a.sigma == b.sigma) { return a.index < b.index; }
        /* from 32 on, one ulp of sigma (2^-47 or more) moves pow(B, sigma) by 0.23 x 2^-47 = 7 x 2^-52 relative or more;
           pow (under one ulp) and the product with the common prior (half an ulp) move each side by at most
           1.5 x 2^-52: they can neither merge nor reorder the two, the smaller sigma is the larger p */
        if(fmin(a.sigma, b.sigma) >= 32.0) { return a.sigma < b.sigma; }
    }
    const double pa = reference_power(base, a.sigma) * a.prior;
    const double pb = reference_power(base, b.sigma) * b.prior;
    return pa > pb || (pa == pb && a.index < b.index);
}

/*  The tie pass proper. ONE THREAD PER QUEUED READ: the reads of a queue name two to a dozen candidates each, so a
    lane per barcode (a warp per read, later eight lanes per read) leaves most lanes idle while every read still pays
    the warp-wide set-up, a butterfly of comparisons and the decision. A thread instead

      1. loads its 128-byte record and turns every position into the shared-memory address of its score: the CTA holds
         ONE table of 512 doubles indexed by Phred byte | mismatch << 7 | no-call << 8 (phred.cpp:39-72: the true
         positive quality when the base matches, the quality itself when it does not, UNIFORM_BASE_QUALITY for a base
         that is not A / C / G / T, 0 at Phred 0; 4 KB aligned, so the mismatch bit is ORed into the address): a
         candidate's position costs a shift, a LOP3 and an LDS.64 next to the four DADDs of its Kahan step;
      2. walks its candidates — named in the record, in the pool, or the members of the flagged runs — and forms each
         one's sigma_q exactly like Barcode::compensated_decoding_probability (barcode.h:147-162), keeping the one the
         reference's strict > would keep (`beats` is a strict total order, so folding in any order finds the same one);
      3. takes the decision and updates the accumulators.

    A read whose candidates the scan could not bound (TIE_RESCAN: rare) is scanned by its whole warp afterwards, lanes =
    barcodes, and handed back to its thread. */
constexpr int TIE_THREADS = 128;
constexpr int TIE_STAGE_ENTRIES = 1024;
/* CTAs per SM: the per-position addresses of a read stay in registers (4 G of them) */
__host__ __device__ constexpr int tie_resident(int G) { return G <= 4 ? 6 : 4; }
/* rows of the tie kernel's per-CTA accumulator tables (N + 1), 0 when they stay in global memory */
__host__ __device__ constexpr int tie_accumulator_rows(int N) { return N + 1 <= 300 ? N + 1 : 0; }
constexpr int TIE_SCORE_ENTRIES = 512;
__host__ __device__ constexpr size_t tie_shared_bytes(int N) {
    return 4096                                                             /* alignment slack of the score table */
         + TIE_SCORE_ENTRIES * 8 + 128 * 8                                  /* scores, mismatch ratios */
         + (N <= TIE_STAGE_ENTRIES ? static_cast< size_t >(N) * sizeof(BarcodeEntry) : 0)
         + static_cast< size_t >(tie_accumulator_rows(N)) * (ACC_F64_COLUMNS * 8 + ACC_U64_COLUMNS * 4);
}

/* sigma_q of a candidate: the Kahan sum of the per-position scores in position order, bit for bit barcode.h:147-162.
   score_address[j] = table + 8 q_j + 2048 no-call_j; the mismatch bit j of m goes to bit 10 (128 entries of 8 bytes).
   Two candidates at a time: a step is a chain of four dependent DADDs, and a thread with one chain waits on it. */
template < int G >
__device__ __forceinline__ void tie_sigma_pair(const uint32_t (&score_address)[4 * G], uint32_t m0, uint32_t m1, int L, double& sigma0, double& sigma1) {
    double s0 = 0.0, c0 = 0.0, s1 = 0.0, c1 = 0.0;
    #pragma unroll
    for(int j = 0; j < 4 * G; ++j) {
        if(j > 4 * (G - 1) && j >= L) { break; }
        const uint32_t moved0 = j <= 10 ? (m0 << (j <= 10 ? 10 - j : 0)) : (m0 >> (j <= 10 ? 0 : j - 10));
        const uint32_t moved1 = j <= 10 ? (m1 << (j <= 10 ? 10 - j : 0)) : (m1 >> (j <= 10 ? 0 : j - 10));
        uint32_t address0, address1;
        asm("lop3.b32 %0, %1, 0x400, %2, 0xEA;" : "=r"(address0) : "r"(moved0), "r"(score_address[j]));
        asm("lop3.b32 %0, %1, 0x400, %2, 0xEA;" : "=r"(address1) : "r"(moved1), "r"(score_address[j]));
        double value0, value1;
        asm("ld.shared.f64 %0, [%1];" : "=d"(value0) : "r"(address0));
        asm("ld.shared.f64 %0, [%1];" : "=d"(value1) : "r"(address1));
        const double y0 = __dsub_rn(value0, c0);
        const double y1 = __dsub_rn(value1, c1);
        const double t0 = __dadd_rn(s0, y0);
        const double t1 = __dadd_rn(s1, y1);
        c0 = __dsub_rn(__dsub_rn(t0, s0), y0);
        c1 = __dsub_rn(__dsub_rn(t1, s1), y1);
        s0 = t0;
        s1 = t1;
    }
    sigma0 = s0;
    sigma1 = s1;
}
template < int G >
__device__ __forceinline__ double tie_sigma(const uint32_t (&score_address)[4 * G], uint32_t m, int L) {
    double sigma = 0.0, compensation = 0.0;
    #pragma unroll
    for(int j = 0; j < 4 * G; ++j) {
        if(j > 4 * (G - 1) && j >= L) { break; }
        const uint32_t moved = j <= 10 ? (m << (j <= 10 ? 10 - j : 0)) : (m >> (j <= 10 ? 0 : j - 10));
        uint32_t address;
        asm("lop3.b32 %0, %1, 0x400, %2, 0xEA;" : "=r"(address) : "r"(moved), "r"(score_address[j]));
        double value;
        asm("ld.shared.f64 %0, [%1];" : "=d"(value) : "r"(address));
        const double y = __dsub_rn(value, compensation);
        const double t = __dadd_rn(sigma, y);
        compensation = __dsub_rn(__dsub_rn(t, sigma), y);
        sigma = t;
    }
    return sigma;
}
/* the mismatch product of a barcode over the mismatched, unambiguous positions (ascending), from the ratio table */
template < int G >
__device__ __forceinline__ double tie_product(const uint32_t (&score_address)[4 * G], uint32_t ratio_table, uint32_t counted, int L) {
    double t = 1.0;
    #pragma unroll
    for(int j = 0; j < 4 * G; ++j) {
        if(j > 4 * (G - 1) && j >= L) { break; }
        if((counted >> j) & 1u) {
            double value;
            asm("ld.shared.f64 %0, [%1];" : "=d"(value) : "r"(ratio_table + (score_address[j] & 0x3f8u)));
            t *= value;
        }
    }
    return t;
}

template < int G >
__global__ void __launch_bounds__(TIE_THREADS, tie_resident(G))
pamld_tie_kernel(const DecoderParams P, const TileArguments A) {
    extern __shared__ __align__(16) unsigned char tie_smem[];
    __shared__ uint32_t block_counter[4];
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int N = P.barcode_cardinality;
    const unsigned tie_cardinality = *P.tie_count;
    if(blockIdx.x * TIE_THREADS >= tie_cardinality) { return; }

    /* ---- shared memory: score table (4 KB aligned), mismatch ratios, the barcode table when it is small, accumulator rows */
    const uint32_t window = shared_address(tie_smem);
    const uint32_t slack = (4096u - (window & 4095u)) & 4095u;
    double* const score = reinterpret_cast< double* >(tie_smem + slack);
    double* const ratio = score + TIE_SCORE_ENTRIES;
    unsigned char* cursor = reinterpret_cast< unsigned char* >(ratio + 128);
    const uint32_t score_table = window + slack;
    const uint32_t ratio_table = score_table + TIE_SCORE_ENTRIES * 8;
    const double uniform_quality = P.phred[PHRED_UNIFORM_QUALITY];
    const double base = P.phred[PHRED_BASE];
    for(int i = tid; i < TIE_SCORE_ENTRIES; i += blockDim.x) {
        const int q = i & 127;
        score[i] = q == 0 ? 0.0 : ((i >> 8) ? uniform_quality : (((i >> 7) & 1) ? static_cast< double >(q) : P.phred[PHRED_TRUE_POSITIVE_QUALITY + q]));
    }
    for(int i = tid; i < 128; i += blockDim.x) { ratio[i] = P.phred[PHRED_MISMATCH_RATIO + i]; }
    const BarcodeEntry* barcodes = P.barcodes;
    if(N <= TIE_STAGE_ENTRIES) {
        uint4* const stage = reinterpret_cast< uint4* >(cursor);
        for(int i = tid; i < N; i += blockDim.x) { stage[i] = reinterpret_cast< const uint4* >(P.barcodes)[i]; }
        barcodes = reinterpret_cast< const BarcodeEntry* >(cursor);
        cursor += static_cast< size_t >(N) * sizeof(BarcodeEntry);
    }
    if(tid < 4) { block_counter[tid] = 0; }
    /* per-CTA accumulator tables (small codecs): the queued reads of a batch hit a handful of rows — the undetermined
       one above all — and global atomics on one address serialise */
    const int accumulator_rows = tie_accumulator_rows(N);
    Accumulator accumulator;
    accumulator.shared_u32 = nullptr;
    accumulator.shared_f64 = nullptr;
    accumulator.global_u64 = P.acc_u64;
    accumulator.global_f64 = P.acc_f64;
    if(accumulator_rows > 0) {
        accumulator.shared_f64 = reinterpret_cast< double* >(cursor);
        accumulator.shared_u32 = reinterpret_cast< uint32_t* >(accumulator.shared_f64 + accumulator_rows * ACC_F64_COLUMNS);
        for(int i = tid; i < accumulator_rows * ACC_F64_COLUMNS; i += blockDim.x) { accumulator.shared_f64[i] = 0.0; }
        for(int i = tid; i < accumulator_rows * ACC_U64_COLUMNS; i += blockDim.x) { accumulator.shared_u32[i] = 0u; }
    }
    __syncthreads();

    const int L = P.nucleotide_cardinality;
    /* a warp takes the next 32 records of the queue: what a read costs varies with its candidates by an order of magnitude,
       and a fixed split left a quarter of the SM cycles idle at the end */
    for(;;) {
        unsigned first_item = 0;
        if(lane == 0) { first_item = atomicAdd(P.tie_count + 1, 32u); }
        first_item = __shfl_sync(FULL_MASK, first_item, 0);
        if(first_item >= tie_cardinality) { break; }
        const unsigned item = first_item + lane;
        const bool live = item < tie_cardinality;
        /* everything the scan knew about the read travels in the record: one 128-byte line per thread */
        TieRecord record;
        {
            uint4* const words = reinterpret_cast< uint4* >(&record);
            const uint4* const source = reinterpret_cast< const uint4* >(P.tie_record + (live ? item : 0u));
            #pragma unroll
            for(int i = 0; i < 8; ++i) { words[i] = source[i]; }
        }
        const uint32_t o_lo = record.o_lo, o_hi = record.o_hi, nmask = record.nmask;
        uint32_t score_address[4 * G];
        #pragma unroll
        for(int j = 0; j < 4 * G; ++j) {
            const uint32_t q = phred_quality((record.quality[j >> 2] >> (8 * (j & 3))) & 0xffu);
            score_address[j] = score_table + q * 8u + ((nmask >> j) & 1u) * 2048u;
        }

        /* ---- the candidates: a list (in the record or in the pool) or the members of the flagged runs */
        const uint32_t count_word = record.candidate_count;
        const bool rescan = live && count_word == TIE_RESCAN;
        const bool blocks = live && count_word == TIE_BLOCKS;
        const bool masks = live && count_word == TIE_MASKS;        /* the separable scan: words of part A x words of part B */
        const bool pooled = live && !blocks && !masks && !rescan && (count_word & TIE_POOLED) != 0u;
        const uint32_t* const named = pooled ? P.tie_pool + record.candidate[0] : P.tie_record[live ? item : 0u].candidate;
        const bool grid_entries = blocks && record.candidate[2] != 0u;
        const uint32_t scanned = static_cast< uint32_t >(grid_entries ? P.grid_entries : N);      /* what a block mask counts */
        const uint32_t run = 4u << (record.candidate[1] & 31u);
        uint32_t pending_runs = (blocks || masks) ? record.candidate[0] : 0u;    /* flagged runs, or words of part A */
        uint32_t pending_words = 0u;                                               /* words of part B still to pair with the current A word */
        uint32_t next = 0u;
        uint32_t last = (!live || rescan || blocks || masks) ? 0u : (pooled ? (count_word & 0xffffu) : count_word);
        Candidate best;
        best.prior = 0; best.sigma = 0; best.index = -1;
        /* the next candidate of this thread, -1 when it has none left */
        auto pull = [&]() -> int {
            for(;;) {
                if(masks) {
                    if(pending_words == 0u) {
                        if(pending_runs == 0u) { return -1; }
                        next = static_cast< uint32_t >(__ffs(static_cast< int >(pending_runs)) - 1) * record.candidate[2];     /* a x KB */
                        pending_runs &= pending_runs - 1u;
                        pending_words = record.candidate[1];
                        continue;
                    }
                    const uint32_t e = next + static_cast< uint32_t >(__ffs(static_cast< int >(pending_words)) - 1);
                    pending_words &= pending_words - 1u;
                    const int b = static_cast< int >(reinterpret_cast< const uint4* >(P.grid)[P.grid_a + P.grid_b + e].y);
                    if(b < N) { return b; }
                    continue;
                }
                if(next >= last) {
                    if(pending_runs == 0u) { return -1; }
                    const uint32_t bit = static_cast< uint32_t >(__ffs(static_cast< int >(pending_runs)) - 1);
                    pending_runs &= pending_runs - 1u;
                    next = bit * run;
                    last = min(next + run, scanned);
                    continue;
                }
                int b;
                if(blocks) { b = grid_entries ? static_cast< int >(reinterpret_cast< const uint4* >(P.grid)[P.grid_a + P.grid_b + next].y) : static_cast< int >(next); }
                else { b = static_cast< int >(named[next]); }
                ++next;
                if(b < N) { return b; }
            }
        };
        for(;;) {
            const int b0 = pull();
            if(b0 < 0) { break; }
            const int b1 = pull();
            const uint4 raw0 = *reinterpret_cast< const uint4* >(barcodes + b0);
            const uint4 raw1 = *reinterpret_cast< const uint4* >(barcodes + max(b1, 0));
            const uint32_t m0 = ((o_lo ^ raw0.x) | (o_hi ^ raw0.y)) | nmask;
            const uint32_t m1 = ((o_lo ^ raw1.x) | (o_hi ^ raw1.y)) | nmask;
            Candidate first, second;
            tie_sigma_pair< G >(score_address, m0, m1, L, first.sigma, second.sigma);
            first.prior = __hiloint2double(static_cast< int >(raw0.w), static_cast< int >(raw0.z));
            first.index = b0;
            second.prior = __hiloint2double(static_cast< int >(raw1.w), static_cast< int >(raw1.z));
            second.index = b1;                              /* -1 = none: beats() lets it lose */
            if(beats(second, first, base)) { first = second; }
            if(beats(first, best, base)) { best = first; }
        }

        /* ---- reads without a bound on their candidates: the warp scans the whole table for one read at a time; barcodes
           within 2^-18 of the scan's maximum are evaluated, every lane folds its own, a butterfly picks the winner */
        unsigned unbounded = __ballot_sync(FULL_MASK, rescan);
        while(unbounded != 0u) {
            const int owner = __ffs(static_cast< int >(unbounded)) - 1;
            unbounded &= unbounded - 1u;
            const uint32_t r_lo = __shfl_sync(FULL_MASK, o_lo, owner), r_hi = __shfl_sync(FULL_MASK, o_hi, owner), r_n = __shfl_sync(FULL_MASK, nmask, owner);
            uint32_t r_address[4 * G];
            #pragma unroll
            for(int j = 0; j < 4 * G; ++j) { r_address[j] = __shfl_sync(FULL_MASK, score_address[j], owner); }
            const int scan_high = __shfl_sync(FULL_MASK, __double2hiint(record.best), owner);
            const double threshold = __hiloint2double(scan_high, 0) * (1.0 - 3.814697265625e-06);
            Candidate own;
            own.prior = 0; own.sigma = 0; own.index = -1;
            #pragma unroll 1
            for(int b = lane; b < N; b += WARP_SIZE) {
                const uint4 raw = *reinterpret_cast< const uint4* >(barcodes + b);
                const uint32_t m = ((r_lo ^ raw.x) | (r_hi ^ raw.y)) | r_n;
                const double prior = __hiloint2double(static_cast< int >(raw.w), static_cast< int >(raw.z));
                if(tie_product< G >(r_address, ratio_table, m & ~r_n, L) * prior >= threshold) {
                    Candidate other;
                    other.sigma = tie_sigma< G >(r_address, m, L);
                    other.prior = prior;
                    other.index = b;
                    if(beats(other, own, base)) { own = other; }
                }
            }
            #pragma unroll
            for(int offset = WARP_SIZE / 2; offset > 0; offset >>= 1) {
                Candidate other;
                other.prior = __shfl_xor_sync(FULL_MASK, own.prior, offset);
                other.sigma = __shfl_xor_sync(FULL_MASK, own.sigma, offset);
                other.index = __shfl_xor_sync(FULL_MASK, own.index, offset);
                if(beats(other, own, base)) { own = other; }
            }
            if(lane == owner) { best = own; }
        }

        /* ---- the decision (pamld.cpp:87-122) */
        bool passes = false;
        if(live) {
            const int winner = max(best.index, 0);
            const uint4 winner_entry = *reinterpret_cast< const uint4* >(barcodes + winner);
            const uint32_t m = ((o_lo ^ winner_entry.x) | (o_hi ^ winner_entry.y)) | nmask;
            const double t = tie_product< G >(score_address, ratio_table, m & ~nmask, L);
            const long long r = record.read;
            const double prior = __hiloint2double(static_cast< int >(winner_entry.w), static_cast< int >(winner_entry.z));
            /* everything but the winner: the scan's total minus the winner. The winner is within 2^-18 of
               the scan's maximum, so the first difference is exact (Sterbenz) and nothing cancels. */
            const double others = (record.best - t * prior) + record.rest;
            const uint32_t qcfail = A.qcfail[r];
            const Verdict v = pamld_decide(P, accumulator, &block_counter[3], winner, m, t, prior, others, record.base_probability,
                                           record.uniform != 0u, record.high_quality_mask, qcfail);
            A.qcfail[r] = static_cast< uint8_t >(v.qcfail);
            store_result(A, r, v.decoded, v.distance, v.confidence, v.qcfail);
            passes = !v.qcfail;
        }
        const unsigned decided = __ballot_sync(FULL_MASK, live);
        const unsigned passing = __ballot_sync(FULL_MASK, passes);
        if(lane == 0) {
            atomicAdd(&block_counter[0], static_cast< uint32_t >(__popc(decided)));
            if(passing) { atomicAdd(&block_counter[1], static_cast< uint32_t >(__popc(passing))); }
        }
    }
    __syncthreads();
    if(tid < 2 && P.totals != nullptr && block_counter[tid]) { atomicAdd(&P.totals[tid], static_cast< unsigned long long >(block_counter[tid])); }
    if(accumulator_rows > 0) { flush_accumulators(accumulator, accumulator_rows, P); }
    if(tid == 3 && P.diagnostics != nullptr && block_counter[3]) { atomicAdd(&P.diagnostics[DIAG_THRESHOLD_BAND], static_cast< unsigned long long >(block_counter[3])); }
    if(tid == 2 && P.diagnostics != nullptr && blockIdx.x == 0 && tie_cardinality) { atomicAdd(&P.diagnostics[DIAG_EXACT_PATH], static_cast< unsigned long long >(tie_cardinality)); }
}

/*  The tie pass of pamld_long_kernel: pamld_tie_kernel's thread per queued read, with the observation read again from
    the tile through the record's read index (a record has no room for 64 quality bytes) and the candidates taken from
    the flagged runs of barcodes, the only form that scan queues. Position j of the split form is bit j of word 0 for
    j < 4 H and bit j - 4 H of word 1 after it; the Kahan sums run over positions 0 .. L - 1 in order. */
__host__ __device__ constexpr size_t long_tie_shared_bytes(int N) {
    return 4096 + TIE_SCORE_ENTRIES * 8 + 128 * 8
         + (N <= TIE_STAGE_ENTRIES ? static_cast< size_t >(N) * sizeof(LongBarcodeEntry) : 0)
         + static_cast< size_t >(tie_accumulator_rows(N)) * (ACC_F64_COLUMNS * 8 + ACC_U64_COLUMNS * 4);
}
/* bit j of the split form of m moved to bit 10 (the mismatch bit of a score address); j is a constant after unrolling */
template < int H >
__device__ __forceinline__ uint32_t long_moved(uint32_t m0, uint32_t m1, int j) {
    const int at = j < 4 * H ? j : j - 4 * H;
    const uint32_t word = j < 4 * H ? m0 : m1;
    return at <= 10 ? (word << (at <= 10 ? 10 - at : 0)) : (word >> (at <= 10 ? 0 : at - 10));
}
/* sigma_q of two candidates (tie_sigma_pair over the split form) */
template < int H >
__device__ __forceinline__ void long_tie_sigma_pair(const uint32_t (&score_address)[8 * H], uint32_t a0, uint32_t a1, uint32_t b0, uint32_t b1, int L,
                                                    double& sigma0, double& sigma1) {
    double s0 = 0.0, c0 = 0.0, s1 = 0.0, c1 = 0.0;
    #pragma unroll
    for(int j = 0; j < 8 * H; ++j) {
        if(j >= 8 * (H - 1) && j >= L) { break; }
        uint32_t address0, address1;
        asm("lop3.b32 %0, %1, 0x400, %2, 0xEA;" : "=r"(address0) : "r"(long_moved< H >(a0, a1, j)), "r"(score_address[j]));
        asm("lop3.b32 %0, %1, 0x400, %2, 0xEA;" : "=r"(address1) : "r"(long_moved< H >(b0, b1, j)), "r"(score_address[j]));
        double value0, value1;
        asm("ld.shared.f64 %0, [%1];" : "=d"(value0) : "r"(address0));
        asm("ld.shared.f64 %0, [%1];" : "=d"(value1) : "r"(address1));
        const double y0 = __dsub_rn(value0, c0);
        const double y1 = __dsub_rn(value1, c1);
        const double t0 = __dadd_rn(s0, y0);
        const double t1 = __dadd_rn(s1, y1);
        c0 = __dsub_rn(__dsub_rn(t0, s0), y0);
        c1 = __dsub_rn(__dsub_rn(t1, s1), y1);
        s0 = t0;
        s1 = t1;
    }
    sigma0 = s0;
    sigma1 = s1;
}
/* the mismatch product over the counted positions (tie_product over the split form) */
template < int H >
__device__ __forceinline__ double long_tie_product(const uint32_t (&score_address)[8 * H], uint32_t ratio_table, uint32_t counted0, uint32_t counted1, int L) {
    double t = 1.0;
    #pragma unroll
    for(int j = 0; j < 8 * H; ++j) {
        if(j >= 8 * (H - 1) && j >= L) { break; }
        if(((j < 4 * H ? counted0 : counted1) >> (j < 4 * H ? j : j - 4 * H)) & 1u) {
            double value;
            asm("ld.shared.f64 %0, [%1];" : "=d"(value) : "r"(ratio_table + (score_address[j] & 0x3f8u)));
            t *= value;
        }
    }
    return t;
}

template < int H >
__global__ void __launch_bounds__(TIE_THREADS, 2)
pamld_long_tie_kernel(const DecoderParams P, const TileArguments A) {
    extern __shared__ __align__(16) unsigned char tie_smem[];
    __shared__ uint32_t block_counter[4];
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int N = P.barcode_cardinality;
    const unsigned tie_cardinality = *P.tie_count;
    if(blockIdx.x * TIE_THREADS >= tie_cardinality) { return; }

    /* ---- shared memory: score table (4 KB aligned), mismatch ratios, the barcode table when it is small, accumulator rows */
    const uint32_t window = shared_address(tie_smem);
    const uint32_t slack = (4096u - (window & 4095u)) & 4095u;
    double* const score = reinterpret_cast< double* >(tie_smem + slack);
    double* const ratio = score + TIE_SCORE_ENTRIES;
    unsigned char* cursor = reinterpret_cast< unsigned char* >(ratio + 128);
    const uint32_t score_table = window + slack;
    const uint32_t ratio_table = score_table + TIE_SCORE_ENTRIES * 8;
    const double uniform_quality = P.phred[PHRED_UNIFORM_QUALITY];
    const double base = P.phred[PHRED_BASE];
    for(int i = tid; i < TIE_SCORE_ENTRIES; i += blockDim.x) {
        const int q = i & 127;
        score[i] = q == 0 ? 0.0 : ((i >> 8) ? uniform_quality : (((i >> 7) & 1) ? static_cast< double >(q) : P.phred[PHRED_TRUE_POSITIVE_QUALITY + q]));
    }
    for(int i = tid; i < 128; i += blockDim.x) { ratio[i] = P.phred[PHRED_MISMATCH_RATIO + i]; }
    const LongBarcodeEntry* barcodes = P.long_barcodes;
    if(N <= TIE_STAGE_ENTRIES) {
        uint4* const stage = reinterpret_cast< uint4* >(cursor);
        for(int i = tid; i < 2 * N; i += blockDim.x) { stage[i] = reinterpret_cast< const uint4* >(P.long_barcodes)[i]; }
        barcodes = reinterpret_cast< const LongBarcodeEntry* >(cursor);
        cursor += static_cast< size_t >(N) * sizeof(LongBarcodeEntry);
    }
    if(tid < 4) { block_counter[tid] = 0; }
    const int accumulator_rows = tie_accumulator_rows(N);
    Accumulator accumulator;
    accumulator.shared_u32 = nullptr;
    accumulator.shared_f64 = nullptr;
    accumulator.global_u64 = P.acc_u64;
    accumulator.global_f64 = P.acc_f64;
    if(accumulator_rows > 0) {
        accumulator.shared_f64 = reinterpret_cast< double* >(cursor);
        accumulator.shared_u32 = reinterpret_cast< uint32_t* >(accumulator.shared_f64 + accumulator_rows * ACC_F64_COLUMNS);
        for(int i = tid; i < accumulator_rows * ACC_F64_COLUMNS; i += blockDim.x) { accumulator.shared_f64[i] = 0.0; }
        for(int i = tid; i < accumulator_rows * ACC_U64_COLUMNS; i += blockDim.x) { accumulator.shared_u32[i] = 0u; }
    }
    __syncthreads();

    const int L = P.nucleotide_cardinality;
    const int G = (L + 3) >> 2;
    for(;;) {
        unsigned first_item = 0;
        if(lane == 0) { first_item = atomicAdd(P.tie_count + 1, 32u); }
        first_item = __shfl_sync(FULL_MASK, first_item, 0);
        if(first_item >= tie_cardinality) { break; }
        const unsigned item = first_item + lane;
        const bool live = item < tie_cardinality;
        const TieRecord& record = P.tie_record[live ? item : 0u];
        const long long r = live ? static_cast< long long >(record.read) : 0;
        LongObservation o;
        uint32_t score_address[8 * H];
        uint32_t high_quality[2] = { 0u, 0u };
        o.lo[0] = o.lo[1] = o.hi[0] = o.hi[1] = o.nmask[0] = o.nmask[1] = 0u;
        #pragma unroll
        for(int j = 0; j < 8 * H; ++j) { score_address[j] = score_table; }
        if(live) {
            o = fetch_long_observation(A, r, 4 * H);
            #pragma unroll
            for(int g = 0; g < 2 * H; ++g) {
                const uint32_t word = g < G ? quality_word(A, r, g) : 0u;
                #pragma unroll
                for(int k = 0; k < 4; ++k) {
                    const int j = 4 * g + k;
                    const int half = j < 4 * H ? 0 : 1;
                    const int at = j - 4 * H * half;
                    const uint32_t raw = (word >> (8 * k)) & 0xffu;
                    if(j < L && static_cast< int >(raw) >= P.high_quality_threshold) { high_quality[half] |= 1u << at; }
                    score_address[j] = score_table + phred_quality(raw) * 8u + ((o.nmask[half] >> at) & 1u) * 2048u;
                }
            }
        }

        /* ---- the candidates: the members of the flagged runs */
        const uint32_t run = 4u << (record.candidate[1] & 31u);
        uint32_t pending_runs = live ? record.candidate[0] : 0u;
        uint32_t next = 0u, last = 0u;
        Candidate best;
        best.prior = 0; best.sigma = 0; best.index = -1;
        auto pull = [&]() -> int {
            for(;;) {
                if(next >= last) {
                    if(pending_runs == 0u) { return -1; }
                    const uint32_t bit = static_cast< uint32_t >(__ffs(static_cast< int >(pending_runs)) - 1);
                    pending_runs &= pending_runs - 1u;
                    next = bit * run;
                    last = min(next + run, static_cast< uint32_t >(N));
                    continue;
                }
                return static_cast< int >(next++);
            }
        };
        for(;;) {
            const int b0 = pull();
            if(b0 < 0) { break; }
            const int b1 = pull();
            const LongBarcodeEntry e0 = barcodes[b0];
            const LongBarcodeEntry e1 = barcodes[max(b1, 0)];
            const uint32_t m00 = ((o.lo[0] ^ e0.lo0) | (o.hi[0] ^ e0.hi0)) | o.nmask[0];
            const uint32_t m01 = ((o.lo[1] ^ e0.lo1) | (o.hi[1] ^ e0.hi1)) | o.nmask[1];
            const uint32_t m10 = ((o.lo[0] ^ e1.lo0) | (o.hi[0] ^ e1.hi0)) | o.nmask[0];
            const uint32_t m11 = ((o.lo[1] ^ e1.lo1) | (o.hi[1] ^ e1.hi1)) | o.nmask[1];
            Candidate first, second;
            long_tie_sigma_pair< H >(score_address, m00, m01, m10, m11, L, first.sigma, second.sigma);
            first.prior = e0.prior;
            first.index = b0;
            second.prior = e1.prior;
            second.index = b1;                              /* -1 = none: beats() lets it lose */
            if(beats(second, first, base)) { first = second; }
            if(beats(first, best, base)) { best = first; }
        }

        /* ---- the decision (pamld.cpp:87-122) */
        bool passes = false;
        if(live) {
            const int winner = max(best.index, 0);
            const LongBarcodeEntry e = barcodes[winner];
            const uint32_t m0 = ((o.lo[0] ^ e.lo0) | (o.hi[0] ^ e.hi0)) | o.nmask[0];
            const uint32_t m1 = ((o.lo[1] ^ e.lo1) | (o.hi[1] ^ e.hi1)) | o.nmask[1];
            const double t = long_tie_product< H >(score_address, ratio_table, m0 & ~o.nmask[0], m1 & ~o.nmask[1], L);
            /* everything but the winner: the scan's total minus the winner (see pamld_tie_kernel) */
            const double others = (record.best - t * e.prior) + record.rest;
            const Verdict v = pamld_decide_counted(P, accumulator, &block_counter[3], winner, __popc(m0) + __popc(m1),
                                                   __popc(m0 & high_quality[0]) + __popc(m1 & high_quality[1]), t, e.prior, others,
                                                   record.base_probability, record.uniform != 0u, o.qcfail);
            A.qcfail[r] = static_cast< uint8_t >(v.qcfail);
            store_result(A, r, v.decoded, v.distance, v.confidence, v.qcfail);
            passes = !v.qcfail;
        }
        const unsigned decided = __ballot_sync(FULL_MASK, live);
        const unsigned passing = __ballot_sync(FULL_MASK, passes);
        if(lane == 0) {
            atomicAdd(&block_counter[0], static_cast< uint32_t >(__popc(decided)));
            if(passing) { atomicAdd(&block_counter[1], static_cast< uint32_t >(__popc(passing))); }
        }
    }
    __syncthreads();
    if(tid < 2 && P.totals != nullptr && block_counter[tid]) { atomicAdd(&P.totals[tid], static_cast< unsigned long long >(block_counter[tid])); }
    if(accumulator_rows > 0) { flush_accumulators(accumulator, accumulator_rows, P); }
    if(tid == 3 && P.diagnostics != nullptr && block_counter[3]) { atomicAdd(&P.diagnostics[DIAG_THRESHOLD_BAND], static_cast< unsigned long long >(block_counter[3])); }
    if(tid == 2 && P.diagnostics != nullptr && blockIdx.x == 0 && tie_cardinality) { atomicAdd(&P.diagnostics[DIAG_EXACT_PATH], static_cast< unsigned long long >(tie_cardinality)); }
}

/* ------------------------------------------------------------------ MDD */
template < int SEGMENTS >      /* 0 = run-time segment count */
__global__ void __launch_bounds__(MAX_WARPS * WARP_SIZE, 2)
mdd_kernel(const DecoderParams P, const TileArguments A) {
    extern __shared__ __align__(256) unsigned char smem[];
    const BlockState S = block_prologue(smem, P, false);
    const BarcodeStream stream(S, P);
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int L = P.nucleotide_cardinality;
    const int segment_cardinality = SEGMENTS > 0 ? SEGMENTS : P.segment_cardinality;
    const uint32_t all_positions = (L >= 32) ? 0xffffffffu : ((1u << L) - 1u);

    /* either all reads of the launch or, after mdd_table_kernel, the few it queued */
    const long long item_cardinality = A.index_list != nullptr ? static_cast< long long >(*A.index_count) : A.n_reads;
    const long long tile_cardinality = (item_cardinality + blockDim.x - 1) / blockDim.x;
    const long long my_tiles = tile_cardinality > blockIdx.x ? (tile_cardinality - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const unsigned long long total_iterations = static_cast< unsigned long long >(my_tiles) * stream.chunk_cardinality;
    unsigned iteration = 0;
    if(tid == 0 && total_iterations > 0) { stream.issue(0); }
    const bool resident = stream.chunk_cardinality == 1;
    const BarcodeEntry* resident_stage = nullptr;
    if(resident && total_iterations > 0) { resident_stage = stream.wait(0); }

    for(long long tile = blockIdx.x; tile < tile_cardinality; tile += gridDim.x) {
        const long long item = tile * blockDim.x + tid;
        const bool valid = item < item_cardinality;
        const long long r = (valid && A.index_list != nullptr) ? A.index_list[item] : item;
        uint32_t o_lo = 0, o_hi = 0, nmask = 0, present = 0, masked = 0, qcfail = 0;
        if(valid) {
            const uint32_t w0 = load_stream(A.bases + r);
            o_lo = w0 & 0xffffu;
            o_hi = w0 >> 16;
            nmask = load_stream(A.nmask + r);
            if(P.word_cardinality > 1) {
                const uint32_t w1 = load_stream(A.bases + A.pitch + r);
                o_lo |= w1 << 16;
                o_hi |= w1 & 0xffff0000u;
                nmask |= load_stream(A.nmask + A.pitch + r) << 16;
            }
            /* a position the read does not have is packed as ambiguous with both base bits set (a real ambiguous base
               has them clear); the quality byte is a Phred value like any other, 255 included */
            present = ~(nmask & o_lo & o_hi) & all_positions;
            if(P.quality_masking_threshold > 0) {
                for(int g = 0; g < P.quality_word_cardinality; ++g) {
                    const uint32_t qw = quality_word(A, r, g);
                    #pragma unroll
                    for(int k = 0; k < 4; ++k) {
                        if(static_cast< int >((qw >> (8 * k)) & 0xffu) < P.quality_masking_threshold) { masked |= 1u << (g * 4 + k); }
                    }
                }
                masked &= present;
            }
            qcfail = A.qcfail[r];
        }
        const bool complete = present == all_positions;

        /* exact match first (mdd.cpp:44-46), else the first barcode within tolerance in every segment (mdd.cpp:50-80) */
        int exact_index = -1, found_index = -1, found_distance = 0;
        for(int chunk = 0; chunk < stream.chunk_cardinality; ++chunk) {
            const BarcodeEntry* stage;
            if(resident) {
                stage = resident_stage;
            } else {
                if(tid == 0 && iteration + 1 < total_iterations) { stream.issue(iteration + 1); }
                stage = stream.wait(iteration);
            }
            const int count = stream.count(chunk);
            const int first = chunk * S.plan.stage_capacity;
            #pragma unroll 4
            for(int i = 0; i < count; ++i) {
                const uint2 raw = *reinterpret_cast< const uint2* >(stage + i);
                const uint32_t m = ((o_lo ^ raw.x) | (o_hi ^ raw.y)) | nmask;
                const uint32_t error = (m | masked) & present;
                bool within = true;
                #pragma unroll
                for(int s = 0; s < (SEGMENTS > 0 ? SEGMENTS : PHQ_MAX_SEGMENTS); ++s) {
                    if(s < segment_cardinality) {
                        within = within && (__popc(error & P.segment_mask[s]) <= P.distance_tolerance[s]);
                    }
                }
                if(complete && m == 0u && exact_index < 0) { exact_index = first + i; }
                if(within && found_index < 0) { found_index = first + i; found_distance = __popc(error); }
            }
            if(!resident) {
                __syncthreads();
                ++iteration;
            }
        }

        if(valid) {
            int decoded = 0, distance = 0;
            if(exact_index >= 0) { decoded = exact_index + 1; }
            else if(found_index >= 0) { decoded = found_index + 1; distance = found_distance; }
            if(decoded == 0) { qcfail = 1; }
            if(decoded > 0 && distance > 0) {
                S.accumulator.add_pair(decoded, ACC_DISTANCE, ACC_PF_DISTANCE, static_cast< uint32_t >(distance), !qcfail);
            }
            S.accumulator.add_pair(decoded, ACC_COUNT, ACC_PF_COUNT, 1u, !qcfail);
            A.qcfail[r] = static_cast< uint8_t >(qcfail);
            store_result(A, r, decoded, distance, 0.0, qcfail);
        }
        if(P.totals != nullptr) {
            const unsigned live = __ballot_sync(FULL_MASK, valid);
            const unsigned pass = __ballot_sync(FULL_MASK, valid && !qcfail);
            if(lane == 0) {
                atomicAdd(&S.misc[0], static_cast< uint32_t >(__popc(live)));
                atomicAdd(&S.misc[1], static_cast< uint32_t >(__popc(pass)));
            }
        }
    }
    block_epilogue(S, P);
}

/* mdd_kernel for 33-64 nucleotides: the same scan over the split form (LongBarcodeEntry, segment_mask / segment_mask_long) */
template < int SEGMENTS >      /* 0 = run-time segment count */
__global__ void __launch_bounds__(MAX_WARPS * WARP_SIZE, 2)
mdd_long_kernel(const DecoderParams P, const TileArguments A) {
    extern __shared__ __align__(256) unsigned char smem[];
    const BlockState S = block_prologue(smem, P, false, long_stage_blob(P.barcode_cardinality));
    const LongBarcodeStream stream(S, P);
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int L = P.nucleotide_cardinality;
    const int split = P.long_split;
    const int segment_cardinality = SEGMENTS > 0 ? SEGMENTS : P.segment_cardinality;
    const uint32_t all_positions[2] = { split >= 32 ? 0xffffffffu : ((1u << split) - 1u), L - split >= 32 ? 0xffffffffu : ((1u << (L - split)) - 1u) };

    const long long item_cardinality = A.n_reads;
    const long long tile_cardinality = (item_cardinality + blockDim.x - 1) / blockDim.x;
    const long long my_tiles = tile_cardinality > blockIdx.x ? (tile_cardinality - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const unsigned long long total_iterations = static_cast< unsigned long long >(my_tiles) * stream.chunk_cardinality;
    unsigned iteration = 0;
    if(tid == 0 && total_iterations > 0) { stream.issue(0); }
    const bool resident = stream.chunk_cardinality == 1;
    const LongBarcodeEntry* resident_stage = nullptr;
    if(resident && total_iterations > 0) { resident_stage = stream.wait(0); }

    for(long long tile = blockIdx.x; tile < tile_cardinality; tile += gridDim.x) {
        const long long r = tile * blockDim.x + tid;
        const bool valid = r < item_cardinality;
        LongObservation o;
        o.lo[0] = o.lo[1] = o.hi[0] = o.hi[1] = o.nmask[0] = o.nmask[1] = 0u;
        o.qcfail = 0;
        uint32_t present[2] = { 0u, 0u }, masked[2] = { 0u, 0u };
        if(valid) {
            o = fetch_long_observation(A, r, split);
            /* absent positions: ambiguous with both base bits set (mdd_kernel) */
            #pragma unroll
            for(int h = 0; h < 2; ++h) { present[h] = ~(o.nmask[h] & o.lo[h] & o.hi[h]) & all_positions[h]; }
            if(P.quality_masking_threshold > 0) {
                for(int g = 0; g < P.quality_word_cardinality; ++g) {
                    const uint32_t qw = quality_word(A, r, g);
                    #pragma unroll
                    for(int k = 0; k < 4; ++k) {
                        const int j = g * 4 + k;
                        if(static_cast< int >((qw >> (8 * k)) & 0xffu) < P.quality_masking_threshold) {
                            if(j < split) { masked[0] |= 1u << j; } else { masked[1] |= 1u << (j - split); }
                        }
                    }
                }
                masked[0] &= present[0];
                masked[1] &= present[1];
            }
        }
        const bool complete = present[0] == all_positions[0] && present[1] == all_positions[1];
        const uint32_t qcfail_in = o.qcfail;

        int exact_index = -1, found_index = -1, found_distance = 0;
        for(int chunk = 0; chunk < stream.chunk_cardinality; ++chunk) {
            const LongBarcodeEntry* stage;
            if(resident) {
                stage = resident_stage;
            } else {
                if(tid == 0 && iteration + 1 < total_iterations) { stream.issue(iteration + 1); }
                stage = stream.wait(iteration);
            }
            const int count = stream.count(chunk);
            const int first = chunk * stream.capacity;
            #pragma unroll 4
            for(int i = 0; i < count; ++i) {
                const uint4 raw = *reinterpret_cast< const uint4* >(stage + i);
                const uint32_t m0 = ((o.lo[0] ^ raw.x) | (o.hi[0] ^ raw.y)) | o.nmask[0];
                const uint32_t m1 = ((o.lo[1] ^ raw.z) | (o.hi[1] ^ raw.w)) | o.nmask[1];
                const uint32_t error0 = (m0 | masked[0]) & present[0];
                const uint32_t error1 = (m1 | masked[1]) & present[1];
                bool within = true;
                #pragma unroll
                for(int s = 0; s < (SEGMENTS > 0 ? SEGMENTS : PHQ_MAX_SEGMENTS); ++s) {
                    if(s < segment_cardinality) {
                        within = within && (__popc(error0 & P.segment_mask[s]) + __popc(error1 & P.segment_mask_long[s]) <= P.distance_tolerance[s]);
                    }
                }
                if(complete && (m0 | m1) == 0u && exact_index < 0) { exact_index = first + i; }
                if(within && found_index < 0) { found_index = first + i; found_distance = __popc(error0) + __popc(error1); }
            }
            if(!resident) {
                __syncthreads();
                ++iteration;
            }
        }

        uint32_t qcfail = qcfail_in;
        if(valid) {
            int decoded = 0, distance = 0;
            if(exact_index >= 0) { decoded = exact_index + 1; }
            else if(found_index >= 0) { decoded = found_index + 1; distance = found_distance; }
            if(decoded == 0) { qcfail = 1; }
            if(decoded > 0 && distance > 0) {
                S.accumulator.add_pair(decoded, ACC_DISTANCE, ACC_PF_DISTANCE, static_cast< uint32_t >(distance), !qcfail);
            }
            S.accumulator.add_pair(decoded, ACC_COUNT, ACC_PF_COUNT, 1u, !qcfail);
            A.qcfail[r] = static_cast< uint8_t >(qcfail);
            store_result(A, r, decoded, distance, 0.0, qcfail);
        }
        if(P.totals != nullptr) {
            const unsigned live = __ballot_sync(FULL_MASK, valid);
            const unsigned pass = __ballot_sync(FULL_MASK, valid && !qcfail);
            if(lane == 0) {
                atomicAdd(&S.misc[0], static_cast< uint32_t >(__popc(live)));
                atomicAdd(&S.misc[1], static_cast< uint32_t >(__popc(pass)));
            }
        }
    }
    block_epilogue(S, P);
}

/* ------------------------------------------------------------------ MDD by lookup
   See MddSlot in kernels.cuh. Per read: one probe sequence per segment and one for the tuple of words, instead
   of a scan over every barcode. The exact match of mdd.cpp:44-46 (tested before quality masking) is the same
   lookup with distance 0 on the unmasked observation. Reads that miss positions (short tokens: the reference
   counts only the observed length) are queued for mdd_kernel. Only the base and ambiguity planes are read
   unless quality masking is on. */
/*  Open addressing probe. The tables are built at load factor <= 1/4, so the home slot or its neighbour answer
    almost every lookup: both are fetched up front (two independent LDS.128) and the loop only runs for the
    rare longer cluster, which keeps the lanes of a warp converged. STAGED = tables in shared memory. */
template < bool STAGED >
__device__ __forceinline__ uint2 mdd_slot(const MddSlot* __restrict__ table, uint32_t at) {
    if(STAGED) {
        uint2 v;
        asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(shared_address(table) + at * 8u));
        return v;
    }
    return __ldg(reinterpret_cast< const uint2* >(table) + at);
}
/* slot words: x = key_lo, y = key_hi | value << 16 */
template < bool STAGED >
__device__ __forceinline__ bool mdd_probe(const MddSlot* __restrict__ table, uint32_t mask, uint32_t key_lo, uint32_t key_hi, uint32_t& value) {
    uint32_t at = mdd_hash(key_lo, key_hi) & mask;
    const uint2 first = mdd_slot< STAGED >(table, at);
    const uint2 second = mdd_slot< STAGED >(table, (at + 1u) & mask);
    if(first.x == key_lo && (first.y & 0xffffu) == key_hi && (first.y >> 16) != MDD_EMPTY) { value = first.y >> 16; return true; }
    if((first.y >> 16) == MDD_EMPTY) { return false; }
    if(second.x == key_lo && (second.y & 0xffffu) == key_hi && (second.y >> 16) != MDD_EMPTY) { value = second.y >> 16; return true; }
    if((second.y >> 16) == MDD_EMPTY) { return false; }
    #pragma unroll 1
    for(uint32_t step = 2; step <= mask; ++step) {
        const uint2 slot = mdd_slot< STAGED >(table, (at + step) & mask);
        if((slot.y >> 16) == MDD_EMPTY) { return false; }
        if(slot.x == key_lo && (slot.y & 0xffffu) == key_hi) { value = slot.y >> 16; return true; }
    }
    return false;
}

/* one lookup pass over the SEGMENTS segments with the given ambiguity plane: barcode index or -1, total distance */
template < int SEGMENTS, bool STAGED >
__device__ __forceinline__ int mdd_lookup(const DecoderParams& P, const MddSlot* __restrict__ tables, uint32_t o_lo, uint32_t o_hi, uint32_t ambiguity, int& total) {
    uint32_t word[4] = { 0u, 0u, 0u, 0u };
    total = 0;
    #pragma unroll
    for(int s = 0; s < SEGMENTS; ++s) {
        const uint32_t field = (1u << P.segment_length[s]) - 1u;
        const uint32_t n = (ambiguity >> P.segment_offset[s]) & field;
        const uint32_t keep = field & ~n;           /* bases under an ambiguous / masked position do not take part in the key */
        const uint32_t lo = (o_lo >> P.segment_offset[s]) & keep;
        const uint32_t hi = (o_hi >> P.segment_offset[s]) & keep;
        uint32_t value = 0;
        if(!mdd_probe< STAGED >(tables + P.mdd_first[s], static_cast< uint32_t >(P.mdd_mask[s]), lo | (hi << 16), n, value)) { return -1; }
        word[s] = value & 0xfffu;
        total += static_cast< int >(value >> 12);
    }
    uint32_t value = 0;
    if(!mdd_probe< STAGED >(tables + P.mdd_first[SEGMENTS], static_cast< uint32_t >(P.mdd_mask[SEGMENTS]),
                            word[0] | (word[1] << 12) | (word[2] << 24), (word[2] >> 8) | (word[3] << 4), value)) { return -1; }
    return static_cast< int >(value);
}

template < int SEGMENTS, bool MASKING, bool STAGED >
__global__ void __launch_bounds__(256, 4)
mdd_table_kernel(const DecoderParams P, const TileArguments A, int* queue, unsigned* queue_count) {
    constexpr bool staged = STAGED;
    extern __shared__ __align__(256) unsigned char smem[];
    const BlockState S = block_prologue(smem, P, false, staged ? (P.mdd_slots + 1) / 2 : 1);
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const MddSlot* tables = P.mdd_tables;
    if(staged) {
        if(tid == 0) {
            const uint32_t bytes = static_cast< uint32_t >(P.mdd_slots) * 8u;        /* mdd_slots is kept even: 16-byte granules */
            mbarrier_expect_tx(&S.mbarrier[0], bytes);
            tma_bulk_load(smem + S.plan.off_stage, P.mdd_tables, bytes, &S.mbarrier[0]);
        }
        mbarrier_wait(&S.mbarrier[0], 0);
        tables = reinterpret_cast< const MddSlot* >(smem + S.plan.off_stage);
    }
    const bool two_words = P.word_cardinality > 1;

    /* the planes of the next tile are requested before the current tile is worked on */
    struct Planes { uint32_t w0, w1, n0, n1, qcfail; };
    auto fetch = [&](long long r) {
        Planes p;
        p.w0 = 0; p.w1 = 0; p.n0 = 0; p.n1 = 0; p.qcfail = 0;
        if(r < A.n_reads) {
            p.w0 = load_stream(A.bases + r);
            p.n0 = load_stream(A.nmask + r);
            if(two_words) {
                p.w1 = load_stream(A.bases + A.pitch + r);
                p.n1 = load_stream(A.nmask + A.pitch + r);
            }
            p.qcfail = A.qcfail[r];
        }
        return p;
    };
    const long long tile_cardinality = (A.n_reads + blockDim.x - 1) / blockDim.x;
    Planes next = fetch(static_cast< long long >(blockIdx.x) * blockDim.x + tid);
    for(long long tile = blockIdx.x; tile < tile_cardinality; tile += gridDim.x) {
        const long long r = tile * blockDim.x + tid;
        const bool valid = r < A.n_reads;
        const Planes now = next;
        next = fetch((tile + gridDim.x) * blockDim.x + tid);
        const uint32_t o_lo = (now.w0 & 0xffffu) | (now.w1 << 16);
        const uint32_t o_hi = (now.w0 >> 16) | (now.w1 & 0xffff0000u);
        const uint32_t nmask = now.n0 | (now.n1 << 16);
        uint32_t qcfail = now.qcfail;
        /* a position the read does not have is packed as ambiguous with both base bits set */
        const bool partial = valid && (nmask & o_lo & o_hi) != 0u;
        const bool decided = valid && !partial;

        int decoded = 0, distance = 0;
        if(decided) {
            /* the unmasked observation: final when masking is off, and the exact match (mdd.cpp:44-46) otherwise */
            int total;
            int barcode = mdd_lookup< SEGMENTS, STAGED >(P, tables, o_lo, o_hi, nmask, total);
            if(MASKING && !(barcode >= 0 && total == 0)) {
                /* quality masking (sequence.h:321-332): positions below the threshold always count as errors */
                uint32_t masked = 0;
                for(int g = 0; g < P.quality_word_cardinality; ++g) {
                    const uint32_t qw = quality_word(A, r, g);
                    #pragma unroll
                    for(int k = 0; k < 4; ++k) {
                        if(static_cast< int >((qw >> (8 * k)) & 0xffu) < P.quality_masking_threshold) { masked |= 1u << (g * 4 + k); }
                    }
                }
                masked &= (P.nucleotide_cardinality >= 32) ? 0xffffffffu : ((1u << P.nucleotide_cardinality) - 1u);
                barcode = mdd_lookup< SEGMENTS, STAGED >(P, tables, o_lo, o_hi, nmask | masked, total);
            }
            if(barcode >= 0) { decoded = barcode + 1; distance = total; }
        }

        const unsigned queued = __ballot_sync(FULL_MASK, partial);
        if(queued) {
            unsigned slot = 0;
            if(lane == 0) { slot = atomicAdd(queue_count, static_cast< unsigned >(__popc(queued))); }
            slot = __shfl_sync(FULL_MASK, slot, 0);
            if(partial) { queue[slot + __popc(queued & ((1u << lane) - 1u))] = static_cast< int >(r); }
        }
        if(decided) {
            if(decoded == 0) { qcfail = 1; }
            if(distance > 0) {
                S.accumulator.add_pair(decoded, ACC_DISTANCE, ACC_PF_DISTANCE, static_cast< uint32_t >(distance), !qcfail);
            }
            S.accumulator.add_pair(decoded, ACC_COUNT, ACC_PF_COUNT, 1u, !qcfail);
            A.qcfail[r] = static_cast< uint8_t >(qcfail);
            store_result(A, r, decoded, distance, 0.0, qcfail);
        }
        if(P.totals != nullptr) {
            const unsigned live = __ballot_sync(FULL_MASK, decided);
            const unsigned pass = __ballot_sync(FULL_MASK, decided && !qcfail);
            if(lane == 0) {
                atomicAdd(&S.misc[0], static_cast< uint32_t >(__popc(live)));
                atomicAdd(&S.misc[1], static_cast< uint32_t >(__popc(pass)));
            }
        }
    }
    block_epilogue(S, P);
}

/* ------------------------------------------------------------------ naive / passthrough bookkeeping */
__global__ void __launch_bounds__(256)
count_kernel(const DecoderParams P, const TileArguments A) {
    __shared__ unsigned long long block_count[2];
    if(threadIdx.x < 2) { block_count[threadIdx.x] = 0; }
    __syncthreads();
    unsigned long long live = 0, pass = 0;
    for(long long r = static_cast< long long >(blockIdx.x) * blockDim.x + threadIdx.x; r < A.n_reads; r += static_cast< long long >(gridDim.x) * blockDim.x) {
        ++live;
        if(!A.qcfail[r]) { ++pass; }
        store_result(A, r, 0, 0, 0.0, A.qcfail[r]);
    }
    #pragma unroll
    for(int offset = 16; offset > 0; offset >>= 1) {
        live += __shfl_xor_sync(FULL_MASK, live, offset);
        pass += __shfl_xor_sync(FULL_MASK, pass, offset);
    }
    if((threadIdx.x & 31) == 0) {
        atomicAdd(&block_count[0], live);
        atomicAdd(&block_count[1], pass);
    }
    __syncthreads();
    if(threadIdx.x == 0) {
        if(P.acc_u64 != nullptr) {
            if(block_count[0]) { atomicAdd(&P.acc_u64[ACC_COUNT], block_count[0]); }
            if(block_count[1]) { atomicAdd(&P.acc_u64[ACC_PF_COUNT], block_count[1]); }
        }
        if(P.totals != nullptr) {
            if(block_count[0]) { atomicAdd(&P.totals[0], block_count[0]); }
            if(block_count[1]) { atomicAdd(&P.totals[1], block_count[1]); }
        }
    }
}

/* pow(B, sigma) as the tie pass forms it, for the parity tests (phq_reference_power) */
__global__ void reference_power_kernel(const double* __restrict__ sigma, double* __restrict__ out, long long n, double base) {
    for(long long i = static_cast< long long >(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast< long long >(gridDim.x) * blockDim.x) {
        out[i] = reference_power(base, sigma[i]);
    }
}

/* the tie pass over the reads the scan queued; the queue length is only known on the device: a fixed grid strides over it */
template < int G >
cudaError_t launch_tie(const DecoderParams& params, const TileArguments& tile, const LaunchGeometry& geometry, cudaStream_t stream) {
    const size_t tie_bytes = tie_shared_bytes(params.barcode_cardinality);
    const cudaError_t status = cudaFuncSetAttribute(pamld_tie_kernel< G >, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast< int >(tie_bytes));
    if(status != cudaSuccess) { return status; }
    /* as many CTAs as stay resident: every CTA stages the tables and flushes its accumulator rows once,
       and the flushes of all CTAs meet on the same few hundred global addresses */
    if(params.whitelist != nullptr) {
        /* header word [1], the tie pass' work counter, was the whitelist scan's own: the other scans clear it with the queue length */
        const cudaError_t cleared = cudaMemsetAsync(params.tie_count + 1, 0, sizeof(unsigned), stream);
        if(cleared != cudaSuccess) { return cleared; }
    }
    pamld_tie_kernel< G ><<< geometry.multiprocessor_count * tie_resident(G), TIE_THREADS, tie_bytes, stream >>>(params, tile);
    return cudaGetLastError();
}

template < int G >
cudaError_t launch_pamld_groups(const DecoderParams& params, const TileArguments& tile, const LaunchGeometry& geometry, cudaStream_t stream) {
    const SharedPlan plan = make_plan(params.barcode_cardinality, true);
    const size_t per_warp = static_cast< size_t >(G) * 16 * WARP_SIZE * sizeof(double);
    if(plan.fixed_bytes + per_warp > geometry.shared_memory_per_block_optin) { return cudaErrorInvalidConfiguration; }
    int warps = static_cast< int >((geometry.shared_memory_per_block_optin - plan.fixed_bytes) / per_warp);
    warps = warps > pamld_warps(G) ? pamld_warps(G) : warps;
    const size_t bytes = plan.fixed_bytes + per_warp * warps;
    cudaError_t status = cudaFuncSetAttribute(pamld_kernel< G >, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast< int >(bytes));
    if(status != cudaSuccess) { return status; }
    const int threads = warps * WARP_SIZE;
    const long long tiles = (tile.n_reads + threads - 1) / threads;
    const int grid = static_cast< int >(tiles < geometry.multiprocessor_count ? tiles : geometry.multiprocessor_count);
    status = cudaMemsetAsync(params.tie_count, 0, 2 * sizeof(unsigned), stream);      /* the tie queue's length and the tie pass' work counter */
    if(status != cudaSuccess) { return status; }
    pamld_kernel< G ><<< grid, threads, bytes, stream >>>(params, tile);
    status = cudaGetLastError();
    if(status != cudaSuccess) { return status; }
    return launch_tie< G >(params, tile, geometry, stream);
}

/* the combinatorial scan: staging area = the grid blob instead of the barcode table */
template < int LA, int LB, int KBP, bool UNIFORM >
cudaError_t launch_pamld_grid_as(const DecoderParams& params, const TileArguments& tile, const LaunchGeometry& geometry, cudaStream_t stream) {
    constexpr int W = GRID_GROUP_WIDTH;
    constexpr int G = (LA + LB + 3) / 4;
    constexpr int GA = (LA + W - 1) / W;
    constexpr int GB = (LB + W - 1) / W;
    const int blob_entries = params.grid_a + params.grid_b + params.grid_entries;
    const SharedPlan plan = make_plan(params.barcode_cardinality, true, blob_entries);
    const size_t fixed = plan.fixed_bytes;
    const size_t per_warp = static_cast< size_t >(GA + GB) * (256 << W) + (KBP > 0 ? 0 : static_cast< size_t >(params.grid_b) * 256);
    if(fixed + per_warp > geometry.shared_memory_per_block_optin) { return cudaErrorInvalidConfiguration; }
    int warps = static_cast< int >((geometry.shared_memory_per_block_optin - fixed) / per_warp);
    warps = warps > GRID_MAX_WARPS ? GRID_MAX_WARPS : warps;
    const size_t bytes = fixed + per_warp * warps;
    cudaError_t status = cudaFuncSetAttribute(pamld_grid_kernel< LA, LB, W, KBP, UNIFORM >, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast< int >(bytes));
    if(status != cudaSuccess) { return status; }
    const int threads = warps * WARP_SIZE;
    const long long tiles = (tile.n_reads + threads - 1) / threads;
    const int grid = static_cast< int >(tiles < geometry.multiprocessor_count ? tiles : geometry.multiprocessor_count);
    status = cudaMemsetAsync(params.tie_count, 0, 2 * sizeof(unsigned), stream);      /* the tie queue's length and the tie pass' work counter */
    if(status != cudaSuccess) { return status; }
    pamld_grid_kernel< LA, LB, W, KBP, UNIFORM ><<< grid, threads, bytes, stream >>>(params, tile);
    status = cudaGetLastError();
    if(status != cudaSuccess) { return status; }
    return launch_tie< G >(params, tile, geometry, stream);
}
template < int LA, int LB, bool DENSE >
cudaError_t launch_pamld_grid(const DecoderParams& params, const TileArguments& tile, const LaunchGeometry& geometry, cudaStream_t stream) {
    if(params.grid_uniform) { return launch_pamld_grid_as< LA, LB, 1, true >(params, tile, geometry, stream); }
    if(DENSE && params.grid_dense == 8) { return launch_pamld_grid_as< LA, LB, 8, false >(params, tile, geometry, stream); }
    if(DENSE && params.grid_dense == 16) { return launch_pamld_grid_as< LA, LB, 16, false >(params, tile, geometry, stream); }
    return launch_pamld_grid_as< LA, LB, 0, false >(params, tile, geometry, stream);
}

/* the prefilter scan over every read of the launch, then the exact scan over the reads it left, then the tie pass */
template < int G, bool UNIFORM >
cudaError_t launch_pamld_fast_groups_as(const DecoderParams& params, const TileArguments& tile, const LaunchGeometry& geometry, cudaStream_t stream) {
    const SharedPlan plan = make_plan(params.barcode_cardinality, true, 0, true);
    const size_t per_warp = static_cast< size_t >(G) * FAST_GROUP_FLOATS * sizeof(float);
    if(plan.fixed_bytes + per_warp > geometry.shared_memory_per_block_optin) { return cudaErrorInvalidConfiguration; }
    int warps = static_cast< int >((geometry.shared_memory_per_block_optin - plan.fixed_bytes) / per_warp);
    warps = warps > fast_warps(G, UNIFORM) ? fast_warps(G, UNIFORM) : warps;
    const size_t bytes = plan.fixed_bytes + per_warp * warps;
    cudaError_t status = cudaFuncSetAttribute(pamld_fast_kernel< G, UNIFORM >, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast< int >(bytes));
    if(status != cudaSuccess) { return status; }
    const int threads = warps * WARP_SIZE;
    const long long tiles = (tile.n_reads + threads - 1) / threads;
    const int grid = static_cast< int >(tiles < geometry.multiprocessor_count ? tiles : geometry.multiprocessor_count);
    status = cudaMemsetAsync(params.tie_count + 2, 0, sizeof(unsigned), stream);
    if(status != cudaSuccess) { return status; }
    pamld_fast_kernel< G, UNIFORM ><<< grid, threads, bytes, stream >>>(params, tile);
    status = cudaGetLastError();
    if(status != cudaSuccess) { return status; }
    TileArguments rest(tile);
    rest.index_list = params.hard_list;
    rest.index_count = params.tie_count + 2;
    return launch_pamld_groups< G >(params, rest, geometry, stream);
}
/* the prefilter scan over every read of the launch, then the exact scan over the reads it left, then the tie pass */
template < int G >
cudaError_t launch_pamld_fast_groups(const DecoderParams& params, const TileArguments& tile, const LaunchGeometry& geometry, cudaStream_t stream) {
    return params.fast_uniform_prior > 0.0f ? launch_pamld_fast_groups_as< G, true >(params, tile, geometry, stream)
                                            : launch_pamld_fast_groups_as< G, false >(params, tile, geometry, stream);
}
template < int LA, int LB, int KBP >
cudaError_t launch_pamld_fast_grid_as(const DecoderParams& params, const TileArguments& tile, const LaunchGeometry& geometry, cudaStream_t stream) {
    constexpr int GROUPS = (LA + 3) / 4 + (LB + 3) / 4;
    const int blob_entries = params.grid_a + params.grid_b + params.grid_entries;
    const SharedPlan plan = make_plan(params.barcode_cardinality, true, blob_entries, true);
    const size_t per_warp = static_cast< size_t >(GROUPS) * FAST_GROUP_FLOATS * sizeof(float);
    const size_t dense_bytes = KBP > 0 ? (static_cast< size_t >(params.grid_entries) * sizeof(float) + 15) / 16 * 16 : 0;
    if(plan.fixed_bytes + dense_bytes + per_warp > geometry.shared_memory_per_block_optin) { return cudaErrorInvalidConfiguration; }
    int warps = static_cast< int >((geometry.shared_memory_per_block_optin - plan.fixed_bytes - dense_bytes) / per_warp);
    warps = warps > fast_grid_warps(KBP) ? fast_grid_warps(KBP) : warps;
    const size_t bytes = plan.fixed_bytes + per_warp * warps + dense_bytes;
    cudaError_t status = cudaFuncSetAttribute(pamld_fast_grid_kernel< LA, LB, KBP >, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast< int >(bytes));
    if(status != cudaSuccess) { return status; }
    const int threads = warps * WARP_SIZE;
    const long long tiles = (tile.n_reads + threads - 1) / threads;
    const int grid = static_cast< int >(tiles < geometry.multiprocessor_count ? tiles : geometry.multiprocessor_count);
    status = cudaMemsetAsync(params.tie_count + 2, 0, sizeof(unsigned), stream);
    if(status != cudaSuccess) { return status; }
    pamld_fast_grid_kernel< LA, LB, KBP ><<< grid, threads, bytes, stream >>>(params, tile);
    status = cudaGetLastError();
    if(status != cudaSuccess) { return status; }
    TileArguments rest(tile);
    rest.index_list = params.hard_list;
    rest.index_count = params.tie_count + 2;
    if(KBP == 0) { return launch_pamld_grid_as< LA, LB, 1, true >(params, rest, geometry, stream); }
    return launch_pamld_grid_as< LA, LB, (KBP == 0 ? 8 : KBP), false >(params, rest, geometry, stream);
}
/* the prefilter exists for the separable form (any supported shape) and for the dense form of the 8 + 8 and 10 + 10 shapes */
template < int LA, int LB, bool DENSE >
cudaError_t launch_pamld_fast_grid(const DecoderParams& params, const TileArguments& tile, const LaunchGeometry& geometry, cudaStream_t stream) {
    if(params.grid_uniform) { return launch_pamld_fast_grid_as< LA, LB, 0 >(params, tile, geometry, stream); }
    if(DENSE && params.grid_dense == 8) { return launch_pamld_fast_grid_as< LA, LB, 8 >(params, tile, geometry, stream); }
    if(DENSE && params.grid_dense == 16) { return launch_pamld_fast_grid_as< LA, LB, 16 >(params, tile, geometry, stream); }
    return cudaErrorInvalidValue;
}

/* the long scan (H = ceil(L / 8) groups per lane), then its tie pass */
template < int H >
cudaError_t launch_pamld_long(const DecoderParams& params, const TileArguments& tile, const LaunchGeometry& geometry, cudaStream_t stream) {
    const SharedPlan plan = make_plan(params.barcode_cardinality, true, long_stage_blob(params.barcode_cardinality));
    const size_t per_warp = static_cast< size_t >(H) * 16 * WARP_SIZE * sizeof(double);
    if(plan.fixed_bytes + per_warp > geometry.shared_memory_per_block_optin) { return cudaErrorInvalidConfiguration; }
    int warps = static_cast< int >((geometry.shared_memory_per_block_optin - plan.fixed_bytes) / per_warp);
    warps = warps > LONG_MAX_WARPS ? LONG_MAX_WARPS : warps;
    const size_t bytes = plan.fixed_bytes + per_warp * warps;
    cudaError_t status = cudaFuncSetAttribute(pamld_long_kernel< H >, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast< int >(bytes));
    if(status != cudaSuccess) { return status; }
    const int reads_per_tile = warps * WARP_SIZE / 2;
    const long long tiles = (tile.n_reads + reads_per_tile - 1) / reads_per_tile;
    const int grid = static_cast< int >(tiles < geometry.multiprocessor_count ? tiles : geometry.multiprocessor_count);
    status = cudaMemsetAsync(params.tie_count, 0, 2 * sizeof(unsigned), stream);      /* the tie queue's length and the tie pass' work counter */
    if(status != cudaSuccess) { return status; }
    pamld_long_kernel< H ><<< grid, warps * WARP_SIZE, bytes, stream >>>(params, tile);
    status = cudaGetLastError();
    if(status != cudaSuccess) { return status; }
    const size_t tie_bytes = long_tie_shared_bytes(params.barcode_cardinality);
    status = cudaFuncSetAttribute(pamld_long_tie_kernel< H >, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast< int >(tie_bytes));
    if(status != cudaSuccess) { return status; }
    pamld_long_tie_kernel< H ><<< geometry.multiprocessor_count * 2, TIE_THREADS, tie_bytes, stream >>>(params, tile);
    return cudaGetLastError();
}

template < int SEGMENTS >
cudaError_t launch_mdd_long_as(const DecoderParams& params, const TileArguments& tile, const LaunchGeometry& geometry, cudaStream_t stream) {
    const size_t bytes = make_plan(params.barcode_cardinality, false, long_stage_blob(params.barcode_cardinality)).fixed_bytes;
    const int threads = 256;
    const long long tiles = (tile.n_reads + threads - 1) / threads;
    const long long resident = static_cast< long long >(geometry.multiprocessor_count) * 4;
    const cudaError_t status = cudaFuncSetAttribute(mdd_long_kernel< SEGMENTS >, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast< int >(bytes));
    if(status != cudaSuccess) { return status; }
    mdd_long_kernel< SEGMENTS ><<< static_cast< int >(tiles < resident ? tiles : resident), threads, bytes, stream >>>(params, tile);
    return cudaGetLastError();
}

}   /* namespace */

static cudaError_t launch_pamld_whitelist(const DecoderParams& params, const TileArguments& tile, const LaunchGeometry& geometry, cudaStream_t stream) {
    constexpr int G = 4;
    if(WL_FIXED_BYTES + WL_WARP_BYTES > geometry.shared_memory_per_block_optin) { return cudaErrorInvalidConfiguration; }
    int warps = static_cast< int >((geometry.shared_memory_per_block_optin - WL_FIXED_BYTES) / WL_WARP_BYTES);
    warps = warps > WHITELIST_MAX_WARPS ? WHITELIST_MAX_WARPS : warps;
    const size_t bytes = WL_FIXED_BYTES + static_cast< size_t >(WL_WARP_BYTES) * warps;
    cudaError_t status = cudaFuncSetAttribute(pamld_whitelist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast< int >(bytes));
    if(status != cudaSuccess) { return status; }
    const long long units = (tile.n_reads + 31) / 32;
    const long long wanted = (units + warps - 1) / warps;
    const int grid = static_cast< int >(wanted < geometry.multiprocessor_count ? wanted : geometry.multiprocessor_count);
    /* the queue header: [0] tie queue length, [1] the next unit of 32 reads */
    status = cudaMemsetAsync(params.tie_count, 0, 4 * sizeof(unsigned), stream);
    if(status != cudaSuccess) { return status; }
    pamld_whitelist_kernel<<< grid, warps * WARP_SIZE, bytes, stream >>>(params, tile, params.tie_count + 1);
    status = cudaGetLastError();
    if(status != cudaSuccess) { return status; }
    return launch_tie< G >(params, tile, geometry, stream);
}

cudaError_t launch_pamld(const DecoderParams& params, const TileArguments& tile, const LaunchGeometry& geometry, cudaStream_t stream) {
    if(tile.n_reads <= 0) { return cudaSuccess; }
    if(params.nucleotide_cardinality > LONG_NUCLEOTIDES) {
        switch((params.nucleotide_cardinality + 7) / 8) {
            case 5: return launch_pamld_long< 5 >(params, tile, geometry, stream);
            case 6: return launch_pamld_long< 6 >(params, tile, geometry, stream);
            case 7: return launch_pamld_long< 7 >(params, tile, geometry, stream);
            case 8: return launch_pamld_long< 8 >(params, tile, geometry, stream);
            default: return cudaErrorInvalidValue;
        }
    }
    if(params.whitelist != nullptr) { return launch_pamld_whitelist(params, tile, geometry, stream); }
    if(params.fast_barcodes != nullptr) {
        /* f32 prefilter scan first (see pamld_fast_kernel); the api only offers it for the shapes handled here */
        if(params.grid != nullptr) {
            if(params.grid_split == 6 && params.nucleotide_cardinality == 12) { return launch_pamld_fast_grid< 6, 6, false >(params, tile, geometry, stream); }
            if(params.grid_split == 8 && params.nucleotide_cardinality == 16) { return launch_pamld_fast_grid< 8, 8, true >(params, tile, geometry, stream); }
            if(params.grid_split == 10 && params.nucleotide_cardinality == 20) { return launch_pamld_fast_grid< 10, 10, true >(params, tile, geometry, stream); }
            if(params.grid_split == 12 && params.nucleotide_cardinality == 24) { return launch_pamld_fast_grid< 12, 12, false >(params, tile, geometry, stream); }
            return cudaErrorInvalidValue;
        }
        switch(params.group_cardinality) {
            case 1: return launch_pamld_fast_groups< 1 >(params, tile, geometry, stream);
            case 2: return launch_pamld_fast_groups< 2 >(params, tile, geometry, stream);
            case 3: return launch_pamld_fast_groups< 3 >(params, tile, geometry, stream);
            case 4: return launch_pamld_fast_groups< 4 >(params, tile, geometry, stream);
            case 5: return launch_pamld_fast_groups< 5 >(params, tile, geometry, stream);
            case 6: return launch_pamld_fast_groups< 6 >(params, tile, geometry, stream);
            case 7: return launch_pamld_fast_groups< 7 >(params, tile, geometry, stream);
            case 8: return launch_pamld_fast_groups< 8 >(params, tile, geometry, stream);
            default: return cudaErrorInvalidValue;
        }
    }
    if(params.grid != nullptr) {
        if(params.grid_split == 6 && params.nucleotide_cardinality == 12) { return launch_pamld_grid< 6, 6, false >(params, tile, geometry, stream); }
        if(params.grid_split == 8 && params.nucleotide_cardinality == 16) { return launch_pamld_grid< 8, 8, true >(params, tile, geometry, stream); }
        if(params.grid_split == 10 && params.nucleotide_cardinality == 20) { return launch_pamld_grid< 10, 10, true >(params, tile, geometry, stream); }
        if(params.grid_split == 12 && params.nucleotide_cardinality == 24) { return launch_pamld_grid< 12, 12, false >(params, tile, geometry, stream); }
    }
    switch(params.group_cardinality) {
        case 1: return launch_pamld_groups< 1 >(params, tile, geometry, stream);
        case 2: return launch_pamld_groups< 2 >(params, tile, geometry, stream);
        case 3: return launch_pamld_groups< 3 >(params, tile, geometry, stream);
        case 4: return launch_pamld_groups< 4 >(params, tile, geometry, stream);
        case 5: return launch_pamld_groups< 5 >(params, tile, geometry, stream);
        case 6: return launch_pamld_groups< 6 >(params, tile, geometry, stream);
        case 7: return launch_pamld_groups< 7 >(params, tile, geometry, stream);
        case 8: return launch_pamld_groups< 8 >(params, tile, geometry, stream);
        default: return cudaErrorInvalidValue;
    }
}

static cudaError_t launch_mdd_scan(const DecoderParams& params, const TileArguments& tile, const LaunchGeometry& geometry, cudaStream_t stream) {
    const SharedPlan plan = make_plan(params.barcode_cardinality, false);
    const size_t bytes = plan.fixed_bytes;
    const int threads = 256;
    const long long tiles = (tile.n_reads + threads - 1) / threads;
    const long long resident = static_cast< long long >(geometry.multiprocessor_count) * 4;
    const int grid = static_cast< int >(tiles < resident ? tiles : resident);
    cudaError_t status;
    switch(params.segment_cardinality) {
        case 1:
            status = cudaFuncSetAttribute(mdd_kernel< 1 >, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast< int >(bytes));
            if(status != cudaSuccess) { return status; }
            mdd_kernel< 1 ><<< grid, threads, bytes, stream >>>(params, tile);
            break;
        case 2:
            status = cudaFuncSetAttribute(mdd_kernel< 2 >, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast< int >(bytes));
            if(status != cudaSuccess) { return status; }
            mdd_kernel< 2 ><<< grid, threads, bytes, stream >>>(params, tile);
            break;
        default:
            status = cudaFuncSetAttribute(mdd_kernel< 0 >, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast< int >(bytes));
            if(status != cudaSuccess) { return status; }
            mdd_kernel< 0 ><<< grid, threads, bytes, stream >>>(params, tile);
            break;
    }
    return cudaGetLastError();
}

cudaError_t launch_mdd(const DecoderParams& params, const TileArguments& tile, const LaunchGeometry& geometry, cudaStream_t stream) {
    if(tile.n_reads <= 0) { return cudaSuccess; }
    if(params.nucleotide_cardinality > LONG_NUCLEOTIDES) {
        switch(params.segment_cardinality) {
            case 1: return launch_mdd_long_as< 1 >(params, tile, geometry, stream);
            case 2: return launch_mdd_long_as< 2 >(params, tile, geometry, stream);
            default: return launch_mdd_long_as< 0 >(params, tile, geometry, stream);
        }
    }
    if(params.mdd_tables == nullptr) { return launch_mdd_scan(params, tile, geometry, stream); }
    /* lookup kernel, then the scan kernel over the reads it queued (short tokens) */
    int* const queue = reinterpret_cast< int* >(reinterpret_cast< unsigned char* >(params.tie_record));
    unsigned* const queue_count = params.tie_count;
    cudaError_t status = cudaMemsetAsync(queue_count, 0, sizeof(unsigned), stream);
    if(status != cudaSuccess) { return status; }
    const SharedPlan staged_plan = make_plan(params.barcode_cardinality, false, (params.mdd_slots + 1) / 2);
    const bool staged = staged_plan.fixed_bytes <= 54 * 1024;          /* keep four CTAs per SM */
    const SharedPlan plan = staged ? staged_plan : make_plan(params.barcode_cardinality, false, 1);
    const int threads = 256;
    const long long tiles = (tile.n_reads + threads - 1) / threads;
    const long long resident = static_cast< long long >(geometry.multiprocessor_count) * 4;
    const int grid = static_cast< int >(tiles < resident ? tiles : resident);
    const bool masking = params.quality_masking_threshold > 0;
    #define PHQ_LAUNCH_MDD_TABLE_AS(SEGMENTS, MASKING, STAGED) { \
            status = cudaFuncSetAttribute(mdd_table_kernel< SEGMENTS, MASKING, STAGED >, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast< int >(plan.fixed_bytes)); \
            if(status != cudaSuccess) { return status; } \
            mdd_table_kernel< SEGMENTS, MASKING, STAGED ><<< grid, threads, plan.fixed_bytes, stream >>>(params, tile, queue, queue_count); }
    #define PHQ_LAUNCH_MDD_TABLE(SEGMENTS) \
        if(masking && staged) PHQ_LAUNCH_MDD_TABLE_AS(SEGMENTS, true, true) \
        else if(masking) PHQ_LAUNCH_MDD_TABLE_AS(SEGMENTS, true, false) \
        else if(staged) PHQ_LAUNCH_MDD_TABLE_AS(SEGMENTS, false, true) \
        else PHQ_LAUNCH_MDD_TABLE_AS(SEGMENTS, false, false)
    switch(params.segment_cardinality) {
        case 1: PHQ_LAUNCH_MDD_TABLE(1) break;
        case 2: PHQ_LAUNCH_MDD_TABLE(2) break;
        case 3: PHQ_LAUNCH_MDD_TABLE(3) break;
        default: PHQ_LAUNCH_MDD_TABLE(4) break;
    }
    #undef PHQ_LAUNCH_MDD_TABLE_AS
    #undef PHQ_LAUNCH_MDD_TABLE
    status = cudaGetLastError();
    if(status != cudaSuccess) { return status; }
    TileArguments rest(tile);
    rest.index_list = queue;
    rest.index_count = queue_count;
    return launch_mdd_scan(params, rest, geometry, stream);
}

cudaError_t launch_reference_power(const double* sigma, double* out, long long n, double base, cudaStream_t stream) {
    if(n <= 0) { return cudaSuccess; }
    reference_power_kernel<<< 296, 256, 0, stream >>>(sigma, out, n, base);
    return cudaGetLastError();
}

cudaError_t launch_count(const DecoderParams& params, const TileArguments& tile, const LaunchGeometry& geometry, cudaStream_t stream) {
    if(tile.n_reads <= 0) { return cudaSuccess; }
    const int threads = 256;
    const long long blocks = (tile.n_reads + threads - 1) / threads;
    const long long resident = static_cast< long long >(geometry.multiprocessor_count) * 8;
    const int grid = static_cast< int >(blocks < resident ? blocks : resident);
    count_kernel<<< grid, threads, 0, stream >>>(params, tile);
    return cudaGetLastError();
}

/* the kernels launch_pamld / launch_mdd / launch_count pick for these parameters, for reports and profiles */
void describe_kernels(const DecoderParams& params, int algorithm, char* buffer, size_t capacity) {
    if(buffer == nullptr || capacity == 0) { return; }
    const int L = params.nucleotide_cardinality;
    if(algorithm <= 1 && L > LONG_NUCLEOTIDES) {
        if(algorithm == 0) { snprintf(buffer, capacity, "pamld_long_kernel<%d> + pamld_long_tie_kernel<%d>", (L + 7) / 8, (L + 7) / 8); }
        else { snprintf(buffer, capacity, "mdd_long_kernel<%d>", params.segment_cardinality <= 2 ? params.segment_cardinality : 0); }
    } else if(algorithm == 0) {
        const bool grid = params.grid != nullptr && grid_shape_supported(params.grid_split, L);
        if(params.whitelist != nullptr) {
            snprintf(buffer, capacity, "pamld_whitelist_kernel + pamld_tie_kernel<4>");
        } else if(grid) {
            const bool dense = params.grid_dense != 0 && (params.grid_split == 8 || params.grid_split == 10);
            char prefilter[64] = "";
            if(params.fast_barcodes != nullptr) { snprintf(prefilter, sizeof(prefilter), "pamld_fast_grid_kernel<%d, %d, %d> + ", params.grid_split, L - params.grid_split, params.grid_uniform ? 0 : params.grid_dense); }
            snprintf(buffer, capacity, "%spamld_grid_kernel<%d, %d, %d, %d, %d> + pamld_tie_kernel<%d>", prefilter, params.grid_split, L - params.grid_split,
                     GRID_GROUP_WIDTH, params.grid_uniform ? 1 : (dense ? params.grid_dense : 0), params.grid_uniform ? 1 : 0, (L + 3) / 4);
        } else {
            char prefilter[64] = "";
            if(params.fast_barcodes != nullptr) { snprintf(prefilter, sizeof(prefilter), "pamld_fast_kernel<%d, %d> + ", params.group_cardinality, params.fast_uniform_prior > 0.0f ? 1 : 0); }
            snprintf(buffer, capacity, "%spamld_kernel<%d> + pamld_tie_kernel<%d>", prefilter, params.group_cardinality, params.group_cardinality);
        }
    } else if(algorithm == 1) {
        const int scan = params.segment_cardinality <= 2 ? params.segment_cardinality : 0;
        if(params.mdd_tables != nullptr) {
            snprintf(buffer, capacity, "mdd_table_kernel<%d> + mdd_kernel<%d> (short reads)", params.segment_cardinality < 4 ? params.segment_cardinality : 4, scan);
        } else {
            snprintf(buffer, capacity, "mdd_kernel<%d>", scan);
        }
    } else {
        snprintf(buffer, capacity, "count_kernel");
    }
}

cudaError_t prepare_kernels(const LaunchGeometry&) {
    return cudaSuccess;
}

}   /* namespace phq */
