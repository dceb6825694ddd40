/*  api.cu — the C ABI of include/pheniqs_b200.h: handle, device memory, host packer, launches.

    The handle plays the role of one thread's TranscodingDecoder (transcode.h:40-65,
    transcode.cpp:60-195): it owns the decoder chain, their barcode tables and accumulators.
    File:line citations are relative to the reference tree.
*/
#include "kernels.cuh"
#include "pack.cuh"
#include "spec.hpp"
#include "report.hpp"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>               /* types only: the entry points are resolved at run time (NcclLibrary) */

#include <array>
#include <cmath>
#include <exception>
#include <functional>
#include <thread>
#include <cstring>
#include <string>
#include <vector>

using namespace phq;

namespace {

thread_local std::string global_error;

#define PHQ_CUDA(call) do { cudaError_t status_ = (call); if(status_ != cudaSuccess) { \
    throw phq::Error(status_ == cudaErrorMemoryAllocation ? PHQ_OUT_OF_MEMORY_ERROR : PHQ_INTERNAL_ERROR, \
        std::string("Internal error : CUDA ") + cudaGetErrorName(status_) + " : " + cudaGetErrorString(status_) + " in " #call); } } while(0)

/* iupac.h:107-124 BamToReverseComplementBam */
const uint8_t BAM_REVERSE_COMPLEMENT[16] = { 0x0, 0x8, 0x4, 0xc, 0x2, 0xa, 0x6, 0xe, 0x1, 0x9, 0x5, 0xd, 0x3, 0xb, 0x7, 0xf };

/* the per-segment scratch an Observation keeps from read to read (sequence.h:264-300) */
struct ScratchSegment {
    std::vector< uint8_t > code;
    std::vector< uint8_t > quality;
    int32_t length;
    ScratchSegment() : code(PHQ_MAX_NUCLEOTIDES * 4 + 64, 0), quality(PHQ_MAX_NUCLEOTIDES * 4 + 64, 0), length(0) {}
};

/* threads phq_pack spreads a batch over: PHQ_PACK_THREADS, else the hardware's, at most 16, and 1 below 32 Ki reads */
inline int pack_workers(int64_t n_reads) {
    const char* const value(getenv("PHQ_PACK_THREADS"));
    int workers(value != NULL && atoi(value) > 0 ? atoi(value) : static_cast< int >(std::thread::hardware_concurrency()));
    if(workers > 16) { workers = 16; }
    if(value == NULL && n_reads < 32768) { workers = 1; }
    if(static_cast< int64_t >(workers) > n_reads) { workers = n_reads > 0 ? static_cast< int >(n_reads) : 1; }
    return workers < 1 ? 1 : workers;
}

/* device memory of T, freed with its owner; the owner makes the device current before it goes (destroy) */
template < class T > struct DeviceBuffer {
    T* pointer;
    size_t capacity;
    DeviceBuffer() : pointer(NULL), capacity(0) {}
    DeviceBuffer(const DeviceBuffer&) = delete;
    DeviceBuffer& operator=(const DeviceBuffer&) = delete;
    DeviceBuffer(DeviceBuffer&& other) noexcept : pointer(other.pointer), capacity(other.capacity) { other.pointer = NULL; other.capacity = 0; }
    DeviceBuffer& operator=(DeviceBuffer&& other) noexcept {
        if(this != &other) { release(); pointer = other.pointer; capacity = other.capacity; other.pointer = NULL; other.capacity = 0; }
        return *this;
    }
    ~DeviceBuffer() { release(); }
    /* grow only: staging buffers keep their memory from call to call */
    void reserve(size_t count) {
        if(count > capacity) {
            release();
            PHQ_CUDA(cudaMalloc(reinterpret_cast< void** >(&pointer), count * sizeof(T)));
            capacity = count;
        }
    }
    /* the whole table, in memory allocated at its size (at least `minimum` elements): nothing stale lies past its end */
    void upload(const std::vector< T >& table, size_t minimum = 0) {
        release();
        reserve(table.size() > minimum ? table.size() : minimum);
        PHQ_CUDA(cudaMemcpy(pointer, table.data(), table.size() * sizeof(T), cudaMemcpyHostToDevice));
    }
    /* no CUDA call on an empty buffer: a host-only handle never touches the runtime */
    void release() {
        if(pointer != NULL) { cudaFree(pointer); pointer = NULL; capacity = 0; }
    }
};

/* one 16-byte record of a combinatorial codec blob (pamld_grid_kernel) */
struct GridCell { uint32_t a, b, c, d; };

/*  The device tables of one decoder and what their builders derive. Each builder resets its own part and fills it
    where its kernel applies; an empty buffer (NULL) means the kernel does not run for this decoder. */
struct DecoderTables {
    DeviceBuffer< BarcodeEntry > barcodes;      /* padded to whole WHITELIST_CHUNK groups with zero entries (prior 0) */
    DeviceBuffer< LongBarcodeEntry > long_barcodes;     /* decoders of more than LONG_NUCLEOTIDES (kernels.cuh) instead of `barcodes` */
    DeviceBuffer< FastEntry > fast;             /* f32 form of the barcode table for the prefilter scans */
    DeviceBuffer< GridCell > grid;              /* combinatorial codec blob (kernels.cuh) */
    int32_t grid_a = 0, grid_b = 0, grid_entries = 0, grid_split = 0, grid_dense = 0, grid_uniform = 0;
    DeviceBuffer< unsigned char > whitelist;    /* chunked whitelist blob (kernels.cuh) */
    int32_t whitelist_chunks = 0;
    double prior_maximum = 0;
    DeviceBuffer< MddSlot > mdd;                /* MDD lookup tables (kernels.cuh), empty where the scan kernel is used */
    int32_t mdd_first[PHQ_MAX_SEGMENTS + 1] = {}, mdd_mask[PHQ_MAX_SEGMENTS + 1] = {}, mdd_slots = 0;    /* where `mdd` holds tables: first slot and mask of every table, total slots */
    DeviceBuffer< uint8_t > barcode_code;       /* tag synthesis: [(N + 1)][L] BAM codes, row 0 undetermined */
};

/* device staging of one in-flight sub-batch of phq_decode_batch */
struct StagingSlot {
    cudaStream_t stream;
    cudaEvent_t done;
    std::vector< DeviceBuffer< uint32_t > > bases;
    std::vector< DeviceBuffer< uint16_t > > nmask;
    std::vector< DeviceBuffer< uint32_t > > quality;
    std::vector< DeviceBuffer< phq_result > > results;
    DeviceBuffer< uint8_t > qcfail;
    DeviceBuffer< unsigned char > tie_list;  /* queue of the PAMLD tie pass: counter, read indices, records */
    std::vector< DeviceBuffer< uint8_t > > raw_sequence;    /* feed bytes of phq_decode_batch_raw, per input segment */
    std::vector< DeviceBuffer< uint8_t > > raw_quality;
    std::vector< DeviceBuffer< long long > > raw_offset;
    DeviceBuffer< uint8_t > aux;                /* tag synthesis: auxiliary records and their lengths */
    DeviceBuffer< int32_t > aux_length;
    StagingSlot() : stream(NULL), done(NULL) {}
    ~StagingSlot() {
        if(done != NULL) { cudaEventDestroy(done); }
        if(stream != NULL) { cudaStreamDestroy(stream); }
    }
};

constexpr int STAGING_SLOTS = 3;
constexpr long long SUB_BATCH_READS = 1ll << 22;

}   /* namespace */

struct phq_handle {
    int device;
    Json job;                                   /* the compiled job as given (codec records for the report) */
    std::vector< DecoderSpec > chain;
    std::vector< DecoderParams > params;
    std::vector< std::vector< ScratchSegment > > scratch;
    std::vector< DecoderTables > tables;        /* per decoder */
    DeviceBuffer< uint8_t > device_read_group_text;     /* tag synthesis: read group IDs of the sample decoder */
    DeviceBuffer< int32_t > device_read_group_offset;
    int32_t read_group_longest;
    bool tags_ready;
    DeviceBuffer< float > device_phred32;       /* f32 mismatch ratios */
    bool fast_enabled;                          /* PHQ_DISABLE_FAST=1 keeps every PAMLD decoder on the exact scans */
    DeviceBuffer< double > device_phred;
    DeviceBuffer< unsigned char > device_accumulators;
    std::vector< int64_t > offset_u64;
    std::vector< int64_t > offset_f64;
    int64_t n_u64;
    int64_t n_f64;
    LaunchGeometry geometry;
    StagingSlot slot[STAGING_SLOTS];
    DeviceBuffer< unsigned char > tie_list;  /* tie queue of the device path (one batch in flight per handle) */
    cudaEvent_t timing_start;
    cudaEvent_t timing_stop;
    cudaStream_t timing_stream;
    bool timing_valid;
    uint64_t kernel_launches;
    long long sub_batch_reads;              /* reads per in-flight sub-batch of the host-buffer calls */
    bool collected;                         /* the tables hold the sums of all ranks (phq_collect): no decode / collect until reset */
    std::string error;

    phq_handle() : device(0), read_group_longest(0), tags_ready(false), fast_enabled(true), n_u64(0), n_f64(0),
        timing_start(NULL), timing_stop(NULL), timing_stream(NULL), timing_valid(false), kernel_launches(0), sub_batch_reads(SUB_BATCH_READS), collected(false) {
        /* PHQ_SUB_BATCH_READS: smaller sub-batches (tests exercise the boundaries with small inputs) */
        const char* const value(getenv("PHQ_SUB_BATCH_READS"));
        if(value != NULL && atoll(value) > 0) { sub_batch_reads = atoll(value); }
        const char* const disable(getenv("PHQ_DISABLE_FAST"));
        if(disable != NULL && atoi(disable) > 0) { fast_enabled = false; }
    }
    ~phq_handle() {
        if(timing_start != NULL) { cudaEventDestroy(timing_start); }
        if(timing_stop != NULL) { cudaEventDestroy(timing_stop); }
    }

    unsigned long long* u64_plane() const { return reinterpret_cast< unsigned long long* >(device_accumulators.pointer); }
    double* f64_plane() const { return reinterpret_cast< double* >(device_accumulators.pointer + n_u64 * 8); }
    unsigned long long* totals() const { return u64_plane() + n_u64 - 4; }
    unsigned long long* diagnostics() const { return u64_plane() + n_u64 - 2; }
};

namespace {

/* phred.h:33-34, phred.cpp:24-72 with the host libm, then the factored forms the kernels consume */
void assemble_phred(std::vector< double >& table, double& uniform_quality, double& base) {
    table.assign(PHRED_TABLE_SIZE, 0.0);
    uniform_quality = 10.0 * log10(4);
    base = pow(10.0, -0.1);
    table[PHRED_MATCH_FACTOR] = 1.0;
    table[PHRED_MISMATCH_RATIO] = 1.0;
    for(int q(1); q < 0x80; ++q) {
        const double false_positive_probability(pow(base, q));
        const double true_positive_probability(1.0 - false_positive_probability);
        const double true_positive_quality(-10.0 * log10(true_positive_probability));
        table[PHRED_TRUE_POSITIVE_QUALITY + q] = true_positive_quality;
        table[PHRED_MATCH_FACTOR + q] = pow(base, true_positive_quality);
        table[PHRED_MISMATCH_RATIO + q] = pow(base, static_cast< double >(q) - true_positive_quality);
    }
    table[PHRED_UNIFORM_QUALITY] = uniform_quality;
    table[PHRED_BASE] = base;
    table[PHRED_UNIFORM_FACTOR] = pow(base, uniform_quality);
}

/* the 2-bit code the barcode tables hold for a BAM base code: A 0, C 1, G 2, T 3 */
inline uint32_t two_bit_code(uint8_t code) { return code == 1 ? 0u : code == 2 ? 1u : code == 4 ? 2u : 3u; }

/* positions [from, to) of barcode b as low / high bit-planes, position `from` at bit 0 */
void barcode_planes(const DecoderSpec& d, int32_t b, int32_t from, int32_t to, uint32_t& lo, uint32_t& hi) {
    lo = 0; hi = 0;
    for(int32_t j(from); j < to; ++j) {
        const uint32_t two(two_bit_code(d.barcode[static_cast< size_t >(b) * d.nucleotide_cardinality + j]));
        lo |= (two & 1u) << (j - from);
        hi |= (two >> 1) << (j - from);
    }
}

void upload_barcodes(phq_handle* h, size_t k) {
    const DecoderSpec& d(h->chain[k]);
    if(d.nucleotide_cardinality > LONG_NUCLEOTIDES) {
        /* split form: positions [0, split) in the first word of each plane, [split, L) in the second */
        const int32_t split(long_split(d.nucleotide_cardinality));
        std::vector< LongBarcodeEntry > table(static_cast< size_t >(d.barcode_cardinality));
        for(int32_t b(0); b < d.barcode_cardinality; ++b) {
            LongBarcodeEntry e;
            memset(&e, 0, sizeof(e));
            barcode_planes(d, b, 0, split, e.lo0, e.hi0);
            barcode_planes(d, b, split, d.nucleotide_cardinality, e.lo1, e.hi1);
            e.prior = d.concentration[b];
            table[b] = e;
        }
        h->tables[k].long_barcodes.upload(table);
        return;
    }
    /* padded to whole whitelist groups with zero entries (prior 0): pamld_whitelist_kernel may look a padding barcode up */
    std::vector< BarcodeEntry > table((static_cast< size_t >(d.barcode_cardinality) + WHITELIST_CHUNK - 1) / WHITELIST_CHUNK * WHITELIST_CHUNK);
    for(int32_t b(0); b < d.barcode_cardinality; ++b) {
        BarcodeEntry e;
        barcode_planes(d, b, 0, d.nucleotide_cardinality, e.lo, e.hi);
        e.prior = d.concentration[b];
        table[b] = e;
    }
    h->tables[k].barcodes.upload(table);
}

/* the barcode table in the form the f32 prefilter scans read (pamld_fast_kernel) */
void upload_fast(phq_handle* h, size_t k) {
    const DecoderSpec& d(h->chain[k]);
    h->tables[k].fast.release();
    /* no prefilter for long decoders: its f32 error bound is argued for at most 32 positions, and 4^-64 is below the
       smallest normal float */
    if(d.algorithm != PHQ_PAMLD || !h->fast_enabled || d.nucleotide_cardinality > LONG_NUCLEOTIDES) { return; }
    std::vector< FastEntry > table(static_cast< size_t >(d.barcode_cardinality));
    for(int32_t b(0); b < d.barcode_cardinality; ++b) {
        FastEntry e;
        e.pad = 0;
        barcode_planes(d, b, 0, d.nucleotide_cardinality, e.lo, e.hi);
        e.prior = static_cast< float >(d.concentration[b]);
        table[b] = e;
    }
    h->tables[k].fast.upload(table, 1);
}

/*  Combinatorial codecs (C1: 12 distinct i7 words x 8 distinct i5 words = 96 barcodes): group the barcodes
    by the word of their first segment and index the distinct words of the remaining segments, so the scan
    forms each word's probability once per read (pamld_grid_kernel). Built when it pays: at least two
    segments, a supported shape, and far fewer distinct words than barcodes. */
void upload_grid(phq_handle* h, size_t k) {
    const DecoderSpec& d(h->chain[k]);
    DecoderTables& tables(h->tables[k]);
    tables.grid.release();
    tables.grid_a = tables.grid_b = tables.grid_entries = tables.grid_split = tables.grid_dense = tables.grid_uniform = 0;
    if(d.algorithm != PHQ_PAMLD || d.segment_cardinality < 2) { return; }
    const int32_t split(d.segment_length[0]);
    const int32_t L(d.nucleotide_cardinality);
    if(!grid_shape_supported(split, L)) { return; }
    std::map< std::pair< uint32_t, uint32_t >, std::vector< int32_t > > by_prefix;
    std::map< std::pair< uint32_t, uint32_t >, int32_t > suffix_index;
    std::vector< std::pair< uint32_t, uint32_t > > suffix_word;
    std::vector< int32_t > suffix_of(static_cast< size_t >(d.barcode_cardinality));
    for(int32_t b(0); b < d.barcode_cardinality; ++b) {
        uint32_t lo, hi;
        barcode_planes(d, b, 0, split, lo, hi);
        by_prefix[std::make_pair(lo, hi)].push_back(b);
        barcode_planes(d, b, split, L, lo, hi);
        const auto key(std::make_pair(lo, hi));
        auto found(suffix_index.find(key));
        if(found == suffix_index.end()) {
            found = suffix_index.emplace(key, static_cast< int32_t >(suffix_word.size())).first;
            suffix_word.push_back(key);
        }
        suffix_of[b] = found->second;
    }
    const size_t KA(by_prefix.size()), KB(suffix_word.size());
    if((KA + KB) * 2 > static_cast< size_t >(d.barcode_cardinality) || KB > 64) { return; }
    /* dense form when the codec fills most of the KA x KB grid: every A word gets KBP consecutive entries in B
       word order, absent combinations carry prior 0 (pamld_grid_kernel, KBP > 0) */
    /* separable form: the full KA x KB grid under one prior (the default of a multiplexed run before prior
       estimation); entries are the KA x KB matrix and the kernel evaluates KA + KB words per read */
    bool uniform(static_cast< size_t >(d.barcode_cardinality) == KA * KB);
    for(int32_t b(1); b < d.barcode_cardinality && uniform; ++b) { uniform = d.concentration[b] == d.concentration[0]; }
    const size_t KBP(uniform ? KB : (KB <= 8 ? 8 : 16));
    const bool shape_dense((split == 8 && L == 16) || (split == 10 && L == 20));
    const bool dense(uniform || (shape_dense && KB <= 16 && static_cast< size_t >(d.barcode_cardinality) * 10 >= KA * KBP * 6));
    std::vector< GridCell > blob(KA + (dense ? KBP : KB));
    std::vector< GridCell > entries;
    size_t at(0);
    for(const auto& run : by_prefix) {
        GridCell header;
        header.a = run.first.first; header.b = run.first.second;
        header.c = static_cast< uint32_t >(entries.size());
        if(dense) {
            GridCell none;
            none.a = 0; none.b = 0; none.c = 0; none.d = 0;
            const size_t first(entries.size());
            entries.resize(first + KBP, none);
            for(int32_t b : run.second) {
                GridCell& e(entries[first + static_cast< size_t >(suffix_of[b])]);
                e.a = static_cast< uint32_t >(suffix_of[b]) * 256u;
                e.b = static_cast< uint32_t >(b);
                memcpy(&e.c, &d.concentration[b], sizeof(double));
            }
        } else {
            for(int32_t b : run.second) {
                GridCell e;
                e.a = static_cast< uint32_t >(suffix_of[b]) * 256u;
                e.b = static_cast< uint32_t >(b);
                memcpy(&e.c, &d.concentration[b], sizeof(double));
                entries.push_back(e);
            }
            while(entries.size() % 4 != 0) {        /* pad the run with prior 0: the product is 0 and never wins */
                GridCell e;
                e.a = 0; e.b = 0; e.c = 0; e.d = 0;
                entries.push_back(e);
            }
        }
        header.d = static_cast< uint32_t >(entries.size()) - header.c;
        blob[at++] = header;
    }
    for(size_t i(0); i < (dense ? KBP : KB); ++i) {
        GridCell w;
        w.a = i < KB ? suffix_word[i].first : 0u; w.b = i < KB ? suffix_word[i].second : 0u; w.c = 0; w.d = 0;
        blob[at++] = w;
    }
    blob.insert(blob.end(), entries.begin(), entries.end());
    if(blob.size() * 16 > 64 * 1024) { return; }
    tables.grid.upload(blob);
    tables.grid_a = static_cast< int32_t >(KA);
    tables.grid_b = static_cast< int32_t >(dense ? KBP : KB);
    tables.grid_entries = static_cast< int32_t >(entries.size());
    tables.grid_split = split;
    tables.grid_dense = dense ? static_cast< int32_t >(KBP) : 0;
    tables.grid_uniform = uniform ? 1 : 0;
}

/*  Large single-word codecs (a cellular whitelist): the chunked blob pamld_whitelist_kernel streams — per chunk of
    WHITELIST_CHUNK barcodes the equality planes of its blocks of 32, the barcode words and the priors (kernels.cuh). */
void upload_whitelist(phq_handle* h, size_t k) {
    const DecoderSpec& d(h->chain[k]);
    DecoderTables& tables(h->tables[k]);
    tables.whitelist.release();
    tables.whitelist_chunks = 0;
    tables.prior_maximum = 0;
    long long minimum(WHITELIST_MINIMUM_BARCODES);
    const char* const value(getenv("PHQ_WHITELIST_MINIMUM"));
    if(value != NULL && atoll(value) > 0) { minimum = atoll(value); }
    if(d.algorithm != PHQ_PAMLD || d.nucleotide_cardinality > WHITELIST_POSITIONS || d.barcode_cardinality < minimum) { return; }
    const int32_t L(d.nucleotide_cardinality);
    const size_t chunks((static_cast< size_t >(d.barcode_cardinality) + WHITELIST_CHUNK - 1) / WHITELIST_CHUNK);
    std::vector< unsigned char > blob(chunks * WHITELIST_CHUNK_BYTES, 0);
    double largest(0);
    for(size_t c(0); c < chunks; ++c) {
        uint32_t* const equality(reinterpret_cast< uint32_t* >(blob.data() + c * WHITELIST_CHUNK_BYTES));
        /* plane (position j, code c) of block b at word ((j * planes + c) * blocks + b): one 16-byte load per position covers the group */
        for(int32_t block(0); block < WHITELIST_BLOCKS; ++block) {
            for(int32_t j(0); j < WHITELIST_POSITIONS; ++j) { equality[(j * WHITELIST_PLANES + 4) * WHITELIST_BLOCKS + block] = 0xffffffffu; }
        }
        for(int32_t i(0); i < WHITELIST_CHUNK; ++i) {
            const size_t b(c * WHITELIST_CHUNK + static_cast< size_t >(i));
            if(b >= static_cast< size_t >(d.barcode_cardinality)) { break; }      /* padding: no plane bit, prior 0 */
            for(int32_t j(0); j < L; ++j) {
                const int32_t two(static_cast< int32_t >(two_bit_code(d.barcode[b * L + j])));
                equality[(j * WHITELIST_PLANES + two) * WHITELIST_BLOCKS + (i >> 5)] |= 1u << (i & 31);
            }
            if(d.concentration[b] > largest) { largest = d.concentration[b]; }
        }
    }
    tables.whitelist.upload(blob);
    tables.whitelist_chunks = static_cast< int32_t >(chunks);
    tables.prior_maximum = largest;
}

/*  MDD lookup tables (MddSlot, kernels.cuh). Built when the reference's scan is provably a lookup: every segment
    is at most 16 nucleotides, at most four segments, and every tolerance is within the segment's Shannon bound
    (metric.h:87-111), so the spheres of radius `tolerance` around the distinct words of a segment are disjoint. */
void upload_mdd_tables(phq_handle* h, size_t k) {
    const DecoderSpec& d(h->chain[k]);
    DecoderTables& tables(h->tables[k]);
    tables.mdd.release();
    tables.mdd_slots = 0;
    if(d.algorithm != PHQ_MDD || d.segment_cardinality > 4 || d.barcode_cardinality > MDD_MAX_BARCODES) { return; }
    if(d.nucleotide_cardinality > LONG_NUCLEOTIDES) { return; }        /* the lookup kernel reads 32-position planes */
    const int32_t S(d.segment_cardinality);
    const int32_t L(d.nucleotide_cardinality);
    std::vector< std::vector< std::vector< uint8_t > > > words(static_cast< size_t >(S));      /* distinct words per segment, 2-bit codes */
    std::vector< std::vector< int32_t > > word_of(static_cast< size_t >(S), std::vector< int32_t >(static_cast< size_t >(d.barcode_cardinality)));
    for(int32_t s(0); s < S; ++s) {
        if(d.segment_length[s] > 16) { return; }
        std::map< std::vector< uint8_t >, int32_t > index;
        for(int32_t b(0); b < d.barcode_cardinality; ++b) {
            std::vector< uint8_t > w;
            for(int32_t j(d.segment_offset[s]); j < d.segment_offset[s + 1]; ++j) {
                w.push_back(static_cast< uint8_t >(two_bit_code(d.barcode[static_cast< size_t >(b) * L + j])));
            }
            auto found(index.find(w));
            if(found == index.end()) {
                found = index.emplace(w, static_cast< int32_t >(words[s].size())).first;
                words[s].push_back(w);
            }
            word_of[s][b] = found->second;
        }
        if(words[s].size() > static_cast< size_t >(MDD_MAX_WORDS)) { return; }
        /* Shannon bound of the segment: (minimum pairwise distance - 1) / 2 */
        int32_t minimum(d.segment_length[s]);
        if(words[s].size() > 4096) { return; }          /* the pairwise scan is quadratic */
        for(size_t i(0); i < words[s].size(); ++i) {
            for(size_t j(i + 1); j < words[s].size(); ++j) {
                int32_t distance(0);
                for(size_t p(0); p < words[s][i].size(); ++p) { distance += words[s][i][p] != words[s][j][p]; }
                minimum = std::min(minimum, distance);
            }
        }
        const int32_t bound((minimum - 1) / 2);
        if(words[s].size() > 1 && d.distance_tolerance[s] > bound) { return; }
        if(d.distance_tolerance[s] >= d.segment_length[s] || d.distance_tolerance[s] < 0 || d.distance_tolerance[s] > 3) { return; }
    }
    /* enumerate every variant within tolerance: a subset of positions, each replaced by another base or made ambiguous */
    struct Entry { uint32_t key_lo, key_hi, value; };
    std::vector< std::vector< Entry > > entries(static_cast< size_t >(S) + 1);
    for(int32_t s(0); s < S; ++s) {
        const int32_t n(d.segment_length[s]);
        const int32_t tolerance(d.distance_tolerance[s]);
        std::map< std::pair< uint32_t, uint32_t >, uint32_t > seen;
        for(size_t w(0); w < words[s].size(); ++w) {
            std::vector< int32_t > position;
            std::function< bool(int32_t, uint32_t, uint32_t, uint32_t, int32_t) > visit;
            bool clash(false);
            visit = [&](int32_t from, uint32_t lo, uint32_t hi, uint32_t amb, int32_t changed) -> bool {
                const uint32_t key_lo((lo & ~amb) | ((hi & ~amb) << 16));
                const uint32_t value(static_cast< uint32_t >(w) | (static_cast< uint32_t >(changed) << 12));
                auto inserted(seen.emplace(std::make_pair(key_lo, amb), value));
                if(!inserted.second && (inserted.first->second & 0xfffu) != static_cast< uint32_t >(w)) { clash = true; return false; }
                if(inserted.second) {
                    Entry e; e.key_lo = key_lo; e.key_hi = amb; e.value = value;
                    entries[s].push_back(e);
                    if(entries[s].size() > 200000) { clash = true; return false; }
                }
                if(changed == tolerance) { return true; }
                for(int32_t p(from); p < n; ++p) {
                    const uint32_t bit(1u << p);
                    const uint32_t original(((lo >> p) & 1u) | (((hi >> p) & 1u) << 1));
                    for(uint32_t alternative(0); alternative < 4; ++alternative) {
                        if(alternative == original) { continue; }
                        const uint32_t lo2((lo & ~bit) | ((alternative & 1u) << p));
                        const uint32_t hi2((hi & ~bit) | ((alternative >> 1) << p));
                        if(!visit(p + 1, lo2, hi2, amb, changed + 1)) { return false; }
                    }
                    if(!visit(p + 1, lo, hi, amb | bit, changed + 1)) { return false; }
                }
                return true;
            };
            uint32_t lo(0), hi(0);
            for(int32_t p(0); p < n; ++p) { lo |= (words[s][w][p] & 1u) << p; hi |= (static_cast< uint32_t >(words[s][w][p]) >> 1) << p; }
            visit(0, lo, hi, 0u, 0);
            if(clash) { return; }
        }
    }
    /* the tuple of words -> barcode (for one segment: word -> barcode, words are in first-occurrence order) */
    for(int32_t b(0); b < d.barcode_cardinality; ++b) {
        uint32_t id[4] = { 0u, 0u, 0u, 0u };
        for(int32_t s(0); s < S; ++s) { id[s] = static_cast< uint32_t >(word_of[s][b]); }
        Entry e;
        e.key_lo = id[0] | (id[1] << 12) | (id[2] << 24);
        e.key_hi = (id[2] >> 8) | (id[3] << 4);
        e.value = static_cast< uint32_t >(b);
        entries[S].push_back(e);
    }
    /* open addressing tables, load factor <= 1/4 (mdd_probe fetches the home slot and its neighbour up front) */
    std::vector< MddSlot > blob;
    for(int32_t t(0); t <= S; ++t) {
        size_t slots(4);
        while(slots < entries[t].size() * 4) { slots *= 2; }
        const size_t first(blob.size());
        MddSlot empty; empty.key_lo = 0; empty.key_hi = 0; empty.value = static_cast< uint16_t >(MDD_EMPTY);
        blob.resize(first + slots, empty);
        for(const auto& e : entries[t]) {
            size_t at(mdd_hash(e.key_lo, e.key_hi) & (slots - 1));
            while(blob[first + at].value != MDD_EMPTY) { at = (at + 1) & (slots - 1); }
            blob[first + at].key_lo = e.key_lo; blob[first + at].key_hi = static_cast< uint16_t >(e.key_hi); blob[first + at].value = static_cast< uint16_t >(e.value);
        }
        tables.mdd_first[t] = static_cast< int32_t >(first);
        tables.mdd_mask[t] = static_cast< int32_t >(slots - 1);
    }
    if(blob.size() > (1u << 20)) { return; }
    tables.mdd.upload(blob);
    tables.mdd_slots = static_cast< int32_t >(blob.size());
}

/* every device table of decoder k, from its codec and its priors */
void build_tables(phq_handle* h, size_t k) {
    upload_barcodes(h, k);
    upload_fast(h, k);
    upload_grid(h, k);
    upload_whitelist(h, k);
    upload_mdd_tables(h, k);
}

void refresh_params(phq_handle* h, size_t k) {
    const DecoderSpec& d(h->chain[k]);
    DecoderParams& p(h->params[k]);
    memset(&p, 0, sizeof(p));
    p.algorithm = d.algorithm;
    p.barcode_cardinality = d.barcode_cardinality;
    p.nucleotide_cardinality = d.nucleotide_cardinality;
    p.word_cardinality = d.word_cardinality();
    p.quality_word_cardinality = d.quality_word_cardinality();
    p.group_cardinality = d.quality_word_cardinality();
    p.segment_cardinality = d.segment_cardinality;
    const bool long_form(d.nucleotide_cardinality > LONG_NUCLEOTIDES);
    p.long_split = long_form ? long_split(d.nucleotide_cardinality) : 0;
    for(int32_t s(0); s < d.segment_cardinality && s < PHQ_MAX_SEGMENTS; ++s) {
        /* long decoders: the mask in split form (kernels.cuh), word 0 here and word 1 in segment_mask_long */
        uint64_t mask(0);
        for(int32_t j(d.segment_offset[s]); j < d.segment_offset[s + 1]; ++j) { mask |= static_cast< uint64_t >(1) << j; }
        p.segment_mask[s] = static_cast< uint32_t >(long_form ? (mask & ((static_cast< uint64_t >(1) << p.long_split) - 1)) : mask);
        p.segment_mask_long[s] = long_form ? static_cast< uint32_t >(mask >> p.long_split) : 0u;
        p.distance_tolerance[s] = d.algorithm == PHQ_MDD ? d.distance_tolerance[s] : 0;
    }
    p.high_quality_threshold = d.high_quality_threshold;
    p.high_quality_distance_threshold = d.high_quality_distance_threshold;
    p.quality_masking_threshold = d.quality_masking_threshold;
    p.adjusted_noise_probability = d.noise * d.random_barcode_probability;           /* pamld.cpp:29 */
    p.confidence_threshold = d.confidence_threshold;
    p.random_barcode_probability = d.random_barcode_probability;
    {
        /* sigma_q of an observation whose every position scores UNIFORM_BASE_QUALITY (barcode.h:147-163) */
        const double U(10.0 * log10(4));
        double y(0), t(0), sigma(0), compensation(0);
        for(int32_t j(0); j < d.nucleotide_cardinality; ++j) {
            y = U - compensation;
            t = sigma + y;
            compensation = (t - sigma) - y;
            sigma = t;
        }
        p.uniform_observation_probability = pow(pow(10.0, -0.1), sigma);
    }
    const DecoderTables& tables(h->tables[k]);
    p.barcodes = tables.barcodes.pointer;
    p.long_barcodes = tables.long_barcodes.pointer;
    p.phred = h->device_phred.pointer;
    p.acc_u64 = h->u64_plane() + h->offset_u64[k];
    p.acc_f64 = h->f64_plane() + h->offset_f64[k];
    p.totals = NULL;
    p.diagnostics = h->diagnostics();
    for(int32_t s(0); s < d.segment_cardinality && s < PHQ_MAX_SEGMENTS; ++s) {
        p.segment_offset[s] = d.segment_offset[s];
        p.segment_length[s] = d.segment_length[s];
    }
    p.mdd_tables = tables.mdd.pointer;
    if(p.mdd_tables != NULL) {
        for(int32_t t(0); t <= d.segment_cardinality; ++t) { p.mdd_first[t] = tables.mdd_first[t]; p.mdd_mask[t] = tables.mdd_mask[t]; }
        p.mdd_slots = tables.mdd_slots;
    }
    p.whitelist = tables.whitelist.pointer;
    p.whitelist_chunks = tables.whitelist_chunks;
    p.prior_maximum = tables.prior_maximum;
    p.grid = tables.grid.pointer;
    p.grid_a = tables.grid_a;
    p.grid_b = tables.grid_b;
    p.grid_entries = tables.grid_entries;
    p.grid_split = tables.grid_split;
    p.grid_dense = tables.grid_dense;
    p.grid_uniform = tables.grid_uniform;
    {
        /* one bit of a tie block mask per (4 << shift) scanned barcodes / grid entries: at most 32 bits */
        const int32_t scanned(p.grid != NULL ? p.grid_entries : p.barcode_cardinality);
        int32_t shift(0);
        while((((scanned + 3) >> 2) + (1 << shift) - 1) >> shift > 32) { ++shift; }
        p.tie_block_shift = shift;
    }
    /* the prefilter scan exists for the generic scan and for the dense forms of the combinatorial one (upload_grid
       builds a dense grid only for the separable form and the 8 + 8 and 10 + 10 shapes) */
    const bool prefilter(tables.fast.pointer != NULL && p.whitelist == NULL && (p.grid == NULL || p.grid_dense != 0));
    p.fast_barcodes = prefilter ? tables.fast.pointer : NULL;
    p.phred32 = h->device_phred32.pointer;
    p.fast_uniform_prior = 0.0f;
    if(prefilter && d.barcode_cardinality > 0) {
        bool uniform(true);
        for(int32_t b(1); b < d.barcode_cardinality && uniform; ++b) { uniform = d.concentration[b] == d.concentration[0]; }
        if(uniform && static_cast< float >(d.concentration[0]) > 0.0f) { p.fast_uniform_prior = static_cast< float >(d.concentration[0]); }
    }
}

void destroy(phq_handle* h) {
    if(h == NULL) { return; }
    if(h->device >= 0) { cudaSetDevice(h->device); }       /* its buffers, streams and events go on its own device */
    delete h;
}

/* launch the chain on device-resident planes (TranscodingDecoder::classify order, transcode.h:51-60) */
void launch_chain(phq_handle* h, int64_t n_reads, const phq_tile* tiles, uint8_t* qcfail, phq_result* const* results, phq_compact_result* const* compact,
                  DeviceBuffer< unsigned char >& tie_list, cudaStream_t stream) {
    const size_t n_decoders(h->chain.size());
    /* the PAMLD tie queue (80-byte records) and the MDD short-read queue (read indices) share one buffer:
       [16 bytes: counter][queue]; launches cover at most PAMLD_LAUNCH_READS reads so it stays bounded */
    bool needs_queue(false);
    for(size_t k(0); k < n_decoders; ++k) { needs_queue = needs_queue || h->chain[k].algorithm == PHQ_PAMLD || h->params[k].mdd_tables != NULL; }
    const long long queue_reads(n_reads < PAMLD_LAUNCH_READS ? n_reads : PAMLD_LAUNCH_READS);
    /* [16 bytes: counters][tie records][hard list of the prefilter scans: one int per read][candidate pool] */
    if(needs_queue) { tie_list.reserve(16 + static_cast< size_t >(queue_reads) * (sizeof(TieRecord) + sizeof(int) + TIE_POOL_PER_READ * sizeof(uint32_t))); }
    for(size_t k(0); k < n_decoders; ++k) {
        DecoderParams p(h->params[k]);
        p.totals = (k + 1 == n_decoders) ? h->totals() : NULL;
        if(tie_list.pointer != NULL) {
            p.tie_count = reinterpret_cast< unsigned* >(tie_list.pointer);
            p.tie_record = reinterpret_cast< TieRecord* >(tie_list.pointer + 16);
            p.hard_list = reinterpret_cast< int* >(tie_list.pointer + 16 + static_cast< size_t >(queue_reads) * sizeof(TieRecord));
            p.tie_pool = reinterpret_cast< uint32_t* >(p.hard_list + queue_reads);
            p.tie_pool_capacity = static_cast< uint32_t >(queue_reads * TIE_POOL_PER_READ);
        }
        TileArguments a;
        memset(&a, 0, sizeof(a));
        a.n_reads = n_reads;
        a.qcfail = qcfail;
        a.results = results != NULL ? results[k] : NULL;
        a.compact = compact != NULL ? compact[k] : NULL;
        a.quality_bits = 8;
        a.nucleotides = h->chain[k].nucleotide_cardinality;
        cudaError_t status(cudaSuccess);
        if(h->chain[k].tiled()) {
            if(tiles == NULL || tiles[k].bases == NULL || tiles[k].nmask == NULL || tiles[k].quality == NULL) {
                throw InternalError("decoder " + std::to_string(k) + " needs a tile");
            }
            if(tiles[k].pitch < n_reads) { throw InternalError("tile pitch is smaller than the number of reads"); }
            a.bases = tiles[k].bases;
            a.nmask = tiles[k].nmask;
            a.quality = tiles[k].quality;
            a.pitch = tiles[k].pitch;
            a.quality_bits = tiles[k].quality_bits == 0 ? 8 : tiles[k].quality_bits;
            if(a.quality_bits != 8 && a.quality_bits != 4 && a.quality_bits != 2) { throw InternalError("quality_bits must be 8, 4 or 2"); }
            memcpy(a.codebook, tiles[k].quality_codebook, 16);
            /* sub-launches over read ranges keep the queues bounded; planes are [word][read], so a range is a pointer offset */
            for(long long begin(0); begin < n_reads && status == cudaSuccess; begin += PAMLD_LAUNCH_READS) {
                TileArguments part(a);
                part.n_reads = (n_reads - begin) < PAMLD_LAUNCH_READS ? (n_reads - begin) : PAMLD_LAUNCH_READS;
                part.bases = a.bases + begin;
                part.nmask = a.nmask + begin;
                part.quality = a.quality + begin;
                part.qcfail = a.qcfail + begin;
                part.results = a.results != NULL ? a.results + begin : NULL;
                part.compact = a.compact != NULL ? a.compact + begin : NULL;
                if(h->chain[k].algorithm == PHQ_PAMLD) {
                    status = launch_pamld(p, part, h->geometry, stream);
                    h->kernel_launches += pamld_launches(p);
                } else {
                    status = launch_mdd(p, part, h->geometry, stream);
                    h->kernel_launches += p.mdd_tables != NULL ? 2 * MDD_KERNEL_LAUNCHES : MDD_KERNEL_LAUNCHES;
                }
            }
        } else {
            status = launch_count(p, a, h->geometry, stream);
            h->kernel_launches += COUNT_KERNEL_LAUNCHES;
        }
        PHQ_CUDA(status);
    }
}

/* a retry after a failure creates only what the failed call did not */
void ensure_slots(phq_handle* h) {
    const size_t n(h->chain.size());
    for(auto& s : h->slot) {
        if(s.stream == NULL) { PHQ_CUDA(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking)); }
        if(s.done == NULL) { PHQ_CUDA(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming)); }
        s.bases.resize(n); s.nmask.resize(n); s.quality.resize(n); s.results.resize(n);
    }
}

/*  The status of the exception in flight; its message goes where phq_last_error finds it: on the handle, or in the
    thread's global error without one. Call it from a catch(...) block. */
int record_error(phq_handle* h) {
    int status;
    std::string message;
    try { throw; }
    catch(const phq::Error& e) { status = e.code; message = e.what(); }
    catch(const JsonError& e) { status = PHQ_CONFIGURATION_ERROR; message = std::string("Configuration error : ") + e.what(); }
    catch(const std::bad_alloc&) { status = PHQ_OUT_OF_MEMORY_ERROR; message = "Out of memory error"; }
    catch(const std::exception& e) { status = PHQ_UNKNOWN_ERROR; message = e.what(); }
    (h != NULL ? h->error : global_error) = message;
    return status;
}

template < class F > int guarded(phq_handle* h, F body) {
    try {
        if(h == NULL) { throw InternalError("null handle"); }
        if(h->device < 0) { throw InternalError("this handle was created without a device (host-only); there is no CPU classification path"); }
        PHQ_CUDA(cudaSetDevice(h->device));
        body();
        return PHQ_OK;
    } catch(...) { return record_error(h); }
}

/* a handle whose accumulators hold the sums of all ranks must be reset before it accumulates again (phq_collect) */
void refuse_collected(const phq_handle* h) {
    if(h->collected) { throw InternalError("the accumulators of this handle were collected across ranks; phq_reset_accumulators before the next pass"); }
}
/* phq_compact_result carries the barcode index in 24 bits and the distance in 6 */
void require_compact_range(const phq_handle* h) {
    for(const auto& d : h->chain) {
        if(d.tiled() && d.barcode_cardinality >= 0xffffff) {
            throw ConfigurationError("a decoder with " + std::to_string(d.barcode_cardinality) + " barcodes does not fit the 24 bit index of phq_compact_result; use the phq_result forms");
        }
        if(d.tiled() && d.nucleotide_cardinality > 63) {
            throw ConfigurationError("a decoder of " + std::to_string(d.nucleotide_cardinality) + " nucleotides does not fit the 6 bit distance of phq_compact_result; use the phq_result forms");
        }
    }
}

/*  The host-buffer decode calls: reads [0, n_reads) in sub-batches rotating over the staging slots, so that one
    sub-batch's copies overlap another's kernels. On the slot's stream, per sub-batch: qcfail in, stage_tiles (fills
    the slot's tile buffers of every tiled decoder), the chain, after_chain, then results and qcfail out. Both steps
    take (slot, first read, reads, pitch of the slot buffers); stage_tiles also the device tiles, after_chain the
    device results. */
template < class StageTiles, class AfterChain >
void decode_staged(phq_handle* h, int64_t n_reads, bool tags, const uint8_t* qcfail_in, phq_result* const* results,
                   phq_compact_result* const* compact, uint8_t* qcfail_out, StageTiles stage_tiles, AfterChain after_chain) {
    refuse_collected(h);
    if(compact != NULL) { require_compact_range(h); }
    ensure_slots(h);
    const size_t n_decoders(h->chain.size());
    /* compact results take the 8-byte form on the device, unless the tag kernel reads them: it reads the 16-byte form */
    const bool compact_on_device(compact != NULL && !tags);
    const long long sub(n_reads < h->sub_batch_reads ? (n_reads > 0 ? n_reads : 1) : h->sub_batch_reads);
    int turn(0);
    for(long long begin(0); begin < n_reads; begin += sub, ++turn) {
        const long long count((n_reads - begin) < sub ? (n_reads - begin) : sub);
        StagingSlot& s(h->slot[turn % STAGING_SLOTS]);
        if(turn >= STAGING_SLOTS) { PHQ_CUDA(cudaEventSynchronize(s.done)); }
        s.qcfail.reserve(static_cast< size_t >(sub));
        if(qcfail_in != NULL) { PHQ_CUDA(cudaMemcpyAsync(s.qcfail.pointer, qcfail_in + begin, static_cast< size_t >(count), cudaMemcpyHostToDevice, s.stream)); }
        else { PHQ_CUDA(cudaMemsetAsync(s.qcfail.pointer, 0, static_cast< size_t >(count), s.stream)); }
        std::vector< phq_tile > device_tiles(n_decoders);
        std::vector< phq_result* > device_results(n_decoders, static_cast< phq_result* >(NULL));
        std::vector< phq_compact_result* > device_compact(n_decoders, static_cast< phq_compact_result* >(NULL));
        for(size_t k(0); k < n_decoders; ++k) {
            const DecoderSpec& d(h->chain[k]);
            if(d.tiled()) {
                s.bases[k].reserve(static_cast< size_t >(sub) * d.word_cardinality());
                s.nmask[k].reserve(static_cast< size_t >(sub) * d.word_cardinality());
                s.quality[k].reserve(static_cast< size_t >(sub) * d.quality_word_cardinality());
                device_tiles[k].bases = s.bases[k].pointer;
                device_tiles[k].nmask = s.nmask[k].pointer;
                device_tiles[k].quality = s.quality[k].pointer;
                device_tiles[k].pitch = sub;
            }
            if((results != NULL && results[k] != NULL) || (compact != NULL && compact[k] != NULL) || (tags && d.tiled())) {
                /* the staging buffer is sized for the 16-byte form and reused for the 8-byte one */
                s.results[k].reserve(static_cast< size_t >(sub));
                if(compact_on_device) { device_compact[k] = reinterpret_cast< phq_compact_result* >(s.results[k].pointer); }
                else { device_results[k] = s.results[k].pointer; }
            }
        }
        stage_tiles(s, begin, count, sub, device_tiles.data());
        launch_chain(h, count, device_tiles.data(), s.qcfail.pointer, device_results.data(), device_compact.data(), s.tie_list, s.stream);
        after_chain(s, begin, count, sub, device_results.data());
        for(size_t k(0); k < n_decoders; ++k) {
            if(device_results[k] != NULL && results != NULL && results[k] != NULL) {
                PHQ_CUDA(cudaMemcpyAsync(results[k] + begin, device_results[k], static_cast< size_t >(count) * sizeof(phq_result), cudaMemcpyDeviceToHost, s.stream));
            }
            if(device_compact[k] != NULL) {
                PHQ_CUDA(cudaMemcpyAsync(compact[k] + begin, device_compact[k], static_cast< size_t >(count) * sizeof(phq_compact_result), cudaMemcpyDeviceToHost, s.stream));
            }
        }
        if(qcfail_out != NULL) { PHQ_CUDA(cudaMemcpyAsync(qcfail_out + begin, s.qcfail.pointer, static_cast< size_t >(count), cudaMemcpyDeviceToHost, s.stream)); }
        PHQ_CUDA(cudaEventRecord(s.done, s.stream));
    }
    for(int i(0); i < STAGING_SLOTS && i < turn; ++i) { PHQ_CUDA(cudaStreamSynchronize(h->slot[i].stream)); }
}

/* for entry points that are pure host work and therefore also serve host-only handles */
template < class F > int guarded_host(phq_handle* h, F body) {
    try {
        if(h == NULL) { throw InternalError("null handle"); }
        body();
        return PHQ_OK;
    } catch(...) { return record_error(h); }
}

/* a malloc'd copy the caller releases with phq_free */
char* duplicate(const std::string& text) {
    char* out(static_cast< char* >(malloc(text.size() + 1)));
    if(out == NULL) { throw phq::Error(PHQ_OUT_OF_MEMORY_ERROR, "Out of memory error"); }
    memcpy(out, text.c_str(), text.size() + 1);
    return out;
}

}   /* namespace */

extern "C" {

const char* phq_last_global_error(void) { return global_error.c_str(); }
const char* phq_last_error(const phq_handle* handle) { return handle != NULL ? handle->error.c_str() : global_error.c_str(); }
void phq_free(void* pointer) { free(pointer); }

int phq_compile_job(const char* job_json, char** compiled_json) {
    try {
        if(job_json == NULL || compiled_json == NULL) { throw InternalError("null argument"); }
        Json compiled(compile_job(Json::parse(job_json)));
        *compiled_json = duplicate(compiled.dump(-1, 4));     /* shortest round-trip decimals: priors must survive the text form bit for bit */
        return PHQ_OK;
    } catch(...) { return record_error(NULL); }
}

int phq_load_job(const char* path, char** job_json) {
    if(path == NULL || job_json == NULL) { global_error = "Internal error : illegal argument"; return PHQ_INTERNAL_ERROR; }
    *job_json = NULL;
    try {
        std::set< std::string > visited;
        const Json job(load_job_with_import(path, visited));
        *job_json = duplicate(job.dump(-1, 4));
        return PHQ_OK;
    } catch(...) { return record_error(NULL); }
}

int phq_create(const char* compiled_job_json, int device, phq_handle** handle) {
    phq_handle* h(NULL);
    try {
        if(compiled_job_json == NULL || handle == NULL) { throw InternalError("null argument"); }
        *handle = NULL;
        const Json job(Json::parse(compiled_job_json));
        std::vector< DecoderSpec > chain(parse_compiled_job(job));
        for(const auto& d : chain) {
            /* candidate keys of the whitelist scan (owner lane << 27 | barcode) and of the tie pass (slot << 28 | barcode) */
            if(d.algorithm == PHQ_PAMLD && d.barcode_cardinality >= (1 << 27)) {
                throw ConfigurationError("a PAMLD codec holds at most 2^27 - 1 barcodes on this path, not " + std::to_string(d.barcode_cardinality));
            }
        }

        if(device < 0) {
            /* host-only handle: configuration, phq_pack and phq_decoder_describe work; anything that
               needs the GPU fails with an internal error. For feed threads and CPU-only tests. */
            h = new phq_handle();
            h->device = -1;
            h->job = job;
            h->chain = chain;
            h->scratch.resize(chain.size());
            for(size_t k(0); k < chain.size(); ++k) { h->scratch[k].resize(static_cast< size_t >(chain[k].segment_cardinality)); }
            *handle = h;
            return PHQ_OK;
        }
        int device_count(0);
        cudaError_t status(cudaGetDeviceCount(&device_count));
        if(status != cudaSuccess || device_count < 1) {
            throw InternalError(std::string("no usable CUDA device (") + cudaGetErrorString(status) + "); this path has no CPU fallback");
        }
        if(device < 0 || device >= device_count) { throw InternalError("device " + std::to_string(device) + " out of range"); }
        PHQ_CUDA(cudaSetDevice(device));
        cudaDeviceProp prop;
        PHQ_CUDA(cudaGetDeviceProperties(&prop, device));
        if(prop.major < 10) { throw InternalError(std::string("device ") + prop.name + " is not sm_100 class; this library is built for sm_100a only"); }

        h = new phq_handle();
        h->device = device;
        h->job = job;
        h->chain = chain;
        h->geometry.multiprocessor_count = prop.multiProcessorCount;
        h->geometry.shared_memory_per_block_optin = prop.sharedMemPerBlockOptin;
        const size_t n(chain.size());
        h->params.resize(n);
        h->tables.resize(n);
        h->scratch.resize(n);
        h->offset_u64.resize(n);
        h->offset_f64.resize(n);
        int64_t at_u(0), at_f(0);
        for(size_t k(0); k < n; ++k) {
            h->scratch[k].resize(static_cast< size_t >(chain[k].segment_cardinality));
            h->offset_u64[k] = at_u;
            h->offset_f64[k] = at_f;
            at_u += static_cast< int64_t >(chain[k].barcode_cardinality + 1) * ACC_U64_COLUMNS;
            at_f += static_cast< int64_t >(chain[k].barcode_cardinality + 1) * ACC_F64_COLUMNS;
        }
        h->n_u64 = at_u + 4;        /* + totals count, pf_count + diagnostics exact path, threshold band */
        h->n_f64 = at_f;
        h->device_accumulators.reserve(static_cast< size_t >(h->n_u64 + h->n_f64) * 8);
        PHQ_CUDA(cudaMemset(h->device_accumulators.pointer, 0, static_cast< size_t >(h->n_u64 + h->n_f64) * 8));

        std::vector< double > phred;
        double uniform_quality, base;
        assemble_phred(phred, uniform_quality, base);
        h->device_phred.upload(phred);
        {
            std::vector< float > ratio32(128);
            for(int q(0); q < 128; ++q) { ratio32[q] = static_cast< float >(phred[PHRED_MISMATCH_RATIO + q]); }
            h->device_phred32.upload(ratio32);
        }

        for(size_t k(0); k < n; ++k) {
            if(chain[k].tiled()) { build_tables(h, k); }
            refresh_params(h, k);
        }
        PHQ_CUDA(cudaEventCreate(&h->timing_start));
        PHQ_CUDA(cudaEventCreate(&h->timing_stop));
        PHQ_CUDA(prepare_kernels(h->geometry));
        *handle = h;
        return PHQ_OK;
    } catch(...) {
        const int status(record_error(NULL));
        destroy(h);
        return status;
    }
}

void phq_destroy(phq_handle* handle) { destroy(handle); }

int phq_decoder_count(const phq_handle* handle) { return handle != NULL ? static_cast< int >(handle->chain.size()) : 0; }

int phq_decoder_describe(const phq_handle* handle, int decoder, phq_decoder_info* info) {
    if(handle == NULL || info == NULL || decoder < 0 || decoder >= static_cast< int >(handle->chain.size())) {
        global_error = "Internal error : decoder index out of range";
        return PHQ_INTERNAL_ERROR;
    }
    const DecoderSpec& d(handle->chain[decoder]);
    memset(info, 0, sizeof(*info));
    info->algorithm = d.algorithm;
    info->topic = d.topic;
    info->index = d.index;
    info->barcode_cardinality = d.barcode_cardinality;
    info->segment_cardinality = d.segment_cardinality;
    info->nucleotide_cardinality = d.nucleotide_cardinality;
    for(int32_t s(0); s < d.segment_cardinality && s < PHQ_MAX_SEGMENTS; ++s) { info->segment_length[s] = d.segment_length[s]; }
    info->word_cardinality = d.word_cardinality();
    info->quality_word_cardinality = d.quality_word_cardinality();
    info->has_tile = d.tiled() ? 1 : 0;
    return PHQ_OK;
}

int phq_pack(phq_handle* handle, int64_t n_reads, int32_t n_input_segments,
             const uint8_t* const* code, const uint8_t* const* quality, const int64_t* const* offset,
             phq_tile* tiles) {
    return guarded_host(handle, [&]() {
        phq_handle* h(handle);
        if(n_reads < 0 || tiles == NULL) { throw InternalError("illegal argument"); }
        for(size_t k(0); k < h->chain.size(); ++k) {
            const DecoderSpec& d(h->chain[k]);
            if(!d.tiled()) { continue; }
            phq_tile& tile(tiles[k]);
            if(tile.bases == NULL || tile.nmask == NULL || tile.quality == NULL || tile.pitch < n_reads) { throw InternalError("decoder " + std::to_string(k) + " has no host tile to pack into"); }
            for(const auto& t : d.transform) {
                if(t.input_segment_index >= n_input_segments) {
                    throw ConfigurationError("invalid input feed reference " + std::to_string(t.input_segment_index) + " in token " + std::to_string(t.token_index));
                }
            }
            uint32_t* out_bases(const_cast< uint32_t* >(tile.bases));
            uint16_t* out_nmask(const_cast< uint16_t* >(tile.nmask));
            uint32_t* out_quality(const_cast< uint32_t* >(tile.quality));
            const int32_t words(d.word_cardinality());
            const int32_t quality_words(d.quality_word_cardinality());
            const bool stale_semantics(d.algorithm == PHQ_PAMLD);
            const int64_t pitch(tile.pitch);

            /* reads [begin, end) in order on top of `scratch`; returns whether any of them was short (an observed segment
               shorter than the barcode segment), which is when a read's tile depends on the reads before it */
            auto pack_range = [&](int64_t begin, int64_t end, std::vector< ScratchSegment >& scratch, bool* seen) -> bool {
                bool any_short(false);
                for(int64_t r(begin); r < end; ++r) {
                    /* Observation::clear + Rule::apply (sequence.h:296-300, transform.h:142-169) */
                    for(auto& sg : scratch) { sg.length = 0; sg.code[0] = 0; sg.quality[0] = 0; }
                    for(const auto& t : d.transform) {
                        const int64_t from(offset[t.input_segment_index][r]);
                        const int32_t from_length(static_cast< int32_t >(offset[t.input_segment_index][r + 1] - from));
                        const uint8_t* from_code(code[t.input_segment_index] + from);
                        const uint8_t* from_quality(quality[t.input_segment_index] + from);
                        ScratchSegment& to(scratch[t.output_segment_index]);
                        const int32_t start(t.absolute_start(from_length));
                        const int32_t end_of_token(t.absolute_end(from_length));
                        const int32_t size(end_of_token - start);
                        if(size > 0) {
                            if(to.length + size + 1 > static_cast< int32_t >(to.code.size())) { throw SequenceError("token extracts more nucleotides than the barcode segment holds"); }
                            if(!t.reverse_complement) {
                                memcpy(to.code.data() + to.length, from_code + start, size);
                                memcpy(to.quality.data() + to.length, from_quality + start, size);
                            } else {
                                for(int32_t i(0); i < size; ++i) {
                                    to.code[to.length + i] = BAM_REVERSE_COMPLEMENT[from_code[end_of_token - i - 1] & 0xf];
                                    to.quality[to.length + i] = from_quality[end_of_token - i - 1];
                                }
                            }
                            to.length += size;
                            to.code[to.length] = 0;
                            to.quality[to.length] = 0;
                        }
                    }
                    /* 2-bit planes + ambiguity mask + Phred bytes */
                    uint64_t lo(0), hi(0), ambiguous(0);
                    uint8_t phred[PHQ_MAX_NUCLEOTIDES];
                    memset(phred, 0, sizeof(phred));
                    for(int32_t sgm(0); sgm < d.segment_cardinality; ++sgm) {
                        const ScratchSegment& from(scratch[sgm]);
                        any_short = any_short || from.length < d.segment_length[sgm];
                        for(int32_t i(0); i < d.segment_length[sgm]; ++i) {
                            const int32_t j(d.segment_offset[sgm] + i);
                            if(!stale_semantics && i >= from.length) {
                                /* Sequence::distance_from stops at the observed length: the position is absent, marked as
                                   an ambiguous position whose base bits are both set (a real ambiguous base has them clear),
                                   quality PHQ_ABSENT_QUALITY */
                                phred[j] = PHQ_ABSENT_QUALITY;
                                lo |= static_cast< uint64_t >(1) << j;
                                hi |= static_cast< uint64_t >(1) << j;
                                ambiguous |= static_cast< uint64_t >(1) << j;
                                continue;
                            }
                            /* PAMLD reads the expected length: terminator, then stale bytes (barcode.h:150) */
                            const uint8_t c(from.code[i]);
                            const uint64_t bit(static_cast< uint64_t >(1) << j);
                            switch(c) {
                                case 1: break;
                                case 2: lo |= bit; break;
                                case 4: hi |= bit; break;
                                case 8: lo |= bit; hi |= bit; break;
                                default: ambiguous |= bit; break;
                            }
                            phred[j] = from.quality[i];
                        }
                    }
                    for(int32_t w(0); w < words; ++w) {
                        out_bases[w * pitch + r] = static_cast< uint32_t >((lo >> (16 * w)) & 0xffffu) | (static_cast< uint32_t >((hi >> (16 * w)) & 0xffffu) << 16);
                        out_nmask[w * pitch + r] = static_cast< uint16_t >((ambiguous >> (16 * w)) & 0xffffu);
                    }
                    for(int32_t w(0); w < quality_words; ++w) {
                        out_quality[w * pitch + r] = static_cast< uint32_t >(phred[4 * w]) | (static_cast< uint32_t >(phred[4 * w + 1]) << 8)
                            | (static_cast< uint32_t >(phred[4 * w + 2]) << 16) | (static_cast< uint32_t >(phred[4 * w + 3]) << 24);
                    }
                    for(int32_t j(0); j < d.nucleotide_cardinality; ++j) { seen[phred[j]] = true; }
                }
                return any_short;
            };

            bool seen[256];
            memset(seen, 0, sizeof(seen));
            /*  A read's tile only depends on the reads before it when some read is short (the stale bytes of the
                reference's Observation, barcode.h:150). Large batches are therefore packed by several threads on
                private Observations; if any of them meets a short read the batch is packed again in order. */
            const int workers(pack_workers(n_reads));
            bool in_order(workers <= 1);
            if(!in_order) {
                std::vector< std::vector< ScratchSegment > > private_scratch(static_cast< size_t >(workers), h->scratch[k]);
                std::vector< std::array< bool, 256 > > private_seen(static_cast< size_t >(workers));
                std::vector< char > met_short(static_cast< size_t >(workers), 0);
                std::vector< std::exception_ptr > failure(static_cast< size_t >(workers));
                std::vector< std::thread > pool;
                for(int w(0); w < workers; ++w) {
                    private_seen[w].fill(false);
                    pool.emplace_back([&, w]() {
                        try {
                            met_short[w] = pack_range(n_reads * w / workers, n_reads * (w + 1) / workers, private_scratch[w], private_seen[w].data()) ? 1 : 0;
                        } catch(...) { failure[w] = std::current_exception(); }
                    });
                }
                for(auto& t : pool) { t.join(); }
                for(int w(0); w < workers; ++w) { if(failure[w]) { std::rethrow_exception(failure[w]); } }
                for(int w(0); w < workers; ++w) { in_order = in_order || met_short[w] != 0; }
                if(!in_order) {
                    for(int w(0); w < workers; ++w) { for(int v(0); v < 256; ++v) { seen[v] = seen[v] || private_seen[w][v]; } }
                    h->scratch[k] = private_scratch[static_cast< size_t >(workers) - 1];       /* full length reads: the last one's Observation */
                }
            }
            if(in_order) {
                memset(seen, 0, sizeof(seen));
                pack_range(0, n_reads, h->scratch[k], seen);
            }
            /* quality form: Phred bytes as written above, or indices into a codebook of the distinct values */
            int32_t wanted(tile.quality_bits);
            int32_t distinct(0);
            uint8_t codebook[256];
            uint8_t index_of[256];
            memset(index_of, 0, sizeof(index_of));
            for(int v(0); v < 256; ++v) { if(seen[v]) { index_of[v] = static_cast< uint8_t >(distinct); codebook[distinct++] = static_cast< uint8_t >(v); } }
            if(wanted == -1) { wanted = distinct <= 4 ? 2 : (distinct <= 16 ? 4 : 8); }
            if(wanted == 0) { wanted = 8; }
            if(wanted != 8 && wanted != 4 && wanted != 2) { throw ConfigurationError("quality_bits must be -1, 0, 2, 4 or 8"); }
            if(wanted != 8 && distinct > (1 << wanted)) {
                throw ConfigurationError(std::to_string(distinct) + " distinct quality values do not fit " + std::to_string(wanted) + " bit indices");
            }
            memset(tile.quality_codebook, 0, sizeof(tile.quality_codebook));
            if(wanted != 8) {
                memcpy(tile.quality_codebook, codebook, static_cast< size_t >(distinct));
                const int32_t per_word(32 / wanted);
                const int32_t packed_words((d.nucleotide_cardinality * wanted + 31) / 32);
                auto encode_range = [&](int64_t begin, int64_t end) {
                    for(int64_t r(begin); r < end; ++r) {
                        uint32_t packed[PHQ_MAX_NUCLEOTIDES / 4];
                        memset(packed, 0, sizeof(packed));
                        for(int32_t j(0); j < d.nucleotide_cardinality; ++j) {
                            const uint8_t q(static_cast< uint8_t >((out_quality[(j >> 2) * tile.pitch + r] >> (8 * (j & 3))) & 0xffu));
                            packed[j / per_word] |= static_cast< uint32_t >(index_of[q]) << (wanted * (j % per_word));
                        }
                        for(int32_t w(0); w < packed_words; ++w) { out_quality[w * tile.pitch + r] = packed[w]; }
                    }
                };
                if(workers <= 1) { encode_range(0, n_reads); }
                else {
                    std::vector< std::thread > pool;
                    for(int w(0); w < workers; ++w) { pool.emplace_back(encode_range, n_reads * w / workers, n_reads * (w + 1) / workers); }
                    for(auto& t : pool) { t.join(); }
                }
            }
            tile.quality_bits = wanted;
        }
    });
}

static int decode_device(phq_handle* handle, int64_t n_reads, const phq_tile* device_tiles, uint8_t* device_qcfail,
                         phq_result* const* device_results, phq_compact_result* const* device_compact, void* stream) {
    return guarded(handle, [&]() {
        if(n_reads < 0 || n_reads > 0x7fffffffll) { throw OverflowError("a batch holds at most 2^31 - 1 reads"); }
        if(device_qcfail == NULL) { throw InternalError("device_qcfail is required"); }
        refuse_collected(handle);
        if(device_compact != NULL) { require_compact_range(handle); }
        cudaStream_t s(static_cast< cudaStream_t >(stream));
        PHQ_CUDA(cudaEventRecord(handle->timing_start, s));
        launch_chain(handle, n_reads, device_tiles, device_qcfail, device_results, device_compact, handle->tie_list, s);
        PHQ_CUDA(cudaEventRecord(handle->timing_stop, s));
        handle->timing_stream = s;
        handle->timing_valid = true;
    });
}
int phq_decode_batch_device(phq_handle* handle, int64_t n_reads, const phq_tile* device_tiles,
                            uint8_t* device_qcfail, phq_result* const* device_results, void* stream) {
    return decode_device(handle, n_reads, device_tiles, device_qcfail, device_results, NULL, stream);
}
int phq_decode_batch_device_compact(phq_handle* handle, int64_t n_reads, const phq_tile* device_tiles,
                                    uint8_t* device_qcfail, phq_compact_result* const* device_compact, void* stream) {
    return decode_device(handle, n_reads, device_tiles, device_qcfail, NULL, device_compact, stream);
}

static int decode_host(phq_handle* handle, int64_t n_reads, const phq_tile* tiles, const uint8_t* qcfail_in,
                       phq_result* const* results, phq_compact_result* const* compact, uint8_t* qcfail_out) {
    return guarded(handle, [&]() {
        phq_handle* h(handle);
        if(n_reads < 0) { throw InternalError("illegal read count"); }
        auto copy_tiles = [&](StagingSlot& s, long long begin, long long count, long long sub, phq_tile* device_tiles) {
            for(size_t k(0); k < h->chain.size(); ++k) {
                const DecoderSpec& d(h->chain[k]);
                if(!d.tiled()) { continue; }
                if(tiles == NULL || tiles[k].bases == NULL) { throw InternalError("decoder " + std::to_string(k) + " needs a tile"); }
                const int32_t words(d.word_cardinality());
                const int32_t bits(tiles[k].quality_bits == 0 ? 8 : tiles[k].quality_bits);
                /* only the rows the chosen quality form occupies travel */
                const int32_t quality_words((d.nucleotide_cardinality * bits + 31) / 32);
                PHQ_CUDA(cudaMemcpy2DAsync(s.bases[k].pointer, static_cast< size_t >(sub) * 4, tiles[k].bases + begin, static_cast< size_t >(tiles[k].pitch) * 4,
                                           static_cast< size_t >(count) * 4, words, cudaMemcpyHostToDevice, s.stream));
                PHQ_CUDA(cudaMemcpy2DAsync(s.nmask[k].pointer, static_cast< size_t >(sub) * 2, tiles[k].nmask + begin, static_cast< size_t >(tiles[k].pitch) * 2,
                                           static_cast< size_t >(count) * 2, words, cudaMemcpyHostToDevice, s.stream));
                PHQ_CUDA(cudaMemcpy2DAsync(s.quality[k].pointer, static_cast< size_t >(sub) * 4, tiles[k].quality + begin, static_cast< size_t >(tiles[k].pitch) * 4,
                                           static_cast< size_t >(count) * 4, quality_words, cudaMemcpyHostToDevice, s.stream));
                device_tiles[k].quality_bits = tiles[k].quality_bits;
                memcpy(device_tiles[k].quality_codebook, tiles[k].quality_codebook, sizeof(tiles[k].quality_codebook));
            }
        };
        decode_staged(h, n_reads, false, qcfail_in, results, compact, qcfail_out, copy_tiles, [](auto&&...) {});
    });
}
int phq_decode_batch(phq_handle* handle, int64_t n_reads, const phq_tile* tiles,
                     const uint8_t* qcfail_in, phq_result* const* results, uint8_t* qcfail_out) {
    return decode_host(handle, n_reads, tiles, qcfail_in, results, NULL, qcfail_out);
}
int phq_decode_batch_compact(phq_handle* handle, int64_t n_reads, const phq_tile* tiles,
                             const uint8_t* qcfail_in, phq_compact_result* const* compact_results) {
    return decode_host(handle, n_reads, tiles, qcfail_in, NULL, compact_results, NULL);
}

/* ------------------------------------------------------------------ feed bytes in: pack on the device (pack.cuh) */
namespace {

/* host mirror of the kernel's view of one read of one output segment, for the state the Observation is left in */
struct RawReader {
    const DecoderSpec& d;
    const phq_raw_segment* segments;
    int32_t phred_offset;
    bool bam_input;
    int64_t begin(int32_t i, int64_t r) const { return segments[i].offset != NULL ? segments[i].offset[r] : r * segments[i].length; }
    int32_t length(int32_t i, int64_t r) const { return segments[i].offset != NULL ? static_cast< int32_t >(segments[i].offset[r + 1] - segments[i].offset[r]) : static_cast< int32_t >(segments[i].length); }
    int32_t observed_length(int64_t r, int32_t s) const {
        int32_t total(0);
        for(const auto& t : d.transform) {
            if(t.output_segment_index != s) { continue; }
            const int32_t n(length(t.input_segment_index, r));
            const int32_t size(t.absolute_end(n) - t.absolute_start(n));
            total += size > 0 ? size : 0;
        }
        return total;
    }
    void fetch(int64_t r, int32_t s, int32_t i, uint8_t& code, uint8_t& quality) const {
        int32_t at(0);
        for(const auto& t : d.transform) {
            if(t.output_segment_index != s) { continue; }
            const int32_t n(length(t.input_segment_index, r));
            const int32_t start(t.absolute_start(n)), end(t.absolute_end(n));
            const int32_t size(end - start);
            if(size <= 0) { continue; }
            if(i < at + size) {
                const int64_t source(begin(t.input_segment_index, r) + (t.reverse_complement ? (end - (i - at) - 1) : (start + (i - at))));
                code = bam_input ? static_cast< uint8_t >(segments[t.input_segment_index].sequence[source] & 0xf) : ascii_to_bam(segments[t.input_segment_index].sequence[source]);
                if(t.reverse_complement) { code = BAM_REVERSE_COMPLEMENT[code & 0xf]; }
                quality = static_cast< uint8_t >(segments[t.input_segment_index].quality[source] - phred_offset);
                return;
            }
            at += size;
        }
    }
    /* the Observation after reads [0, r_last] on top of `scratch` (the state before read 0); r_last = -1 keeps scratch */
    void state_after(int64_t r_last, const std::vector< ScratchSegment >& scratch, uint8_t* code, uint8_t* quality) const {
        for(int32_t s(0); s < d.segment_cardinality; ++s) {
            for(int32_t i(0); i < d.segment_length[s]; ++i) {
                const int32_t j(d.segment_offset[s] + i);
                code[j] = scratch[s].code[i];
                quality[j] = scratch[s].quality[i];
                for(int64_t r(r_last); r >= 0; --r) {
                    const int32_t reach(observed_length(r, s));
                    if(reach == i) { code[j] = 0; quality[j] = 0; break; }
                    if(reach > i) { fetch(r, s, i, code[j], quality[j]); break; }
                }
            }
        }
    }
};

/* bytes one read's auxiliary record can take: every tag of every topic at its longest (Auxiliary::encode, auxiliary.cpp:320-361) */
int32_t tag_record_bytes(const phq_handle* h) {
    int32_t bytes(0);
    for(int topic(0); topic < 3; ++topic) {
        int32_t raw(0), corrected(0);
        bool present(false), probabilistic(false);
        for(const auto& d : h->chain) {
            if(d.topic != topic) { continue; }
            present = true;
            if(!d.transform.empty()) { raw += d.nucleotide_cardinality; }
            if(d.tiled()) { corrected += d.nucleotide_cardinality; }
            probabilistic = probabilistic || d.algorithm == PHQ_PAMLD;
        }
        if(!present) { continue; }
        if(topic == PHQ_SAMPLE) { bytes += 3 + h->read_group_longest + 1; }
        if(raw > 0) { bytes += 2 * (3 + raw + 1); }
        if(corrected > 0 && topic != PHQ_SAMPLE) { bytes += (topic == PHQ_MOLECULAR ? 2 : 1) * (3 + corrected + 1); }
        if(probabilistic) { bytes += 3 + 4; }
    }
    return (bytes + 15) / 16 * 16;
}

/* the longest read group ID of the sample decoder (decode_tag_id_by_index, classifier.cpp:79-98): host only */
int32_t host_read_group_longest(const phq_handle* h) {
    int32_t longest(0);
    const Json* element(h->job.find("sample"));
    if(element == NULL || !element->is_object()) { return 0; }
    auto measure = [&](const Json* record) {
        if(record != NULL && record->is_object()) {
            const int32_t length(static_cast< int32_t >(get_string(*record, "ID").size()));
            if(length > longest) { longest = length; }
        }
    };
    measure(element->find("undetermined"));
    const Json* codec(element->find("codec"));
    if(codec != NULL && codec->is_object()) { for(const auto& record : codec->members()) { measure(&record.second); } }
    return longest;
}

/* device tables of the tag kernel: barcode codes by index (row 0 = undetermined) and the read group IDs */
void ensure_tags(phq_handle* h) {
    if(h->tags_ready) { return; }
    const char* name[3] = { "sample", "molecular", "cellular" };
    for(size_t k(0); k < h->chain.size(); ++k) {
        const DecoderSpec& d(h->chain[k]);
        if(!d.tiled()) { continue; }
        const size_t L(static_cast< size_t >(d.nucleotide_cardinality));
        std::vector< uint8_t > table((static_cast< size_t >(d.barcode_cardinality) + 1) * L, 0);
        memcpy(table.data() + L, d.barcode.data(), static_cast< size_t >(d.barcode_cardinality) * L);
        h->tables[k].barcode_code.upload(table, 1);
        if(d.topic == PHQ_SAMPLE) {
            /* decode_tag_id_by_index (classifier.h): the ID of the undetermined element, then of every barcode by index */
            const Json* element(h->job.find(name[0]));
            std::vector< int32_t > offset(1, 0);
            std::string text;
            auto push = [&](const Json* record) {
                if(record != NULL && record->is_object()) { text += get_string(*record, "ID"); }
                offset.push_back(static_cast< int32_t >(text.size()));
                const int32_t length(offset[offset.size() - 1] - offset[offset.size() - 2]);
                if(length > h->read_group_longest) { h->read_group_longest = length; }
            };
            push(element != NULL ? element->find("undetermined") : NULL);
            const Json* codec(element != NULL ? element->find("codec") : NULL);
            for(const auto& key : d.barcode_key) { push(codec != NULL ? codec->find(key) : NULL); }
            h->device_read_group_text.upload(std::vector< uint8_t >(text.begin(), text.end()), 1);
            h->device_read_group_offset.upload(offset);
        }
    }
    h->tags_ready = true;
}

/* a token in the form the pack and tag kernels read */
PackToken pack_token(const TransformSpec& t) {
    PackToken to;
    to.input_segment = t.input_segment_index; to.start = t.start; to.end = t.end; to.end_terminated = t.end_terminated ? 1 : 0;
    to.output_segment = t.output_segment_index; to.reverse_complement = t.reverse_complement ? 1 : 0;
    return to;
}

int decode_raw(phq_handle* handle, int64_t n_reads, int32_t n_input_segments, const phq_raw_segment* segments, int32_t phred_offset,
               const uint8_t* qcfail_in, phq_result* const* results, phq_compact_result* const* compact, uint8_t* qcfail_out,
               uint8_t* aux = NULL, int32_t* aux_length = NULL, int32_t aux_stride = 0, bool bam_input = false) {
    return guarded(handle, [&]() {
        phq_handle* h(handle);
        const bool tags(aux != NULL);
        if(tags) {
            if(aux_length == NULL) { throw InternalError("illegal argument"); }
            if(h->chain.size() > static_cast< size_t >(TAG_MAX_DECODERS)) { throw ConfigurationError("more than " + std::to_string(TAG_MAX_DECODERS) + " decoders are not supported by the tag path"); }
            ensure_tags(h);
            if(aux_stride < tag_record_bytes(h) || aux_stride % 4 != 0) { throw ConfigurationError("auxiliary record stride must be a multiple of 4 and at least " + std::to_string(tag_record_bytes(h))); }
        }
        if(n_reads < 0 || n_input_segments < 0 || (n_input_segments > 0 && segments == NULL)) { throw InternalError("illegal argument"); }
        if(n_input_segments > PACK_MAX_INPUT_SEGMENTS) { throw ConfigurationError("more than " + std::to_string(PACK_MAX_INPUT_SEGMENTS) + " input segments are not supported on this path"); }
        const size_t n_decoders(h->chain.size());
        std::vector< bool > used(static_cast< size_t >(n_input_segments), false);
        for(size_t k(0); k < n_decoders; ++k) {
            const DecoderSpec& d(h->chain[k]);
            if(!d.tiled() && !(tags && !d.transform.empty())) { continue; }
            if(tags && d.transform.size() > static_cast< size_t >(TAG_MAX_TOKENS)) { throw ConfigurationError("more than " + std::to_string(TAG_MAX_TOKENS) + " tokens per decoder are not supported by the tag path"); }
            if(d.transform.size() > static_cast< size_t >(PACK_MAX_TOKENS)) { throw ConfigurationError("more than " + std::to_string(PACK_MAX_TOKENS) + " tokens per decoder are not supported on this path"); }
            for(const auto& t : d.transform) {
                if(t.input_segment_index >= n_input_segments) {
                    throw ConfigurationError("invalid input feed reference " + std::to_string(t.input_segment_index) + " in token " + std::to_string(t.token_index));
                }
                used[static_cast< size_t >(t.input_segment_index)] = true;
            }
        }
        for(int32_t i(0); i < n_input_segments; ++i) {
            if(used[i] && (segments[i].sequence == NULL || segments[i].quality == NULL || (segments[i].offset == NULL && segments[i].length < 0))) {
                throw InternalError("input segment " + std::to_string(i) + " has no bytes");
            }
        }
        /* the bytes of the current sub-batch's reads, as they sit in the feed buffers: filled by upload_and_pack, read by the tag step */
        RawSegmentView view[PACK_MAX_INPUT_SEGMENTS];
        auto upload_and_pack = [&](StagingSlot& s, long long begin, long long count, long long sub, phq_tile*) {
            s.raw_sequence.resize(static_cast< size_t >(n_input_segments));
            s.raw_quality.resize(static_cast< size_t >(n_input_segments));
            s.raw_offset.resize(static_cast< size_t >(n_input_segments));
            memset(view, 0, sizeof(view));
            for(int32_t i(0); i < n_input_segments; ++i) {
                if(!used[i]) { continue; }
                const phq_raw_segment& g(segments[i]);
                const int64_t first_byte(g.offset != NULL ? g.offset[begin] : begin * g.length);
                const int64_t last_byte(g.offset != NULL ? g.offset[begin + count] : (begin + count) * g.length);
                const size_t bytes(static_cast< size_t >(last_byte - first_byte));
                s.raw_sequence[i].reserve(bytes ? bytes : 1);
                s.raw_quality[i].reserve(bytes ? bytes : 1);
                if(bytes) {
                    PHQ_CUDA(cudaMemcpyAsync(s.raw_sequence[i].pointer, g.sequence + first_byte, bytes, cudaMemcpyHostToDevice, s.stream));
                    PHQ_CUDA(cudaMemcpyAsync(s.raw_quality[i].pointer, g.quality + first_byte, bytes, cudaMemcpyHostToDevice, s.stream));
                }
                view[i].sequence = s.raw_sequence[i].pointer - first_byte;
                view[i].quality = s.raw_quality[i].pointer - first_byte;
                view[i].length = g.length;
                view[i].first = 0;
                if(g.offset != NULL) {
                    s.raw_offset[i].reserve(static_cast< size_t >(sub) + 1);
                    PHQ_CUDA(cudaMemcpyAsync(s.raw_offset[i].pointer, g.offset + begin, static_cast< size_t >(count + 1) * sizeof(long long), cudaMemcpyHostToDevice, s.stream));
                    view[i].offset = s.raw_offset[i].pointer;
                } else {
                    view[i].first = begin;      /* r * length is absolute like the offsets */
                }
            }
            for(size_t k(0); k < n_decoders; ++k) {
                const DecoderSpec& d(h->chain[k]);
                if(!d.tiled()) { continue; }
                PackPlan plan;
                memset(&plan, 0, sizeof(plan));
                plan.token_cardinality = static_cast< int32_t >(d.transform.size());
                plan.segment_cardinality = d.segment_cardinality;
                plan.nucleotide_cardinality = d.nucleotide_cardinality;
                plan.stale_semantics = d.algorithm == PHQ_PAMLD ? 1 : 0;
                plan.phred_offset = phred_offset;
                plan.bam_input = bam_input ? 1 : 0;
                for(int32_t i(0); i <= d.segment_cardinality; ++i) { plan.segment_offset[i] = d.segment_offset[i]; }
                for(size_t i(0); i < d.transform.size(); ++i) { plan.token[i] = pack_token(d.transform[i]); }
                memcpy(plan.input, view, sizeof(view));
                if(plan.stale_semantics) {
                    const RawReader reader{ d, segments, phred_offset, bam_input };
                    reader.state_after(begin - 1, h->scratch[k], plan.carry_code, plan.carry_quality);
                }
                PHQ_CUDA(launch_pack(plan, count, s.bases[k].pointer, s.nmask[k].pointer, s.quality[k].pointer, sub, h->geometry.multiprocessor_count, s.stream));
                h->kernel_launches += 1;
            }
        };
        auto synthesize_tags = [&](StagingSlot& s, long long begin, long long count, long long sub, phq_result* const* device_results) {
            if(!tags) { return; }
            TagPlan plan;
            memset(&plan, 0, sizeof(plan));
            plan.decoder_cardinality = static_cast< int32_t >(n_decoders);
            plan.phred_offset = phred_offset;
            plan.bam_input = bam_input ? 1 : 0;
            plan.stride = aux_stride;
            plan.read_group_text = h->device_read_group_text.pointer;
            plan.read_group_offset = h->device_read_group_offset.pointer;
            memcpy(plan.input, view, sizeof(view));
            for(size_t k(0); k < n_decoders; ++k) {
                const DecoderSpec& d(h->chain[k]);
                TagDecoder& to(plan.decoder[k]);
                to.topic = d.topic;
                to.algorithm = d.algorithm;
                to.corrected_quality = d.corrected_quality;
                to.token_cardinality = static_cast< int32_t >(d.transform.size());
                to.segment_cardinality = d.transform.empty() ? 0 : d.segment_cardinality;
                to.nucleotide_cardinality = d.nucleotide_cardinality;
                for(int32_t i(0); i <= d.segment_cardinality && i <= PHQ_MAX_SEGMENTS && !d.transform.empty(); ++i) { to.segment_offset[i] = d.segment_offset[i]; }
                for(size_t i(0); i < d.transform.size(); ++i) { to.token[i] = pack_token(d.transform[i]); }
                to.results = d.tiled() ? device_results[k] : NULL;
                to.barcode_code = h->tables[k].barcode_code.pointer;
            }
            s.aux.reserve(static_cast< size_t >(sub) * aux_stride);
            s.aux_length.reserve(static_cast< size_t >(sub));
            PHQ_CUDA(launch_tags(plan, count, s.aux.pointer, s.aux_length.pointer, h->geometry.multiprocessor_count, s.stream));
            h->kernel_launches += 1;
            PHQ_CUDA(cudaMemcpyAsync(aux + begin * aux_stride, s.aux.pointer, static_cast< size_t >(count) * aux_stride, cudaMemcpyDeviceToHost, s.stream));
            PHQ_CUDA(cudaMemcpyAsync(aux_length + begin, s.aux_length.pointer, static_cast< size_t >(count) * sizeof(int32_t), cudaMemcpyDeviceToHost, s.stream));
        };
        decode_staged(h, n_reads, tags, qcfail_in, results, compact, qcfail_out, upload_and_pack, synthesize_tags);
        /* leave the Observations as a single reference thread would: later calls (raw or phq_pack) continue from here */
        for(size_t k(0); k < n_decoders && n_reads > 0; ++k) {
            const DecoderSpec& d(h->chain[k]);
            if(!d.tiled() || d.algorithm != PHQ_PAMLD) { continue; }
            uint8_t code[PHQ_MAX_NUCLEOTIDES], quality[PHQ_MAX_NUCLEOTIDES];
            const RawReader reader{ d, segments, phred_offset, bam_input };
            reader.state_after(n_reads - 1, h->scratch[k], code, quality);
            for(int32_t sgm(0); sgm < d.segment_cardinality; ++sgm) {
                for(int32_t i(0); i < d.segment_length[sgm]; ++i) {
                    h->scratch[k][sgm].code[i] = code[d.segment_offset[sgm] + i];
                    h->scratch[k][sgm].quality[i] = quality[d.segment_offset[sgm] + i];
                }
            }
        }
    });
}

}   /* namespace */

int phq_decode_batch_raw(phq_handle* handle, int64_t n_reads, int32_t n_input_segments, const phq_raw_segment* segments, int32_t phred_offset,
                         const uint8_t* qcfail_in, phq_result* const* results, uint8_t* qcfail_out) {
    return decode_raw(handle, n_reads, n_input_segments, segments, phred_offset, qcfail_in, results, NULL, qcfail_out);
}
int phq_decode_batch_raw_compact(phq_handle* handle, int64_t n_reads, int32_t n_input_segments, const phq_raw_segment* segments, int32_t phred_offset,
                                 const uint8_t* qcfail_in, phq_compact_result* const* compact_results) {
    return decode_raw(handle, n_reads, n_input_segments, segments, phred_offset, qcfail_in, NULL, compact_results, NULL);
}

int phq_tag_record_bytes(phq_handle* handle, int32_t* bytes) {
    return guarded_host(handle, [&]() {           /* pure host work: also answers for a host-only handle */
        if(bytes == NULL) { throw InternalError("illegal argument"); }
        if(!handle->tags_ready) {
            const int32_t longest(host_read_group_longest(handle));
            if(longest > handle->read_group_longest) { handle->read_group_longest = longest; }
        }
        *bytes = tag_record_bytes(handle);
    });
}
int phq_decode_batch_raw_tags(phq_handle* handle, int64_t n_reads, int32_t n_input_segments, const phq_raw_segment* segments, int32_t phred_offset,
                              const uint8_t* qcfail_in, uint8_t* aux, int32_t aux_stride, int32_t* aux_length, uint8_t* qcfail_out, phq_result* const* results) {
    if(aux == NULL) { return PHQ_INTERNAL_ERROR; }
    return decode_raw(handle, n_reads, n_input_segments, segments, phred_offset, qcfail_in, results, NULL, qcfail_out, aux, aux_length, aux_stride);
}

/* the same three calls over the reference's own in-memory form of a segment (sequence.h:264-300): BAM codes, Phred bytes */
int phq_decode_batch_bam(phq_handle* handle, int64_t n_reads, int32_t n_input_segments, const phq_raw_segment* segments,
                         const uint8_t* qcfail_in, phq_result* const* results, uint8_t* qcfail_out) {
    return decode_raw(handle, n_reads, n_input_segments, segments, 0, qcfail_in, results, NULL, qcfail_out, NULL, NULL, 0, true);
}
int phq_decode_batch_bam_compact(phq_handle* handle, int64_t n_reads, int32_t n_input_segments, const phq_raw_segment* segments,
                                 const uint8_t* qcfail_in, phq_compact_result* const* compact_results) {
    return decode_raw(handle, n_reads, n_input_segments, segments, 0, qcfail_in, NULL, compact_results, NULL, NULL, NULL, 0, true);
}
int phq_decode_batch_bam_tags(phq_handle* handle, int64_t n_reads, int32_t n_input_segments, const phq_raw_segment* segments,
                              const uint8_t* qcfail_in, uint8_t* aux, int32_t aux_stride, int32_t* aux_length, uint8_t* qcfail_out, phq_result* const* results) {
    if(aux == NULL) { return PHQ_INTERNAL_ERROR; }
    return decode_raw(handle, n_reads, n_input_segments, segments, 0, qcfail_in, results, NULL, qcfail_out, aux, aux_length, aux_stride, true);
}

int phq_host_alloc(void** pointer, size_t bytes) {
    if(pointer == NULL) { return PHQ_INTERNAL_ERROR; }
    cudaError_t status(cudaHostAlloc(pointer, bytes ? bytes : 1, cudaHostAllocDefault));
    if(status != cudaSuccess) {
        global_error = std::string("Out of memory error : ") + cudaGetErrorString(status);
        return PHQ_OUT_OF_MEMORY_ERROR;
    }
    return PHQ_OK;
}
void phq_host_free(void* pointer) { if(pointer != NULL) { cudaFreeHost(pointer); } }

int phq_accumulators(phq_handle* handle, int decoder, uint64_t* u64_table, double* f64_table) {
    return guarded(handle, [&]() {
        if(decoder < 0 || decoder >= static_cast< int >(handle->chain.size())) { throw InternalError("decoder index out of range"); }
        PHQ_CUDA(cudaDeviceSynchronize());
        const size_t rows(static_cast< size_t >(handle->chain[decoder].barcode_cardinality) + 1);
        if(u64_table != NULL) { PHQ_CUDA(cudaMemcpy(u64_table, handle->u64_plane() + handle->offset_u64[decoder], rows * ACC_U64_COLUMNS * 8, cudaMemcpyDeviceToHost)); }
        if(f64_table != NULL) { PHQ_CUDA(cudaMemcpy(f64_table, handle->f64_plane() + handle->offset_f64[decoder], rows * ACC_F64_COLUMNS * 8, cudaMemcpyDeviceToHost)); }
    });
}

int phq_totals(phq_handle* handle, uint64_t* count, uint64_t* pf_count) {
    return guarded(handle, [&]() {
        unsigned long long t[2];
        PHQ_CUDA(cudaDeviceSynchronize());
        PHQ_CUDA(cudaMemcpy(t, handle->totals(), sizeof(t), cudaMemcpyDeviceToHost));
        if(count != NULL) { *count = t[0]; }
        if(pf_count != NULL) { *pf_count = t[1]; }
    });
}

int phq_accumulator_buffer(phq_handle* handle, void** device_pointer, int64_t* n_u64, int64_t* n_f64) {
    return guarded(handle, [&]() {
        if(device_pointer != NULL) { *device_pointer = handle->device_accumulators.pointer; }
        if(n_u64 != NULL) { *n_u64 = handle->n_u64; }
        if(n_f64 != NULL) { *n_f64 = handle->n_f64; }
    });
}

int phq_reset_accumulators(phq_handle* handle) {
    return guarded(handle, [&]() {
        PHQ_CUDA(cudaDeviceSynchronize());
        PHQ_CUDA(cudaMemset(handle->device_accumulators.pointer, 0, static_cast< size_t >(handle->n_u64 + handle->n_f64) * 8));
        handle->collected = false;
    });
}

int phq_reset_accumulators_async(phq_handle* handle, void* stream) {
    return guarded(handle, [&]() {
        PHQ_CUDA(cudaMemsetAsync(handle->device_accumulators.pointer, 0, static_cast< size_t >(handle->n_u64 + handle->n_f64) * 8, static_cast< cudaStream_t >(stream)));
        handle->collected = false;
    });
}

int phq_estimate_priors(phq_handle* handle, int decoder, double* estimated_noise, double* estimated_concentration) {
    return guarded(handle, [&]() {
        if(decoder < 0 || decoder >= static_cast< int >(handle->chain.size())) { throw InternalError("decoder index out of range"); }
        const int32_t N(handle->chain[decoder].barcode_cardinality);
        std::vector< uint64_t > u(static_cast< size_t >(N + 1) * ACC_U64_COLUMNS);
        PHQ_CUDA(cudaDeviceSynchronize());
        PHQ_CUDA(cudaMemcpy(u.data(), handle->u64_plane() + handle->offset_u64[decoder], u.size() * 8, cudaMemcpyDeviceToHost));
        /* PamlDecoder::finalize (pamld.h:40-48) and Classifier::finalize (classifier.h:94-124) */
        uint64_t classified_count(0), pf_classified_count(0), low_conditional_confidence_count(0), low_confidence_count(0);
        for(int32_t i(1); i <= N; ++i) {
            classified_count += u[i * ACC_U64_COLUMNS + ACC_COUNT];
            pf_classified_count += u[i * ACC_U64_COLUMNS + ACC_PF_COUNT];
            if(handle->chain[decoder].algorithm == PHQ_PAMLD) {
                low_conditional_confidence_count += u[i * ACC_U64_COLUMNS + ACC_LOW_CONDITIONAL];
                low_confidence_count += u[i * ACC_U64_COLUMNS + ACC_LOW_CONFIDENCE];
            }
        }
        const uint64_t count(classified_count + u[ACC_COUNT]);
        double estimated_noise_count(low_conditional_confidence_count);
        double confident_noise_ratio(estimated_noise_count / (estimated_noise_count + pf_classified_count));
        if(low_confidence_count > 0) {
            estimated_noise_count += double(low_confidence_count) * confident_noise_ratio;
        }
        const double estimated_noise_prior(estimated_noise_count / double(count));
        const double estimated_not_noise_prior(1.0 - estimated_noise_prior);
        if(estimated_noise != NULL) { *estimated_noise = estimated_noise_prior; }
        if(estimated_concentration != NULL) {
            for(int32_t i(1); i <= N; ++i) {
                double pf_pooled_classified_fraction(0);
                const uint64_t pf_count(u[i * ACC_U64_COLUMNS + ACC_PF_COUNT]);
                if(pf_count > 0 && pf_classified_count > 0) {                      /* selector.cpp:87-99 */
                    pf_pooled_classified_fraction = double(pf_count) / double(pf_classified_count);
                }
                estimated_concentration[i - 1] = estimated_not_noise_prior * pf_pooled_classified_fraction;
            }
        }
    });
}

int phq_set_priors(phq_handle* handle, int decoder, double noise, const double* concentration) {
    return guarded(handle, [&]() {
        if(decoder < 0 || decoder >= static_cast< int >(handle->chain.size())) { throw InternalError("decoder index out of range"); }
        DecoderSpec& d(handle->chain[decoder]);
        if(!d.tiled()) { throw ConfigurationError("decoder has no priors"); }
        if(noise < 0 || noise > 1) { throw ConfigurationError("noise value " + std::to_string(noise) + " not between 0 and 1"); }
        d.noise = noise;
        if(concentration != NULL) {
            for(int32_t i(0); i < d.barcode_cardinality; ++i) { d.concentration[i] = concentration[i]; }
        }
        PHQ_CUDA(cudaDeviceSynchronize());
        build_tables(handle, static_cast< size_t >(decoder));
        refresh_params(handle, static_cast< size_t >(decoder));
    });
}

/* ------------------------------------------------------------------ the collective (classifier.h:87-93 across GPUs) */
extern "C++" {
namespace {

/*  NCCL resolved at run time: dlopen("libnccl.so.2") returns the copy already mapped into the process when there is
    one (a PyTorch host brings its own), else the system library. A host that never collects never needs it. */
struct NcclLibrary {
    void* library;
    ncclResult_t (*get_unique_id)(ncclUniqueId*);
    ncclResult_t (*comm_init_rank)(ncclComm_t*, int, ncclUniqueId, int);
    ncclResult_t (*comm_destroy)(ncclComm_t);
    ncclResult_t (*comm_count)(const ncclComm_t, int*);
    ncclResult_t (*all_reduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t);
    ncclResult_t (*group_start)();
    ncclResult_t (*group_end)();
    const char* (*get_error_string)(ncclResult_t);
    NcclLibrary() : library(NULL) {
        const char* const candidates[] = { "libnccl.so.2", "libnccl.so" };
        for(const char* name : candidates) {
            library = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if(library != NULL) { break; }
        }
        if(library == NULL) { throw InternalError(std::string("NCCL is not available : ") + dlerror()); }
        resolve(get_unique_id, "ncclGetUniqueId");
        resolve(comm_init_rank, "ncclCommInitRank");
        resolve(comm_destroy, "ncclCommDestroy");
        resolve(comm_count, "ncclCommCount");
        resolve(all_reduce, "ncclAllReduce");
        resolve(group_start, "ncclGroupStart");
        resolve(group_end, "ncclGroupEnd");
        resolve(get_error_string, "ncclGetErrorString");
    }
    template < class F > void resolve(F& target, const char* name) {
        target = reinterpret_cast< F >(dlsym(library, name));
        if(target == NULL) { throw InternalError(std::string("NCCL symbol missing : ") + name); }
    }
    void check(ncclResult_t status, const char* what) const {
        if(status != ncclSuccess) { throw InternalError(std::string("Internal error : NCCL ") + what + " : " + get_error_string(status)); }
    }
};
const NcclLibrary& nccl() {
    static const NcclLibrary instance;
    return instance;
}

template < class F > int guarded_global(F body) {
    try { body(); return PHQ_OK; }
    catch(...) { return record_error(NULL); }
}

}   /* namespace */
}   /* extern "C++" */

int phq_comm_unique_id(uint8_t* id) {
    return guarded_global([&]() {
        if(id == NULL) { throw InternalError("null argument"); }
        static_assert(sizeof(ncclUniqueId) == PHQ_COMM_ID_BYTES, "PHQ_COMM_ID_BYTES is NCCL_UNIQUE_ID_BYTES");
        ncclUniqueId value;
        nccl().check(nccl().get_unique_id(&value), "ncclGetUniqueId");
        memcpy(id, &value, sizeof(value));
    });
}

int phq_comm_create(const uint8_t* id, int rank, int world_size, int device, void** nccl_comm) {
    return guarded_global([&]() {
        if(id == NULL || nccl_comm == NULL || rank < 0 || rank >= world_size) { throw InternalError("illegal argument"); }
        PHQ_CUDA(cudaSetDevice(device));
        ncclUniqueId value;
        memcpy(&value, id, sizeof(value));
        ncclComm_t comm(NULL);
        nccl().check(nccl().comm_init_rank(&comm, world_size, value, rank), "ncclCommInitRank");
        *nccl_comm = comm;
    });
}

int phq_comm_destroy(void* nccl_comm) {
    return guarded_global([&]() {
        if(nccl_comm != NULL) { nccl().check(nccl().comm_destroy(static_cast< ncclComm_t >(nccl_comm)), "ncclCommDestroy"); }
    });
}

int phq_collect(phq_handle* handle, void* nccl_comm, void* stream) {
    return guarded(handle, [&]() {
        if(nccl_comm == NULL) { throw InternalError("null communicator"); }
        refuse_collected(handle);
        const NcclLibrary& library(nccl());
        ncclComm_t comm(static_cast< ncclComm_t >(nccl_comm));
        cudaStream_t s(static_cast< cudaStream_t >(stream));
        int world(0);
        library.check(library.comm_count(comm, &world), "ncclCommCount");
        /* behind the last device batch of this handle, whatever stream it was launched on */
        if(handle->timing_valid && handle->timing_stream != s) { PHQ_CUDA(cudaStreamWaitEvent(s, handle->timing_stop, 0)); }
        library.check(library.group_start(), "ncclGroupStart");
        library.check(library.all_reduce(handle->u64_plane(), handle->u64_plane(), static_cast< size_t >(handle->n_u64), ncclUint64, ncclSum, comm, s), "ncclAllReduce (u64 plane)");
        library.check(library.all_reduce(handle->f64_plane(), handle->f64_plane(), static_cast< size_t >(handle->n_f64), ncclFloat64, ncclSum, comm, s), "ncclAllReduce (f64 plane)");
        library.check(library.group_end(), "ncclGroupEnd");
        handle->collected = world > 1;
    });
}

int phq_statistics(phq_handle* handle, uint64_t* kernel_launches, uint64_t* exact_path_reads, uint64_t* threshold_band_reads) {
    return guarded(handle, [&]() {
        unsigned long long d[2];
        PHQ_CUDA(cudaDeviceSynchronize());
        PHQ_CUDA(cudaMemcpy(d, handle->diagnostics(), sizeof(d), cudaMemcpyDeviceToHost));
        if(kernel_launches != NULL) { *kernel_launches = handle->kernel_launches; }
        if(exact_path_reads != NULL) { *exact_path_reads = d[DIAG_EXACT_PATH]; }
        if(threshold_band_reads != NULL) { *threshold_band_reads = d[DIAG_THRESHOLD_BAND]; }
    });
}

/* ------------------------------------------------------------------ report and prior adjusted job (report.hpp) */
int phq_encode_report(phq_handle* handle, const uint64_t* const* u64_tables, const double* const* f64_tables, uint64_t count, uint64_t pf_count,
                      uint64_t incoming_count, uint64_t incoming_pf_count, int precision, char** report_json) {
    return guarded_host(handle, [&]() {
        if(u64_tables == NULL || f64_tables == NULL || report_json == NULL) { throw InternalError("null argument"); }
        std::vector< AccumulatorTables > tables(handle->chain.size());
        for(size_t k(0); k < handle->chain.size(); ++k) {
            if(u64_tables[k] == NULL || f64_tables[k] == NULL) { throw InternalError("null accumulator table"); }
            tables[k].u64 = u64_tables[k];
            tables[k].f64 = f64_tables[k];
        }
        const Json report(encode_job_report(handle->job, handle->chain, tables, count, pf_count, incoming_count, incoming_pf_count));
        *report_json = duplicate(report.dump(precision, 4));
    });
}

int phq_report(phq_handle* handle, uint64_t incoming_count, uint64_t incoming_pf_count, int precision, char** report_json) {
    return guarded(handle, [&]() {
        if(report_json == NULL) { throw InternalError("null argument"); }
        if(handle->device < 0) { throw InternalError("handle was created without a device"); }
        std::vector< uint64_t > u(static_cast< size_t >(handle->n_u64));
        std::vector< double > f(static_cast< size_t >(handle->n_f64));
        PHQ_CUDA(cudaDeviceSynchronize());
        PHQ_CUDA(cudaMemcpy(u.data(), handle->u64_plane(), u.size() * 8, cudaMemcpyDeviceToHost));
        PHQ_CUDA(cudaMemcpy(f.data(), handle->f64_plane(), f.size() * 8, cudaMemcpyDeviceToHost));
        std::vector< AccumulatorTables > tables(handle->chain.size());
        for(size_t k(0); k < handle->chain.size(); ++k) {
            tables[k].u64 = u.data() + handle->offset_u64[k];
            tables[k].f64 = f.data() + handle->offset_f64[k];
        }
        const uint64_t count(u[u.size() - 4]), pf_count(u[u.size() - 3]);
        const Json report(encode_job_report(handle->job, handle->chain, tables, count, pf_count, incoming_count, incoming_pf_count));
        *report_json = duplicate(report.dump(precision, 4));
    });
}

int phq_adjust_job(const char* job_json, const char* report_json, int precision, char** adjusted_json) {
    try {
        if(job_json == NULL || report_json == NULL || adjusted_json == NULL) { throw InternalError("null argument"); }
        Json adjusted(adjust_job(Json::parse(job_json), Json::parse(report_json)));
        adjusted.sort_keys();
        *adjusted_json = duplicate(adjusted.dump(precision, 4));
        return PHQ_OK;
    } catch(...) { return record_error(NULL); }
}

int phq_reference_power(phq_handle* handle, int64_t n, const double* sigma, double* power) {
    return guarded(handle, [&]() {
        if(n < 0 || (n > 0 && (sigma == NULL || power == NULL))) { throw InternalError("illegal argument"); }
        if(n == 0) { return; }
        DeviceBuffer< double > in, out;
        in.reserve(static_cast< size_t >(n));
        out.reserve(static_cast< size_t >(n));
        std::vector< double > phred;
        double uniform_quality, base;
        assemble_phred(phred, uniform_quality, base);
        cudaError_t status(cudaMemcpy(in.pointer, sigma, static_cast< size_t >(n) * sizeof(double), cudaMemcpyHostToDevice));
        if(status == cudaSuccess) { status = launch_reference_power(in.pointer, out.pointer, n, base, NULL); }
        if(status == cudaSuccess) { status = cudaMemcpy(power, out.pointer, static_cast< size_t >(n) * sizeof(double), cudaMemcpyDeviceToHost); }
        in.release();
        out.release();
        PHQ_CUDA(status);
    });
}

int phq_kernel_description(phq_handle* handle, int decoder, char* buffer, size_t capacity) {
    return guarded(handle, [&]() {
        if(decoder < 0 || static_cast< size_t >(decoder) >= handle->chain.size()) { throw InternalError("decoder index out of range"); }
        if(handle->device < 0) { throw InternalError("handle was created without a device"); }
        describe_kernels(handle->params[static_cast< size_t >(decoder)], static_cast< int >(handle->chain[static_cast< size_t >(decoder)].algorithm), buffer, capacity);
    });
}

int phq_last_kernel_milliseconds(phq_handle* handle, float* milliseconds) {
    return guarded(handle, [&]() {
        if(!handle->timing_valid) { throw InternalError("no device batch has been decoded yet"); }
        PHQ_CUDA(cudaEventSynchronize(handle->timing_stop));
        PHQ_CUDA(cudaEventElapsedTime(milliseconds, handle->timing_start, handle->timing_stop));
    });
}

}   /* extern "C" */
