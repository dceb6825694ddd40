/*  kernels.cuh — device-side data layout and launch interface of the classification kernels.

    HBM layout (see DESIGN.md):
      tiles        structure-of-arrays planes, read index fastest (phq_tile in pheniqs_b200.h)
      barcodes     one 16-byte entry per barcode: low bit-plane, high bit-plane (32 positions
                   each, position j = bit j) and the f64 prior  -> replaces vector< Barcode >
                   (classifier.h:49) for the scoring loop
      phred        f64 tables derived on the host with libm exactly as phred.cpp:24-72 does
      accumulators [(N+1)][6] u64 then [(N+1)][2] f64 per decoder, inside one buffer per handle
*/
#ifndef PHQ_KERNELS_CUH
#define PHQ_KERNELS_CUH

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pheniqs_b200.h"

namespace phq {

struct __align__(16) BarcodeEntry {
    uint32_t lo;            /* bit j = low bit of the 2-bit code of barcode position j */
    uint32_t hi;            /* bit j = high bit */
    double prior;           /* Barcode::concentration (barcode.h:37) */
};

/*  The same barcode for the f32 prefilter scans (pamld_fast_kernel): planes and the prior rounded to f32. */
struct __align__(16) FastEntry {
    uint32_t lo;
    uint32_t hi;
    float prior;
    uint32_t pad;
};

/*  Decoders of more than LONG_NUCLEOTIDES positions (up to PHQ_MAX_NUCLEOTIDES) take the long kernels
    (pamld_long_kernel, pamld_long_tie_kernel, mdd_long_kernel) and this table instead of the 16-byte one. Their
    positions travel in SPLIT FORM, two 32-bit words per plane: word 0 holds positions [0, split), word 1 positions
    [split, L), split = long_split(L) = 4 x ceil(L / 8), so each word covers at most ceil(L / 8) groups of four
    positions and the PAMLD scan gives one word to each lane of a lane pair. */
constexpr int LONG_NUCLEOTIDES = 32;
__host__ __device__ inline int long_split(int nucleotides) { return 4 * ((nucleotides + 7) / 8); }
struct __align__(16) LongBarcodeEntry {
    uint32_t lo0, hi0;      /* low / high bit-plane of positions [0, split) */
    uint32_t lo1, hi1;      /* of positions [split, L), position split + j = bit j */
    double prior;
    double pad;
};
static_assert(sizeof(LongBarcodeEntry) == 32, "one long barcode entry is 32 bytes");

/* offsets into the f64 Phred table uploaded once per handle */
enum {
    PHRED_MATCH_FACTOR   = 0,       /* [128]  B ^ true_positive_quality[q]      (q = 0 -> 1)            */
    PHRED_MISMATCH_RATIO = 128,     /* [128]  B ^ (q - true_positive_quality[q]) (q = 0 -> 1)           */
    PHRED_TRUE_POSITIVE_QUALITY = 256, /* [128] phred.cpp:34-38, used by the exact tie path            */
    PHRED_UNIFORM_QUALITY = 384,    /* UNIFORM_BASE_QUALITY, phred.h:33                                  */
    PHRED_BASE = 385,               /* PHRED_PROBABILITY_BASE, phred.h:34                                */
    PHRED_UNIFORM_FACTOR = 386,     /* B ^ UNIFORM_BASE_QUALITY                                          */
    PHRED_TABLE_SIZE = 388
};

enum { ACC_COUNT = 0, ACC_PF_COUNT = 1, ACC_DISTANCE = 2, ACC_LOW_CONDITIONAL = 3, ACC_LOW_CONFIDENCE = 4, ACC_PF_DISTANCE = 5, ACC_U64_COLUMNS = 6 };
enum { ACC_CONFIDENCE = 0, ACC_PF_CONFIDENCE = 1, ACC_F64_COLUMNS = 2 };
enum { DIAG_EXACT_PATH = 0, DIAG_THRESHOLD_BAND = 1, DIAG_COLUMNS = 2 };

/*  MDD lookup tables (mdd_table_kernel). When every segment's tolerance is within its Shannon bound, at most one
    distinct word of a segment lies within tolerance of an observed segment, so the reference's scan
    (mdd.cpp:50-80) is a lookup: every variant of every distinct word within tolerance (substitutions and N /
    masked positions) is a key of an open addressing hash table whose value is the word and the distance, and the
    tuple of words is looked up in a second table that holds the barcodes. */
struct __align__(8) MddSlot {
    uint32_t key_lo;            /* segment: low plane | high plane << 16; combination: word 0 | word 1 << 12 | word 2 << 24 (low 8 bits) */
    uint16_t key_hi;            /* segment: ambiguity plane; combination: word 2 >> 8 | word 3 << 4 */
    uint16_t value;             /* segment: word | distance << 12; combination: barcode index; 0xffff = empty slot */
};
constexpr uint32_t MDD_EMPTY = 0xffffu;
constexpr int MDD_MAX_WORDS = 4095;             /* distinct words per segment (12 bits) */
constexpr int MDD_MAX_BARCODES = 65535;         /* barcode index in 16 bits, 0xffff reserved */
__host__ __device__ inline uint32_t mdd_hash(uint32_t key_lo, uint32_t key_hi) {
    uint32_t h = (key_lo * 0x9E3779B1u) ^ (key_hi * 0x85EBCA77u) ^ 0x27D4EB2Fu;
    h ^= h >> 15;
    h *= 0x2C1B3C6Du;
    h ^= h >> 13;
    return h;
}

/*  Whitelist blob (pamld_whitelist_kernel; large single-word codecs such as a 737 K x 16 nt cellular whitelist).
    The table is cut into groups of WHITELIST_CHUNK barcodes, each one contiguous so that ONE TMA bulk copy stages it:
      equality planes  [position 0..15][code A, C, G, T, "not counted"][block of 32 barcodes] u32 — bit k of
                       plane (j, c, block) is set when barcode 32 * block + k has base c at position j; the
                       fifth plane is all ones (positions a read does not count read it); the four blocks of a
                       (position, code) are one 16-byte load
    The exact path reads the barcode word and prior of a candidate from `barcodes`; the padding of the last group
    has no plane bit set, so it is never a candidate. */
constexpr int WHITELIST_CHUNK = 128;
constexpr int WHITELIST_POSITIONS = 16;
constexpr int WHITELIST_PLANES = 5;
constexpr int WHITELIST_BLOCKS = WHITELIST_CHUNK / 32;
constexpr int WHITELIST_EQUALITY_WORDS = WHITELIST_BLOCKS * WHITELIST_POSITIONS * WHITELIST_PLANES;
constexpr int WHITELIST_CHUNK_BYTES = WHITELIST_EQUALITY_WORDS * 4;
constexpr int WHITELIST_MINIMUM_BARCODES = 4096;    /* smaller codecs use the exhaustive scans (PHQ_WHITELIST_MINIMUM overrides, for tests) */

/* what the scan kernel hands to the tie kernel for a queued read */
constexpr int TIE_CANDIDATES = 11;                  /* barcodes the scan can name as possible winners of a queued read */
constexpr uint32_t TIE_RESCAN = 0xffffffffu;        /* candidate_count of a read whose candidates the tie kernel has to find itself */
constexpr uint32_t TIE_BLOCKS = 0xfffffffeu;        /* candidate_count: candidate[0] is a bit mask over runs of (4 << candidate[1]) consecutive barcodes (grid entries when candidate[2]) that hold every possible winner */
constexpr uint32_t TIE_MASKS = 0xfffffffdu;         /* candidate_count: candidate[0] x candidate[1] are bit masks over the distinct words of the two parts of a full grid of candidate[2] B words per A word */
constexpr uint32_t TIE_POOLED = 0x40000000u;        /* candidate_count flag: the (count & 0xffff) candidates are in the pool from entry candidate[0] on */
constexpr int TIE_POOLED_CANDIDATES = 64;           /* the most a scan names for one read (the whitelist scan: noise reads tie a dozen ways) */
constexpr int TIE_POOL_PER_READ = 4;                /* pool entries per read of the launch */
struct __align__(16) TieRecord {
    double best;                /* the scan's maximum prior adjusted product (relative to P0) */
    double rest;                /* the scan's sum of all other products */
    double base_probability;    /* P0 */
    uint32_t high_quality_mask;
    uint32_t uniform;
    uint32_t o_lo, o_hi, nmask; /* the observation */
    uint32_t read;              /* read index within the launch */
    uint32_t quality[8];
    uint32_t candidate_count;   /* barcodes named below; more than TIE_CANDIDATES (TIE_RESCAN) = scan the whole table */
    uint32_t candidate[TIE_CANDIDATES];     /* every barcode whose product is within 2^-19 of the maximum is among them */
};
static_assert(sizeof(TieRecord) == 128, "one tie record is 128 bytes");

struct DecoderParams {
    int32_t algorithm;
    int32_t barcode_cardinality;
    int32_t nucleotide_cardinality;
    int32_t word_cardinality;
    int32_t quality_word_cardinality;
    int32_t group_cardinality;                  /* ceil(nucleotide_cardinality / 4) */
    int32_t segment_cardinality;
    uint32_t segment_mask[PHQ_MAX_SEGMENTS];    /* positions of each segment in the concatenated observation */
    int32_t distance_tolerance[PHQ_MAX_SEGMENTS];
    int32_t high_quality_threshold;
    int32_t high_quality_distance_threshold;
    int32_t quality_masking_threshold;
    double adjusted_noise_probability;          /* noise * random barcode probability, pamld.cpp:29 */
    double confidence_threshold;
    double random_barcode_probability;
    double uniform_observation_probability;     /* pow(B, Kahan sum of L copies of U) computed with the host libm */
    const BarcodeEntry* barcodes;               /* [N] device */
    const double* phred;                        /* [PHRED_TABLE_SIZE] device */
    unsigned long long* acc_u64;                /* [(N+1)][6] device */
    double* acc_f64;                            /* [(N+1)][2] device */
    unsigned long long* totals;                 /* [2] count, pf_count; NULL unless this is the last decoder of the chain */
    unsigned long long* diagnostics;            /* [DIAG_COLUMNS] */
    const MddSlot* mdd_tables;                  /* NULL = scan every barcode (mdd_kernel) */
    int32_t mdd_first[PHQ_MAX_SEGMENTS + 1];   /* first slot of each segment table; [segment_cardinality] = the combination table */
    int32_t mdd_mask[PHQ_MAX_SEGMENTS + 1];    /* slots - 1 of each table (powers of two) */
    int32_t mdd_slots;                          /* total slots */
    int32_t segment_offset[PHQ_MAX_SEGMENTS];
    int32_t segment_length[PHQ_MAX_SEGMENTS];
    const void* grid;                           /* combinatorial codec blob: grid_a headers, grid_b words, grid_entries entries (16 B each); NULL = generic scan */
    int32_t grid_a;
    int32_t grid_b;
    int32_t grid_entries;
    int32_t grid_split;                         /* nucleotides of the first segment */
    int32_t grid_dense;                         /* 0, or the padded B word count (8 / 16) of the dense form: entries = grid_a x grid_dense */
    int32_t grid_uniform;                       /* dense form with every combination present under one prior */
    const unsigned char* whitelist;             /* chunked blob of pamld_whitelist_kernel (WhitelistLayout); NULL = the other scans */
    int32_t whitelist_chunks;
    double prior_maximum;                       /* largest barcode prior: the pruning bound of pamld_whitelist_kernel */
    TieRecord* tie_record;                      /* [reads of the launch] queue of reads whose winner needs the exact tie path (PAMLD) */
    unsigned* tie_count;                        /* queue header: [0] tie queue length, [1] work counter (of the whitelist scan, then of the tie pass), [2] hard list length, [3] pool cursor */
    const FastEntry* fast_barcodes;             /* [N] device; NULL = no f32 prefilter scan for this decoder (exact scan over every read) */
    const float* phred32;                       /* [128] mismatch ratios rounded to f32 */
    float fast_uniform_prior;                   /* the common prior (f32) when every barcode has the same one, else 0: the prefilter scan then multiplies once per read */
    int* hard_list;                             /* [reads of the launch] reads the prefilter scan leaves to the exact scan */
    int32_t tie_block_shift;                    /* log2 of the blocks of four barcodes (grid entries) one bit of a TIE_BLOCKS mask stands for */
    uint32_t* tie_pool;                         /* candidates of the reads that name more than a record holds; cursor = tie_count[3] */
    uint32_t tie_pool_capacity;
    /* decoders of more than LONG_NUCLEOTIDES positions: `barcodes` is NULL, segment_mask holds word 0 of the split form */
    const LongBarcodeEntry* long_barcodes;      /* [N] device */
    int32_t long_split;                         /* long_split(nucleotide_cardinality) */
    uint32_t segment_mask_long[PHQ_MAX_SEGMENTS];   /* word 1 of each segment's mask in split form (MDD) */
};

struct TileArguments {
    const uint32_t* bases;
    const uint16_t* nmask;
    const uint32_t* quality;
    long long pitch;
    long long n_reads;
    uint8_t* qcfail;                            /* in/out running flag, [n_reads] */
    phq_result* results;                        /* may be NULL */
    phq_compact_result* compact;                /* may be NULL; written instead of `results` when set */
    int quality_bits;                           /* 8, 4 or 2 (phq_tile) */
    int nucleotides;                            /* nucleotide cardinality of the decoder */
    const int* index_list;                      /* when set, the kernel works on reads index_list[0 .. *index_count) instead of 0 .. n_reads */
    const unsigned* index_count;
    uint32_t codebook[4];                       /* quality_codebook, little endian words */
};

struct LaunchGeometry {
    int multiprocessor_count;
    size_t shared_memory_per_block_optin;
};

/* each returns the CUDA error of the launch; all are asynchronous on `stream`.
   launch_pamld launches two kernels (scan, then the tie pass over the reads the scan queued). */
enum { PAMLD_KERNEL_LAUNCHES = 2, PAMLD_FAST_KERNEL_LAUNCHES = 3, MDD_KERNEL_LAUNCHES = 1, COUNT_KERNEL_LAUNCHES = 1 };
/* kernels launch_pamld launches for these parameters: prefilter scan + exact scan over the reads it left + tie pass, or scan + tie pass */
inline int pamld_launches(const DecoderParams& params) { return (params.fast_barcodes != nullptr && params.whitelist == nullptr) ? PAMLD_FAST_KERNEL_LAUNCHES : PAMLD_KERNEL_LAUNCHES; }
/* PAMLD launches cover at most this many reads, so the tie queue (80 bytes per read, worst case every read) stays bounded */
constexpr long long PAMLD_LAUNCH_READS = 1ll << 24;
cudaError_t launch_pamld(const DecoderParams& params, const TileArguments& tile, const LaunchGeometry& geometry, cudaStream_t stream);
cudaError_t launch_mdd(const DecoderParams& params, const TileArguments& tile, const LaunchGeometry& geometry, cudaStream_t stream);
/* naive / passthrough bookkeeping: count and pf_count of the undetermined row (and the chain totals) */
void describe_kernels(const DecoderParams& params, int algorithm, char* buffer, size_t capacity);
cudaError_t launch_count(const DecoderParams& params, const TileArguments& tile, const LaunchGeometry& geometry, cudaStream_t stream);
cudaError_t prepare_kernels(const LaunchGeometry& geometry);
/* out[i] = pow(base, sigma[i]) as the tie pass forms it (correctly rounded double-double evaluation); device pointers */
cudaError_t launch_reference_power(const double* sigma, double* out, long long n, double base, cudaStream_t stream);
/* (first segment length, total length) pairs the combinatorial scan is instantiated for */
inline bool grid_shape_supported(int split, int total) { return (split == 6 && total == 12) || (split == 8 && total == 16) || (split == 10 && total == 20) || (split == 12 && total == 24); }

}   /* namespace phq */
#endif
