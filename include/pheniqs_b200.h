/*  pheniqs_b200.h — C ABI of the B200-native Pheniqs barcode classification path.

    This is the drop-in boundary for ONE path of the reference (Pheniqs 2.1.0): per-read
    barcode classification by the PAMLD and MDD decoders (plus the bookkeeping of the naive /
    passthrough decoders) over sample, molecular and cellular barcode sets. Everything the
    reference does on that path one read at a time through

        Classifier< Barcode >::classify(const Read&, Read&)      classifier.h:78-86
          <- PamlDecoder::classify / MdDecoder::classify          pamld.cpp:37-123, mdd.cpp:37-86
          <- TranscodingDecoder::classify                         transcode.h:51-65

    is done here for a whole batch of reads per call on one B200 (sm_100a). File:line
    citations are relative to the reference tree. Plain pointers and sizes only; no C++,
    torch or CUDA types appear in any signature (streams travel as void*).

    One handle = the ordered decoder chain of one job (sample, then molecular[], then
    cellular[]: transcode.h:51-60) on one GPU, owned by one host thread, exactly as one
    TranscodingThread owns a private TranscodingDecoder (transcode.cpp:2296).

    Every function returns a phq_status whose values are the reference's ErrorCode
    (error.h:32-44); the message of the last failure is read with phq_last_error().
*/
#ifndef PHENIQS_B200_H
#define PHENIQS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PHQ_VERSION "0.1.0"
#define PHQ_MAX_SEGMENTS 8          /* output segments of one decoder's Observation */
#define PHQ_MAX_NUCLEOTIDES 64      /* nucleotide cardinality of one decoder (four 16-base words); no struct of this
                                       header is sized by it. Decoders of more than 32 run on kernels of their own
                                       and cannot use the compact result forms above 63 (a 6-bit distance) */
#define PHQ_ABSENT_QUALITY 0xFF     /* quality byte phq_pack writes at a position the (short) read does not have; the
                                       kernels recognise such a position by its planes (phq_tile), not by this byte */

/* error.h:32-44 */
typedef enum {
    PHQ_OK                      = 0,
    PHQ_UNKNOWN_ERROR           = 1,
    PHQ_INTERNAL_ERROR          = 2,
    PHQ_CONFIGURATION_ERROR     = 3,
    PHQ_OUT_OF_MEMORY_ERROR     = 4,
    PHQ_COMMAND_LINE_ERROR      = 5,
    PHQ_IO_ERROR                = 6,
    PHQ_SEQUENCE_ERROR          = 7,
    PHQ_OVERFLOW_ERROR          = 8
} phq_status;

/* atom.h:348-355 (Algorithm) and classifier.h:28-33 (ClassifierType) */
typedef enum { PHQ_PAMLD = 0, PHQ_MDD = 1, PHQ_NAIVE = 2, PHQ_PASSTHROUGH = 3 } phq_algorithm;
typedef enum { PHQ_SAMPLE = 0, PHQ_MOLECULAR = 1, PHQ_CELLULAR = 2 } phq_topic;

typedef struct phq_handle phq_handle;

/*  Shape of decoder k of the chain, as compiled (decoder.h:44-52, classifier.h:54-60). */
typedef struct {
    int32_t algorithm;                  /* phq_algorithm */
    int32_t topic;                      /* phq_topic */
    int32_t index;                      /* "index" within its topic */
    int32_t barcode_cardinality;        /* codec entries, undetermined excluded; barcode rows are 1..N in sorted codec-key order */
    int32_t segment_cardinality;
    int32_t nucleotide_cardinality;
    int32_t segment_length[PHQ_MAX_SEGMENTS];
    int32_t word_cardinality;           /* ceil(nucleotide_cardinality / 16): uint32 base words and uint16 mask words per read */
    int32_t quality_word_cardinality;   /* ceil(nucleotide_cardinality / 4): uint32 quality words per read */
    int32_t has_tile;                   /* 1 when the decoder consumes a phq_tile (PAMLD, MDD), 0 otherwise */
} phq_decoder_info;

/*  One decoder's view of a batch: the Observation that Rule::apply (transform.h:142-169)
    extracts, for every read, as three structure-of-arrays planes. Position j of the
    concatenated observation (segments in order) lives in word j / 16, bit j % 16.

      bases[w * pitch + r]    bits 0..15  = low bit,  bits 16..31 = high bit of the 2-bit code
                              (A=0, C=1, G=2, T=3) of the 16 bases of word w of read r
      nmask[w * pitch + r]    bit j set   = base j is not one of A, C, G, T (N, IUPAC, '=' ...)
      quality[w * pitch + r]  byte k      = Phred value (offset removed) of base 4w + k, any of 0..255

    A base a short read does not have (MDD) is marked in the planes: its nmask bit and both base bits
    set, which no observed base has (an ambiguous base has its base bits clear). Its quality byte is
    PHQ_ABSENT_QUALITY, but an observed base may carry that byte too. PAMLD scores a Phred byte above
    127 as 0 (no information); MDD compares it with the masking threshold as it is.

    Binned qualities (current Illumina instruments emit 4 distinct values) can travel as indices
    into a per-tile codebook: with quality_bits = 4 or 2, position j occupies quality_bits bits at
    bit (j * quality_bits) % 32 of word (j * quality_bits) / 32 of the quality plane and
    quality_codebook[index] is its Phred value. quality_bits = 0 or 8 means plain bytes. This only
    changes how the bytes travel to the device (a 16-base observation shrinks from 22 to 10 bytes
    with 2-bit indices); the kernels see the same Phred values.

    Replaces the byte-per-base Segment / Observation containers of sequence.h:264-300. */
typedef struct {
    const uint32_t* bases;
    const uint16_t* nmask;
    const uint32_t* quality;
    int64_t pitch;                      /* elements between consecutive words of a plane (>= n_reads) */
    int32_t quality_bits;               /* 0 or 8: Phred bytes; 4 or 2: indices into quality_codebook */
    uint8_t quality_codebook[16];
} phq_tile;

/*  What one decoder decides for one read: decoded->index (0 = undetermined), edit_distance and
    decoding_confidence (classifier.h:47, decoder.h:34, pamld.h:35). MDD / naive confidence is 0. */
typedef struct {
    int32_t index;
    int32_t distance;
    double confidence;
} phq_result;

/*  The same decision in the 8 bytes the reference's OUTPUT carries for one decoder: the channel /
    read group index, the distance, the running qcfail flag and the error probability exactly as
    Read::flush forms it, float(1.0 - confidence) (read.h:187-199, the XB / XC / XM tags). Lossless
    with respect to the reference's output when a topic has one decoder; with several decoders of one
    topic the reference multiplies the f64 confidences first (read.h:279-285), which needs phq_result. */
typedef struct {
    uint32_t packed;                    /* bits 0-23 index, 24-29 distance, 30 qcfail after this decoder */
    float error_probability;            /* float(1.0 - confidence); 1 for an undetermined read */
} phq_compact_result;
#define PHQ_COMPACT_INDEX(p) ((p) & 0xffffffu)
#define PHQ_COMPACT_DISTANCE(p) (((p) >> 24) & 0x3fu)
#define PHQ_COMPACT_QCFAIL(p) (((p) >> 30) & 1u)

/* ------------------------------------------------------------------ configuration */

/*  Compile the decoder directives of a job the way Transcode::compile_decoder does
    (transcode.cpp:735-768, 824-1039; metric.h:87-111, 216-242; defaults configuration.json:368-376,
    423-501): barcode index by sorted codec key, concentrations normalised to 1 - noise,
    default random barcode probability 4^-n, default knit, default / validated distance
    tolerance. Input: {"sample": {...}, "molecular": [...], "cellular": [...]}. The compiled
    JSON (same keys as the reference's --compile output for those sections) is returned in a
    buffer the caller releases with phq_free. Host only; no GPU needed. */
int phq_compile_job(const char* job_json, char** compiled_json);
/*  The job document at `path` with the documents its "import" list names merged underneath it, depth first, each
    path relative to the importing document and visited once (Job::load_instruction_with_import, job.cpp:160-224).
    phq_compile_job then resolves `base` references between the decoders of the "decoder" repository and from the
    sample / molecular / cellular decoders into it (Transcode::apply_inheritance, transcode.cpp:328-442), values
    the "<topic>:decoder" / "<topic>:barcode" projections from the job root and the decoder
    (Transcode::compile_topic, transcode.cpp:769-823; configuration.json:423-501) and infers PU / ID of every
    barcode (transcode.cpp:1224-1260), so an unmodified reference job file can be fed in. Host only. */
int phq_load_job(const char* path, char** job_json);
void phq_free(void* pointer);
/* message of the last failure of a call that had no handle to attach it to (calling thread) */
const char* phq_last_global_error(void);

/* ------------------------------------------------------------------ lifecycle */

/*  Build the decoder chain from COMPILED decoder JSON, as the reference's decoder constructors
    do from the compiled ontology (classifier.h:54-60, decoder.h:44-52, pamld.cpp:24-31,
    mdd.cpp:24-27; factory transcode.cpp:66-161), and upload barcode tables, priors and Phred
    tables to `device`. Fails with PHQ_INTERNAL_ERROR when no CUDA device is usable: there is
    no CPU fallback. device < 0 builds a host-only handle (configuration + phq_pack only). */
int phq_create(const char* compiled_job_json, int device, phq_handle** handle);
void phq_destroy(phq_handle* handle);
const char* phq_last_error(const phq_handle* handle);

int phq_decoder_count(const phq_handle* handle);
int phq_decoder_describe(const phq_handle* handle, int decoder, phq_decoder_info* info);

/* ------------------------------------------------------------------ host side of the feed seam */

/*  Rule::apply (transform.h:142-169, token slicing transform.h:65-80, '~' reverse complement
    iupac.h:107-124) for every tiled decoder over a batch of reads held the way the reference
    holds them (one BAM 4-bit code byte and one Phred byte per base; segment s of read r is
    code[s][offset[s][r] .. offset[s][r+1])), packed into caller-provided HOST planes
    tiles[k] (k over all decoders; entries of untiled decoders are ignored).
    Short tokens: PAMLD tiles reproduce what a single reference thread sees (terminator, then
    the bytes left in its Observation by earlier reads, barcode.h:150 / sequence.h:296-300);
    MDD tiles mark missing positions as ambiguous with both base bits set, quality PHQ_ABSENT_QUALITY
    (sequence.h:90-98 iterate the observed length). The handle carries the Observation scratch from call to call.
    tiles[k].quality_bits selects how qualities are written: 0 / 8 = Phred bytes, 4 / 2 = codebook
    indices (PHQ_CONFIGURATION_ERROR if the batch has more distinct values than fit), -1 = the
    smallest that fits; on return quality_bits and quality_codebook describe what was written. The
    quality plane must be allocated for the byte form (quality_word_cardinality words). */
int phq_pack(phq_handle* handle, int64_t n_reads, int32_t n_input_segments,
             const uint8_t* const* code, const uint8_t* const* quality, const int64_t* const* offset,
             phq_tile* tiles);

/* ------------------------------------------------------------------ classification */

/*  TranscodingDecoder::classify (transcode.h:51-65) for n_reads reads with HOST buffers:
    tiles[k], results[k] (may be NULL for a decoder whose per-read results are not wanted) and
    the per-read qcfail flags (qcfail_in may be NULL = all clear; qcfail_out receives the
    running flag after the whole chain: input flag OR every decoder's verdict, read.h:94-103).
    Copies host->device, launches the kernels and copies back on internal streams, pipelined
    over sub-batches; returns when the outputs are in host memory. Accumulates into the
    handle's device-resident tables. Pinned host memory (phq_host_alloc) makes the copies
    asynchronous. */
int phq_decode_batch(phq_handle* handle, int64_t n_reads, const phq_tile* tiles,
                     const uint8_t* qcfail_in, phq_result* const* results, uint8_t* qcfail_out);

/*  Same, returning phq_compact_result records (8 bytes per read and decoder instead of 16 + the
    qcfail byte). compact_results[k] may be NULL. */
int phq_decode_batch_compact(phq_handle* handle, int64_t n_reads, const phq_tile* tiles,
                             const uint8_t* qcfail_in, phq_compact_result* const* compact_results);

/*  Same with DEVICE pointers, asynchronous on `stream` (a cudaStream_t, NULL = default
    stream): `qcfail` is read and updated in place. Nothing is copied; the caller synchronises. */
int phq_decode_batch_device(phq_handle* handle, int64_t n_reads, const phq_tile* device_tiles,
                            uint8_t* device_qcfail, phq_result* const* device_results, void* stream);

int phq_decode_batch_device_compact(phq_handle* handle, int64_t n_reads, const phq_tile* device_tiles,
                                    uint8_t* device_qcfail, phq_compact_result* const* device_compact_results, void* stream);

/* ------------------------------------------------------------------ feed bytes in (SURVEY.md §8 f1)

   The same classification from the bytes of the FASTQ records themselves: the device does what the feed and
   Rule::apply do on the host in the reference — AsciiToAmbiguousBam and `quality - phred offset` (fastq.h:55-78,
   iupac.h:153-171), token slicing and reverse complement (transform.h:65-80, 142-169) — and packs the tiles, so the
   host only hands over the barcode-bearing input segments as they sit in its feed buffers (feed.h:281-456). */
typedef struct phq_raw_segment {
    const uint8_t* sequence;    /* ASCII nucleotides (IUPAC) of every read of the batch, concatenated */
    const uint8_t* quality;     /* ASCII qualities (Phred + phred offset), same layout */
    const int64_t* offset;      /* [n_reads + 1] first byte of every read; NULL when every read has `length` bytes */
    int64_t length;             /* bytes per read when offset is NULL */
} phq_raw_segment;

/* phq_decode_batch / phq_decode_batch_compact with `segments[n_input_segments]` (host pointers; input segments no
   token refers to may be left NULL) in place of packed tiles. Results, accumulators and the state short tokens
   leave behind (see phq_pack) are identical to phq_pack of the decoded reads followed by phq_decode_batch. */
int phq_decode_batch_raw(phq_handle* handle, int64_t n_reads, int32_t n_input_segments, const phq_raw_segment* segments,
                         int32_t phred_offset, const uint8_t* qcfail_in, phq_result* const* results, uint8_t* qcfail_out);
int phq_decode_batch_raw_compact(phq_handle* handle, int64_t n_reads, int32_t n_input_segments, const phq_raw_segment* segments,
                                 int32_t phred_offset, const uint8_t* qcfail_in, phq_compact_result* const* compact_results);

/* The same from the form the reference itself keeps a decoded read in: `sequence` holds one BAM 4-bit code per base
   (Sequence::code, sequence.h:264-300: A=1 C=2 G=4 T=8 N=15, what FastqRecord decoding and bam_seqi produce) and
   `quality` one Phred value per base with the offset already removed (ObservedSequence::quality). A host whose feed
   has decoded its input (HTS input, hts.h; or FASTQ through fastq.h:55-78) hands its Segment buffers over unchanged
   and skips phq_pack: token slicing, reverse complement and the tile packing happen on the device. */
int phq_decode_batch_bam(phq_handle* handle, int64_t n_reads, int32_t n_input_segments, const phq_raw_segment* segments,
                         const uint8_t* qcfail_in, phq_result* const* results, uint8_t* qcfail_out);
int phq_decode_batch_bam_compact(phq_handle* handle, int64_t n_reads, int32_t n_input_segments, const phq_raw_segment* segments,
                                 const uint8_t* qcfail_in, phq_compact_result* const* compact_results);

/* ------------------------------------------------------------------ tags out (SURVEY.md §8 f2)

   What Read::flush (read.h:187-237) assembles from the decoders' verdicts and Auxiliary::encode
   (auxiliary.cpp:320-361) appends to every output record, produced on the device as the BAM auxiliary bytes
   themselves (tag, type, value; strings NUL terminated, floats little endian) in the reference's order:

       RG:Z                    ID of the sample barcode the read was assigned to (pamld.cpp:139, mdd.cpp:101)
       BC:Z QT:Z XB:f          raw sample barcode, its qualities (Phred + 33), float(1 - sample confidence)
       RX:Z QX:Z OX:Z BZ:Z XM:f corrected / raw molecular barcode and qualities (sequence.h:382-398: a corrected
                               base carries `corrected quality`)
       CB:Z CR:Z CY:Z XC:f      corrected / raw cellular barcode, its qualities, float(1 - cellular confidence)

   A string tag is left out when empty, a float tag unless 0 < confidence < 1, like the reference. Confidences of
   several decoders of a topic are multiplied in f64 first (read.h:279-285); an undetermined cellular or molecular
   decoder zeroes its topic (pamld.cpp:153-159). The host appends aux[r * aux_stride .. + aux_length[r]) to record r
   (every segment of the read carries the same block, read.h:219-231) and sets the QC fail flag from qcfail_out.
   Known divergence: QX of a second corrected molecular segment — the reference indexes the observed bases from
   the length the corrected barcode already has (sequence.h:388) and can run past the segment into stale memory;
   positions past the segment's terminator count as different here. */
int phq_tag_record_bytes(phq_handle* handle, int32_t* bytes);   /* the smallest aux_stride the job needs (multiple of 16) */
/* phq_decode_batch_raw that also writes the auxiliary block of every read; `results` may be NULL */
int phq_decode_batch_raw_tags(phq_handle* handle, int64_t n_reads, int32_t n_input_segments, const phq_raw_segment* segments, int32_t phred_offset,
                              const uint8_t* qcfail_in, uint8_t* aux, int32_t aux_stride, int32_t* aux_length, uint8_t* qcfail_out,
                              phq_result* const* results);

/* phq_decode_batch_raw_tags over BAM code / Phred byte segments (see phq_decode_batch_bam) */
int phq_decode_batch_bam_tags(phq_handle* handle, int64_t n_reads, int32_t n_input_segments, const phq_raw_segment* segments,
                              const uint8_t* qcfail_in, uint8_t* aux, int32_t aux_stride, int32_t* aux_length, uint8_t* qcfail_out,
                              phq_result* const* results);

int phq_host_alloc(void** pointer, size_t bytes);       /* pinned host memory */
void phq_host_free(void* pointer);

/* ------------------------------------------------------------------ accumulators and priors */

/*  Per-barcode accumulators of decoder k (AccumulatingOption, selector.h:32-60), row 0 =
    undetermined, rows 1..N = barcodes. u64 columns: count, pf_count, accumulated_distance,
    low_conditional_confidence_count, low_confidence_count, accumulated_pf_distance; f64
    columns: accumulated_confidence, accumulated_pf_confidence. Synchronises the device. */
int phq_accumulators(phq_handle* handle, int decoder, uint64_t* u64_table /* [(N+1)*6] */, double* f64_table /* [(N+1)*2] */);
/* TranscodingDecoder::count / pf_count (transcode.h:44-45) */
int phq_totals(phq_handle* handle, uint64_t* count, uint64_t* pf_count);
/*  The device buffer holding ALL accumulators of the handle, laid out as n_u64 unsigned 64-bit
    integers followed by n_f64 doubles, so the one collective of the path — the sum the
    reference does thread by thread in collect() (transcode.cpp:162-179, classifier.h:87-93,
    selector.cpp:68-77) — is one in-place all-reduce(sum) per plane. */
int phq_accumulator_buffer(phq_handle* handle, void** device_pointer, int64_t* n_u64, int64_t* n_f64);
int phq_reset_accumulators(phq_handle* handle);
/* the same without synchronising the device: the tables are cleared in `stream` order (a cudaStream_t, NULL = default
   stream), for hosts that keep decode -> collect -> reset on one stream */
int phq_reset_accumulators_async(phq_handle* handle, void* stream);

/* ------------------------------------------------------------------ the collective

   Classifier::collect across the GPUs of a job (classifier.h:87-93, selector.cpp:68-77, 185-196; the serial loop over
   threads of transcode.cpp:162-179): ONE in-place ncclAllReduce(sum) per plane of the handle's accumulator buffer
   (u64 counters as ncclUint64, f64 sums as ncclFloat64, grouped into one NCCL launch), asynchronous on `stream`
   (a cudaStream_t, NULL = default stream). `nccl_comm` is the host's own ncclComm_t with one rank per handle; the
   library finds NCCL at run time (the libnccl.so.2 already loaded into the process, else the system one), so hosts
   that never collect do not need it. The collective waits for the last phq_decode_batch_device of this handle
   whatever stream that ran on. Afterwards every rank holds the sums of the whole job: phq_accumulators,
   phq_estimate_priors and phq_report answer for the job. A handle whose tables were collected refuses to decode or
   collect again (PHQ_INTERNAL_ERROR) until phq_reset_accumulators: the sums would be counted once per rank. */
int phq_collect(phq_handle* handle, void* nccl_comm, void* stream);
/* Convenience for hosts without a communicator of their own: ncclGetUniqueId on one rank (the 128 bytes travel to the
   other ranks by whatever channel the host has), ncclCommInitRank on every rank (call after cudaSetDevice-equivalent
   `device`), ncclCommDestroy. */
#define PHQ_COMM_ID_BYTES 128
int phq_comm_unique_id(uint8_t* id /* [PHQ_COMM_ID_BYTES] */);
int phq_comm_create(const uint8_t* id, int rank, int world_size, int device, void** nccl_comm);
int phq_comm_destroy(void* nccl_comm);

/*  Classifier::finalize prior estimation (classifier.h:94-124 with pamld.h:40-48,
    decoder.h:77-83, selector.cpp:78-101) from the current accumulators of decoder k. */
int phq_estimate_priors(phq_handle* handle, int decoder, double* estimated_noise, double* estimated_concentration /* [N] */);
/*  Install a noise prior and per-barcode concentration priors (taken as already normalised,
    as Classifier::adjust_prior writes them, classifier.h:125-160) for the next pass. */
int phq_set_priors(phq_handle* handle, int decoder, double noise, const double* concentration /* [N] */);

/* ------------------------------------------------------------------ report and prior adjusted job */

/* The decoder sections of the job report Transcode::finalize assembles (transcode.cpp:1811-1863): "outgoing",
   "sample", "molecular", "cellular" with every AccumulatingSelector / AccumulatingOption key the reference
   encodes (selector.cpp:102-135, 215-247; classifier.h:161-177; barcode.cpp:53-67), the estimated priors
   (classifier.h:94-124), read group tags on the sample elements, cleaned and key sorted (json.cpp:834-893),
   written with at most `precision` decimal places (the reference's float precision, 15 by default).
   "incoming" (feed statistics, not part of this path) is encoded when incoming_count > 0.
   Reads the device accumulators of this handle; after an all-reduce of phq_accumulator_buffer it is the report
   of the whole job. *report_json is malloc'd; release with phq_free. */
int phq_report(phq_handle* handle, uint64_t incoming_count, uint64_t incoming_pf_count, int precision, char** report_json);
/* the same from caller-held tables (u64_tables[k]: [(N_k + 1)][6], f64_tables[k]: [(N_k + 1)][2], chain order) and
   chain totals; pure host work, also available on a host-only handle */
int phq_encode_report(phq_handle* handle, const uint64_t* const* u64_tables, const double* const* f64_tables,
                      uint64_t count, uint64_t pf_count, uint64_t incoming_count, uint64_t incoming_pf_count,
                      int precision, char** report_json);
/* The prior adjusted job: `noise` and every codec `concentration` of the sample / molecular / cellular decoders of
   job_json replaced by the report's "estimated noise" / "estimated concentration" (barcodes matched by their
   segments; 0 where the report has no estimate), as tool/pheniqs-prior-api.py:39-56, 186-215 and
   Classifier::adjust_prior (classifier.h:125-160) do; key sorted. Host only. */
int phq_adjust_job(const char* job_json, const char* report_json, int precision, char** adjusted_json);

/* ------------------------------------------------------------------ instrumentation */

/* kernels launched by this handle so far, reads that needed the exact tie path, and reads whose PAMLD decision fell
   within the accuracy of the path of a threshold (diagnostic "band" counter): within 1e-12 (relative) for the exact
   and prefilter scans, within 2^-21 (1 - confidence) of the confidence threshold for the pruned whitelist scan,
   whose sigma_p can lack up to that much (DESIGN.md §4.9): such a read may be decided differently from the reference */
int phq_statistics(phq_handle* handle, uint64_t* kernel_launches, uint64_t* exact_path_reads, uint64_t* threshold_band_reads);
/* names of the kernels decoder `decoder` launches with its current tables ("pamld_grid_kernel<8, 8, 2, 8, 1> +
   pamld_tie_kernel<4>"), NUL terminated into buffer[capacity]; for reports and profiles. No reference counterpart. */
int phq_kernel_description(phq_handle* handle, int decoder, char* buffer, size_t capacity);
/* power[i] = pow(PHRED_PROBABILITY_BASE, sigma[i]) (phred.h:34, barcode.h:163) as the device forms it where the
   reference's decision depends on the rounding of pow itself (ties between barcodes whose Kahan sums differ in the
   last bits): a correctly rounded double-double evaluation, which is what glibc's pow returns except within 2^-68 of a
   rounding boundary. Host buffers; for parity tests. */
int phq_reference_power(phq_handle* handle, int64_t n, const double* sigma, double* power);
/* device time (ms) of the kernels of the last phq_decode_batch_device call, measured with CUDA
   events on the launching stream; synchronises that stream */
int phq_last_kernel_milliseconds(phq_handle* handle, float* milliseconds);

#ifdef __cplusplus
}
#endif
#endif /* PHENIQS_B200_H */
