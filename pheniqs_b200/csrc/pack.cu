/*  pack.cu — the feed -> tile kernel (pack.cuh). Lane = read. */
#include "pack.cuh"

#include <type_traits>

namespace phq {
namespace {

/* iupac.h:153-171 AsciiToAmbiguousBam, rows 0x30-0x7f; everything else is 15 */
__constant__ uint8_t ASCII_TO_BAM[80] = {
     1, 2, 4, 8, 15,15,15,15, 15,15,15,15, 15, 0,15,15,
    15, 1,14, 2, 13,15,15, 4, 11,15,15,12, 15, 3,15,15,
    15,15, 5, 6,  8,15, 7, 9, 15,10,15,15, 15,15,15,15,
    15, 1,14, 2, 13,15,15, 4, 11,15,15,12, 15, 3,15,15,
    15,15, 5, 6,  8,15, 7, 9, 15,10,15,15, 15,15,15,15,
};
/* iupac.h BamToAmbiguousAscii */
__constant__ uint8_t BAM_TO_ASCII[16] = { '=', 'A', 'C', 'M', 'G', 'R', 'S', 'V', 'T', 'W', 'Y', 'H', 'K', 'D', 'B', 'N' };
/* sequence.h BamToReverseComplementBam */
__constant__ uint8_t BAM_COMPLEMENT[16] = { 0x0, 0x8, 0x4, 0xc, 0x2, 0xa, 0x6, 0xe, 0x1, 0x9, 0x5, 0xd, 0x3, 0xb, 0x7, 0xf };

struct Base { uint32_t code; uint32_t quality; };

__device__ __forceinline__ long long read_begin(const RawSegmentView& v, long long r) {
    return v.offset != nullptr ? v.offset[v.first + r] : (v.first + r) * v.length;
}
__device__ __forceinline__ int read_length(const RawSegmentView& v, long long r) {
    return v.offset != nullptr ? static_cast< int >(v.offset[v.first + r + 1] - v.offset[v.first + r]) : static_cast< int >(v.length);
}
/* transform.h:65-80 */
__device__ __forceinline__ int absolute_end(const PackToken& t, int n) {
    if(t.end_terminated) {
        if(t.end < 0) { const int v = n + t.end; return v < 0 ? 0 : v; }
        return t.end > n ? n : t.end;
    }
    return n;
}
__device__ __forceinline__ int absolute_start(const PackToken& t, int n) {
    if(t.start < 0) { const int v = n + t.start; return v < 0 ? 0 : v; }
    return t.start > n ? 0 : t.start;
}

/* the tokens of one decoder over the raw segments of the launch */
struct TokenView {
    const PackToken* token;
    int token_cardinality;
    const RawSegmentView* input;
    int phred_offset;
    int bam_input;
};
__device__ __forceinline__ TokenView view_of(const PackPlan& plan) {
    TokenView v;
    v.token = plan.token; v.token_cardinality = plan.token_cardinality; v.input = plan.input; v.phred_offset = plan.phred_offset; v.bam_input = plan.bam_input;
    return v;
}

/* nucleotides Rule::apply appends to output segment s for read r (transform.h:142-169) */
__device__ __forceinline__ int observed_length(const TokenView& plan, const uint8_t* table, long long r, int s) {
    int length = 0;
    for(int k = 0; k < plan.token_cardinality; ++k) {
        const PackToken& t = plan.token[k];
        if(t.output_segment != s) { continue; }
        const int n = read_length(plan.input[t.input_segment], r);
        const int size = absolute_end(t, n) - absolute_start(t, n);
        length += size > 0 ? size : 0;
    }
    return length;
}
/* nucleotide i (< observed length) of output segment s of read r */
__device__ __forceinline__ Base fetch(const TokenView& plan, const uint8_t* table, long long r, int s, int i) {
    Base b;
    b.code = 0; b.quality = 0;
    int at = 0;
    for(int k = 0; k < plan.token_cardinality; ++k) {
        const PackToken& t = plan.token[k];
        if(t.output_segment != s) { continue; }
        const RawSegmentView& v = plan.input[t.input_segment];
        const int n = read_length(v, r);
        const int start = absolute_start(t, n);
        const int end = absolute_end(t, n);
        const int size = end - start;
        if(size <= 0) { continue; }
        if(i < at + size) {
            const int within = i - at;
            const long long source = read_begin(v, r) + (t.reverse_complement ? (end - within - 1) : (start + within));
            const uint32_t letter = v.sequence[source];
            /* FASTQ text through AsciiToAmbiguousBam (iupac.h:153-171), or the BAM code a decoded feed already holds */
            uint32_t code = plan.bam_input ? (letter & 0xfu) : ((letter >= 0x30u && letter < 0x80u) ? table[letter - 0x30u] : 15u);
            if(t.reverse_complement) { code = table[80 + code]; }
            b.code = code;
            b.quality = (static_cast< uint32_t >(v.quality[source]) - static_cast< uint32_t >(plan.phred_offset)) & 0xffu;     /* char arithmetic, fastq.h:73 */
            return b;
        }
        at += size;
    }
    return b;
}

/*  MAX = the most nucleotides the instantiation packs: 32 (one 32-bit word per plane) or PHQ_MAX_NUCLEOTIDES (64-bit
    planes, for decoders of more than 32 nucleotides) */
template < int MAX >
__global__ void __launch_bounds__(256)
pack_kernel(const __grid_constant__ PackPlan pack_plan, const long long n_reads, uint32_t* __restrict__ bases, uint16_t* __restrict__ nmask,
            uint32_t* __restrict__ quality, const long long pitch) {
    typedef typename std::conditional< (MAX <= 32), uint32_t, uint64_t >::type Plane;
    __shared__ uint8_t table[96];
    if(threadIdx.x < 80) { table[threadIdx.x] = ASCII_TO_BAM[threadIdx.x]; }
    else if(threadIdx.x < 96) { table[threadIdx.x] = BAM_COMPLEMENT[threadIdx.x - 80]; }
    __syncthreads();
    const TokenView plan = view_of(pack_plan);
    const int L = pack_plan.nucleotide_cardinality;
    for(long long r = blockIdx.x * static_cast< long long >(blockDim.x) + threadIdx.x; r < n_reads; r += static_cast< long long >(gridDim.x) * blockDim.x) {
        Plane lo = 0, hi = 0, ambiguous = 0;
        uint32_t phred[MAX / 4];
        #pragma unroll
        for(int w = 0; w < MAX / 4; ++w) { phred[w] = 0; }
        for(int s = 0; s < pack_plan.segment_cardinality; ++s) {
            const int expected = pack_plan.segment_offset[s + 1] - pack_plan.segment_offset[s];
            const int length = observed_length(plan, table, r, s);
            for(int i = 0; i < expected; ++i) {
                const int j = pack_plan.segment_offset[s] + i;
                const Plane bit = static_cast< Plane >(1) << j;
                Base b;
                if(i < length) {
                    b = fetch(plan, table, r, s, i);
                } else if(!pack_plan.stale_semantics) {
                    /* absent position (phq_pack): quality PHQ_ABSENT_QUALITY, ambiguous with both base bits set */
                    lo |= bit; hi |= bit; ambiguous |= bit;
                    phred[j >> 2] |= static_cast< uint32_t >(PHQ_ABSENT_QUALITY) << (8 * (j & 3));
                    continue;
                } else if(i == length) {
                    b.code = 0; b.quality = 0;                      /* the terminator the last append wrote */
                } else {
                    /* what an earlier read left there: the nearest one that reached position i */
                    b.code = pack_plan.carry_code[j]; b.quality = pack_plan.carry_quality[j];
                    for(long long earlier = r - 1; earlier >= 0; --earlier) {
                        const int reach = observed_length(plan, table, earlier, s);
                        if(reach == i) { b.code = 0; b.quality = 0; break; }
                        if(reach > i) { b = fetch(plan, table, earlier, s, i); break; }
                    }
                }
                switch(b.code) {
                    case 1: break;
                    case 2: lo |= bit; break;
                    case 4: hi |= bit; break;
                    case 8: lo |= bit; hi |= bit; break;
                    default: ambiguous |= bit; break;
                }
                phred[j >> 2] |= b.quality << (8 * (j & 3));
            }
        }
        if(MAX <= 32) {
            bases[r] = (static_cast< uint32_t >(lo) & 0xffffu) | ((static_cast< uint32_t >(hi) & 0xffffu) << 16);
            nmask[r] = static_cast< uint16_t >(static_cast< uint32_t >(ambiguous) & 0xffffu);
            if(L > 16) {
                bases[pitch + r] = (static_cast< uint32_t >(lo) >> 16) | (static_cast< uint32_t >(hi) & 0xffff0000u);
                nmask[pitch + r] = static_cast< uint16_t >(static_cast< uint32_t >(ambiguous) >> 16);
            }
        } else {
            #pragma unroll
            for(int w = 0; w < MAX / 16; ++w) {
                if(16 * w < L) {
                    bases[w * pitch + r] = static_cast< uint32_t >((lo >> (16 * w)) & 0xffffu) | (static_cast< uint32_t >((hi >> (16 * w)) & 0xffffu) << 16);
                    nmask[w * pitch + r] = static_cast< uint16_t >((ambiguous >> (16 * w)) & 0xffffu);
                }
            }
        }
        #pragma unroll
        for(int w = 0; w < MAX / 4; ++w) {
            if(4 * w < L) { quality[w * pitch + r] = phred[w]; }
        }
    }
}


/* ------------------------------------------------------------------ tag synthesis (pack.cuh) */
constexpr int TAG_WARPS = 4;

/* one read's auxiliary record being written into shared memory */
struct TagWriter {
    uint8_t* out;
    int at;
    __device__ __forceinline__ void put(uint32_t byte) { out[at++] = static_cast< uint8_t >(byte); }
    __device__ __forceinline__ int open(char a, char b, char type) { const int mark = at; put(a); put(b); put(type); return mark; }
    /* a Z tag is only encoded when its string is not empty (auxiliary.cpp:334-353) */
    __device__ __forceinline__ void close_string(int mark) { if(at == mark + 3) { at = mark; } else { put(0u); } }
    __device__ __forceinline__ void put_float(char a, char b, float value) {
        if(value > 0) {
            open(a, b, 'f');
            const uint32_t bits = __float_as_uint(value);
            put(bits & 0xffu); put((bits >> 8) & 0xffu); put((bits >> 16) & 0xffu); put(bits >> 24);
        }
    }
};

enum TagContent { TAG_RAW_SEQUENCE, TAG_RAW_QUALITY, TAG_CORRECTED_SEQUENCE, TAG_CORRECTED_QUALITY };

/*  One string tag of one topic: the decoders of the topic in chain order, their output segments in order
    (read.h:239-278: append_to_raw_* / append_to_corrected_*_sequence). Corrected content only comes from decoders
    with a codec; a corrected base keeps the observed quality where the observed base (indexed as
    Sequence::append_corrected does, sequence.h:382-398: from the length the corrected barcode already has) equals
    the corrected one or the barcode is undetermined ('='), and gets `corrected quality` elsewhere. */
__device__ __forceinline__ void put_string(TagWriter& w, const TagPlan& plan, const uint8_t* table, long long r, int topic, char a, char b, TagContent content) {
    const int mark = w.open(a, b, 'Z');
    int appended = 0;                       /* nucleotides this tag holds so far */
    for(int k = 0; k < plan.decoder_cardinality; ++k) {
        const TagDecoder& d = plan.decoder[k];
        if(d.topic != topic || d.token_cardinality == 0) { continue; }
        const bool corrected = content == TAG_CORRECTED_SEQUENCE || content == TAG_CORRECTED_QUALITY;
        if(corrected && d.results == nullptr) { continue; }
        TokenView view;
        view.token = d.token; view.token_cardinality = d.token_cardinality; view.input = plan.input; view.phred_offset = plan.phred_offset; view.bam_input = plan.bam_input;
        const uint8_t* barcode = nullptr;
        if(corrected) { barcode = d.barcode_code + static_cast< long long >(d.results[r].index) * d.nucleotide_cardinality; }
        for(int s = 0; s < d.segment_cardinality; ++s) {
            const int length = observed_length(view, table, r, s);
            const int expected = d.segment_offset[s + 1] - d.segment_offset[s];
            const int start = appended;
            for(int i = 0; i < length; ++i) {
                if(content == TAG_RAW_SEQUENCE) {
                    w.put(table[96 + fetch(view, table, r, s, i).code]);
                } else if(content == TAG_RAW_QUALITY) {
                    w.put((fetch(view, table, r, s, i).quality + 33u) & 0xffu);
                } else {
                    /* the barcode segment holds `expected` nucleotides and a terminator */
                    const uint32_t code = i < expected ? barcode[d.segment_offset[s] + i] : 0u;
                    if(content == TAG_CORRECTED_SEQUENCE) {
                        w.put(table[96 + code]);
                    } else {
                        const int probe = start + i;
                        const uint32_t observed = probe < length ? fetch(view, table, r, s, probe).code : (probe == length ? 0u : 0xffu);
                        const uint32_t quality = (observed == code || code == 0u) ? fetch(view, table, r, s, i).quality : static_cast< uint32_t >(d.corrected_quality);
                        w.put((quality + 33u) & 0xffu);
                    }
                }
                ++appended;
            }
        }
    }
    w.close_string(mark);
}

/*  Read level confidence of a topic (read.h:279-285 and the decoders' routing, pamld.cpp:133-180): the product over
    the topic's PAMLD decoders; a cellular or molecular decoder that leaves the read undetermined sets it to 0.
    Returns float(1 - confidence) when 0 < confidence < 1 (read.h:188-199), else 0. */
__device__ __forceinline__ float topic_error_probability(const TagPlan& plan, long long r, int topic) {
    double confidence = 1.0;
    for(int k = 0; k < plan.decoder_cardinality; ++k) {
        const TagDecoder& d = plan.decoder[k];
        if(d.topic != topic || d.algorithm != PHQ_PAMLD || d.results == nullptr) { continue; }
        const phq_result result = d.results[r];
        if(topic == PHQ_SAMPLE || result.index > 0) {
            confidence = confidence == 1.0 ? result.confidence : confidence * result.confidence;
        } else {
            confidence = 0.0;
        }
    }
    return (confidence > 0.0 && confidence < 1.0) ? static_cast< float >(1.0 - confidence) : 0.0f;
}

__global__ void __launch_bounds__(TAG_WARPS * 32)
tag_kernel(const __grid_constant__ TagPlan plan, const long long n_reads, uint8_t* __restrict__ aux, int32_t* __restrict__ aux_length) {
    extern __shared__ __align__(16) uint8_t tag_stage[];    /* [warp][32 records of stride + 4 bytes]: the pad spreads the lanes over the banks */
    __shared__ uint8_t table[96 + 16];
    if(threadIdx.x < 80) { table[threadIdx.x] = ASCII_TO_BAM[threadIdx.x]; }
    else if(threadIdx.x < 96) { table[threadIdx.x] = BAM_COMPLEMENT[threadIdx.x - 80]; }
    else if(threadIdx.x < 112) { table[threadIdx.x] = BAM_TO_ASCII[threadIdx.x - 96]; }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int stride = plan.stride;
    const int padded = stride + 4;
    uint8_t* const stage = tag_stage + static_cast< size_t >(warp) * 32 * padded;
    const long long step = static_cast< long long >(gridDim.x) * TAG_WARPS * 32;
    for(long long first = (static_cast< long long >(blockIdx.x) * TAG_WARPS + warp) * 32; first < n_reads; first += step) {
        const long long r = first + lane;
        TagWriter w;
        w.out = stage + lane * padded;
        w.at = 0;
        if(r < n_reads) {
            for(int topic = 0; topic < 3; ++topic) {
                bool present = false;
                for(int k = 0; k < plan.decoder_cardinality; ++k) { present = present || plan.decoder[k].topic == topic; }
                if(!present) { continue; }
                if(topic == PHQ_SAMPLE) {
                    /* set_RG(rg_by_barcode_index[decoded->index]) of the sample decoder (pamld.cpp:139, mdd.cpp:101) */
                    for(int k = 0; k < plan.decoder_cardinality; ++k) {
                        const TagDecoder& d = plan.decoder[k];
                        if(d.topic == PHQ_SAMPLE && d.results != nullptr && plan.read_group_offset != nullptr) {
                            const int index = d.results[r].index;
                            const int mark = w.open('R', 'G', 'Z');
                            for(int i = plan.read_group_offset[index]; i < plan.read_group_offset[index + 1]; ++i) { w.put(plan.read_group_text[i]); }
                            w.close_string(mark);
                        }
                    }
                    put_string(w, plan, table, r, topic, 'B', 'C', TAG_RAW_SEQUENCE);
                    put_string(w, plan, table, r, topic, 'Q', 'T', TAG_RAW_QUALITY);
                    w.put_float('X', 'B', topic_error_probability(plan, r, topic));
                } else if(topic == PHQ_MOLECULAR) {
                    put_string(w, plan, table, r, topic, 'R', 'X', TAG_CORRECTED_SEQUENCE);
                    put_string(w, plan, table, r, topic, 'Q', 'X', TAG_CORRECTED_QUALITY);
                    put_string(w, plan, table, r, topic, 'O', 'X', TAG_RAW_SEQUENCE);
                    put_string(w, plan, table, r, topic, 'B', 'Z', TAG_RAW_QUALITY);
                    w.put_float('X', 'M', topic_error_probability(plan, r, topic));
                } else {
                    put_string(w, plan, table, r, topic, 'C', 'B', TAG_CORRECTED_SEQUENCE);
                    put_string(w, plan, table, r, topic, 'C', 'R', TAG_RAW_SEQUENCE);
                    put_string(w, plan, table, r, topic, 'C', 'Y', TAG_RAW_QUALITY);
                    w.put_float('X', 'C', topic_error_probability(plan, r, topic));
                }
            }
            aux_length[r] = w.at;
            for(int i = w.at; i < stride; ++i) { w.out[i] = 0; }
        }
        __syncwarp();
        /* 32 records leave as one contiguous run of words */
        const long long live = (n_reads - first) < 32 ? (n_reads - first) : 32;
        const int words = stride >> 2;
        uint32_t* const target = reinterpret_cast< uint32_t* >(aux + first * stride);
        for(int i = lane; i < live * words; i += 32) {
            const int record = i / words;
            const int word = i - record * words;
            target[i] = *reinterpret_cast< const uint32_t* >(stage + record * padded + word * 4);
        }
        __syncwarp();
    }
}

}   /* namespace */

cudaError_t launch_pack(const PackPlan& plan, long long n_reads, uint32_t* bases, uint16_t* nmask, uint32_t* quality, long long pitch,
                        int multiprocessor_count, cudaStream_t stream) {
    if(n_reads <= 0) { return cudaSuccess; }
    const int threads = 256;
    const long long blocks = (n_reads + threads - 1) / threads;
    const long long resident = static_cast< long long >(multiprocessor_count) * 8;
    const int grid = static_cast< int >(blocks < resident ? blocks : resident);
    if(plan.nucleotide_cardinality > 32) {
        pack_kernel< PHQ_MAX_NUCLEOTIDES ><<< grid, threads, 0, stream >>>(plan, n_reads, bases, nmask, quality, pitch);
    } else {
        pack_kernel< 32 ><<< grid, threads, 0, stream >>>(plan, n_reads, bases, nmask, quality, pitch);
    }
    return cudaGetLastError();
}

cudaError_t launch_tags(const TagPlan& plan, long long n_reads, uint8_t* aux, int32_t* aux_length, int multiprocessor_count, cudaStream_t stream) {
    if(n_reads <= 0) { return cudaSuccess; }
    const size_t bytes = static_cast< size_t >(TAG_WARPS) * 32 * (plan.stride + 4);
    cudaError_t status = cudaFuncSetAttribute(tag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast< int >(bytes));
    if(status != cudaSuccess) { return status; }
    const long long blocks = (n_reads + TAG_WARPS * 32 - 1) / (TAG_WARPS * 32);
    const long long resident = static_cast< long long >(multiprocessor_count) * 4;
    tag_kernel<<< static_cast< int >(blocks < resident ? blocks : resident), TAG_WARPS * 32, bytes, stream >>>(plan, n_reads, aux, aux_length);
    return cudaGetLastError();
}

}   /* namespace phq */
