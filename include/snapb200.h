/*
 * snapb200.h -- C ABI of the B200-native Snappy codec (libsnapb200.so).
 *
 * This is the drop-in boundary for rust-snappy's raw/frame hot path: a Rust
 * `snap` shim (see INTEGRATION.md, rust/) binds exactly these symbols. Each
 * entry point cites the reference interface it replaces (paths relative to the
 * rust-snappy checkout). Plain pointers and sizes only -- no torch/CUDA types.
 *
 * All work is done by sm_100a CUDA kernels; there is NO CPU fallback. When no
 * CUDA device is usable every compute call returns SB_E_NO_DEVICE.
 */
#ifndef SNAPB200_H
#define SNAPB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* snap::Error variant index (declaration order of src/error.rs:72-180) plus
 * the payload fields of that variant in a, b, c. 0 = Ok. */
enum {
    SB_OK = 0,
    SB_TOO_BIG = 1,                  /* a=given  b=max                         */
    SB_BUFFER_TOO_SMALL = 2,         /* a=given  b=min                         */
    SB_EMPTY = 3,
    SB_HEADER = 4,
    SB_HEADER_MISMATCH = 5,          /* a=expected_len b=got_len               */
    SB_LITERAL = 6,                  /* a=len a=src_len c=dst_len              */
    SB_COPY_READ = 7,                /* a=len b=src_len                        */
    SB_COPY_WRITE = 8,               /* a=len b=dst_len                        */
    SB_OFFSET = 9,                   /* a=offset b=dst_pos                     */
    SB_STREAM_HEADER = 10,           /* a=byte                                 */
    SB_STREAM_HEADER_MISMATCH = 11,  /* a=6 body bytes, little endian          */
    SB_UNSUPPORTED_CHUNK_TYPE = 12,  /* a=byte                                 */
    SB_UNSUPPORTED_CHUNK_LENGTH = 13,/* a=len b=header(0/1)                    */
    SB_CHECKSUM = 14,                /* a=expected b=got                       */
    SB_IO_UNEXPECTED_EOF = 100,      /* io::ErrorKind::UnexpectedEof (read_exact, src/read.rs:439-455) */
    /* library-level failures (never produced by the reference) */
    SB_E_NO_DEVICE = 200,            /* no usable CUDA device / kernel image   */
    SB_E_CUDA = 201,                 /* a=cudaError_t                          */
    SB_E_INVALID = 202               /* bad argument (null pointer, ...)       */
};

typedef struct sb_error {
    uint32_t code;
    uint32_t _pad;
    uint64_t a, b, c;
} sb_error;

/* Outcome of a stream-ordered frame call, written to device memory by the last kernel of the call. */
typedef struct sb_frame_result {
    sb_error status;                 /* SB_OK or the first error in stream order                  */
    uint64_t bytes;                  /* encode: stream length; decode: bytes produced before the error */
    uint32_t nchunks;                /* data chunks in the stream                                  */
    uint32_t _pad;
} sb_frame_result;

/* ---- scalar API: host pointers, mirrors snap::raw ------------------------ */

/* snap::raw::max_compress_len  (src/compress.rs:42-53). Pure arithmetic. */
size_t sb_max_compress_len(size_t input_len);

/* snap::raw::Encoder::compress (src/compress.rs:99-154): `in` is compressed
 * as ONE raw stream (varint header + 64KB blocks) into out[..cap]; on success
 * returns 0 and *out_n = bytes written. Errors: TooBig, BufferTooSmall. */
int sb_compress(const uint8_t* in, size_t n, uint8_t* out, size_t cap, size_t* out_n, sb_error* err);

/* snap::raw::decompress_len (src/decompress.rs:30-35). Header parse only. */
int sb_decompress_len(const uint8_t* in, size_t n, size_t* out_len, sb_error* err);

/* snap::raw::Decoder::decompress (src/decompress.rs:75-95). Exact error
 * variant and payload of the reference on corrupt input. */
int sb_decompress(const uint8_t* in, size_t n, uint8_t* out, size_t cap, size_t* out_n, sb_error* err);

/* crc32::CheckSummer::crc32c_masked (src/crc32.rs:35-38), computed on device. */
int sb_crc32c_masked(const uint8_t* in, size_t n, uint32_t* out, sb_error* err);

/* ---- batched host API: many independent raw streams per call -------------
 * What a Rust caller holding many buffers (or the frame writers below) uses:
 * one call, pinned staging + H2D/D2H pipelined against the kernels inside.
 * Unit i reads in_base[in_offs[i] .. +in_lens[i]) and writes out_base[out_offs[i] ..];
 * out capacity per unit is out_caps[i]. statuses may be NULL for compress. */
int sb_compress_batch_host(const uint8_t* in_base, const uint64_t* in_offs, const uint32_t* in_lens,
                           uint8_t* out_base, const uint64_t* out_offs, const uint32_t* out_caps,
                           uint32_t* out_lens, size_t count, sb_error* err);
int sb_decompress_batch_host(const uint8_t* in_base, const uint64_t* in_offs, const uint32_t* in_lens,
                             uint8_t* out_base, const uint64_t* out_offs, const uint32_t* out_caps,
                             uint32_t* out_lens, sb_error* statuses, size_t count, sb_error* err);
/* Same compress, but the LIBRARY lays the streams out back to back in out_base[0 .. out_cap) and reports where:
 * out_offs receives count+1 entries (out_offs[count] = total bytes). A caller cannot know compressed sizes in
 * advance, so this is the form whose drain is one D2H copy per wave; sb_max_compress_len(len) summed over the
 * units is always enough capacity. Units are one block each (in_lens[i] <= 65536, else TooBig). */
int sb_compress_batch_host_packed(const uint8_t* in_base, const uint64_t* in_offs, const uint32_t* in_lens,
                                  uint8_t* out_base, uint64_t out_cap, uint64_t* out_offs, uint32_t* out_lens,
                                  size_t count, sb_error* err);

/* ---- batched device API: device pointers, stream ordered ------------------
 * The kernels' native interface (and what bench.py's `value` times). All
 * pointers are device pointers; `stream` is a cudaStream_t passed as void*
 * (NULL is the legacy default stream, exactly as in the CUDA runtime).
 * Addressing is base + i*stride (uniform) -- or per-unit pointer arrays when
 * in_ptrs/out_ptrs are non-NULL. in_lens/out_caps NULL => the uniform value. */
typedef struct sb_batch {
    const uint8_t* const* in_ptrs;  const uint8_t* in_base;  uint64_t in_stride;
    const uint32_t* in_lens;        uint32_t in_len_uniform;
    uint8_t* const* out_ptrs;       uint8_t* out_base;       uint64_t out_stride;
    const uint32_t* out_caps;       uint32_t out_cap_uniform;
    uint32_t* out_lens;             /* device, count entries (required)      */
    sb_error* statuses;             /* device, count entries (decode; may be NULL for encode) */
    uint32_t count;
} sb_batch;

/* Each unit is ONE BLOCK: at most 65536 bytes, and its output slot must hold
 * sb_max_compress_len(len) bytes; the unit becomes one raw stream exactly as
 * Encoder::compress would produce it (one parser/emitter warp pair per unit, 12
 * pairs per SM). A unit that breaks either limit is skipped: out_lens[i] = 0 and,
 * when `statuses` is given, TooBig{given,max=65536} / BufferTooSmall{given,min}
 * (src/compress.rs:104-117); uniform lengths/caps are also checked on the host.
 * Larger inputs go through sb_compress / sb_frame_encode_device, which cut them
 * into blocks. Compress launches share a per-device scratch (event rings,
 * L2-resident hash tables, work counter): launches issued on different streams
 * of one device are ordered after each other on the device. */
int sb_compress_batch_device(const sb_batch* batch, void* stream, sb_error* err);
/* Each unit is one raw stream; statuses[i] carries the reference's error. */
int sb_decompress_batch_device(const sb_batch* batch, void* stream, sb_error* err);
/* Masked CRC-32C of each unit (frame chunks): out_lens[i] receives the CRC. */
int sb_crc32c_masked_batch_device(const sb_batch* batch, void* stream, sb_error* err);

/* ---- frame format (snap::write::FrameEncoder / snap::read::FrameDecoder) --
 * One-shot forms over host memory. sb_frame_encode(in) produces exactly the
 * bytes of `FrameEncoder::new(vec![]).write_all(in); into_inner()`
 * (src/write.rs:123-192): stream identifier + one chunk per <=65536-byte slice;
 * empty input => empty output. */
size_t sb_frame_max_len(size_t n);
int sb_frame_encode(const uint8_t* in, size_t n, uint8_t* out, size_t cap, size_t* out_n, sb_error* err);
/* The chunk loop of write::Inner::write alone (src/write.rs:171-190): chunks for
 * `in` with (include_ident=1) or without the leading stream identifier -- what
 * a streaming FrameEncoder calls for every buffer it hands down. */
int sb_frame_encode_ex(const uint8_t* in, size_t n, uint8_t* out, size_t cap, size_t* out_n, int include_ident, sb_error* err);
/* `FrameDecoder::new(in).read_to_end()` (src/read.rs:104-239): pass out=NULL to
 * size the output (*out_n). Errors carry the reference's variant/payload. */
int sb_frame_decode(const uint8_t* in, size_t n, uint8_t* out, size_t cap, size_t* out_n, sb_error* err);

/* Device-resident frame encode of n bytes at d_in (device) into d_out (device,
 * cap >= sb_frame_max_len(n)); *out_n (host) = stream length. include_ident=0
 * omits the 10-byte stream identifier (ranks > 0 of a sharded stream).
 * Convenience form: pooled scratch, waits for the result. */
int sb_frame_encode_device(const uint8_t* d_in, uint64_t n, uint8_t* d_out, uint64_t cap,
                           int include_ident, uint64_t* out_n, void* stream, sb_error* err);

/* ---- stream-ordered frame calls with caller-provided scratch ---------------
 * No allocation, no host synchronisation (n > 0): every kernel of the call is
 * enqueued on `stream` and the outcome is written to *d_result (device memory).
 *   scratch: device memory of at least sb_frame_{encode,decode}_scratch_bytes(..).
 * Encode (src/write.rs:165-192 + src/frame.rs:62-104): K1 compresses every chunk
 * and leaves its masked CRC-32C beside it, a two-level scan places the chunks,
 * one gather writes headers + bodies. d_chunk_offs (optional, device, nchunks+1
 * entries) receives the offset of every chunk header in d_out and the total --
 * the chunk index sb_frame_decode_device_ws accepts. */
uint64_t sb_frame_encode_scratch_bytes(uint64_t n);
int sb_frame_encode_device_ws(const uint8_t* d_in, uint64_t n, uint8_t* d_out, uint64_t cap, int include_ident,
                              uint64_t* d_chunk_offs, sb_frame_result* d_result, void* scratch, uint64_t scratch_bytes,
                              void* stream, sb_error* err);
/* Decode (read::FrameDecoder, src/read.rs:104-239) of a frame stream in device
 * memory. With d_chunk_offs/nchunks (the encoder's index; d_chunk_offs[nchunks]
 * = n) the chunk headers are parsed in parallel; without it (or when the index
 * does not describe a clean run of data chunks) one thread walks the headers in
 * stream order exactly like the reference's reader. Then one warp per chunk:
 * raw decode (K2) or copy, masked CRC-32C of the produced bytes against the
 * header. d_result: first error in stream order + bytes produced before it.
 *   flags bit0: no stream identifier expected (a rank's fragment of a sharded stream)
 *   max_chunks: capacity of the chunk table carved from scratch (SB_E_INVALID{a=max_chunks,b=1} if exceeded) */
uint64_t sb_frame_decode_scratch_bytes(uint32_t max_chunks);
int sb_frame_decode_device_ws(const uint8_t* d_in, uint64_t n, uint8_t* d_out, uint64_t cap,
                              const uint64_t* d_chunk_offs, uint32_t nchunks, uint32_t flags,
                              sb_frame_result* d_result, void* scratch, uint64_t scratch_bytes, uint32_t max_chunks,
                              void* stream, sb_error* err);
/* Convenience form: pooled scratch, waits and returns the result on the host. */
int sb_frame_decode_device(const uint8_t* d_in, uint64_t n, uint8_t* d_out, uint64_t cap,
                           const uint64_t* d_chunk_offs, uint32_t nchunks, uint32_t flags,
                           sb_frame_result* result, void* stream, sb_error* err);

/* ---- batches of raw streams of any size (units above 64KB) ----------------
 * Unit i = d_in_ptrs[i][0 .. d_in_lens[i]) (device pointer and length arrays); each becomes exactly
 * Encoder::compress(unit) (src/compress.rs:99-154): one varint of the unit's length, then its 64KB blocks.
 * The library lays the streams out back to back in d_out[0 .. cap) and reports where: d_out_offs receives count+1
 * entries (d_out_offs[count] = total bytes). The whole batch is one launch sequence on `stream` -- no allocation, no
 * host synchronisation; the outcome lands in *d_result (device): status, bytes = total, nchunks = 64KB blocks.
 *   total_in: a host-side upper bound on the sum of the lengths; it sizes the scratch and the launch
 *     (units + total_in/65536 block slots). A sum above it is SB_E_INVALID{a=sum, b=total_in} and nothing is written.
 *   A unit with sb_max_compress_len(len) == 0 is refused with TooBig{given=len, max=2^32-1} and gets an empty
 *     stream (d_out_offs[i+1] == d_out_offs[i]); the other units are compressed. d_result reports the first such unit.
 *   Output larger than cap: nothing is written, d_result (and every status) is BufferTooSmall{given=cap, min=total};
 *     the offsets are still reported, so a caller can size a retry. sum(sb_max_compress_len(len)) is always enough.
 *   d_statuses (may be NULL): per unit Ok / TooBig, or the call's failure.
 *   scratch: device memory of at least sb_compress_streams_scratch_bytes(count, total_in). */
uint64_t sb_compress_streams_scratch_bytes(uint32_t count, uint64_t total_in);
int sb_compress_streams_device_ws(const uint8_t* const* d_in_ptrs, const uint64_t* d_in_lens, uint32_t count,
                                  uint64_t total_in, uint8_t* d_out, uint64_t cap, uint64_t* d_out_offs,
                                  sb_error* d_statuses, sb_frame_result* d_result,
                                  void* scratch, uint64_t scratch_bytes, void* stream, sb_error* err);
/* Host buffers: unit i = in_base[in_offs[i] .. +in_lens[i]), streams packed back to back into out_base[0 .. out_cap)
 * with out_offs[0..count] reported (count+1 entries). Pipelined waves like sb_compress_batch_host_packed; a unit larger
 * than a wave gets a wave of its own. Any unit with sb_max_compress_len(len) == 0 fails the call up front with TooBig
 * for the first such unit. For sb_reserve, a wave of this call counts its units plus the 64KB blocks they span. */
int sb_compress_streams_host_packed(const uint8_t* in_base, const uint64_t* in_offs, const uint64_t* in_lens, size_t count,
                                    uint8_t* out_base, uint64_t out_cap, uint64_t* out_offs, sb_error* err);
/* Unit i = one raw stream d_in_ptrs[i][0 .. d_in_lens[i]) (device). Output sizes come from the streams' own varint
 * headers (0 for an unusable header) and are laid out back to back in d_out (d_out_offs: count+1 entries);
 * d_statuses[i] (required) = Decoder::decompress's result for unit i (src/decompress.rs:75-95), decoded by K2 exactly
 * as sb_decompress_batch_device does; a stream longer than 2^32-1 bytes is SB_E_INVALID for that unit, as in
 * sb_decompress. If the total exceeds cap no unit is decoded, and d_result and every status are
 * BufferTooSmall{given=cap, min=total}. Otherwise d_result = the first failing unit's status (or Ok), bytes = total,
 * nchunks = count. Stream ordered, no allocation, no host synchronisation.
 *   scratch: device memory of at least sb_decompress_streams_scratch_bytes(count). */
uint64_t sb_decompress_streams_scratch_bytes(uint32_t count);
int sb_decompress_streams_device_ws(const uint8_t* const* d_in_ptrs, const uint64_t* d_in_lens, uint32_t count,
                                    uint8_t* d_out, uint64_t cap, uint64_t* d_out_offs, sb_error* d_statuses,
                                    sb_frame_result* d_result, void* scratch, uint64_t scratch_bytes,
                                    void* stream, sb_error* err);

/* ---- resources -------------------------------------------------------------
 * The host entry points keep grow-only per-device pools (device staging, pinned
 * descriptors, streams, events): the first calls size them, the steady state
 * allocates nothing. sb_reserve sizes them ahead of time for waves of up to
 * wave_units units / wave_in_bytes input / wave_out_bytes output;
 * sb_alloc_count() = allocations + event/stream creations since load (a caller
 * can assert it stays flat). First use of a device is thread safe. */
int sb_reserve(size_t wave_units, size_t wave_in_bytes, size_t wave_out_bytes, sb_error* err);
uint64_t sb_alloc_count(void);
/* Pin the calling thread to the CPUs of the NUMA node of `device` (so that pinned staging it allocates afterwards
 * and its copies stay on the near socket). Returns the node, or -1 when the topology is not exposed. */
int sb_bind_host_thread_to_device_numa(int device);

/* ---- libsnappy-compatible C API ------------------------------------------
 * The four functions the reference's `snappy-cpp` crate binds
 * (snappy-cpp/src/lib.rs:66-88, snappy-c.h): linking the reference's test/ and
 * bench/ crates with `--features cpp` against this library runs their
 * cross-implementation tests on the GPU codec. 0 = SNAPPY_OK, 1 = INVALID_INPUT,
 * 2 = BUFFER_TOO_SMALL. */
int snappy_compress(const char* input, size_t input_length, char* compressed, size_t* compressed_length);
int snappy_uncompress(const char* compressed, size_t compressed_length, char* uncompressed, size_t* uncompressed_length);
size_t snappy_max_compressed_length(size_t source_length);
int snappy_uncompressed_length(const char* compressed, size_t compressed_length, size_t* result);

/* ---- misc ---------------------------------------------------------------- */
/* Number of kernel launches issued by this library since load (bench.py's
 * gpu_launches evidence). */
uint64_t sb_launch_count(void);
/* Device-side helper used by tests/bench: fills unit i (i < count) at
 * d_out + i*stride with text[off_i .. off_i+len), off_i = ((first+i)*mul) % (text_len-len). */
int sb_generate_blocks_device(const uint8_t* d_text, uint64_t text_len, uint8_t* d_out, uint64_t stride,
                              uint32_t len, uint64_t first, uint64_t count, uint64_t mul, void* stream, sb_error* err);
const char* sb_version(void);

#ifdef __cplusplus
}
#endif
#endif
