/* swcgpu.h — C ABI of libswcgpu.so: B200 (sm_100a) batched decompression engine that replaces the decode hot path of
 * tsolomko/SWCompression 4.9.0 (pure Swift).  The reference has no FFI layer; its "operator API" is the set of Swift
 * static functions cited next to each entry point below.  A Swift / ctypes shim keeps those names and signatures and
 * routes the bodies through this header (see INTEGRATION.md for the module map + Swift binding).
 *
 * Conventions
 *   - extern "C", no exceptions, no torch types.  Return value / status[] entries are `enum swc_status` codes
 *     (include/swc_status.h): 0 = OK, <base>+k = k-th case of the corresponding Swift error enum.
 *   - "payload-carrying" errors (wrongCRC(Data), checksumMismatch([Data]), wrongAdler32(Data), wrongCheck([Data]))
 *     return the status AND the decoded bytes, as the Swift errors do.
 *   - single-unit calls take HOST pointers, run on the current device and return a buffer allocated with swc_alloc
 *     (caller frees with swc_free).  *_batch calls take DEVICE pointers and are asynchronous on `cuda_stream`.
 *     *_batch_host calls take HOST pointers and include the host<->device copies (blocking).
 *   - every decode reports how much input it consumed, because the reference's wrappers keep parsing after the
 *     payload (GzipArchive.swift:88-94, ZlibArchive.swift:31-37, ZipContainer.swift:74-79, XZBlock.swift:78-82).
 *   - there is no CPU fallback: without a CUDA device every call returns SWC_ERR_NO_DEVICE.
 *   - threading: like the reference, the library may be called from any number of host threads.  Mutable state is one lazily
 *     created context per device (scratch arenas, staging streams, pinned result buffers) behind a per-device mutex: calls on
 *     the same device are serialised, calls on different devices run concurrently.  The asynchronous *_batch calls only hold
 *     the mutex while they enqueue; when several of them are in flight on one device at the same time each needs its own
 *     `scratch` (the NULL = library-pool form shares one arena).
 *   - multi-member / multi-stream / multi-block archives are discovered up front and decoded as one batch; the
 *     reference's in-order walk is kept as the validator, so results and errors are those of the sequential loop.
 *
 * Batch layout (all arrays have n entries, device memory):
 *   unit i reads  in_base[in_off[i] .. in_off[i]+in_len[i])           (any byte alignment; 16-B aligned is fastest)
 *   unit i writes out_base[out_off[i] .. out_off[i]+out_cap[i])       (out_off[i] must be a multiple of 16)
 *   results: out_len[i] (bytes produced; on SWC_ERR_OUTPUT_OVERFLOW the size required), consumed[i], status[i].
 *   Output regions must not overlap.  Bytes between out_len[i] and out_cap[i] are scratch and may be clobbered.
 */
#ifndef SWCGPU_H
#define SWCGPU_H

#include <stddef.h>
#include <stdint.h>
#include "swc_status.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- library / memory ---- */
int32_t     swc_device_count(void);
int32_t     swc_set_device(int32_t device);
const char *swc_last_error_string(void);               /* thread-local text for the last SWC_ERR_CUDA */
const char *swc_status_name(int32_t status);           /* "DeflateError.wrongSymbol", ... */
void       *swc_alloc(size_t bytes);                   /* host memory for single-unit results */
void        swc_free(void *p);
void       *swc_alloc_pinned(size_t bytes);            /* page-locked host memory for *_batch_host callers */
void        swc_free_pinned(void *p);
uint64_t    swc_kernel_launches(void);                 /* number of CUDA kernels this library has launched so far */
int32_t     swc_release_scratch(void);                 /* free the per-device scratch pools */
/* measurement aid: while enabled, every batched call drops CUDA events on its stream before/between/after its kernels;
 * swc_timing_collect (after a stream sync) returns the elapsed ms of each interval in launch order */
void        swc_timing_enable(int32_t on);
int32_t     swc_timing_collect(float *ms, int32_t max_n);

/* ---- Deflate ------------------------------------------------------------------------------------------------
 * Deflate.decompress(data:)                Sources/Deflate/Deflate.swift:24-28
 * Deflate.decompress(_: LsbBitReader)      Sources/Deflate/Deflate.swift:30-249   (start_bit/consumed_bits form) */
int32_t swc_deflate_decompress(const uint8_t *in, size_t in_len, size_t start_bit,
                               uint8_t **out, size_t *out_len, size_t *consumed_bits);
/* scratch the batched call needs for `out_capacity_total` bytes of output buffer */
size_t  swc_deflate_batch_scratch_bytes(uint64_t n, uint64_t out_capacity_total);
/* Device batch: every out_off[i] must be a multiple of 16 (the kernels store whole 8- and 16-byte words inside
 * [out_off[i], out_off[i] + out_cap[i])); out_base itself must be 16-byte aligned. in_off may have any alignment. */
int32_t swc_deflate_decompress_batch(const uint8_t *in_base, const uint64_t *in_off, const uint64_t *in_len,
                                     const uint8_t *start_bits /* n entries 0..7, or NULL */,
                                     uint8_t *out_base, const uint64_t *out_off, const uint64_t *out_cap,
                                     uint64_t out_capacity_total,
                                     uint64_t *out_len, uint64_t *consumed_bits, int32_t *status,
                                     uint64_t n, void *scratch, size_t scratch_bytes /* NULL,0 = library pool */,
                                     void *cuda_stream);
int32_t swc_deflate_decompress_batch_host(const uint8_t *in_base, const uint64_t *in_off, const uint64_t *in_len,
                                          uint64_t in_total,
                                          uint8_t *out_base, const uint64_t *out_off, const uint64_t *out_cap,
                                          uint64_t out_capacity_total,
                                          uint64_t *out_len, uint64_t *consumed_bits, int32_t *status, uint64_t n);

/* ---- LZ4 ----------------------------------------------------------------------------------------------------
 * LZ4.decompress(data:)                                   Sources/LZ4/LZ4.swift:49-51
 * LZ4.decompress(data:dictionary:dictionaryID:)           Sources/LZ4/LZ4.swift:73-91
 * LZ4.multiDecompress(data:dictionary:dictionaryID:)      Sources/LZ4/LZ4.swift:116-146
 * LZ4.process(block:_:) (private raw-block decoder)       Sources/LZ4/LZ4.swift:332-413  -> *_block_batch */
int32_t swc_lz4_decompress(const uint8_t *in, size_t in_len, const uint8_t *dict /* NULL = nil */, size_t dict_len,
                           int32_t has_dict_id, uint32_t dict_id,
                           uint8_t **out, size_t *out_len, size_t *consumed_bytes);
/* frames are concatenated into *out; frame_ends[i] = end offset of frame i; returns the number of frames in *n_frames */
int32_t swc_lz4_multi_decompress(const uint8_t *in, size_t in_len, const uint8_t *dict, size_t dict_len,
                                 int32_t has_dict_id, uint32_t dict_id,
                                 uint8_t **out, size_t *out_len, size_t **frame_ends, size_t *n_frames);
/* raw blocks; dict (device pointer, may be NULL) is the prefix every block may reference (independent-block mode).
 * As for Deflate, every out_off[i] must be a multiple of 16 and out_base 16-byte aligned: the kernels store 16-byte words. */
int32_t swc_lz4_block_decompress_batch(const uint8_t *in_base, const uint64_t *in_off, const uint64_t *in_len,
                                       const uint8_t *dict, uint64_t dict_len,
                                       uint8_t *out_base, const uint64_t *out_off, const uint64_t *out_cap,
                                       uint64_t *out_len, int32_t *status, uint64_t n, void *cuda_stream);
int32_t swc_lz4_block_decompress_batch_host(const uint8_t *in_base, const uint64_t *in_off, const uint64_t *in_len,
                                            uint64_t in_total,
                                            uint8_t *out_base, const uint64_t *out_off, const uint64_t *out_cap,
                                            uint64_t out_capacity_total,
                                            uint64_t *out_len, int32_t *status, uint64_t n);

/* ---- BZip2 --------------------------------------------------------------------------------------------------
 * BZip2.decompress(data:)            Sources/BZip2/BZip2.swift:22-26
 * BZip2.multiDecompress(data:)       Sources/BZip2/BZip2.swift:40-48
 * BZip2.decompress(_: MsbBitReader)  Sources/BZip2/BZip2.swift:50-95 */
int32_t swc_bzip2_decompress(const uint8_t *in, size_t in_len, size_t start_bit,
                             uint8_t **out, size_t *out_len, size_t *consumed_bits);
int32_t swc_bzip2_multi_decompress(const uint8_t *in, size_t in_len,
                                   uint8_t **out, size_t *out_len, size_t **stream_ends, size_t *n_streams);
/* one .bz2 stream per unit */
int32_t swc_bzip2_decompress_batch(const uint8_t *in_base, const uint64_t *in_off, const uint64_t *in_len,
                                   uint8_t *out_base, const uint64_t *out_off, const uint64_t *out_cap,
                                   uint64_t *out_len, uint64_t *consumed_bits, int32_t *status,
                                   uint64_t n, void *cuda_stream);

/* ---- LZMA / LZMA2 -------------------------------------------------------------------------------------------
 * LZMA.decompress(data:)                                   Sources/LZMA/LZMA.swift:25-34
 * LZMA.decompress(data:properties:uncompressedSize:)       Sources/LZMA/LZMA.swift:56-61
 * LZMA2.decompress(data:)                                  Sources/LZMA2/LZMA2.swift:25-30
 * LZMA2.decompress(_:_:) (reader + dict byte, used by XZ)  Sources/LZMA2/LZMA2.swift:32-36 */
int32_t swc_lzma_decompress(const uint8_t *in, size_t in_len, uint8_t **out, size_t *out_len, size_t *consumed_bytes);
int32_t swc_lzma_decompress_raw(const uint8_t *in, size_t in_len, int32_t lc, int32_t lp, int32_t pb,
                                int64_t dictionary_size, int64_t uncompressed_size /* <0 = nil */,
                                uint8_t **out, size_t *out_len, size_t *consumed_bytes);
int32_t swc_lzma2_decompress(const uint8_t *in, size_t in_len, uint8_t **out, size_t *out_len, size_t *consumed_bytes);
/* one raw LZMA stream per unit (the ZIP / 7-Zip form, LZMA.decompress(data:properties:uncompressedSize:), LZMA.swift:56-61):
 * props[i] = lc | lp << 8 | pb << 16, dict_size[i] as in LZMAProperties, uncompressed_size[i] < 0 = nil (end marker).
 * lc + lp must be <= 4 in the batched form (the literal coders live in shared memory); other units report SWC_ERR_UNSUPPORTED. */
int32_t swc_lzma_decompress_batch(const uint8_t *in_base, const uint64_t *in_off, const uint64_t *in_len,
                                  const uint32_t *props, const int64_t *dict_size, const int64_t *uncompressed_size,
                                  uint8_t *out_base, const uint64_t *out_off, const uint64_t *out_cap,
                                  uint64_t *out_len, uint64_t *consumed_bytes, int32_t *status,
                                  uint64_t n, void *cuda_stream);
/* one raw LZMA2 stream per unit; dict_bytes[i] is the XZ filter property byte */
int32_t swc_lzma2_decompress_batch(const uint8_t *in_base, const uint64_t *in_off, const uint64_t *in_len,
                                   const uint8_t *dict_bytes,
                                   uint8_t *out_base, const uint64_t *out_off, const uint64_t *out_cap,
                                   uint64_t *out_len, uint64_t *consumed_bytes, int32_t *status,
                                   uint64_t n, void *cuda_stream);

/* ---- wrappers -----------------------------------------------------------------------------------------------
 * GzipArchive.unarchive(archive:) / multiUnarchive   Sources/GZip/GzipArchive.swift:38-77
 * ZlibArchive.unarchive(archive:)                     Sources/Zlib/ZlibArchive.swift:25-42
 * XZArchive.unarchive(archive:) / splitUnarchive      Sources/XZ/XZArchive.swift:27-88 */
/* GzipHeader(archive:) / GzipHeader.init(_: LsbBitReader)   Sources/GZip/GzipHeader.swift:10-60, 63-199
 * ZlibHeader(archive:)                                       Sources/Zlib/ZlibHeader.swift:10-40, 42-93
 * Pure framing: these two calls need no device.  String / extra-field bytes are returned as offsets into `in`
 * (file name and comment are ISO-Latin-1, GzipHeader.swift:160,178; extra fields are the SI1 SI2 LEN data... records). */
typedef struct swc_gzip_header {
    int32_t  compression_method;     /* CompressionMethod.deflate = 8 */
    uint32_t modification_time;      /* MTIME; 0 = nil */
    uint8_t  os_type;                /* raw OS byte (FileSystemType(rawOsType)) */
    uint8_t  is_text_file;           /* FTEXT */
    uint8_t  has_file_name, has_comment;
    size_t   file_name_off, file_name_len;     /* without the terminating zero */
    size_t   comment_off, comment_len;
    size_t   extra_off, extra_len;             /* the XLEN bytes behind the XLEN field (0,0 without FEXTRA) */
    size_t   header_len;                       /* bytes from the member start to the first Deflate byte */
} swc_gzip_header;
typedef struct swc_zlib_header {
    int32_t compression_method;      /* always 8 */
    int32_t compression_level;       /* ZlibHeader.CompressionLevel raw value 0..3 */
    int32_t window_size;             /* 1 << (CINFO + 8) */
    size_t  header_len;              /* 2, or 6 with FDICT */
} swc_zlib_header;
int32_t swc_gzip_header_parse(const uint8_t *in, size_t in_len, size_t member_off, swc_gzip_header *hdr);
int32_t swc_zlib_header_parse(const uint8_t *in, size_t in_len, swc_zlib_header *hdr);
int32_t swc_gzip_unarchive(const uint8_t *in, size_t in_len, uint8_t **out, size_t *out_len, size_t *consumed_bytes);
/* GzipArchive.multiUnarchive -> [Member] (GzipArchive.swift:13-22, 52-77): as swc_gzip_multi_unarchive, plus the offset of
 * every member inside `in` (n_members + 1 entries, the last one = where the walk stopped) so the caller can rebuild
 * Member.header with swc_gzip_header_parse.  On SWC_GZIP_WRONG_CRC the failing member is the last one returned. */
int32_t swc_gzip_multi_unarchive_members(const uint8_t *in, size_t in_len,
                                         uint8_t **out, size_t *out_len, size_t **member_ends, size_t **member_in_off,
                                         size_t *n_members);
int32_t swc_gzip_multi_unarchive(const uint8_t *in, size_t in_len,
                                 uint8_t **out, size_t *out_len, size_t **member_ends, size_t *n_members);
int32_t swc_zlib_unarchive(const uint8_t *in, size_t in_len, uint8_t **out, size_t *out_len);
int32_t swc_xz_unarchive(const uint8_t *in, size_t in_len, uint8_t **out, size_t *out_len);
int32_t swc_xz_split_unarchive(const uint8_t *in, size_t in_len,
                               uint8_t **out, size_t *out_len, size_t **stream_ends, size_t *n_streams);

/* ---- ZIP container -------------------------------------------------------------------------------------------
 * ZipContainer.open(container:) -> [ZipEntry]     Sources/ZIP/ZipContainer.swift:43-58 (entry data: getEntryData :62-125)
 * ZipContainer.info(container:) -> [ZipEntryInfo] Sources/ZIP/ZipContainer.swift:132-134 (host only, no device needed)
 * One entry per central-directory record, in its order.  All Deflate / BZip2 / LZMA entries of a container are decoded as
 * one batch each; errors (and the entries returned with SWC_ZIP_WRONG_CRC: the failing one last) are those of the reference's
 * entry-by-entry loop.  `*out` holds every entry's data at [data_off, data_off + data_len); free both results with swc_free. */
typedef struct swc_zip_entry {
    uint64_t name_off, name_len;         /* ZipEntryInfo.name: bytes inside the container (central directory) */
    uint64_t comment_off, comment_len;   /* ZipEntryInfo.comment */
    uint64_t data_off, data_len;         /* ZipEntry.data inside *out (0, 0 for directories and for swc_zip_info) */
    uint64_t size;                       /* ZipEntryInfo.size */
    uint32_t crc;                        /* ZipEntryInfo.crc */
    uint32_t external_attrs;             /* externalFileAttributes: permissions = (attrs & 0x0FFF0000) >> 16, dosAttributes = attrs & 0xFF */
    uint16_t method;                     /* raw compression method: 0 copy, 8 deflate, 12 bzip2, 14 lzma, else .other */
    uint16_t version_made_by;            /* FileSystemType(versionMadeBy) */
    uint16_t internal_attrs;             /* isTextFile = internal_attrs & 1 */
    uint16_t dos_time, dos_date;         /* native modification time */
    uint8_t  is_directory;               /* ZipEntryInfo.type == .directory */
    uint8_t  utf8;                       /* general purpose bit 11: name / comment are UTF-8 (else CP437 unless the bytes need UTF-8) */
} swc_zip_entry;
int32_t swc_zip_open(const uint8_t *in, size_t in_len, uint8_t **out, size_t *out_len, swc_zip_entry **entries, size_t *n_entries);
int32_t swc_zip_info(const uint8_t *in, size_t in_len, swc_zip_entry **entries, size_t *n_entries);

/* ---- checks (device-side, used by the wrappers; exposed for the shim and the tests) ---------------------------
 * CheckSums.crc32 / bzip2crc32 / crc64 / adler32   Sources/Common/CheckSums.swift:12-57
 * XxHash32.hash                                     Sources/LZ4/XxHash32.swift:24-83
 * Sha256.hash                                       Sources/XZ/Sha256.swift */
int32_t swc_crc32(const uint8_t *in, size_t n, uint32_t *result);
int32_t swc_bzip2_crc32(const uint8_t *in, size_t n, uint32_t *result);
int32_t swc_crc64(const uint8_t *in, size_t n, uint64_t *result);
int32_t swc_adler32(const uint8_t *in, size_t n, uint32_t *result);
int32_t swc_xxh32(const uint8_t *in, size_t n, uint32_t *result);
int32_t swc_sha256(const uint8_t *in, size_t n, uint8_t digest[32]);
/* batched epilogues on DEVICE buffers (asynchronous on `cuda_stream`): one result per unit in_base[off[i] .. off[i]+len[i]).
 * `status` may be NULL; units whose status[i] != 0 are not read (their result is 0). */
int32_t swc_crc32_batch(const uint8_t *in_base, const uint64_t *off, const uint64_t *len, const int32_t *status,
                        uint32_t *result, uint64_t n, void *cuda_stream);
int32_t swc_xxh32_batch(const uint8_t *in_base, const uint64_t *off, const uint64_t *len,
                        uint32_t *result, uint64_t n, void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* SWCGPU_H */
