/*
 * dtb200_io.h -- C ABI of libdtb200_io.so: the raster files either side of the descriptor path
 * (SURVEY.md section 8 f3).
 *
 * The reference reads its inputs and writes its class map with rasterio / GDAL
 * (Example/example.py:33-39, :106, :201-217): single-band GeoTIFFs, LZW-compressed 128 x 128 tiles
 * (12_dem / 12_fdr / 12_fac) or plain strips (WB_12_100y, output/hand_class), float32 / uint8, with the
 * georeferencing in the ModelPixelScale / ModelTiepoint / GeoKey tags and the nodata value in GDAL_NODATA.
 * This library is a native, multi-threaded codec for exactly that family of files (classic TIFF and
 * BigTIFF -- a 40 000 x 40 000 float32 raster is 6.4 GB): a reader that decodes row blocks into
 * caller-owned (pinned) host memory so the blocks can go to the device while the next ones are being
 * decoded, and a writer that takes row blocks as they come back.  It is host code; it has no CUDA in it
 * and does no arithmetic of the descriptor path.
 *
 * Conventions: plain pointers and sizes, int status (0 = ok, negative = error, dtbio_last_error() holds
 * the text for the calling thread); handles are created by *_open / *_create and freed by dtbio_close;
 * rasters are row-major, band 1 only (SamplesPerPixel == 1, what every file of the reference is).
 */
#ifndef DTB200_IO_H
#define DTB200_IO_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DTBIO_ABI_VERSION 1

enum {
    DTBIO_OK = 0,
    DTBIO_ERR_INVALID = -1,     /* bad argument                                         */
    DTBIO_ERR_IO = -2,          /* open / read / write failed                           */
    DTBIO_ERR_FORMAT = -3,      /* not a TIFF, or a damaged one                         */
    DTBIO_ERR_UNSUPPORTED = -4, /* a TIFF this codec does not read (multi-band, JPEG ...) */
    DTBIO_ERR_ORDER = -5        /* writer: row block not on a chunk boundary             */
};

/* element types (the NumPy dtypes rasterio hands back, example.py:33-39) */
enum {
    DTBIO_U8 = 0, DTBIO_I8 = 1, DTBIO_U16 = 2, DTBIO_I16 = 3, DTBIO_U32 = 4, DTBIO_I32 = 5,
    DTBIO_U64 = 6, DTBIO_I64 = 7, DTBIO_F32 = 8, DTBIO_F64 = 9
};

/* TIFF compression codes understood (tag 259) */
enum { DTBIO_COMP_NONE = 1, DTBIO_COMP_LZW = 5, DTBIO_COMP_DEFLATE = 8, DTBIO_COMP_PACKBITS = 32773 };

typedef struct dtbio_info {
    int64_t rows, cols;       /* ImageLength, ImageWidth                                          */
    int32_t dtype;            /* DTBIO_*                                                          */
    int32_t compression;      /* tag 259 (32946, old deflate, is reported as DTBIO_COMP_DEFLATE)  */
    int32_t predictor;        /* tag 317: 1 none, 2 horizontal differencing, 3 floating point     */
    int32_t tile_rows;        /* TileLength, 0 for a striped file                                  */
    int32_t tile_cols;        /* TileWidth, 0 for a striped file                                   */
    int32_t rows_per_strip;   /* RowsPerStrip, 0 for a tiled file                                  */
    int32_t bigtiff;          /* 1 = BigTIFF (8-byte offsets)                                      */
    int32_t big_endian;       /* 1 = 'MM' file (reader swaps; the writer always writes 'II')       */
    int32_t has_nodata;       /* GDAL_NODATA (tag 42113) present and numeric                       */
    int32_t has_georef;       /* ModelPixelScale + ModelTiepoint present                           */
    double nodata;
    double pixel_scale[3];    /* tag 33550                                                         */
    double tiepoint[6];       /* tag 33922 (first tie point)                                       */
} dtbio_info;

typedef struct dtbio_reader dtbio_reader;
typedef struct dtbio_writer dtbio_writer;

int dtbio_abi_version(void);
const char *dtbio_error_string(int code);
const char *dtbio_last_error(void);          /* detail of the calling thread's last failure */
int64_t dtbio_dtype_size(int dtype);

/* ---- reader: replaces rasterio.open(path).read(1) (example.py:33-39, :106) ---------------------- */
int dtbio_open(const char *path, dtbio_reader **out);
int dtbio_get_info(const dtbio_reader *r, dtbio_info *info);
/* Raw access to a tag of the first IFD (values converted to host byte order, ASCII as stored).
 * *type is the TIFF field type (1 BYTE, 2 ASCII, 3 SHORT, 4 LONG, 12 DOUBLE, 16 LONG8 ...), *count the
 * number of values, *data a pointer owned by the reader.  Returns DTBIO_ERR_INVALID if absent.
 * Used for the georeferencing tags 33550, 33922, 34264, 34735, 34736, 34737, 42112, 42113. */
int dtbio_get_tag(const dtbio_reader *r, int tag, int *type, int64_t *count, const void **data);
/* Decode rows [row0, row0 + nrows) into dst (host memory, typically pinned; row i of the block starts at
 * dst + i * dst_stride_bytes, dst_stride_bytes >= cols * element size).  The tiles / strips that overlap
 * the block are decoded by `threads` worker threads (<= 0: one per hardware thread, at most 64). */
int dtbio_read_rows(dtbio_reader *r, int64_t row0, int64_t nrows, void *dst, int64_t dst_stride_bytes, int threads);

/* ---- writer: replaces rasterio.open(path, "w", **meta).write(...) (example.py:201-217) ---------- */
/* Only rows, cols, dtype, compression, predictor, tile_rows, tile_cols, rows_per_strip, bigtiff are read
 * from *info (tile_rows == 0: strips of rows_per_strip rows, 0 -> about 8 KB like GDAL; bigtiff: 1 force,
 * 0 = only when the uncompressed raster would not fit a classic file). */
int dtbio_create(const char *path, const dtbio_info *info, dtbio_writer **out);
/* the layout the writer settled on (default strip height, BigTIFF decision) */
int dtbio_writer_info(const dtbio_writer *w, dtbio_info *info);
/* add / replace a tag written with the IFD at close (the georeferencing tags, GDAL_NODATA, ...);
 * `data` holds `count` values of TIFF field type `type` in host byte order and is copied */
int dtbio_set_tag(dtbio_writer *w, int tag, int type, int64_t count, const void *data);
/* Encode rows [row0, row0 + nrows): row0 must be a multiple of the chunk height (tile_rows or
 * rows_per_strip) and the block must end on one or at the last row; blocks may arrive in any order and
 * each chunk exactly once. */
int dtbio_write_rows(dtbio_writer *w, int64_t row0, int64_t nrows, const void *src, int64_t src_stride_bytes, int threads);
/* Chunks encoded elsewhere (dtb_tiff_encode_chunks, include/dtb200.h): chunk first_chunk + i is the sizes[i] bytes at
 * blob + offsets[i]; the blob (blob_bytes long) is written with one call and the chunk table points into it.
 * The streams must match the writer's compression / predictor / chunk geometry. */
int dtbio_write_encoded(dtbio_writer *w, int64_t first_chunk, int64_t n_chunks, const void *blob, int64_t blob_bytes,
                        const int64_t *offsets, const int64_t *sizes);
/* ---- one file, several writers (a row-band run: every rank writes the chunks it encoded) ----------
 * The main writer (dtbio_create) owns the file: it writes the header and the IFD at close, and removes the file if a
 * chunk is missing then.  dtbio_open_part opens the file the main writer created: it checks *info exactly as
 * dtbio_create does and settles the same layout and BigTIFF decision, but never truncates the file; closing it only
 * closes its descriptor (no header, no IFD, no unlink).  A part writer takes dtbio_write_encoded_at only.
 * dtbio_write_encoded_at: as dtbio_write_encoded, but the blob goes to file_offset (even, at least 16: the bytes the
 *   header reserves) instead of the end of the file; the writer's end of data becomes at least the blob's end.
 * dtbio_place_chunks: records chunks another writer put at file_offsets[i] (sizes[i] bytes), on the main writer.
 * Both refuse chunks outside the raster, chunks already recorded, odd offsets or offsets inside the header, chunks
 * that overlap each other or a chunk placed before, a classic file past 4 GB, and a writer that has appended chunks
 * (dtbio_write_rows / dtbio_write_encoded): a file takes its chunks either appended or at given offsets. */
int dtbio_open_part(const char *path, const dtbio_info *info, dtbio_writer **out);
int dtbio_write_encoded_at(dtbio_writer *w, int64_t first_chunk, int64_t n_chunks, const void *blob, int64_t blob_bytes,
                           const int64_t *offsets, const int64_t *sizes, int64_t file_offset);
int dtbio_place_chunks(dtbio_writer *w, int64_t first_chunk, int64_t n_chunks, const int64_t *file_offsets, const int64_t *sizes);
/* number of bytes in the file so far (header + chunks written) */
int64_t dtbio_bytes_written(const dtbio_writer *w);

/* the writer's IFD goes out at close, so its status matters; a writer with missing chunks removes its file */
int dtbio_close_reader(dtbio_reader *r);
int dtbio_close_writer(dtbio_writer *w);

#ifdef __cplusplus
}
#endif
#endif /* DTB200_IO_H */
