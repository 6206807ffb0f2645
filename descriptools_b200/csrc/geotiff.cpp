// geotiff.cpp -- libdtb200_io.so: native single-band GeoTIFF codec for the rasters either side of the
// descriptor path (include/dtb200_io.h; SURVEY.md section 8 f3).
//
// The reference delegates raster I/O to rasterio / GDAL (Example/example.py:33-39 reads 12_dem / 12_fdr /
// 12_fac -- LZW, 128 x 128 tiles -- and :106 the strip-organised benchmark map; :201-217 writes the class
// map with the DEM's georeferencing).  Nothing of GDAL is restated here: this is a TIFF 6.0 / BigTIFF codec
// written against the format itself.  Chunks (tiles or strips) are independent, so a row block is decoded
// or encoded by a team of threads, one chunk at a time each, straight into / out of the caller's (pinned)
// buffer; the Python side (descriptools_b200/raster.py) overlaps that with the host<->device copies.
#include "../../include/dtb200_io.h"
#include "lzw.cuh"  // the decoder shared with the device tile decoder (tiffcodec.cu)

#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cerrno>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <new>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

namespace {

thread_local std::string g_err;

int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}

// no C++ exception crosses the C ABI (a damaged file can ask for absurd allocations)
template <typename F>
int guarded(F body) {
    try {
        return body();
    } catch (const std::bad_alloc &) {
        return fail(DTBIO_ERR_IO, "out of memory");
    } catch (const std::exception &e) {
        return fail(DTBIO_ERR_IO, e.what());
    }
}

// ---------------------------------------------------------------------------------------------------
// TIFF field types
// ---------------------------------------------------------------------------------------------------
enum { T_BYTE = 1, T_ASCII = 2, T_SHORT = 3, T_LONG = 4, T_RATIONAL = 5, T_SBYTE = 6, T_UNDEF = 7, T_SSHORT = 8,
       T_SLONG = 9, T_SRATIONAL = 10, T_FLOAT = 11, T_DOUBLE = 12, T_IFD = 13, T_LONG8 = 16, T_SLONG8 = 17, T_IFD8 = 18 };

int type_size(int t) {
    switch (t) {
        case T_BYTE: case T_ASCII: case T_SBYTE: case T_UNDEF: return 1;
        case T_SHORT: case T_SSHORT: return 2;
        case T_LONG: case T_SLONG: case T_FLOAT: case T_IFD: return 4;
        case T_RATIONAL: case T_SRATIONAL: case T_DOUBLE: case T_LONG8: case T_SLONG8: case T_IFD8: return 8;
    }
    return 0;
}
// width of the unit that is byte-swapped (a RATIONAL is two LONGs)
int swap_unit(int t) { return (t == T_RATIONAL || t == T_SRATIONAL) ? 4 : type_size(t); }

void swap_bytes(uint8_t *p, size_t n_units, int unit) {
    if (unit == 2) for (size_t i = 0; i < n_units; ++i) std::swap(p[2 * i], p[2 * i + 1]);
    else if (unit == 4) for (size_t i = 0; i < n_units; ++i) { std::swap(p[4 * i], p[4 * i + 3]); std::swap(p[4 * i + 1], p[4 * i + 2]); }
    else if (unit == 8) for (size_t i = 0; i < n_units; ++i) for (int k = 0; k < 4; ++k) std::swap(p[8 * i + k], p[8 * i + 7 - k]);
}

struct Tag {
    int type = 0;
    uint64_t count = 0;
    std::vector<uint8_t> data;  // host byte order
    uint64_t uint_at(uint64_t i) const {
        const uint8_t *p = data.data();
        switch (type) {
            case T_BYTE: case T_UNDEF: return p[i];
            case T_SHORT: { uint16_t v; memcpy(&v, p + 2 * i, 2); return v; }
            case T_LONG: case T_IFD: { uint32_t v; memcpy(&v, p + 4 * i, 4); return v; }
            case T_LONG8: case T_IFD8: { uint64_t v; memcpy(&v, p + 8 * i, 8); return v; }
            case T_SSHORT: { int16_t v; memcpy(&v, p + 2 * i, 2); return (uint64_t)(int64_t)v; }
            case T_SLONG: { int32_t v; memcpy(&v, p + 4 * i, 4); return (uint64_t)(int64_t)v; }
            case T_SLONG8: { int64_t v; memcpy(&v, p + 8 * i, 8); return (uint64_t)v; }
        }
        return 0;
    }
};

const int DT_SIZE[10] = {1, 1, 2, 2, 4, 4, 8, 8, 4, 8};

// SampleFormat (tag 339): 1 unsigned, 2 signed, 3 IEEE float
int dtype_from(int bits, int fmt) {
    if (fmt == 3) return bits == 32 ? DTBIO_F32 : bits == 64 ? DTBIO_F64 : -1;
    if (fmt == 2) return bits == 8 ? DTBIO_I8 : bits == 16 ? DTBIO_I16 : bits == 32 ? DTBIO_I32 : bits == 64 ? DTBIO_I64 : -1;
    if (fmt == 1 || fmt == 4) return bits == 8 ? DTBIO_U8 : bits == 16 ? DTBIO_U16 : bits == 32 ? DTBIO_U32 : bits == 64 ? DTBIO_U64 : -1;
    return -1;
}
int sample_format_of(int dtype) {
    if (dtype == DTBIO_F32 || dtype == DTBIO_F64) return 3;
    if (dtype == DTBIO_I8 || dtype == DTBIO_I16 || dtype == DTBIO_I32 || dtype == DTBIO_I64) return 2;
    return 1;
}

// ---------------------------------------------------------------------------------------------------
// LZW, the TIFF flavour: MSB-first codes of 9..12 bits, Clear = 256, EOI = 257, the code width grows one
// code early (TIFF 6.0 section 13).  The decoder lives in lzw.cuh.
// ---------------------------------------------------------------------------------------------------
struct LzwEncoder {
    static const int HBITS = 14, HSIZE = 1 << HBITS;
    std::vector<int32_t> keys;
    std::vector<uint16_t> codes;
    LzwEncoder() : keys(HSIZE), codes(HSIZE) {}

    void encode(const uint8_t *in, size_t n, std::vector<uint8_t> &out) {
        out.clear();
        out.reserve(n / 2 + 64);
        uint64_t acc = 0;
        int have = 0;
        auto put = [&](int code, int nbits) {
            acc = (acc << nbits) | (uint64_t)code;
            have += nbits;
            while (have >= 8) {
                out.push_back((uint8_t)(acc >> (have - 8)));
                have -= 8;
            }
        };
        int nbits = 9, next = 258, maxcode = 511;
        std::fill(keys.begin(), keys.end(), -1);
        put(256, nbits);
        if (n == 0) {
            put(257, nbits);
            if (have) out.push_back((uint8_t)(acc << (8 - have)));
            return;
        }
        int ent = in[0];
        for (size_t i = 1; i < n; ++i) {
            int c = in[i];
            int32_t key = (ent << 8) | c;
            uint32_t h = ((uint32_t)key * 2654435761u) >> (32 - HBITS);
            bool found = false;
            while (keys[h] >= 0) {
                if (keys[h] == key) {
                    ent = codes[h];
                    found = true;
                    break;
                }
                h = (h + 1) & (HSIZE - 1);
            }
            if (found) continue;
            put(ent, nbits);
            ent = c;
            keys[h] = key;
            codes[h] = (uint16_t)next++;
            if (next == 4094) {  // table full: start over
                put(256, nbits);
                std::fill(keys.begin(), keys.end(), -1);
                nbits = 9;
                next = 258;
                maxcode = 511;
            } else if (next > maxcode) {
                ++nbits;
                maxcode = (1 << nbits) - 1;
            }
        }
        put(ent, nbits);
        // the decoder adds one more entry for that code before it reads EOI
        ++next;
        if (next == 4094) {
            put(256, nbits);
            nbits = 9;
        } else if (next > maxcode) {
            ++nbits;
        }
        put(257, nbits);
        if (have) out.push_back((uint8_t)((acc << (8 - have)) & 0xFF));
    }
};

int64_t packbits_decode(const uint8_t *in, size_t n, uint8_t *out, size_t cap) {
    size_t ip = 0, op = 0;
    while (ip < n && op < cap) {
        int8_t c = (int8_t)in[ip++];
        if (c >= 0) {
            size_t k = (size_t)c + 1;
            if (ip + k > n) k = n - ip;
            if (op + k > cap) k = cap - op;
            memcpy(out + op, in + ip, k);
            ip += (size_t)c + 1;
            op += k;
        } else if (c != -128) {
            size_t k = (size_t)(-c) + 1;
            if (ip >= n) break;
            if (op + k > cap) k = cap - op;
            memset(out + op, in[ip++], k);
            op += k;
        }
    }
    return (int64_t)op;
}

// ---------------------------------------------------------------------------------------------------
// predictors (tag 317), applied per chunk row of `width` samples of `bps` bytes
// ---------------------------------------------------------------------------------------------------
template <typename T>
void hacc(uint8_t *row, size_t width) {
    T *p = reinterpret_cast<T *>(row);
    for (size_t i = 1; i < width; ++i) p[i] = (T)(p[i] + p[i - 1]);
}
template <typename T>
void hdiff(uint8_t *row, size_t width) {
    T *p = reinterpret_cast<T *>(row);
    for (size_t i = width; i-- > 1;) p[i] = (T)(p[i] - p[i - 1]);
}
void predictor2(uint8_t *row, size_t width, int bps, bool decode) {
    switch (bps) {
        case 1: decode ? hacc<uint8_t>(row, width) : hdiff<uint8_t>(row, width); break;
        case 2: decode ? hacc<uint16_t>(row, width) : hdiff<uint16_t>(row, width); break;
        case 4: decode ? hacc<uint32_t>(row, width) : hdiff<uint32_t>(row, width); break;
        case 8: decode ? hacc<uint64_t>(row, width) : hdiff<uint64_t>(row, width); break;
    }
}
// floating-point predictor (Adobe TIFF technical note 3): the row is stored as `bps` byte planes, most
// significant byte of every sample first, then differenced byte by byte over the whole row
void predictor3_decode(uint8_t *row, size_t width, int bps, std::vector<uint8_t> &tmp) {
    size_t n = width * bps;
    for (size_t i = 1; i < n; ++i) row[i] = (uint8_t)(row[i] + row[i - 1]);
    tmp.assign(row, row + n);
    for (size_t i = 0; i < width; ++i)
        for (int b = 0; b < bps; ++b) row[i * bps + b] = tmp[(size_t)(bps - 1 - b) * width + i];  // little-endian host
}
void predictor3_encode(uint8_t *row, size_t width, int bps, std::vector<uint8_t> &tmp) {
    size_t n = width * bps;
    tmp.assign(row, row + n);
    for (size_t i = 0; i < width; ++i)
        for (int b = 0; b < bps; ++b) row[(size_t)(bps - 1 - b) * width + i] = tmp[i * bps + b];
    for (size_t i = n; i-- > 1;) row[i] = (uint8_t)(row[i] - row[i - 1]);
}

// ---------------------------------------------------------------------------------------------------
// a team of threads over independent chunks
// ---------------------------------------------------------------------------------------------------
int team_size(int threads, int64_t n) {
    int t = threads;
    if (t <= 0) {
        t = (int)std::thread::hardware_concurrency();
        if (t <= 0) t = 4;
        if (t > 64) t = 64;
    }
    if ((int64_t)t > n) t = (int)n;
    return t < 1 ? 1 : t;
}

template <typename Fn>  // Fn(int64_t item, int worker) -> int status; a failing item leaves its text in g_err
int run_team(int64_t n, int threads, Fn fn) {
    if (n <= 0) return DTBIO_OK;
    int t = team_size(threads, n);
    std::atomic<int64_t> next(0);
    std::atomic<int> status(DTBIO_OK);
    std::mutex m;
    std::string first_error;
    auto work = [&](int worker) {
        for (;;) {
            int64_t i = next.fetch_add(1);
            if (i >= n || status.load() != DTBIO_OK) return;
            int rc = guarded([&] { return fn(i, worker); });
            if (rc != DTBIO_OK) {
                std::lock_guard<std::mutex> g(m);
                if (status.load() == DTBIO_OK) {
                    status.store(rc);
                    first_error = g_err;
                }
                return;
            }
        }
    };
    if (t == 1) {
        work(0);
    } else {
        std::vector<std::thread> team;
        team.reserve(t - 1);
        for (int k = 1; k < t; ++k) team.emplace_back(work, k);
        work(0);
        for (auto &th : team) th.join();
    }
    if (status.load() != DTBIO_OK) g_err = first_error;
    return status.load();
}

bool pread_all(int fd, void *buf, size_t n, uint64_t off) {
    uint8_t *p = (uint8_t *)buf;
    while (n) {
        ssize_t k = pread(fd, p, n, (off_t)off);
        if (k < 0 && errno == EINTR) continue;
        if (k <= 0) return false;
        p += k;
        off += (uint64_t)k;
        n -= (size_t)k;
    }
    return true;
}
bool pwrite_all(int fd, const void *buf, size_t n, uint64_t off) {
    const uint8_t *p = (const uint8_t *)buf;
    while (n) {
        ssize_t k = pwrite(fd, p, n, (off_t)off);
        if (k < 0 && errno == EINTR) continue;
        if (k <= 0) return false;
        p += k;
        off += (uint64_t)k;
        n -= (size_t)k;
    }
    return true;
}

// geometry shared by reader and writer
struct Layout {
    int64_t rows = 0, cols = 0;
    int bps = 1;            // bytes per sample
    int64_t ch = 0, cw = 0;  // chunk height / width in samples (cw == cols for strips)
    int64_t across = 1, down = 1;
    bool tiled = false;
    int64_t n_chunks() const { return across * down; }
    // rows of chunk-row cy that hold data
    int64_t rows_in(int64_t cy) const { return std::min(ch, rows - cy * ch); }
    // rows a chunk is stored with (tiles are always whole)
    int64_t stored_rows(int64_t cy) const { return tiled ? ch : rows_in(cy); }
    void set(int64_t r, int64_t c, int b, int64_t tile_rows, int64_t tile_cols, int64_t rps) {
        rows = r; cols = c; bps = b;
        tiled = tile_rows > 0 && tile_cols > 0;
        if (tiled) { ch = tile_rows; cw = tile_cols; }
        else { ch = rps > 0 ? std::min(rps, std::max<int64_t>(r, 1)) : std::max<int64_t>(r, 1); cw = c; }
        across = tiled ? (cols + cw - 1) / cw : 1;
        down = (rows + ch - 1) / ch;
    }
};

}  // namespace

// =====================================================================================================
// reader
// =====================================================================================================
struct dtbio_reader {
    ~dtbio_reader() { if (fd >= 0) close(fd); }
    int fd = -1;
    uint64_t file_size = 0;
    bool big = false, swap = false;
    std::map<int, Tag> tags;
    dtbio_info info{};
    Layout lay;
    const Tag *offsets = nullptr, *counts = nullptr;
};

namespace {

int read_ifd(dtbio_reader *r) {
    uint8_t hdr[16];
    if (r->file_size < 8 || !pread_all(r->fd, hdr, 8, 0)) return fail(DTBIO_ERR_FORMAT, "file shorter than a TIFF header");
    if (hdr[0] == 'I' && hdr[1] == 'I') r->swap = false;
    else if (hdr[0] == 'M' && hdr[1] == 'M') r->swap = true;
    else return fail(DTBIO_ERR_FORMAT, "not a TIFF file (no II/MM byte-order mark)");
    auto rd16 = [&](const uint8_t *p) { uint16_t v; memcpy(&v, p, 2); if (r->swap) v = (uint16_t)((v >> 8) | (v << 8)); return v; };
    auto rd32 = [&](const uint8_t *p) { uint32_t v; memcpy(&v, p, 4); if (r->swap) v = __builtin_bswap32(v); return v; };
    auto rd64 = [&](const uint8_t *p) { uint64_t v; memcpy(&v, p, 8); if (r->swap) v = __builtin_bswap64(v); return v; };
    uint16_t magic = rd16(hdr + 2);
    uint64_t ifd;
    if (magic == 42) {
        r->big = false;
        ifd = rd32(hdr + 4);
    } else if (magic == 43) {
        r->big = true;
        if (!pread_all(r->fd, hdr + 8, 8, 8)) return fail(DTBIO_ERR_FORMAT, "truncated BigTIFF header");
        if (rd16(hdr + 4) != 8) return fail(DTBIO_ERR_FORMAT, "BigTIFF offset size is not 8");
        ifd = rd64(hdr + 8);
    } else {
        return fail(DTBIO_ERR_FORMAT, "not a TIFF file (magic is neither 42 nor 43)");
    }
    const int esz = r->big ? 20 : 12, csz = r->big ? 8 : 2, inl = r->big ? 8 : 4;
    uint8_t cnt[8];
    if (ifd > r->file_size - csz || !pread_all(r->fd, cnt, csz, ifd)) return fail(DTBIO_ERR_FORMAT, "IFD offset outside the file");
    uint64_t n = r->big ? rd64(cnt) : rd16(cnt);
    if (n == 0 || n > 65535 || n * esz > r->file_size - ifd - csz) return fail(DTBIO_ERR_FORMAT, "implausible IFD entry count");
    std::vector<uint8_t> ent(n * esz);
    if (!pread_all(r->fd, ent.data(), ent.size(), ifd + csz)) return fail(DTBIO_ERR_IO, "cannot read the IFD");
    for (uint64_t i = 0; i < n; ++i) {
        const uint8_t *e = ent.data() + i * esz;
        int tag = rd16(e), type = rd16(e + 2);
        uint64_t count = r->big ? rd64(e + 4) : rd32(e + 4);
        int ts = type_size(type);
        if (ts == 0) continue;  // unknown field type: skip, as the specification asks
        if (count > (1ull << 40) / ts) return fail(DTBIO_ERR_FORMAT, "implausible tag count");
        uint64_t bytes = count * ts;
        Tag t;
        t.type = type;
        t.count = count;
        const uint8_t *val = e + (r->big ? 12 : 8);
        if (bytes <= (uint64_t)inl) {
            t.data.assign(val, val + bytes);
        } else {
            uint64_t off = r->big ? rd64(val) : rd32(val);
            if (bytes > r->file_size || off > r->file_size - bytes)  // before anything is allocated for it
                return fail(DTBIO_ERR_FORMAT, "tag " + std::to_string(tag) + " points outside the file");
            t.data.resize(bytes);
            if (!pread_all(r->fd, t.data.data(), bytes, off)) return fail(DTBIO_ERR_IO, "cannot read tag " + std::to_string(tag));
        }
        if (r->swap) swap_bytes(t.data.data(), bytes / swap_unit(type), swap_unit(type));
        r->tags[tag] = std::move(t);
    }
    return DTBIO_OK;
}

uint64_t tag_uint(const dtbio_reader *r, int tag, uint64_t dflt) {
    auto it = r->tags.find(tag);
    if (it == r->tags.end() || it->second.count == 0) return dflt;
    return it->second.uint_at(0);
}

int interpret(dtbio_reader *r) {
    dtbio_info &in = r->info;
    in.cols = (int64_t)tag_uint(r, 256, 0);
    in.rows = (int64_t)tag_uint(r, 257, 0);
    if (in.rows <= 0 || in.cols <= 0) return fail(DTBIO_ERR_FORMAT, "ImageWidth / ImageLength missing");
    if (tag_uint(r, 277, 1) != 1) return fail(DTBIO_ERR_UNSUPPORTED, "more than one sample per pixel (only single-band rasters are read)");
    int bits = (int)tag_uint(r, 258, 1), fmt = (int)tag_uint(r, 339, 1);
    in.dtype = dtype_from(bits, fmt);
    if (in.dtype < 0) return fail(DTBIO_ERR_UNSUPPORTED, "unsupported BitsPerSample/SampleFormat " + std::to_string(bits) + "/" + std::to_string(fmt));
    int comp = (int)tag_uint(r, 259, 1);
    if (comp == 32946) comp = DTBIO_COMP_DEFLATE;
    if (comp != DTBIO_COMP_NONE && comp != DTBIO_COMP_LZW && comp != DTBIO_COMP_DEFLATE && comp != DTBIO_COMP_PACKBITS)
        return fail(DTBIO_ERR_UNSUPPORTED, "unsupported compression " + std::to_string(comp));
    in.compression = comp;
    in.predictor = (int)tag_uint(r, 317, 1);
    if (in.predictor < 1 || in.predictor > 3) return fail(DTBIO_ERR_UNSUPPORTED, "unknown predictor");
    // the predictor belongs to the LZW / Deflate codecs; libtiff and GDAL ignore the tag on stored and PackBits data
    if (comp == DTBIO_COMP_NONE || comp == DTBIO_COMP_PACKBITS) in.predictor = 1;
    if (in.predictor == 3 && in.dtype != DTBIO_F32 && in.dtype != DTBIO_F64) return fail(DTBIO_ERR_FORMAT, "floating-point predictor on integer samples");
    if (tag_uint(r, 266, 1) != 1) return fail(DTBIO_ERR_UNSUPPORTED, "FillOrder 2");
    in.bigtiff = r->big;
    in.big_endian = r->swap;
    if (r->tags.count(322) && r->tags.count(323)) {
        in.tile_cols = (int32_t)tag_uint(r, 322, 0);
        in.tile_rows = (int32_t)tag_uint(r, 323, 0);
        if (in.tile_cols <= 0 || in.tile_rows <= 0) return fail(DTBIO_ERR_FORMAT, "bad tile size");
        r->offsets = r->tags.count(324) ? &r->tags[324] : nullptr;
        r->counts = r->tags.count(325) ? &r->tags[325] : nullptr;
    } else {
        uint64_t rps = tag_uint(r, 278, (uint64_t)in.rows);
        if (rps == 0 || rps > (uint64_t)in.rows) rps = (uint64_t)in.rows;
        in.rows_per_strip = (int32_t)rps;
        r->offsets = r->tags.count(273) ? &r->tags[273] : nullptr;
        r->counts = r->tags.count(279) ? &r->tags[279] : nullptr;
    }
    r->lay.set(in.rows, in.cols, DT_SIZE[in.dtype], in.tile_rows, in.tile_cols, in.rows_per_strip);
    if ((double)r->lay.ch * (double)r->lay.cw * r->lay.bps > 2147483647.0)
        return fail(DTBIO_ERR_UNSUPPORTED, "a chunk of more than 2 GiB (one strip for a huge raster?)");
    if (!r->offsets || r->offsets->count < (uint64_t)r->lay.n_chunks()) return fail(DTBIO_ERR_FORMAT, "chunk offsets missing or too few");
    if (r->counts && r->counts->count < (uint64_t)r->lay.n_chunks()) return fail(DTBIO_ERR_FORMAT, "chunk byte counts too few");
    if (!r->counts && in.compression != DTBIO_COMP_NONE) return fail(DTBIO_ERR_FORMAT, "compressed file without chunk byte counts");
    // GDAL_NODATA: ASCII number
    auto nd = r->tags.find(42113);
    if (nd != r->tags.end() && nd->second.type == T_ASCII && nd->second.count > 0) {
        std::string s((const char *)nd->second.data.data(), nd->second.data.size());
        char *end = nullptr;
        double v = strtod(s.c_str(), &end);
        if (end != s.c_str()) {
            in.has_nodata = 1;
            in.nodata = v;
        }
    }
    auto ps = r->tags.find(33550), tp = r->tags.find(33922);
    if (ps != r->tags.end() && tp != r->tags.end() && ps->second.type == T_DOUBLE && tp->second.type == T_DOUBLE &&
        ps->second.count >= 2 && tp->second.count >= 6) {
        in.has_georef = 1;
        memcpy(in.pixel_scale, ps->second.data.data(), sizeof(double) * std::min<uint64_t>(3, ps->second.count));
        memcpy(in.tiepoint, tp->second.data.data(), sizeof(double) * 6);
    }
    return DTBIO_OK;
}

struct Scratch {
    std::vector<uint8_t> comp, raw, tmp;
    std::vector<dtb::LzwWideSlot> lzw;
    LzwEncoder *enc = nullptr;
    ~Scratch() { delete enc; }
};

int decode_chunk(dtbio_reader *r, int64_t chunk, int64_t row0, int64_t row1, uint8_t *dst, int64_t stride, Scratch &s) {
    const Layout &L = r->lay;
    int64_t cy = chunk / L.across, cx = chunk % L.across;
    int64_t srows = L.stored_rows(cy);
    size_t row_bytes = (size_t)(L.cw * L.bps), raw_bytes = row_bytes * (size_t)srows;
    uint64_t off = r->offsets->uint_at((uint64_t)chunk);
    uint64_t len = r->counts ? r->counts->uint_at((uint64_t)chunk) : raw_bytes;
    // the rows / columns of this chunk that the caller asked for
    int64_t y0 = std::max(row0, cy * L.ch), y1 = std::min(row1, cy * L.ch + L.rows_in(cy));
    int64_t x0 = cx * L.cw, x1 = std::min(L.cols, x0 + L.cw);
    size_t copy_bytes = (size_t)((x1 - x0) * L.bps);
    const uint8_t *src = nullptr;
    if (len == 0 || off == 0) {  // sparse file (GDAL SPARSE_OK): an absent chunk reads as zeros
        for (int64_t y = y0; y < y1; ++y) memset(dst + (y - row0) * stride + x0 * L.bps, 0, copy_bytes);
        return DTBIO_OK;
    }
    if (len > r->file_size || off > r->file_size - len) return fail(DTBIO_ERR_FORMAT, "chunk " + std::to_string(chunk) + " lies outside the file");
    const int comp = r->info.compression;
    if (comp == DTBIO_COMP_NONE && r->info.predictor == 1 && !r->swap) {
        // read just the rows that are wanted, straight into place when the chunk spans whole rows
        if (len < raw_bytes && y1 > y0 && (uint64_t)(y1 - cy * L.ch) * row_bytes > len) return fail(DTBIO_ERR_FORMAT, "short uncompressed chunk");
        for (int64_t y = y0; y < y1; ++y) {
            uint64_t o = off + (uint64_t)(y - cy * L.ch) * row_bytes;
            if (!pread_all(r->fd, dst + (y - row0) * stride + x0 * L.bps, copy_bytes, o)) return fail(DTBIO_ERR_IO, "read failed");
        }
        return DTBIO_OK;
    }
    s.comp.resize(len);
    if (!pread_all(r->fd, s.comp.data(), len, off)) return fail(DTBIO_ERR_IO, "read failed");
    if (comp == DTBIO_COMP_NONE) {
        if (len < raw_bytes) return fail(DTBIO_ERR_FORMAT, "short uncompressed chunk");
        src = s.comp.data();
    } else {
        s.raw.resize(raw_bytes);
        int64_t got = 0;
        if (comp == DTBIO_COMP_LZW) {
            s.lzw.resize(dtb::kLzwTableSlots);
            got = dtb::lzw_decode(s.comp.data(), len, s.raw.data(), raw_bytes, s.lzw.data());
            if (got == -2) return fail(DTBIO_ERR_UNSUPPORTED, "old-style (pre TIFF 6.0) LZW");
        } else if (comp == DTBIO_COMP_DEFLATE) {
            uLongf n = (uLongf)raw_bytes;
            int rc = uncompress(s.raw.data(), &n, s.comp.data(), (uLong)len);
            got = (rc == Z_OK || rc == Z_BUF_ERROR) ? (int64_t)n : -1;
        } else {
            got = packbits_decode(s.comp.data(), len, s.raw.data(), raw_bytes);
        }
        if (got < 0) return fail(DTBIO_ERR_FORMAT, "corrupt compressed data in chunk " + std::to_string(chunk));
        if ((size_t)got < raw_bytes) {
            // tolerate a short last chunk only beyond the rows that carry data
            if ((size_t)got < row_bytes * (size_t)L.rows_in(cy)) return fail(DTBIO_ERR_FORMAT, "chunk " + std::to_string(chunk) + " decodes short");
            memset(s.raw.data() + got, 0, raw_bytes - (size_t)got);
        }
        src = s.raw.data();
    }
    uint8_t *buf = const_cast<uint8_t *>(src);
    const int pred = r->info.predictor;
    if (r->swap && pred != 3 && L.bps > 1) swap_bytes(buf, raw_bytes / L.bps, L.bps);
    if (pred != 1) {
        // rows above y1 are not needed, but the accumulation is per row, so only the wanted rows are undone
        for (int64_t y = y0; y < y1; ++y) {
            uint8_t *row = buf + (size_t)(y - cy * L.ch) * row_bytes;
            if (pred == 2) predictor2(row, (size_t)L.cw, L.bps, true);
            else predictor3_decode(row, (size_t)L.cw, L.bps, s.tmp);
        }
    }
    for (int64_t y = y0; y < y1; ++y)
        memcpy(dst + (y - row0) * stride + x0 * L.bps, buf + (size_t)(y - cy * L.ch) * row_bytes, copy_bytes);
    return DTBIO_OK;
}

}  // namespace

// =====================================================================================================
// writer
// =====================================================================================================
struct dtbio_writer {
    ~dtbio_writer() { if (fd >= 0) close(fd); }
    int fd = -1;
    std::string path;
    dtbio_info info{};
    Layout lay;
    bool big = false;
    std::atomic<uint64_t> pos{0};
    std::vector<uint64_t> offsets, counts;
    std::map<int, Tag> extra;
    bool part = false;                  // dtbio_open_part: writes chunks only, never the header / IFD
    bool appended = false;              // chunks went to the end of the file (write_rows / write_encoded)
    std::map<uint64_t, uint64_t> spans;  // [start, end) of the chunks written or placed at given offsets
};

namespace {

int encode_chunk(dtbio_writer *w, int64_t chunk, int64_t row0, const uint8_t *src, int64_t stride, Scratch &s) {
    const Layout &L = w->lay;
    int64_t cy = chunk / L.across, cx = chunk % L.across;
    int64_t srows = L.stored_rows(cy), drows = L.rows_in(cy);
    size_t row_bytes = (size_t)(L.cw * L.bps), raw_bytes = row_bytes * (size_t)srows;
    int64_t x0 = cx * L.cw, x1 = std::min(L.cols, x0 + L.cw);
    size_t copy_bytes = (size_t)((x1 - x0) * L.bps);
    const int comp = w->info.compression, pred = w->info.predictor;
    const uint8_t *first = src + (cy * L.ch - row0) * stride + x0 * L.bps;
    const uint8_t *payload;
    size_t payload_bytes;
    if (comp == DTBIO_COMP_NONE && pred == 1 && copy_bytes == row_bytes && (stride == (int64_t)row_bytes || srows == 1) && srows == drows) {
        payload = first;  // a strip of whole rows, already contiguous in the caller's buffer
        payload_bytes = raw_bytes;
    } else {
        s.raw.resize(raw_bytes);
        for (int64_t y = 0; y < srows; ++y) {
            uint8_t *row = s.raw.data() + (size_t)y * row_bytes;
            if (y < drows) {
                memcpy(row, first + y * stride, copy_bytes);
                // pad a partial tile by repeating the last sample / row: compresses well, never read back
                for (size_t b = copy_bytes; b < row_bytes; b += L.bps) memcpy(row + b, row + copy_bytes - L.bps, L.bps);
            } else {
                memcpy(row, s.raw.data() + (size_t)(drows - 1) * row_bytes, row_bytes);
            }
        }
        if (pred == 2) for (int64_t y = 0; y < srows; ++y) predictor2(s.raw.data() + (size_t)y * row_bytes, (size_t)L.cw, L.bps, false);
        if (pred == 3) for (int64_t y = 0; y < srows; ++y) predictor3_encode(s.raw.data() + (size_t)y * row_bytes, (size_t)L.cw, L.bps, s.tmp);
        if (comp == DTBIO_COMP_LZW) {
            if (!s.enc) s.enc = new LzwEncoder();
            s.enc->encode(s.raw.data(), raw_bytes, s.comp);
            payload = s.comp.data();
            payload_bytes = s.comp.size();
        } else if (comp == DTBIO_COMP_DEFLATE) {
            uLongf n = compressBound((uLong)raw_bytes);
            s.comp.resize(n);
            if (compress2(s.comp.data(), &n, s.raw.data(), (uLong)raw_bytes, 6) != Z_OK) return fail(DTBIO_ERR_IO, "deflate failed");
            payload = s.comp.data();
            payload_bytes = n;
        } else {
            payload = s.raw.data();
            payload_bytes = raw_bytes;
        }
    }
    uint64_t at = w->pos.fetch_add((payload_bytes + 1) & ~(uint64_t)1);
    if (!w->big && at + payload_bytes > 0xFFFFFFF0ull) return fail(DTBIO_ERR_UNSUPPORTED, "classic TIFF would exceed 4 GB: create the file with bigtiff = 1");
    if (!pwrite_all(w->fd, payload, payload_bytes, at)) return fail(DTBIO_ERR_IO, std::string("write failed: ") + strerror(errno));
    w->offsets[(size_t)chunk] = at;
    w->counts[(size_t)chunk] = payload_bytes;
    return DTBIO_OK;
}

void put_tag(std::map<int, Tag> &m, int tag, int type, const std::vector<uint64_t> &vals) {
    Tag t;
    t.type = type;
    t.count = vals.size();
    int ts = type_size(type);
    t.data.resize(vals.size() * ts);
    for (size_t i = 0; i < vals.size(); ++i) {
        if (ts == 2) { uint16_t v = (uint16_t)vals[i]; memcpy(&t.data[i * 2], &v, 2); }
        else if (ts == 4) { uint32_t v = (uint32_t)vals[i]; memcpy(&t.data[i * 4], &v, 4); }
        else { uint64_t v = vals[i]; memcpy(&t.data[i * 8], &v, 8); }
    }
    m[tag] = std::move(t);
}

int finish(dtbio_writer *w) {
    for (size_t i = 0; i < w->offsets.size(); ++i)
        if (w->counts[i] == 0) return fail(DTBIO_ERR_ORDER, "chunk " + std::to_string(i) + " was never written");
    std::map<int, Tag> tags = w->extra;
    const Layout &L = w->lay;
    const int dt = w->info.dtype;
    put_tag(tags, 256, L.cols > 65535 ? T_LONG : T_SHORT, {(uint64_t)L.cols});
    put_tag(tags, 257, L.rows > 65535 ? T_LONG : T_SHORT, {(uint64_t)L.rows});
    put_tag(tags, 258, T_SHORT, {(uint64_t)DT_SIZE[dt] * 8});
    put_tag(tags, 259, T_SHORT, {(uint64_t)w->info.compression});
    put_tag(tags, 262, T_SHORT, {1});  // BlackIsZero
    put_tag(tags, 277, T_SHORT, {1});
    put_tag(tags, 284, T_SHORT, {1});
    put_tag(tags, 339, T_SHORT, {(uint64_t)sample_format_of(dt)});
    if (w->info.predictor != 1) put_tag(tags, 317, T_SHORT, {(uint64_t)w->info.predictor});
    const int otype = w->big ? T_LONG8 : T_LONG;
    if (L.tiled) {
        put_tag(tags, 322, T_SHORT, {(uint64_t)L.cw});
        put_tag(tags, 323, T_SHORT, {(uint64_t)L.ch});
        put_tag(tags, 324, otype, w->offsets);
        put_tag(tags, 325, otype, w->counts);
    } else {
        put_tag(tags, 273, otype, w->offsets);
        put_tag(tags, 278, L.ch > 65535 ? T_LONG : T_SHORT, {(uint64_t)L.ch});
        put_tag(tags, 279, otype, w->counts);
    }
    // out-of-line values first, then the IFD (tags ascending: std::map order)
    const int esz = w->big ? 20 : 12, inl = w->big ? 8 : 4;
    uint64_t at = (w->pos.load() + 1) & ~(uint64_t)1;
    std::vector<uint8_t> ifd;
    uint64_t n = tags.size();
    if (w->big) { ifd.resize(8); memcpy(ifd.data(), &n, 8); }
    else { uint16_t n16 = (uint16_t)n; ifd.resize(2); memcpy(ifd.data(), &n16, 2); }
    for (auto &kv : tags) {
        const Tag &t = kv.second;
        uint8_t e[20] = {0};
        uint16_t tag16 = (uint16_t)kv.first, type16 = (uint16_t)t.type;
        memcpy(e, &tag16, 2);
        memcpy(e + 2, &type16, 2);
        uint8_t *val;
        if (w->big) { memcpy(e + 4, &t.count, 8); val = e + 12; }
        else { uint32_t c32 = (uint32_t)t.count; memcpy(e + 4, &c32, 4); val = e + 8; }
        if (t.data.size() <= (size_t)inl) {
            memcpy(val, t.data.data(), t.data.size());
        } else {
            if (!w->big && at + t.data.size() > 0xFFFFFFF0ull) return fail(DTBIO_ERR_UNSUPPORTED, "classic TIFF would exceed 4 GB");
            if (!pwrite_all(w->fd, t.data.data(), t.data.size(), at)) return fail(DTBIO_ERR_IO, "write failed");
            if (w->big) memcpy(val, &at, 8);
            else { uint32_t a32 = (uint32_t)at; memcpy(val, &a32, 4); }
            at = (at + t.data.size() + 1) & ~(uint64_t)1;
        }
        ifd.insert(ifd.end(), e, e + esz);
    }
    uint64_t zero = 0;
    ifd.insert(ifd.end(), (uint8_t *)&zero, (uint8_t *)&zero + (w->big ? 8 : 4));  // no next IFD
    if (!w->big && at + ifd.size() > 0xFFFFFFF0ull) return fail(DTBIO_ERR_UNSUPPORTED, "classic TIFF would exceed 4 GB");
    if (!pwrite_all(w->fd, ifd.data(), ifd.size(), at)) return fail(DTBIO_ERR_IO, "write failed");
    w->pos.store(at + ifd.size());
    uint8_t hdr[16] = {'I', 'I'};
    if (w->big) {
        hdr[2] = 43; hdr[4] = 8;
        memcpy(hdr + 8, &at, 8);
        if (!pwrite_all(w->fd, hdr, 16, 0)) return fail(DTBIO_ERR_IO, "write failed");
    } else {
        hdr[2] = 42;
        uint32_t a32 = (uint32_t)at;
        memcpy(hdr + 4, &a32, 4);
        if (!pwrite_all(w->fd, hdr, 8, 0)) return fail(DTBIO_ERR_IO, "write failed");
    }
    return DTBIO_OK;
}

constexpr uint64_t kHeaderBytes = 16;  // reserved for the header, patched in at close (classic TIFF uses 8)

// Chunks first .. first + n - 1 at base + rel[i] (sizes[i] bytes): in the raster, not recorded yet, even, past the
// header, inside the classic-TIFF 4 GB limit, and disjoint from each other and from every chunk placed before.  On
// success `r` holds their [start, end) in chunk order.
int check_placement(const dtbio_writer *w, int64_t first, int64_t n, uint64_t base, const int64_t *rel, const int64_t *sizes,
                    std::vector<std::pair<uint64_t, uint64_t>> &r) {
    if (w->appended) return fail(DTBIO_ERR_ORDER, "chunks at given offsets cannot follow chunks appended to the file");
    if (first + n > w->lay.n_chunks()) return fail(DTBIO_ERR_INVALID, "chunk range outside the raster");
    r.clear();
    for (int64_t i = 0; i < n; ++i) {
        const std::string which = "chunk " + std::to_string(first + i);
        if (sizes[i] <= 0 || rel[i] < 0) return fail(DTBIO_ERR_INVALID, which + ": bad offset or size");
        if (w->counts[(size_t)(first + i)]) return fail(DTBIO_ERR_ORDER, which + " written twice");
        const uint64_t at = base + (uint64_t)rel[i];
        if (at & 1) return fail(DTBIO_ERR_INVALID, which + ": TIFF offsets must be even");
        if (at < kHeaderBytes) return fail(DTBIO_ERR_INVALID, which + " overlaps the header");
        if (!w->big && at + (uint64_t)sizes[i] > 0xFFFFFFF0ull) return fail(DTBIO_ERR_UNSUPPORTED, "classic TIFF would exceed 4 GB: create the file with bigtiff = 1");
        r.emplace_back(at, at + (uint64_t)sizes[i]);
    }
    std::vector<std::pair<uint64_t, uint64_t>> sorted(r);
    std::sort(sorted.begin(), sorted.end());
    for (size_t k = 0; k < sorted.size(); ++k) {
        bool clash = k > 0 && sorted[k].first < sorted[k - 1].second;
        auto it = w->spans.upper_bound(sorted[k].first);
        if (it != w->spans.end() && it->first < sorted[k].second) clash = true;
        if (it != w->spans.begin() && std::prev(it)->second > sorted[k].first) clash = true;
        if (clash) return fail(DTBIO_ERR_INVALID, "chunks overlap at file offset " + std::to_string(sorted[k].first));
    }
    return DTBIO_OK;
}

void record_placement(dtbio_writer *w, int64_t first, const std::vector<std::pair<uint64_t, uint64_t>> &r) {
    for (size_t i = 0; i < r.size(); ++i) {
        w->offsets[(size_t)first + i] = r[i].first;
        w->counts[(size_t)first + i] = r[i].second - r[i].first;
        w->spans[r[i].first] = r[i].second;
    }
}

// what dtbio_create and dtbio_open_part share: the checks of *info and the layout / BigTIFF decision
int setup_writer(dtbio_writer *w, const char *path, const dtbio_info *info) {
    if (info->rows <= 0 || info->cols <= 0) return fail(DTBIO_ERR_INVALID, "raster size must be positive");
    if (info->dtype < 0 || info->dtype > DTBIO_F64) return fail(DTBIO_ERR_INVALID, "bad dtype");
    int comp = info->compression == 0 ? DTBIO_COMP_NONE : info->compression;
    if (comp != DTBIO_COMP_NONE && comp != DTBIO_COMP_LZW && comp != DTBIO_COMP_DEFLATE) return fail(DTBIO_ERR_UNSUPPORTED, "the writer compresses with LZW or Deflate only");
    int pred = info->predictor == 0 ? 1 : info->predictor;
    if (pred < 1 || pred > 3) return fail(DTBIO_ERR_INVALID, "bad predictor");
    if (comp == DTBIO_COMP_NONE) pred = 1;  // a predictor without a codec is not part of the format (GDAL drops it too)
    if (pred == 3 && info->dtype != DTBIO_F32 && info->dtype != DTBIO_F64) return fail(DTBIO_ERR_INVALID, "predictor 3 needs floating-point samples");
    if ((info->tile_rows > 0) != (info->tile_cols > 0)) return fail(DTBIO_ERR_INVALID, "give both tile sizes or neither");
    if (info->tile_rows > 0 && ((info->tile_rows % 16) || (info->tile_cols % 16))) return fail(DTBIO_ERR_INVALID, "tile sizes must be multiples of 16");
    w->info = *info;
    w->info.compression = comp;
    w->info.predictor = pred;
    const int bps = DT_SIZE[info->dtype];
    int64_t rps = info->rows_per_strip;
    if (info->tile_rows == 0 && rps <= 0) rps = std::max<int64_t>(1, 8192 / (info->cols * bps));
    w->lay.set(info->rows, info->cols, bps, info->tile_rows, info->tile_cols, rps);
    w->info.rows_per_strip = w->lay.tiled ? 0 : (int32_t)w->lay.ch;
    const double raw = (double)info->rows * (double)info->cols * bps;
    w->big = info->bigtiff || raw > (comp == DTBIO_COMP_NONE ? 4.0e9 : 2.0e9);
    w->info.bigtiff = w->big;
    w->info.big_endian = 0;
    w->offsets.assign((size_t)w->lay.n_chunks(), 0);
    w->counts.assign((size_t)w->lay.n_chunks(), 0);
    w->path = path;
    w->pos.store(kHeaderBytes);
    return DTBIO_OK;
}

}  // namespace

// =====================================================================================================
// C ABI
// =====================================================================================================
extern "C" {

int dtbio_abi_version(void) { return DTBIO_ABI_VERSION; }

const char *dtbio_error_string(int code) {
    switch (code) {
        case DTBIO_OK: return "ok";
        case DTBIO_ERR_INVALID: return "invalid argument";
        case DTBIO_ERR_IO: return "I/O error";
        case DTBIO_ERR_FORMAT: return "not a valid TIFF";
        case DTBIO_ERR_UNSUPPORTED: return "unsupported TIFF feature";
        case DTBIO_ERR_ORDER: return "row block not on a chunk boundary";
    }
    return "unknown error";
}

const char *dtbio_last_error(void) { return g_err.c_str(); }

int64_t dtbio_dtype_size(int dtype) { return (dtype >= 0 && dtype < 10) ? DT_SIZE[dtype] : 0; }

int dtbio_open(const char *path, dtbio_reader **out) {
    if (!path || !out) return fail(DTBIO_ERR_INVALID, "null argument");
    *out = nullptr;
    int fd = open(path, O_RDONLY | O_CLOEXEC);
    if (fd < 0) return fail(DTBIO_ERR_IO, std::string("cannot open ") + path + ": " + strerror(errno));
    struct stat st;
    if (fstat(fd, &st) != 0) { close(fd); return fail(DTBIO_ERR_IO, "fstat failed"); }
    return guarded([&]() -> int {
        std::unique_ptr<dtbio_reader> r;
        try {
            r.reset(new dtbio_reader());
        } catch (...) {
            close(fd);
            throw;
        }
        r->fd = fd;  // closed by the reader from here on
        r->file_size = (uint64_t)st.st_size;
        int rc = read_ifd(r.get());
        if (rc == DTBIO_OK) rc = interpret(r.get());
        if (rc != DTBIO_OK) return rc;
        *out = r.release();
        return DTBIO_OK;
    });
}

int dtbio_get_info(const dtbio_reader *r, dtbio_info *info) {
    if (!r || !info) return fail(DTBIO_ERR_INVALID, "null argument");
    *info = r->info;
    return DTBIO_OK;
}

int dtbio_get_tag(const dtbio_reader *r, int tag, int *type, int64_t *count, const void **data) {
    if (!r) return fail(DTBIO_ERR_INVALID, "null argument");
    auto it = r->tags.find(tag);
    if (it == r->tags.end()) return fail(DTBIO_ERR_INVALID, "tag " + std::to_string(tag) + " not present");
    if (type) *type = it->second.type;
    if (count) *count = (int64_t)it->second.count;
    if (data) *data = it->second.data.data();
    return DTBIO_OK;
}

int dtbio_read_rows(dtbio_reader *r, int64_t row0, int64_t nrows, void *dst, int64_t stride, int threads) {
    if (!r || (!dst && nrows > 0)) return fail(DTBIO_ERR_INVALID, "null argument");
    const Layout &L = r->lay;
    if (row0 < 0 || nrows < 0 || row0 + nrows > L.rows) return fail(DTBIO_ERR_INVALID, "row block outside the raster");
    if (stride < L.cols * L.bps) return fail(DTBIO_ERR_INVALID, "destination stride shorter than a row");
    if (nrows == 0) return DTBIO_OK;
    int64_t cy0 = row0 / L.ch, cy1 = (row0 + nrows - 1) / L.ch + 1;
    int64_t n = (cy1 - cy0) * L.across;
    return guarded([&]() -> int {
        int t = team_size(threads, n);
        std::vector<Scratch> scratch((size_t)t);
        return run_team(n, t, [&](int64_t i, int worker) {
            return decode_chunk(r, cy0 * L.across + i, row0, row0 + nrows, (uint8_t *)dst, stride, scratch[(size_t)worker]);
        });
    });
}

int dtbio_create(const char *path, const dtbio_info *info, dtbio_writer **out) {
    if (!path || !info || !out) return fail(DTBIO_ERR_INVALID, "null argument");
    *out = nullptr;
    return guarded([&]() -> int {
    std::unique_ptr<dtbio_writer> w(new dtbio_writer());
    const int rc = setup_writer(w.get(), path, info);
    if (rc != DTBIO_OK) return rc;
    w->fd = open(path, O_WRONLY | O_CREAT | O_TRUNC | O_CLOEXEC, 0644);
    if (w->fd < 0) return fail(DTBIO_ERR_IO, std::string("cannot create ") + path + ": " + strerror(errno));
    *out = w.release();
    return DTBIO_OK;
    });
}

int dtbio_open_part(const char *path, const dtbio_info *info, dtbio_writer **out) {
    if (!path || !info || !out) return fail(DTBIO_ERR_INVALID, "null argument");
    *out = nullptr;
    return guarded([&]() -> int {
    std::unique_ptr<dtbio_writer> w(new dtbio_writer());
    const int rc = setup_writer(w.get(), path, info);
    if (rc != DTBIO_OK) return rc;
    w->part = true;
    w->fd = open(path, O_WRONLY | O_CLOEXEC);
    if (w->fd < 0) return fail(DTBIO_ERR_IO, std::string("cannot open ") + path + ": " + strerror(errno));
    *out = w.release();
    return DTBIO_OK;
    });
}

int dtbio_set_tag(dtbio_writer *w, int tag, int type, int64_t count, const void *data) {
    if (!w || count < 0 || (count > 0 && !data)) return fail(DTBIO_ERR_INVALID, "null argument");
    int ts = type_size(type);
    if (ts == 0 || tag <= 0 || tag > 65535) return fail(DTBIO_ERR_INVALID, "bad tag or field type");
    return guarded([&]() -> int {
        Tag t;
        t.type = type;
        t.count = (uint64_t)count;
        t.data.assign((const uint8_t *)data, (const uint8_t *)data + (size_t)count * ts);
        w->extra[tag] = std::move(t);
        return DTBIO_OK;
    });
}

int dtbio_write_rows(dtbio_writer *w, int64_t row0, int64_t nrows, const void *src, int64_t stride, int threads) {
    if (!w || (!src && nrows > 0)) return fail(DTBIO_ERR_INVALID, "null argument");
    const Layout &L = w->lay;
    if (row0 < 0 || nrows < 0 || row0 + nrows > L.rows) return fail(DTBIO_ERR_INVALID, "row block outside the raster");
    if (stride < L.cols * L.bps) return fail(DTBIO_ERR_INVALID, "source stride shorter than a row");
    if (nrows == 0) return DTBIO_OK;
    if (w->part) return fail(DTBIO_ERR_ORDER, "a part writer writes chunks at given offsets only");
    if (row0 % L.ch) return fail(DTBIO_ERR_ORDER, "row block does not start on a chunk boundary");
    if ((row0 + nrows) % L.ch && row0 + nrows != L.rows) return fail(DTBIO_ERR_ORDER, "row block does not end on a chunk boundary");
    int64_t cy0 = row0 / L.ch, cy1 = (row0 + nrows - 1) / L.ch + 1;
    int64_t n = (cy1 - cy0) * L.across;
    for (int64_t i = 0; i < n; ++i)
        if (w->counts[(size_t)(cy0 * L.across + i)]) return fail(DTBIO_ERR_ORDER, "chunk written twice");
    w->appended = true;
    return guarded([&]() -> int {
        int t = team_size(threads, n);
        std::vector<Scratch> scratch((size_t)t);
        return run_team(n, t, [&](int64_t i, int worker) {
            return encode_chunk(w, cy0 * L.across + i, row0, (const uint8_t *)src, stride, scratch[(size_t)worker]);
        });
    });
}

int dtbio_write_encoded(dtbio_writer *w, int64_t first_chunk, int64_t n_chunks, const void *blob, int64_t blob_bytes,
                        const int64_t *offsets, const int64_t *sizes) {
    if (!w || n_chunks < 0 || first_chunk < 0 || blob_bytes < 0) return fail(DTBIO_ERR_INVALID, "bad argument");
    if (n_chunks == 0) return DTBIO_OK;
    if (!blob || !offsets || !sizes) return fail(DTBIO_ERR_INVALID, "null argument");
    if (first_chunk + n_chunks > w->lay.n_chunks()) return fail(DTBIO_ERR_INVALID, "chunk range outside the raster");
    if (w->part) return fail(DTBIO_ERR_ORDER, "a part writer writes chunks at given offsets only");
    for (int64_t i = 0; i < n_chunks; ++i) {
        if (sizes[i] <= 0 || offsets[i] < 0 || offsets[i] + sizes[i] > blob_bytes) return fail(DTBIO_ERR_INVALID, "chunk " + std::to_string(first_chunk + i) + " lies outside the blob");
        if (w->counts[(size_t)(first_chunk + i)]) return fail(DTBIO_ERR_ORDER, "chunk written twice");
    }
    w->appended = true;
    uint64_t at = w->pos.fetch_add(((uint64_t)blob_bytes + 1) & ~(uint64_t)1);
    if (!w->big && at + (uint64_t)blob_bytes > 0xFFFFFFF0ull) return fail(DTBIO_ERR_UNSUPPORTED, "classic TIFF would exceed 4 GB: create the file with bigtiff = 1");
    if (!pwrite_all(w->fd, blob, (size_t)blob_bytes, at)) return fail(DTBIO_ERR_IO, std::string("write failed: ") + strerror(errno));
    for (int64_t i = 0; i < n_chunks; ++i) {
        w->offsets[(size_t)(first_chunk + i)] = at + (uint64_t)offsets[i];
        w->counts[(size_t)(first_chunk + i)] = (uint64_t)sizes[i];
    }
    return DTBIO_OK;
}

int dtbio_write_encoded_at(dtbio_writer *w, int64_t first_chunk, int64_t n_chunks, const void *blob, int64_t blob_bytes,
                           const int64_t *offsets, const int64_t *sizes, int64_t file_offset) {
    if (!w || n_chunks < 0 || first_chunk < 0 || blob_bytes < 0 || file_offset < 0) return fail(DTBIO_ERR_INVALID, "bad argument");
    if (n_chunks == 0) return DTBIO_OK;
    if (!blob || !offsets || !sizes) return fail(DTBIO_ERR_INVALID, "null argument");
    if (file_offset & 1) return fail(DTBIO_ERR_INVALID, "TIFF offsets must be even");
    if ((uint64_t)file_offset < kHeaderBytes) return fail(DTBIO_ERR_INVALID, "the blob overlaps the header");
    if (!w->big && (uint64_t)file_offset + (uint64_t)blob_bytes > 0xFFFFFFF0ull) return fail(DTBIO_ERR_UNSUPPORTED, "classic TIFF would exceed 4 GB: create the file with bigtiff = 1");
    for (int64_t i = 0; i < n_chunks; ++i)
        if (sizes[i] <= 0 || offsets[i] < 0 || offsets[i] + sizes[i] > blob_bytes) return fail(DTBIO_ERR_INVALID, "chunk " + std::to_string(first_chunk + i) + " lies outside the blob");
    return guarded([&]() -> int {
        std::vector<std::pair<uint64_t, uint64_t>> r;
        const int rc = check_placement(w, first_chunk, n_chunks, (uint64_t)file_offset, offsets, sizes, r);
        if (rc != DTBIO_OK) return rc;
        if (!pwrite_all(w->fd, blob, (size_t)blob_bytes, (uint64_t)file_offset)) return fail(DTBIO_ERR_IO, std::string("write failed: ") + strerror(errno));
        record_placement(w, first_chunk, r);
        const uint64_t end = (uint64_t)file_offset + (uint64_t)blob_bytes;
        uint64_t cur = w->pos.load();
        while (cur < end && !w->pos.compare_exchange_weak(cur, end)) {
        }
        return DTBIO_OK;
    });
}

int dtbio_place_chunks(dtbio_writer *w, int64_t first_chunk, int64_t n_chunks, const int64_t *file_offsets, const int64_t *sizes) {
    if (!w || n_chunks < 0 || first_chunk < 0) return fail(DTBIO_ERR_INVALID, "bad argument");
    if (n_chunks == 0) return DTBIO_OK;
    if (!file_offsets || !sizes) return fail(DTBIO_ERR_INVALID, "null argument");
    return guarded([&]() -> int {
        std::vector<std::pair<uint64_t, uint64_t>> r;
        const int rc = check_placement(w, first_chunk, n_chunks, 0, file_offsets, sizes, r);
        if (rc != DTBIO_OK) return rc;
        record_placement(w, first_chunk, r);
        uint64_t end = 0, cur = w->pos.load();
        for (const auto &x : r) end = std::max(end, x.second);
        while (cur < end && !w->pos.compare_exchange_weak(cur, end)) {
        }
        return DTBIO_OK;
    });
}

int dtbio_writer_info(const dtbio_writer *w, dtbio_info *info) {
    if (!w || !info) return fail(DTBIO_ERR_INVALID, "null argument");
    *info = w->info;
    return DTBIO_OK;
}

int64_t dtbio_bytes_written(const dtbio_writer *w) { return w ? (int64_t)w->pos.load() : 0; }

int dtbio_close_reader(dtbio_reader *r) {
    delete r;  // closes the file
    return DTBIO_OK;
}

int dtbio_close_writer(dtbio_writer *w) {
    if (!w) return DTBIO_OK;
    if (w->part) {  // the main writer owns the header, the IFD and the file's fate
        int rc = close(w->fd) == 0 ? DTBIO_OK : fail(DTBIO_ERR_IO, std::string("close failed: ") + strerror(errno));
        w->fd = -1;
        delete w;
        return rc;
    }
    int rc = guarded([&]() -> int { return finish(w); });
    if (close(w->fd) != 0 && rc == DTBIO_OK) rc = fail(DTBIO_ERR_IO, std::string("close failed: ") + strerror(errno));
    w->fd = -1;
    if (rc != DTBIO_OK) {
        std::string keep = g_err;
        unlink(w->path.c_str());
        g_err = keep;
    }
    delete w;
    return rc;
}

}  // extern "C"
