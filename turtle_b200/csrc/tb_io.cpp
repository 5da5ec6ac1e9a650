/*
 * tb_io.cpp -- readers / writers of the reference's DEM formats (see tb_io.hpp).
 *
 * Reference behaviour restated per format (file:line in the reference's sources):
 *   hgt  src/turtle/io/hgt.c:61-147      name -> origin and size; big-endian int16, north first
 *   png  src/turtle/io/png16.c:195-377   16-bit gray, JSON "topography" object in a text chunk
 *        src/turtle/io/png16.c:456-546   writer: tEXt "Comment" with %a formatted bounds
 *   tif  src/turtle/io/geotiff16.c:166-260  int16 strips, ModelPixelScale / ModelTiepoint
 *        src/turtle/io/geotiff16.c:262-330  writer (z scale must be (-32767, 1), no projection)
 *   grd  src/turtle/io/grd.c:45-155      "y0 y1 x0 x1 dy dx" then values, south first
 *   asc  src/turtle/io/asc.c:44-145      ESRI header, cell-centred origin, north first
 * The reference goes through libpng / libtiff (dlopen); here the containers are parsed
 * directly and only zlib's inflate / deflate / crc32 are borrowed.
 */
#include "tb_io.hpp"

#include <float.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <zlib.h>

#include <exception>

#include "tb_core.cuh"

namespace tbio {

static int fail(Error & error, enum turtle_return code, const char * file, const char * format,
    ...)
{
        char buffer[1024];
        va_list args;
        va_start(args, format);
        vsnprintf(buffer, sizeof buffer, format, args);
        va_end(args);
        error.code = code;
        error.message = buffer;
        error.file = file;
        return -1;
}

const char * extension(const char * path)
{
        const char * ext = NULL;
        for (const char * p = path; *p != 0x0; p++) {
                if (*p == '.') ext = p + 1;
                if ((*p == '/') || (*p == '\\')) ext = NULL;
        }
        return ext;
}

int known_extension(const char * ext)
{
        static const char * known[] = { "tif", "grd", "hgt", "png", "asc" };
        if (ext == NULL) return 0;
        for (size_t i = 0; i < sizeof(known) / sizeof(*known); i++)
                if (strcmp(ext, known[i]) == 0) return 1;
        return 0;
}

static int read_file(const char * path, std::vector<uint8_t> & bytes)
{
        FILE * fid = fopen(path, "rb");
        if (fid == NULL) return -1;
        fseek(fid, 0, SEEK_END);
        const long size = ftell(fid);
        fseek(fid, 0, SEEK_SET);
        bytes.resize(size > 0 ? (size_t)size : 0);
        const size_t got = bytes.empty() ? 0 : fread(bytes.data(), 1, bytes.size(), fid);
        fclose(fid);
        return (got == bytes.size()) ? 0 : -1;
}

/* The reference's `(uint16_t)d` of a rounded double (map.c:41-44 set_z and its copies):
 * in range it is the value; out of range it is what the x86-64 code of the reference
 * does, a 32-bit truncation whose low half is kept. */
static uint16_t to_u16(double d)
{
        if (d >= 0. && d <= 65535.) return (uint16_t)d;
        if (!(d > -2147483649.) || !(d < 2147483648.)) return 0;
        return (uint16_t)(uint32_t)(int32_t)d;
}

/* ---- hgt ------------------------------------------------------------------------ */
static const char * HGT_C = "src/turtle/io/hgt.c";

static int hgt_header(const char * path, Header & h, Error & error)
{
        const char * filename = path;
        for (const char * p = path; *p != 0x0; p++)
                if ((*p == '/') || (*p == '\\')) filename = p + 1;
        int bad = strlen(filename) < 8;
        double x0 = 0., y0 = 0.;
        if (!bad) {
                x0 = atoi(filename + 4);
                if (filename[3] == 'W')
                        x0 = -x0;
                else if (filename[3] != 'E')
                        bad = 1;
                y0 = atoi(filename + 1);
                if (filename[0] == 'S')
                        y0 = -y0;
                else if (filename[0] != 'N')
                        bad = 1;
        }
        const char * ext = NULL;
        if (!bad) {
                for (const char * p = filename + 7; *p != 0x0; p++)
                        if (*p == '.') ext = p + 1;
                if (ext == NULL) bad = 1;
        }
        if (bad)
                return fail(error, TURTLE_RETURN_BAD_FORMAT, HGT_C,
                    "invalid hgt filename for `%s'", path);
        const int n = (int)(ext - filename) - 8;
        const int nxy = ((n == 0) || (strncmp(filename + 8, "SRTMGL1", n - 1) == 0)) ? 3601 : 1201;
        h.nx = h.ny = nxy;
        h.x0 = x0;
        h.y0 = y0;
        h.z0 = -32767.;
        h.dz = 1.;
        h.dx = h.dy = 1. / (nxy - 1);
        h.kind = tb::NODE_DIRECT_I16;
        h.projection.clear();
        return 0;
}

static int hgt_read(const char * path, Header & h, RawLayout & layout,
    std::vector<uint16_t> & raw, Error & error)
{
        if (hgt_header(path, h, error) != 0) return -1;
        FILE * fid = fopen(path, "rb");
        if (fid == NULL)
                return fail(error, TURTLE_RETURN_PATH_ERROR, HGT_C, "could not open file `%s'",
                    path);
        raw.resize((size_t)h.nx * h.ny);
        const size_t got = fread(raw.data(), sizeof(uint16_t), raw.size(), fid);
        fclose(fid);
        if (got != raw.size())
                return fail(error, TURTLE_RETURN_BAD_FORMAT, HGT_C,
                    "missing data when reading file `%s'", path);
        layout.big_endian = 1;
        layout.north_first = 1;
        return 0;
}

/* ---- png ------------------------------------------------------------------------ */
static const char * PNG_C = "src/turtle/io/png16.c";

static uint32_t be32(const uint8_t * p)
{
        return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3];
}

/* A JSON token in the manner of the reference's tokenizer (jsmn, non strict): objects
 * count their keys, strings exclude the quotes, a primitive runs to the next delimiter. */
struct Token {
        int type; /* 0 primitive, 1 object, 2 array, 3 string */
        int start, end, size;
};

static int json_tokens(const char * js, int length, std::vector<Token> & tokens)
{
        tokens.clear();
        std::vector<int> open; /* enclosing containers */
        int super = -1;
        for (int pos = 0; pos < length && js[pos] != 0x0; pos++) {
                const char c = js[pos];
                if ((c == '{') || (c == '[')) {
                        if (super >= 0) tokens[super].size++;
                        Token t = { (c == '{') ? 1 : 2, pos, -1, 0 };
                        tokens.push_back(t);
                        open.push_back((int)tokens.size() - 1);
                        super = (int)tokens.size() - 1;
                } else if ((c == '}') || (c == ']')) {
                        if (open.empty()) return -1;
                        Token & t = tokens[open.back()];
                        if (t.type != ((c == '}') ? 1 : 2)) return -1;
                        t.end = pos + 1;
                        open.pop_back();
                        super = open.empty() ? -1 : open.back();
                } else if (c == '"') {
                        int e = pos + 1;
                        while ((e < length) && (js[e] != '"')) {
                                if ((js[e] == '\\') && (e + 1 < length)) e++;
                                e++;
                        }
                        if (e >= length) return -1;
                        Token t = { 3, pos + 1, e, 0 };
                        tokens.push_back(t);
                        if (super >= 0) tokens[super].size++;
                        pos = e;
                } else if ((c == '\t') || (c == '\r') || (c == '\n') || (c == ' ')) {
                        continue;
                } else if (c == ':') {
                        super = (int)tokens.size() - 1;
                } else if (c == ',') {
                        if ((super >= 0) && (tokens[super].type != 1) && (tokens[super].type != 2))
                                super = open.empty() ? -1 : open.back();
                } else {
                        int e = pos;
                        while ((e < length) && (js[e] != 0x0) && (strchr("\t\r\n ,]}:", js[e]) == NULL))
                                e++;
                        Token t = { 0, pos, e, 0 };
                        tokens.push_back(t);
                        if (super >= 0) tokens[super].size++;
                        pos = e - 1;
                }
        }
        return open.empty() ? (int)tokens.size() : -1;
}

/* png16.c:268-363: a text chunk holding {"topography" : {7 fields}} sets the meta data.
 * Returns -1 on a malformed topography object, 0 otherwise (used or ignored). */
static int png_topography(const char * path, std::string text, Header & h, Error & error)
{
        std::vector<Token> tok;
        const int r = json_tokens(text.c_str(), (int)text.size(), tok);
        if (r != 17) return 0; /* fewer: not ours; more: the reference's 17-token parse fails */
        if ((tok[0].type != 1) || (tok[1].type != 3)) return 0;
#define KEY_IS(t, name) (strncmp(text.c_str() + (t).start, name, (t).end - (t).start) == 0)
        if (!KEY_IS(tok[1], "topography")) return 0;
        if ((tok[2].type != 1) || (tok[2].size != 7))
                return fail(error, TURTLE_RETURN_BAD_FORMAT, PNG_C,
                    "invalid meta data for png file `%s'", path);
        double x1 = 0., y1 = 0., z1 = 0.;
        int done[7] = { 0, 0, 0, 0, 0, 0, 0 };
        static const char * names[7] = { "projection", "x0", "y0", "z0", "x1", "y1", "z1" };
        for (int j = 0; j < 7; j++) {
                const Token & key = tok[3 + 2 * j];
                const Token & value = tok[4 + 2 * j];
                if (!done[0] && KEY_IS(key, names[0])) {
                        if (value.type != 3)
                                return fail(error, TURTLE_RETURN_BAD_FORMAT, PNG_C,
                                    "invalid projection for png file `%s'", path);
                        h.projection = text.substr(value.start, value.end - value.start);
                        done[0] = 1;
                        continue;
                }
                if (value.type != 0)
                        return fail(error, TURTLE_RETURN_BAD_FORMAT, PNG_C,
                            "invalid type for a key in png file `%s'", path);
                double * where[7] = { NULL, &h.x0, &h.y0, &h.z0, &x1, &y1, &z1 };
                int k = 1;
                for (; k < 7; k++)
                        if (!done[k] && KEY_IS(key, names[k])) break;
                if (k == 7)
                        return fail(error, TURTLE_RETURN_BAD_FORMAT, PNG_C,
                            "invalid key for png file `%s'", path);
                sscanf(text.c_str() + value.start, "%la", where[k]);
                done[k] = 1;
        }
#undef KEY_IS
        h.dx = (x1 - h.x0) / (h.nx - 1);
        h.dy = (y1 - h.y0) / (h.ny - 1);
        h.dz = (z1 - h.z0) / 65535;
        return 0;
}

static int inflate_all(const uint8_t * src, size_t n, std::vector<uint8_t> & out, size_t hint)
{
        z_stream zs;
        memset(&zs, 0x0, sizeof zs);
        if (inflateInit(&zs) != Z_OK) return -1;
        out.resize(hint ? hint : 4096);
        zs.next_in = (Bytef *)src;
        zs.avail_in = (uInt)n;
        size_t have = 0;
        int rc = Z_OK;
        while (rc != Z_STREAM_END) {
                if (have == out.size()) out.resize(out.size() * 2);
                zs.next_out = out.data() + have;
                zs.avail_out = (uInt)(out.size() - have);
                rc = inflate(&zs, Z_NO_FLUSH);
                have = out.size() - zs.avail_out;
                if ((rc != Z_OK) && (rc != Z_STREAM_END)) {
                        inflateEnd(&zs);
                        return -1;
                }
                if ((rc == Z_OK) && (zs.avail_in == 0) && (zs.avail_out != 0)) {
                        inflateEnd(&zs);
                        return -1; /* truncated stream */
                }
        }
        inflateEnd(&zs);
        out.resize(have);
        return 0;
}

static int png_read(const char * path, Header & h, RawLayout * layout,
    std::vector<uint16_t> * raw, Error & error)
{
        std::vector<uint8_t> f;
        if (read_file(path, f) != 0)
                return fail(error, TURTLE_RETURN_PATH_ERROR, PNG_C, "could not open file `%s'",
                    path);
        static const uint8_t signature[8] = { 0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a };
        if ((f.size() < 8) || (memcmp(f.data(), signature, 8) != 0))
                return fail(error, TURTLE_RETURN_BAD_FORMAT, PNG_C, "invalid header for png `%s'",
                    path);
        h = Header();
        h.kind = tb::NODE_AFFINE_U16;
        std::vector<uint8_t> idat;
        int seen_header = 0, seen_data = 0, seen_end = 0, interlaced = 0;
        size_t pos = 8;
        while (!seen_end) {
                if (pos + 12 > f.size()) break;
                const uint32_t length = be32(&f[pos]);
                const uint8_t * type = &f[pos + 4];
                const uint8_t * data = &f[pos + 8];
                if ((size_t)length > f.size() - pos - 12) break;
                if (be32(data + length) != (uint32_t)crc32(crc32(0L, Z_NULL, 0), type, length + 4))
                        return fail(error, TURTLE_RETURN_BAD_FORMAT, PNG_C,
                            "a libpng error occured when loading file `%s'", path);
                pos += 12 + (size_t)length;
                if (memcmp(type, "IHDR", 4) == 0) {
                        if (length < 13) break;
                        h.nx = (int)be32(data);
                        h.ny = (int)be32(data + 4);
                        if (data[9] != 0)
                                return fail(error, TURTLE_RETURN_BAD_FORMAT, PNG_C,
                                    "invalid color scheme for png file `%s'", path);
                        if (data[8] != 16)
                                return fail(error, TURTLE_RETURN_BAD_FORMAT, PNG_C,
                                    "invalid bit depth (%d != 16) for file `%s'", data[8], path);
                        if ((data[12] > 1) || (h.nx <= 0) || (h.ny <= 0)) break;
                        interlaced = data[12];
                        seen_header = 1;
                } else if (memcmp(type, "IDAT", 4) == 0) {
                        seen_data = 1;
                        if (raw == NULL) break; /* header only: the text chunks were read */
                        idat.insert(idat.end(), data, data + length);
                } else if (memcmp(type, "IEND", 4) == 0) {
                        seen_end = 1;
                } else if (!seen_data && seen_header &&
                    ((memcmp(type, "tEXt", 4) == 0) || (memcmp(type, "zTXt", 4) == 0) ||
                        (memcmp(type, "iTXt", 4) == 0))) {
                        /* only the text that precedes the image is known when the reference
                         * looks for it (png16.c:262-267, after png_read_info) */
                        const uint8_t * end = data + length;
                        const uint8_t * p = (const uint8_t *)memchr(data, 0x0, length);
                        if (p == NULL) continue;
                        p++;
                        std::string text;
                        if (type[0] == 't') {
                                text.assign((const char *)p, end - p);
                        } else {
                                int compressed = 1;
                                if (type[0] == 'i') {
                                        if (end - p < 2) continue;
                                        compressed = p[0];
                                        p += 2;
                                        for (int k = 0; k < 2; k++) { /* language, translated key */
                                                const uint8_t * q =
                                                    (const uint8_t *)memchr(p, 0x0, end - p);
                                                if (q == NULL) {
                                                        p = end;
                                                        break;
                                                }
                                                p = q + 1;
                                        }
                                } else {
                                        if (end - p < 1) continue;
                                        p++; /* compression method */
                                }
                                if (compressed) {
                                        std::vector<uint8_t> plain;
                                        if (inflate_all(p, end - p, plain, 0) != 0) continue;
                                        text.assign((const char *)plain.data(), plain.size());
                                } else {
                                        text.assign((const char *)p, end - p);
                                }
                        }
                        if (png_topography(path, text, h, error) != 0) return -1;
                }
        }
        if (!seen_header || !seen_data)
                return fail(error, TURTLE_RETURN_BAD_FORMAT, PNG_C,
                    "a libpng error occured when loading file `%s'", path);
        if (raw == NULL) return 0;

        /* the passes of the image: one, or the seven of Adam7 (libpng's png_read_image
         * de-interlaces, png16.c:440) -- { x0, y0, dx, dy } */
        static const int adam7[7][4] = { { 0, 0, 8, 8 }, { 4, 0, 8, 8 }, { 0, 4, 4, 8 },
                { 2, 0, 4, 4 }, { 0, 2, 2, 4 }, { 1, 0, 2, 2 }, { 0, 1, 1, 2 } };
        static const int whole[1][4] = { { 0, 0, 1, 1 } };
        const int(*passes)[4] = interlaced ? adam7 : whole;
        const int n_passes = interlaced ? 7 : 1;
        size_t expected = 0;
        for (int k = 0; k < n_passes; k++) {
                const size_t w = ((size_t)h.nx - passes[k][0] + passes[k][2] - 1) / passes[k][2];
                const size_t n = ((size_t)h.ny - passes[k][1] + passes[k][3] - 1) / passes[k][3];
                if ((h.nx > passes[k][0]) && (h.ny > passes[k][1])) expected += (2 * w + 1) * n;
        }
        std::vector<uint8_t> px;
        if ((double)expected > 1100. * (double)idat.size() + 65536.)
                return fail(error, TURTLE_RETURN_BAD_FORMAT, PNG_C,
                    "a libpng error occured when loading file `%s'", path);
        if ((inflate_all(idat.data(), idat.size(), px, expected) != 0) || (px.size() < expected))
                return fail(error, TURTLE_RETURN_BAD_FORMAT, PNG_C,
                    "a libpng error occured when loading file `%s'", path);
        raw->resize((size_t)h.nx * h.ny);
        uint8_t * out = (uint8_t *)raw->data();
        std::vector<uint8_t> lines[2];
        const uint8_t * in = px.data();
        for (int k = 0; k < n_passes; k++) {
                if ((h.nx <= passes[k][0]) || (h.ny <= passes[k][1])) continue; /* empty pass */
                const size_t w = ((size_t)h.nx - passes[k][0] + passes[k][2] - 1) / passes[k][2];
                const size_t n = ((size_t)h.ny - passes[k][1] + passes[k][3] - 1) / passes[k][3];
                const size_t stride = 2 * w;
                lines[0].assign(stride, 0);
                lines[1].assign(stride, 0);
                for (size_t r = 0; r < n; r++) { /* undo the scanline filters, 2 bytes per pixel */
                        uint8_t * cur = lines[r & 1].data();
                        const uint8_t * up = lines[(r & 1) ^ 1].data(); /* zeros above row 0 */
                        const int filter = in[0];
                        in++;
                        if ((filter < 0) || (filter > 4))
                                return fail(error, TURTLE_RETURN_BAD_FORMAT, PNG_C,
                                    "a libpng error occured when loading file `%s'", path);
                        for (size_t i = 0; i < stride; i++) {
                                const int a = (i >= 2) ? cur[i - 2] : 0;
                                const int b = up[i];
                                const int c = (i >= 2) ? up[i - 2] : 0;
                                int pred = 0;
                                if (filter == 1) pred = a;
                                else if (filter == 2) pred = b;
                                else if (filter == 3) pred = (a + b) >> 1;
                                else if (filter == 4) {
                                        const int p0 = a + b - c;
                                        const int pa = abs(p0 - a), pb = abs(p0 - b),
                                                  pc = abs(p0 - c);
                                        pred = ((pa <= pb) && (pa <= pc)) ? a : ((pb <= pc) ? b : c);
                                }
                                cur[i] = (uint8_t)(in[i] + pred);
                        }
                        in += stride;
                        uint8_t * row = out +
                            2 * ((size_t)(passes[k][1] + r * passes[k][3]) * h.nx + passes[k][0]);
                        if (passes[k][2] == 1) {
                                memcpy(row, cur, stride);
                        } else {
                                for (size_t i = 0; i < w; i++) {
                                        row[2 * i * passes[k][2]] = cur[2 * i];
                                        row[2 * i * passes[k][2] + 1] = cur[2 * i + 1];
                                }
                        }
                }
        }
        layout->big_endian = 1;
        layout->north_first = 1;
        return 0;
}

static void put_be32(std::vector<uint8_t> & v, uint32_t x)
{
        v.push_back((uint8_t)(x >> 24));
        v.push_back((uint8_t)(x >> 16));
        v.push_back((uint8_t)(x >> 8));
        v.push_back((uint8_t)x);
}

static void png_chunk(std::vector<uint8_t> & out, const char * type, const uint8_t * data,
    size_t n)
{
        put_be32(out, (uint32_t)n);
        const size_t start = out.size();
        out.insert(out.end(), type, type + 4);
        if (n) out.insert(out.end(), data, data + n);
        put_be32(out, (uint32_t)crc32(crc32(0L, Z_NULL, 0), &out[start], (uInt)(n + 4)));
}

static double node_z(const Header & h, uint16_t raw)
{
        return tb::node_decode(h.kind, h.z0, h.dz, raw);
}

static int png_write(const char * path, const Header & h, const std::vector<uint16_t> & nodes,
    Error & error)
{
        std::vector<uint8_t> out;
        static const uint8_t signature[8] = { 0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a };
        out.insert(out.end(), signature, signature + 8);
        std::vector<uint8_t> ihdr;
        put_be32(ihdr, (uint32_t)h.nx);
        put_be32(ihdr, (uint32_t)h.ny);
        const uint8_t tail[5] = { 16, 0, 0, 0, 0 };
        ihdr.insert(ihdr.end(), tail, tail + 5);
        png_chunk(out, "IHDR", ihdr.data(), ihdr.size());
        /* png16.c:497-515 */
        const double x1 = h.x0 + h.dx * (h.nx - 1);
        const double y1 = h.y0 + h.dy * (h.ny - 1);
        const double z1 = h.z0 + h.dz * 65535;
        char json[2048];
        snprintf(json, sizeof json,
            "{\"topography\" : {\"x0\" : %a, \"y0\" : %a, \"z0\" : %a, \"x1\" : %a, "
            "\"y1\" : %a, \"z1\" : %a, \"projection\" : \"%s\"}}",
            h.x0, h.y0, h.z0, x1, y1, z1, h.projection.c_str());
        std::string text = std::string("Comment") + '\0' + json;
        png_chunk(out, "tEXt", (const uint8_t *)text.data(), text.size());
        /* png16.c:523-536: rows north first, big-endian, re-quantised through get_z */
        const size_t stride = 2 * (size_t)h.nx;
        std::vector<uint8_t> px((stride + 1) * (size_t)h.ny);
        for (int i = 0; i < h.ny; i++) {
                uint8_t * row = &px[(size_t)i * (stride + 1)];
                row[0] = 0;
                const uint16_t * src = &nodes[(size_t)(h.ny - 1 - i) * h.nx];
                for (int j = 0; j < h.nx; j++) {
                        const uint16_t u = to_u16(round((node_z(h, src[j]) - h.z0) / h.dz));
                        row[1 + 2 * j] = (uint8_t)(u >> 8);
                        row[2 + 2 * j] = (uint8_t)u;
                }
        }
        uLongf bound = compressBound((uLong)px.size());
        std::vector<uint8_t> packed(bound);
        if (compress2(packed.data(), &bound, px.data(), (uLong)px.size(), 6) != Z_OK)
                return fail(error, TURTLE_RETURN_MEMORY_ERROR, PNG_C,
                    "could not allocate memory for png proxy");
        png_chunk(out, "IDAT", packed.data(), bound);
        png_chunk(out, "IEND", NULL, 0);
        FILE * fid = fopen(path, "wb+");
        if (fid == NULL)
                return fail(error, TURTLE_RETURN_PATH_ERROR, PNG_C, "could not open file `%s'",
                    path);
        const size_t n = fwrite(out.data(), 1, out.size(), fid);
        fclose(fid);
        if (n != out.size())
                return fail(error, TURTLE_RETURN_PATH_ERROR, PNG_C, "could not open file `%s'",
                    path);
        return 0;
}

/* ---- tif ------------------------------------------------------------------------ */
static const char * TIF_C = "src/turtle/io/geotiff16.c";

struct TiffReader {
        const std::vector<uint8_t> & f;
        int big;
        explicit TiffReader(const std::vector<uint8_t> & f_) : f(f_), big(0) {}
        int ok(size_t at, size_t n) const { return (at <= f.size()) && (n <= f.size() - at); }
        uint16_t u16(size_t at) const
        {
                return big ? (uint16_t)((f[at] << 8) | f[at + 1]) :
                             (uint16_t)((f[at + 1] << 8) | f[at]);
        }
        uint32_t u32(size_t at) const
        {
                return big ? be32(&f[at]) :
                             ((uint32_t)f[at + 3] << 24) | ((uint32_t)f[at + 2] << 16) |
                        ((uint32_t)f[at + 1] << 8) | f[at];
        }
        double f64(size_t at) const
        {
                uint64_t v = 0;
                for (int i = 0; i < 8; i++)
                        v |= (uint64_t)f[at + (big ? 7 - i : i)] << (8 * i);
                double d;
                memcpy(&d, &v, sizeof d);
                return d;
        }
};

/* TIFF LZW (compression 5): MSB-first codes of 9 to 12 bits, ClearCode 256, EndOfInformation
 * 257, the code width growing one code early ("early change") as every libtiff-written
 * file does. Returns 0 on success. */
static int lzw_decode(const uint8_t * src, size_t n, std::vector<uint8_t> & out, size_t expect)
{
        out.clear();
        out.reserve(expect);
        struct Entry { int prefix; uint8_t first, last; uint16_t length; };
        std::vector<Entry> table(4096);
        for (int i = 0; i < 256; i++) {
                table[i].prefix = -1;
                table[i].first = table[i].last = (uint8_t)i;
                table[i].length = 1;
        }
        int next = 258, width = 9, previous = -1;
        uint64_t bits = 0;
        int have = 0;
        size_t at = 0;
        std::vector<uint8_t> scratch;
        for (;;) {
                while ((have < width) && (at < n)) {
                        bits = (bits << 8) | src[at++];
                        have += 8;
                }
                if (have < width) break; /* no EOI: accept what was decoded */
                const int code = (int)((bits >> (have - width)) & ((1u << width) - 1u));
                have -= width;
                if (code == 257) break;
                if (code == 256) {
                        next = 258;
                        width = 9;
                        previous = -1;
                        continue;
                }
                int emit;
                if (code < next) {
                        emit = code;
                } else if ((code == next) && (previous >= 0)) {
                        emit = -1; /* previous string + its own first byte */
                } else {
                        return -1;
                }
                if (emit >= 0) {
                        const int len = table[emit].length;
                        const size_t base = out.size();
                        out.resize(base + len);
                        for (int c = emit, k = len - 1; c >= 0; c = table[c].prefix, k--)
                                out[base + k] = table[c].last;
                } else {
                        const int len = table[previous].length;
                        const size_t base = out.size();
                        out.resize(base + len + 1);
                        for (int c = previous, k = len - 1; c >= 0; c = table[c].prefix, k--)
                                out[base + k] = table[c].last;
                        out[base + len] = table[previous].first;
                }
                if ((previous >= 0) && (next < 4096)) {
                        table[next].prefix = previous;
                        table[next].first = table[previous].first;
                        table[next].last = (emit >= 0) ? table[emit].first : table[previous].first;
                        table[next].length = (uint16_t)(table[previous].length + 1);
                        next++;
                }
                previous = code;
                if (next + 1 >= (1 << width) && (width < 12)) width++; /* early change */
                if (out.size() > expect + 4096) return -1;
        }
        return 0;
}

static int tif_read(const char * path, Header & h, RawLayout * layout,
    std::vector<uint16_t> * raw, Error & error)
{
        std::vector<uint8_t> f;
        if (read_file(path, f) != 0)
                return fail(error, TURTLE_RETURN_PATH_ERROR, TIF_C, "could not open file `%s'",
                    path);
        TiffReader t(f);
        const char * bad = "a libtiff error occured when reading file `%s'";
        if ((f.size() < 8) || !(((f[0] == 'I') && (f[1] == 'I')) || ((f[0] == 'M') && (f[1] == 'M'))))
                return fail(error, TURTLE_RETURN_PATH_ERROR, TIF_C, "could not open file `%s'",
                    path);
        t.big = f[0] == 'M';
        if (t.u16(2) != 42)
                return fail(error, TURTLE_RETURN_PATH_ERROR, TIF_C, "could not open file `%s'",
                    path);
        const size_t ifd = t.u32(4);
        if (!t.ok(ifd, 2)) return fail(error, TURTLE_RETURN_BAD_FORMAT, TIF_C, bad, path);
        const int n_entries = t.u16(ifd);
        if (!t.ok(ifd + 2, (size_t)n_entries * 12))
                return fail(error, TURTLE_RETURN_BAD_FORMAT, TIF_C, bad, path);

        uint32_t width = 0, height = 0, bits = 1, compression = 1, samples = 1, rows_per_strip = 0;
        uint32_t predictor = 1, tiled = 0;
        std::vector<uint32_t> offsets, counts;
        std::vector<double> scale, tie;
        static const int type_size[13] = { 0, 1, 1, 2, 4, 8, 1, 1, 2, 4, 8, 4, 8 };
        for (int e = 0; e < n_entries; e++) {
                const size_t at = ifd + 2 + 12 * (size_t)e;
                const int tag = t.u16(at), type = t.u16(at + 2);
                const uint32_t count = t.u32(at + 4);
                if ((type < 1) || (type > 12)) continue;
                const size_t bytes = (size_t)type_size[type] * count;
                const size_t where = (bytes <= 4) ? at + 8 : t.u32(at + 8);
                if (!t.ok(where, bytes)) return fail(error, TURTLE_RETURN_BAD_FORMAT, TIF_C, bad, path);
                std::vector<uint32_t> ints;
                if ((type == 3) || (type == 4) || (type == 1))
                        for (uint32_t k = 0; k < count; k++)
                                ints.push_back((type == 3) ? t.u16(where + 2 * k) :
                                                             ((type == 4) ? t.u32(where + 4 * k) :
                                                                            f[where + k]));
                const uint32_t first = ints.empty() ? 0 : ints[0];
                switch (tag) {
                case 256: width = first; break;
                case 257: height = first; break;
                case 258: bits = first; break;
                case 259: compression = first; break;
                case 273: offsets = ints; break;
                case 277: samples = first; break;
                case 278: rows_per_strip = first; break;
                case 279: counts = ints; break;
                case 317: predictor = first; break;
                case 322: case 324: tiled = 1; break;
                case 33550:
                        if (type == 12)
                                for (uint32_t k = 0; k < count; k++)
                                        scale.push_back(t.f64(where + 8 * k));
                        break;
                case 33922:
                        if (type == 12)
                                for (uint32_t k = 0; k < count; k++)
                                        tie.push_back(t.f64(where + 8 * k));
                        break;
                default: break;
                }
        }
        /* geotiff16.c:186-215 */
        h = Header();
        h.z0 = -32767.;
        h.dz = 1.;
        h.kind = tb::NODE_DIRECT_I16;
        h.ny = (int)height;
        h.nx = (int)(((size_t)width * bits * samples + 7) / 8 / sizeof(int16_t));
        if (scale.size() == 3) {
                h.dx = scale[0];
                h.dy = scale[1];
        }
        if (tie.size() == 6) {
                h.x0 = tie[3];
                h.y0 = tie[4] + (1 - h.ny) * h.dy;
        }
        if (raw == NULL) return 0;

        if ((bits != 16) || (samples != 1) || tiled || (h.nx <= 0) || (h.ny <= 0) ||
            offsets.empty() || (offsets.size() != counts.size()) ||
            !((compression == 1) || (compression == 5) || (compression == 8) ||
                (compression == 32946)))
                return fail(error, TURTLE_RETURN_BAD_FORMAT, TIF_C, bad, path);
        if (rows_per_strip == 0) rows_per_strip = height;
        /* (deflate expands at most ~1032 times: a grid no file of this size can hold is a
         * corrupt header, not a request for memory) */
        if ((double)h.nx * (double)h.ny * 2. > 1100. * (double)f.size() + 65536.)
                return fail(error, TURTLE_RETURN_BAD_FORMAT, TIF_C, bad, path);
        raw->assign((size_t)h.nx * h.ny, 0);
        const size_t stride = 2 * (size_t)h.nx;
        std::vector<uint8_t> plain;
        for (size_t s = 0; s < offsets.size(); s++) {
                const size_t row0 = s * (size_t)rows_per_strip;
                if (row0 >= height) break;
                const size_t rows = ((row0 + rows_per_strip) <= height) ? rows_per_strip : height - row0;
                if (!t.ok(offsets[s], counts[s]))
                        return fail(error, TURTLE_RETURN_BAD_FORMAT, TIF_C, bad, path);
                const uint8_t * src = &f[offsets[s]];
                size_t have = counts[s];
                if (compression != 1) {
                        const int rc = (compression == 5) ?
                            lzw_decode(src, have, plain, rows * stride) :
                            inflate_all(src, have, plain, rows * stride);
                        if (rc != 0) return fail(error, TURTLE_RETURN_BAD_FORMAT, TIF_C, bad, path);
                        src = plain.data();
                        have = plain.size();
                }
                if (have < rows * stride) return fail(error, TURTLE_RETURN_BAD_FORMAT, TIF_C, bad, path);
                for (size_t r = 0; r < rows; r++) {
                        uint16_t * dst = raw->data() + (row0 + r) * (size_t)h.nx;
                        const uint8_t * p = src + r * stride;
                        for (int i = 0; i < h.nx; i++)
                                dst[i] = t.big ? (uint16_t)((p[2 * i] << 8) | p[2 * i + 1]) :
                                                 (uint16_t)((p[2 * i + 1] << 8) | p[2 * i]);
                        if (predictor == 2)
                                for (int i = 1; i < h.nx; i++) dst[i] = (uint16_t)(dst[i] + dst[i - 1]);
                }
        }
        layout->big_endian = 0; /* converted to native above */
        layout->north_first = 1;
        return 0;
}

static int tif_write(const char * path, const Header & h, const std::vector<uint16_t> & nodes,
    Error & error)
{
        if ((h.z0 != -32767.) || (h.dz != 1.))
                return fail(error, TURTLE_RETURN_BAD_FORMAT, TIF_C,
                    "unsupported z scale when dumping map to `%s'", path);
        if (!h.projection.empty())
                return fail(error, TURTLE_RETURN_BAD_FORMAT, TIF_C,
                    "unsupported projection when dumping map to `%s'", path);
        std::vector<uint8_t> out;
        auto put16 = [&out](uint32_t v) {
                out.push_back((uint8_t)v);
                out.push_back((uint8_t)(v >> 8));
        };
        auto put32 = [&out](uint32_t v) {
                for (int i = 0; i < 4; i++) out.push_back((uint8_t)(v >> (8 * i)));
        };
        auto put64 = [&out](double d) {
                uint64_t v;
                memcpy(&v, &d, sizeof v);
                for (int i = 0; i < 8; i++) out.push_back((uint8_t)(v >> (8 * i)));
        };
        out.push_back('I');
        out.push_back('I');
        put16(42);
        put32(0); /* directory offset, patched below */
        const size_t data_at = out.size();
        for (int i = 0; i < h.ny; i++) { /* geotiff16.c:307-320: rows north first */
                const uint16_t * src = &nodes[(size_t)(h.ny - 1 - i) * h.nx];
                for (int j = 0; j < h.nx; j++) {
                        const double d = round(node_z(h, src[j]));
                        put16((uint16_t)(int16_t)d);
                }
        }
        const size_t scale_at = out.size();
        put64(h.dx);
        put64(h.dy);
        put64(0.);
        const size_t tie_at = out.size();
        const double tie[6] = { 0., 0., 0., h.x0, h.y0 + (h.ny - 1) * h.dy, 0. };
        for (int i = 0; i < 6; i++) put64(tie[i]);
        if (out.size() & 1) out.push_back(0);
        const size_t ifd = out.size();
        struct entry { uint16_t tag, type; uint32_t count, value; };
        const entry entries[] = {
                { 256, 4, 1, (uint32_t)h.nx }, { 257, 4, 1, (uint32_t)h.ny }, { 258, 3, 1, 16 },
                { 259, 3, 1, 1 }, { 262, 3, 1, 1 }, { 273, 4, 1, (uint32_t)data_at },
                { 274, 3, 1, 1 }, { 277, 3, 1, 1 }, { 278, 4, 1, (uint32_t)h.ny },
                { 279, 4, 1, (uint32_t)(2 * (size_t)h.nx * h.ny) }, { 284, 3, 1, 1 },
                { 296, 3, 1, 1 }, { 33550, 12, 3, (uint32_t)scale_at },
                { 33922, 12, 6, (uint32_t)tie_at } };
        const int n = (int)(sizeof(entries) / sizeof(*entries));
        put16(n);
        for (int i = 0; i < n; i++) {
                put16(entries[i].tag);
                put16(entries[i].type);
                put32(entries[i].count);
                if ((entries[i].type == 3) && (entries[i].count == 1)) {
                        put16(entries[i].value);
                        put16(0);
                } else {
                        put32(entries[i].value);
                }
        }
        put32(0);
        for (int i = 0; i < 4; i++) out[4 + i] = (uint8_t)(ifd >> (8 * i));
        FILE * fid = fopen(path, "wb+");
        if (fid == NULL)
                return fail(error, TURTLE_RETURN_PATH_ERROR, TIF_C, "could not create file `%s'",
                    path);
        const size_t w = fwrite(out.data(), 1, out.size(), fid);
        fclose(fid);
        if (w != out.size())
                return fail(error, TURTLE_RETURN_BAD_FORMAT, TIF_C,
                    "a libtiff error occured when writing to file `%s'", path);
        return 0;
}

/* ---- grd / asc (text grids) ------------------------------------------------------ */

/* Both readers scan the values once for the z range with the reference's exact rule
 * (grd.c:86-108, asc.c:84-113: `zmax` starts at -DBL_MIN and a value that lowers zmin
 * never raises zmax), then quantise with z0 = zmin, dz = (zmax - zmin) / 65535. */
static int text_range(FILE * fid, const char * path, const char * file, Header & h,
    const double * nodata, Error & error)
{
        const long offset = ftell(fid);
        double zmin = DBL_MAX, zmax = -DBL_MIN;
        for (int i = 0; i < h.ny; i++)
                for (int j = 0; j < h.nx; j++) {
                        double d;
                        if (fscanf(fid, "%lf", &d) != 1)
                                return fail(error, TURTLE_RETURN_BAD_FORMAT, file,
                                    "inconsistent data in file `%s'", path);
                        if ((nodata != NULL) && (d == *nodata)) continue;
                        if (d < zmin)
                                zmin = d;
                        else if (d > zmax)
                                zmax = d;
                }
        fseek(fid, offset, SEEK_SET);
        h.z0 = zmin;
        h.dz = (zmax - zmin) / 65535;
        h.kind = tb::NODE_AFFINE_U16;
        return 0;
}

static int grd_read(const char * path, Header & h, RawLayout * layout,
    std::vector<uint16_t> * raw, Error & error)
{
        static const char * GRD_C = "src/turtle/io/grd.c";
        FILE * fid = fopen(path, "r");
        if (fid == NULL)
                return fail(error, TURTLE_RETURN_PATH_ERROR, GRD_C, "could not open file `%s'",
                    path);
        h = Header();
        double v[6];
        if (fscanf(fid, "%lf %lf %lf %lf %lf %lf", v, v + 1, v + 2, v + 3, v + 4, v + 5) != 6) {
                fclose(fid);
                return fail(error, TURTLE_RETURN_BAD_FORMAT, GRD_C,
                    "could not read the header of file `%s'", path);
        }
        h.x0 = v[2];
        h.dx = v[5];
        h.y0 = v[0];
        h.dy = v[4];
        h.nx = (int)round((v[3] - v[2]) / v[5]) + 1;
        h.ny = (int)round((v[1] - v[0]) / v[4]) + 1;
        if (text_range(fid, path, GRD_C, h, NULL, error) != 0) {
                fclose(fid);
                return -1;
        }
        if (raw != NULL) { /* grd.c:130-149: line chunks of 127 characters, strtod tokens */
                raw->assign((size_t)h.nx * h.ny, 0);
                long i = 0;
                const long n = (long)h.nx * h.ny;
                char buffer[128];
                while (fgets(buffer, sizeof(buffer), fid) != NULL) {
                        char *start = buffer, *end;
                        for (;; i++) {
                                const double d = strtod(start, &end);
                                if (start == end) break;
                                start = end;
                                if (i < n) /* (the reference writes past the map here) */
                                        (*raw)[i] = to_u16(round((d - h.z0) / h.dz));
                        }
                }
                layout->big_endian = 0;
                layout->north_first = 0;
        }
        fclose(fid);
        return 0;
}

static int asc_read(const char * path, Header & h, RawLayout * layout,
    std::vector<uint16_t> * raw, Error & error)
{
        static const char * ASC_C = "src/turtle/io/asc.c";
        FILE * fid = fopen(path, "r");
        if (fid == NULL)
                return fail(error, TURTLE_RETURN_PATH_ERROR, ASC_C, "could not open file `%s'",
                    path);
        h = Header();
        double nodata;
        if ((fscanf(fid, "%*s %d", &h.nx) != 1) || (fscanf(fid, "%*s %d", &h.ny) != 1) ||
            (fscanf(fid, "%*s %lf", &h.x0) != 1) || (fscanf(fid, "%*s %lf", &h.y0) != 1) ||
            (fscanf(fid, "%*s %lf", &h.dx) != 1) || (fscanf(fid, "%*s %lf", &nodata) != 1)) {
                fclose(fid);
                return fail(error, TURTLE_RETURN_BAD_FORMAT, ASC_C,
                    "could not read the header of file `%s'", path);
        }
        h.dy = h.dx;
        h.x0 += 0.5 * h.dx; /* asc.c:80-82: cell corner -> cell centre */
        h.y0 += 0.5 * h.dy;
        if (text_range(fid, path, ASC_C, h, &nodata, error) != 0) {
                fclose(fid);
                return -1;
        }
        if (raw != NULL) { /* asc.c:138-145: reading order is north first */
                raw->assign((size_t)h.nx * h.ny, 0);
                for (int iy = 0; iy < h.ny; iy++)
                        for (int ix = 0; ix < h.nx; ix++) {
                                double d;
                                if (fscanf(fid, "%lf", &d) != 1) d = 0.;
                                (*raw)[(size_t)iy * h.nx + ix] = to_u16(round((d - h.z0) / h.dz));
                        }
                layout->big_endian = 0;
                layout->north_first = 1;
        }
        fclose(fid);
        return 0;
}

/* ---- dispatch (io.c:73-103) ------------------------------------------------------- */

static int dispatch(const char * path, Header & h, RawLayout * layout,
    std::vector<uint16_t> * raw, Error & error)
{
        const char * ext = extension(path);
        if (!known_extension(ext))
                return fail(error, TURTLE_RETURN_BAD_EXTENSION, "src/turtle/io.c",
                    "no valid format for file `%s'", path);
        int rc;
        RawLayout scratch;
        if (layout == NULL) layout = &scratch;
        if (strcmp(ext, "hgt") == 0)
                rc = (raw != NULL) ? hgt_read(path, h, *layout, *raw, error) :
                                     hgt_header(path, h, error);
        else if (strcmp(ext, "png") == 0)
                rc = png_read(path, h, layout, raw, error);
        else if (strcmp(ext, "tif") == 0)
                rc = tif_read(path, h, layout, raw, error);
        else if (strcmp(ext, "grd") == 0)
                rc = grd_read(path, h, layout, raw, error);
        else
                rc = asc_read(path, h, layout, raw, error);
        if (rc == 0) h.encoding = ext;
        return rc;
}

/* A corrupt header can ask for any amount of memory: allocation failures inside a reader
 * are reported like the reference reports its failed malloc (map.c:131-135), they do not
 * cross the C ABI as exceptions. */
static int guarded(const char * path, Header & h, RawLayout * layout,
    std::vector<uint16_t> * raw, Error & error)
{
        try {
                const int rc = dispatch(path, h, layout, raw, error);
                if ((rc == 0) && ((h.nx <= 0) || (h.ny <= 0)))
                        return fail(error, TURTLE_RETURN_BAD_FORMAT, "src/turtle/io.c",
                            "invalid grid size in file `%s'", path);
                return rc;
        } catch (const std::exception &) {
                return fail(error, TURTLE_RETURN_MEMORY_ERROR, "src/turtle/map.c",
                    "could not allocate memory for map `%s'", path);
        }
}

int read_header(const char * path, Header & header, Error & error)
{
        return guarded(path, header, NULL, NULL, error);
}

int read_map(const char * path, Header & header, RawLayout & layout,
    std::vector<uint16_t> & raw, Error & error)
{
        return guarded(path, header, &layout, &raw, error);
}

void normalise(const Header & h, const RawLayout & layout, std::vector<uint16_t> & raw)
{
        if (layout.big_endian)
                for (size_t i = 0; i < raw.size(); i++)
                        raw[i] = (uint16_t)((raw[i] << 8) | (raw[i] >> 8));
        if (layout.north_first) {
                std::vector<uint16_t> row(h.nx);
                for (int r = 0; r < h.ny / 2; r++) {
                        uint16_t * a = &raw[(size_t)r * h.nx];
                        uint16_t * b = &raw[(size_t)(h.ny - 1 - r) * h.nx];
                        memcpy(row.data(), a, sizeof(uint16_t) * h.nx);
                        memcpy(a, b, sizeof(uint16_t) * h.nx);
                        memcpy(b, row.data(), sizeof(uint16_t) * h.nx);
                }
        }
}

int write_map(const char * path, const Header & header, const std::vector<uint16_t> & nodes,
    Error & error)
{
        const char * ext = extension(path);
        if (!known_extension(ext))
                return fail(error, TURTLE_RETURN_BAD_EXTENSION, "src/turtle/io.c",
                    "no valid format for file `%s'", path);
        if (strcmp(ext, "png") == 0) return png_write(path, header, nodes, error);
        if (strcmp(ext, "tif") == 0) return tif_write(path, header, nodes, error);
        /* hgt.c:51-55, grd.c:52-56, asc.c:50-54 have no writer: their `open` refuses mode "wb" */
        const char * file = (strcmp(ext, "hgt") == 0) ? "src/turtle/io/hgt.c" :
            ((strcmp(ext, "grd") == 0) ? "src/turtle/io/grd.c" : "src/turtle/io/asc.c");
        return fail(error, TURTLE_RETURN_BAD_FORMAT, file,
            "invalid write format for file `%s'", path);
}

} /* namespace tbio */
