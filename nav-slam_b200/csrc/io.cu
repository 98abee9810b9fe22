// io.cu -- the data formats either side of the path (SURVEY 8f #3, #4), host code inside the C-ABI
// library: the L9 CSV reader of src/main.c:77-128 and the 25-column CSV row writer of
// src/main.c:243,320-352, both byte/bit compatible with the reference and several times faster
// (no fscanf / fprintf in the loop).  These are the callers' formats, not kernels: nothing here touches
// the GPU, and frames are parsed straight into caller memory (pinned memory from nav_host_alloc
// makes them a DMA source for the frame calls).
#include <ctype.h>
#include <errno.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/navslam_b200.h"
#include "csv_fixed2.cuh"

extern "C" const char *nav_last_error(void);
int nav_io_fail(const char *fmt, ...);  // defined in capi.cu (sets the thread-local error)

// ---------------------------------------------------------------------------------- reader -----
// src/main.c:86-118: skip one header line (at most 255 characters are consumed by the reference's
// fgets), then records "%d,%d,%d,%lf,%lf,%lf,%d" until the first one that does not parse.  A record
// whose row/col is out of range is skipped without touching the frame bookkeeping; a change of the
// frame number starts the next frame slot.  Unlike the reference (col > MAX_COLS, main.c:100) a
// record with col == cols is rejected instead of written out of bounds.
namespace {

inline const char *skip_ws(const char *p, const char *end) {  // fscanf directives skip leading white space
    while (p < end && (*p == ' ' || *p == '\n' || *p == '\t' || *p == '\r' || *p == '\v' || *p == '\f')) ++p;
    return p;
}

inline bool parse_int(const char *&p, const char *end, int &out) {
    p = skip_ws(p, end);
    const char *q = p;
    bool neg = false;
    if (q < end && (*q == '-' || *q == '+')) neg = *q++ == '-';
    if (q >= end || *q < '0' || *q > '9') return false;
    long long v = 0;
    while (q < end && *q >= '0' && *q <= '9') {
        v = v * 10 + (*q++ - '0');
        if (v > 0x7fffffffLL + 1) v = 0x7fffffffLL + 1;
    }
    out = (int)(neg ? -v : v);
    p = q;
    return true;
}

inline bool parse_double(const char *&p, const char *end, double &out) {
    p = skip_ws(p, end);
    if (p >= end) return false;
    // fast path: optional sign, up to 15 significant digits with an optional fraction, no exponent:
    // the value is an exactly representable integer divided by an exactly representable power of ten,
    // which one IEEE division rounds correctly -- the same result strtod / fscanf("%lf") give.
    const char *q = p;
    bool neg = false;
    if (*q == '-' || *q == '+') neg = *q++ == '-';
    unsigned long long mant = 0;
    int digits = 0, frac = 0;
    bool any = false;
    while (q < end && *q >= '0' && *q <= '9') {
        mant = mant * 10 + (unsigned)(*q++ - '0');
        if (mant) ++digits;
        any = true;
    }
    if (q < end && *q == '.') {
        ++q;
        while (q < end && *q >= '0' && *q <= '9') {
            mant = mant * 10 + (unsigned)(*q++ - '0');
            if (mant) ++digits;
            ++frac;
            any = true;
        }
    }
    static const double p10[] = {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12, 1e13, 1e14, 1e15,
                                 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22};
    const bool simple = any && digits <= 15 && frac <= 22 && (q >= end || (*q != 'e' && *q != 'E' && *q != 'x' && *q != 'X' &&
                                                                          *q != 'n' && *q != 'N' && *q != 'i' && *q != 'I'));
    if (simple) {
        const double v = (double)mant / p10[frac];
        out = neg ? -v : v;
        p = q;
        return true;
    }
    // anything else (exponents, inf/nan, long mantissas): the C library, on a bounded copy
    char tmp[512];
    size_t len = (size_t)(end - p) < sizeof(tmp) - 1 ? (size_t)(end - p) : sizeof(tmp) - 1;
    memcpy(tmp, p, len);
    tmp[len] = 0;
    char *stop = nullptr;
    const double v = strtod(tmp, &stop);
    if (stop == tmp) return false;
    out = v;
    p += stop - tmp;
    return true;
}

inline bool expect(const char *&p, const char *end, char c) {  // a literal in the format: no white-space skipping
    if (p < end && *p == c) {
        ++p;
        return true;
    }
    return false;
}

}  // namespace

namespace {

// the record loop of both L9 readers.  store(i, v) puts the record's x y z into pixel i (frame-major) and returns the
// index (0..2) of a value it cannot store, or -1; a refused value fails the call with its line and text.
template <class Store>
int l9_csv_parse(const char *fn, const char *path, int rows, int cols, size_t max_frames, int *timestamps_out,
                 size_t *n_frames_out, Store store) {
    *n_frames_out = 0;
    FILE *fp = fopen(path, "rb");
    if (!fp) return nav_io_fail("%s: cannot open %s: %s", fn, path, strerror(errno));
    std::string text;
    {
        char chunk[1 << 16];
        size_t got;
        while ((got = fread(chunk, 1, sizeof(chunk), fp)) > 0) text.append(chunk, got);
        fclose(fp);
    }
    const char *p = text.data(), *end = p + text.size();
    {   // fgets(header, 256): at most 255 characters, stopping after the first newline
        size_t n = 0;
        while (p < end && n < 255) {
            ++n;
            if (*p++ == '\n') break;
        }
        if (n == 0) return 0;  // empty file: zero frames, like the reference
    }
    const size_t npx = (size_t)rows * cols;
    long long current = -1;
    bool have_frame = false;
    size_t count = 0;  // index of the frame being filled
    while (true) {
        int frame, row, col, conf;
        double v[3];
        const char *tok[3], *tok_end[3];  // where each of x y z was read (for the error of a refused value)
        const char *q = p;
        auto coord = [&](int k) {
            tok[k] = q;
            const bool ok = parse_double(q, end, v[k]);
            tok_end[k] = q;
            return ok;
        };
        if (!(parse_int(q, end, frame) && expect(q, end, ',') && parse_int(q, end, row) && expect(q, end, ',') &&
              parse_int(q, end, col) && expect(q, end, ',') && coord(0) && expect(q, end, ',') && coord(1) &&
              expect(q, end, ',') && coord(2) && expect(q, end, ',') && parse_int(q, end, conf)))
            break;
        p = q;
        if (row < 0 || row >= rows || col < 0 || col >= cols) continue;
        if (!have_frame || frame != current) {
            if (have_frame) ++count;
            if (count >= max_frames) {  // the reference overruns its lidarData[10] here; stop instead
                *n_frames_out = max_frames;
                return nav_io_fail("%s: more than %zu frames in %s", fn, max_frames, path);
            }
            have_frame = true;
            current = frame;
            if (timestamps_out) timestamps_out[count] = frame;
        }
        const int bad = store(count * npx + (size_t)row * cols + col, v);
        if (bad >= 0) {
            const char *t = skip_ws(tok[bad], tok_end[bad]);
            size_t line = 1;
            for (const char *c = text.data(); c < t; ++c) line += *c == '\n';
            return nav_io_fail("%s: line %zu of %s: %c = '%.*s' is not a whole number of millimetres that int32 holds "
                               "with the same binary64 bits (fractions, |v| > 2^31-1, inf, nan and -0 are refused)",
                               fn, line, path, "xyz"[bad], (int)(tok_end[bad] - t), t);
        }
    }
    *n_frames_out = have_frame ? count + 1 : 0;
    return 0;
}

}  // namespace

extern "C" int nav_l9_csv_read(const char *path, int rows, int cols, size_t max_frames, nav_point *frames_out,
                               int *timestamps_out, size_t *n_frames_out) {
    if (!path || !frames_out || !n_frames_out || rows < 1 || cols < 1)
        return nav_io_fail("nav_l9_csv_read: bad argument");
    return l9_csv_parse("nav_l9_csv_read", path, rows, cols, max_frames, timestamps_out, n_frames_out,
                        [&](size_t i, const double v[3]) {
                            frames_out[i].x = v[0];
                            frames_out[i].y = v[1];
                            frames_out[i].z = v[2];
                            return -1;
                        });
}

extern "C" int nav_l9_csv_read_mm(const char *path, int rows, int cols, size_t max_frames, int32_t *frames_out,
                                  int *timestamps_out, size_t *n_frames_out) {
    if (!path || !frames_out || !n_frames_out || rows < 1 || cols < 1)
        return nav_io_fail("nav_l9_csv_read_mm: bad argument");
    return l9_csv_parse("nav_l9_csv_read_mm", path, rows, cols, max_frames, timestamps_out, n_frames_out,
                        [&](size_t i, const double v[3]) {
                            for (int k = 0; k < 3; ++k) {
                                // in range first (the conversion of anything else is undefined), then the
                                // bits: this refuses fractions and -0.0, whose int32 widens to +0.0
                                if (!(v[k] >= -2147483648.0 && v[k] <= 2147483647.0)) return k;
                                const int32_t m = (int32_t)v[k];
                                const double back = (double)m;
                                if (memcmp(&back, &v[k], sizeof(double)) != 0) return k;
                                frames_out[i * 3 + k] = m;
                            }
                            return -1;
                        });
}

// ---------------------------------------------------------------------------------- writer -----
namespace {

// printf("%.2f") of any double: the integer path of csv_fixed2.cuh, the C library for inf / nan / >= 2^57
inline char *fmt_fixed2(char *o, double v) {
    bool neg;
    unsigned long long q;
    if (nav::fixed2_scaled(v, neg, q)) return nav::put_fixed2(o, neg, q);
    char tmp[400];
    const int n = snprintf(tmp, sizeof(tmp), "%.2f", v);
    memcpy(o, tmp, (size_t)n);
    return o + n;
}

inline char *fmt_uint(char *o, unsigned long long v) { return nav::put_uint(o, v, nav::dec_len(v)); }
inline char *fmt_int(char *o, long long v) { return nav::put_int(o, v); }

}  // namespace

namespace nav {
// ",%.2f" x 18 + "\n" (src/main.c:331-348); out needs 18 * 340 + 2 bytes for arbitrary doubles
size_t csv_pose_columns(char *out, const double imu[6], const nav_pos *lidar_pos, const nav_pos *ekf_pos) {
    char *t = out;
    const double zero6[6] = {0, 0, 0, 0, 0, 0};
    const double *im = imu ? imu : zero6;
    for (int i = 0; i < 6; ++i) {
        *t++ = ',';
        t = fmt_fixed2(t, im[i]);
    }
    const double lp[6] = {lidar_pos->x, lidar_pos->y, lidar_pos->z, lidar_pos->roll, lidar_pos->pitch, lidar_pos->yaw};
    for (int i = 0; i < 6; ++i) {
        *t++ = ',';
        t = fmt_fixed2(t, lp[i]);
    }
    const double ep[6] = {ekf_pos ? ekf_pos->x : 0, ekf_pos ? ekf_pos->y : 0, ekf_pos ? ekf_pos->z : 0,
                          ekf_pos ? ekf_pos->roll : 0, ekf_pos ? ekf_pos->pitch : 0, ekf_pos ? ekf_pos->yaw : 0};
    for (int i = 0; i < 6; ++i) {
        *t++ = ',';
        t = fmt_fixed2(t, ep[i]);
    }
    *t++ = '\n';
    return (size_t)(t - out);
}
}  // namespace nav

extern "C" const char *nav_csv_header(void) {
    // src/main.c:243
    return "Timestamp,Row,Col,x,y,z,distance,IMU_x,IMU_y,IMU_z,IMU_roll,IMU_pitch,IMU_yaw,LiDAR_x,LiDAR_y,LiDAR_z,"
           "LiDAR_roll,LiDAR_pitch,LiDAR_yaw,EKF_x,EKF_y,EKF_z,EKF_roll,EKF_pitch,EKF_yaw\n";
}

// One frame = rows*cols lines of src/main.c:324-349 (the L5 handler, which passes a double to every
// %.2f).  distances == NULL prints 0, imu == NULL / ekf_pos == NULL print 0.00 in their six columns: what
// the L9 handler (main.c:437-461) means by its literal 0 arguments -- as written it hands ints to %.2f,
// which is undefined behaviour and not reproduced.
extern "C" size_t nav_csv_format_frame(char *buf, size_t cap, unsigned long long timestamp, int rows, int cols,
                                       const nav_point *global_cloud, const int *distances, const double imu[6],
                                       const nav_pos *lidar_pos, const nav_pos *ekf_pos) {
    if (!buf || !global_cloud || !lidar_pos || rows < 1 || cols < 1) return 0;
    // the 18 pose columns are the same text on every line of the frame
    char tail[18 * 340 + 4];
    const size_t tail_len = nav::csv_pose_columns(tail, imu, lidar_pos, ekf_pos);
    char *o = buf;
    char *const lim = buf + cap;
    char head[3 * 340 + 80];
    for (int r = 0; r < rows; ++r) {
        for (int c = 0; c < cols; ++c) {
            const nav_point &p = global_cloud[(size_t)r * cols + c];
            char *h = fmt_uint(head, timestamp);
            *h++ = ',';
            h = fmt_int(h, r);
            *h++ = ',';
            h = fmt_int(h, c);
            *h++ = ',';
            h = fmt_fixed2(h, p.x);
            *h++ = ',';
            h = fmt_fixed2(h, p.y);
            *h++ = ',';
            h = fmt_fixed2(h, p.z);
            *h++ = ',';
            h = fmt_int(h, distances ? distances[(size_t)r * cols + c] : 0);
            const size_t head_len = (size_t)(h - head);
            if ((size_t)(lim - o) < head_len + tail_len) return 0;  // caller's buffer too small
            memcpy(o, head, head_len);
            memcpy(o + head_len, tail, tail_len);
            o += head_len + tail_len;
        }
    }
    return (size_t)(o - buf);
}

// ------------------------------------------------------------------------- L5 JSON readers -----
// LidarProcessData / IMUProcessData (src/main.c:12-75,130-178) read `parsed_data.json` through
// jansson: a top-level array of objects {"time_main": int, "distance": [int...], "params": [6 reals]}.
// This is a small validating JSON scanner for exactly that use: the whole document must be one valid
// JSON value followed by white space only (json_loadf with flags 0), otherwise nothing is read.
// Differences from jansson that do not matter for data files: invalid UTF-8 inside strings is accepted.
namespace {

struct JsonScan {
    const char *p, *end;
    bool ok = true;
    void ws() {
        while (p < end && (*p == ' ' || *p == '\n' || *p == '\t' || *p == '\r')) ++p;
    }
    bool lit(const char *s) {
        const size_t n = strlen(s);
        if ((size_t)(end - p) >= n && memcmp(p, s, n) == 0) {
            p += n;
            return true;
        }
        return ok = false;
    }
    // string: returns its raw bytes (escapes are validated, not decoded: keys of interest have none)
    bool str(std::string *out) {
        if (p >= end || *p != '"') return ok = false;
        ++p;
        const char *s0 = p;
        while (p < end && *p != '"') {
            if ((unsigned char)*p < 0x20) return ok = false;
            if (*p == '\\') {
                ++p;
                if (p >= end) return ok = false;
                if (*p == 'u') {
                    for (int i = 1; i <= 4; ++i)
                        if (p + i >= end || !isxdigit((unsigned char)p[i])) return ok = false;
                    p += 4;
                } else if (!strchr("\"\\/bfnrt", *p)) {
                    return ok = false;
                }
            }
            ++p;
        }
        if (p >= end) return ok = false;
        if (out) out->assign(s0, p);
        ++p;
        return true;
    }
    // number: JSON grammar; integer iff it has no fraction and no exponent (jansson's rule)
    bool num(bool *is_int, long long *iv, double *dv) {
        const char *s0 = p;
        if (p < end && *p == '-') ++p;
        if (p >= end) return ok = false;
        if (*p == '0') {
            ++p;
        } else if (*p >= '1' && *p <= '9') {
            while (p < end && *p >= '0' && *p <= '9') ++p;
        } else {
            return ok = false;
        }
        bool integer = true;
        if (p < end && *p == '.') {
            integer = false;
            ++p;
            if (p >= end || *p < '0' || *p > '9') return ok = false;
            while (p < end && *p >= '0' && *p <= '9') ++p;
        }
        if (p < end && (*p == 'e' || *p == 'E')) {
            integer = false;
            ++p;
            if (p < end && (*p == '+' || *p == '-')) ++p;
            if (p >= end || *p < '0' || *p > '9') return ok = false;
            while (p < end && *p >= '0' && *p <= '9') ++p;
        }
        char tmp[400];
        const size_t len = (size_t)(p - s0);
        if (len >= sizeof(tmp)) return ok = false;
        memcpy(tmp, s0, len);
        tmp[len] = 0;
        errno = 0;
        if (integer) {
            const long long v = strtoll(tmp, nullptr, 10);
            if (errno == ERANGE) return ok = false;  // jansson: "too big integer"
            if (iv) *iv = v;
        } else {
            const double v = strtod(tmp, nullptr);
            if (errno == ERANGE && (v == HUGE_VAL || v == -HUGE_VAL)) return ok = false;  // jansson: real overflow
            if (dv) *dv = v;
        }
        if (is_int) *is_int = integer;
        return true;
    }
    bool skip_value(int depth = 0) {
        if (depth > 2048) return ok = false;  // jansson's JSON_PARSER_MAX_DEPTH
        ws();
        if (p >= end) return ok = false;
        switch (*p) {
            case '{': {
                ++p;
                ws();
                if (p < end && *p == '}') return ++p, true;
                while (true) {
                    ws();
                    if (!str(nullptr)) return false;
                    ws();
                    if (p >= end || *p != ':') return ok = false;
                    ++p;
                    if (!skip_value(depth + 1)) return false;
                    ws();
                    if (p < end && *p == ',') {
                        ++p;
                        continue;
                    }
                    if (p < end && *p == '}') return ++p, true;
                    return ok = false;
                }
            }
            case '[': {
                ++p;
                ws();
                if (p < end && *p == ']') return ++p, true;
                while (true) {
                    if (!skip_value(depth + 1)) return false;
                    ws();
                    if (p < end && *p == ',') {
                        ++p;
                        continue;
                    }
                    if (p < end && *p == ']') return ++p, true;
                    return ok = false;
                }
            }
            case '"': return str(nullptr);
            case 't': return lit("true");
            case 'f': return lit("false");
            case 'n': return lit("null");
            default: return num(nullptr, nullptr, nullptr);
        }
    }
};

struct JsonNum {
    bool is_num, is_int;
    long long iv;
    double dv;
};

// one element of the top-level array: what the two readers look at
struct L5Record {
    bool is_object = false;
    bool has_time = false;  // "time_main" present and an integer
    long long time_main = 0;
    bool has_distance = false, has_params = false;  // present and arrays
    std::vector<JsonNum> distance, params;
};

bool read_num_array(JsonScan &js, std::vector<JsonNum> &out) {  // at '[': every element recorded, numbers decoded
    out.clear();
    ++js.p;
    js.ws();
    if (js.p < js.end && *js.p == ']') return ++js.p, true;
    while (true) {
        js.ws();
        JsonNum v = {false, false, 0, 0.0};
        if (js.p < js.end && (*js.p == '-' || (*js.p >= '0' && *js.p <= '9'))) {
            v.is_num = true;
            if (!js.num(&v.is_int, &v.iv, &v.dv)) return false;
        } else if (!js.skip_value(1)) {
            return false;
        }
        out.push_back(v);
        js.ws();
        if (js.p < js.end && *js.p == ',') {
            ++js.p;
            continue;
        }
        if (js.p < js.end && *js.p == ']') return ++js.p, true;
        return js.ok = false;
    }
}

bool read_record(JsonScan &js, L5Record &r) {
    js.ws();
    if (js.p >= js.end) return js.ok = false;
    if (*js.p != '{') return js.skip_value(1);
    r.is_object = true;
    ++js.p;
    js.ws();
    if (js.p < js.end && *js.p == '}') return ++js.p, true;
    while (true) {
        js.ws();
        std::string key;
        if (!js.str(&key)) return false;
        js.ws();
        if (js.p >= js.end || *js.p != ':') return js.ok = false;
        ++js.p;
        js.ws();
        // a repeated key replaces the earlier value, as in jansson's object
        if (key == "time_main") {
            r.has_time = false;
            if (js.p < js.end && (*js.p == '-' || (*js.p >= '0' && *js.p <= '9'))) {
                bool is_int;
                long long iv = 0;
                if (!js.num(&is_int, &iv, nullptr)) return false;
                r.has_time = is_int;
                r.time_main = iv;
            } else if (!js.skip_value(1)) {
                return false;
            }
        } else if (key == "distance" || key == "params") {
            bool &has = key == "distance" ? r.has_distance : r.has_params;
            std::vector<JsonNum> &dst = key == "distance" ? r.distance : r.params;
            has = false;
            if (js.p < js.end && *js.p == '[') {
                if (!read_num_array(js, dst)) return false;
                has = true;
            } else if (!js.skip_value(1)) {
                return false;
            }
        } else if (!js.skip_value(1)) {
            return false;
        }
        js.ws();
        if (js.p < js.end && *js.p == ',') {
            ++js.p;
            continue;
        }
        if (js.p < js.end && *js.p == '}') return ++js.p, true;
        return js.ok = false;
    }
}

// the whole document -> records; false if it is not valid JSON (then the reference reads nothing either)
int load_l5_records(const char *fn, const char *path, std::vector<L5Record> &recs, bool *root_is_array) {
    FILE *fp = fopen(path, "rb");
    if (!fp) return nav_io_fail("%s: cannot open %s: %s", fn, path, strerror(errno));
    std::string text;
    char chunk[1 << 16];
    size_t got;
    while ((got = fread(chunk, 1, sizeof(chunk), fp)) > 0) text.append(chunk, got);
    fclose(fp);
    JsonScan js;
    js.p = text.data();
    js.end = js.p + text.size();
    js.ws();
    *root_is_array = js.p < js.end && *js.p == '[';
    if (!*root_is_array) {
        if (!js.skip_value()) return nav_io_fail("%s: %s is not valid JSON", fn, path);
    } else {
        ++js.p;
        js.ws();
        if (js.p < js.end && *js.p == ']') {
            ++js.p;
        } else {
            while (true) {
                recs.emplace_back();
                if (!read_record(js, recs.back())) return nav_io_fail("%s: %s is not valid JSON", fn, path);
                js.ws();
                if (js.p < js.end && *js.p == ',') {
                    ++js.p;
                    continue;
                }
                if (js.p < js.end && *js.p == ']') {
                    ++js.p;
                    break;
                }
                return nav_io_fail("%s: %s is not valid JSON", fn, path);
            }
        }
    }
    js.ws();
    if (js.p != js.end) return nav_io_fail("%s: %s has text after the JSON value", fn, path);
    return 0;
}

}  // namespace

extern "C" int nav_l5_json_read(const char *path, int rows, int cols, size_t max_frames, int *distances_out,
                                int *timestamps_out, size_t *n_frames_out) {
    if (!path || !distances_out || !n_frames_out || rows < 1 || cols < 1)
        return nav_io_fail("nav_l5_json_read: bad argument");
    *n_frames_out = 0;
    std::vector<L5Record> recs;
    bool is_array = false;
    if (load_l5_records("nav_l5_json_read", path, recs, &is_array)) return 1;
    if (!is_array) return 0;  // main.c:31: nothing to do unless the root is a non-empty array
    if (recs.size() > max_frames)  // the reference overruns lidarData[100] here
        return nav_io_fail("nav_l5_json_read: %zu frames in %s, room for %zu", recs.size(), path, max_frames);
    const size_t npx = (size_t)rows * cols;
    for (size_t f = 0; f < recs.size(); ++f) {
        const L5Record &r = recs[f];
        if (r.is_object) {
            if (r.has_time && timestamps_out) timestamps_out[f] = (int)r.time_main;  // main.c:44-48
            if (r.has_distance)
                for (size_t i = 0; i < r.distance.size() && i < npx; ++i)           // main.c:55-63
                    if (r.distance[i].is_num && r.distance[i].is_int) distances_out[f * npx + i] = (int)r.distance[i].iv;
        }
    }
    *n_frames_out = recs.size();  // main.c:67: every array element advances the frame count
    return 0;
}

extern "C" int nav_imu_json_read(const char *path, size_t max_frames, double *params_out, int *timestamps_out,
                                 size_t *n_frames_out) {
    if (!path || !params_out || !n_frames_out) return nav_io_fail("nav_imu_json_read: bad argument");
    *n_frames_out = 0;
    std::vector<L5Record> recs;
    bool is_array = false;
    if (load_l5_records("nav_imu_json_read", path, recs, &is_array)) return 1;
    if (!is_array) return 0;
    size_t count = 0;
    for (const L5Record &r : recs) {
        if (!r.is_object) continue;  // main.c:157: only objects advance the IMU count
        if (count >= max_frames) return nav_io_fail("nav_imu_json_read: more than %zu frames in %s", max_frames, path);
        if (r.has_time && timestamps_out) timestamps_out[count] = (int)r.time_main;
        if (r.has_params && r.params.size() == 6)  // main.c:168-176; json_real_value() is 0.0 for a non-real
            for (int k = 0; k < 6; ++k)
                params_out[count * 6 + k] = (r.params[k].is_num && !r.params[k].is_int) ? r.params[k].dv : 0.0;
        ++count;
    }
    *n_frames_out = count;
    return 0;
}
