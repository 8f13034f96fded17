// track.cu -- host-side track-to-geometry compiler and device upload.
//
// Restates (not copies) the reference's track pipeline for the hot path:
//   ft_grandprix/chunk.py:39-64    threshold (R+G+B == 765), 20x20-px chunk scan in
//                                  column-major (i outer, j inner) order, empty chunks dropped
//   template/mushr.em.xml:19-20    size_x = 20*scale/horizontal_chunks (likewise y)
//   template/mushr.em.xml:55,92    one hfield per chunk at (size_x*i, -size_y*j, -0.1),
//                                  half extents size/2, elevation range 0.3, base 1e-4
//   MuJoCo hfield-from-PNG         rows flipped (PNG top = +Y), data normalised to [0,1];
//                                  a constant (all-wall) chunk normalises to all zeros
//   ft_grandprix/curve.py:6-18     centreline = svg.path Path.point(i/100)
// Output is the packed device blob described in common.h.
#include <cctype>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <algorithm>
#include "common.h"

namespace ftgp {
static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};
void set_error(const char* fmt, ...) {
    va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof g_err, fmt, ap); va_end(ap);
}
bool cuda_ok(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return true;
    set_error("CUDA error %s: %s", what, cudaGetErrorString(e));
    return false;
}
void count_launch(int n) { g_launches += n; }
}  // namespace ftgp
using namespace ftgp;

extern "C" const char* ftgp_last_error(void) { return g_err; }
extern "C" int ftgp_abi_version(void) { return 3; }
extern "C" int64_t ftgp_launch_count(void) { return g_launches.load(); }

extern "C" ftgp_track* ftgp_track_create(const uint8_t* px, int w, int h, int channels,
                                         double scale, int chunk_px) {
    if (!px || w <= 0 || h <= 0 || (channels != 1 && channels != 3 && channels != 4) ||
        chunk_px < 2 || chunk_px > 20 || !(scale > 0)) {
        set_error("ftgp_track_create: bad argument (w=%d h=%d channels=%d chunk_px=%d)", w, h, channels, chunk_px);
        return nullptr;
    }
    auto is_wall = [&](int x, int y) -> bool {
        const uint8_t* p = px + ((size_t)y * w + x) * channels;
        if (channels == 1) return p[0] != 0;
        return (int)p[0] + (int)p[1] + (int)p[2] == 765;      // chunk.py:41
    };
    ftgp_track* t = new ftgp_track();
    t->w = w; t->h = h; t->chunk_px = chunk_px; t->scale = scale;
    t->hc = (w + chunk_px - 1) / chunk_px;
    t->vc = (h + chunk_px - 1) / chunk_px;
    if (t->hc * t->vc >= 0xFFFF) { set_error("track too large: %d x %d chunks", t->hc, t->vc); delete t; return nullptr; }
    t->size_x = 20.0 * scale / t->hc;
    t->size_y = 20.0 * scale / t->vc;
    for (int i = 0; i < t->hc; i++) {
        for (int j = 0; j < t->vc; j++) {
            int x0 = i * chunk_px, y0 = j * chunk_px;
            int ncol = std::min(chunk_px, w - x0), nrow = std::min(chunk_px, h - y0);
            uint32_t m[13] = {0};
            int count = 0;
            for (int r = 0; r < nrow; r++)                       // hfield row r = image row nrow-1-r
                for (int c = 0; c < ncol; c++)
                    if (is_wall(x0 + c, y0 + (nrow - 1 - r))) {
                        int bit = r * ncol + c;
                        m[bit >> 5] |= 1u << (bit & 31);
                        count++;
                    }
            if (count == 0) continue;                            // chunk.py:59
            if (ncol < 2 || nrow < 2) {
                set_error("chunk %dx%d is %dx%d px: MuJoCo needs >= 2x2 hfield samples", i, j, ncol, nrow);
                delete t; return nullptr;
            }
            if (count == ncol * nrow) memset(m, 0, sizeof m);    // constant image -> all-zero elevation
            t->ij.push_back(i); t->ij.push_back(j);
            t->counts.push_back(count);
            t->dims.push_back((uint8_t)ncol); t->dims.push_back((uint8_t)nrow);
            t->masks.insert(t->masks.end(), m, m + 13);
        }
    }
    return t;
}

extern "C" void ftgp_track_destroy(ftgp_track* t) { delete t; }

extern "C" int ftgp_track_meta(const ftgp_track* t, int32_t* out6, double* size_xy2) {
    if (!t || !out6) { set_error("ftgp_track_meta: null"); return FTGP_ERR_ARG; }
    out6[0] = t->hc; out6[1] = t->vc; out6[2] = (int32_t)t->counts.size();
    out6[3] = t->w; out6[4] = t->h; out6[5] = t->chunk_px;
    if (size_xy2) { size_xy2[0] = t->size_x; size_xy2[1] = t->size_y; }
    return FTGP_OK;
}

extern "C" int ftgp_track_chunks(const ftgp_track* t, int32_t* ij, int32_t* counts) {
    if (!t) { set_error("ftgp_track_chunks: null"); return FTGP_ERR_ARG; }
    if (ij) memcpy(ij, t->ij.data(), t->ij.size() * sizeof(int32_t));
    if (counts) memcpy(counts, t->counts.data(), t->counts.size() * sizeof(int32_t));
    return FTGP_OK;
}

// ---------------------------------------------------------------- centreline
// svg.path 6.3 semantics: Path = [Move, CubicBezier | Line ..., Close]; length of a cubic by
// recursive chord bisection (error 1e-12, min depth 5); Path.point(t) picks the segment by
// cumulative length fraction (bisect_right) and evaluates it at the *linear* local parameter.
namespace {
struct Seg { int kind; double p[8]; double len; };   // 0 move, 1 line, 2 cubic
inline void seg_eval(const Seg& s, double u, double& x, double& y) {
    if (s.kind == 0) { x = s.p[0]; y = s.p[1]; }
    else if (s.kind == 1) { x = s.p[0] + (s.p[2] - s.p[0]) * u; y = s.p[1] + (s.p[3] - s.p[1]) * u; }
    else {
        double v = 1 - u;
        double b0 = v * v * v, b1 = 3 * v * v * u, b2 = 3 * v * u * u, b3 = u * u * u;
        x = b0 * s.p[0] + b1 * s.p[2] + b2 * s.p[4] + b3 * s.p[6];
        y = b0 * s.p[1] + b1 * s.p[3] + b2 * s.p[5] + b3 * s.p[7];
    }
}
double bisect_len(const Seg& s, double a, double b, double ax, double ay, double bx, double by, int depth) {
    double m = (a + b) / 2, mx, my;
    seg_eval(s, m, mx, my);
    double chord = std::hypot(bx - ax, by - ay);
    double two = std::hypot(mx - ax, my - ay) + std::hypot(bx - mx, by - my);
    if ((two - chord > 1e-12 || depth < 5) && depth < 40)
        return bisect_len(s, a, m, ax, ay, mx, my, depth + 1) + bisect_len(s, m, b, mx, my, bx, by, depth + 1);
    return two;
}
bool next_number(const char*& p, double& v) {
    while (*p && (isspace((unsigned char)*p) || *p == ',')) p++;
    if (!*p) return false;
    char* e; v = strtod(p, &e);
    if (e == p) return false;
    p = e; return true;
}
}  // namespace

extern "C" int ftgp_centreline(const char* d, int npoints, int img_w, int img_h, int chunk_w,
                               int chunk_h, double scale, double* out) {
    if (!d || !out || npoints <= 0 || img_w <= 0 || img_h <= 0) { set_error("ftgp_centreline: bad argument"); return FTGP_ERR_ARG; }
    std::vector<Seg> segs;
    double cx = 0, cy = 0, sx = 0, sy = 0;
    const char* p = d;
    char cmd = 0;
    for (;;) {
        while (*p && (isspace((unsigned char)*p) || *p == ',')) p++;
        if (!*p) break;
        if (isalpha((unsigned char)*p)) { cmd = *p++; if (cmd != 'z' && cmd != 'Z') continue; }
        bool rel = islower((unsigned char)cmd);
        Seg s{}; double v[6];
        if (cmd == 'm' || cmd == 'M') {
            if (!next_number(p, v[0]) || !next_number(p, v[1])) goto bad;
            if (rel) { v[0] += cx; v[1] += cy; }
            cx = sx = v[0]; cy = sy = v[1];
            s.kind = 0; s.p[0] = cx; s.p[1] = cy; segs.push_back(s);
            cmd = rel ? 'l' : 'L';
        } else if (cmd == 'l' || cmd == 'L') {
            if (!next_number(p, v[0]) || !next_number(p, v[1])) goto bad;
            if (rel) { v[0] += cx; v[1] += cy; }
            s.kind = 1; s.p[0] = cx; s.p[1] = cy; s.p[2] = v[0]; s.p[3] = v[1]; segs.push_back(s);
            cx = v[0]; cy = v[1];
        } else if (cmd == 'c' || cmd == 'C') {
            for (int k = 0; k < 6; k++) if (!next_number(p, v[k])) goto bad;
            if (rel) for (int k = 0; k < 6; k += 2) { v[k] += cx; v[k + 1] += cy; }
            s.kind = 2; s.p[0] = cx; s.p[1] = cy;
            for (int k = 0; k < 6; k++) s.p[2 + k] = v[k];
            segs.push_back(s); cx = v[4]; cy = v[5];
        } else if (cmd == 'z' || cmd == 'Z') {
            s.kind = 1; s.p[0] = cx; s.p[1] = cy; s.p[2] = sx; s.p[3] = sy; segs.push_back(s);
            cx = sx; cy = sy; cmd = 0;
        } else goto bad;
    }
    if (segs.empty()) goto bad;
    {
        double total = 0;
        for (auto& s : segs) {
            if (s.kind == 0) s.len = 0;
            else if (s.kind == 1) s.len = std::hypot(s.p[2] - s.p[0], s.p[3] - s.p[1]);
            else { double ax, ay, bx, by; seg_eval(s, 0, ax, ay); seg_eval(s, 1, bx, by); s.len = bisect_len(s, 0, 1, ax, ay, bx, by, 0); }
            total += s.len;
        }
        std::vector<double> frac(segs.size());
        double f = 0;
        for (size_t k = 0; k < segs.size(); k++) { f += total > 0 ? segs[k].len / total : 0; frac[k] = f; }
        frac.back() = 1.0;
        for (int q = 0; q < npoints; q++) {
            double pos = (double)q / (double)npoints, x, y;
            if (pos == 0.0 || total == 0.0) seg_eval(segs[0], 0.0, x, y);
            else {
                size_t i = 0;
                while (i < segs.size() && frac[i] <= pos) i++;
                if (i >= segs.size()) i = segs.size() - 1;
                double u = i == 0 ? pos / frac[0] : (pos - frac[i - 1]) / (frac[i] - frac[i - 1]);
                seg_eval(segs[i], u, x, y);
            }
            out[2 * q] = x / img_w * chunk_w * scale;            // custom.py:1185
            out[2 * q + 1] = -y / img_h * chunk_h * scale;       // custom.py:1186
        }
    }
    return FTGP_OK;
bad:
    set_error("ftgp_centreline: cannot parse path data near '%.20s'", p);
    return FTGP_ERR_ARG;
}

// ---------------------------------------------------------------- device upload
// the geometry blob (layout: common.h) of up to FTGP_MAX_TRACKS compiled tracks; empty on error
static std::vector<uint32_t> build_blob(const ftgp_track* const* tracks, const double* const* paths, int ntracks) {
    if (!tracks || ntracks < 1 || ntracks > FTGP_MAX_TRACKS) { set_error("geometry: ntracks must be 1..%d", FTGP_MAX_TRACKS); return {}; }
    std::vector<uint32_t> blob(sizeof(GeomHeader) / 4, 0);
    GeomHeader gh{};
    gh.ntracks = ntracks;
    std::vector<int> thdr_off(ntracks);
    for (int k = 0; k < ntracks; k++) {
        const ftgp_track* t = tracks[k];
        if (!t) { set_error("geometry: track %d is null", k); return {}; }
        TrackHeader th{};
        th.hc = t->hc; th.vc = t->vc; th.nchunks = (int)t->counts.size(); th.chunk_px = t->chunk_px;
        th.size_x = (float)t->size_x; th.size_y = (float)t->size_y;
        th.inv_size_x = (float)(1.0 / t->size_x); th.inv_size_y = (float)(1.0 / t->size_y);
        th.dsize_x = t->size_x; th.dsize_y = t->size_y;
        th.dinv_size_x = 1.0 / th.dsize_x; th.dinv_size_y = 1.0 / th.dsize_y;
        th.path_off = -1;
        while (blob.size() % 2) blob.push_back(0);               // 8-byte align the header (doubles inside)
        gh.track_off[k] = thdr_off[k] = (int)blob.size();
        blob.resize(blob.size() + sizeof(TrackHeader) / 4);
        th.index_off = (int)blob.size();
        size_t ncell = (size_t)t->hc * t->vc;
        std::vector<uint16_t> index(ncell + (ncell & 1), EMPTY_CHUNK);
        for (int c = 0; c < th.nchunks; c++) {
            int i = t->ij[2 * c], j = t->ij[2 * c + 1];
            index[(size_t)(t->vc - 1 - j) * t->hc + i] = (uint16_t)c;
        }
        blob.resize(blob.size() + index.size() / 2);
        memcpy(&blob[th.index_off], index.data(), index.size() * 2);
        th.chunks_off = (int)blob.size();
        for (int c = 0; c < th.nchunks; c++) {
            for (int wd = 0; wd < 13; wd++) blob.push_back(t->masks[(size_t)c * 13 + wd]);
            const int ncol = t->dims[2 * c], nrow = t->dims[2 * c + 1];
            blob.push_back((uint32_t)ncol | ((uint32_t)nrow << 8));
            int cmin = 255, cmax = 0, rmin = 255, rmax = 0;
            for (int r = 0; r < nrow; r++)
                for (int cc = 0; cc < ncol; cc++) {
                    const int bit = r * ncol + cc;
                    if ((t->masks[(size_t)c * 13 + (bit >> 5)] >> (bit & 31)) & 1u) {
                        cmin = std::min(cmin, cc); cmax = std::max(cmax, cc); rmin = std::min(rmin, r); rmax = std::max(rmax, r);
                    }
                }
            if (cmin > cmax) { cmin = 200; cmax = 100; rmin = 200; rmax = 100; }      // no wall vertex: empty box
            blob.push_back((uint32_t)cmin | ((uint32_t)cmax << 8) | ((uint32_t)rmin << 16) | ((uint32_t)rmax << 24));
            uint32_t mt[13] = {0};                                   // transposed copy
            for (int r = 0; r < nrow; r++)
                for (int cc = 0; cc < ncol; cc++) {
                    const int bit = r * ncol + cc;
                    if ((t->masks[(size_t)c * 13 + (bit >> 5)] >> (bit & 31)) & 1u) { const int bt = cc * nrow + r; mt[bt >> 5] |= 1u << (bt & 31); }
                }
            for (int wd = 0; wd < 13; wd++) blob.push_back(mt[wd]);
        }
        memcpy(&blob[thdr_off[k]], &th, sizeof th);
    }
    gh.lidar_words = (int)blob.size();
    for (int k = 0; k < ntracks; k++) {
        if (!paths || !paths[k]) continue;
        while (blob.size() % 2) blob.push_back(0);
        TrackHeader th; memcpy(&th, &blob[thdr_off[k]], sizeof th);
        th.path_off = (int)blob.size();
        blob.resize(blob.size() + FTGP_NPATH * 2 * 2);
        memcpy(&blob[th.path_off], paths[k], sizeof(double) * FTGP_NPATH * 2);
        memcpy(&blob[thdr_off[k]], &th, sizeof th);
    }
    while (blob.size() % 4) blob.push_back(0);
    gh.total_words = (int)blob.size();
    memcpy(blob.data(), &gh, sizeof gh);
    return blob;
}

extern "C" int64_t ftgp_geom_blob(const ftgp_track* const* tracks, const double* const* paths, int ntracks,
                                  uint32_t* out, int64_t cap_words) {
    const std::vector<uint32_t> blob = build_blob(tracks, paths, ntracks);
    if (blob.empty()) return -1;
    if (out && cap_words >= (int64_t)blob.size()) memcpy(out, blob.data(), blob.size() * 4);
    return (int64_t)blob.size();
}

extern "C" int ftgp_blob_track_view(const uint32_t* blob, int track, int32_t* out4, double* size_xy2) {
    if (!blob || !out4 || !size_xy2) { set_error("ftgp_blob_track_view: bad argument"); return FTGP_ERR_ARG; }
    GeomHeader gh; memcpy(&gh, blob, sizeof gh);
    if (track < 0 || track >= gh.ntracks) { set_error("ftgp_blob_track_view: no such track"); return FTGP_ERR_ARG; }
    TrackHeader th; memcpy(&th, blob + gh.track_off[track], sizeof th);
    out4[0] = th.index_off; out4[1] = th.chunks_off; out4[2] = th.hc; out4[3] = th.vc;
    size_xy2[0] = th.dsize_x; size_xy2[1] = th.dsize_y;
    return FTGP_OK;
}

extern "C" ftgp_geom* ftgp_geom_create(const ftgp_track* const* tracks, const double* const* paths,
                                       int ntracks, int device) {
    std::vector<uint32_t> blob = build_blob(tracks, paths, ntracks);
    if (blob.empty()) return nullptr;
    ftgp_geom* g = new ftgp_geom();
    g->device = device; g->ntracks = ntracks; g->bytes = (int64_t)blob.size() * 4;
    g->h_blob = blob;
    if (!cuda_ok(cudaSetDevice(device), "cudaSetDevice") ||
        !cuda_ok(cudaMalloc(&g->d_blob, g->bytes), "cudaMalloc(geom)") ||
        !cuda_ok(cudaMemcpy(g->d_blob, blob.data(), g->bytes, cudaMemcpyHostToDevice), "cudaMemcpy(geom)") ||
        !cuda_ok(cudaStreamCreateWithFlags(&g->host_stream, cudaStreamNonBlocking), "cudaStreamCreate")) {
        if (g->d_blob) cudaFree(g->d_blob);
        delete g;
        return nullptr;
    }
    return g;
}

extern "C" void ftgp_geom_destroy(ftgp_geom* g) {
    if (!g) return;
    cudaSetDevice(g->device);
    ftgp::forget_geom(g);
    if (g->d_scratch) cudaFree(g->d_scratch);
    if (g->d_blob) cudaFree(g->d_blob);
    if (g->host_stream) cudaStreamDestroy(g->host_stream);
    delete g;
}
extern "C" int ftgp_geom_device(const ftgp_geom* g) { return g ? g->device : -1; }
extern "C" int64_t ftgp_geom_bytes(const ftgp_geom* g) { return g ? g->bytes : 0; }
