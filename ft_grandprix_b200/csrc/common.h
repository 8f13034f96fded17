// common.h -- shared internals of libftgp.so (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>
#include "../../include/ftgp.h"

namespace ftgp {

void set_error(const char* fmt, ...);
bool cuda_ok(cudaError_t e, const char* what);
void count_launch(int n = 1);


#define FTGP_CUDA(call)                                        \
    do {                                                       \
        if (!ftgp::cuda_ok((call), #call)) return FTGP_ERR_CUDA; \
    } while (0)

// ---- policy bank (policy.cu) ----------------------------------------------
// checked before any CUDA call: a bank needs weights and at least one policy; FTGP_DRIVER_POLICY as the default needs a bank
inline bool bad_policy_args(const ftgp_policy_args* p, int default_kind) {
    if (!p) return default_kind == FTGP_DRIVER_POLICY;
    return !p->weights || p->npolicies < 1;
}
// the POLICY cars of the fleet, grouped by policy id, then evaluated (after drivers_kernel, which skips them)
int launch_policy(const ftgp_policy_args* p, const float* ranges, const int32_t* kind, int default_kind, const double* qpos,
                  const double* qvel, const int32_t* lap, double* ctrl, int64_t ncars, cudaStream_t stream);
// the per-stream scratch of the grouping (step.cu keeps it with the step's, so captured ticks see it re-allocated):
// int32 hist[npolicies], cursor[npolicies], total[1], list[ncars]
int policy_scratch(int64_t ncars, int npolicies, cudaStream_t stream, int32_t** buf);

// ---- device geometry blob -------------------------------------------------
// One blob per ftgp_geom, replicated on a GPU and staged into shared memory by
// the lidar kernel.  All offsets are in 32-bit words from the start of the blob.
//
//   GeomHeader
//   per track: TrackHeader, index grid uint16[vc][hc] (row gy grows with +Y world,
//              gy = vc-1-j), chunk table uint32[nchunks][CHUNK_WORDS]
//   per track: centreline double[100][2] (8-byte aligned), or absent
//
// chunk record: words 0..12 = 400 vertex bits (bit r*ncol + c set = wall vertex,
// hfield row r = 0 at the -Y edge, i.e. the PNG chunk's bottom pixel row, SURVEY C.2),
// word 13 = ncol | nrow << 8; word 14 = bounding box of the wall vertices: cmin | cmax << 8 | rmin << 16 | rmax << 24
// words 15..27 = the same 400 vertex bits transposed (bit c * nrow + r), for rays that cross fewer columns than rows
// (cmin > cmax when the chunk has no wall vertex left, i.e. an all-wall chunk whose elevation normalises to 0)
constexpr int CHUNK_WORDS = 28;   // 13 mask words (row-major), dims, wall bounding box, 13 mask words (column-major)
constexpr uint16_t EMPTY_CHUNK = 0xFFFF;

struct TrackHeader {
    int32_t hc, vc, nchunks, chunk_px;
    float size_x, size_y;          // chunk pitch in metres (mushr.em.xml:19-20)
    float inv_size_x, inv_size_y;
    int32_t index_off, chunks_off; // word offsets from blob start
    int32_t path_off;              // word offset of double[100][2], or -1
    int32_t pad;
    double dsize_x, dsize_y;       // fp64 copies for the step kernel
    double dinv_size_x, dinv_size_y;   // 1 / dsize (the lidar's ray set-up divides by the chunk pitch for every ray)
};

struct GeomHeader {
    int32_t ntracks, total_words;
    int32_t track_off[FTGP_MAX_TRACKS];   // word offset of each TrackHeader
    int32_t lidar_words;                  // words the lidar kernel stages into shared memory
    int32_t pad;
};

}  // namespace ftgp

struct ftgp_track {
    int w, h, chunk_px, hc, vc;
    double scale, size_x, size_y;
    std::vector<int32_t> ij;          // 2*nchunks, chunk.py scan order
    std::vector<int32_t> counts;      // wall pixels per chunk
    std::vector<uint8_t> dims;        // 2*nchunks (ncol, nrow)
    std::vector<uint32_t> masks;      // nchunks * 13 words
};

namespace ftgp { void forget_geom(const struct ::ftgp_geom* geom); }   // drops captured tick graphs that reference the geometry

struct ftgp_geom {
    int device = 0;
    int ntracks = 0;
    uint32_t* d_blob = nullptr;
    std::vector<uint32_t> h_blob;
    int64_t bytes = 0;
    cudaStream_t host_stream = nullptr;   // for *_host variants
    // scratch for *_host variants (grown on demand)
    void* d_scratch = nullptr;
    size_t scratch_bytes = 0;
};
