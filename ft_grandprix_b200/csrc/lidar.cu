// lidar.cu -- the rangefinder kernel (SURVEY.md §8 a3).
//
// Replaces `data.sensordata[vehicle_state.sensors]` (ft_grandprix/custom.py:1395), i.e. the
// 90 `rangefinder` sensors per car of template/mushr.em.xml:112-117,204-206, which MuJoCo
// evaluates with mj_ray against the hfield walls (mushr.em.xml:92), the ground plane
// (mushr.em.xml:94) and, in multi-car worlds, the other cars' lidar cylinders
// (mushr.em.xml:108).  Semantics restated in SURVEY.md B.10.
//
// Design (B200):
//   * the whole compiled track (chunk index grid + 400-bit vertex masks, ~40-60 KB) is staged
//     once per CTA into shared memory by a persistent grid of 148 x k CTAs;
//   * one warp per car, lane l traces beams l, l+32, l+64 (< 90): within one round the 32
//     lanes hold 32 angularly adjacent beams (4 deg apart) and the 32 results are written as
//     one coalesced 128-byte store;
//   * two-level traversal: Amanatides-Woo DDA over the 0.5 m chunk grid (empty chunks cost
//     one shared-memory load), then a major-axis sweep over the 19x19 cells of a non-empty
//     chunk where only cells with at least one wall vertex (4 mask bits) are intersected;
//   * a cell is two height-field triangles split along (c,r)-(c+1,r+1) exactly as mj_rayHfield
//     does; the chunk's vertical side faces count as hits below the boundary elevation profile;
//   * pose math (quaternion -> ray origin/direction -> grid coordinates) is done in fp64, the
//     traversal in fp32 on cell-relative coordinates (error budget ~4e-6 m << 1e-4 m);
//   * a warp-level min-reduction yields the per-car closest obstacle (min_range).
#include <math.h>
#include <algorithm>
#include "common.h"
#include "mushr_mesh.h"

namespace ftgp {

__constant__ double c_beam_sc[FTGP_NBEAMS][2];   // (sin b, cos b), b = radians(4j - 90)
// the chassis mesh's own 33 triangles in the car frame (mushr.em.xml:38,119): what mj_ray tests on another car (SURVEY B.10)
__constant__ double c_chassis_tri[MUSHR_CHASSIS_NTRI][9];
__constant__ double c_chassis_box[6];            // bounding box of those triangles (lo[3], hi[3]), grown by 1e-9
static bool g_beam_ready[16] = {false};

constexpr float HF_RANGE = 0.3f;      // hfield elevation range: border_height + affordance (mushr.em.xml:16,22,55)
constexpr float HF_Z0 = -0.1f;        // hfield geom z (mushr.em.xml:92)
constexpr float PLANE_Z = 0.01f;      // ground plane (mushr.em.xml:94)
constexpr float PLANE_HALF = 300.0f;
constexpr float CELL_EPS = 1e-4f;     // inside-test tolerance in cell units (~2.6 um)
constexpr float BIG = 3.0e38f;

struct Ray {
    int ix0, iy0;        // chunk cell containing the origin (may be outside the grid)
    float fx0, fy0;      // fractional position inside that cell, [0,1)
    float dgx, dgy;      // chunk-grid units per metre of ray parameter
    float lz, dz;        // height above the hfield base plane (z + 0.1), vertical direction
};

__device__ __forceinline__ uint32_t mask_bits2(const uint32_t* m, int bit) {
    // two consecutive vertex bits starting at `bit` (may straddle a word)
    int w = bit >> 5, s = bit & 31;
    uint32_t lo = m[w], hi = m[min(w + 1, 12)];
    return __funnelshift_r(lo, hi, s) & 3u;
}
// n (<= 20) consecutive vertex bits starting at `bit`
__device__ __forceinline__ uint32_t mask_line(const uint32_t* m, int bit, int n) {
    int w = bit >> 5, sh = bit & 31;
    return __funnelshift_r(m[w], m[min(w + 1, 12)], sh) & ((1u << n) - 1u);
}
__device__ __forceinline__ uint32_t mask_bit(const uint32_t* m, int bit) {
    return (m[bit >> 5] >> (bit & 31)) & 1u;
}

// Intersect the ray (cell-local start (u,v), height z, per-metre increments du,dv,dz) with
// the two triangles of one cell.  bits: b0 = (c,r), b1 = (c+1,r), b2 = (c,r+1), b3 = (c+1,r+1).
// Returns the smallest parameter s >= smin at which it hits, or BIG.  `unsure` is set when an
// inside test landed within CELL_EPS of a triangle edge (or s within 1e-5 of smin): there the
// fp32 decision is not trustworthy (a ray grazing a ridge by microns) and the caller re-runs
// the cell in fp64 (cell_hit_exact).
__device__ __forceinline__ float cell_hit(uint32_t bits, float u, float v, float z,
                                          float du, float dv, float dz, float smin, bool& unsure) {
    float h00 = (bits & 1u) ? HF_RANGE : 0.f, h10 = (bits & 2u) ? HF_RANGE : 0.f;
    float h01 = (bits & 4u) ? HF_RANGE : 0.f, h11 = (bits & 8u) ? HF_RANGE : 0.f;
    float best = BIG;
    {   // triangle {(c,r), (c+1,r+1), (c+1,r)}: v <= u
        float a = h10 - h00, b = h11 - h10;
        float den = dz - a * du - b * dv;
        float num = z - h00 - a * u - b * v;
        if (fabsf(den) > 1e-15f) {
            float s = __fdividef(-num, den);        // (2 ulp; hits within CELL_EPS of an edge are re-done in fp64 anyway)
            float uu = u + s * du, vv = v + s * dv;
            float m = fminf(fminf(vv, uu - vv), 1.f - uu);          // > 0 inside
            if (s >= smin - 1e-5f && m >= -CELL_EPS) {
                if (m <= CELL_EPS || s < smin + 1e-5f) unsure = true; else best = s;
            }
        }
    }
    {   // triangle {(c,r), (c+1,r+1), (c,r+1)}: v >= u
        float a = h11 - h01, b = h01 - h00;
        float den = dz - a * du - b * dv;
        float num = z - h00 - a * u - b * v;
        if (fabsf(den) > 1e-15f) {
            float s = __fdividef(-num, den);        // (2 ulp; hits within CELL_EPS of an edge are re-done in fp64 anyway)
            float uu = u + s * du, vv = v + s * dv;
            float m = fminf(fminf(uu, vv - uu), 1.f - vv);
            if (s >= smin - 1e-5f && m >= -CELL_EPS) {
                if (m <= CELL_EPS || s < smin + 1e-5f) unsure = true; else if (s < best) best = s;
            }
        }
    }
    return best;
}

// fp64 re-evaluation of one cell for a grazing ray: the ray is rebuilt from the car pose exactly as
// the CPU restatement does, and the two triangles are tested without tolerance (hit point inside
// the closed triangle, s >= 0).  Returns the absolute ray parameter or BIG.  Rare path (~1e-4 of cells).
__device__ __noinline__ float cell_hit_exact(const TrackHeader* th, const double* __restrict__ pose7, int beam,
                                             int ix, int iy, int ncol, int nrow, int cc, int rr, uint32_t bits) {
    double q[7];
#pragma unroll
    for (int k = 0; k < 7; k++) q[k] = pose7[k];
    double n = sqrt(q[3] * q[3] + q[4] * q[4] + q[5] * q[5] + q[6] * q[6]);
    double w = q[3], x = q[4], y = q[5], z = q[6];
    if (n < 1e-15) { w = 1; x = y = z = 0; } else { w /= n; x /= n; y /= n; z /= n; }
    const double R0 = 1 - 2 * (y * y + z * z), R1 = 2 * (x * y - w * z), R2 = 2 * (x * z + w * y);
    const double R3 = 2 * (x * y + w * z), R4 = 1 - 2 * (x * x + z * z), R5 = 2 * (y * z - w * x);
    const double R6 = 2 * (x * z - w * y), R7 = 2 * (y * z + w * x), R8 = 1 - 2 * (x * x + y * y);
    const double sb = c_beam_sc[beam][0], cb = c_beam_sc[beam][1];
    const double rx = -0.0525, rz = 0.065, lr = 0.030;
    const double dx = sb * R0 - cb * R1, dy = sb * R3 - cb * R4, dz = sb * R6 - cb * R7;
    const double lx = rx - lr * sb, ly = lr * cb;
    const double ox = q[0] + R0 * lx + R1 * ly + R2 * rz, oy = q[1] + R3 * lx + R4 * ly + R5 * rz,
                 oz = q[2] + R6 * lx + R7 * ly + R8 * rz;
    // chunk (ix, iy) is centred at (size_x * ix, size_y * (iy - (vc-1))); cell pitch = size / (n - 1)
    const double cw = th->dsize_x / (ncol - 1), chh = th->dsize_y / (nrow - 1);
    const double u = (ox - th->dsize_x * ix + 0.5 * th->dsize_x) / cw - cc;
    const double v = (oy - th->dsize_y * (iy - (th->vc - 1)) + 0.5 * th->dsize_y) / chh - rr;
    const double du = dx / cw, dv = dy / chh, zz = oz + 0.1;      // hfield geom z = -0.1 (mushr.em.xml:92)
    const double H = 0.2 + 0.1;                                      // border_height + affordance (mushr.em.xml:55)
    const double h00 = (bits & 1u) ? H : 0., h10 = (bits & 2u) ? H : 0., h01 = (bits & 4u) ? H : 0., h11 = (bits & 8u) ? H : 0.;
    double best = 1e300;
    {
        double a = h10 - h00, b = h11 - h10, den = dz - a * du - b * dv, num = zz - h00 - a * u - b * v;
        if (fabs(den) > 1e-15) {
            double s = -num / den, uu = u + s * du, vv = v + s * dv;
            if (s >= 0 && vv >= 0 && vv <= uu && uu <= 1) best = s;
        }
    }
    {
        double a = h11 - h01, b = h01 - h00, den = dz - a * du - b * dv, num = zz - h00 - a * u - b * v;
        if (fabs(den) > 1e-15) {
            double s = -num / den, uu = u + s * du, vv = v + s * dv;
            if (s >= 0 && s < best && uu >= 0 && uu <= vv && vv <= 1) best = s;
        }
    }
    return best < 1e300 ? (float)best : BIG;
}

// Vertical side face of a chunk's top box, crossed at parameter t.  axis 0: face normal to x
// (profile runs along rows), axis 1: normal to y.  far_side: the +x / +y face.
__device__ __forceinline__ bool face_hit(const uint32_t* m, int ncol, int nrow, int axis, bool far_side,
                                         float along, float zt) {
    if (zt < 0.f || zt > 1.f) return false;
    int n = axis == 0 ? nrow : ncol;
    if (along < -CELL_EPS || along > (float)(n - 1) + CELL_EPS) return false;
    float y0 = fminf(fmaxf(floorf(along), 0.f), (float)(n - 2));
    int k = (int)y0;
    uint32_t z0, z1;
    if (axis == 0) {
        int col = far_side ? ncol - 1 : 0;
        z0 = mask_bit(m, k * ncol + col); z1 = mask_bit(m, (k + 1) * ncol + col);
    } else {
        int row = far_side ? nrow - 1 : 0;
        z0 = mask_bit(m, row * ncol + k); z1 = mask_bit(m, row * ncol + k + 1);
    }
    float prof = (float)z0 * (y0 + 1.f - along) + (float)z1 * (along - y0);
    return zt < prof;
}

// other car's lidar cylinder (mushr.em.xml:108): r = 0.03, half height 0.015, centred at
// (rx, 0, rz - lh/2) in that car's frame.  p/v: ray in the cylinder frame.  fp64: the target is 3 cm
// wide, so b^2 - a c cancels badly in fp32 for grazing rays (mju_rayGeom's cylinder branch restated).
__device__ __forceinline__ double ray_cylinder(double px, double py, double pz, double vx, double vy, double vz,
                                               double r, double hh) {
    double best = -1.0;
    const double a = vx * vx + vy * vy, b = px * vx + py * vy, c = px * px + py * py - r * r;
    if (a > 1e-15) {
        double det = b * b - a * c;
        if (det >= 1e-15) {
            det = sqrt(det);
            const double x0 = (-b - det) / a, x1 = (-b + det) / a;
            const double s = x0 >= 0 ? x0 : (x1 >= 0 ? x1 : -1.0);
            if (s >= 0 && fabs(pz + s * vz) <= hh) best = s;
        }
    }
    if (fabs(vz) > 1e-15) {
#pragma unroll
        for (int side = -1; side <= 1; side += 2) {
            const double s = ((double)side * hh - pz) / vz;
            if (s >= 0) {
                const double x = px + s * vx, y = py + s * vy;
                if (x * x + y * y <= r * r && (best < 0 || s < best)) best = s;
            }
        }
    }
    return best;
}

// other car's wheel ellipsoid (mushr.em.xml:69), ray in the geom frame: quadratic in the scaled space (mju_rayGeom)
__device__ __forceinline__ double ray_ellipsoid(double px, double py, double pz, double vx, double vy, double vz,
                                                double sx, double sy, double sz) {
    const double ix = 1.0 / (sx * sx), iy = 1.0 / (sy * sy), iz = 1.0 / (sz * sz);
    const double a = ix * vx * vx + iy * vy * vy + iz * vz * vz, b = ix * px * vx + iy * py * vy + iz * pz * vz,
                 c = ix * px * px + iy * py * py + iz * pz * pz - 1.0;
    if (a < 1e-15) return -1.0;
    double det = b * b - a * c;
    if (det < 1e-15) return -1.0;
    det = sqrt(det);
    const double x0 = (-b - det) / a, x1 = (-b + det) / a;
    return x0 >= 0 ? x0 : (x1 >= 0 ? x1 : -1.0);
}
// one triangle of the other car's chassis mesh (mj_rayMesh), ray in that car's frame
__device__ __forceinline__ double ray_triangle(const double* t, double px, double py, double pz, double vx, double vy, double vz) {
    const double e1x = t[3] - t[0], e1y = t[4] - t[1], e1z = t[5] - t[2], e2x = t[6] - t[0], e2y = t[7] - t[1], e2z = t[8] - t[2];
    const double hx = vy * e2z - vz * e2y, hy = vz * e2x - vx * e2z, hz = vx * e2y - vy * e2x;
    const double det = e1x * hx + e1y * hy + e1z * hz;
    if (fabs(det) < 1e-300) return -1.0;
    const double tx = px - t[0], ty = py - t[1], tz = pz - t[2];
    const double u = (tx * hx + ty * hy + tz * hz) / det;
    if (u < 0 || u > 1) return -1.0;
    const double qx = ty * e1z - tz * e1y, qy = tz * e1x - tx * e1z, qz = tx * e1y - ty * e1x;
    const double v = (vx * qx + vy * qy + vz * qz) / det;
    if (v < 0 || u + v > 1) return -1.0;
    const double x = (e2x * qx + e2y * qy + e2z * qz) / det;
    return x >= 0 ? x : -1.0;
}
// Nearest lidar-visible geom of ANOTHER car along the ray (p, v given in that car's frame): lidar cylinder, chassis mesh
// triangles, four wheel ellipsoids (their pose follows the suspension slide and, at the front, the steering hinge; the
// ellipsoid is a body of revolution about the axle, so the throttle angle drops out).  jq: susp[4], steer[2].
// Everything of the car lies inside the sphere |x - (0, 0, 0.02)| < 0.145, which culls almost every (ray, car) pair.
// The rare parts live in functions of their own: inlined, the 33 triangles, four ellipsoids and a sincos made the set-up
// block 27 KB of code that evicted the traversal loop from the 32 KB instruction cache every round (ncu: stall_no_instruction
// 3.0 cycles per issued instruction against 0.26 in the single-car kernel, 2.3 ms against 1.1 ms for the same rays).
__device__ __noinline__ double ray_chassis_mesh(double px, double py, double pz, double vx, double vy, double vz) {
    // only if the ray crosses the triangles' bounding box (slab test)
    double t0 = 0.0, t1 = 1e300;
    const double p[3] = {px, py, pz}, v[3] = {vx, vy, vz};
#pragma unroll
    for (int a = 0; a < 3; a++) {
        if (fabs(v[a]) > 1e-30) {
            const double i = 1.0 / v[a], ta = (c_chassis_box[a] - p[a]) * i, tb = (c_chassis_box[3 + a] - p[a]) * i;
            t0 = fmax(t0, fmin(ta, tb)); t1 = fmin(t1, fmax(ta, tb));
        } else if (p[a] < c_chassis_box[a] || p[a] > c_chassis_box[3 + a]) t1 = -1.0;
    }
    double best = -1.0;
    if (t0 <= t1 * (1 + 1e-12) + 1e-12)
#pragma unroll 1
        for (int f = 0; f < MUSHR_CHASSIS_NTRI; f++) {
            const double x = ray_triangle(c_chassis_tri[f], px, py, pz, vx, vy, vz);
            if (x >= 0 && (best < 0 || x < best)) best = x;
        }
    return best;
}
__device__ __noinline__ double ray_wheels(double px, double py, double pz, double vx, double vy, double vz, const double* jq) {
    double best = -1.0;
#pragma unroll 1
    for (int w = 0; w < 4; w++) {
        const double cx = w < 2 ? 0.06925 : -0.079, cy = (w & 1) ? -0.0575 : 0.0575, cz = 0.0244 + jq[w];
        const double qx = px - cx, qy = py - cy, qz = pz - cz;
        {   // the ellipsoid (0.03, 0.01, 0.03) lies inside the sphere of radius 0.03 about its centre
            const double b = qx * vx + qy * vy + qz * vz, c = qx * qx + qy * qy + qz * qz - 0.03 * 0.03 * (1 + 1e-9);
            if (c > 0 && (b > 0 || b * b - c < 0)) continue;
        }
        double sn = 0.0, cs = 1.0;
        if (w < 2) sincos(jq[4 + w], &sn, &cs);
        const double x = ray_ellipsoid(cs * qx + sn * qy, -sn * qx + cs * qy, qz, cs * vx + sn * vy, -sn * vx + cs * vy, vz, 0.03, 0.01, 0.03);
        if (x >= 0 && (best < 0 || x < best)) best = x;
    }
    return best;
}
__device__ __noinline__ double ray_other_car(double px, double py, double pz, double vx, double vy, double vz, const double* jq) {
    const double b = px * vx + py * vy + (pz - 0.02) * vz;
    {
        const double cz = pz - 0.02, c = px * px + py * py + cz * cz - 0.145 * 0.145;
        if (c > 0 && (b > 0 || b * b - c < 0)) return -1.0;
    }
    double best = -1.0;
    {   // lidar cylinder, behind its own bounding sphere
        const double qx = px + 0.0525, qz = pz - (0.065 - 0.015 / 2);
        const double bb = qx * vx + py * vy + qz * vz, cc = qx * qx + py * py + qz * qz - (0.03 * 0.03 + 0.015 * 0.015) * (1 + 1e-9);
        if (!(cc > 0 && (bb > 0 || bb * bb - cc < 0))) best = ray_cylinder(qx, py, qz, vx, vy, vz, 0.03, 0.015);
    }
    // Inside the bounding sphere the ray stays within 0.145 |vz| of the height of its closest approach to the sphere's centre.
    // On level ground the beams pass 2 cm above every chassis and wheel: that interval misses both height ranges and the
    // mesh / wheel tests are not even called.
    const double zc = pz - b * vz, dz = 0.145 * fabs(vz), zlo = zc - dz - 1e-9, zhi = zc + dz + 1e-9;
    if (!(zlo > c_chassis_box[5] || zhi < c_chassis_box[2])) {
        const double x = ray_chassis_mesh(px, py, pz, vx, vy, vz);
        if (x >= 0 && (best < 0 || x < best)) best = x;
    }
    const double jmax = fmax(fmax(jq[0], jq[1]), fmax(jq[2], jq[3])), jmin = fmin(fmin(jq[0], jq[1]), fmin(jq[2], jq[3]));
    if (!(zlo > 0.0244 + 0.03 + jmax || zhi < 0.0244 - 0.03 + jmin)) {
        const double x = ray_wheels(px, py, pz, vx, vy, vz, jq);
        if (x >= 0 && (best < 0 || x < best)) best = x;
    }
    return best;
}

// ---------------------------------------------------------------------------------------------------
// Traversal as a per-lane state machine.  A warp owns a batch of cars (whole worlds) and a pool of
// 90 x ncars rays; every lane runs IDLE -> CHUNK (one Amanatides-Woo step over the 0.5 m chunk grid)
// -> SWEEP (one major-axis column of 19x19 cells inside a non-empty chunk) -> ... -> IDLE, and an idle
// lane pulls the next ray of the pool.  Each loop iteration executes ONE of two code blocks for the whole warp --
// "leave the previous chunk and walk to the next non-empty one" or "sweep the lines of the current chunk" -- the one
// most lanes are waiting for (a warp-uniform vote), so that lanes in the same state are served together and the
// other block's instructions are not issued at all for a handful of lanes
// (the first version traced beams l, l+32, l+64 per lane with nested loops: 6.5 of 32 lanes active).
enum { ST_IDLE = 0, ST_CHUNK = 1, ST_SWEEP = 2, ST_ADV = 3 };
// scheduling knobs of the state machine (tools/build_variant.py experiments; the defaults are what ships)
#ifndef FTGP_AB_HYST_A
#define FTGP_AB_HYST_A 0            // > 0: keep sweeping while at least A lanes sweep ...
#endif
#ifndef FTGP_AB_HYST_B
#define FTGP_AB_HYST_B 0            // ... and keep walking while at least B lanes walk (0/0: plain majority vote)
#endif
#ifndef FTGP_AB_WALK_MAX
#define FTGP_AB_WALK_MAX 5          // at most this many empty chunks per round (0: unbounded; measured 1.30 -> 1.14 ms at 65,536 cars)
#endif
#ifndef FTGP_AB_VOTE_BIAS
#define FTGP_AB_VOTE_BIAS 0         // the walk block runs when n_walk + bias >= n_sweep (and somebody walks)
#endif
#ifndef FTGP_AB_WALK_VOTE
#define FTGP_AB_WALK_VOTE 0         // K > 0: the walk goes on while at least K/4 of the lanes that started it are still walking
#endif
#ifndef FTGP_AB_LINE_MAX
#define FTGP_AB_LINE_MAX 0          // > 0: at most this many candidate-free lines per round
#endif
#ifndef FTGP_AB_REFILL
#define FTGP_AB_REFILL 8            // idle lanes that trigger a refill
#endif
#ifndef FTGP_AB_LANESTATS
#define FTGP_AB_LANESTATS 0         // 1: count rounds and active lanes per block into g_lane_stats (ftgp_lidar_lanestats)
#endif
#if FTGP_AB_LANESTATS
// per block: rounds, lanes that entered; per inner loop: iterations, active lanes summed over them
enum { LS_SETUP_ROUNDS, LS_SETUP_LANES, LS_WALK_ROUNDS, LS_WALK_LANES, LS_SWEEP_ROUNDS, LS_SWEEP_LANES, LS_HOP_ITERS,
       LS_HOP_LANES, LS_LINE_ITERS, LS_LINE_LANES, LS_CELL_ITERS, LS_CELL_LANES, LS_N };
__device__ unsigned long long g_lane_stats[LS_N];
static int64_t g_lane_launch[4];      // shared memory, CTAs per SM, track staged, cars per batch of the last launch
#define LANESTAT_ROUND(k, n) do { if (lane == 0) { ls[k]++; ls[(k) + 1] += (n); } } while (0)
#define LANESTAT_LOOP(k) do { const unsigned am_ = __activemask(); if (lane == __ffs(am_) - 1) { ls[k]++; ls[(k) + 1] += __popc(am_); } } while (0)
#else
#define LANESTAT_ROUND(k, n) do { } while (0)
#define LANESTAT_LOOP(k) do { } while (0)
#endif
constexpr int BATCH = 8;              // max cars per warp batch (a batch holds whole worlds of 1..8 cars)
constexpr int MULTI_WORDS = BATCH * FTGP_NBEAMS + 64 + 66;   // per warp, multi-car worlds: nearest other-car hit per ray, beam window and running count per (car, other car)
constexpr int FRAME_DOUBLES = 21;     // p[3], R[9], suspension travel [4], front steering angle [2], centre of the car's bounding sphere [3]

struct Lane {
    // ray
    int ix0, iy0; float fx0, fy0, dgx, dgy, lz, dz;
    float inv_dgx, inv_dgy; int stepx, stepy;
    float tz0, tend, best;
    // chunk DDA
    int ix, iy; float t0; int entry_axis;
    // current chunk
    const uint32_t* m; int ncol, nrow; float fxo, dfx, fyo, dfy, t1; int exit_axis; bool nonempty;
    // sweep
    float ta, span, xa, ya, za, dM, dm, Ma, ma, inv_dM; int nM, nm, sg, c, cend; bool floor_reach, major_x;
    // bookkeeping
    int rid, state;
    const TrackHeader* th;
};

__device__ __forceinline__ void finish(Lane& L, float val, float* __restrict__ ranges, float* __restrict__ min_range,
                                       int64_t base_car) {
    const int car = L.rid / FTGP_NBEAMS, beam = L.rid - car * FTGP_NBEAMS;
    ranges[(base_car + car) * FTGP_NBEAMS + beam] = val;
    if (min_range && val >= 0.f) atomicMin(reinterpret_cast<unsigned int*>(min_range + base_car + car), __float_as_uint(val));
    L.state = ST_IDLE;
}

// MULTI: worlds of 2..8 cars (the other cars' geoms are ray targets); single-car worlds compile without that code
template <bool MULTI>
__global__ void __launch_bounds__(512)
lidar_kernel(const uint32_t* __restrict__ blob, int lidar_words, const double* __restrict__ qpos,
             int64_t stride, const int32_t* __restrict__ track_id, const uint8_t* __restrict__ visible,
             const int32_t* __restrict__ lap, int64_t ncars, int cpw, int bsz, int stage, float* __restrict__ ranges,
             float* __restrict__ min_range) {
    extern __shared__ __align__(16) uint32_t sm[];
    // the compiled tracks are staged into shared memory when they fit (one or two tracks); otherwise they are
    // read through L1/L2 from the global blob
    if (stage) {
        const uint4* src = reinterpret_cast<const uint4*>(blob);
        uint4* dst = reinterpret_cast<uint4*>(sm);
        int n4 = (lidar_words + 3) >> 2;
        for (int i = threadIdx.x; i < n4; i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    const uint32_t* geo = stage ? sm : blob;
    uint32_t* scratch = stage ? sm + ((lidar_words + 3) & ~3) : sm;
    const GeomHeader* gh = reinterpret_cast<const GeomHeader*>(geo);
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int warps_per_block = blockDim.x >> 5;
    double* frames = reinterpret_cast<double*>(scratch) + (size_t)wib * BATCH * FRAME_DOUBLES;
    int* meta = reinterpret_cast<int*>(reinterpret_cast<double*>(scratch) +
                                       (size_t)warps_per_block * BATCH * FRAME_DOUBLES) + wib * BATCH;
    // multi-car worlds: the other cars' hits are found in a pass of their own before the traversal (below)
    uint32_t* obest = reinterpret_cast<uint32_t*>(reinterpret_cast<int*>(reinterpret_cast<double*>(scratch) +
                                                  (size_t)warps_per_block * BATCH * FRAME_DOUBLES) + warps_per_block * BATCH) +
                      (size_t)wib * MULTI_WORDS;
    uint32_t* prange = obest + BATCH * FTGP_NBEAMS;
    int* ppre = reinterpret_cast<int*>(prange + 64);
    const int64_t nwarps = (int64_t)gridDim.x * warps_per_block;
    const int64_t nbatch = (ncars + bsz - 1) / bsz;
    const double rx = -0.0525, rz = 0.065, lr = 0.030;   // mushr.em.xml:101-103
    const unsigned lt = (1u << lane) - 1u;
#if FTGP_AB_LANESTATS
    unsigned ls[LS_N] = {};
#endif

    for (int64_t batch = (int64_t)blockIdx.x * warps_per_block + wib; batch < nbatch; batch += nwarps) {
        const int64_t base_car = batch * bsz;
        const int nb = (int)min((int64_t)bsz, ncars - base_car);
        __syncwarp();
        if (lane < nb) {            // pose frame of each car of the batch: position + rotation matrix, fp64
            const double* q = qpos + (base_car + lane) * stride;
            double w = q[3], x = q[4], y = q[5], z = q[6];
            const double n = sqrt(w * w + x * x + y * y + z * z);
            if (n < 1e-15) { w = 1; x = y = z = 0; } else { w /= n; x /= n; y /= n; z /= n; }
            double* F = frames + lane * FRAME_DOUBLES;
            F[0] = q[0]; F[1] = q[1]; F[2] = q[2];
            F[3] = 1 - 2 * (y * y + z * z); F[4] = 2 * (x * y - w * z); F[5] = 2 * (x * z + w * y);
            F[6] = 2 * (x * y + w * z); F[7] = 1 - 2 * (x * x + z * z); F[8] = 2 * (y * z - w * x);
            F[9] = 2 * (x * z - w * y); F[10] = 2 * (y * z + w * x); F[11] = 1 - 2 * (x * x + y * y);
            // wheel poses for the other cars' rays (full state rows only; a bare pose leaves the joints at qpos0)
            if (MULTI) {
                const bool full = stride >= FTGP_NQ;
                F[12] = full ? q[8] : 0.0; F[13] = full ? q[15] : 0.0; F[14] = full ? q[22] : 0.0; F[15] = full ? q[28] : 0.0;
                F[16] = full ? q[9] : 0.0; F[17] = full ? q[16] : 0.0;
                F[18] = F[0] + 0.02 * F[5]; F[19] = F[1] + 0.02 * F[8]; F[20] = F[2] + 0.02 * F[11];      // car-frame (0, 0, 0.02)
            }
            int tid = track_id ? track_id[base_car + lane] : 0;
            if (tid < 0 || tid >= gh->ntracks) tid = 0;
            // bit 8: other cars do not see this car (shadowed, custom.py:1455-1464); bit 9: its own rangefinders are
            // switched off (mjSENS_USER after shadow(), custom.py:1438): the ranges row keeps its stale values
            int flags = tid;
            if (visible && !visible[base_car + lane]) flags |= 0x100;
            if (lap && lap[(base_car + lane) * FTGP_LAP_FIELDS + FTGP_LAP_FINISHED]) flags |= 0x300;
            meta[lane] = flags;
            if (min_range) min_range[base_car + lane] = INFINITY;
        }
        __syncwarp();
        const int nrays = nb * FTGP_NBEAMS;
        if (MULTI) {
            // ---------------- [block: other cars of the world, one pass per batch]
            // The other cars' lidar cylinder, chassis mesh and wheels (mushr.em.xml:108,119,69) as ray targets.  Tested inside the
            // ray set-up, the exact test ran for one or two lanes at a time (a third of the kernel's instructions at 1.5 active
            // lanes).  Here: per ordered pair (car A, other car) the window of A's beams that can reach the other car's bounding
            // sphere, then the (A, other, beam) triples of all windows dealt out to the 32 lanes.
            for (int i = lane; i < nrays; i += 32) obest[i] = __float_as_uint(BIG);
            for (int pidx = lane; pidx < 64; pidx += 32) {
                uint32_t win = 0;                                        // beam window: first beam | count << 8
                const int A = pidx / cpw, oc = (A / cpw) * cpw + pidx % cpw;
                if (pidx < nb * cpw && oc < nb && oc != A && !(meta[oc] & 0x100) && !(meta[A] & 0x200)) {
                    const double* F = frames + A * FRAME_DOUBLES; const double* Q = frames + oc * FRAME_DOUBLES;
                    // e = centre of the other car's sphere - A's lidar axis point (rx, 0, rz), in A's frame.  A beam starts within
                    // 0.03 m of that point, so it reaches the sphere (r = 0.145) only if its direction passes within 0.175 m.
                    const double wx = Q[18] - (F[0] + F[3] * rx + F[5] * rz), wy = Q[19] - (F[1] + F[6] * rx + F[8] * rz),
                                 wz = Q[20] - (F[2] + F[9] * rx + F[11] * rz);
                    const float ex = (float)(F[3] * wx + F[6] * wy + F[9] * wz), ey = (float)(F[4] * wx + F[7] * wy + F[10] * wz),
                                ez = (float)(F[5] * wx + F[8] * wy + F[11] * wz);
                    const float RR = 0.175f, e2 = ex * ex + ey * ey + ez * ez, rho = sqrtf(ex * ex + ey * ey);
                    if (e2 <= RR * RR * 1.01f) win = 0u | (90u << 8);
                    else {
                        const float kappa = sqrtf(e2 - RR * RR) / fmaxf(rho, 1e-20f);
                        if (kappa < 1.f) {
                            // beam j points along azimuth 4 j - 180 degrees in A's frame (site +Z = (sin b, -cos b, 0), b = 4 j - 90)
                            const float phi = atan2f(ey, ex) * 57.29578f, half = acosf(kappa) * 57.29578f + 4.5f;   // one beam of margin
                            const float jc = (phi + 180.f) * 0.25f, hw = half * 0.25f;
                            int jlo = (int)floorf(jc - hw), cnt = (int)ceilf(jc + hw) - jlo + 1;
                            if (cnt >= 90) win = 90u << 8;
                            else win = (uint32_t)(((jlo % 90) + 90) % 90) | ((uint32_t)cnt << 8);
                        }
                    }
                }
                prange[pidx] = win;
            }
            __syncwarp();
            int total = 0;                                               // running count over the 64 windows (every lane, redundantly)
            for (int pidx = 0; pidx < nb * cpw; pidx++) { if (lane == 0) ppre[pidx] = total; total += (int)(prange[pidx] >> 8); }
            if (lane == 0) ppre[nb * cpw] = total;
            __syncwarp();
            for (int t = lane; t < total; t += 32) {
                int lo = 0, hi = nb * cpw;                                // the window that holds triple t
                while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (ppre[mid] <= t) lo = mid; else hi = mid; }
                const uint32_t win = prange[lo];
                const int A = lo / cpw, oc = (A / cpw) * cpw + lo % cpw;
                int j = (int)(win & 0xFF) + (t - ppre[lo]); if (j >= FTGP_NBEAMS) j -= FTGP_NBEAMS;
                const double* F = frames + A * FRAME_DOUBLES; const double* Q = frames + oc * FRAME_DOUBLES;
                const double sb = c_beam_sc[j][0], cb = c_beam_sc[j][1];
                const double dwx = sb * F[3] - cb * F[4], dwy = sb * F[6] - cb * F[7], dwz = sb * F[9] - cb * F[10];
                const double lx = rx - lr * sb, ly = lr * cb;
                const double owx = F[0] + F[3] * lx + F[4] * ly + F[5] * rz;
                const double owy = F[1] + F[6] * lx + F[7] * ly + F[8] * rz;
                const double owz = F[2] + F[9] * lx + F[10] * ly + F[11] * rz;
                const double ex = owx - Q[0], ey = owy - Q[1], ez = owz - Q[2];
                const double sc = ray_other_car(Q[3] * ex + Q[6] * ey + Q[9] * ez, Q[4] * ex + Q[7] * ey + Q[10] * ez,
                                                Q[5] * ex + Q[8] * ey + Q[11] * ez, Q[3] * dwx + Q[6] * dwy + Q[9] * dwz,
                                                Q[4] * dwx + Q[7] * dwy + Q[10] * dwz, Q[5] * dwx + Q[8] * dwy + Q[11] * dwz, Q + 12);
                if (sc >= 0) atomicMin(&obest[A * FTGP_NBEAMS + j], __float_as_uint((float)sc));
            }
            __syncwarp();
        }
        int next = 0;
        Lane L;
        L.state = ST_IDLE;
        int mode = ST_CHUNK;
        for (;;) {
            const unsigned idle = __ballot_sync(0xffffffffu, L.state == ST_IDLE);
            const bool refill = next < nrays && (__popc(idle) >= FTGP_AB_REFILL || idle == 0xffffffffu);
            if (!refill && idle == 0xffffffffu) break;
            if (refill) {
                const int r = next + __popc(idle & lt);
                LANESTAT_ROUND(LS_SETUP_ROUNDS, min(__popc(idle), nrays - next));
                next += __popc(idle);
                if (L.state == ST_IDLE && r < nrays) {
                    // ---------------- ray set-up (fp64 pose math, then fp32 cell-relative coordinates)
                    const int car = r / FTGP_NBEAMS, j = r - car * FTGP_NBEAMS;
                    const int flags = meta[car];
                    if (!(flags & 0x200)) {
                        L.rid = r;
                        const double* F = frames + car * FRAME_DOUBLES;
                        const TrackHeader* th = reinterpret_cast<const TrackHeader*>(geo + gh->track_off[flags & 0xFF]);
                        L.th = th;
                        const double sb = c_beam_sc[j][0], cb = c_beam_sc[j][1];
                        // site +Z axis in the car frame = (sin b, -cos b, 0); origin = lidar axis - lr * dir
                        const double dwx = sb * F[3] - cb * F[4], dwy = sb * F[6] - cb * F[7], dwz = sb * F[9] - cb * F[10];
                        const double lx = rx - lr * sb, ly = lr * cb;
                        const double owx = F[0] + F[3] * lx + F[4] * ly + F[5] * rz;
                        const double owy = F[1] + F[6] * lx + F[7] * ly + F[8] * rz;
                        const double owz = F[2] + F[9] * lx + F[10] * ly + F[11] * rz;
                        const double inv_sx = th->dinv_size_x, inv_sy = th->dinv_size_y;
                        const double gxd = owx * inv_sx + 0.5, gyd = owy * inv_sy + 0.5 + (double)(th->vc - 1);
                        const double fgx = floor(gxd), fgy = floor(gyd);
                        L.ix0 = (int)fgx; L.iy0 = (int)fgy;
                        L.fx0 = (float)(gxd - fgx); L.fy0 = (float)(gyd - fgy);
                        L.dgx = (float)(dwx * inv_sx); L.dgy = (float)(dwy * inv_sy);
                        L.lz = (float)(owz + 0.1); L.dz = (float)dwz;
                        float best = BIG;
                        if (MULTI) best = __uint_as_float(obest[r]);      // nearest hit on another car of the world (pass above)
                        // ground plane: hit only from the front side, inside the 300 m rendered square
                        if (L.dz < -1e-15f) {
                            float tp = -(L.lz + HF_Z0 - PLANE_Z) / L.dz;
                            if (tp >= 0.f) {
                                float ppx = ((float)L.ix0 + L.fx0 - 0.5f + tp * L.dgx) * th->size_x;
                                float ppy = ((float)(L.iy0 - (th->vc - 1)) + L.fy0 - 0.5f + tp * L.dgy) * th->size_y;
                                if (fabsf(ppx) <= PLANE_HALF && fabsf(ppy) <= PLANE_HALF) best = fminf(best, tp);
                            }
                        }
                        L.best = best;
                        // parameter interval in which the ray is inside the walls' height slab [0, 0.3]
                        float tz0 = 0.f, tz1 = BIG;
                        if (fabsf(L.dz) > 1e-15f) {
                            float a = (0.f - L.lz) / L.dz, b2 = (HF_RANGE - L.lz) / L.dz;
                            tz0 = fmaxf(0.f, fminf(a, b2)); tz1 = fmaxf(a, b2);
                        } else if (L.lz < 0.f || L.lz > HF_RANGE) tz1 = -1.f;
                        const float tend = fminf(tz1, best);
                        L.tz0 = tz0; L.tend = tend;
                        bool go = tend >= tz0;
                        // clip against the chunk grid [0,hc] x [0,vc]
                        const int hc = th->hc, vc = th->vc;
                        const float gx = (float)L.ix0 + L.fx0, gy = (float)L.iy0 + L.fy0;
                        float tg0 = 0.f, tg1 = tend;
                        int enter_axis = -1;
                        L.inv_dgx = fabsf(L.dgx) > 1e-20f ? 1.f / L.dgx : 0.f;
                        L.inv_dgy = fabsf(L.dgy) > 1e-20f ? 1.f / L.dgy : 0.f;
                        if (L.inv_dgx != 0.f) {
                            float a = (0.f - gx) * L.inv_dgx, b2 = ((float)hc - gx) * L.inv_dgx;
                            float lo = fminf(a, b2), hi = fmaxf(a, b2);
                            if (lo > tg0) { tg0 = lo; enter_axis = 0; }
                            tg1 = fminf(tg1, hi);
                        } else if (gx < 0.f || gx >= (float)hc) tg1 = -1.f;
                        if (L.inv_dgy != 0.f) {
                            float a = (0.f - gy) * L.inv_dgy, b2 = ((float)vc - gy) * L.inv_dgy;
                            float lo = fminf(a, b2), hi = fmaxf(a, b2);
                            if (lo > tg0) { tg0 = lo; enter_axis = 1; }
                            tg1 = fminf(tg1, hi);
                        } else if (gy < 0.f || gy >= (float)vc) tg1 = -1.f;
                        if (tg1 < tg0) go = false;
                        float ts = tg0;
                        if (tz0 > ts) { ts = tz0; enter_axis = -1; }   // dropping into the slab from above: no side face
                        if (ts > tend) go = false;
                        if (!go) finish(L, best < BIG ? best : -1.f, ranges, min_range, base_car);
                        else {
                            L.stepx = L.dgx >= 0.f ? 1 : -1; L.stepy = L.dgy >= 0.f ? 1 : -1;
                            // chunk containing the start point (relative to the origin cell to keep fp32 exact)
                            const float relx = L.fx0 + ts * L.dgx, rely = L.fy0 + ts * L.dgy;
                            int ix = L.ix0 + (int)floorf(relx), iy = L.iy0 + (int)floorf(rely);
                            if (enter_axis == 0) ix = L.stepx > 0 ? 0 : hc - 1;
                            if (enter_axis == 1) iy = L.stepy > 0 ? 0 : vc - 1;
                            L.ix = min(max(ix, 0), hc - 1); L.iy = min(max(iy, 0), vc - 1);
                            L.t0 = ts; L.entry_axis = enter_axis;
                            L.state = ST_CHUNK;
                        }
                    }
                }
            }
            // ---------------- which block runs this round: the state with the most lanes
            const int n_chunk = __popc(__ballot_sync(0xffffffffu, L.state == ST_CHUNK || L.state == ST_ADV));
            const int n_sweep = __popc(__ballot_sync(0xffffffffu, L.state == ST_SWEEP));
            int pick = (n_chunk + FTGP_AB_VOTE_BIAS >= n_sweep && (n_chunk > 0 || n_sweep == 0)) ? ST_CHUNK : ST_SWEEP;
            if (FTGP_AB_VOTE_BIAS < 0 && n_sweep == 0) pick = ST_CHUNK;
            if (FTGP_AB_HYST_A > 0) {
                if (mode == ST_SWEEP) pick = (n_sweep >= FTGP_AB_HYST_A || n_chunk == 0) ? ST_SWEEP : ST_CHUNK;
                else pick = (n_chunk >= FTGP_AB_HYST_B && n_chunk > 0) || n_sweep == 0 ? ST_CHUNK : ST_SWEEP;
                mode = pick;
            }
            if (pick == ST_CHUNK) LANESTAT_ROUND(LS_WALK_ROUNDS, n_chunk); else LANESTAT_ROUND(LS_SWEEP_ROUNDS, n_sweep);
            // ---------------- leave the previous chunk (exit side face, step of the chunk DDA) ...
            if (pick == ST_CHUNK && L.state == ST_ADV) {
                bool done = false;
                if (L.t1 <= L.tend) {                                // exit side face
                    const bool far_side = L.exit_axis == 0 ? L.stepx > 0 : L.stepy > 0;
                    const float along = L.exit_axis == 0 ? L.fyo + L.t1 * L.dfy : L.fxo + L.t1 * L.dfx;
                    if (face_hit(L.m, L.ncol, L.nrow, L.exit_axis, far_side, along, (L.lz + L.t1 * L.dz) * (1.f / HF_RANGE))) {
                        finish(L, fminf(L.best, L.t1), ranges, min_range, base_car); done = true;
                    }
                }
                if (!done) {
                    if (L.t1 >= L.tend) finish(L, L.best < BIG ? L.best : -1.f, ranges, min_range, base_car);
                    else {
                        if (L.exit_axis == 0) L.ix += L.stepx; else L.iy += L.stepy;
                        if (L.ix < 0 || L.ix >= L.th->hc || L.iy < 0 || L.iy >= L.th->vc)
                            finish(L, L.best < BIG ? L.best : -1.f, ranges, min_range, base_car);
                        else { L.t0 = L.t1; L.entry_axis = L.exit_axis; L.state = ST_CHUNK; }
                    }
                }
            }
            // ---------------- ... and on over the chunk grid to the next non-empty chunk (empty chunks: one shared-memory load each)
            if (pick == ST_CHUNK && L.state == ST_CHUNK) {
                const TrackHeader* th = L.th;
                const int hc = th->hc, vc = th->vc;
                const uint16_t* index = reinterpret_cast<const uint16_t*>(geo + th->index_off);
                uint32_t cid;
                bool more = false;
                const int entered = FTGP_AB_WALK_VOTE > 0 ? __popc(__activemask()) : 0;
                for (int hop = 0;; hop++) {
                    LANESTAT_LOOP(LS_HOP_ITERS);
                    if (FTGP_AB_WALK_MAX > 0 && hop == FTGP_AB_WALK_MAX) { more = true; break; }
                    if (FTGP_AB_WALK_VOTE > 0 && hop > 0 && __popc(__activemask()) * 4 < entered * FTGP_AB_WALK_VOTE) { more = true; break; }
                    const float tmx = L.inv_dgx != 0.f ? ((float)(L.ix - L.ix0 + (L.stepx > 0 ? 1 : 0)) - L.fx0) * L.inv_dgx : BIG;
                    const float tmy = L.inv_dgy != 0.f ? ((float)(L.iy - L.iy0 + (L.stepy > 0 ? 1 : 0)) - L.fy0) * L.inv_dgy : BIG;
                    L.exit_axis = tmx <= tmy ? 0 : 1;
                    L.t1 = fminf(tmx, tmy);
                    cid = index[L.iy * hc + L.ix];
                    if (cid != EMPTY_CHUNK) break;
                    // empty chunk: nothing to hit, leave it at once
                    if (L.t1 >= L.tend) { finish(L, L.best < BIG ? L.best : -1.f, ranges, min_range, base_car); break; }
                    if (L.exit_axis == 0) L.ix += L.stepx; else L.iy += L.stepy;
                    if (L.ix < 0 || L.ix >= hc || L.iy < 0 || L.iy >= vc) { finish(L, L.best < BIG ? L.best : -1.f, ranges, min_range, base_car); break; }
                    L.t0 = L.t1; L.entry_axis = L.exit_axis;
                }
                L.nonempty = L.state == ST_CHUNK && !more;
                if (L.nonempty) L.state = ST_ADV;           // unless the sweep below takes over (or a face ends the ray)
                if (L.nonempty) {
                    const uint32_t* m = geo + th->chunks_off + cid * CHUNK_WORDS;
                    L.m = m;
                    L.ncol = m[13] & 0xFF; L.nrow = (m[13] >> 8) & 0xFF;
                    const float nx = (float)(L.ncol - 1), ny = (float)(L.nrow - 1);
                    // fine-cell coordinates inside this chunk: f(t) = fo + t * df
                    L.fxo = ((float)(L.ix0 - L.ix) + L.fx0) * nx; L.dfx = L.dgx * nx;
                    L.fyo = ((float)(L.iy0 - L.iy) + L.fy0) * ny; L.dfy = L.dgy * ny;
                    const float inv_h = 1.f / HF_RANGE;
                    bool done = false;
                    if (L.entry_axis >= 0 && L.t0 <= L.tend) {       // entry side face
                        const bool far_side = L.entry_axis == 0 ? L.stepx < 0 : L.stepy < 0;
                        const float along = L.entry_axis == 0 ? L.fyo + L.t0 * L.dfy : L.fxo + L.t0 * L.dfx;
                        if (face_hit(m, L.ncol, L.nrow, L.entry_axis, far_side, along, (L.lz + L.t0 * L.dz) * inv_h)) {
                            finish(L, fminf(L.best, L.t0), ranges, min_range, base_car); done = true;
                        }
                    }
                    if (!done) {
                        float ta = fmaxf(L.t0, L.tz0), tb = fminf(L.t1, L.tend);
                        if (ta <= tb) {
                            const float za0 = L.lz + ta * L.dz;
                            // (a ray that ENDS on the base plane -- it started below the ground plane, so nothing stops it before
                            // z = -0.1 -- reaches height 0 only up to fp32 rounding: without the margin the flat floor cells were
                            // sometimes not candidates and the ray was reported as a miss where mj_rayHfield hits the floor)
                            L.floor_reach = fminf(za0, za0 + (tb - ta) * L.dz) <= 1e-5f;
                            if (!L.floor_reach) {
                                // only cells with a wall vertex can be hit: clip to the chunk's wall bounding box (+1 cell)
                                const uint32_t bb = m[14];
                                const float xlo = (float)(bb & 0xFF) - 1.01f, xhi = (float)((bb >> 8) & 0xFF) + 1.01f;
                                const float ylo = (float)((bb >> 16) & 0xFF) - 1.01f, yhi = (float)(bb >> 24) + 1.01f;
                                if (fabsf(L.dfx) > 1e-20f) {
                                    const float i = __fdividef(1.f, L.dfx), a = (xlo - L.fxo) * i, b2 = (xhi - L.fxo) * i;
                                    ta = fmaxf(ta, fminf(a, b2)); tb = fminf(tb, fmaxf(a, b2));
                                } else if (L.fxo < xlo || L.fxo > xhi) tb = -BIG;
                                if (fabsf(L.dfy) > 1e-20f) {
                                    const float i = __fdividef(1.f, L.dfy), a = (ylo - L.fyo) * i, b2 = (yhi - L.fyo) * i;
                                    ta = fmaxf(ta, fminf(a, b2)); tb = fminf(tb, fmaxf(a, b2));
                                } else if (L.fyo < ylo || L.fyo > yhi) tb = -BIG;
                            }
                            if (ta <= tb) {
                                // re-origin at ta
                                L.ta = ta; L.span = tb - ta;
                                L.xa = L.fxo + ta * L.dfx; L.ya = L.fyo + ta * L.dfy; L.za = L.lz + ta * L.dz;
                                // iterate over the lines of the SLOW axis (rows if |dy| <= |dx|, columns otherwise); the run of
                                // cells a line covers along the fast axis is tested at once against the line-pair occupancy bits
                                L.major_x = fabsf(L.dfx) < fabsf(L.dfy);          // true: lines are columns (transposed masks)
                                L.dM = L.major_x ? L.dfx : L.dfy; L.dm = L.major_x ? L.dfy : L.dfx;
                                L.Ma = L.major_x ? L.xa : L.ya; L.ma = L.major_x ? L.ya : L.xa;
                                L.nM = L.major_x ? L.ncol - 1 : L.nrow - 1; L.nm = L.major_x ? L.nrow - 1 : L.ncol - 1;
                                L.sg = L.dM >= 0.f ? 1 : -1;
                                L.inv_dM = fabsf(L.dM) > 1e-20f ? __fdividef(1.f, L.dM) : 0.f;      // (the line intervals carry a 1e-3 cell slack)
                                const float Mb = L.Ma + L.span * L.dM;
                                int c = (int)floorf(L.Ma - (float)L.sg * 1e-3f), cend = (int)floorf(Mb + (float)L.sg * 1e-3f);
                                L.c = min(max(c, 0), L.nM - 1); L.cend = min(max(cend, 0), L.nM - 1);
                                L.state = ST_SWEEP;
                            }
                        }
                    }
                }
            }
            // ---------------- inside the current chunk: on to the next line of cells with a candidate, then test them
            if (pick == ST_SWEEP && L.state == ST_SWEEP) {
                uint32_t cand, lineA, lineB;
                const uint32_t* mk = L.major_x ? L.m + 15 : L.m;        // row-major masks for rows, transposed for columns
                const int nline = L.major_x ? L.nrow : L.ncol;          // vertices per line
                for (int hop = 0;; hop++) {
                    LANESTAT_LOOP(LS_LINE_ITERS);
                    float s0 = 0.f, s1 = L.span;
                    if (L.inv_dM != 0.f) {
                        const float e0 = ((float)(L.c + (L.sg > 0 ? 0 : 1)) - L.Ma) * L.inv_dM;
                        const float e1 = ((float)(L.c + (L.sg > 0 ? 1 : 0)) - L.Ma) * L.inv_dM;
                        s0 = fmaxf(s0, e0); s1 = fminf(s1, e1);
                    }
                    const float m0 = L.ma + s0 * L.dm, m1 = L.ma + s1 * L.dm;
                    int rlo = (int)floorf(fminf(m0, m1) - 1e-3f), rhi = (int)floorf(fmaxf(m0, m1) + 1e-3f);
                    rlo = min(max(rlo, 0), L.nm - 1); rhi = min(max(rhi, 0), L.nm - 1);
                    // vertex bits of lines c and c+1 along the fast axis
                    lineA = mask_line(mk, L.c * nline, nline); lineB = mask_line(mk, (L.c + 1) * nline, nline);
                    uint32_t occ = lineA | lineB;
                    occ |= occ >> 1;                                    // cell k has a wall vertex among its 4 corners
                    const uint32_t range = (2u << rhi) - (1u << rlo);   // cells rlo..rhi
                    cand = L.floor_reach ? range : (occ & range);
                    if (cand || L.c == L.cend) break;
                    if (FTGP_AB_LINE_MAX > 0 && hop + 1 == FTGP_AB_LINE_MAX) break;      // (cand == 0: the tail below moves on one line)
                    L.c += L.sg;
                }
                float found = BIG;
                while (cand && found == BIG) {
                    LANESTAT_LOOP(LS_CELL_ITERS);
                    const int k = L.dm >= 0.f ? __ffs(cand) - 1 : 31 - __clz(cand);
                    cand &= ~(1u << k);
                    const uint32_t a2 = (lineA >> k) & 3u, b2 = (lineB >> k) & 3u;
                    // corner bits b0 = (c,r), b1 = (c+1,r), b2 = (c,r+1), b3 = (c+1,r+1)
                    const uint32_t bits = L.major_x ? ((a2 & 1u) | ((b2 & 1u) << 1) | ((a2 & 2u) << 1) | ((b2 & 2u) << 2)) : (a2 | (b2 << 2));
                    const int cc = L.major_x ? L.c : k, rr = L.major_x ? k : L.c;
                    bool unsure = false;
                    float s = cell_hit(bits, L.xa - (float)cc, L.ya - (float)rr, L.za, L.dfx, L.dfy, L.dz, -L.ta, unsure);
                    if (unsure) {
                        const int car = L.rid / FTGP_NBEAMS;
                        const float sx = cell_hit_exact(L.th, qpos + (base_car + car) * stride, L.rid - car * FTGP_NBEAMS,
                                                        L.ix, L.iy, L.ncol, L.nrow, cc, rr, bits);
                        s = sx < BIG ? sx - L.ta : BIG;
                    }
                    if (s <= L.span + 1e-4f) found = fminf(found, s);
                }
                if (found < BIG) finish(L, fminf(L.best, fmaxf(L.ta + found, 0.f)), ranges, min_range, base_car);
                else if (L.c == L.cend) L.state = ST_ADV;
                else L.c += L.sg;
            }
        }
    }
#if FTGP_AB_LANESTATS
    for (int k = 0; k < LS_N; k++)
        if (ls[k]) atomicAdd(&g_lane_stats[k], (unsigned long long)ls[k]);
#endif
}

static int ensure_beams(int device) {
    if (device >= 0 && device < 16 && g_beam_ready[device]) return FTGP_OK;
    double h[FTGP_NBEAMS][2];
    const double PI = 3.14159265358979323846;
    for (int j = 0; j < FTGP_NBEAMS; j++) {
        double b = (360.0 / FTGP_NBEAMS * j - 90.0) * PI / 180.0;   // radians(inter_ray_angle*j - 90), mushr.em.xml:21,114
        h[j][0] = sin(b); h[j][1] = cos(b);
    }
    FTGP_CUDA(cudaMemcpyToSymbol(c_beam_sc, h, sizeof h));
    const double tri[MUSHR_CHASSIS_NTRI][9] = MUSHR_CHASSIS_TRI;
    FTGP_CUDA(cudaMemcpyToSymbol(c_chassis_tri, tri, sizeof tri));
    double box[6] = {1e300, 1e300, 1e300, -1e300, -1e300, -1e300};
    for (int f = 0; f < MUSHR_CHASSIS_NTRI; f++)
        for (int k = 0; k < 9; k++) { box[k % 3] = std::min(box[k % 3], tri[f][k] - 1e-9); box[3 + k % 3] = std::max(box[3 + k % 3], tri[f][k] + 1e-9); }
    FTGP_CUDA(cudaMemcpyToSymbol(c_chassis_box, box, sizeof box));
    if (device >= 0 && device < 16) g_beam_ready[device] = true;
    return FTGP_OK;
}

int launch_lidar(const ftgp_geom* g, const double* qpos, int64_t stride, const int32_t* track_id,
                 const uint8_t* visible, const int32_t* lap, int64_t ncars, int cpw, float* ranges, float* min_range,
                 cudaStream_t stream) {
    if (cpw < 1 || cpw > BATCH) { set_error("ftgp_lidar: cars_per_world must be 1..8"); return FTGP_ERR_UNSUPPORTED; }
    GeomHeader gh; memcpy(&gh, g->h_blob.data(), sizeof gh);
    const int threads = 512;
    const size_t scratch = (size_t)(threads / 32) * (BATCH * (FRAME_DOUBLES * 8 + 4) + (cpw > 1 ? MULTI_WORDS * 4 : 0));
    const size_t blob_bytes = (size_t)((gh.lidar_words + 3) / 4) * 16;
    const int stage = blob_bytes + scratch <= 200 * 1024;
    const size_t smem = (stage ? blob_bytes : 0) + scratch;
    static int sm_count[16] = {0};
    int dev = g->device;
    if (dev < 16 && sm_count[dev] == 0) {
        FTGP_CUDA(cudaDeviceGetAttribute(&sm_count[dev], cudaDevAttrMultiProcessorCount, dev));
        FTGP_CUDA(cudaFuncSetAttribute(lidar_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        FTGP_CUDA(cudaFuncSetAttribute(lidar_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    }
    int rc = ensure_beams(dev); if (rc) return rc;
    // CTAs that can be resident on one SM at once, registers included: at 512 threads the kernel's registers leave room
    // for one.  The grid is one wave of those, and the batch size below fills it; counting the shared memory alone
    // gave 2, i.e. a second wave of CTAs queued behind the first and half the cars per batch.
    static size_t occ_smem[16][2];
    static int occ_ctas[16][2];
    const int multi = cpw > 1;
    int per_sm = 1;
    if (dev < 16 && occ_smem[dev][multi] == smem && occ_ctas[dev][multi] > 0) per_sm = occ_ctas[dev][multi];
    else {
        FTGP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, multi ? lidar_kernel<true> : lidar_kernel<false>,
                                                                threads, smem));
        per_sm = std::max(1, std::min(4, per_sm));
        if (dev < 16) { occ_smem[dev][multi] = smem; occ_ctas[dev][multi] = per_sm; }
    }
    int nsm = dev < 16 ? sm_count[dev] : 148;
    // cars per warp batch: 8 for big fleets (best lane utilisation), fewer when the fleet would not fill the GPU
    int wpb = BATCH / cpw;                                      // whole worlds per batch
    while (wpb > 1 && (ncars + wpb * cpw - 1) / (wpb * cpw) < (int64_t)nsm * per_sm * (threads / 32) * 2) wpb >>= 1;
    const int bsz = wpb * cpw;
    int64_t need = ((ncars + bsz - 1) / bsz + (threads / 32) - 1) / (threads / 32);
    int grid = (int)std::min<int64_t>(need, (int64_t)nsm * per_sm);
    if (grid < 1) return FTGP_OK;
    if (cpw > 1)
        lidar_kernel<true><<<grid, threads, smem, stream>>>(g->d_blob, gh.lidar_words, qpos, stride, track_id, visible, lap,
                                                            ncars, cpw, bsz, stage, ranges, min_range);
    else
        lidar_kernel<false><<<grid, threads, smem, stream>>>(g->d_blob, gh.lidar_words, qpos, stride, track_id, visible, lap,
                                                             ncars, cpw, bsz, stage, ranges, min_range);
    count_launch();
    FTGP_CUDA(cudaGetLastError());
#if FTGP_AB_LANESTATS
    g_lane_launch[0] = (int64_t)smem; g_lane_launch[1] = per_sm; g_lane_launch[2] = stage; g_lane_launch[3] = bsz;
#endif
    return FTGP_OK;
}

}  // namespace ftgp
using namespace ftgp;

extern "C" int ftgp_lidar(const ftgp_geom* g, const double* qpos, int64_t qpos_stride,
                          const int32_t* track_id, const uint8_t* visible, const int32_t* lap, int64_t ncars,
                          int cars_per_world, float* ranges, float* min_range, void* stream) {
    if (!g || !qpos || !ranges || ncars < 0 || qpos_stride < 7 || cars_per_world < 1) {
        set_error("ftgp_lidar: bad argument"); return FTGP_ERR_ARG;
    }
    if (ncars == 0) return FTGP_OK;
    FTGP_CUDA(cudaSetDevice(g->device));
    return launch_lidar(g, qpos, qpos_stride, track_id, visible, lap, ncars, cars_per_world, ranges, min_range,
                        (cudaStream_t)stream);
}

extern "C" int ftgp_lidar_host(const ftgp_geom* g, const double* qpos, int64_t qpos_stride,
                               const int32_t* track_id, int64_t ncars, float* ranges) {
    if (!g || !qpos || !ranges || ncars < 0 || qpos_stride < 7) { set_error("ftgp_lidar_host: bad argument"); return FTGP_ERR_ARG; }
    if (ncars == 0) return FTGP_OK;
    FTGP_CUDA(cudaSetDevice(g->device));
    ftgp_geom* gm = const_cast<ftgp_geom*>(g);
    size_t b_pose = (size_t)ncars * 7 * sizeof(double), b_tid = track_id ? (size_t)ncars * 4 : 0;
    size_t b_rng = (size_t)ncars * FTGP_NBEAMS * sizeof(float);
    size_t o_tid = (b_pose + 255) & ~(size_t)255, o_rng = (o_tid + b_tid + 255) & ~(size_t)255;
    size_t need = o_rng + b_rng;
    if (need > gm->scratch_bytes) {
        if (gm->d_scratch) cudaFree(gm->d_scratch);
        gm->d_scratch = nullptr; gm->scratch_bytes = 0;
        FTGP_CUDA(cudaMalloc(&gm->d_scratch, need));
        gm->scratch_bytes = need;
    }
    char* base = (char*)gm->d_scratch;
    cudaStream_t s = gm->host_stream;
    // only the free-joint pose (7 doubles per car) crosses the bus
    FTGP_CUDA(cudaMemcpy2DAsync(base, 7 * sizeof(double), qpos, qpos_stride * sizeof(double), 7 * sizeof(double),
                                ncars, cudaMemcpyHostToDevice, s));
    if (track_id) FTGP_CUDA(cudaMemcpyAsync(base + o_tid, track_id, b_tid, cudaMemcpyHostToDevice, s));
    int rc = launch_lidar(g, (const double*)base, 7, track_id ? (const int32_t*)(base + o_tid) : nullptr, nullptr, nullptr,
                          ncars, 1, (float*)(base + o_rng), nullptr, s);
    if (rc) return rc;
    FTGP_CUDA(cudaMemcpyAsync(ranges, base + o_rng, b_rng, cudaMemcpyDeviceToHost, s));
    FTGP_CUDA(cudaStreamSynchronize(s));
    return FTGP_OK;
}

#if FTGP_AB_LANESTATS
// A/B builds only (tools/lidar_ab.py): out[0..LS_N) = the counters summed since the last call, which zeroes them,
// then shared memory, CTAs per SM, track staged, cars per batch of the last launch.
extern "C" int ftgp_lidar_lanestats(unsigned long long* out) {
    FTGP_CUDA(cudaDeviceSynchronize());
    FTGP_CUDA(cudaMemcpyFromSymbol(out, g_lane_stats, sizeof g_lane_stats));
    const unsigned long long zero[LS_N] = {};
    FTGP_CUDA(cudaMemcpyToSymbol(g_lane_stats, zero, sizeof zero));
    for (int k = 0; k < 4; k++) out[LS_N + k] = (unsigned long long)g_lane_launch[k];
    return FTGP_OK;
}
#endif
