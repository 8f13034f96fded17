// fleet.cu -- the per-car, per-tick kernels around the two heavy ones (lidar.cu, step.cu):
//
//   reset_kernel    mj_resetData + position_vehicles      ft_grandprix/custom.py:1092,1232-1245
//   drivers_kernel  the bundled disparity-extender drivers ft_grandprix/nidc.py:116-131,
//                                                          ft_grandprix/fast.py:118-139,
//                                                          ft_grandprix/lobotomy.py:1-3
//                   + the control write                    ft_grandprix/custom.py:1418-1423
//   lap_kernel      progress / lap state machine           ft_grandprix/custom.py:1340-1372
//   reload_kernel   reload() of the worlds whose race is over, ft_grandprix/custom.py:1089-1128
//                   with the race tally of their cars
//
// Layout: one warp per car for the driver (lane l owns beams l, l+32, l+64 of the 68-beam
// front window, so the ranges row is read with coalesced 128-byte loads and the sequential
// "extend disparities" loop runs as warp-uniform control flow with shuffles); one thread per
// world for the lap logic (cars of one world are ranked in car order, exactly as the
// reference's `for vehicle_state in self.vehicle_states` loop does).
#include <math.h>
#include "common.h"

namespace ftgp {

// ------------------------------------------------------------------ reset
__device__ __forceinline__ void reset_car(int64_t i, double* __restrict__ qpos, double* __restrict__ qvel, double* __restrict__ warm,
                                          double* __restrict__ ctrl, const double* __restrict__ xy, const double* __restrict__ yaw) {
    double* q = qpos + i * FTGP_NQ;
    // qpos0: free joint at the body pos (0, 2, 0) with identity quat, hinges/slides 0, balls identity
    // (mushr.em.xml:96); position_vehicles then overwrites x, y and the quaternion (custom.py:1244-1245)
    for (int k = 0; k < FTGP_NQ; k++) q[k] = 0.0;
    q[0] = xy[2 * i]; q[1] = xy[2 * i + 1]; q[2] = 0.0;
    // euler_to_quaternion([yaw, 0, 0]) (custom.py:81-87): cr = cp = 1, sr = sp = 0
    const double h = yaw[i] * 0.5;
    q[3] = cos(h); q[4] = 0.0; q[5] = 0.0; q[6] = sin(h);
    q[11] = 1.0; q[18] = 1.0; q[24] = 1.0; q[30] = 1.0;          // ball joints of the four softener bodies
    for (int k = 0; k < FTGP_NV; k++) { qvel[i * FTGP_NV + k] = 0.0; warm[i * FTGP_NV + k] = 0.0; }
    if (ctrl) { ctrl[2 * i] = 0.0; ctrl[2 * i + 1] = 0.0; }
}

__global__ void reset_kernel(double* __restrict__ qpos, double* __restrict__ qvel, double* __restrict__ warm,
                             double* __restrict__ ctrl, const double* __restrict__ xy,
                             const double* __restrict__ yaw, int64_t ncars) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ncars) return;
    reset_car(i, qpos, qvel, warm, ctrl, xy, yaw);
}

// ------------------------------------------------------------------ reload of finished worlds (custom.py:1089-1128)
// One thread per world, as the lap kernel: the due test reads the FINISHED flags of every car of the world and
// race_start[w], and the reset writes both, so the thread that decides is the only one that writes the world (worlds of
// 3, 5, 6 or 7 cars do not align to warps).  A world that is not due costs one int32 load (race_start, when race_ticks
// decides) or the FINISHED flags up to the first car still racing, and no store.
__global__ void reload_kernel(double* __restrict__ qpos, double* __restrict__ qvel, double* __restrict__ warm,
                              double* __restrict__ ctrl, float* __restrict__ ranges, int32_t* __restrict__ lap,
                              int32_t* __restrict__ times, int32_t* __restrict__ winners, int32_t* __restrict__ status,
                              int64_t ncars, int cpw, const double* __restrict__ start_xy, const double* __restrict__ start_yaw,
                              const int32_t* __restrict__ start_offset, int32_t* __restrict__ race_start,
                              int32_t* __restrict__ tally, int32_t race_ticks, int32_t steps, const int32_t* __restrict__ steps_dev) {
    const int64_t world = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t first = world * cpw;
    if (first >= ncars) return;
    const int64_t end = first + cpw < ncars ? first + cpw : ncars;
    if (steps_dev) steps = *steps_dev;              // graph-replayed tick: the value the lap kernel reads after this one
    bool due = race_ticks > 0 && (int64_t)steps - race_start[world] >= race_ticks;
    if (!due) {
        due = true;
        for (int64_t car = first; car < end; car++)
            if (!lap[car * FTGP_LAP_FIELDS + FTGP_LAP_FINISHED]) { due = false; break; }
    }
    if (!due) return;
    for (int64_t car = first; car < end; car++) {
        int32_t* s = lap + car * FTGP_LAP_FIELDS;
        int32_t* tm = times + car * FTGP_MAX_LAPTIMES;
        if (tally) {                                  // the race that just ended
            int32_t* t = tally + car * FTGP_RACE_FIELDS;
            const int nt = s[FTGP_LAP_NTIMES] < FTGP_MAX_LAPTIMES ? s[FTGP_LAP_NTIMES] : FTGP_MAX_LAPTIMES;
            int32_t sum = 0, best = t[FTGP_RACE_BEST_LAP];
            for (int k = 0; k < nt; k++) {
                const int32_t v = tm[k];
                sum += v;
                if (v > 0 && (best == 0 || v < best)) best = v;
            }
            t[FTGP_RACE_RACES] += 1;
            t[FTGP_RACE_FINISHED] += s[FTGP_LAP_FINISHED];
            t[FTGP_RACE_WINS] += s[FTGP_LAP_RANK] == 1;
            t[FTGP_RACE_RANK_SUM] += s[FTGP_LAP_RANK];
            t[FTGP_RACE_LAPS_SUM] += s[FTGP_LAP_LAPS];
            if (s[FTGP_LAP_FINISHED]) t[FTGP_RACE_TIME_SUM] += sum;
            t[FTGP_RACE_BEST_LAP] = best;
            t[FTGP_RACE_OFFTRACK_TICKS] += s[FTGP_LAP_OFFTRACK_TICKS];
            t[FTGP_RACE_CONTACT_TICKS] += s[FTGP_LAP_CONTACT_TICKS];
        }
        // what Fleet.reset(xy, yaw) leaves: ftgp_reset, then ranges / lap / times / status zero, VehicleState(offset,
        // good_start=True) (custom.py:96-118); START = steps keeps every lap time equal to a fresh fleet's
        reset_car(car, qpos, qvel, warm, ctrl, start_xy, start_yaw);
        for (int k = 0; k < FTGP_NBEAMS; k++) ranges[car * FTGP_NBEAMS + k] = 0.0f;
        for (int k = 0; k < FTGP_MAX_LAPTIMES; k++) tm[k] = 0;
        for (int k = 0; k < FTGP_LAP_FIELDS; k++) s[k] = 0;
        s[FTGP_LAP_OFFSET] = start_offset[car];
        s[FTGP_LAP_GOOD_START] = 1;
        s[FTGP_LAP_START] = steps;
        if (status) status[car] = 0;
    }
    if (winners) winners[world] = 0;
    if (race_start) race_start[world] = steps;
}

int launch_reload(const ftgp_tick_args* a, const ftgp_reload_args* r, int32_t steps, cudaStream_t stream,
                  const int32_t* steps_dev) {
    const int64_t nworlds = (a->ncars + a->cars_per_world - 1) / a->cars_per_world;
    const int threads = 128;
    reload_kernel<<<(unsigned)((nworlds + threads - 1) / threads), threads, 0, stream>>>(
        a->qpos, a->qvel, a->warm, a->ctrl, a->ranges, a->lap, a->times, a->winners, a->status, a->ncars, a->cars_per_world,
        r->start_xy, r->start_yaw, r->start_offset, r->race_start, r->tally, r->race_ticks, steps, steps_dev);
    count_launch();
    FTGP_CUDA(cudaGetLastError());
    return FTGP_OK;
}

// ------------------------------------------------------------------ option naive_flatten (custom.py:981,1338-1339)
// qpos[3:7] = euler_to_quaternion([quaternion_to_angle(*qpos[3:7]), 0, 0]) (custom.py:62-87): keep the yaw, drop pitch / roll
__global__ void flatten_kernel(double* __restrict__ qpos, int64_t stride, int64_t ncars) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ncars) return;
    double* q = qpos + i * stride + 3;
    const double w = q[0], x = q[1], y = q[2], z = q[3];
    const double yaw = atan2(2.0 * (w * z + x * y), 1.0 - 2.0 * (y * y + z * z));
    q[0] = cos(yaw / 2); q[1] = 0.0; q[2] = 0.0; q[3] = sin(yaw / 2);
}
int launch_flatten(double* qpos, int64_t stride, int64_t ncars, cudaStream_t stream) {
    flatten_kernel<<<(unsigned)((ncars + 127) / 128), 128, 0, stream>>>(qpos, stride, ncars);
    count_launch();
    FTGP_CUDA(cudaGetLastError());
    return FTGP_OK;
}

// ------------------------------------------------------------------ drivers
constexpr int NPROC = 68;             // 90 - 2 * int(90 / 8)          nidc.py:17-18
constexpr int EIGHTH = 11;

__device__ __forceinline__ double pick(double e0, double e1, double e2, int idx) {
    // value of element idx of the warp-distributed array (uniform idx)
    int slot = idx >> 5;
    double v = slot == 0 ? e0 : (slot == 1 ? e1 : e2);
    return __shfl_sync(0xffffffffu, v, idx & 31);
}

// Field F of the reference row of a bundled kind (include/ftgp.h FTGP_DRV_*), folded at compile time.
__device__ __forceinline__ double default_field(bool nidc, int f) {
    const double PI = 3.141592653589793;
    switch (f) {
    case FTGP_DRV_CAR_WIDTH:            return nidc ? 0.12 : 0.06;               // nidc.py:5, fast.py:4
    case FTGP_DRV_SAFETY_PERCENTAGE:    return 300.;                             // nidc.py:10
    case FTGP_DRV_DIFFERENCE_THRESHOLD: return 0.6;                              // nidc.py:7
    case FTGP_DRV_SPEED:                return 0.5;                              // nidc.py:8
    case FTGP_DRV_SPEED_DIVISOR:        return nidc ? 1.57 * 2 : PI;             // nidc.py:130, fast.py:138
    case FTGP_DRV_MAX_STEER:            return 90.0 * (PI / 180.0);              // nidc.py:113
    case FTGP_DRV_BOOST_SPEED:          return 7;                                // fast.py:136
    case FTGP_DRV_BOOST_MAX_STEER:      return nidc ? 0.0 : 0.1;                 // fast.py:135 (nidc: never)
    case FTGP_DRV_BOOST_MIN_REAR_RANGE: return 0.5;                              // fast.py:135
    default:                            return nidc ? INFINITY : 2.0;            // fast.py:138 SPEED_CAP
    }
}
// the car's row (lane-uniform address: one broadcast load per field), or its kind's reference row
template <int F> __device__ __forceinline__ double drv(const double* __restrict__ row, int k) {
    return row ? row[F] : default_field(k == FTGP_DRIVER_NIDC, F);
}

__global__ void __launch_bounds__(256)
drivers_kernel(const float* __restrict__ ranges, const int32_t* __restrict__ kind, int default_kind,
               const double* __restrict__ params, const int32_t* __restrict__ lap, double* __restrict__ ctrl, int64_t ncars,
               int32_t* __restrict__ steps_dev, bool bank) {
    const int lane = threadIdx.x & 31;
    const int64_t car = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    // graph-replayed tick: the lap kernel (earlier on this stream) has read the tick counter; nothing else reads it this tick
    if (steps_dev && blockIdx.x == 0 && threadIdx.x == 0) *steps_dev += 1;
    if (car >= ncars) return;
    int k = kind ? kind[car] : default_kind;
    if (lap && lap[car * FTGP_LAP_FIELDS + FTGP_LAP_FINISHED]) k = FTGP_DRIVER_LOBOTOMY;   // shadow(): custom.py:1437
    if (k == FTGP_DRIVER_POLICY) {                  // policy_kernel (policy.cu) drives it; without a bank it is inert
        if (bank) return;
        k = FTGP_DRIVER_LOBOTOMY;
    }
    double* out = ctrl + 2 * car;
    if (k == FTGP_DRIVER_LOBOTOMY) { if (lane == 0) { out[0] = 0.0; out[1] = 0.0; } return; }
    const double* prow = params ? params + car * FTGP_DRV_FIELDS : nullptr;
    const float* row = ranges + car * FTGP_NBEAMS;
    const double PI = 3.141592653589793;
    const double rpp = (2 * PI) / FTGP_NBEAMS;                  // nidc.py:121
    // proc = ranges[11:79]
    double e0 = (double)row[EIGHTH + lane];
    double e1 = (double)row[EIGHTH + 32 + lane];
    double e2 = lane < NPROC - 64 ? (double)row[EIGHTH + 64 + lane] : 0.0;
    const float r0 = row[0];
    // disparities from the unmodified array (nidc.py:123-124): |proc[i] - proc[i-1]| > threshold, i >= 1
    const double thr = drv<FTGP_DRV_DIFFERENCE_THRESHOLD>(prow, k);
    double p0 = __shfl_up_sync(0xffffffffu, e0, 1);
    double l0 = __shfl_sync(0xffffffffu, e0, 31), l1 = __shfl_sync(0xffffffffu, e1, 31);
    double p1 = __shfl_up_sync(0xffffffffu, e1, 1); if (lane == 0) p1 = l0;
    double p2 = __shfl_up_sync(0xffffffffu, e2, 1); if (lane == 0) p2 = l1;
    unsigned m0 = __ballot_sync(0xffffffffu, lane > 0 && fabs(e0 - p0) > thr);
    unsigned m1 = __ballot_sync(0xffffffffu, fabs(e1 - p1) > thr);
    unsigned m2 = __ballot_sync(0xffffffffu, lane < NPROC - 64 && fabs(e2 - p2) > thr);
    // nidc.py:93; with the reference rows this equals the constant the literals fold to, bit for bit
    const double width = (drv<FTGP_DRV_CAR_WIDTH>(prow, k) / 2) * (1 + drv<FTGP_DRV_SAFETY_PERCENTAGE>(prow, k) / 100);
    bool raised = false;
    for (int seg = 0; seg < 3 && !raised; seg++) {
        unsigned m = seg == 0 ? m0 : (seg == 1 ? m1 : m2);
        while (m) {
            int i = 32 * seg + __ffs(m) - 1; m &= m - 1;
            int first = i - 1;
            double a = pick(e0, e1, e2, first), b = pick(e0, e1, e2, first + 1);
            // np.argmin / np.argmax over two elements: first NaN wins, ties -> index 0
            int amin = isnan(a) ? 0 : (isnan(b) ? 1 : (b < a ? 1 : 0));
            int amax = isnan(a) ? 0 : (isnan(b) ? 1 : (b > a ? 1 : 0));
            int close = first + amin, far = first + amax;
            double dist = amin ? b : a;
            double angle = 2 * atan(width / (2 * dist));               // nidc.py:57
            double np_ = ceil(angle / rpp);                            // nidc.py:58
            if (isnan(np_)) { raised = true; break; }                  // int(nan) -> ValueError -> ctrl kept
            long num = (long)np_;
            // cover_points (nidc.py:71-84): indices close+1 .. close+num (right) or close-1 .. close-num (left)
            long lo, hi;
            if (close < far) { lo = close + 1; hi = close + num; } else { lo = close - num; hi = close - 1; }
            int j0 = lane, j1 = lane + 32, j2 = lane + 64;
            if (j0 >= lo && j0 <= hi && e0 > dist) e0 = dist;
            if (j1 >= lo && j1 <= hi && e1 > dist) e1 = dist;
            if (j2 >= lo && j2 <= hi && j2 < NPROC && e2 > dist) e2 = dist;
        }
    }
    if (raised) return;                                               // custom.py:1409-1411
    // np.argmax: first maximum, first NaN wins
    double bv = e0; int bi = lane;
    bool bn = isnan(e0);
    if (!bn) {
        if (isnan(e1)) { bv = e1; bi = lane + 32; bn = true; }
        else if (e1 > bv) { bv = e1; bi = lane + 32; }
    }
    if (!bn && lane < NPROC - 64) {
        if (isnan(e2)) { bv = e2; bi = lane + 64; bn = true; }
        else if (e2 > bv) { bv = e2; bi = lane + 64; }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        double ov = __shfl_xor_sync(0xffffffffu, bv, off);
        int oi = __shfl_xor_sync(0xffffffffu, bi, off);
        bool on = isnan(ov);
        bool take;
        if (bn || on) take = on && (!bn || oi < bi);
        else take = ov > bv || (ov == bv && oi < bi);
        if (take) { bv = ov; bi = oi; bn = on; }
    }
    if (lane == 0) {
        double ang = ((double)bi - (NPROC / 2.0)) * rpp;              // nidc.py:112
        const double lim = drv<FTGP_DRV_MAX_STEER>(prow, k);          // nidc.py:113
        double st = ang < -lim ? -lim : (ang > lim ? lim : ang);
        double sp;
        if (fabs(st) < drv<FTGP_DRV_BOOST_MAX_STEER>(prow, k) && (double)r0 > drv<FTGP_DRV_BOOST_MIN_REAR_RANGE>(prow, k))
            sp = drv<FTGP_DRV_BOOST_SPEED>(prow, k);                                        // fast.py:135-136
        else {                                                                              // nidc.py:130, fast.py:138
            const double s = drv<FTGP_DRV_SPEED>(prow, k) * 5 * (1 - fabs(st) / drv<FTGP_DRV_SPEED_DIVISOR>(prow, k));
            const double cap = drv<FTGP_DRV_SPEED_CAP>(prow, k);
            sp = s < cap ? s : cap;
        }
        out[0] = sp; out[1] = st;                                      // custom.py:1422-1423
    }
}

// ------------------------------------------------------------------ lap logic
__device__ __forceinline__ int pymod(int a, int b) { int r = a % b; return r < 0 ? r + b : r; }

__global__ void lap_kernel(const uint32_t* __restrict__ blob, const double* __restrict__ qpos, int64_t stride,
                           const int32_t* __restrict__ track_id, int32_t* __restrict__ lap,
                           int32_t* __restrict__ times, int32_t* __restrict__ winners,
                           const int32_t* __restrict__ status, int64_t ncars, int cpw, int32_t steps,
                           int32_t lap_target, const int32_t* __restrict__ steps_dev) {
    if (steps_dev) steps = *steps_dev;              // graph-replayed tick: self.steps lives on the device
    const int64_t world = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t first = world * cpw;
    if (first >= ncars) return;
    const GeomHeader* gh = reinterpret_cast<const GeomHeader*>(blob);
    int32_t nwin = winners ? winners[world] : 0;
    for (int64_t car = first; car < first + cpw && car < ncars; car++) {
        int tid = track_id ? track_id[car] : 0;
        if (tid < 0 || tid >= gh->ntracks) tid = 0;
        const TrackHeader* th = reinterpret_cast<const TrackHeader*>(blob + gh->track_off[tid]);
        int32_t* s = lap + car * FTGP_LAP_FIELDS;
        if (status && ((status[car] >> 16) & 0xFF)) s[FTGP_LAP_CONTACT_TICKS] += 1;
        if (th->path_off < 0) continue;
        const double* path = reinterpret_cast<const double*>(blob + th->path_off);
        const double x = qpos[car * stride], y = qpos[car * stride + 1];
        int closest = 0; double best = 0;
        for (int k = 0; k < FTGP_NPATH; k++) {                        // custom.py:1341-1342
            double dx = path[2 * k] - x, dy = path[2 * k + 1] - y;
            double d = dx * dx + dy * dy;
            if (k == 0 || d < best) { best = d; closest = k; }
        }
        const int off = best > 1;                                     // custom.py:1343-1344
        s[FTGP_LAP_OFF_TRACK] = off;
        if (off) { s[FTGP_LAP_OFFTRACK_TICKS] += 1; continue; }
        const int completion = pymod(closest - s[FTGP_LAP_OFFSET], 100);
        const int draw = completion - s[FTGP_LAP_COMPLETION];
        const int delta = pymod(draw + 50, 100) - 50;
        s[FTGP_LAP_DELTA] = delta;
        if (abs(draw) > 90) {
            const int lap_steps = steps - s[FTGP_LAP_START];
            if (delta < 0) {
                s[FTGP_LAP_LAPS] -= 1; s[FTGP_LAP_GOOD_START] = 0;
                if (s[FTGP_LAP_NTIMES] != 0) s[FTGP_LAP_NTIMES] -= 1;
            } else if (delta > 0) {
                if (s[FTGP_LAP_GOOD_START]) {
                    int n = s[FTGP_LAP_NTIMES];
                    if (n < FTGP_MAX_LAPTIMES) times[car * FTGP_MAX_LAPTIMES + n] = lap_steps;
                    s[FTGP_LAP_NTIMES] = n + 1;
                    s[FTGP_LAP_START] = steps;
                }
                s[FTGP_LAP_LAPS] += 1; s[FTGP_LAP_GOOD_START] = 1;
            }
        }
        if (s[FTGP_LAP_LAPS] >= lap_target) {                         // custom.py:1367-1371
            if (s[FTGP_LAP_RANK] == 0) { nwin += 1; s[FTGP_LAP_RANK] = nwin; }
            s[FTGP_LAP_FINISHED] = 1;
        }
        s[FTGP_LAP_COMPLETION] = completion;                          // custom.py:1372
    }
    if (winners) winners[world] = nwin;
}

int launch_drivers(const float* ranges, const int32_t* kind, int default_kind, const double* params, const int32_t* lap,
                   double* ctrl, int64_t ncars, cudaStream_t stream, int32_t* steps_dev, bool bank) {
    const int threads = 256;
    int64_t blocks = (ncars * 32 + threads - 1) / threads;
    drivers_kernel<<<(unsigned)blocks, threads, 0, stream>>>(ranges, kind, default_kind, params, lap, ctrl, ncars, steps_dev, bank);
    count_launch();
    FTGP_CUDA(cudaGetLastError());
    return FTGP_OK;
}

int launch_lap(const ftgp_geom* g, const double* qpos, int64_t stride, const int32_t* track_id, int32_t* lap,
               int32_t* times, int32_t* winners, const int32_t* status, int64_t ncars, int cpw, int32_t steps,
               int32_t lap_target, cudaStream_t stream, const int32_t* steps_dev) {
    int64_t nworlds = (ncars + cpw - 1) / cpw;
    const int threads = 128;
    lap_kernel<<<(unsigned)((nworlds + threads - 1) / threads), threads, 0, stream>>>(
        g->d_blob, qpos, stride, track_id, lap, times, winners, status, ncars, cpw, steps, lap_target, steps_dev);
    count_launch();
    FTGP_CUDA(cudaGetLastError());
    return FTGP_OK;
}

}  // namespace ftgp
using namespace ftgp;

extern "C" int ftgp_reset(double* qpos, double* qvel, double* warm, double* ctrl, const double* xy,
                          const double* yaw, int64_t ncars, void* stream) {
    if (!qpos || !qvel || !warm || !xy || !yaw || ncars < 0) { set_error("ftgp_reset: bad argument"); return FTGP_ERR_ARG; }
    if (ncars == 0) return FTGP_OK;
    reset_kernel<<<(unsigned)((ncars + 127) / 128), 128, 0, (cudaStream_t)stream>>>(qpos, qvel, warm, ctrl, xy, yaw, ncars);
    count_launch();
    FTGP_CUDA(cudaGetLastError());
    return FTGP_OK;
}

extern "C" int ftgp_naive_flatten(double* qpos, int64_t qpos_stride, int64_t ncars, void* stream) {
    if (!qpos || ncars < 0 || qpos_stride < 7) { set_error("ftgp_naive_flatten: bad argument"); return FTGP_ERR_ARG; }
    if (ncars == 0) return FTGP_OK;
    return launch_flatten(qpos, qpos_stride, ncars, (cudaStream_t)stream);
}

extern "C" int ftgp_drivers_policy(const float* ranges, const int32_t* kind, int default_kind, const double* params,
                                   const ftgp_policy_args* policy, const double* qpos, const double* qvel, const int32_t* lap,
                                   double* ctrl, int64_t ncars, void* stream) {
    if (!ranges || !ctrl || ncars < 0 || default_kind < 0 || default_kind > FTGP_DRIVER_POLICY) { set_error("ftgp_drivers: bad argument"); return FTGP_ERR_ARG; }
    if (bad_policy_args(policy, default_kind) || (policy && (!qpos || !qvel))) { set_error("ftgp_drivers: bad policy argument"); return FTGP_ERR_ARG; }
    if (ncars == 0) return FTGP_OK;
    int rc = launch_drivers(ranges, kind, default_kind, params, lap, ctrl, ncars, (cudaStream_t)stream, nullptr, policy != nullptr);
    if (!rc && policy) rc = launch_policy(policy, ranges, kind, default_kind, qpos, qvel, lap, ctrl, ncars, (cudaStream_t)stream);
    return rc;
}

extern "C" int ftgp_drivers_params(const float* ranges, const int32_t* kind, int default_kind, const double* params,
                                   const int32_t* lap, double* ctrl, int64_t ncars, void* stream) {
    return ftgp_drivers_policy(ranges, kind, default_kind, params, nullptr, nullptr, nullptr, lap, ctrl, ncars, stream);
}

extern "C" int ftgp_drivers(const float* ranges, const int32_t* kind, int default_kind, const int32_t* lap,
                            double* ctrl, int64_t ncars, void* stream) {
    return ftgp_drivers_params(ranges, kind, default_kind, nullptr, lap, ctrl, ncars, stream);
}

extern "C" int ftgp_lap_update(const ftgp_geom* g, const double* qpos, int64_t qpos_stride,
                               const int32_t* track_id, int32_t* lap, int32_t* times, int32_t* winners,
                               const int32_t* status, int64_t ncars, int cars_per_world, int32_t steps,
                               int32_t lap_target, void* stream) {
    if (!g || !qpos || !lap || !times || ncars < 0 || cars_per_world < 1 || qpos_stride < 2) {
        set_error("ftgp_lap_update: bad argument"); return FTGP_ERR_ARG;
    }
    if (ncars == 0) return FTGP_OK;
    FTGP_CUDA(cudaSetDevice(g->device));
    return launch_lap(g, qpos, qpos_stride, track_id, lap, times, winners, status, ncars, cars_per_world, steps,
                      lap_target, (cudaStream_t)stream, nullptr);
}
