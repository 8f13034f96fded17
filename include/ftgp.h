/*
 * ftgp.h -- C ABI of libftgp.so: the B200-native replacement for the engine
 * boundary that ft_grandprix's per-tick loop sits on (SURVEY.md §8 b, B2).
 *
 * Every entry point cites the reference interface it replaces (paths relative to
 * the reference repo FT-Autonomous/ft_grandprix).  Conventions:
 *   - plain pointers and sizes, no C++/torch types; every call returns an int
 *     status (0 = ok) unless it returns a handle (NULL = error);
 *     ftgp_last_error() gives the thread-local message.
 *   - "device pointer" arguments are CUDA device memory on the geometry's device,
 *     owned by the caller (torch allocations); `stream` is a cudaStream_t passed
 *     as void* (NULL = legacy default stream).  Device calls are asynchronous on
 *     that stream and never synchronise; *_host variants take host buffers, copy
 *     in/out on an internal stream and return when the result is in host memory.
 *   - state layout (one row per car, row-major, fp64 like MuJoCo's mjtNum):
 *       qpos[ncars][34], qvel[ncars][29], warm[ncars][29], ctrl[ncars][2]
 *     ctrl = (forward #i, turn #i) = (speed, steering_angle)  (custom.py:1422-1423)
 *     ranges[ncars][90] fp32, -1 on miss                     (custom.py:1395)
 *   - there is no CPU fallback: on a machine without a CUDA device every device
 *     call fails with FTGP_ERR_CUDA.
 */
#ifndef FTGP_H
#define FTGP_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FTGP_NBEAMS 90   /* custom.py:1158 rangefinders=90 */
#define FTGP_NQ 34       /* template/mushr.em.xml:95-174 */
#define FTGP_NV 29
#define FTGP_NU 2
#define FTGP_NPATH 100   /* curve.py:8 points=100 */
#define FTGP_MAX_TRACKS 4
#define FTGP_MAX_LAPTIMES 16

enum {
    FTGP_OK = 0,
    FTGP_ERR_ARG = 1,
    FTGP_ERR_CUDA = 2,
    FTGP_ERR_ALLOC = 3,
    FTGP_ERR_UNSUPPORTED = 4
};

enum { FTGP_DRIVER_NIDC = 0, FTGP_DRIVER_FAST = 1, FTGP_DRIVER_LOBOTOMY = 2, FTGP_DRIVER_POLICY = 3 };
enum { FTGP_OPT_NAIVE_FLATTEN = 1, FTGP_OPT_BUBBLE_WRAP = 2 };   /* path-relevant options of custom.py:946-989 */

const char* ftgp_last_error(void);
int ftgp_abi_version(void);
/* number of kernels this library has launched in this process (bench gpu_launches) */
int64_t ftgp_launch_count(void);

/* ------------------------------------------------------------------ track (host) */
typedef struct ftgp_track ftgp_track;

/* Replaces ft_grandprix.chunk.chunk() (chunk.py:10-80) + the hfield placement that
 * produce_mjcf()/mushr.em.xml emit (map.py:27-65, mushr.em.xml:19-20,55,92).
 * pixels: uint8[h][w][channels]; channels == 3: RGB, wall iff R+G+B == 765
 * (chunk.py:39-43); channels == 1: wall iff non-zero.  scale: chunk(scale=2.0)
 * (custom.py:1155); chunk_px: 20. */
ftgp_track* ftgp_track_create(const uint8_t* pixels, int w, int h, int channels,
                              double scale, int chunk_px);
void ftgp_track_destroy(ftgp_track* t);
/* metadata.json fields (chunk.py:67-79): out[0]=horizontal_chunks, [1]=vertical_chunks,
 * [2]=number of non-empty chunks, [3]=width, [4]=height, [5]=chunk_px */
int ftgp_track_meta(const ftgp_track* t, int32_t* out6, double* size_xy2);
/* metadata["chunks"]: ij[2*k], ij[2*k+1] in chunk.py's scan order; counts[k] = wall pixels */
int ftgp_track_chunks(const ftgp_track* t, int32_t* ij, int32_t* counts);
/* Replaces extract_path_from_svg (curve.py:6-18) + custom.py:1184-1186.  d = the SVG path
 * data string; out: double[npoints][2] metres. */
int ftgp_centreline(const char* svg_d, int npoints, int img_w, int img_h, int chunk_w,
                    int chunk_h, double scale, double* out);

/* ------------------------------------------------------------------ geometry (device) */
typedef struct ftgp_geom ftgp_geom;
/* Replaces MjModel.from_xml_path for the static world (custom.py:1178): packs up to
 * FTGP_MAX_TRACKS compiled tracks (chunk index grid + per-chunk vertex bit masks) plus
 * their centrelines (double[100][2] each, may be NULL) into one device blob on `device`. */
ftgp_geom* ftgp_geom_create(const ftgp_track* const* tracks, const double* const* paths,
                            int ntracks, int device);
void ftgp_geom_destroy(ftgp_geom* g);
/* Host-only: the same geometry blob in host memory (no CUDA device needed; for tools and the CPU test harness).
 * Returns the blob size in 32-bit words (out may be NULL to query it), -1 on error. */
int64_t ftgp_geom_blob(const ftgp_track* const* tracks, const double* const* paths, int ntracks,
                       uint32_t* out, int64_t cap_words);
/* Where one track sits inside a blob: out4 = {index grid offset, chunk table offset (32-bit words), horizontal_chunks,
 * vertical_chunks}, size_xy2 = chunk pitch in metres.  index grid: uint16[vc][hc] (row vc-1-j), chunk table: 28 words each. */
int ftgp_blob_track_view(const uint32_t* blob, int track, int32_t* out4, double* size_xy2);
int ftgp_geom_device(const ftgp_geom* g);
int64_t ftgp_geom_bytes(const ftgp_geom* g);

/* ------------------------------------------------------------------ lidar */
/* Replaces data.sensordata[vehicle_state.sensors] (custom.py:1395): the 90 rangefinder
 * sensors of mushr.em.xml:112-117,204-206 evaluated by mj_ray from the pose in qpos.
 * qpos: device double[ncars][qpos_stride] (first 7 = free joint).  track_id: device
 * int32[ncars] or NULL (all on track 0).  cars_per_world in 2..8: consecutive cars share a
 * world and see each other's lidar cylinder (mushr.em.xml:108); visible: device
 * uint8[ncars] or NULL (0 = shadowed car, custom.py:1455-1464).
 * lap: device lap state (FTGP_LAP_* rows, see below) or NULL; a car whose FTGP_LAP_FINISHED field
 * is set has been shadow()ed (custom.py:1436-1464): its rangefinders are switched off (its
 * ranges row keeps the stale values) and the other cars no longer see it.
 * ranges: device float[ncars][90].  min_range: device float[ncars] or NULL (smallest
 * non-negative range of the scan, +inf if none). */
int ftgp_lidar(const ftgp_geom* g, const double* qpos, int64_t qpos_stride,
               const int32_t* track_id, const uint8_t* visible, const int32_t* lap, int64_t ncars,
               int cars_per_world, float* ranges, float* min_range, void* stream);
/* host-buffer variant (same arguments in host memory) */
int ftgp_lidar_host(const ftgp_geom* g, const double* qpos, int64_t qpos_stride,
                    const int32_t* track_id, int64_t ncars, float* ranges);

/* ------------------------------------------------------------------ reset */
/* Replaces mj_resetData + position_vehicles (custom.py:1092,1232-1245): qpos = qpos0 with
 * (x, y) = xy[i], z = 0, quat = yaw-only; qvel = warm = ctrl = 0.  xy: device double[ncars][2],
 * yaw: device double[ncars]. */
int ftgp_reset(double* qpos, double* qvel, double* warm, double* ctrl, const double* xy,
               const double* yaw, int64_t ncars, void* stream);

/* ------------------------------------------------------------------ vehicle step */
/* Replaces mujoco.mj_step(model, data) (custom.py:1425) for ncars independent cars of
 * template/mushr.em.xml (timestep 0.004, Newton, pyramidal cones).  status: device
 * int32[ncars] or NULL, per car: bits 0-7 Newton iterations of the last step, bit 8 =
 * state was reset (MuJoCo's bad-state check), bits 16-23 contacts with walls (wheels, chassis hull
 * vertices, lidar cylinder), bits 24-27 wheel-ground contacts, bits 28-30 chassis / lidar-cylinder
 * contacts with the ground (a flipped car), bit 9 = advanced by the coupled world solver, bit 10 = within reach of a
 * wall (the step's own regrouping hint).  g may be NULL (open ground plane, no walls).  lap: device lap state
 * (FTGP_LAP_* rows, see below) or NULL; a car whose FTGP_LAP_FINISHED field is set has been
 * shadow()ed (custom.py:1455-1464: conaffinity 0 / contype 2): it no longer collides with walls.
 * options: FTGP_OPT_* bits; FTGP_OPT_BUBBLE_WRAP = the reference's option bubble_wrap (custom.py:970-972,
 * 1041-1055: the softener spheres of mushr.em.xml:66 get conaffinity 4 and collide with the walls).
 * cars_per_world in 1..8: consecutive cars form one world = one MjModel of the reference (mushr.em.xml:95,
 * template/cars/*.json).  Cars of a world that touch each other (a chassis hull vertex inside the other chassis' hull
 * box) are advanced as ONE constraint problem, as mj_step does for the model (one search direction, one step length,
 * one stopping rule); status bit 9 marks cars advanced that way.  cars_per_world > 1 needs nsteps == 1. */
int ftgp_step(const ftgp_geom* g, double* qpos, double* qvel, double* warm, const double* ctrl,
              const int32_t* track_id, const int32_t* lap, int64_t ncars, int cars_per_world, int nsteps,
              int32_t* status, int options, void* stream);
/* The step keeps per-(device, stream) scratch (regrouping lists, records of the staged solve: about
 * 6 KB per car).  Frees the scratch of `stream` on the current device; call when a fleet is destroyed. */
int ftgp_release_scratch(void* stream);

/* ------------------------------------------------------------------ drivers */
/* Device ports of the bundled drivers (nidc.py:116-131, fast.py:118-139, lobotomy.py:1-3)
 * followed by the control write ctrl[i] = (speed, steering) (custom.py:1418-1423).
 * ranges: device float[ncars][90].  kind: device int32[ncars] (FTGP_DRIVER_*) or NULL
 * (= every car runs `default_kind`).  lap: device lap state (see below) or NULL; a car
 * whose FTGP_LAP_FINISHED field is set runs the lobotomy driver, as shadow() arranges
 * (custom.py:1437).  A scan on which the Python driver would raise (NaN ->
 * ValueError in int(np.ceil(nan))) leaves that car's ctrl untouched (custom.py:1409-1411). */
int ftgp_drivers(const float* ranges, const int32_t* kind, int default_kind, const int32_t* lap,
                 double* ctrl, int64_t ncars, void* stream);

/* Per-car driver parameters: the constants a competitor edits to tune the bundled disparity extender, as one fp64 row
 * per car, params[ncars][FTGP_DRV_FIELDS].  One formula covers both bundled drivers (nidc.py:12-131, fast.py:12-139):
 *   disparity at i >= 1 of proc = ranges[11:79]:  |proc[i] - proc[i-1]| > DIFFERENCE_THRESHOLD
 *   cover width:        (CAR_WIDTH / 2) * (1 + SAFETY_PERCENTAGE / 100)                         nidc.py:93
 *   covered beams:      ceil(2 * atan(width / (2 * dist)) / (2 pi / 90))                        nidc.py:57-58
 *   steering st:        the chosen beam's angle clipped to [-MAX_STEER, MAX_STEER]             nidc.py:112-113
 *   speed:              BOOST_SPEED                      if |st| < BOOST_MAX_STEER and ranges[0] > BOOST_MIN_REAR_RANGE
 *                       s < SPEED_CAP ? s : SPEED_CAP    otherwise, s = SPEED * 5 * (1 - |st| / SPEED_DIVISOR)
 *                                                                                               nidc.py:130, fast.py:135-138
 * The reference instances (the rows used when params is NULL):
 *   field                  nidc                               fast
 *   CAR_WIDTH              0.12                               0.06                  nidc.py:5, fast.py:4
 *   SAFETY_PERCENTAGE      300                                300                   nidc.py:10
 *   DIFFERENCE_THRESHOLD   0.6                                0.6                   nidc.py:7
 *   SPEED                  0.5                                0.5                   nidc.py:8
 *   SPEED_DIVISOR          1.57 * 2                           3.141592653589793     nidc.py:130, fast.py:138
 *   MAX_STEER              90.0 * (3.141592653589793 / 180.0) the same              nidc.py:113 (np.radians(90))
 *   BOOST_SPEED            7                                  7                     fast.py:136
 *   BOOST_MAX_STEER        0 (|st| < 0 never holds)           0.1                   fast.py:135
 *   BOOST_MIN_REAR_RANGE   0.5                                0.5                   fast.py:135 (ranges[0]: the rear beam)
 *   SPEED_CAP              +inf                               2                     fast.py:138
 * The beam window (68 beams from index 11) is fixed.  Rows are not validated: an out-of-range row does exactly what the
 * numpy formula does.  A NaN width (or inf width at inf range) raises at the first disparity and leaves ctrl unchanged,
 * as custom.py:1409-1411 does; a zero or negative width covers nothing; a negative threshold makes every index whose
 * difference is not NaN a disparity, an infinite or NaN one none; atan is bounded, so a disparity covers at most 45
 * beams whatever the width; a NaN speed law gives SPEED_CAP; a NaN MAX_STEER clips nothing. */
enum {
    FTGP_DRV_CAR_WIDTH = 0, FTGP_DRV_SAFETY_PERCENTAGE, FTGP_DRV_DIFFERENCE_THRESHOLD, FTGP_DRV_SPEED,
    FTGP_DRV_SPEED_DIVISOR, FTGP_DRV_MAX_STEER, FTGP_DRV_BOOST_SPEED, FTGP_DRV_BOOST_MAX_STEER,
    FTGP_DRV_BOOST_MIN_REAR_RANGE, FTGP_DRV_SPEED_CAP, FTGP_DRV_FIELDS
};
/* ftgp_drivers with per-car rows: params = device double[ncars][FTGP_DRV_FIELDS] or NULL (= the reference row of each
 * car's kind; ftgp_drivers is this call with NULL).  With rows, a car's row alone decides its driver: kind matters only
 * as FTGP_DRIVER_LOBOTOMY or FTGP_DRIVER_POLICY, and finished cars still run the lobotomy driver.
 * ftgp_drivers_params is ftgp_drivers_policy (below) with no policy bank. */
int ftgp_drivers_params(const float* ranges, const int32_t* kind, int default_kind, const double* params,
                        const int32_t* lap, double* ctrl, int64_t ncars, void* stream);

/* Neural-network drivers: a car of kind FTGP_DRIVER_POLICY runs one policy of a bank, a small MLP of one fixed
 * architecture, fp32.  Inputs x[96], computed per car at the driver's point of the tick (after the lap update, before
 * the step; the ranges are the previous step's, as for the other kinds):
 *   x[j], j = 0..89   r = ranges[j]; (r >= 0 && r < range_clip) ? r / range_clip : 1   (a miss, r >= clip and NaN give 1)
 *   x[90], x[91]      forward and lateral speed in the yaw frame, yaw = atan2(2(wz + xy), 1 - 2(y^2 + z^2)) of qpos[3:7]
 *                     (quaternion_to_euler, custom.py:62-76): fwd = vx cos yaw + vy sin yaw, lat = -vx sin yaw + vy cos yaw,
 *                     (vx, vy) = qvel[0:2]; computed in fp64, rounded to fp32
 *   x[92]             qvel[5]: the free joint's angular velocity about the chassis z axis
 *   x[93], x[94]      the car's ctrl (speed, steering) at the head of the tick (zero after a reset or a reload)
 *   x[95]             0 (padding)
 * Network, hidden width 64, accurate tanhf:
 *   h1 = tanh(b1 + W1^T x),  h2 = tanh(b2 + W2^T h1),  z = b3 + W3^T h2
 *   speed = speed_scale * tanh(z0),  steering = steer_scale * tanh(z1)
 * Every pre-activation is summed in input order, one fused multiply-add per input, starting from the bias, whatever
 * other cars are evaluated with the car: a car's output does not depend on how cars are grouped.
 * One policy = FTGP_POLICY_FLOATS floats (42,016 bytes; every block 16-byte aligned), weights input-major
 * (W[i * width + j] multiplies input i into unit j: the transpose of torch.nn.Linear.weight):
 *   FTGP_POLICY_SCALARS  range_clip, speed_scale, steer_scale, 0
 *   FTGP_POLICY_W1       W1[96][64]        FTGP_POLICY_B1   b1[64]
 *   FTGP_POLICY_W2       W2[64][64]        FTGP_POLICY_B2   b2[64]
 *   FTGP_POLICY_W3       W3[64][2]         FTGP_POLICY_B3   b3[2], 2 floats of padding
 * A POLICY car runs policy policy_id[car] (policy_id NULL: policy 0).  Finished cars run the lobotomy driver; an id
 * outside [0, npolicies) writes (0, 0), as the reference's inert driver on an import failure (custom.py:1106-1109).  The
 * output is written as computed.  Without a bank a POLICY car writes (0, 0). */
enum {
    FTGP_POLICY_NIN = 96, FTGP_POLICY_HIDDEN = 64, FTGP_POLICY_NOUT = 2,
    FTGP_POLICY_SCALARS = 0, FTGP_POLICY_W1 = 4, FTGP_POLICY_B1 = 6148, FTGP_POLICY_W2 = 6212, FTGP_POLICY_B2 = 10308,
    FTGP_POLICY_W3 = 10372, FTGP_POLICY_B3 = 10500, FTGP_POLICY_FLOATS = 10504
};
typedef struct {
    const float* weights;        /* device float[npolicies][FTGP_POLICY_FLOATS] */
    const int32_t* policy_id;    /* device int32[ncars] or NULL (every car on policy 0) */
    int32_t npolicies;           /* >= 1 */
    int32_t reserved;
} ftgp_policy_args;
/* ftgp_drivers_params plus the policy bank: policy NULL is exactly ftgp_drivers_params; with a bank, qpos (device
 * double[ncars][FTGP_NQ]) and qvel (double[ncars][FTGP_NV]) give the inputs x[90..92].  The weights and ids are read by
 * every call (and every graph-replayed tick of ftgp_tick_policy), so a bank rewritten in place in stream order takes
 * effect on the next one.  default_kind in 0..3; FTGP_DRIVER_POLICY needs a bank. */
int ftgp_drivers_policy(const float* ranges, const int32_t* kind, int default_kind, const double* params,
                        const ftgp_policy_args* policy, const double* qpos, const double* qvel, const int32_t* lap,
                        double* ctrl, int64_t ncars, void* stream);

/* ------------------------------------------------------------------ lap logic */
/* Replaces custom.py:1340-1372.  lap: device int32[ncars][FTGP_LAP_FIELDS] (see enum),
 * times: device int32[ncars][FTGP_MAX_LAPTIMES] lap durations in steps (x 0.004 s),
 * winners: device int32[nworlds] = len(self.winners) per world. */
enum {
    FTGP_LAP_OFFSET = 0, FTGP_LAP_COMPLETION, FTGP_LAP_LAPS, FTGP_LAP_START, FTGP_LAP_GOOD_START,
    FTGP_LAP_FINISHED, FTGP_LAP_NTIMES, FTGP_LAP_OFF_TRACK, FTGP_LAP_RANK, FTGP_LAP_DELTA,
    FTGP_LAP_OFFTRACK_TICKS, FTGP_LAP_CONTACT_TICKS, FTGP_LAP_FIELDS
};
int ftgp_lap_update(const ftgp_geom* g, const double* qpos, int64_t qpos_stride,
                    const int32_t* track_id, int32_t* lap, int32_t* times, int32_t* winners,
                    const int32_t* status, int64_t ncars, int cars_per_world, int32_t steps,
                    int32_t lap_target, void* stream);

/* ------------------------------------------------------------------ fused tick */
typedef struct {
    const ftgp_geom* geom;
    double *qpos, *qvel, *warm, *ctrl;     /* device state */
    float* ranges;                          /* device float[ncars][90]: in = last tick's scan */
    const int32_t* track_id;                /* device or NULL */
    const int32_t* driver_kind;             /* device or NULL */
    int32_t *lap, *times, *winners, *status;/* device */
    int64_t ncars;
    int32_t cars_per_world, default_driver, lap_target, steps;
    int32_t options, reserved;              /* FTGP_OPT_* bits: the path-relevant options of custom.py:946-989 */
} ftgp_tick_args;
/* FTGP_OPT_NAIVE_FLATTEN: custom.py:981,1338-1339, every tick keep the chassis' yaw and zero its pitch / roll;
 * FTGP_OPT_BUBBLE_WRAP: custom.py:970-972,1041-1055, the softener spheres collide with the walls */
/* Option naive_flatten on its own (custom.py:1338-1339): qpos[3:7] <- quaternion of (yaw, 0, 0). */
int ftgp_naive_flatten(double* qpos, int64_t qpos_stride, int64_t ncars, void* stream);
/* One iteration of physics_thread (custom.py:1337-1426) for the whole fleet:
 * lap update -> built-in driver on last tick's ranges -> ctrl -> [rangefinders from the
 * pre-step pose, mj_step] ; the same one-tick sensor lag as the reference.
 * cars_per_world > 1: the cars of a world see each other (lidar cylinder, chassis mesh, wheels), are ranked together
 * and collide with each other (see ftgp_step).
 * Fleets of up to 16 384 cars are launch-bound: from the second call with the same arguments and a non-NULL stream the
 * tick is replayed from a CUDA graph captured once (same kernels, same order, bit-identical results; self.steps
 * lives in a device counter).  ftgp_release_graphs() drops the cached graphs. */
int ftgp_tick(const ftgp_tick_args* a, int nticks, void* stream);
int ftgp_release_graphs(void);

/* ------------------------------------------------------------------ race after race (reload(), custom.py:1089-1128) */
/* A world is due at the head of a tick when every one of its cars has FTGP_LAP_FINISHED set, or when race_ticks > 0 and
 * steps - race_start[w] >= race_ticks.  A due world is reloaded before anything else of the tick runs: the race that
 * just ended is added to its cars' tally rows, then its cars are reset exactly as ftgp_reset + a fresh lap state would
 * leave them (qpos / qvel / warm / ctrl from start_xy / start_yaw; ranges, times, status and the lap row zero except
 * FTGP_LAP_OFFSET = start_offset, FTGP_LAP_GOOD_START = 1, FTGP_LAP_START = steps), winners[w] = 0 and
 * race_start[w] = steps.  `steps` is the value the lap update of the same tick sees.  Worlds that are not due are not
 * written.  The start tensors are read when a world is reloaded; the caller may rewrite them between calls. */
enum {
    FTGP_RACE_RACES = 0, FTGP_RACE_FINISHED, FTGP_RACE_WINS, FTGP_RACE_RANK_SUM, FTGP_RACE_LAPS_SUM,
    FTGP_RACE_TIME_SUM, FTGP_RACE_BEST_LAP, FTGP_RACE_OFFTRACK_TICKS, FTGP_RACE_CONTACT_TICKS, FTGP_RACE_FIELDS
};
/* Per car and race: RACES += 1; FINISHED += finished; WINS += rank == 1; RANK_SUM += rank (0 = did not finish);
 * LAPS_SUM += laps; TIME_SUM += the stored lap times (times[0 : min(ntimes, 16)]) of a finished car (run.py:78);
 * BEST_LAP = min(BEST_LAP, stored lap times), 0 = no lap recorded yet; OFFTRACK_TICKS / CONTACT_TICKS += the lap
 * state's FTGP_LAP_OFFTRACK_TICKS / FTGP_LAP_CONTACT_TICKS. */
typedef struct {
    const double* start_xy;      /* device double[ncars][2]  pose of the next race (custom.py:1232-1245) */
    const double* start_yaw;     /* device double[ncars] */
    const int32_t* start_offset; /* device int32[ncars]      FTGP_LAP_OFFSET of the next race */
    int32_t* race_start;         /* device int32[nworlds]    tick at which the world's current race began, or NULL */
    int32_t* tally;              /* device int32[ncars][FTGP_RACE_FIELDS] or NULL (needs race_start) */
    int32_t race_ticks;          /* 0 = a world is due only when all its cars have finished (> 0 needs race_start) */
    int32_t reserved;
} ftgp_reload_args;
/* Un-fused: reload the due worlds now, with steps = a->steps (for loops that issue the tick's pieces one by one). */
int ftgp_reload(const ftgp_tick_args* a, const ftgp_reload_args* r, void* stream);
/* ftgp_tick with the reload at the head of every tick (graph-replayed like ftgp_tick); r == NULL is exactly ftgp_tick. */
int ftgp_tick_reload(const ftgp_tick_args* a, const ftgp_reload_args* r, int nticks, void* stream);
/* ftgp_tick_reload whose drivers read per-car rows (driver_params: device double[ncars][FTGP_DRV_FIELDS] or NULL, see
 * ftgp_drivers_params); ftgp_tick_reload is this call with NULL.  The rows are read by every tick, graph-replayed ones
 * included, so rewriting them in place, in stream order, takes effect on the next tick. */
int ftgp_tick_params(const ftgp_tick_args* a, const ftgp_reload_args* r, const double* driver_params, int nticks,
                     void* stream);
/* ftgp_tick_params whose POLICY cars run the bank (see ftgp_drivers_policy); ftgp_tick_params is this call with
 * policy NULL, and launches exactly the kernels it launched before policies existed.  The cached graph is keyed on the
 * bank's pointers and npolicies; the weights and ids are read by every tick. */
int ftgp_tick_policy(const ftgp_tick_args* a, const ftgp_reload_args* r, const double* driver_params,
                     const ftgp_policy_args* policy, int nticks, void* stream);
/* enable != 0 (default): small fleets replay the captured tick; 0: every tick is issued launch by launch.
 * Returns the previous setting (for A/B timing in the bench). */
int ftgp_tick_use_graphs(int enable);

#ifdef __cplusplus
}
#endif
#endif
