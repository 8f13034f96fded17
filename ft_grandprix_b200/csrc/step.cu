// step.cu -- vehicle-step kernel and the fused per-tick entry point.
//
// ftgp_step replaces mujoco.mj_step(model, data) (ft_grandprix/custom.py:1425) for a fleet of
// independent cars of template/mushr.em.xml; the arithmetic is the block-arrow Newton solver specialised
// for the car's fixed topology (csrc/mushr_step.cuh), mapped four lanes per car, one per wheel chain
// (csrc/mushr_step_quad.cuh), in fp64; cars never interact on this path, so nothing crosses a quad.
// ftgp_tick runs whole iterations of physics_thread (custom.py:1337-1426) without leaving the
// device: lap update -> built-in driver on last tick's ranges -> ctrl -> rangefinders from the
// pre-step pose -> mj_step (the reference's one-tick sensor lag is kept).
#include "common.h"
#include "mushr_consts.h"
#include "mushr_step_quad.cuh"
#include "mushr_world.cuh"
#include <cstdlib>
#include <atomic>
#include <mutex>
#include <utility>

namespace ftgp {
using namespace mushr;

__constant__ ModelConsts c_model;
static bool g_model_ready[16] = {false};
static ModelConsts g_model_host;
static bool g_model_host_ready = false;

static int ensure_model(int device) {
    if (!g_model_host_ready) { g_model_host = model_constants(); g_model_host_ready = true; }
    if (device >= 0 && device < 16 && g_model_ready[device]) return FTGP_OK;
    FTGP_CUDA(cudaMemcpyToSymbol(c_model, &g_model_host, sizeof(ModelConsts)));
    if (device >= 0 && device < 16) g_model_ready[device] = true;
    return FTGP_OK;
}

// the walls of the car's track as the contact rules see them (hfield_contact.cuh); read from global memory (L2-resident, ~50 KB)
__device__ __forceinline__ QHfWalls track_walls(const uint32_t* blob, const int32_t* track_id, int64_t car, bool shadowed, int options) {
    QHfWalls w;
    w.bubble = (options & FTGP_OPT_BUBBLE_WRAP) != 0;       // softener spheres collide with the walls (custom.py:1041-1055)
    w.on = false; w.hv.index = nullptr; w.hv.chunks = nullptr; w.hv.hc = w.hv.vc = 0; w.hv.size_x = w.hv.size_y = 1;
    if (!blob || shadowed) return w;        // a finished ("shadowed") car no longer collides with walls (custom.py:1455-1464)
    const GeomHeader* gh = reinterpret_cast<const GeomHeader*>(blob);
    int tid = track_id ? track_id[car] : 0;
    if (tid < 0 || tid >= gh->ntracks) tid = 0;
    const TrackHeader* th = reinterpret_cast<const TrackHeader*>(blob + gh->track_off[tid]);
    w.on = true;
    w.hv.index = reinterpret_cast<const uint16_t*>(blob + th->index_off);
    w.hv.chunks = blob + th->chunks_off;
    w.hv.hc = th->hc; w.hv.vc = th->vc; w.hv.size_x = th->dsize_x; w.hv.size_y = th->dsize_y;
    return w;
}
__device__ __forceinline__ int status_word(const StepInfo& info, int prev) {
    return (info.iters & 0xFF) | (info.reset ? 0x100 : (prev & 0x100)) | ((info.ncon_wall & 0xFF) << 16) | ((info.ncon_wheel & 0xF) << 24) |
           ((info.ncon_ground > 7 ? 7 : info.ncon_ground) << 28) | (info.near_wall ? 0x400 : 0);
}

// Quad-per-car: four lanes (one per wheel chain) advance one car, 8 cars per warp; see mushr_step_quad.cuh.
// Shared memory: [slot][thread] for the lane-private slots, [slot][car] for the per-car slots, then the table of
// friction-loss row constants.  1 072 B per lane: one 216-thread CTA (54 cars) per SM.
template <int NT> constexpr size_t quad_smem_bytes() { return (size_t)(NT * QP_N + NT / 4 * QC_N + QK_N + 1) * sizeof(double); }

// ONE kernel serves both launches of the staged solve, with ONE inlined copy of the step:
//   resume = 0  the first launch: CTA b steps cars [54 b, 54 b + 54) of the (regrouped) fleet; a car that is not done after
//               max_rounds Newton rounds of its CTA is parked in its record (recs != NULL) and listed in list_out;
//   resume = 1  the continuation: a persistent grid (one CTA per SM) packs the cars listed in list_in, 54 at a time,
//               restores their solver state from the records and goes on (max_rounds <= 0: to convergence).
// Both paths run the same machine code for the solver, so a suspended and resumed car gets bit-identical results to one that
// converges in a single launch: with two kernels (two inlined copies) the compiler contracted a few multiply-adds
// differently and a 6,144-car fleet (staged) differed from its 2,048-car shards (unstaged) by 1e-15; with the step out of
// line (one shared function) the results were identical but the step took 2.50 ms instead of 1.3 (round 2 measurements).
template <int NT, bool LOCK>
__global__ void __launch_bounds__(NT, 1)
step_quad_kernel(const uint32_t* __restrict__ blob, double* __restrict__ qpos, double* __restrict__ qvel,
                 double* __restrict__ warm, const double* __restrict__ ctrl, const int32_t* __restrict__ track_id,
                 const int32_t* __restrict__ lap, const int32_t* __restrict__ perm, int64_t ncars, int nsteps,
                 int32_t* __restrict__ status, double* __restrict__ recs, const int32_t* __restrict__ list_in,
                 const int32_t* __restrict__ count_in, int32_t* __restrict__ list_out, int32_t* __restrict__ count_out,
                 int max_rounds, int options, const uint8_t* __restrict__ world_flag, int cpw, int resume) {
    const int tid = threadIdx.x, cib = tid >> 2;
    constexpr int KO = NT * QP_N + NT / 4 * QC_N, CARS = NT / 4;
    for (int g = tid; g < 25; g += NT) quad_const_entry(c_model, g, quad_sm + KO);
    __syncthreads();
    QuadDev<NT, NT / 4, LOCK> qd;
    qd.w = tid & 3; qd.po = tid; qd.co = NT * QP_N + cib; qd.ko = KO; qd.qs = tid & 28;
    const int64_t nwork = resume ? (int64_t)*count_in : ncars;
    for (int64_t base = (int64_t)blockIdx.x * CARS; base < nwork; base += (int64_t)gridDim.x * CARS) {
        const int64_t e = base + cib;
        bool live = e < nwork;
        int64_t car = live ? e : nwork - 1;             // padding quad: same collectives, no stores
        if (resume) car = list_in[car];
        else if (perm) car = perm[car];                 // cars grouped by their last Newton iteration count
        // a world whose cars touch each other this tick is one coupled problem: world_step_kernel advances it, not this kernel
        if (!resume && world_flag && world_flag[car / cpw]) live = false;
        const bool shadowed = !resume && lap && lap[car * FTGP_LAP_FIELDS + FTGP_LAP_FINISHED];
        const QHfWalls walls = track_walls(resume ? nullptr : blob, track_id, car, shadowed, options);   // (resume: the position stage is behind us)
        const QStage stage{(resume || recs) ? max_rounds : 0, resume != 0, recs ? recs + car * QREC_DOUBLES : nullptr};
        int st = 0;
        bool suspended = false;
        for (int s = 0; s < (resume ? 1 : nsteps) && !suspended; s++) {
            StepInfo info;
            suspended = step_car_quad(qd, c_model, qpos + car * NQ, qvel + car * NV, warm + car * NV, ctrl + 2 * car, walls, live, info, stage);
            if (!suspended) st = status_word(info, st);
        }
        if (live && qd.w == 0) {
            if (suspended) list_out[atomicAdd(count_out, 1)] = (int32_t)car;
            else if (status) status[car] = st;
        }
        if (!resume) break;                             // first launch: one batch per CTA
        __syncthreads();                                // the next batch reuses the shared-memory slots
    }
}

// The quad-per-car kernel runs the cars of a CTA in lock-step, so a CTA takes as many Newton rounds as its slowest
// car.  The iteration count is strongly correlated from one step to the next (measured: mean 2, max over 8 random
// cars 3.6), so cars are grouped by (last iteration count, in wall contact or not) with a counting sort.
constexpr int NBIN = 16;
// bit 10 of the status word: the car was within reach of a wall last step (the gate of quad_prepare).  Only such cars run the
// wall probes, and a warp runs them if ANY of its 8 cars does -- so the cars near walls are kept together.
__device__ __forceinline__ int order_bin(int st) { return min(st & 0xFF, 7) + ((st & 0x400) ? 8 : 0); }
// (cars of a world flagged as coupled sit in the last bin whatever their status word says: inside the fused tick their solver
// is already running beside these kernels and rewrites those words)
__device__ __forceinline__ int order_bin_of(const int32_t* __restrict__ status, const uint8_t* __restrict__ world_flag, int cpw, int64_t i) {
    if (world_flag && world_flag[i / cpw]) return NBIN - 1;
    return order_bin(status[i]);
}
__global__ void order_hist_kernel(const int32_t* __restrict__ status, const uint8_t* __restrict__ world_flag, int cpw, int64_t ncars,
                                  int32_t* __restrict__ hist) {
    __shared__ int h[NBIN];
    if (threadIdx.x < NBIN) h[threadIdx.x] = 0;
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < ncars) atomicAdd(&h[order_bin_of(status, world_flag, cpw, i)], 1);
    __syncthreads();
    if (threadIdx.x < NBIN && h[threadIdx.x]) atomicAdd(&hist[threadIdx.x], h[threadIdx.x]);
}
__global__ void order_scatter_kernel(const int32_t* __restrict__ status, const uint8_t* __restrict__ world_flag, int cpw, int64_t ncars,
                                     const int32_t* __restrict__ hist, int32_t* __restrict__ cursor, int32_t* __restrict__ perm) {
    __shared__ int h[NBIN], base[NBIN];
    if (threadIdx.x < NBIN) h[threadIdx.x] = 0;
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int bin = 0, rank = 0;
    if (i < ncars) { bin = order_bin_of(status, world_flag, cpw, i); rank = atomicAdd(&h[bin], 1); }
    __syncthreads();
    if (threadIdx.x < NBIN) {
        int start = 0;
        for (int b = 0; b < (int)threadIdx.x; b++) start += hist[b];
        base[threadIdx.x] = start + (h[threadIdx.x] ? atomicAdd(&cursor[threadIdx.x], h[threadIdx.x]) : 0);
    }
    __syncthreads();
    if (i < ncars) perm[base[bin] + rank] = (int32_t)i;
}
// one scratch per (device, stream): fleets stepped concurrently on different streams must not share it.  Every access
// (lookup, growth, the launches that use it) happens under g_step_mutex, so host threads never race on it; the launches
// themselves are asynchronous, so the lock is held for microseconds.  ftgp_release_scratch() frees a stream's scratch.
struct StepScratch {
    int dev = -1; cudaStream_t stream = nullptr; uint64_t used = 0;
    int32_t* perm = nullptr; int32_t* counters = nullptr; int64_t cap = 0;                                          // regrouping
    double* recs = nullptr; int32_t* lists = nullptr; int32_t* stage_counts = nullptr; int64_t stage_cap = 0;      // staged solve
    int32_t* world_list = nullptr; uint8_t* world_flag = nullptr; int64_t world_cap = 0;                                // coupled worlds
    void* world_spill = nullptr;                                                                                         // workspaces of warps 1.. of world_step_kernel
    double* qpos_snap = nullptr; int64_t snap_cap = 0;      // fused tick: the poses the rangefinders read while the coupled worlds already move
    bool world_inflight = false;                            // the coupled worlds of this step were started by launch_worlds_early
    cudaStream_t side = nullptr; cudaEvent_t ev_fork = nullptr, ev_join = nullptr;       // ... advanced beside the fast path
    cudaStream_t scan = nullptr; cudaEvent_t ev_scan_fork = nullptr, ev_scan_join = nullptr;    // fused tick: the rangefinders beside the step
    uint64_t generation = 0;     // bumped whenever a buffer is (re)allocated or freed: captured graphs hold these pointers
    void release() {
        if (dev < 0) return;
        int cur = 0;
        cudaGetDevice(&cur); cudaSetDevice(dev);
        if (perm) cudaFree(perm);
        if (counters) cudaFree(counters);
        if (recs) cudaFree(recs);
        if (lists) cudaFree(lists);
        if (stage_counts) cudaFree(stage_counts);
        if (world_list) cudaFree(world_list);
        if (side) cudaStreamDestroy(side);
        if (ev_fork) cudaEventDestroy(ev_fork);
        if (ev_join) cudaEventDestroy(ev_join);
        if (scan) cudaStreamDestroy(scan);
        if (ev_scan_fork) cudaEventDestroy(ev_scan_fork);
        if (ev_scan_join) cudaEventDestroy(ev_scan_join);
        if (world_flag) cudaFree(world_flag);
        if (world_spill) cudaFree(world_spill);
        if (qpos_snap) cudaFree(qpos_snap);
        cudaSetDevice(cur);
        const uint64_t gen = generation + 1;
        *this = StepScratch();
        generation = gen;
    }
};
static StepScratch g_scratch[64];
static std::mutex g_step_mutex;
static uint64_t g_scratch_clock = 0;
static int g_sm_count[16] = {0};
static bool g_attr_ready[16] = {false};

static StepScratch* step_scratch(int dev, cudaStream_t stream) {       // caller holds g_step_mutex
    StepScratch* lru = &g_scratch[0];
    for (auto& o : g_scratch) {
        if (o.dev == dev && o.stream == stream) { o.used = ++g_scratch_clock; return &o; }
        if (o.used < lru->used) lru = &o;
    }
    lru->release();              // not found: a free slot, else the least recently used one (cudaFree waits for its work)
    lru->dev = dev; lru->stream = stream; lru->used = ++g_scratch_clock;
    return lru;
}

// ---- worlds of 2..8 cars (BASELINE config 5): cars that touch each other are ONE constraint problem (mushr_world.cuh).
// world_flag_kernel finds the worlds with a car-car contact this tick (a thread per world, poses only); the quad kernel
// skips their cars; world_step_kernel advances them, one warp per flagged world, lane c = car c.  The world's workspace (206 KB:
// per car the block-arrow M and H, rows, solver vectors; the car-car rows, the Woodbury columns, the small dense system) lives
// in SHARED memory, one world per SM at a time: with the workspace in global memory every access paid the L2 latency and a
// coupled world took 6 ms (measured: 32,768 cars in 8-car worlds, 32 of them coupled, 7.6 ms per tick against 1.6).
__global__ void world_flag_kernel(const double* __restrict__ qpos, const int32_t* __restrict__ lap, int64_t nworlds, int cpw,
                                  uint8_t* __restrict__ flag, int32_t* __restrict__ list, int32_t* __restrict__ count) {
    const int64_t wld = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (wld >= nworlds) return;
    const double* q[WMAXCARS]; bool sh[WMAXCARS];
    for (int c = 0; c < cpw; c++) {
        const int64_t car = wld * cpw + c;
        q[c] = qpos + car * NQ;
        sh[c] = lap && lap[car * FTGP_LAP_FIELDS + FTGP_LAP_FINISHED];
    }
    const bool hit = world_has_contact(cpw, q, sh);
    flag[wld] = hit ? 1 : 0;
    if (hit) list[atomicAdd(count, 1)] = (int32_t)wld;
}

struct WarpComm {                                   // one warp per world: lane c = car c (lanes >= cars idle along)
    int lane, nlanes;
    __device__ __forceinline__ void sync() const { __syncwarp(); }
};

// WORLD_WARPS warps per CTA, one world each: warp 0 works in the CTA's shared memory, further warps would work in a workspace
// in global memory.  Measured with 4 (256 coupled worlds among 32,768 cars): 6.57 ms per tick against 4.57 with one warp
// per SM in two waves -- a world whose workspace is served by L2 takes three times as long, so the shipped value is 1.
constexpr int WORLD_WARPS = 1;
extern __shared__ __align__(16) unsigned char world_sm[];
__global__ void __launch_bounds__(128)      // (a bound of 32 makes ptxas settle on 168 registers and 2.5 KB of spills; with 128 it takes 255 and spills 0.6 KB)
world_step_kernel(const uint32_t* __restrict__ blob, double* __restrict__ qpos, double* __restrict__ qvel, double* __restrict__ warm,
                  const double* __restrict__ ctrl, const int32_t* __restrict__ track_id, const int32_t* __restrict__ lap, int cpw,
                  int32_t* __restrict__ status, const int32_t* __restrict__ list, const int32_t* __restrict__ count, int options,
                  WorldWork* __restrict__ spill) {
    const int n = *count;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if ((int)blockIdx.x * WORLD_WARPS + warp >= n) return;
    WorldWork& W = (WORLD_WARPS == 1 || warp == 0) ? *reinterpret_cast<WorldWork*>(world_sm)
                                                   : spill[(size_t)blockIdx.x * (WORLD_WARPS - 1) + warp - 1];
    WarpComm cm{lane, 32};
    Kin kin;                                        // this lane's position-stage scratch (local memory)
    for (int e = blockIdx.x * WORLD_WARPS + warp; e < n; e += gridDim.x * WORLD_WARPS) {
        const int64_t wld = list[e];
        double *q[WMAXCARS], *v[WMAXCARS], *wm[WMAXCARS]; const double* u[WMAXCARS];
        QHfWalls walls[WMAXCARS]; bool sh[WMAXCARS];
        for (int c = 0; c < cpw; c++) {
            const int64_t car = wld * cpw + c;
            q[c] = qpos + car * NQ; v[c] = qvel + car * NV; wm[c] = warm + car * NV; u[c] = ctrl + 2 * car;
            sh[c] = lap && lap[car * FTGP_LAP_FIELDS + FTGP_LAP_FINISHED];
            walls[c] = track_walls(blob, track_id, car, sh[c], options);
        }
        WorldInfo wi;
        world_step(cm, c_model, cpw, q, v, wm, u, walls, sh, W, kin, wi);
        if (status && lane < cpw) {
            const CarWork& C = W.car[lane];
            StepInfo si; si.iters = wi.iters; si.reset = wi.reset; si.ncon_wheel = C.nwheel; si.ncon_wall = C.nwall; si.ncon_ground = C.nground; si.near_wall = C.nwall > 0;
            status[wld * cpw + lane] = status_word(si, 0) | 0x200;       // bit 9: advanced by the coupled world solver
        }
        __syncwarp();
    }
}

// The production mapping is frozen: 216-thread CTAs (54 cars, 6 warps + 24 lanes), CTA-level lock-step of the Newton
// loop, cars regrouped by (last Newton iteration count, wall contact), staged solve with two Newton rounds in the first
// launch (DESIGN.md 8 lists the measured alternatives; the A/B variants live in tests/host_harness, not in this library).
// NOTE on the 24-lane tail warp: QuadDev's collectives use the full mask; lanes 24-31 of that warp do not exist (they
// count as exited threads, which *_sync primitives ignore), and every quad is 4 lanes inside one warp.
// (tools/build_variant.py compiles A/B variants of these three into separately named libraries for tools/step_ab.py;
// the shipped library always has the defaults)
#ifndef FTGP_AB_LOCK
#define FTGP_AB_LOCK true
#endif
#ifndef FTGP_AB_ROUNDS
#define FTGP_AB_ROUNDS 2
#endif
constexpr int STEP_NT = 216;
constexpr int STAGE_ROUNDS = FTGP_AB_ROUNDS;
constexpr bool STEP_LOCK = FTGP_AB_LOCK;
constexpr int64_t ORDER_MIN_CARS = 1024, STAGE_MIN_CARS = 4096;

static_assert(sizeof(WorldWork) <= 227 * 1024, "the coupled world's workspace must fit one SM's shared memory");

static int step_device_ready(int dev) {             // caller holds g_step_mutex; once per device, not per launch
    int rc = ensure_model(dev); if (rc) return rc;
    if (!g_attr_ready[dev]) {
        constexpr size_t smem = quad_smem_bytes<STEP_NT>();
        FTGP_CUDA(cudaDeviceGetAttribute(&g_sm_count[dev], cudaDevAttrMultiProcessorCount, dev));
        FTGP_CUDA(cudaFuncSetAttribute(step_quad_kernel<STEP_NT, STEP_LOCK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        FTGP_CUDA(cudaFuncSetAttribute(step_quad_kernel<STEP_NT, STEP_LOCK>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        FTGP_CUDA(cudaFuncSetAttribute(world_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(WorldWork)));
        g_attr_ready[dev] = true;
    }
    return FTGP_OK;
}

// worlds of several cars: list the worlds whose cars touch (they leave the fast path) ...
static int world_flag_launch(StepScratch* o, int dev, const double* qpos, const int32_t* lap, int64_t nworlds, int cpw, cudaStream_t stream) {
    if (o->world_cap < nworlds) {
        if (o->world_list) cudaFree(o->world_list);
        if (o->world_flag) cudaFree(o->world_flag);
        o->world_list = nullptr; o->world_flag = nullptr; o->world_cap = 0; o->generation++;
        FTGP_CUDA(cudaMalloc(&o->world_list, (size_t)(nworlds + 1) * sizeof(int32_t)));
        FTGP_CUDA(cudaMalloc(&o->world_flag, (size_t)nworlds));
        o->world_cap = nworlds;
        if (WORLD_WARPS > 1 && !o->world_spill) FTGP_CUDA(cudaMalloc(&o->world_spill, (size_t)g_sm_count[dev] * (WORLD_WARPS - 1) * sizeof(WorldWork)));
        if (!o->side) {
            FTGP_CUDA(cudaStreamCreateWithFlags(&o->side, cudaStreamNonBlocking));
            FTGP_CUDA(cudaEventCreateWithFlags(&o->ev_fork, cudaEventDisableTiming));
            FTGP_CUDA(cudaEventCreateWithFlags(&o->ev_join, cudaEventDisableTiming));
        }
    }
    FTGP_CUDA(cudaMemsetAsync(o->world_list + nworlds, 0, sizeof(int32_t), stream));        // the counter sits behind the list
    world_flag_kernel<<<(unsigned)((nworlds + 127) / 128), 128, 0, stream>>>(qpos, lap, nworlds, cpw, o->world_flag, o->world_list,
                                                                           o->world_list + nworlds);
    count_launch();
    return FTGP_OK;
}
// ... and advance them on a side stream: one warp and 183 KB of shared memory per listed world, launched before the fast
// path's kernel so that its blocks take their SMs first; the two kernels touch disjoint cars, and a coupled world is a
// millisecond-long dependent chain that would otherwise be added to the tick.  The caller joins on ev_join.
static int world_fork_launch(StepScratch* o, int dev, const uint32_t* blob, double* qpos, double* qvel, double* warm, const double* ctrl,
                             const int32_t* track_id, const int32_t* lap, int64_t nworlds, int cpw, int32_t* status, int options,
                             cudaStream_t stream) {
    FTGP_CUDA(cudaEventRecord(o->ev_fork, stream));
    FTGP_CUDA(cudaStreamWaitEvent(o->side, o->ev_fork, 0));
    const int slots = (int)std::min<int64_t>((nworlds + WORLD_WARPS - 1) / WORLD_WARPS, g_sm_count[dev]);
    world_step_kernel<<<slots, 32 * WORLD_WARPS, sizeof(WorldWork), o->side>>>(blob, qpos, qvel, warm, ctrl, track_id, lap, cpw, status,
                                                                               o->world_list, o->world_list + nworlds, options,
                                                                               static_cast<WorldWork*>(o->world_spill));
    count_launch();
    FTGP_CUDA(cudaEventRecord(o->ev_join, o->side));
    return FTGP_OK;
}

// Fused tick, worlds of several cars: the coupled worlds are listed and their solver is started BEFORE the rangefinder
// kernel, which then reads a copy of the poses taken here (mj_step evaluates the rangefinders from the pre-step pose,
// custom.py:1425) while the solver already moves its cars.  launch_step() of the same tick finds the worlds in flight, runs
// only the fast path and joins.  *lidar_qpos receives the copy (row stride FTGP_NQ).
int launch_worlds_early(const ftgp_geom* g, double* qpos, double* qvel, double* warm, const double* ctrl, const int32_t* track_id,
                        const int32_t* lap, int64_t ncars, int cpw, int32_t* status, int options, cudaStream_t stream,
                        const double** lidar_qpos) {
    if (cpw < 2 || cpw > WMAXCARS || ncars % cpw) { set_error("ftgp_tick: cars_per_world must be 1..8 and divide ncars"); return FTGP_ERR_ARG; }
    int dev = 0;
    FTGP_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 16) { set_error("ftgp_tick: device index %d not supported", dev); return FTGP_ERR_UNSUPPORTED; }
    std::lock_guard<std::mutex> lock(g_step_mutex);
    int rc = step_device_ready(dev); if (rc) return rc;
    StepScratch* o = step_scratch(dev, stream);
    const int64_t nworlds = ncars / cpw;
    if (o->world_inflight) {                        // (a tick that failed between the fork and its step: join before starting over)
        o->world_inflight = false;
        FTGP_CUDA(cudaStreamWaitEvent(stream, o->ev_join, 0));
    }
    if ((rc = world_flag_launch(o, dev, qpos, lap, nworlds, cpw, stream))) return rc;
    if (o->snap_cap < ncars) {
        if (o->qpos_snap) cudaFree(o->qpos_snap);
        o->qpos_snap = nullptr; o->snap_cap = 0; o->generation++;
        FTGP_CUDA(cudaMalloc(&o->qpos_snap, (size_t)ncars * NQ * sizeof(double)));
        o->snap_cap = ncars;
    }
    FTGP_CUDA(cudaMemcpyAsync(o->qpos_snap, qpos, (size_t)ncars * NQ * sizeof(double), cudaMemcpyDeviceToDevice, stream));
    if ((rc = world_fork_launch(o, dev, g ? g->d_blob : nullptr, qpos, qvel, warm, ctrl, track_id, lap, nworlds, cpw, status, options, stream))) return rc;
    o->world_inflight = true;
    *lidar_qpos = o->qpos_snap;
    return FTGP_OK;
}

int launch_step(const ftgp_geom* g, double* qpos, double* qvel, double* warm, const double* ctrl,
                const int32_t* track_id, const int32_t* lap, int64_t ncars, int cpw, int nsteps, int32_t* status,
                int options, cudaStream_t stream) {
    if (cpw < 1 || cpw > WMAXCARS || ncars % cpw) { set_error("ftgp_step: cars_per_world must be 1..8 and divide ncars"); return FTGP_ERR_ARG; }
    if (cpw > 1 && nsteps != 1) { set_error("ftgp_step: worlds of several cars are stepped one step per call"); return FTGP_ERR_UNSUPPORTED; }
    int dev = 0;
    FTGP_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 16) { set_error("ftgp_step: device index %d not supported", dev); return FTGP_ERR_UNSUPPORTED; }
    std::lock_guard<std::mutex> lock(g_step_mutex);
    int rc = step_device_ready(dev); if (rc) return rc;
    constexpr size_t smem = quad_smem_bytes<STEP_NT>();
    const uint32_t* blob = g ? g->d_blob : nullptr;
    const bool big = ncars < (int64_t)1 << 31;
    const bool reorder = status && big && ncars >= ORDER_MIN_CARS;
    const bool staged = nsteps == 1 && big && ncars >= STAGE_MIN_CARS;
    StepScratch* o = (reorder || staged || cpw > 1) ? step_scratch(dev, stream) : nullptr;
    const int64_t nworlds = ncars / cpw;
    const bool fork_here = cpw > 1 && !o->world_inflight;          // (inside the fused tick the worlds are in flight already)
    if (fork_here && (rc = world_flag_launch(o, dev, qpos, lap, nworlds, cpw, stream))) return rc;
    // cars grouped by (last Newton iteration count, wall contact) for the kernel that runs 54 cars in lock-step
    const int32_t* perm = nullptr;
    if (reorder) {
        if (o->cap < ncars) {
            if (o->perm) cudaFree(o->perm);
            o->perm = nullptr; o->cap = 0;
            if (!o->counters) FTGP_CUDA(cudaMalloc(&o->counters, 2 * NBIN * sizeof(int32_t)));
            FTGP_CUDA(cudaMalloc(&o->perm, ncars * sizeof(int32_t)));
            o->cap = ncars; o->generation++;
        }
        FTGP_CUDA(cudaMemsetAsync(o->counters, 0, 2 * NBIN * sizeof(int32_t), stream));
        const unsigned nb = (unsigned)((ncars + 255) / 256);
        const uint8_t* wf = cpw > 1 ? o->world_flag : nullptr;
        order_hist_kernel<<<nb, 256, 0, stream>>>(status, wf, cpw, ncars, o->counters);
        order_scatter_kernel<<<nb, 256, 0, stream>>>(status, wf, cpw, ncars, o->counters, o->counters + NBIN, o->perm);
        count_launch(2);
        perm = o->perm;
    }
    // Staged solve (one step of a big fleet): STAGE_ROUNDS Newton rounds in the first launch, then the cars that are not
    // done are packed into fresh CTAs by the persistent continuation kernel.  Measured at 65,536 cars: 1.39 ms unstaged,
    // 1.31 ms staged.  If the records cannot be allocated the step runs unstaged.
    double* recs = nullptr; int32_t* lists = nullptr; int32_t* counts = nullptr;
    if (staged) {
        if (o->stage_cap < ncars) {
            if (o->recs) cudaFree(o->recs);
            if (o->lists) cudaFree(o->lists);
            o->recs = nullptr; o->lists = nullptr; o->stage_cap = 0; o->generation++;
            if (!o->stage_counts) FTGP_CUDA(cudaMalloc(&o->stage_counts, 4 * sizeof(int32_t)));
            if (cudaMalloc(&o->recs, (size_t)ncars * QREC_DOUBLES * sizeof(double)) == cudaSuccess &&
                cudaMalloc(&o->lists, (size_t)ncars * 2 * sizeof(int32_t)) == cudaSuccess) o->stage_cap = ncars;
            else {
                cudaGetLastError();
                if (o->recs) cudaFree(o->recs);
                o->recs = nullptr; o->lists = nullptr;
            }
        }
        if (o->stage_cap >= ncars) {
            recs = o->recs; lists = o->lists; counts = o->stage_counts;
            FTGP_CUDA(cudaMemsetAsync(counts, 0, 4 * sizeof(int32_t), stream));
        }
    }
    if (fork_here && (rc = world_fork_launch(o, dev, blob, qpos, qvel, warm, ctrl, track_id, lap, nworlds, cpw, status, options, stream))) return rc;
    constexpr int CARS = STEP_NT / 4;
    step_quad_kernel<STEP_NT, STEP_LOCK><<<(unsigned)((ncars + CARS - 1) / CARS), STEP_NT, smem, stream>>>(
        blob, qpos, qvel, warm, ctrl, track_id, lap, perm, ncars, nsteps, status, recs, nullptr, nullptr, lists, counts, STAGE_ROUNDS,
        options, cpw > 1 ? o->world_flag : nullptr, cpw, 0);
    count_launch();
    if (recs) {                                     // continuation: the same kernel, persistent grid over the suspended cars
        step_quad_kernel<STEP_NT, STEP_LOCK><<<g_sm_count[dev], STEP_NT, smem, stream>>>(
            nullptr, qpos, qvel, warm, ctrl, track_id, nullptr, nullptr, ncars, 1, status, recs, lists, counts, lists + ncars, counts + 1, 0,
            options, nullptr, cpw, 1);
        count_launch();
    }
    if (cpw > 1) {                                  // join: the coupled worlds are done as well
        o->world_inflight = false;
        FTGP_CUDA(cudaStreamWaitEvent(stream, o->ev_join, 0));
    }
    FTGP_CUDA(cudaGetLastError());
    return FTGP_OK;
}

int launch_lidar(const ftgp_geom* g, const double* qpos, int64_t stride, const int32_t* track_id,
                 const uint8_t* visible, const int32_t* lap, int64_t ncars, int cpw, float* ranges, float* min_range,
                 cudaStream_t stream);
int launch_drivers(const float* ranges, const int32_t* kind, int default_kind, const double* params, const int32_t* lap,
                   double* ctrl, int64_t ncars, cudaStream_t stream, int32_t* steps_dev);
int launch_lap(const ftgp_geom* g, const double* qpos, int64_t stride, const int32_t* track_id, int32_t* lap,
               int32_t* times, int32_t* winners, const int32_t* status, int64_t ncars, int cpw, int32_t steps,
               int32_t lap_target, cudaStream_t stream, const int32_t* steps_dev);

int launch_flatten(double* qpos, int64_t stride, int64_t ncars, cudaStream_t stream);
int launch_reload(const ftgp_tick_args* a, const ftgp_reload_args* r, int32_t steps, cudaStream_t stream,
                  const int32_t* steps_dev);

// Inside the fused tick the rangefinder kernel runs on a side stream against a copy of the poses (mj_step
// evaluates the rangefinders from the pre-step pose, custom.py:1425) while the vehicle step advances the state on the main
// stream.  The two kernels cannot share an SM (227 KB + 80 KB of shared memory), so on a full GPU all there is to win are
// the tails of each other's waves (65,536 cars: 2.97 -> 2.90 ms per tick); small fleets fill the GPU with neither kernel and
// win more (256 cars 0.35 -> 0.28 ms, 1,024 cars 0.52 -> 0.45, 4,096 cars 0.71 -> 0.66, 16,384 cars 1.21 -> 1.13).  Results
// are bit-identical to the serial order (tools/tick_ab.py; tests/test_gpu_step.py, graph-replayed and eager).
static int overlap_fork(double* qpos, int64_t ncars, bool copy, cudaStream_t stream, const double** snap, cudaStream_t* side, cudaEvent_t* join) {
    int dev = 0;
    FTGP_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_step_mutex);
    StepScratch* o = step_scratch(dev, stream);
    if (!o->scan) {
        FTGP_CUDA(cudaStreamCreateWithFlags(&o->scan, cudaStreamNonBlocking));
        FTGP_CUDA(cudaEventCreateWithFlags(&o->ev_scan_fork, cudaEventDisableTiming));
        FTGP_CUDA(cudaEventCreateWithFlags(&o->ev_scan_join, cudaEventDisableTiming));
    }
    if (copy) {                                     // (worlds of several cars: launch_worlds_early has taken the copy already)
        if (o->snap_cap < ncars) {
            if (o->qpos_snap) cudaFree(o->qpos_snap);
            o->qpos_snap = nullptr; o->snap_cap = 0; o->generation++;
            FTGP_CUDA(cudaMalloc(&o->qpos_snap, (size_t)ncars * NQ * sizeof(double)));
            o->snap_cap = ncars;
        }
        FTGP_CUDA(cudaMemcpyAsync(o->qpos_snap, qpos, (size_t)ncars * NQ * sizeof(double), cudaMemcpyDeviceToDevice, stream));
    }
    FTGP_CUDA(cudaEventRecord(o->ev_scan_fork, stream));
    FTGP_CUDA(cudaStreamWaitEvent(o->scan, o->ev_scan_fork, 0));
    *snap = o->qpos_snap; *side = o->scan; *join = o->ev_scan_join;
    return FTGP_OK;
}

// ---- one tick = custom.py:1337-1426 for the whole fleet, in the reference's order; r != NULL: the worlds whose race is
// over are reloaded first (custom.py:1089-1128); dp != NULL: the drivers read the per-car rows (ftgp_drivers_params)
static int issue_tick(const ftgp_tick_args* a, const ftgp_reload_args* r, const double* dp, int32_t steps, int32_t* steps_dev,
                      cudaStream_t s) {
    int rc;
    if (r && (rc = launch_reload(a, r, steps, s, steps_dev))) return rc;
    // custom.py:1338-1339 option naive_flatten
    if ((a->options & FTGP_OPT_NAIVE_FLATTEN) && (rc = launch_flatten(a->qpos, FTGP_NQ, a->ncars, s))) return rc;
    // custom.py:1340-1372 progress + lap logic from the current pose
    if ((rc = launch_lap(a->geom, a->qpos, FTGP_NQ, a->track_id, a->lap, a->times, a->winners, a->status, a->ncars,
                         a->cars_per_world, steps, a->lap_target, s, steps_dev))) return rc;
    // custom.py:1395-1423 driver on the ranges of the previous mj_step, control write
    if ((rc = launch_drivers(a->ranges, a->driver_kind, a->default_driver, dp, a->lap, a->ctrl, a->ncars, s, steps_dev))) return rc;
    // custom.py:1425 mj_step: rangefinders are evaluated from the pre-step pose, then the state advances.  The rangefinder
    // kernel scans a copy of the poses on a stream of its own beside the step; in worlds of several cars the coupled worlds'
    // solver starts here as well, on a third stream (launch_worlds_early takes the copy in that case).
    const double* snap = nullptr; cudaStream_t scan; cudaEvent_t join;
    if (a->cars_per_world > 1 && (rc = launch_worlds_early(a->geom, a->qpos, a->qvel, a->warm, a->ctrl, a->track_id, a->lap, a->ncars,
                                                           a->cars_per_world, a->status, a->options, s, &snap))) return rc;
    if ((rc = overlap_fork(a->qpos, a->ncars, a->cars_per_world == 1, s, &snap, &scan, &join))) return rc;
    if ((rc = launch_lidar(a->geom, snap, FTGP_NQ, a->track_id, nullptr, a->lap, a->ncars, a->cars_per_world, a->ranges, nullptr, scan))) return rc;
    FTGP_CUDA(cudaEventRecord(join, scan));
    rc = launch_step(a->geom, a->qpos, a->qvel, a->warm, a->ctrl, a->track_id, a->lap, a->ncars, a->cars_per_world, 1, a->status, a->options, s);
    FTGP_CUDA(cudaStreamWaitEvent(s, join, 0));           // (also after a failed step: the side stream must rejoin a capture)
    return rc;
}

// ---- small fleets: the tick is launch-bound (4-9 launches of a few microseconds of work each), so it is captured once
// into a CUDA graph per (arguments, stream) and replayed.  The only per-tick value, self.steps, lives in a device counter
// that the lap kernel reads and the driver kernel bumps.  The first tick of a new argument set runs eagerly (it may
// allocate scratch, which a capture must not); graphs are rebuilt when the step scratch they point into is re-allocated.
constexpr int64_t GRAPH_MAX_CARS = 16384;
static std::atomic<int> g_use_graphs{1};
struct TickGraph {
    ftgp_tick_args key{}; bool reload = false; ftgp_reload_args rkey{}; const double* params = nullptr;
    cudaStream_t stream = nullptr; int dev = -1;
    cudaGraphExec_t exec = nullptr; int32_t* steps_dev = nullptr; int32_t shadow = INT32_MIN;
    uint64_t scratch_gen = 0; int launches_per_tick = 0; bool seen = false; uint64_t used = 0;
};
static TickGraph g_graphs[32];
static std::mutex g_graph_mutex;
static uint64_t g_graph_clock = 0;
__global__ void set_i32_kernel(int32_t* p, int32_t v) { *p = v; }

static uint64_t scratch_generation(int dev, cudaStream_t stream) {
    std::lock_guard<std::mutex> lock(g_step_mutex);
    for (auto& o : g_scratch) if (o.dev == dev && o.stream == stream) return o.generation;
    return 0;
}
static bool same_key(const ftgp_tick_args& x, const ftgp_tick_args& y) {
    return x.geom == y.geom && x.qpos == y.qpos && x.qvel == y.qvel && x.warm == y.warm && x.ctrl == y.ctrl && x.ranges == y.ranges &&
           x.track_id == y.track_id && x.driver_kind == y.driver_kind && x.lap == y.lap && x.times == y.times &&
           x.winners == y.winners && x.status == y.status && x.ncars == y.ncars && x.cars_per_world == y.cars_per_world &&
           x.default_driver == y.default_driver && x.lap_target == y.lap_target && x.options == y.options;
}
static bool same_reload(const TickGraph& g, const ftgp_reload_args* r) {
    if (!r) return !g.reload;
    const ftgp_reload_args& x = g.rkey;
    return g.reload && x.start_xy == r->start_xy && x.start_yaw == r->start_yaw && x.start_offset == r->start_offset &&
           x.race_start == r->race_start && x.tally == r->tally && x.race_ticks == r->race_ticks;
}
static void drop_graph(TickGraph& g) {
    if (g.exec) cudaGraphExecDestroy(g.exec);
    if (g.steps_dev) cudaFree(g.steps_dev);
    g = TickGraph();
}

// returns FTGP_OK and sets *done = number of ticks issued through the graph (0: caller runs them eagerly)
static int graph_ticks(const ftgp_tick_args* a, const ftgp_reload_args* r, const double* dp, int nticks, cudaStream_t s,
                       int* done) {
    *done = 0;
    int dev = 0;
    FTGP_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_graph_mutex);
    TickGraph* e = nullptr; TickGraph* lru = &g_graphs[0];
    for (auto& g : g_graphs) {
        if (g.seen && g.dev == dev && g.stream == s && same_key(g.key, *a) && same_reload(g, r) &&
            g.params == dp) { e = &g; break; }
        if (g.used < lru->used) lru = &g;
    }
    int32_t steps = a->steps;
    if (!e) {                                   // first tick with these arguments: register, run ONE tick eagerly
        drop_graph(*lru);
        lru->key = *a; lru->stream = s; lru->dev = dev; lru->seen = true;
        lru->reload = r != nullptr;
        if (r) lru->rkey = *r;
        lru->params = dp;
        e = lru;
        const int rc = issue_tick(a, r, dp, steps, nullptr, s);
        if (rc) return rc;
        steps++; nticks--; *done = 1;
        if (nticks == 0) { e->used = ++g_graph_clock; return FTGP_OK; }
    }
    e->used = ++g_graph_clock;
    const uint64_t gen = scratch_generation(dev, s);
    if (e->exec && e->scratch_gen != gen) { cudaGraphExecDestroy(e->exec); e->exec = nullptr; }
    if (!e->exec) {
        if (!e->steps_dev) FTGP_CUDA(cudaMalloc(&e->steps_dev, sizeof(int32_t)));
        const int64_t l0 = ftgp_launch_count();
        cudaGraph_t graph = nullptr;
        FTGP_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
        const int rc = issue_tick(a, r, dp, 0, e->steps_dev, s);
        const cudaError_t ce = cudaStreamEndCapture(s, &graph);
        if (rc || ce != cudaSuccess || !graph) {                 // capture refused (e.g. scratch had to grow): stay eager
            if (graph) cudaGraphDestroy(graph);
            cudaGetLastError();
            count_launch((int)(l0 - ftgp_launch_count()));
            return FTGP_OK;
        }
        e->launches_per_tick = (int)(ftgp_launch_count() - l0);
        count_launch(-e->launches_per_tick);                     // nothing ran during the capture
        const cudaError_t ie = cudaGraphInstantiate(&e->exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) { e->exec = nullptr; cudaGetLastError(); return FTGP_OK; }
        e->scratch_gen = scratch_generation(dev, s);
        if (e->scratch_gen != gen) { cudaGraphExecDestroy(e->exec); e->exec = nullptr; return FTGP_OK; }
        e->shadow = INT32_MIN;
    }
    if (e->shadow != steps) { set_i32_kernel<<<1, 1, 0, s>>>(e->steps_dev, steps); count_launch(); }
    for (int t = 0; t < nticks; t++) FTGP_CUDA(cudaGraphLaunch(e->exec, s));
    count_launch(nticks * e->launches_per_tick);
    e->shadow = steps + nticks;
    *done += nticks;
    return FTGP_OK;
}

}  // namespace ftgp
using namespace ftgp;

extern "C" int ftgp_step(const ftgp_geom* g, double* qpos, double* qvel, double* warm, const double* ctrl,
                         const int32_t* track_id, const int32_t* lap, int64_t ncars, int cars_per_world, int nsteps,
                         int32_t* status, int options, void* stream) {
    if (!qpos || !qvel || !warm || !ctrl || ncars < 0 || nsteps < 0) { set_error("ftgp_step: bad argument"); return FTGP_ERR_ARG; }
    if (ncars == 0 || nsteps == 0) return FTGP_OK;
    if (g) FTGP_CUDA(cudaSetDevice(g->device));
    return launch_step(g, qpos, qvel, warm, ctrl, track_id, lap, ncars, cars_per_world, nsteps, status, options, (cudaStream_t)stream);
}

extern "C" int ftgp_release_scratch(void* stream) {
    int dev = 0;
    FTGP_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_step_mutex);
    for (auto& o : g_scratch) if (o.dev == dev && o.stream == (cudaStream_t)stream) o.release();
    return FTGP_OK;
}

static bool bad_tick_args(const ftgp_tick_args* a) {
    return !a || !a->geom || !a->qpos || !a->qvel || !a->warm || !a->ctrl || !a->ranges || !a->lap || !a->times ||
           a->ncars < 0 || a->cars_per_world < 1;
}
// checked before any CUDA call: the race cap and the tally both need race_start
static bool bad_reload_args(const ftgp_reload_args* r) {
    return !r || !r->start_xy || !r->start_yaw || !r->start_offset || r->race_ticks < 0 ||
           (r->tally && !r->race_start) || (r->race_ticks > 0 && !r->race_start);
}

extern "C" int ftgp_tick_params(const ftgp_tick_args* a, const ftgp_reload_args* r, const double* driver_params, int nticks,
                                void* stream) {
    if (bad_tick_args(a) || nticks < 0) { set_error("ftgp_tick: bad argument"); return FTGP_ERR_ARG; }
    if (r && bad_reload_args(r)) { set_error("ftgp_tick_reload: bad reload argument"); return FTGP_ERR_ARG; }
    if (a->ncars == 0 || nticks == 0) return FTGP_OK;
    FTGP_CUDA(cudaSetDevice(a->geom->device));
    cudaStream_t s = (cudaStream_t)stream;
    int t0 = 0, rc;
    if (a->ncars <= GRAPH_MAX_CARS && s != nullptr && g_use_graphs.load()) {           // (the legacy default stream cannot be captured)
        if ((rc = graph_ticks(a, r, driver_params, nticks, s, &t0))) return rc;
    }
    for (int t = t0; t < nticks; t++)
        if ((rc = issue_tick(a, r, driver_params, a->steps + t, nullptr, s))) return rc;
    return FTGP_OK;
}

extern "C" int ftgp_tick_reload(const ftgp_tick_args* a, const ftgp_reload_args* r, int nticks, void* stream) {
    return ftgp_tick_params(a, r, nullptr, nticks, stream);
}

extern "C" int ftgp_tick(const ftgp_tick_args* a, int nticks, void* stream) { return ftgp_tick_reload(a, nullptr, nticks, stream); }

extern "C" int ftgp_reload(const ftgp_tick_args* a, const ftgp_reload_args* r, void* stream) {
    if (bad_tick_args(a) || bad_reload_args(r)) { set_error("ftgp_reload: bad argument"); return FTGP_ERR_ARG; }
    if (a->ncars == 0) return FTGP_OK;
    FTGP_CUDA(cudaSetDevice(a->geom->device));
    return launch_reload(a, r, a->steps, (cudaStream_t)stream, nullptr);
}

extern "C" int ftgp_tick_use_graphs(int enable) { return g_use_graphs.exchange(enable ? 1 : 0); }

extern "C" int ftgp_release_graphs(void) {
    std::lock_guard<std::mutex> lock(g_graph_mutex);
    for (auto& g : g_graphs) drop_graph(g);
    return FTGP_OK;
}

namespace ftgp {
void forget_geom(const ftgp_geom* geom) {       // ftgp_geom_destroy: captured ticks point into the geometry blob
    std::lock_guard<std::mutex> lock(g_graph_mutex);
    for (auto& g : g_graphs) if (g.seen && g.key.geom == geom) drop_graph(g);
}
}
