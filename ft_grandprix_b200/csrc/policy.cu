// policy.cu -- neural-network drivers: the cars of kind FTGP_DRIVER_POLICY run one MLP of a bank (include/ftgp.h,
// ftgp_drivers_policy), fp32 on the SIMT pipes, after drivers_kernel (which skips them) and before the step.
//
//   policy_count_kernel    histogram of the POLICY cars' ids; out-of-range ids write (0, 0) here
//   policy_scan_kernel     exclusive prefix sum of the histogram (one CTA)
//   policy_scatter_kernel  the car ids, grouped by policy id (a counting sort into per-stream scratch)
//   policy_kernel          a CTA takes TILE consecutive cars of the grouped list; for each run of one policy in it, the
//                          policy's 42 KB are staged into shared memory once and the run's cars are evaluated as
//                          register-tiled products (4 cars x 4 units per thread)
//
// Neighbouring cars need not share a policy (8-car worlds race 8 variants), so the grouping is what lets a CTA stage
// one policy for many cars.  The order of cars inside a bucket depends on atomics, and correctness never depends on it:
// every pre-activation of a car is the same chain of fmaf in input order, starting from the bias, whichever tile, slot
// or thread evaluates it, so a car's output does not depend on the other cars of its tile.
#include <math.h>
#include "common.h"

namespace ftgp {

constexpr int NIN = FTGP_POLICY_NIN, HID = FTGP_POLICY_HIDDEN, PF = FTGP_POLICY_FLOATS;
constexpr int TILE = 64;               // cars per CTA
constexpr int LD = TILE + 4;           // row pitch of the activations in shared memory (16-byte rows, fewer bank conflicts)
constexpr int NT = 256;                // threads: 16 car groups x 16 unit groups, 4 x 4 outputs each
constexpr size_t POLICY_SMEM = (size_t)(PF + NIN * LD + 2 * HID * LD) * sizeof(float) + TILE * (2 * sizeof(int32_t) + sizeof(float));
static_assert(HID == 64 && NIN % 4 == 0 && PF % 4 == 0, "the tiling assumes width 64");

// the car's bank entry, or -1: not a POLICY car, a finished car (drivers_kernel wrote (0, 0)) or beyond the fleet;
// -2: an id outside [0, npolicies)
__device__ __forceinline__ int policy_key(int64_t i, const int32_t* __restrict__ kind, int default_kind, const int32_t* __restrict__ lap,
                                          const int32_t* __restrict__ policy_id, int npolicies, int64_t ncars) {
    if (i >= ncars) return -1;
    const int k = kind ? kind[i] : default_kind;
    if (k != FTGP_DRIVER_POLICY || (lap && lap[i * FTGP_LAP_FIELDS + FTGP_LAP_FINISHED])) return -1;
    const int id = policy_id ? policy_id[i] : 0;
    return (id < 0 || id >= npolicies) ? -2 : id;
}

// warp-aggregated: the lanes holding the same id add once
__global__ void policy_count_kernel(const int32_t* __restrict__ kind, int default_kind, const int32_t* __restrict__ lap,
                                    const int32_t* __restrict__ policy_id, int npolicies, double* __restrict__ ctrl, int64_t ncars,
                                    int32_t* __restrict__ hist) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int key = policy_key(i, kind, default_kind, lap, policy_id, npolicies, ncars);
    if (key == -2) { ctrl[2 * i] = 0.0; ctrl[2 * i + 1] = 0.0; }          // the inert driver (custom.py:1106-1109)
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    if (key >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[key], __popc(peers));
}

__global__ void __launch_bounds__(1024) policy_scan_kernel(const int32_t* __restrict__ hist, int32_t* __restrict__ cursor,
                                                           int32_t* __restrict__ total, int npolicies) {
    __shared__ int32_t warp_sum[32];
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    const int per = (npolicies + 1023) / 1024;
    const int lo = min(t * per, npolicies), hi = min(lo + per, npolicies);
    int32_t s = 0;
    for (int j = lo; j < hi; j++) s += hist[j];
    int32_t incl = s;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int32_t v = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += v;
    }
    if (lane == 31) warp_sum[w] = incl;
    __syncthreads();
    if (w == 0) {
        int32_t v = warp_sum[lane], x = v;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int32_t u = __shfl_up_sync(0xffffffffu, x, off);
            if (lane >= off) x += u;
        }
        warp_sum[lane] = x - v;                      // exclusive offsets of the warps
    }
    __syncthreads();
    int32_t run = warp_sum[w] + incl - s;
    for (int j = lo; j < hi; j++) { cursor[j] = run; run += hist[j]; }
    if (t == 1023) *total = run;
}

__global__ void policy_scatter_kernel(const int32_t* __restrict__ kind, int default_kind, const int32_t* __restrict__ lap,
                                      const int32_t* __restrict__ policy_id, int npolicies, int64_t ncars,
                                      int32_t* __restrict__ cursor, int32_t* __restrict__ list) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int key = policy_key(i, kind, default_kind, lap, policy_id, npolicies, ncars);
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
    int32_t base = 0;
    if (key >= 0 && lane == leader) base = atomicAdd(&cursor[key], __popc(peers));
    base = __shfl_sync(peers, base, leader);
    if (key >= 0) list[base + __popc(peers & ((1u << lane) - 1))] = (int32_t)i;
}

// One layer of HID units for the cars of slots [first, end) of the tile: out[j][s] = tanh(b[j] + sum_i W[i][j] in[i][s]).
// Thread (cg, hg) owns slots 4cg..4cg+3 and units 4hg..4hg+3; a car group with no slot in the run sits this layer out.
template <int NI>
__device__ __forceinline__ void dense_tanh(const float* __restrict__ W, const float* __restrict__ b, const float* in, float* out,
                                           int first, int end) {
    const int hg = threadIdx.x & 15, cg = threadIdx.x >> 4;
    if (4 * cg >= end || 4 * cg + 4 <= first) return;
    float acc[4][4];
    const float4 bv = *reinterpret_cast<const float4*>(b + 4 * hg);
#pragma unroll
    for (int c = 0; c < 4; c++) { acc[c][0] = bv.x; acc[c][1] = bv.y; acc[c][2] = bv.z; acc[c][3] = bv.w; }
#pragma unroll 4
    for (int i = 0; i < NI; i++) {
        const float4 w = *reinterpret_cast<const float4*>(W + i * HID + 4 * hg);
        const float4 x = *reinterpret_cast<const float4*>(in + i * LD + 4 * cg);
        const float xs[4] = {x.x, x.y, x.z, x.w}, ws[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int c = 0; c < 4; c++)
#pragma unroll
            for (int h = 0; h < 4; h++) acc[c][h] = fmaf(ws[h], xs[c], acc[c][h]);
    }
#pragma unroll
    for (int h = 0; h < 4; h++) {
        float4 o;
        o.x = tanhf(acc[0][h]); o.y = tanhf(acc[1][h]); o.z = tanhf(acc[2][h]); o.w = tanhf(acc[3][h]);
        *reinterpret_cast<float4*>(out + (4 * hg + h) * LD + 4 * cg) = o;
    }
}

__global__ void __launch_bounds__(NT, 2)
policy_kernel(const float* __restrict__ weights, const int32_t* __restrict__ policy_id, const int32_t* __restrict__ list,
              const int32_t* __restrict__ total, const float* __restrict__ ranges, const double* __restrict__ qpos,
              const double* __restrict__ qvel, double* __restrict__ ctrl) {
    extern __shared__ float4 smem4[];
    float* w = reinterpret_cast<float*>(smem4);      // the staged policy, FTGP_POLICY_FLOATS
    float* xs = w + PF;                              // x[96][LD]
    float* h1 = xs + NIN * LD;                       // h1[64][LD]
    float* h2 = h1 + HID * LD;                       // h2[64][LD]
    int32_t* cars = reinterpret_cast<int32_t*>(h2 + HID * LD);
    int32_t* pids = cars + TILE;
    float* clip = reinterpret_cast<float*>(pids + TILE);
    const int t = threadIdx.x;
    const int64_t c0 = (int64_t)blockIdx.x * TILE;
    const int32_t n = *total;
    if (c0 >= n) return;
    const int cnt = n - c0 < TILE ? (int)(n - c0) : TILE;
    if (t < TILE) {
        const int32_t car = t < cnt ? list[c0 + t] : 0;
        const int32_t p = t < cnt ? (policy_id ? policy_id[car] : 0) : -1;
        cars[t] = car; pids[t] = p;
        clip[t] = t < cnt ? weights[(int64_t)p * PF + FTGP_POLICY_SCALARS] : 1.0f;
    }
    __syncthreads();
    // inputs (include/ftgp.h): the ranges row read along the beams, one car after the other
    for (int e = t; e < TILE * FTGP_NBEAMS; e += NT) {
        const int s = e / FTGP_NBEAMS, j = e - s * FTGP_NBEAMS;
        float x = 0.0f;
        if (s < cnt) {
            const float r = ranges[(int64_t)cars[s] * FTGP_NBEAMS + j], c = clip[s];
            x = (r >= 0.0f && r < c) ? r / c : 1.0f;
        }
        xs[j * LD + s] = x;
    }
    if (t < TILE) {
        float f = 0.0f, l = 0.0f, wz = 0.0f, u = 0.0f, st = 0.0f;
        if (t < cnt) {
            const int64_t car = cars[t];
            const double* q = qpos + car * FTGP_NQ;
            const double* v = qvel + car * FTGP_NV;
            const double qw = q[3], qx = q[4], qy = q[5], qz = q[6];
            const double yaw = atan2(2.0 * (qw * qz + qx * qy), 1.0 - 2.0 * (qy * qy + qz * qz));   // custom.py:62-76
            const double cy = cos(yaw), sy = sin(yaw), vx = v[0], vy = v[1];
            f = (float)(vx * cy + vy * sy);
            l = (float)(-vx * sy + vy * cy);
            wz = (float)v[5];
            u = (float)ctrl[2 * car]; st = (float)ctrl[2 * car + 1];
        }
        xs[90 * LD + t] = f; xs[91 * LD + t] = l; xs[92 * LD + t] = wz;
        xs[93 * LD + t] = u; xs[94 * LD + t] = st; xs[95 * LD + t] = 0.0f;
    }
    // one run of equal policy ids after the other (the list is grouped, so a tile holds few runs)
    for (int first = 0; first < cnt;) {
        const int p = pids[first];
        int end = first + 1;
        while (end < cnt && pids[end] == p) end++;
        __syncthreads();                             // inputs written / the previous run's weights no longer read
        const float4* src = reinterpret_cast<const float4*>(weights + (int64_t)p * PF);
        for (int k = t; k < PF / 4; k += NT) smem4[k] = __ldg(src + k);
        __syncthreads();
        dense_tanh<NIN>(w + FTGP_POLICY_W1, w + FTGP_POLICY_B1, xs, h1, first, end);
        __syncthreads();
        dense_tanh<HID>(w + FTGP_POLICY_W2, w + FTGP_POLICY_B2, h1, h2, first, end);
        __syncthreads();
        if (t < 2 * TILE) {
            const int s = t >> 1, o = t & 1;
            if (s >= first && s < end) {
                float z = w[FTGP_POLICY_B3 + o];
#pragma unroll 8
                for (int i = 0; i < HID; i++) z = fmaf(w[FTGP_POLICY_W3 + i * 2 + o], h2[i * LD + s], z);
                ctrl[2 * (int64_t)cars[s] + o] = (double)(w[FTGP_POLICY_SCALARS + 1 + o] * tanhf(z));
            }
        }
        first = end;
    }
}

static bool g_policy_attr[16] = {false};

int launch_policy(const ftgp_policy_args* p, const float* ranges, const int32_t* kind, int default_kind, const double* qpos,
                  const double* qvel, const int32_t* lap, double* ctrl, int64_t ncars, cudaStream_t stream) {
    int dev = 0;
    FTGP_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 16 || !g_policy_attr[dev]) {
        FTGP_CUDA(cudaFuncSetAttribute(policy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)POLICY_SMEM));
        if (dev >= 0 && dev < 16) g_policy_attr[dev] = true;
    }
    int32_t* buf = nullptr;
    int rc = policy_scratch(ncars, p->npolicies, stream, &buf);
    if (rc) return rc;
    const int np = p->npolicies;
    int32_t *hist = buf, *cursor = buf + np, *total = buf + 2 * np, *list = buf + 2 * np + 1;
    FTGP_CUDA(cudaMemsetAsync(hist, 0, (size_t)np * sizeof(int32_t), stream));
    const unsigned nb = (unsigned)((ncars + 255) / 256);
    policy_count_kernel<<<nb, 256, 0, stream>>>(kind, default_kind, lap, p->policy_id, np, ctrl, ncars, hist);
    policy_scan_kernel<<<1, 1024, 0, stream>>>(hist, cursor, total, np);
    policy_scatter_kernel<<<nb, 256, 0, stream>>>(kind, default_kind, lap, p->policy_id, np, ncars, cursor, list);
    policy_kernel<<<(unsigned)((ncars + TILE - 1) / TILE), NT, POLICY_SMEM, stream>>>(p->weights, p->policy_id, list, total, ranges,
                                                                                      qpos, qvel, ctrl);
    count_launch(4);
    FTGP_CUDA(cudaGetLastError());
    return FTGP_OK;
}

}  // namespace ftgp
