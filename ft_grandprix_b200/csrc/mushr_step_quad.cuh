// mushr_step_quad.cuh -- QUAD-PER-CAR version of the vehicle step: four lanes advance one car, one lane per
// wheel chain (same arithmetic as mushr_step.cuh, i.e. mj_step for template/mushr.em.xml; replaces
// mujoco.mj_step at ft_grandprix/custom.py:1425).
//
// Why this mapping (profiles/ncu_summary_r03.md): thread-per-car needs 16.7 KB of scratch per thread, which lives
// in local memory and goes through DRAM 120x more often than the algorithmic state (FP64 pipe 5 % busy);
// warp-per-car keeps the state on chip but executes 5.4x the instructions (serial leader sections, lanes idle).
// The model itself says how to split a car: a 7-dof root plus FOUR IDENTICAL 6-slot wheel chains that are
// coupled only through the root (block-arrow M and H).  So lane w of a quad owns
//   * the chain block W_w (6x6), its border B_w (6x7), its wheel-ground contact, its share of the chassis
//     contacts, its friction-loss / limit / equality rows, and the chain part of every dof vector;
//   * a replica of the 7-entry root part of every dof vector and of the 7x7 root block.
// Chain work (the bulk: Cholesky of W_w, Y_w = L^-1 B_w, Schur term Y_w^T Y_w, J^T D J of the contact rows,
// kinematics / CRB / RNE of the wheel and softener bodies) runs 4-wide with no communication; the root block is
// reduced across the quad with two xor-shuffles per value and then handled redundantly by the four lanes, which
// keeps every loop bound and branch quad-uniform (sums are bit-identical in the four lanes).
// A warp holds 8 cars; per-lane state is ~1/4 of a car and ALL of the solver's persistent state is on chip: lane-private
// slots in shared memory in [slot][thread] layout (conflict-free), root parts of the dof vectors and the root block of M
// once per car in [slot][car] layout (the four lanes read them as a broadcast), the lane's border of M in tensor memory
// (Q::mb_load_row / mb_store_row).  784 B of shared memory and 288 B of tensor memory per lane, so 256 lanes (64 cars)
// are resident per SM; the factorisation itself runs entirely in registers.
// Control flow is WARP-UNIFORM (and CTA-uniform at the Newton loop head): every lane of a warp reaches every
// collective in the same order, so the quad reductions are plain full-mask shuffles and the warps of a CTA walk the
// same code at the same time (one instruction-cache fill serves all of them).  A quad whose car has converged keeps
// going through the motions with its stores switched off until the last car of its CTA is done; the exact line
// search is a per-quad state machine clocked by one warp-uniform cost evaluation per tick.
// Rule for the per-car slots: every lane computes the same value and every lane writes it, always after a quad
// sync that follows the last read of the old value (read phase, sync, write phase).
//
// The code is __host__ __device__ over a communicator policy Q (device: shuffles inside the quad; host tests:
// four OS threads and a barrier, tests/host_harness/step_quad_host.cpp), so its arithmetic is checked against the
// oracle on the CPU build box before it runs on a B200.
#pragma once
#include "mushr_step.cuh"
#include "hfield_contact.cuh"

// The solver's pieces are inlined into the kernel on the device: as separate functions (the ABI saves and restores
// ~100 live registers around every call) the step took 1.93 ms for 65,536 cars, inlined 1.48 ms.
#if defined(__CUDACC__) && defined(FT_QUAD_NOINLINE)
#define FT_QN __host__ __device__ __noinline__
#elif defined(__CUDACC__)
#define FT_QN __host__ __device__ __forceinline__
#else
#define FT_QN __attribute__((noinline))
#endif

namespace ftgp {
namespace mushr {

// ---- shared-memory slots (doubles).  P: private to the lane, C: one copy per car --------------------------------
constexpr int QP_MW = 0;             // 21  chain block of M, lower triangle
constexpr int QP_CJ = 21;            // 18  wheel-ground contact Jacobian, row a x (3 root rotations, 3 chain slots)
constexpr int QP_FRA = 39;           // 6   aref of the friction-loss rows of the chain slots
constexpr int QP_EQ = 45;            // 3   Ackermann equality of a front chain: D (0: none), aref, dP/dx
constexpr int QP_LIM = 48;           // 6   suspension / front steering limit: D[2] (0: inactive), aref[2], sign[2]
constexpr int QP_WC = 54;            // 5   wheel-ground contact: D (0: none), aref[4]
constexpr int QP_VEC = 59;           // 4 x 6 chain parts of the dof vectors below
constexpr int QP_SM_N = 83;          // the slots above are the ones the device keeps in shared memory
constexpr int QP_MB = 83;            // 36  border of M: slot l x root dof j < 6 (column 6 of M's border is zero)
constexpr int QP_N = 119;
// The border of M is written once per step and read a row of six at a time, always through mb_load_row / mb_store_row
// below.  A policy that has those members keeps it elsewhere (QuadDev: in tensor memory, which no kernel of the tick uses
// otherwise; it frees 288 B of shared memory per lane) and there they are warp collectives; for a policy without them
// (the host harnesses) the border is the private slots QP_MB ... QP_N - 1.
constexpr int QC_MR = 0;             // 28  root block of M, lower triangle
constexpr int QC_R6 = 28;            // 4   rows of root dof 6 (steering wheel): friction aref, limit D, aref, sign
constexpr int QC_VEC = 32;           // 4 x 7 root parts of the dof vectors
constexpr int QC_N = 60;
struct QVec { int p, c; };           // dof vector: chain part at P(p + l), root part at C(c + i)
// qfrc_smooth, the iterate x = qacc, M x, and S = right-hand side / solution of the factor-solve (qacc_smooth, then the
// gradient / search direction, then the Euler acceleration).  qacc_smooth itself is not kept: the Gauss term
// (x - qacc_smooth)' M (x - qacc_smooth) / 2 is evaluated as x' (M x / 2 - qfrc_smooth) + qacc_smooth' qfrc_smooth / 2;
// M s lives in registers between the line search and the update of M x.
#define VQFS (QVec{QP_VEC, QC_VEC})
#define VX (QVec{QP_VEC + 6, QC_VEC + 7})
#define VMA (QVec{QP_VEC + 12, QC_VEC + 14})
#define VS (QVec{QP_VEC + 18, QC_VEC + 21})
// model constants of the friction-loss rows (pos = 0, so impedance and regulariser never change): (D, R f, f) for
// chain slot (w, l) at 3 (6 w + l), root dof 6 at 72
constexpr int QK_N = 75;

template <int PS_, int CS_>
struct QuadMem {                     // PS: stride between slots of private data (threads per CTA), CS: cars per CTA
    static constexpr int PS = PS_, CS = CS_;
    double* priv; double* shr; const double* ktab; int w;
    FT_HD double& P(int i) const { return priv[i * PS]; }
    FT_HD double& C(int i) const { return shr[i * CS]; }
    FT_HD double K(int i) const { return ktab[i]; }
    FT_HD int lane() const { return w; }
};

#if defined(__CUDACC__)
extern __shared__ __align__(16) double quad_sm[];      // the kernel's dynamic shared memory (so that accesses are LDS/STS)
template <int PS_, int CS_, bool CTA_LOCKSTEP>
struct QuadDev {                     // po / co / ko: offsets (in doubles) of the lane's, the car's and the table's first slot
    static constexpr int PS = PS_, CS = CS_;
    int po, co, ko, w, qs;           // qs: position of the quad in the warp (lane & 28)
    uint32_t tm;                     // tensor-memory address of the warp's border rows (tmem_border_addr)
    __device__ __forceinline__ double& P(int i) const { return quad_sm[po + i * PS]; }
    __device__ __forceinline__ double& C(int i) const { return quad_sm[co + i * CS]; }
    __device__ __forceinline__ double K(int i) const { return quad_sm[ko + i]; }
    __device__ __forceinline__ int lane() const { return w; }
    // row l of the lane's border of M: 12 columns (six doubles as lo/hi words) from column 12 l of the thread's TMEM lane.
    // tcgen05.ld / st are .sync.aligned warp collectives; the __syncwarp makes sure the warp arrives converged.  The wait
    // sits in the same asm statement so that no use of the loaded registers can be scheduled before it.
    __device__ __forceinline__ void mb_load_row(int l, double* b) const {
        uint32_t r[12];
        __syncwarp();
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%12];\n\t"
                     "tcgen05.ld.sync.aligned.32x32b.x4.b32 {%8, %9, %10, %11}, [%13];\n\t"
                     "tcgen05.wait::ld.sync.aligned;"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                       "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11])
                     : "r"(tm + 12u * l), "r"(tm + 12u * l + 8u));
#pragma unroll
        for (int j = 0; j < 6; j++) b[j] = __hiloint2double((int)r[2 * j + 1], (int)r[2 * j]);
    }
    __device__ __forceinline__ void mb_store_row(int l, const double* b) const {
        uint32_t r[12];
#pragma unroll
        for (int j = 0; j < 6; j++) { r[2 * j] = (uint32_t)__double2loint(b[j]); r[2 * j + 1] = (uint32_t)__double2hiint(b[j]); }
        __syncwarp();
        asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%2, %3, %4, %5, %6, %7, %8, %9};\n\t"
                     "tcgen05.st.sync.aligned.32x32b.x4.b32 [%1], {%10, %11, %12, %13};\n\t"
                     "tcgen05.wait::st.sync.aligned;"
                     :: "r"(tm + 12u * l), "r"(tm + 12u * l + 8u), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]),
                        "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11])
                     : "memory");
    }
    // collectives: called by all 32 lanes of the warp together (cany: by the whole CTA)
    __device__ __forceinline__ double sum(double v) const {
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        return v;
    }
    __device__ __forceinline__ unsigned ballot(bool p) const { return (__ballot_sync(0xffffffffu, p) >> qs) & 0xFu; }
    __device__ __forceinline__ bool any(bool p) const { return ballot(p) != 0; }
    __device__ __forceinline__ bool wany(bool p) const { return __any_sync(0xffffffffu, p) != 0; }
    __device__ __forceinline__ bool cany(bool p) const { return CTA_LOCKSTEP ? __syncthreads_or(p) != 0 : wany(p); }
    __device__ __forceinline__ void sync() const { __syncwarp(); }
};
#endif

template <class Q, class = void> struct HasMbRows { static constexpr bool value = false; };
template <class Q> struct HasMbRows<Q, decltype(static_cast<const Q*>(nullptr)->mb_load_row(0, static_cast<double*>(nullptr)))> {
    static constexpr bool value = true;
};
template <class Q> FT_HD void mb_load_row(const Q& qd, int l, double* b) {
    if constexpr (HasMbRows<Q>::value) qd.mb_load_row(l, b);
    else for (int j = 0; j < 6; j++) b[j] = qd.P(QP_MB + 6 * l + j);
}
template <class Q> FT_HD void mb_store_row(const Q& qd, int l, const double* b) {
    if constexpr (HasMbRows<Q>::value) qd.mb_store_row(l, b);
    else for (int j = 0; j < 6; j++) qd.P(QP_MB + 6 * l + j) = b[j];
}

FT_HDN void quad_const_entry(const ModelConsts& mc, int g, double* t) {      // g: 0..23 chain slot (w, l), 24: root dof 6
    const int p = g < 24 ? NR + g : 6;
    const double f = dof_dummy(p) ? 0.0 : dof_floss(p);
    double K, B, imp, R;
    kbi(0.9, 0.0, mc.dof_invweight0[p], K, B, imp, R);
    t[3 * g] = f > 0 ? 1 / R : 0.0; t[3 * g + 1] = f > 0 ? R * f : 0.0; t[3 * g + 2] = f;
}

// Rare contacts owned by the lane, kept in the lane's frame (local memory) and only touched when present:
//   * up to QMAXCH contacts of the car body's geoms (chassis hull vertices / lidar cylinder against walls and ground):
//     MAXBODYCON = 8 over four lanes, Jacobian over the six chassis dofs only;
//   * up to two "chain contacts" against the walls (bit c of ww): c = 0 the lane's wheel ellipsoid (Jacobian over the six
//     chassis dofs and chain slots 0-2), c = 1 its softener sphere with the option bubble_wrap (chain slots 0-5).
// All of them: condim 3, mu = 1 (hfield / chassis / cylinder / softener friction 1 > wheel 0.3, plane 0.5).
constexpr int QMAXCH = 2, MAXBODYCON = 4 * QMAXCH;
struct QChassis {
    double D[QMAXCH], aref[QMAXCH][4], J[QMAXCH][3][6], dx[QMAXCH][3], ds[QMAXCH][3];
    double wD[2], waref[2][4], wJ[2][3][12], wdx[2][3], wds[2][3];      // chain contacts: wheel-wall, softener-wall
};
struct QState { double cost, gauss, c0; unsigned mask; int nch, ww; };  // c0 = qacc_smooth' qfrc_smooth / 2
constexpr int QB_FR = 0, QB_FR6 = 6, QB_LIM = 7, QB_LIM6 = 9, QB_WC = 10, QB_CH = 14, QB_WW = 22;   // QB_WW + 4 c + rr
constexpr double WC_MU = 0.5, CH_MU = 1.0;
constexpr double REF_B = 2 / (0.95 * 0.02);          // kbi(): B of the default solref with dmax 0.95

FT_HD int popc4(unsigned m) { return (int)((m & 1u) + ((m >> 1) & 1u) + ((m >> 2) & 1u) + ((m >> 3) & 1u)); }
FT_HD double dot6q(const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2] + a[3] * b[3] + a[4] * b[4] + a[5] * b[5]; }

template <class Q> FT_HD void vec_load(const Q& qd, QVec v, double* r, double* c) {
#pragma unroll
    for (int i = 0; i < NR; i++) r[i] = qd.C(v.c + i);
#pragma unroll
    for (int l = 0; l < NC; l++) c[l] = qd.P(v.p + l);
}
template <class Q> FT_HD void vec_store(const Q& qd, QVec v, const double* r, const double* c, bool on = true) {   // caller has synced
    if (!on) return;
#pragma unroll
    for (int i = 0; i < NR; i++) qd.C(v.c + i) = r[i];
#pragma unroll
    for (int l = 0; l < NC; l++) qd.P(v.p + l) = c[l];
}

// wheel contact in its frame n = (0,0,1), t1 = (0,1,0), t2 = (-1,0,0): d3 = J x.  The translation columns of J are
// those unit vectors; the other six (root rotations, chain slots 0-2) are in shared memory.
template <class Q>
FT_HD void wc_dots(const Q& qd, const double* xr, const double* xc, double* d3) {
    d3[0] = xr[2]; d3[1] = xr[1]; d3[2] = -xr[0];
#pragma unroll
    for (int a = 0; a < 3; a++) {
        double s = d3[a];
#pragma unroll
        for (int k = 0; k < 3; k++) s += qd.P(QP_CJ + 6 * a + k) * xr[3 + k] + qd.P(QP_CJ + 6 * a + 3 + k) * xc[k];
        d3[a] = s;
    }
}


// ---- rare contacts, out of line ------------------------------------------------------------------------------------
// The contacts of the car body's geoms and the chain contacts (a wheel / softener against a wall) exist for a few per cent
// of the cars.  Their code is kept OUT OF LINE (one call behind a branch) so that the Newton loop every car runs stays
// small: with it inlined the loop no longer fitted the instruction cache (stall_no_inst 0.7 -> 4.1 cycles per issue, first
// launch 0.93 -> 1.99 ms; profiles/ncu_summary_r11.md).  The helpers take the vectors from shared memory themselves and
// return small structs by value, so that no register array of the caller has its address taken.
#if defined(__CUDACC__)
#define FT_RARE __host__ __device__ __noinline__
#else
#define FT_RARE inline
#endif
struct RareRows { double cost, fr[6], fc[NC]; unsigned mask; };
struct RareHess { double P[21], W[21], B[NC][6]; };
struct RareVec6 { double v[NC]; };
struct RareQuad { double q0, q1, q2; };

// cost / forces / active-row mask of the rare rows at the vector X (root part xr[0..5], chain part xc)
template <class Q>
FT_RARE RareRows rare_rows(const Q& qd, const QChassis& ch, int nch, int ww, QVec X) {
    RareRows o;
    o.cost = 0; o.mask = 0;
    double xr[6], xc[NC];
    for (int i = 0; i < 6; i++) { o.fr[i] = 0; xr[i] = qd.C(X.c + i); }
    for (int l = 0; l < NC; l++) { o.fc[l] = 0; xc[l] = qd.P(X.p + l); }
    for (int s = 0; s < nch; s++) {                                      // contacts of the car body's geoms: root dofs only
        double d3[3];
        for (int a = 0; a < 3; a++) d3[a] = dot6q(ch.J[s][a], xr);
        const double D = ch.D[s];
        for (int rr = 0; rr < 4; rr++) {
            const double sg = (rr & 1) ? -CH_MU : CH_MU; const int ta = 1 + (rr >> 1);
            const double jar = d3[0] + sg * d3[ta] - ch.aref[s][rr];
            if (jar >= 0) continue;
            o.cost += 0.5 * D * jar * jar;
            o.mask |= 1u << (QB_CH + 4 * s + rr);
            const double f = -D * jar;
            for (int col = 0; col < 6; col++) o.fr[col] += (ch.J[s][0][col] + sg * ch.J[s][ta][col]) * f;
        }
    }
    for (int c = 0; c < 2; c++) {                                        // the lane's wheel / softener against a wall
        if (!(ww >> c & 1)) continue;
        double d3[3];
        for (int a = 0; a < 3; a++) d3[a] = dot6q(ch.wJ[c][a], xr) + dot6q(ch.wJ[c][a] + 6, xc);
        for (int rr = 0; rr < 4; rr++) {
            const double sg = (rr & 1) ? -CH_MU : CH_MU; const int ta = 1 + (rr >> 1);
            const double jar = d3[0] + sg * d3[ta] - ch.waref[c][rr];
            if (jar >= 0) continue;
            o.cost += 0.5 * ch.wD[c] * jar * jar;
            o.mask |= 1u << (QB_WW + 4 * c + rr);
            const double f = -ch.wD[c] * jar;
            for (int col = 0; col < 6; col++) o.fr[col] += (ch.wJ[c][0][col] + sg * ch.wJ[c][ta][col]) * f;
            for (int k = 0; k < NC; k++) o.fc[k] += (ch.wJ[c][0][6 + k] + sg * ch.wJ[c][ta][6 + k]) * f;
        }
    }
    return o;
}

// J' D J of the active rare rows: root block (6 x 6 lower triangle), chain block (lower triangle), border (chain x root)
FT_RARE RareHess rare_hessian(const QChassis& ch, int nch, int ww, unsigned mask) {
    RareHess o;
    for (int i = 0; i < 21; i++) { o.P[i] = 0; o.W[i] = 0; }
    for (int l = 0; l < NC; l++) for (int j = 0; j < 6; j++) o.B[l][j] = 0;
    for (int s = 0; s < nch; s++) {
        const double D = ch.D[s];
        for (int rr = 0; rr < 4; rr++) {
            if (!(mask >> (QB_CH + 4 * s + rr) & 1u)) continue;
            const double sg = (rr & 1) ? -CH_MU : CH_MU; const int ta = 1 + (rr >> 1);
            double Jr[6];
            for (int col = 0; col < 6; col++) Jr[col] = ch.J[s][0][col] + sg * ch.J[s][ta][col];
            for (int i = 0; i < 6; i++) { const double di = D * Jr[i]; for (int j = 0; j <= i; j++) o.P[tri(i, j)] += di * Jr[j]; }
        }
    }
    for (int c = 0; c < 2; c++) {
        if (!(ww >> c & 1)) continue;
        for (int rr = 0; rr < 4; rr++) {
            if (!(mask >> (QB_WW + 4 * c + rr) & 1u)) continue;
            const double sg = (rr & 1) ? -CH_MU : CH_MU; const int ta = 1 + (rr >> 1);
            double Jr[12];
            for (int col = 0; col < 12; col++) Jr[col] = ch.wJ[c][0][col] + sg * ch.wJ[c][ta][col];
            for (int i = 0; i < 6; i++) { const double di = ch.wD[c] * Jr[i]; for (int j = 0; j <= i; j++) o.P[tri(i, j)] += di * Jr[j]; }
            for (int l = 0; l < NC; l++) {
                const double dl = ch.wD[c] * Jr[6 + l];
                for (int k = 0; k <= l; k++) o.W[tri(l, k)] += dl * Jr[6 + k];
                for (int j = 0; j < 6; j++) o.B[l][j] += dl * Jr[j];
            }
        }
    }
    return o;
}

// the chain contacts' share of (border of H) x_r, x_r = the first six entries of the root part of V
template <class Q>
FT_RARE RareVec6 rare_border(const Q& qd, const QChassis& ch, int ww, unsigned mask, const double* xr6) {
    RareVec6 o;
    for (int l = 0; l < NC; l++) o.v[l] = 0;
    for (int c = 0; c < 2; c++) {
        if (!(ww >> c & 1)) continue;
        for (int rr = 0; rr < 4; rr++) {
            if (!(mask >> (QB_WW + 4 * c + rr) & 1u)) continue;
            const double sg = (rr & 1) ? -CH_MU : CH_MU; const int ta = 1 + (rr >> 1);
            double sacc = 0;
            for (int col = 0; col < 6; col++) sacc += (ch.wJ[c][0][col] + sg * ch.wJ[c][ta][col]) * xr6[col];
            sacc *= ch.wD[c];
            for (int l = 0; l < NC; l++) o.v[l] += (ch.wJ[c][0][6 + l] + sg * ch.wJ[c][ta][6 + l]) * sacc;
        }
    }
    return o;
}

// line search: J x and J s of the rare contacts (x = VX, s = VS in shared memory) ...
template <class Q>
FT_RARE void rare_ls_init(const Q& qd, QChassis& ch, int nch, int ww) {
    double xr[6], xc[NC], sr[6], sc[NC];
    for (int i = 0; i < 6; i++) { xr[i] = qd.C(VX.c + i); sr[i] = qd.C(VS.c + i); }
    for (int l = 0; l < NC; l++) { xc[l] = qd.P(VX.p + l); sc[l] = qd.P(VS.p + l); }
    for (int s = 0; s < nch; s++)
        for (int a = 0; a < 3; a++) { ch.dx[s][a] = dot6q(ch.J[s][a], xr); ch.ds[s][a] = dot6q(ch.J[s][a], sr); }
    for (int c = 0; c < 2; c++)
        if (ww >> c & 1)
            for (int a = 0; a < 3; a++) {
                ch.wdx[c][a] = dot6q(ch.wJ[c][a], xr) + dot6q(ch.wJ[c][a] + 6, xc);
                ch.wds[c][a] = dot6q(ch.wJ[c][a], sr) + dot6q(ch.wJ[c][a] + 6, sc);
            }
}
// ... and their share of the cost along the line at alpha
FT_RARE RareQuad rare_ls(const QChassis& ch, int nch, int ww, double alpha) {
    RareQuad o;
    o.q0 = o.q1 = o.q2 = 0;
    for (int s = 0; s < nch; s++) {
        const double D = ch.D[s];
        for (int rr = 0; rr < 4; rr++) {
            const double sg = (rr & 1) ? -CH_MU : CH_MU; const int ta = 1 + (rr >> 1);
            const double jar = ch.dx[s][0] + sg * ch.dx[s][ta] - ch.aref[s][rr], jv = ch.ds[s][0] + sg * ch.ds[s][ta];
            if (jar + alpha * jv < 0) { o.q0 += 0.5 * D * jar * jar; o.q1 += D * jar * jv; o.q2 += 0.5 * D * jv * jv; }
        }
    }
    for (int c = 0; c < 2; c++) {
        if (!(ww >> c & 1)) continue;
        const double D = ch.wD[c];
        for (int rr = 0; rr < 4; rr++) {
            const double sg = (rr & 1) ? -CH_MU : CH_MU; const int ta = 1 + (rr >> 1);
            const double jar = ch.wdx[c][0] + sg * ch.wdx[c][ta] - ch.waref[c][rr], jv = ch.wds[c][0] + sg * ch.wds[c][ta];
            if (jar + alpha * jv < 0) { o.q0 += 0.5 * D * jar * jar; o.q1 += D * jar * jv; o.q2 += 0.5 * D * jv * jv; }
        }
    }
    return o;
}

// ---- cost of this lane's rows at the vector X: forces J^T f into fr (root, lane's share) / fc (chain), zone mask --
template <class Q>
FT_QN double rows_eval(const Q& qd, const QChassis& ch, int nch, int ww, QVec X, double* fr, double* fc, unsigned& mask_out) {
    const int w = qd.lane();
    double xr[NR], xc[NC];
    vec_load(qd, X, xr, xc);
    double cost = 0;
    unsigned mask = 0;
#pragma unroll
    for (int i = 0; i < NR; i++) fr[i] = 0;
#pragma unroll
    for (int l = 0; l < NC; l++) {                                       // friction loss: quadratic inside +-R f, linear outside
        const double D = qd.K(3 * (6 * w + l)), Rf = qd.K(3 * (6 * w + l) + 1), f = qd.K(3 * (6 * w + l) + 2);
        const double jar = xc[l] - qd.P(QP_FRA + l);
        const bool lo = jar <= -Rf, hi = jar >= Rf, lin = lo || hi;
        cost += lin ? -0.5 * Rf * f + f * (lo ? -jar : jar) : 0.5 * D * jar * jar;
        fc[l] = lin ? (lo ? f : -f) : -D * jar;
        if (!lin) mask |= 1u << (QB_FR + l);
    }
    {                                                                    // equality (D = 0 on the rear lanes)
        const double D = qd.P(QP_EQ), der = qd.P(QP_EQ + 2), jar = xc[1] - der * xr[6] - qd.P(QP_EQ + 1);
        cost += 0.5 * D * jar * jar;
        const double f = -D * jar;
        fc[1] += f; fr[6] -= der * f;
    }
#pragma unroll
    for (int k = 0; k < 2; k++) {                                        // limits: active when jar < 0 (D = 0: no row)
        const double D = qd.P(QP_LIM + k), sg = qd.P(QP_LIM + 4 + k), jar = sg * xc[k] - qd.P(QP_LIM + 2 + k);
        if (D > 0 && jar < 0) { cost += 0.5 * D * jar * jar; fc[k] += sg * (-D * jar); mask |= 1u << (QB_LIM + k); }
    }
    if (w == 0) {                                                        // rows of the steering-wheel dof
        const double D = qd.K(72), Rf = qd.K(73), f = qd.K(74), jar = xr[6] - qd.C(QC_R6);
        const bool lo = jar <= -Rf, hi = jar >= Rf, lin = lo || hi;
        cost += lin ? -0.5 * Rf * f + f * (lo ? -jar : jar) : 0.5 * D * jar * jar;
        fr[6] += lin ? (lo ? f : -f) : -D * jar;
        if (!lin) mask |= 1u << QB_FR6;
        const double D6 = qd.C(QC_R6 + 1), sg = qd.C(QC_R6 + 3), jar6 = sg * xr[6] - qd.C(QC_R6 + 2);
        if (D6 > 0 && jar6 < 0) { cost += 0.5 * D6 * jar6 * jar6; fr[6] += sg * (-D6 * jar6); mask |= 1u << QB_LIM6; }
    }
    const double Dw = qd.P(QP_WC);
    if (Dw > 0) {                                                        // pyramidal rows of the wheel contact
        double d3[3], F[3] = {0, 0, 0};                                  // F: sum of the row forces in the contact frame
        wc_dots(qd, xr, xc, d3);
#pragma unroll
        for (int rr = 0; rr < 4; rr++) {
            const double sg = (rr & 1) ? -WC_MU : WC_MU; const int ta = 1 + (rr >> 1);
            const double jar = d3[0] + sg * d3[ta] - qd.P(QP_WC + 1 + rr);
            if (jar < 0) { cost += 0.5 * Dw * jar * jar; mask |= 1u << (QB_WC + rr); const double f = -Dw * jar; F[0] += f; F[ta] += sg * f; }
        }
        fr[0] -= F[2]; fr[1] += F[1]; fr[2] += F[0];
#pragma unroll
        for (int k = 0; k < 3; k++) {
            fr[3 + k] += qd.P(QP_CJ + k) * F[0] + qd.P(QP_CJ + 6 + k) * F[1] + qd.P(QP_CJ + 12 + k) * F[2];
            fc[k] += qd.P(QP_CJ + 3 + k) * F[0] + qd.P(QP_CJ + 9 + k) * F[1] + qd.P(QP_CJ + 15 + k) * F[2];
        }
    }
    if (nch | ww) {                                                      // rare contacts (out of line)
        const RareRows o = rare_rows(qd, ch, nch, ww, X);
        cost += o.cost; mask |= o.mask;
#pragma unroll
        for (int i = 0; i < 6; i++) fr[i] += o.fr[i];
#pragma unroll
        for (int l = 0; l < NC; l++) fc[l] += o.fc[l];
    }
    mask_out = mask;
    return cost;
}

// y = M X with M on chip (shared and tensor memory), result in registers (root part replicated)
template <class Q>
FT_QN void quad_mul(const Q& qd, QVec X, double* yr, double* yc) {
    double xr[NR], xc[NC], part[6];
    vec_load(qd, X, xr, xc);
#pragma unroll
    for (int j = 0; j < 6; j++) part[j] = 0;
#pragma unroll
    for (int l = 0; l < NC; l++) {
        double s = 0;
#pragma unroll
        for (int k = 0; k < NC; k++) s += qd.P(QP_MW + (l >= k ? tri(l, k) : tri(k, l))) * xc[k];
        double b[6];
        mb_load_row(qd, l, b);
#pragma unroll
        for (int j = 0; j < 6; j++) { s += b[j] * xr[j]; part[j] += b[j] * xc[l]; }
        yc[l] = s;
    }
#pragma unroll
    for (int i = 0; i < NR; i++) {
        double s = 0;
#pragma unroll
        for (int j = 0; j < NR; j++) s += qd.C(QC_MR + (i >= j ? tri(i, j) : tri(j, i))) * xr[j];
        if (i < 6) s += qd.sum(part[i]);
        yr[i] = s;
    }
}

// cost, Gauss term and gradient (into S) at X (needs MA = M X)
template <class Q>
FT_QN void quad_evaluate(const Q& qd, const QChassis& ch, QState& st, bool on) {
    double fr[NR], fc[NC], g_r[NR], g_c[NC];
    unsigned mask;
    double cc = rows_eval(qd, ch, st.nch, st.ww, VX, fr, fc, mask);
    double g = 0;
#pragma unroll
    for (int l = 0; l < NC; l++) {
        const double ma = qd.P(VMA.p + l), qf = qd.P(VQFS.p + l);
        g += qd.P(VX.p + l) * (0.5 * ma - qf);
        g_c[l] = (ma - qf) - fc[l];
    }
    cc = qd.sum(cc); g = qd.sum(g);
#pragma unroll
    for (int i = 0; i < NR; i++) {
        const double ma = qd.C(VMA.c + i), qf = qd.C(VQFS.c + i);
        g += qd.C(VX.c + i) * (0.5 * ma - qf);
        g_r[i] = (ma - qf) - qd.sum(fr[i]);
    }
    g += st.c0;
    if (on) { st.mask = mask; st.gauss = g; st.cost = cc + g; }
    qd.sync();
    vec_store(qd, VS, g_r, g_c, on);
}

// V <- sign * A^-1 V with A = M (mode 0), M + J^T D J over the rows flagged in st.mask (mode 1), M + h diag(damping)
// (mode 2).  The whole factorisation lives in registers: chain Cholesky, Y = L^-1 B, the lane's share of the Schur
// complement, one 28-value reduction across the quad, root Cholesky (replicated), solve.
template <class Q>
FT_QN void quad_factor_solve(const Q& qd, const QChassis& ch, const QState& st, int mode, QVec V, double sign, bool on) {
    const int w = qd.lane();
    double W[21], B[NC][NR], Pp[28];
    double k00 = 0, k01 = 0, k02 = 0, k11 = 0, k22 = 0, eqb = 0;      // contact-frame K and the equality's border entry (mode 1)
    bool wcon = false;
#pragma unroll
    for (int i = 0; i < 21; i++) W[i] = qd.P(QP_MW + i);
#pragma unroll
    for (int l = 0; l < NC; l++) {
        mb_load_row(qd, l, B[l]);
        B[l][6] = 0;
    }
#pragma unroll
    for (int i = 0; i < 28; i++) Pp[i] = 0;
    if (mode == 2) {
        W[tri(0, 0)] += TIMESTEP * 12.5;
        if (front(w)) W[tri(1, 1)] += TIMESTEP * 0.1;
        W[tri(2, 2)] += TIMESTEP * 0.01;
        if (w == 0) Pp[tri(6, 6)] += TIMESTEP * 0.1;
    } else if (mode == 1) {
        const unsigned mask = st.mask;
        { const double D = qd.P(QP_EQ), der = qd.P(QP_EQ + 2); eqb = -D * der; W[tri(1, 1)] += D; B[1][6] += eqb; Pp[tri(6, 6)] += D * der * der; }
#pragma unroll
        for (int l = 0; l < NC; l++) if (mask >> (QB_FR + l) & 1u) W[tri(l, l)] += qd.K(3 * (6 * w + l));
#pragma unroll
        for (int k = 0; k < 2; k++) if (mask >> (QB_LIM + k) & 1u) W[tri(k, k)] += qd.P(QP_LIM + k);
        if (mask >> QB_FR6 & 1u) Pp[tri(6, 6)] += qd.K(72);
        if (mask >> QB_LIM6 & 1u) Pp[tri(6, 6)] += qd.C(QC_R6 + 1);
        if (mask >> QB_WC & 0xFu) {
            // the active pyramid rows n +- mu t1, n +- mu t2 sum to J^T K J with a 3x3 K in the contact frame
            const double D = qd.P(QP_WC);
            const double a0 = (mask >> QB_WC & 1u) ? 1.0 : 0.0, a1 = (mask >> (QB_WC + 1) & 1u) ? 1.0 : 0.0,
                         a2 = (mask >> (QB_WC + 2) & 1u) ? 1.0 : 0.0, a3 = (mask >> (QB_WC + 3) & 1u) ? 1.0 : 0.0;
            k00 = D * (a0 + a1 + a2 + a3); k01 = D * WC_MU * (a0 - a1); k02 = D * WC_MU * (a2 - a3);
            k11 = D * WC_MU * WC_MU * (a0 + a1); k22 = D * WC_MU * WC_MU * (a2 + a3);
            wcon = true;
            double J[3][9], T[3][9];
            J[0][0] = 0; J[0][1] = 0; J[0][2] = 1; J[1][0] = 0; J[1][1] = 1; J[1][2] = 0; J[2][0] = -1; J[2][1] = 0; J[2][2] = 0;
#pragma unroll
            for (int a = 0; a < 3; a++)
#pragma unroll
                for (int k = 0; k < 6; k++) J[a][3 + k] = qd.P(QP_CJ + 6 * a + k);
#pragma unroll
            for (int col = 0; col < 9; col++) {
                T[0][col] = k00 * J[0][col] + k01 * J[1][col] + k02 * J[2][col];
                T[1][col] = k01 * J[0][col] + k11 * J[1][col];
                T[2][col] = k02 * J[0][col] + k22 * J[2][col];
            }
#pragma unroll
            for (int i = 0; i < 6; i++)
#pragma unroll
                for (int j = 0; j <= i; j++) Pp[tri(i, j)] += J[0][i] * T[0][j] + J[1][i] * T[1][j] + J[2][i] * T[2][j];
#pragma unroll
            for (int l = 0; l < 3; l++) {
#pragma unroll
                for (int k = 0; k <= l; k++) W[tri(l, k)] += J[0][6 + l] * T[0][6 + k] + J[1][6 + l] * T[1][6 + k] + J[2][6 + l] * T[2][6 + k];
#pragma unroll
                for (int j = 0; j < 6; j++) B[l][j] += J[0][6 + l] * T[0][j] + J[1][6 + l] * T[1][j] + J[2][6 + l] * T[2][j];
            }
        }
        if (st.nch | st.ww) {                                            // rare contacts (out of line)
            const RareHess o = rare_hessian(ch, st.nch, st.ww, mask);
#pragma unroll
            for (int i = 0; i < 21; i++) { Pp[i] += o.P[i]; W[i] += o.W[i]; }
#pragma unroll
            for (int l = 0; l < NC; l++)
#pragma unroll
                for (int j = 0; j < 6; j++) B[l][j] += o.B[l][j];
        }
    }
    // chain block: W = L L^T, diagonal keeps 1 / L_jj.  Right-looking (outer-product) order: column j is finished, then the
    // trailing block is updated at once.  Every element sees exactly the same subtractions in the same order as in the
    // dot-product form (bit-identical results), but they are issued as soon as their inputs exist, so the dependent chain
    // per column is one multiply-add + the reciprocal square root instead of j multiply-adds + rsqrt + j multiply-adds: the
    // factorisation is latency-bound with 1.7 warps per scheduler (profiles/ncu_summary_r12.md: the two Cholesky inner
    // products were the two hottest lines of the kernel).
#pragma unroll
    for (int j = 0; j < NC; j++) {
        double d = W[tri(j, j)];
        if (d < MINVAL) d = MINVAL;
        const double id = inv_sqrt(d);
        W[tri(j, j)] = id;
#pragma unroll
        for (int i = j + 1; i < NC; i++) W[tri(i, j)] *= id;
#pragma unroll
        for (int i = j + 1; i < NC; i++)
#pragma unroll
            for (int k = j + 1; k <= i; k++) W[tri(i, k)] -= W[tri(i, j)] * W[tri(k, j)];
    }
    // Y = L^-1 B and the right-hand side's chain part z = L^-1 b_c (column-oriented forward substitution, same order of
    // operations per element as the row-oriented one)
    double z[NC];
#pragma unroll
    for (int l = 0; l < NC; l++) z[l] = qd.P(V.p + l);
#pragma unroll
    for (int k = 0; k < NC; k++) {
#pragma unroll
        for (int col = 0; col < NR; col++) B[k][col] *= W[tri(k, k)];
        z[k] *= W[tri(k, k)];
#pragma unroll
        for (int l = k + 1; l < NC; l++) {
#pragma unroll
            for (int col = 0; col < NR; col++) B[l][col] -= W[tri(l, k)] * B[k][col];
            z[l] -= W[tri(l, k)] * z[k];
        }
    }
    // lane's share of the Schur complement and of the root right-hand side, reduced across the quad
    double R[28], xr[NR];
#pragma unroll
    for (int i = 0; i < NR; i++) {
#pragma unroll
        for (int j = 0; j <= i; j++) {
            double s = Pp[tri(i, j)];
#pragma unroll
            for (int l = 0; l < NC; l++) s -= B[l][i] * B[l][j];
            R[tri(i, j)] = qd.C(QC_MR + tri(i, j)) + qd.sum(s);
        }
        double s = 0;
#pragma unroll
        for (int l = 0; l < NC; l++) s += B[l][i] * z[l];
        xr[i] = qd.C(V.c + i) - qd.sum(s);
    }
    // root block (replicated in the four lanes): right-looking Cholesky and column-oriented forward substitution, as above
#pragma unroll
    for (int j = 0; j < NR; j++) {
        double d = R[tri(j, j)];
        if (d < MINVAL) d = MINVAL;
        const double id = inv_sqrt(d);
        R[tri(j, j)] = id;
#pragma unroll
        for (int i = j + 1; i < NR; i++) R[tri(i, j)] *= id;
#pragma unroll
        for (int i = j + 1; i < NR; i++)
#pragma unroll
            for (int k = j + 1; k <= i; k++) R[tri(i, k)] -= R[tri(i, j)] * R[tri(k, j)];
        xr[j] *= id;
#pragma unroll
        for (int i = j + 1; i < NR; i++) xr[i] -= R[tri(i, j)] * xr[j];
    }
    // back substitution with L^T, column-oriented (every finished x_k is subtracted from the rows above at once)
#pragma unroll
    for (int k = NR - 1; k >= 0; k--) {
        xr[k] *= R[tri(k, k)];
#pragma unroll
        for (int i = 0; i < k; i++) xr[i] -= R[tri(k, i)] * xr[k];
    }
    // chain: x_c = W^-1 (b_c - B x_r) with the ORIGINAL border B, read again from where it is stored (keeping Y = L^-1 B
    // alive across the root factorisation costs 84 registers and spills; rebuilding B x_r costs ~90 DFMA)
    {
        double t[NC];
#pragma unroll
        for (int l = 0; l < NC; l++) {
            double sacc = qd.P(V.p + l), b[6];
            mb_load_row(qd, l, b);
#pragma unroll
            for (int j = 0; j < 6; j++) sacc -= b[j] * xr[j];
            t[l] = sacc;
        }
        t[1] -= eqb * xr[6];
        if (wcon) {
            double v3[3] = {xr[2], xr[1], -xr[0]}, u[3];
#pragma unroll
            for (int a = 0; a < 3; a++)
#pragma unroll
                for (int k = 0; k < 3; k++) v3[a] += qd.P(QP_CJ + 6 * a + k) * xr[3 + k];
            u[0] = k00 * v3[0] + k01 * v3[1] + k02 * v3[2]; u[1] = k01 * v3[0] + k11 * v3[1]; u[2] = k02 * v3[0] + k22 * v3[2];
#pragma unroll
            for (int l = 0; l < 3; l++) t[l] -= qd.P(QP_CJ + 3 + l) * u[0] + qd.P(QP_CJ + 9 + l) * u[1] + qd.P(QP_CJ + 15 + l) * u[2];
        }
        if (mode == 1 && st.ww) {                                        // (the chain contacts' share of the border, as above)
            const double x6[6] = {xr[0], xr[1], xr[2], xr[3], xr[4], xr[5]};
            const RareVec6 o = rare_border(qd, ch, st.ww, st.mask, x6);
#pragma unroll
            for (int l = 0; l < NC; l++) t[l] -= o.v[l];
        }
#pragma unroll
        for (int l = 0; l < NC; l++) z[l] = t[l];
#pragma unroll
        for (int k = 0; k < NC; k++) {
            z[k] *= W[tri(k, k)];
#pragma unroll
            for (int l = k + 1; l < NC; l++) z[l] -= W[tri(l, k)] * z[k];
        }
    }
#pragma unroll
    for (int k = NC - 1; k >= 0; k--) {
        z[k] *= W[tri(k, k)];
#pragma unroll
        for (int l = 0; l < k; l++) z[l] -= W[tri(k, l)] * z[k];
    }
#pragma unroll
    for (int i = 0; i < NR; i++) xr[i] *= sign;
#pragma unroll
    for (int l = 0; l < NC; l++) z[l] *= sign;
    qd.sync();                        // (the reductions above already follow every lane's reads of V's root part)
    vec_store(qd, V, xr, z, on);
}

// ---- exact line search (PrimalSearch) ---------------------------------------------------------------------------
// Everything the cost along the search line needs, gathered once per line search and kept in registers: per row
// the residual at alpha = 0 (j) and its slope (v); always-quadratic terms (Gauss, equality) are folded into c0-c2.
struct QLs {
    double c0, c1, c2;               // lane's always-quadratic rows (added before the quad sum)
    double g0, g1, g2;               // Gauss term (replicated, added after the sum)
    double fj[NC], fv[NC], fD[NC], fRf[NC], ff[NC];          // friction loss of the chain slots
    double lj[2], lv[2], lD[2];      // limits (D = 0: no row)
    double wj[4], wv[4], wD;         // wheel contact pyramid rows (D = 0: no contact)
    double r6j, r6v, l6j, l6v, l6D;  // rows of root dof 6 (lane 0)
};

template <class Q>
FT_HD void quad_ls_eval(const Q& qd, const QChassis& ch, int nch, int ww, const QLs& L, LsPoint& pt, double alpha) {
    double q0 = L.c0, q1 = L.c1, q2 = L.c2;
#pragma unroll
    for (int l = 0; l < NC; l++) {
        const double jar = L.fj[l], jv = L.fv[l], xx = jar + alpha * jv, Rf = L.fRf[l], f = L.ff[l], D = L.fD[l];
        const bool lo = xx <= -Rf, hi = xx >= Rf, lin = lo || hi;
        const double sj = lo ? -1.0 : 1.0;
        q0 += lin ? f * (-0.5 * Rf + sj * jar) : 0.5 * D * jar * jar;
        q1 += lin ? sj * f * jv : D * jar * jv;
        q2 += lin ? 0.0 : 0.5 * D * jv * jv;
    }
#pragma unroll
    for (int k = 0; k < 2; k++) {
        const double D = L.lD[k], jar = L.lj[k], jv = L.lv[k];
        if (D > 0 && jar + alpha * jv < 0) { q0 += 0.5 * D * jar * jar; q1 += D * jar * jv; q2 += 0.5 * D * jv * jv; }
    }
    if (qd.lane() == 0) {
        const double D = qd.K(72), Rf = qd.K(73), f = qd.K(74), jar = L.r6j, jv = L.r6v, xx = jar + alpha * jv;
        const bool lo = xx <= -Rf, hi = xx >= Rf, lin = lo || hi;
        const double sj = lo ? -1.0 : 1.0;
        q0 += lin ? f * (-0.5 * Rf + sj * jar) : 0.5 * D * jar * jar;
        q1 += lin ? sj * f * jv : D * jar * jv;
        q2 += lin ? 0.0 : 0.5 * D * jv * jv;
        const double D6 = L.l6D, j6 = L.l6j, v6 = L.l6v;
        if (D6 > 0 && j6 + alpha * v6 < 0) { q0 += 0.5 * D6 * j6 * j6; q1 += D6 * j6 * v6; q2 += 0.5 * D6 * v6 * v6; }
    }
    if (L.wD > 0) {
#pragma unroll
        for (int rr = 0; rr < 4; rr++) {
            const double jar = L.wj[rr], jv = L.wv[rr];
            if (jar + alpha * jv < 0) { q0 += 0.5 * L.wD * jar * jar; q1 += L.wD * jar * jv; q2 += 0.5 * L.wD * jv * jv; }
        }
    }
    if (nch | ww) { const RareQuad o = rare_ls(ch, nch, ww, alpha); q0 += o.q0; q1 += o.q1; q2 += o.q2; }     // rare contacts (out of line)
    q0 = qd.sum(q0) + L.g0; q1 = qd.sum(q1) + L.g1; q2 = qd.sum(q2) + L.g2;
    pt.alpha = alpha; pt.cost = alpha * alpha * q2 + alpha * q1 + q0;
    pt.d0 = 2 * alpha * q2 + q1; pt.d1 = 2 * q2;
    if (pt.d1 <= 0) pt.d1 = MINVAL;
}

// MuJoCo's PrimalSearch as a state machine: every tick of the warp-uniform loop evaluates the cost once, at the
// point each quad asked for, then each quad moves on by itself (no collectives in the transitions).
template <class Q>
FT_QN double quad_line_search(const Q& qd, QChassis& ch, const QState& st, double scale, bool on, double* mv_r, double* mv_c) {
    QLs L;
    double snorm;
    {
        double sr[NR], sc[NC], xr[NR], xc[NC];
        vec_load(qd, VS, sr, sc);
        double sn = 0;
#pragma unroll
        for (int l = 0; l < NC; l++) sn += sc[l] * sc[l];
        sn = qd.sum(sn);
#pragma unroll
        for (int i = 0; i < NR; i++) sn += sr[i] * sr[i];
        snorm = sqrt(sn);
        quad_mul(qd, VS, mv_r, mv_c);
        double g1 = 0, g2 = 0;
#pragma unroll
        for (int l = 0; l < NC; l++) { g1 += sc[l] * (qd.P(VMA.p + l) - qd.P(VQFS.p + l)); g2 += 0.5 * sc[l] * mv_c[l]; }
        g1 = qd.sum(g1); g2 = qd.sum(g2);
#pragma unroll
        for (int i = 0; i < NR; i++) { g1 += sr[i] * (qd.C(VMA.c + i) - qd.C(VQFS.c + i)); g2 += 0.5 * sr[i] * mv_r[i]; }
        L.g0 = st.gauss; L.g1 = g1; L.g2 = g2;
        vec_load(qd, VX, xr, xc);
        const int w = qd.lane();
#pragma unroll
        for (int l = 0; l < NC; l++) {
            L.fD[l] = qd.K(3 * (6 * w + l)); L.fRf[l] = qd.K(3 * (6 * w + l) + 1); L.ff[l] = qd.K(3 * (6 * w + l) + 2);
            L.fj[l] = xc[l] - qd.P(QP_FRA + l); L.fv[l] = sc[l];
        }
        {
            const double De = qd.P(QP_EQ), der = qd.P(QP_EQ + 2), je = xc[1] - der * xr[6] - qd.P(QP_EQ + 1), ve = sc[1] - der * sr[6];
            L.c0 = 0.5 * De * je * je; L.c1 = De * je * ve; L.c2 = 0.5 * De * ve * ve;
        }
#pragma unroll
        for (int k = 0; k < 2; k++) {
            const double sg = qd.P(QP_LIM + 4 + k);
            L.lD[k] = qd.P(QP_LIM + k); L.lj[k] = sg * xc[k] - qd.P(QP_LIM + 2 + k); L.lv[k] = sg * sc[k];
        }
        {
            const double sg = qd.C(QC_R6 + 3);
            L.r6j = xr[6] - qd.C(QC_R6); L.r6v = sr[6];
            L.l6D = qd.C(QC_R6 + 1); L.l6j = sg * xr[6] - qd.C(QC_R6 + 2); L.l6v = sg * sr[6];
        }
        L.wD = qd.P(QP_WC);
        if (L.wD > 0) {
            double dx[3], ds[3];
            wc_dots(qd, xr, xc, dx); wc_dots(qd, sr, sc, ds);
#pragma unroll
            for (int rr = 0; rr < 4; rr++) {
                const double sg = (rr & 1) ? -WC_MU : WC_MU; const int ta = 1 + (rr >> 1);
                L.wj[rr] = dx[0] + sg * dx[ta] - qd.P(QP_WC + 1 + rr); L.wv[rr] = ds[0] + sg * ds[ta];
            }
        } else {
#pragma unroll
            for (int rr = 0; rr < 4; rr++) { L.wj[rr] = 0; L.wv[rr] = 0; }
        }
        if (st.nch | st.ww) rare_ls_init(qd, ch, st.nch, st.ww);        // (reads x and s from shared memory itself)
    }
    const int nch = st.nch, ww = st.ww;
    const double gtol = SOLVER_TOL * LS_TOL * snorm / scale;
    enum { S_P0, S_P1, S_NEWTON, S_MID, S_A1, S_A2, S_DONE };
    int state = (on && snorm >= MINVAL) ? S_P0 : S_DONE, it = 0;
    double alpha = 0, res = 0, dir = 1;
    bool p2update = false;
    LsPoint p0, p1, p2, pm, a1, pt;
    p0.alpha = p0.cost = p0.d0 = 0; p0.d1 = 1; p1 = p0; p2 = p0; pm = p0; a1 = p0;
    while (qd.wany(state != S_DONE)) {
        quad_ls_eval(qd, ch, nch, ww, L, pt, alpha);
        bool loop1 = false, loop2 = false;
        switch (state) {
        case S_P0:
            p0 = pt; alpha = p0.alpha - p0.d0 / p0.d1; state = S_P1;
            break;
        case S_P1:
            p1 = pt;
            if (p0.cost < p1.cost) p1 = p0;
            if (fabs(p1.d0) < gtol) { res = p1.alpha; state = S_DONE; break; }
            dir = p1.d0 < 0 ? 1.0 : -1.0;
            p2 = p1;
            loop1 = true;
            break;
        case S_NEWTON:
            p1 = pt; it++;
            if (fabs(p1.d0) < gtol) { res = p1.alpha; state = S_DONE; break; }
            loop1 = true;
            break;
        case S_MID:
            pm = pt; it++; alpha = p1.alpha - p1.d0 / p1.d1; state = S_A1;
            break;
        case S_A1:
            a1 = pt; alpha = p2.alpha - p2.d0 / p2.d1; state = S_A2;
            break;
        case S_A2: {
            const LsPoint a2 = pt;
            if (fabs(a1.d0) < gtol) { res = a1.alpha; state = S_DONE; break; }
            if (fabs(a2.d0) < gtol) { res = a2.alpha; state = S_DONE; break; }
            if (fabs(pm.d0) < gtol) { res = pm.alpha; state = S_DONE; break; }
            bool b1 = false, b2 = false;
            double lo = fmin(p1.alpha, p2.alpha), hi = fmax(p1.alpha, p2.alpha);
            for (int cnd = 0; cnd < 3; cnd++) {
                const LsPoint q = cnd == 0 ? a1 : (cnd == 1 ? a2 : pm);
                if (q.alpha <= lo || q.alpha >= hi) continue;
                if ((q.d0 < 0) == (p1.d0 < 0)) { p1 = q; b1 = true; } else { p2 = q; b2 = true; }
                lo = fmin(p1.alpha, p2.alpha); hi = fmax(p1.alpha, p2.alpha);
            }
            if (!b1 && !b2) { res = p1.cost <= p2.cost ? p1.alpha : p2.alpha; state = S_DONE; break; }
            loop2 = true;
            break;
        }
        default: break;
        }
        if (loop1) {                 // while (p1.d0 * dir <= -gtol && it < LS_ITER) { p2 = p1; p1 = newton step from p1 }
            if (p1.d0 * dir <= -gtol && it < LS_ITER) { p2 = p1; p2update = true; alpha = p1.alpha - p1.d0 / p1.d1; state = S_NEWTON; }
            else if (it >= LS_ITER || !p2update) { res = p1.alpha; state = S_DONE; }
            else loop2 = true;
        }
        if (loop2) {                 // bracketing: midpoint and the two Newton steps
            if (it < LS_ITER) { alpha = 0.5 * (p1.alpha + p2.alpha); state = S_MID; }
            else { res = p1.cost <= p2.cost ? p1.alpha : p2.alpha; state = S_DONE; }
        }
    }
    return res;
}

// ---- position + velocity stage of the lane: kinematics, M -> shared memory, bias, smooth force, contacts, rows ----
// WallFn: the height-field walls of the car's track (hfield_contact.cuh rules V and S), or none
struct QNoWalls {                    // open ground
    FT_HD bool enabled() const { return false; }
    FT_HD bool vertex(const double*, QWallHit&) const { return false; }
    FT_HD bool convex(int, const double*, double, const double*, const double*, QWallHit&) const { return false; }
    FT_HD bool bubble_wrap() const { return false; }
    FT_HD bool near_corner(double, double, double, int) const { return false; }
};
struct QHfWalls {                    // walls of one compiled track; bubble: option bubble_wrap (softener spheres collide with them)
    HfView hv; bool on, bubble;
    FT_HD bool enabled() const { return on; }
    FT_HD bool bubble_wrap() const { return bubble; }
    FT_HD bool near_corner(double x, double y, double radius, int k) const { return hf_near_corner(hv, x, y, radius, k); }
    FT_HD bool vertex(const double* p, QWallHit& h) const { return hf_vertex_probe(hv, p, h); }
    FT_HD bool convex(int kind, const double* size, double bound, const double* pos, const double* R, QWallHit& h) const {
        return hf_convex(hv, kind, size, bound, pos, R, h);
    }
};
constexpr double LIDAR_CYL_BOUND = 0.0336;       // > sqrt(0.03^2 + 0.015^2): bounding radius of the lidar cylinder
constexpr double CAR_BOUND = 0.15;               // every geom of the car lies within this distance of the car body's origin, in any pose

template <class Q, class WallFn>
FT_QN void quad_prepare(const Q& qd, const ModelConsts& mc, const double* qr, const double* qc, const double* vr, const double* vc,
                        const double* ctrl, const WallFn& walls, QChassis& ch, QState& st, StepInfo& info) {
    const int w = qd.lane();
    const bool fr = front(w);
    qd.sync();                       // the quad is done with the previous step's shared slots
    // ---- kinematics (root replicated, own wheel chain)
    double q1[4] = {qr[3], qr[4], qr[5], qr[6]}, R1[9];
    quat_norm(q1); quat2mat(R1, q1);
    const double p1[3] = {qr[0], qr[1], qr[2]};
    const double zax[3] = {R1[2], R1[5], R1[8]};
    double p2[3], R2[9];
    { const double c2[3] = {SW_X, 0, SW_Z}; mat_vec3(p2, R1, c2); for (int a = 0; a < 3; a++) p2[a] += p1[a]; }
    { const double cs = cos(qr[7]), sn = sin(qr[7]); const double Rz[9] = {cs, -sn, 0, sn, cs, 0, 0, 0, 1}; mat_mul3(R2, R1, Rz); }
    double pw[3], Rsteer[9], Rw[9], Rs[9], ps[3];
    { const double cw[3] = {wheel_x(w), wheel_y(w), WHEEL_Z + qc[0]}; mat_vec3(pw, R1, cw); for (int a = 0; a < 3; a++) pw[a] += p1[a]; }
    { const double cs = cos(qc[1]), sn = sin(qc[1]); const double Rz[9] = {cs, -sn, 0, sn, cs, 0, 0, 0, 1}; mat_mul3(Rsteer, R1, Rz); }   // rear: angle 0
    { const double cs = cos(qc[2]), sn = sin(qc[2]); const double Ry[9] = {cs, 0, sn, 0, 1, 0, -sn, 0, cs}; mat_mul3(Rw, Rsteer, Ry); }
    {
        double qs[4] = {qc[3], qc[4], qc[5], qc[6]}, Rb[9];
        quat_norm(qs); quat2mat(Rb, qs); mat_mul3(Rs, Rw, Rb);
        const double sc[3] = MUSHR_SOFTENER_CENTER; double t[3];
        mat_vec3(t, Rs, sc);
#pragma unroll
        for (int a = 0; a < 3; a++) ps[a] = pw[a] + t[a];
    }
    double xi1[3], com[3];
    mat_vec3(xi1, R1, mc.ipos1);
    const double mtot = mc.mass1 + SW_MASS + 4 * (WHEEL_MASS + SOFT_MASS);
#pragma unroll
    for (int a = 0; a < 3; a++) {
        xi1[a] += p1[a];
        com[a] = (mc.mass1 * xi1[a] + SW_MASS * p2[a] + qd.sum(WHEEL_MASS * pw[a] + SOFT_MASS * ps[a])) / mtot;
    }
    // spatial inertias about the com
    double cin1[10], cinsw[10], cinw[10], cins[10], d[3];
    const double e0 = (WS1 * WS1 + WS2 * WS2) / 5, e1 = (WS0 * WS0 + WS2 * WS2) / 5, e2 = (WS0 * WS0 + WS1 * WS1) / 5;
    const double is = 0.4 * SOFT_MASS * MUSHR_SOFTENER_RADIUS * MUSHR_SOFTENER_RADIUS;
#pragma unroll
    for (int a = 0; a < 3; a++) d[a] = xi1[a] - com[a];
    inert_com(cin1, mc.inertia1, R1, d, mc.mass1);
#pragma unroll
    for (int a = 0; a < 3; a++) d[a] = p2[a] - com[a];
    inert_com_diag(cinsw, SW_MASS * e0, SW_MASS * e1, SW_MASS * e2, R2, d, SW_MASS);
#pragma unroll
    for (int a = 0; a < 3; a++) d[a] = pw[a] - com[a];
    inert_com_diag(cinw, WHEEL_MASS * e0, WHEEL_MASS * e1, WHEEL_MASS * e2, Rw, d, WHEEL_MASS);
#pragma unroll
    for (int a = 0; a < 3; a++) d[a] = ps[a] - com[a];
    inert_com_diag(cins, is, is, is, Rs, d, SOFT_MASS);
    // motion axes: root rows 0-6 (replicated), chain slots 0-5
    double cdr[NR][6], cd[NC][6], off[3];
#pragma unroll
    for (int p = 0; p < NR; p++) for (int a = 0; a < 6; a++) cdr[p][a] = 0;
#pragma unroll
    for (int l = 0; l < NC; l++) for (int a = 0; a < 6; a++) cd[l][a] = 0;
#pragma unroll
    for (int cc = 0; cc < 3; cc++) cdr[cc][3 + cc] = 1;
#pragma unroll
    for (int a = 0; a < 3; a++) off[a] = com[a] - p1[a];
#pragma unroll
    for (int cc = 0; cc < 3; cc++) { const double ax[3] = {R1[cc], R1[3 + cc], R1[6 + cc]}; for (int a = 0; a < 3; a++) cdr[3 + cc][a] = ax[a]; cross3(cdr[3 + cc] + 3, ax, off); }
#pragma unroll
    for (int a = 0; a < 3; a++) off[a] = com[a] - p2[a];
#pragma unroll
    for (int a = 0; a < 3; a++) cdr[6][a] = zax[a];
    cross3(cdr[6] + 3, zax, off);
#pragma unroll
    for (int a = 0; a < 3; a++) off[a] = com[a] - pw[a];
#pragma unroll
    for (int a = 0; a < 3; a++) cd[0][3 + a] = zax[a];
    if (fr) { for (int a = 0; a < 3; a++) cd[1][a] = zax[a]; cross3(cd[1] + 3, zax, off); }
    { const double ay[3] = {Rsteer[1], Rsteer[4], Rsteer[7]}; for (int a = 0; a < 3; a++) cd[2][a] = ay[a]; cross3(cd[2] + 3, ay, off); }
#pragma unroll
    for (int cc = 0; cc < 3; cc++) { const double ax[3] = {Rs[cc], Rs[3 + cc], Rs[6 + cc]}; for (int a = 0; a < 3; a++) cd[3 + cc][a] = ax[a]; cross3(cd[3 + cc] + 3, ax, off); }
    // ---- composite-rigid-body mass matrix -> shared memory, its border -> Q::mb_store_row
    {
        double crbw[10], crb1[10], buf[6];
#pragma unroll
        for (int a = 0; a < 10; a++) { crbw[a] = cinw[a] + cins[a]; crb1[a] = cin1[a] + cinsw[a] + qd.sum(crbw[a]); }
#pragma unroll
        for (int i = 0; i < 6; i++) {
            inert_mul(buf, crb1, cdr[i]);
#pragma unroll
            for (int j = 0; j <= i; j++) { const double s = dot6q(cdr[j], buf); qd.C(QC_MR + tri(i, j)) = s; }
        }
        inert_mul(buf, cinsw, cdr[6]);
#pragma unroll
        for (int j = 0; j <= 6; j++) { double s = dot6q(cdr[j], buf); if (j == 6) s += dof_armature(6); qd.C(QC_MR + tri(6, j)) = s; }
#pragma unroll
        for (int l = 0; l < NC; l++) {
            inert_mul(buf, l < 3 ? crbw : cins, cd[l]);
#pragma unroll
            for (int kk = 0; kk <= l; kk++) {
                double s = dot6q(cd[kk], buf);
                if (kk == l) s = (l == 1 && !fr) ? 1.0 : s + dof_armature(NR + l);      // rear dummy steering slot: unit diagonal
                qd.P(QP_MW + tri(l, kk)) = s;
            }
            double b[6];
#pragma unroll
            for (int j = 0; j < 6; j++) b[j] = dot6q(cdr[j], buf);
            mb_store_row(qd, l, b);
        }
    }
    // ---- bias forces (recursive Newton-Euler), smooth force
    double bias_r[NR], bias_c[NC];
    {
        double cv1[6] = {0, 0, 0, vr[0], vr[1], vr[2]}, cacc1[6] = {0, 0, 0, 0, 0, GRAV}, dd[6];
        double cvr[6] = {cv1[0], cv1[1], cv1[2], cv1[3], cv1[4], cv1[5]};
#pragma unroll
        for (int cc = 0; cc < 3; cc++) {
            cross_motion(dd, cv1, cdr[3 + cc]);
#pragma unroll
            for (int a = 0; a < 6; a++) { cacc1[a] += dd[a] * vr[3 + cc]; cvr[a] += cdr[3 + cc][a] * vr[3 + cc]; }
        }
#pragma unroll
        for (int a = 0; a < 6; a++) cv1[a] = cvr[a];
        double t[6], t2[6], cfrc1[6], f[6];
        inert_mul(cfrc1, cin1, cacc1);
        inert_mul(t, cin1, cv1); cross_force(t2, cv1, t);
#pragma unroll
        for (int a = 0; a < 6; a++) cfrc1[a] += t2[a];
        {
            double cv[6], ca[6];
            cross_motion(dd, cv1, cdr[6]);
#pragma unroll
            for (int a = 0; a < 6; a++) { ca[a] = cacc1[a] + dd[a] * vr[6]; cv[a] = cv1[a] + cdr[6][a] * vr[6]; }
            inert_mul(f, cinsw, ca);
            inert_mul(t, cinsw, cv); cross_force(t2, cv, t);
#pragma unroll
            for (int a = 0; a < 6; a++) f[a] += t2[a];
            bias_r[6] = dot6q(cdr[6], f);
#pragma unroll
            for (int a = 0; a < 6; a++) cfrc1[a] += f[a];
        }
        double cv[6], ca[6];
#pragma unroll
        for (int a = 0; a < 6; a++) { cv[a] = cv1[a]; ca[a] = cacc1[a]; }
#pragma unroll
        for (int l = 0; l < 3; l++) {                       // rear dummy slot: zero axis and zero velocity
            cross_motion(dd, cv, cd[l]);
#pragma unroll
            for (int a = 0; a < 6; a++) { ca[a] += dd[a] * vc[l]; cv[a] += cd[l][a] * vc[l]; }
        }
        double fw[6];
        inert_mul(fw, cinw, ca);
        inert_mul(t, cinw, cv); cross_force(t2, cv, t);
#pragma unroll
        for (int a = 0; a < 6; a++) fw[a] += t2[a];
        double cvs[6], cas[6];
#pragma unroll
        for (int a = 0; a < 6; a++) { cvs[a] = cv[a]; cas[a] = ca[a]; }
#pragma unroll
        for (int cc = 0; cc < 3; cc++) {
            cross_motion(dd, cv, cd[3 + cc]);
#pragma unroll
            for (int a = 0; a < 6; a++) { cas[a] += dd[a] * vc[3 + cc]; cvs[a] += cd[3 + cc][a] * vc[3 + cc]; }
        }
        double fs[6];
        inert_mul(fs, cins, cas);
        inert_mul(t, cins, cvs); cross_force(t2, cvs, t);
#pragma unroll
        for (int a = 0; a < 6; a++) { fs[a] += t2[a]; fw[a] += fs[a]; cfrc1[a] += qd.sum(fw[a]); }
#pragma unroll
        for (int l = 0; l < NC; l++) bias_c[l] = dot6q(cd[l], l < 3 ? fw : fs);
#pragma unroll
        for (int i = 0; i < 6; i++) bias_r[i] = dot6q(cdr[i], cfrc1);
    }
    {
        double fs_r[NR], fs_c[NC];
#pragma unroll
        for (int i = 0; i < NR; i++) fs_r[i] = -bias_r[i] - dof_damping(i) * vr[i];
#pragma unroll
        for (int l = 0; l < NC; l++) fs_c[l] = -bias_c[l] - dof_damping(NR + l) * vc[l];
        fs_c[0] += -500.0 * (qc[0] - (-0.015));                                           // suspension spring :63
        if (!fr) fs_c[1] = 0;
        fs_r[6] += 20.0 * ctrl[1] - 20.0 * qr[7];                                         // <position kp=20> :179
        const double tv = qd.sum(0.25 * vc[2]);
        double f = 100.0 * ctrl[0] - 100.0 * (0.04 * tv);                                 // <velocity kv=100 gear=0.04> :180
        f = f > 500.0 ? 500.0 : (f < -500.0 ? -500.0 : f);
        fs_c[2] += 0.04 * 0.25 * f;
        vec_store(qd, VQFS, fs_r, fs_c);
        vec_store(qd, VS, fs_r, fs_c);               // right-hand side of qacc_smooth = M^-1 qfrc_smooth
    }
    // ---- rows
    double K, B, imp, R;
#pragma unroll
    for (int l = 0; l < NC; l++) qd.P(QP_FRA + l) = -REF_B * vc[l];
    {
        double a6 = -REF_B * vr[6], D6 = 0, r6 = 0, s6 = 0;
        const double q = qr[7];
        double dist = 0, sign = 0;
        if (q + 1 < 0) { dist = q + 1; sign = 1; } else if (1 - q < 0) { dist = 1 - q; sign = -1; }
        if (sign != 0) {
            kbi(0.9, dist, mc.dof_invweight0[6], K, B, imp, R);
            s6 = sign; D6 = 1 / R; r6 = -B * (sign * vr[6]) - K * imp * dist;
        }
        qd.C(QC_R6) = a6; qd.C(QC_R6 + 1) = D6; qd.C(QC_R6 + 2) = r6; qd.C(QC_R6 + 3) = s6;
    }
    {
        double D = 0, aref = 0, der = 0;
        if (fr) {
            const double x = qr[7], pos = qc[1] - poly_val(w, x);
            der = poly_der(w, x);
            kbi(0.9, pos, mc.dof_invweight0[NR + NC * w + 1] + mc.dof_invweight0[6], K, B, imp, R);
            D = 1 / R; aref = -B * (vc[1] - der * vr[6]) - K * imp * pos;
        }
        qd.P(QP_EQ) = D; qd.P(QP_EQ + 1) = aref; qd.P(QP_EQ + 2) = der;
    }
#pragma unroll
    for (int k = 0; k < 2; k++) {
        double D = 0, aref = 0, sign = 0, dist = 0;
        const double q = qc[k], lo = k == 0 ? -0.03 : -1.0, hi = k == 0 ? 0.0 : 1.0;
        if (!(k == 1 && !fr)) { if (q - lo < 0) { dist = q - lo; sign = 1; } else if (hi - q < 0) { dist = hi - q; sign = -1; } }
        if (sign != 0) {
            kbi(0.9, dist, mc.dof_invweight0[NR + NC * w + k], K, B, imp, R);
            D = 1 / R; aref = -B * (sign * vc[k]) - K * imp * dist;
        }
        qd.P(QP_LIM + k) = D; qd.P(QP_LIM + 2 + k) = aref; qd.P(QP_LIM + 4 + k) = sign;
    }
    // ---- wheel ellipsoid vs ground plane
    {
        const double dl[3] = {-Rw[6], -Rw[7], -Rw[8]};
        double s[3] = {WS0 * dl[0], WS1 * dl[1], WS2 * dl[2]};
        const double nn = sqrt(s[0] * s[0] + s[1] * s[1] + s[2] * s[2]);
        s[0] = WS0 * s[0] / nn; s[1] = WS1 * s[1] / nn; s[2] = WS2 * s[2] / nn;
        double sw[3];
        mat_vec3(sw, Rw, s);
#pragma unroll
        for (int a = 0; a < 3; a++) sw[a] += pw[a];
        const double dist = sw[2] - PLANE_Z;
        const bool on = !(dist > 0);
        double Dw = 0;
        if (on) {
            const double o[3] = {sw[0] - com[0], sw[1] - com[1], sw[2] - 0.5 * dist - com[2]};
            double vel[3] = {vr[2], vr[1], -vr[0]};                       // translation columns of the frame
#pragma unroll
            for (int k = 0; k < 6; k++) {
                const double* ax = k < 3 ? cdr[3 + k] : cd[k - 3];
                double jp[3];
                cross3(jp, ax, o);
#pragma unroll
                for (int a = 0; a < 3; a++) jp[a] += ax[3 + a];
                const double j0 = jp[2], j1 = jp[1], j2 = -jp[0], vk = k < 3 ? vr[3 + k] : vc[k - 3];
                qd.P(QP_CJ + k) = j0; qd.P(QP_CJ + 6 + k) = j1; qd.P(QP_CJ + 12 + k) = j2;
                vel[0] += j0 * vk; vel[1] += j1 * vk; vel[2] += j2 * vk;
            }
            kbi(0.45, dist, mc.wheel_invweight0[w], K, B, imp, R);
            double Rpy = 2 * WC_MU * WC_MU * R; if (Rpy < MINVAL) Rpy = MINVAL;
            Dw = 1 / Rpy;
#pragma unroll
            for (int rr = 0; rr < 4; rr++) {
                const double sg = (rr & 1) ? -1.0 : 1.0;
                qd.P(QP_WC + 1 + rr) = -B * (vel[0] + sg * WC_MU * vel[1 + (rr >> 1)]) - K * imp * dist;
            }
        }
        qd.P(QP_WC) = Dw;
        info.ncon_wheel = popc4(qd.ballot(on));
    }
    // ---- the lane's wheel ellipsoid vs the walls (rule S): one contact, Jacobian over chassis dofs + chain slots 0-2
    st.ww = 0; st.nch = 0;
    info.ncon_wall = 0; info.ncon_ground = 0;
    // (gate: lane k looks at the chunk under corner k of the car's bounding square; most cars are nowhere near a wall)
    // NB the vote is a warp-wide collective: EVERY quad takes part, also one whose car has no walls (a shadowed car)
    const bool near_wall = qd.any(walls.enabled() && walls.near_corner(p1[0], p1[1], CAR_BOUND, w));
    const bool wall_on = walls.enabled() && near_wall;
    info.near_wall = wall_on ? 1 : 0;
    if (qd.wany(wall_on)) {
        if (wall_on) {
            const double wsz[3] = {WS0, WS1, WS2}, ssz[1] = {MUSHR_SOFTENER_RADIUS};
            for (int c = 0; c < (walls.bubble_wrap() ? 2 : 1); c++) {
                QWallHit h;
                // c = 0: wheel ellipsoid (body of the wheel, chain slots 0-2); c = 1: softener sphere behind the ball joint
                // (mushr.em.xml:66, option bubble_wrap: conaffinity 4 against the walls' contype 4; chain slots 0-5)
                const bool hit = c == 0 ? walls.convex(HF_ELLIPSOID, wsz, 0.03, pw, Rw, h)
                                        : walls.convex(HF_SPHERE, ssz, MUSHR_SOFTENER_RADIUS, ps, Rs, h);
                if (!hit) continue;
                st.ww |= 1 << c;
                const int ncol = c == 0 ? 9 : 12;
                const double o[3] = {h.pnt[0] - com[0], h.pnt[1] - com[1], h.pnt[2] - com[2]};
                double vel[3] = {0, 0, 0};
                for (int col = 0; col < 12; col++) {
                    double j0 = 0, j1 = 0, j2 = 0;
                    if (col < ncol) {
                        const double* ax = col < 6 ? cdr[col] : cd[col - 6];
                        double jp[3];
                        cross3(jp, ax, o);
                        for (int a = 0; a < 3; a++) jp[a] += ax[3 + a];
                        j0 = dot3(h.nrm, jp); j1 = dot3(h.t1, jp); j2 = dot3(h.t2, jp);
                        const double vk = col < 6 ? vr[col] : vc[col - 6];
                        vel[0] += j0 * vk; vel[1] += j1 * vk; vel[2] += j2 * vk;
                    }
                    ch.wJ[c][0][col] = j0; ch.wJ[c][1][col] = j1; ch.wJ[c][2][col] = j2;
                }
                kbi(c == 0 ? 0.45 : 0.9, h.dist, c == 0 ? mc.wheel_invweight0[w] : mc.soft_invweight0[w], K, B, imp, R);
                double Rpy = 2 * CH_MU * CH_MU * R; if (Rpy < MINVAL) Rpy = MINVAL;
                ch.wD[c] = 1 / Rpy;
                for (int rr = 0; rr < 4; rr++) {
                    const double sg = (rr & 1) ? -1.0 : 1.0;
                    ch.waref[c][rr] = -B * (vel[0] + sg * CH_MU * vel[1 + (rr >> 1)]) - K * imp * h.dist;
                }
            }
        }
        info.ncon_wall = popc4(qd.ballot(st.ww & 1)) + popc4(qd.ballot(st.ww & 2));
    }
    // ---- contacts of the car body's geoms: candidate c = 2 v (hull vertex v against the walls, rule V), 2 v + 1 (vertex v
    // below the ground plane), 20 (lidar cylinder against the walls, rule S), 21 (cylinder below the ground plane); in that
    // order, the first MAXBODYCON hits count; hit number i goes to lane i & 3, slot i >> 2.
    // Nothing of the body can reach the ground while the bounding box of hull + cylinder stays above the plane:
    const double body_zmin = p1[2] - fabs(R1[6]) * 0.1034 - fabs(R1[7]) * 0.0473 + (R1[8] > 0 ? R1[8] * 0.0151 : R1[8] * 0.0726);
    const bool ground_on = body_zmin < PLANE_Z;
    if (qd.wany(wall_on || ground_on)) {
        const double hull[MUSHR_CHASSIS_NHULL][3] = MUSHR_CHASSIS_HULL;
        const double csz[2] = {0.03, 0.015}, cloc[3] = {-0.0525, 0.0, 0.065 - 0.015 / 2}, down[3] = {0, 0, -1};
        constexpr int NCAND = 2 * MUSHR_CHASSIS_NHULL + 2;
        auto candidate = [&](int c, QWallHit& h) -> bool {
            if (c >= NCAND) return false;
            const bool ground = c & 1;
            if (ground ? !ground_on : !wall_on) return false;
            double p[3];
            if (c < 2 * MUSHR_CHASSIS_NHULL) {
                mat_vec3(p, R1, hull[c >> 1]);
                for (int a = 0; a < 3; a++) p[a] += p1[a];
                return ground ? ground_probe(p, h) : walls.vertex(p, h);
            }
            mat_vec3(p, R1, cloc);
            for (int a = 0; a < 3; a++) p[a] += p1[a];
            if (!ground) return walls.convex(HF_CYLINDER, csz, LIDAR_CYL_BOUND, p, R1, h);
            double sp[3];
            hf_support(HF_CYLINDER, csz, p, R1, down, sp);
            return ground_probe(sp, h);
        };
        unsigned hits = 0;
        for (int k = 0; k < (NCAND + 3) / 4; k++) {
            QWallHit h;
            hits |= qd.ballot(candidate(4 * k + w, h)) << (4 * k);
        }
        if (hits) {
            int rank = 0;
            for (int c = 0; c < NCAND && rank < MAXBODYCON; c++) {
                if (!(hits >> c & 1u)) continue;
                if (c & 1) info.ncon_ground++; else info.ncon_wall++;
                if ((rank & 3) == w) {
                    QWallHit h;
                    candidate(c, h);
                    const int s = st.nch++;
                    double o[3], vel[3] = {0, 0, 0};
                    for (int a = 0; a < 3; a++) o[a] = h.pnt[a] - com[a];
                    for (int col = 0; col < 6; col++) {
                        double jp[3];
                        cross3(jp, cdr[col], o);
                        for (int a = 0; a < 3; a++) jp[a] += cdr[col][3 + a];
                        const double j0 = dot3(h.nrm, jp), j1 = dot3(h.t1, jp), j2 = dot3(h.t2, jp);
                        ch.J[s][0][col] = j0; ch.J[s][1][col] = j1; ch.J[s][2][col] = j2;
                        vel[0] += j0 * vr[col]; vel[1] += j1 * vr[col]; vel[2] += j2 * vr[col];
                    }
                    kbi(0.9, h.dist, mc.chassis_invweight0, K, B, imp, R);
                    double Rpy = 2 * CH_MU * CH_MU * R; if (Rpy < MINVAL) Rpy = MINVAL;
                    ch.D[s] = 1 / Rpy;
                    for (int rr = 0; rr < 4; rr++) {
                        const double sg = (rr & 1) ? -1.0 : 1.0;
                        ch.aref[s][rr] = -B * (vel[0] + sg * CH_MU * vel[1 + (rr >> 1)]) - K * imp * h.dist;
                    }
                }
                rank++;
            }
        }
    }
    qd.sync();                       // per-car slots visible to the quad
}

// state of the lane: root (replicated) + own chain in slot order (susp, steer, throttle, ball)
FT_HD void quad_load(int w, const double* qpos, const double* qvel, double* qr, double* qc, double* vr, double* vc) {
    const int qa = chain_q(w), da = chain_d(w);
    for (int i = 0; i < 8; i++) qr[i] = qpos[i];
    for (int i = 0; i < NR; i++) vr[i] = qvel[i];
    if (front(w)) {
        for (int i = 0; i < 7; i++) qc[i] = qpos[qa + i];
        for (int l = 0; l < NC; l++) vc[l] = qvel[da + l];
    } else {
        qc[0] = qpos[qa]; qc[1] = 0; for (int i = 2; i < 7; i++) qc[i] = qpos[qa + i - 1];
        vc[0] = qvel[da]; vc[1] = 0; for (int l = 2; l < NC; l++) vc[l] = qvel[da + l - 1];
    }
}
FT_HD void quad_store_chain(int w, double* dst, const double* c, int base) {   // 6 chain slots -> dof addresses (rear: no steering dof)
    if (front(w)) { for (int l = 0; l < NC; l++) dst[base + l] = c[l]; }
    else { dst[base] = c[0]; for (int l = 2; l < NC; l++) dst[base + l - 1] = c[l]; }
}

// ---- staged solve: a car that has not converged after `max_rounds` Newton rounds of its CTA is SUSPENDED (its solver
// state -- exactly the shared-memory slots and the border of M plus a few scalars -- goes to a record in global memory) and
// a later launch packs the suspended cars of the whole fleet into fresh CTAs and goes on.  A CTA runs its cars in lock-step,
// so without this every car pays for the slowest of its neighbours: measured mean 2.1 Newton iterations per car,
// 4.5 per CTA (tools/iteration_stats.py).  The arithmetic a car sees does not change (results are bit-identical).
constexpr int QREC_CH = QMAXCH * (1 + 4 + 18), QREC_W1 = 1 + 4 + 36, QREC_WW = 2 * QREC_W1;
constexpr int QREC_LANE = QP_N + QREC_CH + QREC_WW + 2;    // per lane: private slots (border of M included), body contacts, wheel-wall contact, (cost, gauss)
constexpr int QREC_DOUBLES = 4 * QREC_LANE + QC_N + 10;    // + per-car slots + (c0, mask[4], nch[4], ww[4], info) packed below
struct QStage {
    int max_rounds;              // Newton rounds this launch may spend (<= 0: unlimited)
    bool resume;                 // the car's state comes from rec instead of qpos / qvel
    double* rec;                 // this car's record (QREC_DOUBLES doubles), lane-interleaved: element i of lane w at 4 i + w
};

template <class Q>
FT_HD void quad_suspend(const Q& qd, const QChassis& ch, const QState& st, const StepInfo& info, double* rec) {
    const int w = qd.lane();
    for (int i = 0; i < QP_SM_N; i++) rec[4 * i + w] = qd.P(i);      // (the border: quad_suspend_border)
    double* r2 = rec + 4 * QP_N;
    {
        int k = 0;
        for (int s = 0; s < QMAXCH; s++) {                            // (only the contacts that exist travel)
            if (s < st.nch) {
                r2[4 * k++ + w] = ch.D[s];
                for (int rr = 0; rr < 4; rr++) r2[4 * k++ + w] = ch.aref[s][rr];
                for (int a = 0; a < 3; a++) for (int c = 0; c < 6; c++) r2[4 * k++ + w] = ch.J[s][a][c];
            } else k += 1 + 4 + 18;
        }
        for (int c2 = 0; c2 < 2; c2++) {
            if (st.ww >> c2 & 1) {
                r2[4 * k++ + w] = ch.wD[c2];
                for (int rr = 0; rr < 4; rr++) r2[4 * k++ + w] = ch.waref[c2][rr];
                for (int a = 0; a < 3; a++) for (int c = 0; c < 12; c++) r2[4 * k++ + w] = ch.wJ[c2][a][c];
            } else k += QREC_W1;
        }
        r2[4 * k++ + w] = st.cost; r2[4 * k++ + w] = st.gauss;
    }
    double* r3 = rec + 4 * QREC_LANE;
    for (int i = w; i < QC_N; i += 4) r3[i] = qd.C(i);
    double* r4 = r3 + QC_N;
    int* ii = reinterpret_cast<int*>(r4 + 1);
    if (w == 0) {
        r4[0] = st.c0;
        ii[12] = info.iters; ii[13] = info.ncon_wheel; ii[14] = info.ncon_wall; ii[15] = info.reset; ii[16] = info.ncon_ground | (info.near_wall << 8);
    }
    ii[w] = (int)st.mask; ii[4 + w] = st.nch; ii[8 + w] = st.ww;
}
template <class Q>
FT_HD void quad_resume(const Q& qd, QChassis& ch, QState& st, StepInfo& info, const double* rec) {
    const int w = qd.lane();
    for (int i = 0; i < QP_SM_N; i++) qd.P(i) = rec[4 * i + w];      // (the border: quad_resume_border)
    const double* r3 = rec + 4 * QREC_LANE;
    for (int i = 0; i < QC_N; i++) qd.C(i) = r3[i];          // every lane writes the same values
    const double* r4 = r3 + QC_N;
    st.c0 = r4[0];
    const int* ii = reinterpret_cast<const int*>(r4 + 1);
    st.mask = (unsigned)ii[w]; st.nch = ii[4 + w]; st.ww = ii[8 + w];
    info.iters = ii[12]; info.ncon_wheel = ii[13]; info.ncon_wall = ii[14]; info.reset = ii[15]; info.ncon_ground = ii[16] & 0xFF; info.near_wall = ii[16] >> 8;
    const double* r2 = rec + 4 * QP_N;
    {
        int k = 0;
        for (int s = 0; s < QMAXCH; s++) {
            if (s < st.nch) {
                ch.D[s] = r2[4 * k++ + w];
                for (int rr = 0; rr < 4; rr++) ch.aref[s][rr] = r2[4 * k++ + w];
                for (int a = 0; a < 3; a++) for (int c = 0; c < 6; c++) ch.J[s][a][c] = r2[4 * k++ + w];
            } else k += 1 + 4 + 18;
        }
        for (int c2 = 0; c2 < 2; c2++) {
            if (st.ww >> c2 & 1) {
                ch.wD[c2] = r2[4 * k++ + w];
                for (int rr = 0; rr < 4; rr++) ch.waref[c2][rr] = r2[4 * k++ + w];
                for (int a = 0; a < 3; a++) for (int c = 0; c < 12; c++) ch.wJ[c2][a][c] = r2[4 * k++ + w];
            } else k += QREC_W1;
        }
        st.cost = r2[4 * k++ + w]; st.gauss = r2[4 * k++ + w];
    }
}

// The border of M travels with the record as well.  Its accessors are warp collectives, so these two are called by every
// lane of the warp; on: this lane's car is the one suspended / resumed.
template <class Q>
FT_HD void quad_suspend_border(const Q& qd, double* rec, bool on) {
    double* rb = rec + 4 * QP_MB + qd.lane();
#pragma unroll
    for (int l = 0; l < NC; l++) {
        double b[6];
        mb_load_row(qd, l, b);
        if (on) for (int j = 0; j < 6; j++) rb[4 * (6 * l + j)] = b[j];
    }
}
template <class Q>
FT_HD void quad_resume_border(const Q& qd, const double* rec, bool on) {
    const double* rb = rec + 4 * QP_MB + qd.lane();
#pragma unroll
    for (int l = 0; l < NC; l++) {
        double b[6];
        for (int j = 0; j < 6; j++) b[j] = on ? rb[4 * (6 * l + j)] : 0.0;
        mb_store_row(qd, l, b);
    }
}

// ---- the step -----------------------------------------------------------------------------------------------------
// live = false: a padding quad (it re-does the last car so that it can take part in the collectives, and stores
// nothing to global memory)
// (inlined into the one kernel that serves both launches of the staged solve, step.cu)
#define FT_STEP FT_HDN
template <class Q, class WallFn>
FT_STEP bool step_car_quad(const Q& qd, const ModelConsts& mc, double* qpos, double* qvel, double* warm, const double* ctrl,
                          const WallFn& walls, bool live, StepInfo& info, const QStage& stage) {
    const int w = qd.lane();
    const bool fr = front(w);
    const int qa = chain_q(w), da = chain_d(w);
    QChassis ch;
    QState st;
    st.cost = 0; st.gauss = 0; st.mask = 0; st.c0 = 0; st.nch = 0; st.ww = 0;
    info.reset = 0; info.iters = 0; info.ncon_wheel = 0; info.ncon_wall = 0; info.ncon_ground = 0; info.near_wall = 0;
    qd.sync();                                                             // previous step's root state is in memory
    if (stage.resume) {
        if (live) quad_resume(qd, ch, st, info, stage.rec);
        quad_resume_border(qd, stage.rec, live);
        qd.sync();
    } else {
        double qr[8], qc[7], vr[NR], vc[NC];
        quad_load(w, qpos, qvel, qr, qc, vr, vc);
        bool bad = false;                                                  // mj_checkPos / mj_checkVel
        for (int i = 0; i < 8; i++) bad |= bad_value(qr[i]);
        for (int i = 0; i < 7; i++) bad |= bad_value(qc[i]);
        for (int i = 0; i < NR; i++) bad |= bad_value(vr[i]);
        for (int l = 0; l < NC; l++) bad |= bad_value(vc[l]);
        bad = qd.any(bad);
        qd.sync();                                                         // every lane has read the root state
        if (bad) {                                                         // mj_resetData, then the step goes on from qpos0
            info.reset = 1;
            for (int i = 0; i < 8; i++) qr[i] = 0;
            qr[1] = 2.0; qr[3] = 1.0;
            for (int i = 0; i < 7; i++) qc[i] = 0;
            qc[3] = 1.0;
            for (int i = 0; i < NR; i++) vr[i] = 0;
            for (int l = 0; l < NC; l++) vc[l] = 0;
            if (live) {
                if (w == 0) { for (int i = 0; i < 8; i++) qpos[i] = qr[i]; for (int i = 0; i < NR; i++) { qvel[i] = 0; warm[i] = 0; } }
                const int nq = fr ? 7 : 6, nd = fr ? 6 : 5;
                for (int i = 0; i < nq; i++) qpos[qa + i] = (i == nq - 4) ? 1.0 : 0.0;
                for (int i = 0; i < nd; i++) { qvel[da + i] = 0; warm[da + i] = 0; }
            }
        }
        quad_prepare(qd, mc, qr, qc, vr, vc, ctrl, walls, ch, st, info);
    }
    const double scale = 1.0 / (mc.meaninertia * NV);
    // One copy of the factor/solve code serves qacc_smooth (mode 0), every Newton direction (1) and the
    // implicit-damping Euler update (2); mode 3 = finished, waiting for the rest of the CTA.
    // mode 4 = suspended: the CTA has used up this launch's Newton rounds, the car goes on in a later launch.
    int mode = stage.resume ? (live ? 1 : 3) : 0, rounds = 0;
    bool first = !stage.resume;
    for (;;) {
        quad_factor_solve(qd, ch, st, mode >= 3 ? 2 : mode, VS, mode == 1 ? -1.0 : 1.0, mode < 3);
        if (mode == 2) mode = 3;
        if (!first && !qd.cany(mode == 1)) break;
        bool upd = false;
        const bool was_first = first;
        if (first) {
            // warm start if its cost beats qacc_smooth's (mj_fwdConstraint)
            {
                double wr[NR], wc[NC] = {0, 0, 0, 0, 0, 0};
                for (int i = 0; i < NR; i++) wr[i] = warm[i];
                if (fr) { for (int l = 0; l < NC; l++) wc[l] = warm[da + l]; }
                else { wc[0] = warm[da]; for (int l = 2; l < NC; l++) wc[l] = warm[da + l - 1]; }
                if (info.reset) { for (int i = 0; i < NR; i++) wr[i] = 0; for (int l = 0; l < NC; l++) wc[l] = 0; }
                qd.sync();
                vec_store(qd, VX, wr, wc);
            }
            double fr_[NR], fc_[NC]; unsigned m_;
            {
                double mr[NR], mcn[NC];
                quad_mul(qd, VX, mr, mcn);
                qd.sync();
                vec_store(qd, VMA, mr, mcn);
            }
            // S holds qacc_smooth: c0 = qacc_smooth' qfrc_smooth / 2, cost of the warm start and of qacc_smooth
            double c0 = 0, gw = 0;
            for (int l = 0; l < NC; l++) { c0 += qd.P(VS.p + l) * qd.P(VQFS.p + l); gw += qd.P(VX.p + l) * (0.5 * qd.P(VMA.p + l) - qd.P(VQFS.p + l)); }
            c0 = qd.sum(c0); gw = qd.sum(gw);
            for (int i = 0; i < NR; i++) { c0 += qd.C(VS.c + i) * qd.C(VQFS.c + i); gw += qd.C(VX.c + i) * (0.5 * qd.C(VMA.c + i) - qd.C(VQFS.c + i)); }
            st.c0 = 0.5 * c0;
            const double cw = qd.sum(rows_eval(qd, ch, st.nch, st.ww, VX, fr_, fc_, m_)) + (gw + st.c0);
            const double cs = qd.sum(rows_eval(qd, ch, st.nch, st.ww, VS, fr_, fc_, m_));
            double r[NR], c[NC], r2[NR], c2[NC];
            vec_load(qd, VS, r, c); vec_load(qd, VQFS, r2, c2);
            qd.sync();
            vec_store(qd, VX, r, c, cw > cs); vec_store(qd, VMA, r2, c2, cw > cs);
            mode = live ? 1 : 3; first = false;
        } else {
            double xr[NR], xc[NC], mr[NR], mcn[NC];
            const double alpha = quad_line_search(qd, ch, st, scale, mode == 1, mr, mcn);      // mr, mcn: M s
            for (int i = 0; i < NR; i++) { xr[i] = qd.C(VX.c + i) + alpha * qd.C(VS.c + i); mr[i] = qd.C(VMA.c + i) + alpha * mr[i]; }
            for (int l = 0; l < NC; l++) { xc[l] = qd.P(VX.p + l) + alpha * qd.P(VS.p + l); mcn[l] = qd.P(VMA.p + l) + alpha * mcn[l]; }
            upd = mode == 1 && alpha != 0;
            qd.sync();
            vec_store(qd, VX, xr, xc, upd); vec_store(qd, VMA, mr, mcn, upd);
        }
        // cost and gradient (into S) at the new point; a quad that stopped with alpha = 0 gets its gradient back
        const double oldcost = st.cost;
        quad_evaluate(qd, ch, st, mode == 1);
        double gn = 0;
        for (int l = 0; l < NC; l++) gn += qd.P(VS.p + l) * qd.P(VS.p + l);
        gn = qd.sum(gn);
        for (int i = 0; i < NR; i++) gn += qd.C(VS.c + i) * qd.C(VS.c + i);
        if (!was_first && mode == 1) {
            bool done = !upd;                                              // alpha == 0
            if (upd) {
                info.iters++;
                done = scale * (oldcost - st.cost) < SOLVER_TOL || scale * sqrt(gn) < SOLVER_TOL || info.iters >= SOLVER_ITER;
            }
            if (done) mode = 2;
        }
        {
            // mj_Euler with implicit joint damping: (M + h diag(b)) qacc' = qfrc_smooth + qfrc_constraint = M a - grad
            double r[NR], c[NC];
            for (int i = 0; i < NR; i++) r[i] = qd.C(VMA.c + i) - qd.C(VS.c + i);
            for (int l = 0; l < NC; l++) c[l] = qd.P(VMA.p + l) - qd.P(VS.p + l);
            qd.sync();
            vec_store(qd, VS, r, c, mode == 2);
        }
        if (!was_first && stage.max_rounds > 0 && ++rounds >= stage.max_rounds && mode == 1) mode = 4;   // (S = gradient)
    }
    const bool suspended = mode == 4;                                      // the record takes the solver state
    qd.sync();
    if (stage.rec) quad_suspend_border(qd, stage.rec, suspended && live);
    if (suspended && live) quad_suspend(qd, ch, st, info, stage.rec);
    // (a suspended quad still walks through the collectives below with the rest of its warp, then leaves)
    double xr[NR], xc[NC], ar[NR], ac[NC];
    vec_load(qd, VX, xr, xc);
    vec_load(qd, VS, ar, ac);
    bool bad = false;                                                      // mj_checkAcc
    for (int i = 0; i < NR; i++) bad |= bad_value(xr[i]);
    for (int l = 0; l < NC; l++) bad |= bad_value(xc[l]);
    bad = qd.any(bad);
    // ---- velocity, then mj_integratePos with the new velocity (state re-read: it was not kept across the solver)
    double qr[8], qc[7], vr[NR], vc[NC];
    quad_load(w, qpos, qvel, qr, qc, vr, vc);
    qd.sync();                                                             // every lane has re-read the root state
    if (suspended) return true;
    if (bad) {
        info.reset = 1;
        if (!live) return false;
        if (w == 0) { for (int i = 0; i < 8; i++) qpos[i] = (i == 1) ? 2.0 : (i == 3 ? 1.0 : 0.0); for (int i = 0; i < NR; i++) { qvel[i] = 0; warm[i] = 0; } }
        const int nq = fr ? 7 : 6, nd = fr ? 6 : 5;
        for (int i = 0; i < nq; i++) qpos[qa + i] = (i == nq - 4) ? 1.0 : 0.0;
        for (int i = 0; i < nd; i++) { qvel[da + i] = 0; warm[da + i] = 0; }
        return false;
    }
    if (!live) return false;
    for (int i = 0; i < NR; i++) vr[i] += TIMESTEP * ar[i];
    for (int l = 0; l < NC; l++) vc[l] += TIMESTEP * ac[l];
    if (w == 0) {
        for (int a = 0; a < 3; a++) qr[a] += TIMESTEP * vr[a];
        quat_integrate(qr + 3, vr + 3, TIMESTEP);
        qr[7] += TIMESTEP * vr[6];
        for (int i = 0; i < 8; i++) qpos[i] = qr[i];
        for (int i = 0; i < NR; i++) { qvel[i] = vr[i]; warm[i] = xr[i]; }
    }
    for (int l = 0; l < 3; l++) qc[l] += TIMESTEP * vc[l];
    quat_integrate(qc + 3, vc + 3, TIMESTEP);
    if (fr) { for (int i = 0; i < 7; i++) qpos[qa + i] = qc[i]; }
    else { qpos[qa] = qc[0]; for (int i = 2; i < 7; i++) qpos[qa + i - 1] = qc[i]; }
    quad_store_chain(w, qvel, vc, da);
    quad_store_chain(w, warm, xc, da);
    return false;
}

}  // namespace mushr
}  // namespace ftgp
