// TEST-ONLY: the warp-of-quads host harness of step_quad_host.cpp with a communicator policy that keeps the border of M
// the way the device does: outside the private slots, reached only through mb_load_row / mb_store_row, and both are
// collectives (a barrier over the whole host "warp", like the device's tcgen05.ld / st over the 32 lanes).  A call site
// that not every quad of the warp reaches dead-locks here instead of on a GPU.  The private border slots QP_MB.. are
// filled with NaN, so any read of the border that bypasses the accessors changes the results.  Between the two launches
// the border of a suspended car is scribbled over: it has to come back from the record.
// hq_step_warp4 of this library is the border-policy version; the included file's own is renamed out of the way.
#define hq_step_warp4 hq_step_warp4_slots
#include "step_quad_host.cpp"
#undef hq_step_warp4
#include <cmath>

template <int NQ_>
struct WarpQuadHostBorder : WarpQuadHost<NQ_> {
    std::vector<double>* mb;                                           // [36 x 4 NQ] like the device's TMEM columns x lanes
    void mb_load_row(int l, double* b) const {
        this->s->bar.wait();
        for (int j = 0; j < 6; j++) b[j] = (*mb)[(size_t)(6 * l + j) * this->PS + this->tid];
    }
    void mb_store_row(int l, const double* b) const {
        this->s->bar.wait();
        for (int j = 0; j < 6; j++) (*mb)[(size_t)(6 * l + j) * this->PS + this->tid] = b[j];
    }
};
static_assert(HasMbRows<WarpQuadHostBorder<4>>::value && !HasMbRows<WarpQuadHost<4>>::value, "policy detection");

template <int NQ_>
static int warp_step_border(double* qpos, double* qvel, double* warm, const double* ctrl, int* info4, int k1) {
    WarpHostShared sh; sh.bar.nthreads = 4 * NQ_; sh.nq = NQ_;
    sh.slot.assign(4 * NQ_, 0); sh.bits.assign(4 * NQ_, 0); sh.priv.assign((size_t)QP_N * 4 * NQ_, 0); sh.shr.assign((size_t)QC_N * NQ_, 0);
    for (size_t k = (size_t)QP_MB * 4 * NQ_; k < sh.priv.size(); k++) sh.priv[k] = NAN;
    std::vector<double> mb((size_t)(QP_N - QP_MB) * 4 * NQ_, 0);
    for (int g = 0; g < 25; g++) quad_const_entry(g_mc, g, sh.ktab);
    std::vector<double> recs((size_t)QREC_DOUBLES * NQ_);
    std::vector<int> suspended(NQ_, 0);
    std::vector<std::thread> th;
    for (int tid = 0; tid < 4 * NQ_; tid++)
        th.emplace_back([&, tid]() {
            WarpQuadHostBorder<NQ_> q; q.s = &sh; q.tid = tid; q.w = tid & 3; q.quad = tid >> 2; q.mb = &mb;
            const int i = q.quad;
            StepInfo si;
            bool sus = step_car_quad(q, g_mc, qpos + i * NQ, qvel + i * NV, warm + i * NV, ctrl + 2 * i, g_walls, true, si,
                                     QStage{k1, false, recs.data() + (size_t)i * QREC_DOUBLES});
            q.sync();
            if (q.w == 0) suspended[i] = sus;
            if (sus) for (int k = 0; k < QP_N - QP_MB; k++) mb[(size_t)k * q.PS + tid] = -5e55;
            q.sync();
            bool anysus = false; for (int c = 0; c < NQ_; c++) anysus |= suspended[c] != 0;
            if (anysus) {
                StepInfo s2;
                const bool live = suspended[i] != 0;
                step_car_quad(q, g_mc, qpos + i * NQ, qvel + i * NV, warm + i * NV, ctrl + 2 * i, g_walls, live, s2,
                              QStage{0, true, recs.data() + (size_t)i * QREC_DOUBLES});
                if (live) si = s2;
                q.sync();
            }
            if (info4 && q.w == 0) { info4[4 * i] = si.iters; info4[4 * i + 1] = si.ncon_wheel; info4[4 * i + 2] = si.ncon_wall; info4[4 * i + 3] = si.reset; }
        });
    for (auto& t2 : th) t2.join();
    int ns = 0; for (int c = 0; c < NQ_; c++) ns += suspended[c];
    return ns;
}
extern "C" int hq_step_warp4(double* qpos, double* qvel, double* warm, const double* ctrl, int* info4, int k1) {
    if (!g_ready) { g_mc = model_constants(); g_ready = true; }
    return warp_step_border<4>(qpos, qvel, warm, ctrl, info4, k1);
}
