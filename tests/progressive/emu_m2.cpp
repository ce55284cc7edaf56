// emu_m2.cpp -- TEST HELPER: host (g++) build of accumulate_m2_slot (csrc/sqt_paths.cuh), the per-slot function of
// k_accumulate_m2, so that a CPU test can compare it with the oracle's range render.
#include "../../squigly-trace_b200/csrc/sqt_paths.cuh"

using namespace sqt;

extern "C" {

// one round: samples [k0, k1) of every pixel of a single-rank frame, sbuf ks-major ([k1 - k0][npix][3])
void emu_accumulate_m2(int rows, int cols, int spp, const float *sbuf, int k0, int k1, float *accum, float *m2) {
    RenderParams p = {};
    p.rows = rows; p.cols = cols; p.spp = spp; p.world = 1;
    const long long npix = (long long)rows * cols;
    RoundInfo rd = {};
    rd.pixel_list = nullptr; rd.prim = nullptr;
    rd.sbuf = const_cast<float *>(sbuf);
    rd.n_slots = npix; rd.slot_stride = npix;
    rd.k0 = k0; rd.k1 = k1;
    for (long long slot = 0; slot < npix; ++slot) accumulate_m2_slot(p, rd, slot, accum, m2);
}

}
