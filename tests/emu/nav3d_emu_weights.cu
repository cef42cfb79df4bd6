// nav3d_emu_weights.cu — DEBUGGING AID, tests only.  nav3d_set_room_weights in the host emulation: the room-draw table is
// built with the per-element arithmetic of csrc/nav3d_core.cuh (room_weight_ok / room_weight_q / room_cdf_entry), one room
// after the other, and hung on the emulated engine's EngineParams::cdf, where reset_picks and simple_reset_env_philox read
// it through draw_room.  An engine that emu_create made and that was never given a table draws uniformly.  Built as its own
// library around nav3d_emu.cu (tests/emu_weights.py), so it takes the handles emu_create returns.
#include "nav3d_emu.cu"

extern "C" {

// weights NULL = the uniform table; returns the status (0 installed, 1 rejected, table unchanged)
int emu_set_room_weights(void *h, const float *w) {
    Emu *e = (Emu *)h;
    const uint32_t n = (uint32_t)e->P.n_rooms;
    unsigned long long *cdf = const_cast<unsigned long long *>(e->P.cdf);
    if (w) {
        bool bad = false;
        uint32_t mx = 0;
        for (uint32_t j = 0; j < n; j++) { bad |= !room_weight_ok(w[j]); mx = std::max(mx, room_weight_bits(w[j])); }
        if (bad || mx == 0) return 1;
    }
    if (!cdf) cdf = new unsigned long long[n];
    if (!w) {
        for (uint32_t j = 0; j < n; j++) cdf[j] = room_cdf_uniform(j, n);
    } else {
        uint32_t mx = 0;
        for (uint32_t j = 0; j < n; j++) mx = std::max(mx, room_weight_bits(w[j]));
        float w_max;
        std::memcpy(&w_max, &mx, 4);
        unsigned long long total = 0, c = 0;
        for (uint32_t j = 0; j < n; j++) total += room_weight_q(w[j], w_max);
        for (uint32_t j = 0; j < n; j++) { c += room_weight_q(w[j], w_max); cdf[j] = room_cdf_entry(c, total); }
    }
    e->P.cdf = cdf;
    return 0;
}
// the table the draws use: the installed one, or the uniform one when none is
void emu_get_room_cdf(void *h, unsigned long long *out) {
    Emu *e = (Emu *)h;
    const uint32_t n = (uint32_t)e->P.n_rooms;
    for (uint32_t j = 0; j < n; j++) out[j] = e->P.cdf ? e->P.cdf[j] : room_cdf_uniform(j, n);
}
void emu_free_room_cdf(void *h) {
    Emu *e = (Emu *)h;
    delete[] e->P.cdf;
    e->P.cdf = nullptr;
}
}
