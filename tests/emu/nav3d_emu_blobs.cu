// nav3d_emu_blobs.cu — DEBUGGING AID, tests only.  The env-state blob calls (nav3d_save_envs / nav3d_load_envs) in the host
// emulation: the same per-env copy functions of csrc/nav3d_core.cuh that the kernels run, one lane per env.  Built as its
// own library around nav3d_emu.cu (tests/emu_blobs.py), so it takes the handles emu_create returns.
#include "nav3d_emu.cu"

extern "C" {

// The engine signature of the rooms an Emu was created from (nav3d_load_rooms computes the same for a real engine; the
// emulation has no fixed start cells).
unsigned long long emu_signature(void *h, int n_rooms, const int *dims, const int8_t *dense, const unsigned *dense_off,
                                 int wall_code) {
    const Emu *e = (const Emu *)h;
    unsigned long long sig = sig_engine(e->simple ? 1 : 0, e->P.L, e->P.env_stride);
    for (int r = 0; r < n_rooms; r++)
        sig = sig_room(sig, dims[3 * r], dims[3 * r + 1], dims[3 * r + 2], wall_code, dense + dense_off[r], 0xffffffffu);
    return sig;
}
long emu_env_state_bytes(void *h) { return (long)blob_bytes(((Emu *)h)->P); }
void emu_save_envs(void *h, unsigned long long sig, const int *env_ids, int n, const float *obs, uint8_t *blobs) {
    Emu *e = (Emu *)h;
    const unsigned long long B = blob_bytes(e->P);
    for (int i = 0; i < n; i++) save_env_lane(e->P, sig, env_ids ? env_ids[i] : i, obs, blobs + (size_t)i * B, 0, 1);
}
// Under NAV3D_EMU_ASAN the destination env is fenced to the blob's room before the copy, as a reset fences it to its new room.
void emu_load_envs(void *h, unsigned long long sig, const int *env_ids, int n, const uint8_t *blobs, float *obs,
                   uint8_t *status) {
    Emu *e = (Emu *)h;
    const unsigned long long B = blob_bytes(e->P);
    for (int i = 0; i < n; i++) {
        const int env = env_ids ? env_ids[i] : i;
        const uint8_t *blob = blobs + (size_t)i * B;
        const uint8_t st = blob_status(e->P, sig, env, blob);
        if (status) status[i] = st;
        if (st != kBlobLoaded) continue;
        if (!e->simple) fence_env(e, env, reinterpret_cast<const BlobHeader *>(blob)->room);
        load_env_lane(e->P, env, blob, obs, 0, 1);
    }
}
}
