#!/bin/bash
# The device source (csrc/nav3d_core.cuh) compiled for the host under AddressSanitizer + UBSan, every env fenced to the part
# of its knowledge block its current room owns (tests/emu/nav3d_emu.cu: fence_env), driven through the edge-case and
# lock-step tests of tests/test_emu_vs_oracle.py, the env-state blob scenarios of tests/test_env_states_host.py and the
# fused-rollout equivalence tests of tests/test_rollout_actions_host.py and the reward-parameter lock-step tests of
# tests/test_reward_params_host.py (UBSan traps a wrapping episode-return accumulator) and the weighted room-draw scenarios
# of tests/test_room_weights_host.py (the table builder's arithmetic and the binary-search draw).  Stands
# in for compute-sanitizer memcheck/initcheck, which the GPU pool refuses to run.  usage: tools/emu_asan.sh [pytest args]   -> exit code 0 = no report
cd "$(dirname "$0")/.."
export NAV3D_EMU_ASAN=1 ASAN_OPTIONS=detect_leaks=0:halt_on_error=1:abort_on_error=0 UBSAN_OPTIONS=print_stacktrace=1
python -c "import sys; sys.path.insert(0, 'tests'); sys.path.insert(0, '.'); import _nav3d_path, emu_harness, emu_blobs, emu_rollout, emu_weights; emu_harness.build(); emu_blobs.build(); emu_rollout.build(); emu_weights.build()" || exit 2   # build (nvcc must not run under the preload)
LD_PRELOAD=$(gcc -print-file-name=libasan.so):$(gcc -print-file-name=libubsan.so) python -m pytest tests/test_emu_vs_oracle.py tests/test_env_states_host.py tests/test_rollout_actions_host.py tests/test_reward_params_host.py tests/test_room_weights_host.py -x -q "$@"
rc=$?
# negative control: one byte past the K bricks an env owns must be reported (proves the fence and the runtime are live)
LD_PRELOAD=$(gcc -print-file-name=libasan.so):$(gcc -print-file-name=libubsan.so) python - <<'PY' 2>&1 | grep -q "AddressSanitizer: use-after-poison" && echo "negative control: out-of-fence read reported by AddressSanitizer (as it must be)" || { echo "negative control FAILED: the fence did not trigger"; rc=3; }
import ctypes as C, sys
sys.path.insert(0, "tests"); sys.path.insert(0, ".")
import _nav3d_path
from pathlib import Path
from emu_harness import EmuEngine, lib
from nav3d.rooms import load_room_dir
e = EmuEngine(4, load_room_dir(Path("rooms/P1_training"), sort=True), L=10)
e.reset()
L = lib()
L.emu_owned_k_bytes.restype = C.c_long; L.emu_owned_k_bytes.argtypes = [C.c_void_p, C.c_int]
L.emu_probe.argtypes = [C.c_void_p, C.c_int, C.c_long]
small = min(range(4), key=lambda i: L.emu_owned_k_bytes(e.h, i))
L.emu_probe(e.h, small, L.emu_owned_k_bytes(e.h, small))
PY
exit $rc
