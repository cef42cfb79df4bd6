"""Reward-parameter sets for the lock-step tests, and a restatement of the rules by which nav3d_set_reward_params rejects a
set (include/nav3d.h, nav3d_reward_params)."""
import math

from oracle.c_oracle import REWARD_DEFAULTS, REWARD_FIELDS

INT32_MAX = 2 ** 31 - 1


def centi(v: float) -> int:
    """One reward term in 1/100 units: v * 100 in f64, rounded half away from zero."""
    return int(v * 100.0 + (-0.5 if v < 0 else 0.5))


def full(p: dict) -> dict:
    return dict(REWARD_DEFAULTS, **p)


def rejects(p: dict):
    """'saturation', 'overflow' or None for the set `p` (unnamed fields at the reference's values)."""
    p = full(p)
    u, cap = p["revisit_unit"], p["revisit_cap"]
    if not (u == 0.0 or (u > 0.0 and 255.0 * u >= cap)):
        return "saturation"
    rev = max(abs(centi(min(u, cap))), abs(centi(min(255.0 * u, cap))))
    per_step = (abs(centi(p["step_cost"])) + rev + abs(centi(p["near_wall_bonus"]))
                + max(abs(centi(p["repeat_bonus"])), abs(centi(p["reverse_penalty"]))) + abs(centi(p["explore_bonus"])))
    if 65535 * per_step + abs(centi(p["finish_bonus"])) + abs(centi(p["truncation_penalty"])) > INT32_MAX:
        return "overflow"
    return None


def _explore_bound_cents() -> int:
    """The largest explore_bonus, in 1/100 units, that the overflow rule accepts with every other field at its default."""
    d = REWARD_DEFAULTS
    rest = (abs(centi(d["step_cost"])) + abs(centi(min(255 * d["revisit_unit"], d["revisit_cap"]))) +
            abs(centi(d["near_wall_bonus"])) + max(abs(centi(d["repeat_bonus"])), abs(centi(d["reverse_penalty"]))))
    return (INT32_MAX - abs(centi(d["finish_bonus"])) - abs(centi(d["truncation_penalty"]))) // 65535 - rest


def _unit_bound(cap: float) -> float:
    """The smallest revisit_unit with 255.0 * unit >= cap in f64."""
    u = cap / 255.0
    while 255.0 * u < cap:
        u = math.nextafter(u, math.inf)
    while 255.0 * math.nextafter(u, 0.0) >= cap:
        u = math.nextafter(u, 0.0)
    return u


EXPLORE_MAX = _explore_bound_cents() / 100.0
UNIT_MIN = _unit_bound(1.0)

# (id, overrides): the defaults, every field doubled and sign-flipped one at a time, a set that is not in whole cents,
# the revisit term switched off two ways, and sets just inside and just outside each rejection rule
SETS = [("defaults", {})]
for _f in REWARD_FIELDS:
    SETS.append((f"{_f}_x2", {_f: 2 * REWARD_DEFAULTS[_f]}))
    SETS.append((f"{_f}_neg", {_f: -REWARD_DEFAULTS[_f]}))
SETS += [
    ("non_centi", {"step_cost": -0.005, "revisit_unit": 0.004, "near_wall_bonus": 0.125}),
    ("cap0", {"revisit_cap": 0.0}),
    ("unit0", {"revisit_unit": 0.0}),
    ("unit_1e6", {"revisit_unit": 1e6}),                                   # the cap bounds the term: accepted
    ("saturation_in", {"revisit_unit": UNIT_MIN, "revisit_cap": 1.0}),
    ("saturation_out", {"revisit_unit": math.nextafter(UNIT_MIN, 0.0), "revisit_cap": 1.0}),
    ("saturation_unit_0.001", {"revisit_unit": 0.001, "revisit_cap": 1.0}),
    ("overflow_in", {"explore_bonus": EXPLORE_MAX}),
    ("overflow_out", {"explore_bonus": EXPLORE_MAX + 0.01}),
    ("overflow_explore_1e6", {"explore_bonus": 1e6}),
]
ACCEPTED = [(k, p) for k, p in SETS if rejects(p) is None]
REJECTED = [(k, p) for k, p in SETS if rejects(p) is not None]
