"""Map compiler: ASCII SSD map + env_args -> static device tables.

Host-side only (NumPy).  Turns the reference's constructor-time Python work
into flat integer tables the sm_100a kernels index directly:

  * wall mask, apple / waste / spawn point lists  (map_env.py:141-146,
    cleanup.py:72-90, harvest.py:30-34 of the reference)
  * base grid in u8 cell codes                    (cleanup.py:117-125, harvest.py:74-77)
  * spawn-probability LUTs as u32 thresholds      (cleanup.py:189-204, harvest.py:13,20-22,118)
  * colour LUT, full or simplified                (map_env.py:33-62, cleanup.py:14-17,92-105,
    harvest.py:37-48)

The maps are the reference's env definitions (constants.py:13-116), stored
run-length encoded: ``<char><count>`` with ``_`` standing for a blank cell.
"""
from __future__ import annotations

import dataclasses
import hashlib
import math
import re
from dataclasses import dataclass, field

import numpy as np

# cell codes (u8) used everywhere on the device
EMPTY, WALL, APPLE, WASTE, RIVER, STREAM, VOID = 0, 1, 2, 3, 4, 5, 6
AGENT_LUT_BASE = 6            # colour index of agent char c (1..9) is 6 + c
CELL_CHARS = " @AHRS"
# orientation index == position in the reference's ORIENTATIONS dict (map_env.py:28-31)
LEFT, RIGHT, UP, DOWN = 0, 1, 2, 3
ORIENT_VEC = np.array([[-1, 0], [1, 0], [0, -1], [0, 1]], dtype=np.float64)

KIND_CLEANUP, KIND_HARVEST = 0, 1
MAX_AGENTS = 16
MAX_CELLS = 2048

_CLEANUP_SMALL = ["@10", "@H2_3P_B@", "@R2_4B2@", "@H2_5B@", "@R2_4B2@", "@H2_P_3B@",
                  "@R2_4B2@", "@H2_5B@", "@R2P_3B2@", "@10"]
_CLEANUP_BAND = ["@R6_5B5@", "@H6_4P_B4@", "@R6_5B5@", "@R5_7B4@", "@R5_6B5@", "@H4_P_6B4@",
                 "@R5_6B5@", "@H6S6B4@", "@H6S6B4@", "@R5_7B4@", "@H5_6B5@", "@R6_4P_B4@",
                 "@H6_5B5@", "@R5_7B4@", "@H4_7B5@", "@R5_5P_B4@", "@H5_6B5@", "@R5_7B4@",
                 "@H4_P_5B5@", "@R5_7B4@", "@H5_6B5@", "@R5_7B4@", "@H4_7B5@"]
_HARVEST = ["@38", "@_P_3P_11P_10P_4P_2@", "@_8A_3A2_9A3_4A_5@", "@_5A_A3_2A3_4A_4A_A2_A4_3@",
            "@_4A3_A_4A_2A_A3_2A_2A_3A_A_3@", "@_4A_A_7A3_A_2A3_12@", "@_6A3_2A3_2A_6A3_3A3_4@",
            "@_3P_6P_10P_6P_3P_3@", "@38"]

_RLE = {
    "cleanup_n3": _CLEANUP_SMALL,
    "cleanup_n5": ["@18"] + _CLEANUP_BAND + ["@18"],
    "cleanup_n10": ["@18"] + _CLEANUP_BAND + _CLEANUP_BAND + ["@18"],   # the n5 interior stacked twice
    "harvest_n10": _HARVEST,
}
# sha256('\n'.join(rows))[:16] of the reference's constants.py maps (checked in tests/golden)
MAP_SHA = {"cleanup_n3": "39e437e90102227f", "cleanup_n5": "2606d82f1b0a400f",
           "cleanup_n10": "336b8343b9f8cd4b", "harvest_n10": "cf5108fcdd596699"}


def _decode_row(rle: str) -> str:
    return "".join((" " if ch == "_" else ch) * int(cnt or 1) for ch, cnt in re.findall(r"(\D)(\d*)", rle))


def ascii_map(key: str) -> list[str]:
    rows = [_decode_row(r) for r in _RLE[key]]
    assert len({len(r) for r in rows}) == 1
    return rows


def map_sha(rows) -> str:
    return hashlib.sha256("\n".join(rows).encode()).hexdigest()[:16]


@dataclass
class EnvParams:
    """What the reference constructors derive from ``map=`` (cleanup.py:31-54, harvest.py:20-22)."""
    kind: int
    map_key: str
    threshold_depletion: float = 0.0
    threshold_restoration: float = 0.0
    waste_spawn_prob: float = 0.0
    apple_respawn_prob: float = 0.0
    spawn_prob: tuple = (0.0, 0.0, 0.0, 0.0)


def params_for(name: str, map_name: str) -> EnvParams:
    if name == "cleanup":
        if map_name == "default3":
            return EnvParams(KIND_CLEANUP, "cleanup_n3", 0.4, 0.0, 0.5, 0.3)
        if map_name == "default10":
            return EnvParams(KIND_CLEANUP, "cleanup_n10", 0.99, 0.0, 0.5, 0.05)
        # "default5" and every other string select the n5 map (cleanup.py:37-54)
        return EnvParams(KIND_CLEANUP, "cleanup_n5", 0.99, 0.0, 0.5, 0.05)
    if name == "harvest":
        # harvest.py:20-22 sets SPAWN_PROB only for "default10"; every other name crashes in the
        # reference (SURVEY D3).  We define those as the module default harvest.py:13.
        sp = (0.0, 0.05, 0.08, 0.1) if map_name == "default10" else (0.0, 0.005, 0.02, 0.05)
        return EnvParams(KIND_HARVEST, "harvest_n10", spawn_prob=sp)
    raise KeyError(name)


def prob_to_threshold(p: float) -> int:
    """u32 threshold T such that  (k / 2**32 < p)  <=>  (k < T)  for integer k in [0, 2**32)."""
    if not p > 0.0:
        return 0
    return min(int(math.ceil(p * 4294967296.0)), 0xFFFFFFFF)


_AGENT_RGB = [(159, 67, 255), (2, 81, 154), (204, 0, 204), (216, 30, 54), (254, 151, 0),
              (205, 155, 155), (99, 99, 255), (250, 204, 255), (238, 223, 16)]
_CELL_RGB_FULL = {EMPTY: (0, 0, 0), WALL: (180, 180, 180), APPLE: (0, 255, 0),
                  WASTE: (99, 156, 194), RIVER: (113, 75, 24), STREAM: (113, 75, 24)}


def color_lut(kind: int, obs_color: str) -> np.ndarray:
    """[16, 3] u8: rows 0-5 cell codes, 6 = outside the map, 6+c = agent drawn as char c."""
    lut = np.zeros((16, 3), dtype=np.uint8)
    if obs_color == "simplified":
        lut[APPLE] = (0, 255, 0)
        if kind == KIND_CLEANUP:
            lut[WASTE] = (255, 0, 0)
        lut[WALL] = (0, 0, 255)
        lut[AGENT_LUT_BASE + 1:AGENT_LUT_BASE + 10] = (0, 0, 255)
    else:
        for code, rgb in _CELL_RGB_FULL.items():
            lut[code] = rgb
        for c in range(1, 10):
            lut[AGENT_LUT_BASE + c] = _AGENT_RGB[c - 1]
    return lut


def agent_char(i: int) -> int:
    """Agent i is drawn as the first char of str(i % 10 + 1) (map_env.py:370 into a <U1 array)."""
    v = i % 10 + 1
    return 1 if v == 10 else v


@dataclass
class MapSpec:
    kind: int
    rows: list
    H: int
    W: int
    n_agents: int
    view: int
    episode_limit: int
    obs_color: str
    params: EnvParams
    fire_cost: int = 1
    hit_penalty: int = 0
    beam_len: int = 5
    tag_timeout: int = 0          # steps an agent hit by a FIRE ray stays off the map; 0 = never (the reference)
    base_grid: np.ndarray = field(default=None, repr=False)
    wall: np.ndarray = field(default=None, repr=False)
    apple_pts: np.ndarray = field(default=None, repr=False)
    waste_pts: np.ndarray = field(default=None, repr=False)
    spawn_pts: np.ndarray = field(default=None, repr=False)
    thr_apple: np.ndarray = field(default=None, repr=False)
    thr_waste: np.ndarray = field(default=None, repr=False)
    thr_harvest: np.ndarray = field(default=None, repr=False)
    lut: np.ndarray = field(default=None, repr=False)
    # a variant's own shaped-reward parameters (compile_variant key "reward_shaping"): (alpha, beta, decay, prosocial) as
    # float32 values when it gives one dict, or None for the handle's; `preferences` holds every agent's full set
    reward_shaping: tuple = None
    # a variant's own preference sets (reward_preferences): one (alpha, beta, decay, prosocial, svo_angle in radians,
    # svo_weight) tuple per agent, or None for the handle's
    preferences: tuple = None

    @property
    def G(self):
        return self.H * self.W

    @property
    def N(self):
        return 2 * self.view + 1

    @property
    def n_actions(self):
        return 9 if self.kind == KIND_CLEANUP else 8

    def ascii_bytes(self) -> bytes:
        return "".join(self.rows).encode()


def compile_map(name: str, map_name: str, n_agents: int, view: int, episode_limit: int,
                obs_color: str = "simplified", rows=None, params: EnvParams | None = None,
                fire_cost: int = 1, hit_penalty: int = 0, tag_timeout: int = 0) -> MapSpec:
    p = params if params is not None else params_for(name, map_name)
    if not 0 <= int(tag_timeout) <= 255:
        raise ValueError("tag_timeout must be in 0..255")
    rows = list(rows) if rows is not None else ascii_map(p.map_key)
    H, W = len(rows), len(rows[0])
    if H * W > MAX_CELLS:
        raise ValueError("map too large")
    if not 1 <= n_agents <= MAX_AGENTS:
        raise ValueError("num_agents out of range")
    flat = np.frombuffer("".join(rows).encode(), dtype=np.uint8)
    ch = lambda c: flat == ord(c)  # noqa: E731
    wall = ch("@")
    spawn = np.flatnonzero(ch("P")).astype(np.int32)
    if len(spawn) < n_agents:
        # map_env.py:783 'There are not enough spawn points! Check your map?'
        raise AssertionError("There are not enough spawn points! Check your map?")
    base = np.zeros(H * W, dtype=np.uint8)
    base[wall] = WALL
    if p.kind == KIND_CLEANUP:
        base[ch("H")] = WASTE
        base[ch("R")] = RIVER
        base[ch("S")] = STREAM
        apple = np.flatnonzero(ch("B")).astype(np.int32)
        waste = np.flatnonzero(ch("H")).astype(np.int32)
    else:
        base[ch("A")] = APPLE
        apple = np.flatnonzero(ch("A")).astype(np.int32)
        waste = np.zeros(0, dtype=np.int32)
    P = len(waste)
    thr_a = np.zeros(P + 1, dtype=np.uint32)
    thr_w = np.zeros(P + 1, dtype=np.uint32)
    for h in range(P + 1):
        density = 1 - (P - h) / P if P > 0 else 0
        if density >= p.threshold_depletion:
            pa, pw = 0.0, 0.0
        else:
            pw = p.waste_spawn_prob
            if density <= p.threshold_restoration:
                pa = p.apple_respawn_prob
            else:
                pa = (1 - (density - p.threshold_restoration)
                      / (p.threshold_depletion - p.threshold_restoration)) * p.apple_respawn_prob
        thr_a[h] = prob_to_threshold(pa)
        thr_w[h] = 0 if abs(pw) <= 1e-8 else prob_to_threshold(pw)     # np.isclose(pW, 0), cleanup.py:177
    thr_h = np.array([prob_to_threshold(x) for x in p.spawn_prob], dtype=np.uint32)
    return MapSpec(kind=p.kind, rows=rows, H=H, W=W, n_agents=n_agents, view=view,
                   episode_limit=episode_limit, obs_color=obs_color, params=p,
                   fire_cost=fire_cost, hit_penalty=hit_penalty, tag_timeout=int(tag_timeout),
                   base_grid=base, wall=wall.astype(np.uint8), apple_pts=apple, waste_pts=waste,
                   spawn_pts=spawn, thr_apple=thr_a, thr_waste=thr_w, thr_harvest=thr_h,
                   lut=color_lut(p.kind, obs_color))


VARIANT_KEYS_COMMON = ("rows", "fire_cost", "hit_penalty", "tag_timeout", "reward_shaping")
VARIANT_KEYS = {KIND_CLEANUP: VARIANT_KEYS_COMMON + ("threshold_depletion", "threshold_restoration", "waste_spawn_prob",
                                                    "apple_respawn_prob"),
                KIND_HARVEST: VARIANT_KEYS_COMMON + ("spawn_prob",)}


def compile_variant(base: MapSpec, overrides: dict) -> MapSpec:
    """One env variant (``ssd_set_variants``): ``base`` (the handle's creation spec) with ``overrides`` applied.  Keys:
    ``rows`` (an ASCII layout of base's exact H x W), ``fire_cost``, ``hit_penalty``, ``tag_timeout``, and the spawn
    dynamics of the kind -- Cleanup ``threshold_depletion``, ``threshold_restoration``, ``waste_spawn_prob``,
    ``apple_respawn_prob``; Harvest ``spawn_prob`` (4 probabilities); ``reward_shaping`` (a ``reward_shaping`` dict, or a
    list of one per agent, see ``reward_preferences``; absent: the handle's).  ``{}`` is the base config.  Everything else (kind, size, view, agents, episode limit,
    colours) stays the handle's."""
    ov = dict(overrides or {})
    allowed = VARIANT_KEYS[base.kind]
    other = set(VARIANT_KEYS[KIND_HARVEST if base.kind == KIND_CLEANUP else KIND_CLEANUP]) - set(allowed)
    for key in ov:
        if key in other:
            kind = "cleanup" if base.kind == KIND_CLEANUP else "harvest"
            raise ValueError(f"variant key {key!r} does not apply to {kind}")
        if key not in allowed:
            raise ValueError(f"unknown variant key {key!r}; allowed: {sorted(allowed)}")
    rows = list(ov.pop("rows", base.rows))
    if len(rows) != base.H or any(len(r) != base.W for r in rows):
        raise ValueError(f"variant rows must be {base.H} rows of {base.W} characters")
    pk = {k: ov.pop(k) for k in list(ov) if k not in VARIANT_KEYS_COMMON}
    if "spawn_prob" in pk:
        sp = tuple(float(x) for x in pk["spawn_prob"])
        if len(sp) != 4:
            raise ValueError("spawn_prob needs 4 probabilities")
        pk["spawn_prob"] = sp
    params = dataclasses.replace(base.params, **{k: (v if k == "spawn_prob" else float(v)) for k, v in pk.items()})
    spec = compile_map("", "", base.n_agents, base.view, base.episode_limit, obs_color=base.obs_color, rows=rows,
                       params=params, fire_cost=int(ov.get("fire_cost", base.fire_cost)),
                       hit_penalty=int(ov.get("hit_penalty", base.hit_penalty)),
                       tag_timeout=int(ov.get("tag_timeout", base.tag_timeout)))
    if "reward_shaping" in ov:
        spec.preferences = reward_preferences(ov["reward_shaping"], base.n_agents)
        if isinstance(ov["reward_shaping"], dict):
            spec.reward_shaping = spec.preferences[0][:4]
    return spec


# Shaped rewards (ssd_set_reward_shaping; DESIGN.md §3 item 17): inequity aversion (Hughes et al., 2018) and prosocial mixing
# (Peysakhovich & Lerer, 2018).  The default decay is Hughes' gamma * lambda = 0.99 * 0.975, in float32.  Item 20
# (ssd_set_reward_preferences) adds a social value orientation (McKee et al., 2020): a target reward angle svo_angle, given in
# degrees (0 individualistic, 45 prosocial, 90 altruistic) and kept in float32 radians, and its weight svo_weight.
SHAPING_KEYS = ("alpha", "beta", "decay", "prosocial")
SHAPING_DEFAULTS = {"alpha": 0.0, "beta": 0.0, "decay": float(np.float32(0.99 * 0.975)), "prosocial": 0.0}
PREFERENCE_KEYS = SHAPING_KEYS + ("svo_angle", "svo_weight")


def preference(params: dict) -> tuple:
    """``(alpha, beta, decay, prosocial, svo_angle, svo_weight)`` as float32 values from one ``reward_shaping`` dict (svo_angle
    converted once from degrees to radians): unknown keys are refused, missing ones take ``SHAPING_DEFAULTS`` (svo_angle and
    svo_weight 0); every value must be finite, alpha, beta and svo_weight >= 0, decay and prosocial in [0, 1], svo_angle in
    [-180, 180] degrees."""
    if not isinstance(params, dict):
        raise ValueError(f"reward_shaping needs a dict of {list(PREFERENCE_KEYS)}, got {params!r}")
    unknown = set(params) - set(PREFERENCE_KEYS)
    if unknown:
        raise ValueError(f"unknown reward_shaping keys {sorted(unknown)}; allowed: {list(PREFERENCE_KEYS)}")
    with np.errstate(over="ignore"):                        # a value past the float32 range becomes inf and is refused below
        vals = tuple(float(np.float32(params.get(k, SHAPING_DEFAULTS[k]))) for k in SHAPING_KEYS)
        deg, weight = float(params.get("svo_angle", 0.0)), float(np.float32(params.get("svo_weight", 0.0)))
    alpha, beta, decay, prosocial = vals
    if not all(math.isfinite(v) for v in vals) or alpha < 0 or beta < 0 or not 0 <= decay <= 1 or not 0 <= prosocial <= 1:
        raise ValueError("reward_shaping needs finite alpha, beta >= 0 and decay, prosocial in [0, 1], got "
                         f"{dict(zip(SHAPING_KEYS, vals))}")
    if not (math.isfinite(deg) and -180 <= deg <= 180 and math.isfinite(weight) and weight >= 0):
        raise ValueError(f"reward_shaping needs svo_angle in [-180, 180] degrees and a finite svo_weight >= 0, got {deg}, {weight}")
    return vals + (float(np.float32(math.radians(deg))), weight)


def reward_shaping(params: dict) -> tuple:
    """``(alpha, beta, decay, prosocial)`` of one ``reward_shaping`` dict, validated as ``preference`` validates it."""
    return preference(params)[:4]


def reward_preferences(value, n_agents: int) -> tuple:
    """Every agent's preference set (``preference``) from a ``reward_shaping`` value: one dict for every agent, or a list of
    ``n_agents`` dicts, one per agent."""
    if isinstance(value, dict):
        return (preference(value),) * n_agents
    if not isinstance(value, (list, tuple)) or len(value) != n_agents:
        raise ValueError(f"reward_shaping needs one dict or a list of {n_agents} dicts (one per agent), got {value!r}")
    return tuple(preference(d) for d in value)


def dump_maps() -> str:
    """The four shipped maps as plain ASCII (what the run-length rows above decode to), for auditing against
    ``src/envs/ssd/constants.py``:  python -m homophily_marl_b200.mapspec"""
    out = []
    for key in _RLE:
        rows = ascii_map(key)
        out.append(f"{key}  {len(rows)}x{len(rows[0])}  sha {map_sha(rows)}")
        out.extend("  |" + r + "|" for r in rows)
    return "\n".join(out)


if __name__ == "__main__":
    print(dump_maps())
