"""Lattices at and just past every size limit the step kernels dispatch on, the dispatch rule restated in Python,
and the device-vs-oracle matrix that runs them (tests/test_gpu_geometry_edges.py; checked on CPU by
tests/test_geometry_edges_cpu.py).

The limits (a padded lattice is (W+3) x (H+3): the grid points 0..W x 0..H plus a ring of walls):

* ``cc_step_tpe2_kernel`` (small lattices, one-byte cells, a per-cell table): padded width PW <= 32, padded height
  PH <= 16, PW * PH <= 256 (``tpe2_eligible``, csrc/cc_launch_tpe.cu:93-99; ``kT2Max*``, cc_kernel_tpe2.cuh:34).
* ``cc_step_tpe_kernel``, greedy / waiting policies: the occupancy of the lattice is one word per row when PW <= 32
  and PH <= bm_cap, a linear bitmap of ``walk_words = ceil(PW * PH / 32)`` words when walk_words <= bm_cap, and
  register compares otherwise (``launch_tpe_t``, csrc/cc_launch_tpe.cu:25-32).  bm_cap is ``kTpeMaxBitmapWords`` = 16,
  except for float32 rows of even crews, whose bitmap aliases the warp's ring of TMA images:
  ``min(kImgRing * kImgBytes / 128, 16)`` = ``min(3 * A * (3 + 2A) * 8 / 128, 16)``: A=2 -> 2, A=4 -> 8, A=6/8 -> 16.
* every lattice: coordinates up to ``kMaxGeom`` = 120, walk maps up to ``kMaxWalkWords`` = 512 words and reward-table
  indices below ``kRtabSize`` = 400 (cc_kernels.cuh:386-390).
"""

from __future__ import annotations

from dataclasses import dataclass, field

from cases import unchecked

from collectivecrossing_b200.reward_configs import (
    BinaryRewardConfig,
    ConstantNegativeRewardConfig,
    DefaultRewardConfig,
    SimpleDistanceRewardConfig,
)
from collectivecrossing_b200.terminated_configs import (
    AllAtDestinationTerminatedConfig,
    IndividualAtDestinationTerminatedConfig,
)
from collectivecrossing_b200.truncated_configs import MaxStepsTruncatedConfig

# limits of the kernels, as in the sources cited above
T2_MAX_COLS, T2_MAX_ROWS, T2_MAX_CELLS = 32, 16, 256          # cc_kernel_tpe2.cuh:34
TPE_MAX_BITMAP_WORDS = 16                                     # cc_kernel_tpe.cuh:44
TPE_IMG_RING = 3                                              # cc_kernel_tpe.cuh:72
MAX_GEOM, MAX_WALK_WORDS, RTAB_SIZE, Y_BIAS = 120, 512, 400, 128   # cc_kernels.cuh:386-390
NP_RESET = 0x100                                              # ccb::kNpReset, OR-ed into the OBS template argument
OBS_CODE = {"none": 0, "int8": 1, "float32": 4, "table": 16}  # CC_OBS_*


@dataclass(frozen=True)
class Lattice:
    """One named lattice: the config fields that fix its geometry, the limit it pins, and the crews it runs with."""

    name: str
    width: int
    height: int
    division_y: int
    door: tuple[int, int]                      # door posts relative to the tram's left wall
    tram_length: int
    boarding_y: int
    exiting_y: int
    padded: tuple[int, int]                    # (PW, PH) the lattice is named for
    pins: str
    crews: tuple[tuple[int, int], ...]         # (boarding, exiting) crews of the device matrix
    reward: str = "default"
    term: str = "individual"
    max_steps: int = 16
    big_crews: tuple[tuple[int, int], ...] = field(default=())   # crews above 8 (lane-group kernel only)

    def config(self, boarding: int, exiting: int):
        return unchecked(
            width=self.width, height=self.height, division_y=self.division_y, tram_door_left=self.door[0],
            tram_door_right=self.door[1], tram_length=self.tram_length, num_boarding_agents=boarding,
            num_exiting_agents=exiting, exiting_destination_area_y=self.exiting_y, boarding_destination_area_y=self.boarding_y,
            reward_config=REWARDS[self.reward](), terminated_config=TERMS[self.term](),
            truncated_config=MaxStepsTruncatedConfig(max_steps=self.max_steps))


# reward parameters that are not exact in float32 (the device rounds the float64 reward once)
REWARDS = {
    "default": lambda: DefaultRewardConfig(distance_penalty_factor=0.37, tram_door_reward=7.1, tram_area_reward=1 / 3),
    "simple_distance": lambda: SimpleDistanceRewardConfig(distance_penalty_factor=1 / 3),
    "binary": lambda: BinaryRewardConfig(goal_reward=7.1, no_goal_reward=-0.37),
    "constant_negative": lambda: ConstantNegativeRewardConfig(step_penalty=-1 / 3),
}
TERMS = {"individual": IndividualAtDestinationTerminatedConfig, "all": AllAtDestinationTerminatedConfig}

# A door with posts dl and dr opens the cells dl < x < dr of the division row: posts two apart make a door one cell wide.
LATTICES = {lat.name: lat for lat in [
    Lattice("t2_256_wide", 29, 5, 2, (0, 3), 29, boarding_y=5, exiting_y=1, padded=(32, 8),
            pins="tpe2 at its column limit and its cell limit (32 x 8 = 256); tram wall at x = 0; boarding destination y = H, "
                 "exiting destination y = D - 1",
            crews=((5, 3), (1, 1), (2, 2), (3, 4))),
    Lattice("t2_256_square", 13, 13, 6, (10, 12), 13, boarding_y=6, exiting_y=0, padded=(16, 16),
            pins="tpe2 at its row limit and its cell limit (16 x 16 = 256); a one-cell door against the right wall; "
                 "boarding destination y = D",
            crews=((1, 0), (3, 3), (6, 2), (4, 3)), reward="simple_distance", max_steps=14),
    Lattice("t2_narrow_tall", 3, 13, 2, (0, 2), 3, boarding_y=13, exiting_y=1, padded=(6, 16),
            pins="tpe2 on its narrowest lattice with 16 rows (96 cells); a one-cell door; odd W and L",
            crews=((0, 1), (2, 0), (2, 2), (3, 3)), reward="binary", term="all"),
    Lattice("tpe_272", 14, 13, 12, (2, 9), 11, boarding_y=13, exiting_y=11, padded=(17, 16),
            pins="one cell past tpe2 (17 x 16 = 272): tpe row words with PH == bm_cap = 16 (float32 rows of 6 or 8 "
                 "agents, and no rows / table); D = H - 1; exiting destination y = D - 1",
            crews=((4, 2), (2, 0), (5, 3), (1, 2))),
    Lattice("tpe_rows17", 5, 14, 7, (0, 2), 4, boarding_y=14, exiting_y=0, padded=(8, 17),
            pins="one row past tpe2 (8 x 17): tpe linear bitmap of 5 words; even L",
            crews=((1, 1), (3, 1), (4, 4), (2, 5)), reward="constant_negative", max_steps=15),
    Lattice("tpe_cols33", 30, 4, 2, (5, 20), 28, boarding_y=4, exiting_y=0, padded=(33, 7),
            pins="one column past tpe2 (33 x 7): tpe linear bitmap; walk_words = 8 == bm_cap of float32 rows of 4 agents; "
                 "even W and L",
            crews=((1, 0), (2, 2), (4, 2), (5, 3)), term="all"),
    Lattice("tpe_512", 61, 5, 1, (20, 40), 60, boarding_y=5, exiting_y=0, padded=(64, 8),
            pins="tpe linear bitmap at exactly 16 words (64 x 8 = 512) == bm_cap; D = 1",
            crews=((3, 1), (0, 2), (4, 4), (6, 1)), reward="simple_distance"),
    Lattice("tpe_576", 61, 6, 3, (0, 4), 61, boarding_y=6, exiting_y=2, padded=(64, 9),
            pins="one bitmap word past the linear path (64 x 9 = 576, 18 words): tpe register compares; "
                 "exiting destination y = D - 1",
            crews=((1, 0), (2, 2), (5, 3), (3, 3))),
    Lattice("strip_120x4", 120, 4, 2, (100, 116), 117, boarding_y=4, exiting_y=0, padded=(123, 7),
            pins="placements and moves at x up to 120 on a lattice where agents reach their destinations",
            crews=((2, 1), (4, 4), (0, 1), (3, 0)), max_steps=24, big_crews=((5, 4), (40, 24), (80, 48))),
    Lattice("strip_4x120", 4, 120, 60, (1, 3), 4, boarding_y=61, exiting_y=59, padded=(7, 123),
            pins="placements and moves at y up to 120 on a lattice where agents reach their destinations (next to the "
                 "division row, through a one-cell door)",
            crews=((1, 1), (4, 4), (2, 0), (3, 4)), reward="simple_distance", max_steps=24, big_crews=((5, 4), (40, 24), (80, 48))),
    Lattice("max_120", 120, 120, 100, (0, 2), 117, boarding_y=120, exiting_y=0, padded=(123, 123),
            pins="the largest lattice: walk map of 473 words (kMaxWalkWords = 512); the door at the far left, so the "
                 "reward-table index |x - DC| + |y - D| + 128 reaches 345 (kRtabSize = 400)",
            crews=((1, 0), (4, 4), (0, 3), (3, 4)), max_steps=24, big_crews=((5, 4), (40, 24), (80, 48))),
]}
TPE2_LATTICES = ("t2_256_wide", "t2_256_square", "t2_narrow_tall")
TPE_LATTICES = ("tpe_272", "tpe_rows17", "tpe_cols33", "tpe_512", "tpe_576")


def padded(lat_or_cfg) -> tuple[int, int]:
    return lat_or_cfg.width + 3, lat_or_cfg.height + 3


def walk_words(cfg) -> int:
    """Words of one padded-lattice bitmap (``fill_params``, csrc/cc_api.cu:152)."""
    PW, PH = padded(cfg)
    return (PW * PH + 31) // 32


def tpe2_eligible(cfg, A: int, obs: str, tpe2_enabled: bool = True) -> bool:
    """csrc/cc_launch_tpe.cu:93-99 (``CCB200_TPE2=0`` clears ``tpe2_enabled``)."""
    if obs == "float32" and A % 2:
        return False                                   # float32 rows of odd crews: cc_step_tpe_kernel
    PW, PH = padded(cfg)
    return tpe2_enabled and PW <= T2_MAX_COLS and PH <= T2_MAX_ROWS and PW * PH <= T2_MAX_CELLS


def tpe_eligible(A: int, obs: str) -> bool:
    """csrc/cc_api.cu:199-210 for the tensors of BatchedCollectiveCrossing (aligned, float32 rewards, agent order)."""
    return 1 <= A <= 8 and (obs != "int8" or A == 8)


def tpe_bitmap_cap(A: int, obs: str) -> int:
    """bm_cap of ``launch_tpe_t`` (csrc/cc_launch_tpe.cu:28-29): float32 rows of even crews go out through TMA images
    (``TpeLayout::kTma``, cc_kernel_tpe.cuh:70) and the bitmap aliases their ring (128 bytes per word)."""
    if obs == "float32" and A % 2 == 0:
        img_bytes = A * (3 + 2 * A) * 8                # TpeLayout::kImgBytes: A rows of 3 + 2A float pairs
        return min(TPE_IMG_RING * img_bytes // 128, TPE_MAX_BITMAP_WORDS)
    return TPE_MAX_BITMAP_WORDS


def tpe_occupancy_path(cfg, A: int, obs: str, policy: str) -> str | None:
    """Occupancy path of ``launch_tpe_t`` (csrc/cc_launch_tpe.cu:26-32); None where the policy needs no lattice."""
    if policy not in ("greedy", "waiting"):
        return None
    PW, PH = padded(cfg)
    cap = tpe_bitmap_cap(A, obs)
    if PW <= 32 and PH <= cap:
        return "rows"
    if walk_words(cfg) <= cap:
        return "linear"
    return "compares"


def lanes_shape(A: int) -> tuple[int, int]:
    """(lanes per env, agents per lane) of the lane-group kernel (``cc_create``, csrc/cc_api.cu:625-626)."""
    lpe = 4
    while lpe < A and lpe < 32:
        lpe <<= 1
    return lpe, 1 if A <= 32 else (2 if A <= 64 else 4)


def expected_kernel(cfg, A: int, obs: str, policy: str, kernel: str = "auto", *, np_reset: bool = False,
                    tpe2_enabled: bool = True) -> tuple[str, str | None]:
    """(``cc_last_kernel_name`` of a step, tpe occupancy path or None) for a ``BatchedCollectiveCrossing`` with float32
    rewards and agent order.  Name quirks: the README crew's instantiation ``cc_step_tpe2_kernel<8, OBS, 5>`` is named
    without its third argument (csrc/cc_launch_tpe.cu:85), and numpy-mode placements (``reset_rng="numpy"``) OR
    ``kNpReset`` = 256 into the OBS number of all three kernels."""
    code = OBS_CODE[obs] | (NP_RESET if np_reset else 0)
    threads = kernel != "lanes" and tpe_eligible(A, obs)
    if kernel == "threads" and not threads:
        raise ValueError(f"no thread-per-env kernel serves A={A} with {obs} rows")
    if not threads:
        lpe, apl = lanes_shape(A)
        return f"ccb::cc_kernel<{lpe},{apl},{code},step>", None
    if tpe2_eligible(cfg, A, obs, tpe2_enabled):
        return f"ccb::cc_step_tpe2_kernel<{A},{code}>", None
    return f"ccb::cc_step_tpe_kernel<{A},{code}>", tpe_occupancy_path(cfg, A, obs, policy)


def family(cfg, A: int, obs: str, policy: str, kernel: str = "auto", **kw) -> str:
    """Coverage cell of a case: tpe2, tpe_rows, tpe_linear, tpe_compares, tpe (policy without a lattice) or lanes."""
    name, path = expected_kernel(cfg, A, obs, policy, kernel, **kw)
    if "tpe2" in name:
        return "tpe2"
    if "tpe" in name:
        return f"tpe_{path}" if path else "tpe"
    return "lanes"


# ---- the device matrix -------------------------------------------------------------------------------------------
OBS_MODES = ("none", "table", "int8", "float32")
POLICIES = ("greedy", "waiting", "random", "external")


@dataclass(frozen=True)
class Case:
    lattice: str
    boarding: int
    exiting: int
    obs: str
    policy: str
    kernel: str = "auto"

    @property
    def id(self) -> str:
        return f"{self.lattice}-{self.boarding}+{self.exiting}-{self.obs}-{self.policy}-{self.kernel}"

    def config(self):
        return LATTICES[self.lattice].config(self.boarding, self.exiting)

    def expected(self, **kw):
        return expected_kernel(self.config(), self.boarding + self.exiting, self.obs, self.policy, self.kernel, **kw)

    def family(self, **kw):
        return family(self.config(), self.boarding + self.exiting, self.obs, self.policy, self.kernel, **kw)


def device_cases() -> list[Case]:
    """Every lattice x crew in all four output modes, the action source rotating so that each (lattice, output mode)
    sees all four sources; the first crew also on the lane-group kernel; the big crews (lane-group kernel) on the
    largest lattices."""
    out = []
    for lat in LATTICES.values():
        for i, (b, e) in enumerate(lat.crews):
            for j, obs in enumerate(OBS_MODES):
                out.append(Case(lat.name, b, e, obs, POLICIES[(i + j) % 4]))
        b, e = lat.crews[0]
        for j, obs in enumerate(OBS_MODES):
            out.append(Case(lat.name, b, e, obs, POLICIES[(j + 1) % 4], "lanes"))
        for i, (b, e) in enumerate(lat.big_crews):
            out.append(Case(lat.name, b, e, OBS_MODES[(i + 1) % 4], POLICIES[i % 4]))
    return out


def tpe2_off_cases() -> list[Case]:
    """The tpe2 lattices with ``CCB200_TPE2=0``: cc_step_tpe_kernel with bitmap capacities 2, 8 and 16 (float32 rows of
    2, 4 and 6/8 agents) and the compact output modes."""
    crews = {"t2_256_wide": ((1, 1), (2, 2), (5, 3)), "t2_256_square": ((1, 1), (3, 1), (4, 2)), "t2_narrow_tall": ((2, 0), (2, 2), (3, 3))}
    out = []
    for name, cs in crews.items():
        for i, (b, e) in enumerate(cs):
            out.append(Case(name, b, e, "float32", ("greedy", "waiting")[i % 2]))
            out.append(Case(name, b, e, ("none", "table")[i % 2], ("waiting", "greedy", "random")[i % 3]))
    return out
