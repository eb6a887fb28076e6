"""The lattices of tests/geometry_edges.py on CPU: each sits on the size limit it is named for, the C oracle equals the
pure-Python port on every one of them (so it is a trustworthy reference there), and the device matrix of
tests/test_gpu_geometry_edges.py reaches every kernel, occupancy path and output mode, the equality cases included."""

from __future__ import annotations

import re
from pathlib import Path

import pytest
from geometry_edges import (
    LATTICES,
    MAX_GEOM,
    MAX_WALK_WORDS,
    NP_RESET,
    OBS_MODES,
    RTAB_SIZE,
    T2_MAX_CELLS,
    T2_MAX_COLS,
    T2_MAX_ROWS,
    TPE2_LATTICES,
    TPE_IMG_RING,
    TPE_LATTICES,
    TPE_MAX_BITMAP_WORDS,
    Y_BIAS,
    device_cases,
    expected_kernel,
    padded,
    tpe2_off_cases,
    tpe_bitmap_cap,
    walk_words,
)
from test_numpy_reset_cpu import run_against

from collectivecrossing_b200.lowering import lower_config
from oracle.pyport import PyEnv


@pytest.mark.parametrize("name", list(LATTICES))
def test_lattice_lowers_to_its_padded_size(name):
    lat = LATTICES[name]
    for b, e in lat.crews + lat.big_crews:
        low = lower_config(lat.config(b, e))
        assert (low.width + 3, low.height + 3) == lat.padded, name
        assert 0 <= low.tram_left <= low.door_left < low.door_right <= low.tram_right <= low.width <= MAX_GEOM
        assert walk_words(low) <= MAX_WALK_WORDS


def test_lattices_sit_on_the_limits_they_are_named_for():
    PW, PH = {}, {}
    for name, lat in LATTICES.items():
        PW[name], PH[name] = padded(lat)
    cells = {n: PW[n] * PH[n] for n in LATTICES}
    # tpe2: at the column, row and cell limits, and just past each of them
    assert PW["t2_256_wide"] == T2_MAX_COLS and cells["t2_256_wide"] == T2_MAX_CELLS
    assert PH["t2_256_square"] == T2_MAX_ROWS and cells["t2_256_square"] == T2_MAX_CELLS
    assert PH["t2_narrow_tall"] == T2_MAX_ROWS and LATTICES["t2_narrow_tall"].width == 3
    assert PW["tpe_272"] <= T2_MAX_COLS and PH["tpe_272"] == T2_MAX_ROWS and cells["tpe_272"] == T2_MAX_CELLS + 16
    assert PH["tpe_rows17"] == T2_MAX_ROWS + 1 and cells["tpe_rows17"] <= T2_MAX_CELLS
    assert PW["tpe_cols33"] == T2_MAX_COLS + 1 and cells["tpe_cols33"] <= T2_MAX_CELLS and PH["tpe_cols33"] <= T2_MAX_ROWS
    # tpe bitmap: 16 words exactly, one word past; 8 words for the TMA-aliased bitmap of 4 agents
    assert walk_words(LATTICES["tpe_512"]) == TPE_MAX_BITMAP_WORDS and cells["tpe_512"] == 32 * TPE_MAX_BITMAP_WORDS
    assert walk_words(LATTICES["tpe_576"]) == TPE_MAX_BITMAP_WORDS + 2
    assert walk_words(LATTICES["tpe_cols33"]) == tpe_bitmap_cap(4, "float32") == 8
    assert walk_words(LATTICES["tpe_rows17"]) == 5
    # coordinates and tables at their largest
    assert LATTICES["strip_120x4"].width == MAX_GEOM and LATTICES["strip_4x120"].height == MAX_GEOM
    assert padded(LATTICES["max_120"]) == (MAX_GEOM + 3, MAX_GEOM + 3) and walk_words(LATTICES["max_120"]) == 473


def test_restated_limits_match_the_sources():
    """The constants expected_kernel and the lattices are built on are the ones the kernels compile with: moving a limit
    in the sources (say kT2MaxCells to 255 or kTpeMaxBitmapWords to 15) fails here, not only on a GPU."""
    csrc = Path(__file__).resolve().parents[1] / "collectivecrossing_b200" / "csrc"
    text = "".join((csrc / f).read_text() for f in ("cc_kernels.cuh", "cc_kernel_tpe.cuh", "cc_kernel_tpe2.cuh"))

    def const(name):
        m = re.findall(rf"\b{name}\s*=\s*(0x[0-9a-fA-F]+|\d+)\s*[;,]", text)
        assert len(m) == 1, (name, m)
        return int(m[0], 0)

    assert (const("kT2MaxCols"), const("kT2MaxRows"), const("kT2MaxCells")) == (T2_MAX_COLS, T2_MAX_ROWS, T2_MAX_CELLS)
    assert (const("kTpeMaxBitmapWords"), const("kImgRing")) == (TPE_MAX_BITMAP_WORDS, TPE_IMG_RING)
    assert (const("kMaxGeom"), const("kMaxWalkWords"), const("kRtabSize"), const("kYBias")) == (MAX_GEOM, MAX_WALK_WORDS, RTAB_SIZE, Y_BIAS)
    assert const("kNpReset") == NP_RESET


def test_bitmap_capacities():
    assert [tpe_bitmap_cap(a, "float32") for a in range(1, 9)] == [16, 2, 16, 8, 16, 16, 16, 16]
    assert {tpe_bitmap_cap(a, o) for a in range(1, 9) for o in ("none", "table", "int8")} == {16}


def test_reward_table_index_of_the_largest_lattice_is_near_its_bound():
    """|x - DC| + |y - D| + 128 over every grid point of max_120 (the default reward's table index, cc_kernels.cuh:386)."""
    low = lower_config(LATTICES["max_120"].config(1, 0))
    dc = (low.door_left + low.door_right) // 2
    top = max(abs(x - dc) for x in range(low.width + 1)) + max(abs(y - low.division_y) for y in range(low.height + 1)) + Y_BIAS
    assert 340 <= top < RTAB_SIZE


def test_edges_vary_across_the_set():
    lows = {n: lower_config(lat.config(*lat.crews[0])) for n, lat in LATTICES.items()}
    assert any(low.door_right - low.door_left == 2 for low in lows.values())                     # a door one cell wide
    assert any(low.division_y == 1 for low in lows.values())
    assert any(low.division_y == low.height - 1 for low in lows.values())
    assert any(low.boarding_dest_y == low.division_y for low in lows.values())
    assert any(low.boarding_dest_y == low.height for low in lows.values())
    assert any(low.exiting_dest_y == low.division_y - 1 for low in lows.values())
    assert any(low.tram_left == 0 for low in lows.values()) and any(low.tram_right == low.width - 1 for low in lows.values())
    assert {lat.width % 2 for lat in LATTICES.values()} == {0, 1} and {lat.tram_length % 2 for lat in LATTICES.values()} == {0, 1}


def test_expected_kernel_restates_the_dispatch():
    wide, tpe272 = LATTICES["t2_256_wide"].config(5, 3), LATTICES["tpe_272"].config(5, 3)
    assert expected_kernel(wide, 8, "float32", "greedy") == ("ccb::cc_step_tpe2_kernel<8,4>", None)   # README crew: <8,4,5>
    assert expected_kernel(wide, 8, "int8", "random", np_reset=True) == ("ccb::cc_step_tpe2_kernel<8,257>", None)
    assert expected_kernel(wide, 7, "float32", "greedy") == ("ccb::cc_step_tpe_kernel<7,4>", "rows")
    assert expected_kernel(wide, 8, "float32", "greedy", tpe2_enabled=False) == ("ccb::cc_step_tpe_kernel<8,4>", "rows")
    assert expected_kernel(wide, 2, "float32", "waiting", tpe2_enabled=False) == ("ccb::cc_step_tpe_kernel<2,4>", "compares")
    assert expected_kernel(tpe272, 8, "table", "waiting") == ("ccb::cc_step_tpe_kernel<8,16>", "rows")
    assert expected_kernel(tpe272, 8, "table", "external") == ("ccb::cc_step_tpe_kernel<8,16>", None)
    assert expected_kernel(tpe272, 4, "int8", "greedy") == ("ccb::cc_kernel<4,1,1,step>", None)
    assert expected_kernel(tpe272, 8, "none", "greedy", "lanes") == ("ccb::cc_kernel<8,1,0,step>", None)
    assert expected_kernel(tpe272, 128, "table", "greedy", np_reset=True) == ("ccb::cc_kernel<32,4,272,step>", None)
    assert expected_kernel(tpe272, 9, "float32", "greedy") == ("ccb::cc_kernel<16,1,4,step>", None)
    assert expected_kernel(tpe272, 64, "float32", "greedy") == ("ccb::cc_kernel<32,2,4,step>", None)
    with pytest.raises(ValueError):
        expected_kernel(tpe272, 4, "int8", "greedy", "threads")


# ---- the oracle against the pure-Python port at every lattice --------------------------------------------------
@pytest.mark.parametrize("policy", ["greedy", "waiting", "random"])
@pytest.mark.parametrize("name", list(LATTICES))
def test_oracle_equals_pyport_on_edge_lattices(name, policy):
    lat = LATTICES[name]
    seeds = [31 * k + 5 for k in range(4)]
    for b, e in (lat.crews[0], lat.crews[-1]):
        cfg = lat.config(b, e)
        episodes, _, _ = run_against(lambda: PyEnv(cfg), lambda env: env.rng, cfg, 3 * lat.max_steps + 4, policy, seeds)
        assert episodes >= 3 * len(seeds), (name, b, e)


# ---- coverage of the device matrix ------------------------------------------------------------------------------
def _cells(cases, **kw):
    return {(c.family(**kw), c.obs) for c in cases}


def test_device_matrix_covers_every_kernel_path_and_output_mode():
    cases = device_cases()
    assert len({c.id for c in cases}) == len(cases)
    got = _cells(cases)
    want = {(f, o) for f in ("tpe2", "tpe_rows", "tpe_linear", "tpe_compares", "lanes") for o in OBS_MODES}
    assert want <= got, sorted(want - got)
    # the equality cases of the occupancy paths: PH == bm_cap (row words) and walk_words == bm_cap (linear bitmap),
    # the latter also where the bitmap aliases the TMA image ring (cap 8)
    rows_eq, linear_eq = set(), set()
    for c in cases:
        cfg, A = c.config(), c.boarding + c.exiting
        cap = tpe_bitmap_cap(A, c.obs)
        _, path = c.expected()
        if path == "rows" and padded(cfg)[1] == cap:
            rows_eq.add(cap)
        if path == "linear" and walk_words(cfg) == cap:
            linear_eq.add(cap)
    assert 16 in rows_eq and {8, 16} <= linear_eq, (rows_eq, linear_eq)
    # every lattice on the lane-group kernel, crews of 1, 2, 4, 7 and 8, crews without boarding or exiting agents
    assert {c.lattice for c in cases if c.kernel == "lanes"} == set(LATTICES)
    sizes = {c.boarding + c.exiting for c in cases}
    assert {1, 2, 4, 7, 8, 9, 64, 128} <= sizes
    assert any(c.boarding == 0 for c in cases) and any(c.exiting == 0 for c in cases)
    assert {c.policy for c in cases} == {"greedy", "waiting", "random", "external"}
    assert {c.lattice for c in cases} == set(LATTICES)


def test_tpe2_off_matrix_runs_the_small_lattices_through_tpe():
    cases = tpe2_off_cases()
    assert {c.lattice for c in cases} == set(TPE2_LATTICES)
    names = [c.expected(tpe2_enabled=False)[0] for c in cases]
    assert all(n.startswith("ccb::cc_step_tpe_kernel<") for n in names)
    caps = {tpe_bitmap_cap(c.boarding + c.exiting, c.obs) for c in cases if c.obs == "float32"}
    assert caps == {2, 8, 16}
    assert {c.obs for c in cases} == {"float32", "none", "table"}
    assert {c.family(tpe2_enabled=False) for c in cases} >= {"tpe_rows", "tpe_linear", "tpe_compares"}


def test_fused_and_numpy_lattices_exist():
    assert set(TPE2_LATTICES) | set(TPE_LATTICES) <= set(LATTICES)
    for name in TPE2_LATTICES:
        lat = LATTICES[name]
        assert expected_kernel(lat.config(*lat.crews[0]), sum(lat.crews[0]), "table", "greedy")[0].startswith("ccb::cc_step_tpe2_kernel")
    for name in TPE_LATTICES:
        lat = LATTICES[name]
        assert expected_kernel(lat.config(*lat.crews[0]), sum(lat.crews[0]), "table", "greedy")[0].startswith("ccb::cc_step_tpe_kernel")
