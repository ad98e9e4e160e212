"""Randomised differential tests on CPU: the test-only host emulation of the engine (same phase functions as the CUDA
kernels) and the plain-C oracle port against the compiled reference, on random configurations (tests/fuzz_common.py:
2-4 groups, 1x1 .. 2x2 / 1x3 bodies, circle and sector ranges, turn_mode / food_mode / goal_mode / minimap on or off,
random rule sets, walls, random and explicit placements, random call order and acting subset)."""
import os

import pytest

import fuzz_common as fz
import golden_common as gc
import parity_common as pc
from test_emu_parity_cpu import emu  # noqa: F401  (fixture: builds tests/_emu on demand)

HAVE_REF = os.path.exists(pc.REF_LIB)
CHECKER = pc.REF_LIB if HAVE_REF else pc.PORT_LIB


@pytest.mark.parametrize("seed", list(range(0, 24)) + list(range(1000, 1016)))
def test_emulated_engine_matches_checker_on_random_games(emu, seed):
    fz.play(seed, CHECKER, emu, steps=20)


@pytest.mark.parametrize("seed", list(range(100, 116)) + list(range(1100, 1110)))
def test_oracle_port_matches_reference_on_random_games(seed):
    gc.check_reference_result("fuzz/%d" % seed, lambda lib: fz.trace(seed, lib, steps=20), pc.PORT_LIB)


@pytest.mark.parametrize("seed", list(range(200, 212)) + list(range(1200, 1206)))
def test_emulated_engine_matches_checker_with_an_irregular_caller(emu, seed):
    """skipped clear_dead (dead agents keep slots and still get actions), agents added mid-episode, observations
    not fetched every step"""
    fz.play_irregular(seed, CHECKER, emu, steps=20)


@pytest.mark.parametrize("seed", list(range(400, 410)))
def test_emulated_arena_batch_matches_independent_checkers(emu, seed):
    fz.play_batch(seed, CHECKER, emu, n_arenas=1 + seed % 4, steps=10)


# maps in the reference's large_map_mode (more than 99 x 99 cells: movers / turners queued per vertical band, 8 bands;
# 16 bands above 1000 x 1000 cells -- GridWorld.cc:74-85, 403-438), tests/fuzz_common.py LARGE_MAP_SEED / HUGE_MAP_SEED
@pytest.mark.parametrize("seed", list(range(100000, 100008)) + [200000, 200001])
def test_emulated_engine_matches_checker_on_banded_maps(emu, seed):
    fz.play(seed, CHECKER, emu, steps=15)


@pytest.mark.parametrize("seed", list(range(100600, 100604)) + [200002])
def test_oracle_port_matches_reference_on_banded_maps(seed):
    gc.check_reference_result("fuzz/%d" % seed, lambda lib: fz.trace(seed, lib, steps=15), pc.PORT_LIB)


@pytest.mark.parametrize("seed", [101000, 101001, 101002, 201000])
def test_emulated_engine_on_banded_maps_with_an_irregular_caller(emu, seed):
    fz.play_irregular(seed, CHECKER, emu, steps=15)


@pytest.mark.parametrize("seed", [102000, 102001])
def test_emulated_arena_batch_on_banded_maps(emu, seed):
    fz.play_batch(seed, CHECKER, emu, n_arenas=2 + seed % 2, steps=8)


# a caller that reads at every point of the loop, changes the acting subset every step and resets in mid-run
# (fuzz_common.trace_chaotic), replay frames / window queries / density maps included; found: a group reward that
# clear_dead has not collected survives reset(); a long body that kills itself is still fed its own kill_supply (corpse hp)
@pytest.mark.parametrize("seed", list(range(40000, 40016)) + [40029, 47002, 47012, 47086, 110000, 110001, 113018])
def test_emulated_engine_matches_checker_with_a_chaotic_caller(emu, seed):
    fz.play_chaotic(seed, CHECKER, emu)


@pytest.mark.parametrize("seed", list(range(43000, 43008)))
def test_oracle_port_matches_reference_with_a_chaotic_caller(seed):
    gc.check_reference_result("fuzz_chaotic/%d" % seed, lambda lib: fz.chaotic_log(seed, lib), pc.PORT_LIB)


@pytest.mark.parametrize("seed", list(range(60000, 60010)) + [115000, 115001])
def test_emulated_arena_batch_with_a_chaotic_caller(emu, seed):
    """reads at every point of the loop, late adds to all arenas and (select_arena) to one, mid-run reset"""
    fz.play_batch_chaotic(seed, CHECKER, emu, n_arenas=1 + seed % 4)


# 5-8 groups (up to 25 observation channels; fuzz_common.MANY_GROUPS_SEED)
@pytest.mark.parametrize("seed", list(range(70000, 70008)))
def test_emulated_engine_matches_checker_with_many_groups(emu, seed):
    fz.play(seed, CHECKER, emu, steps=15)


@pytest.mark.parametrize("seed", [72000, 72001, 72002, 72003])
def test_emulated_engine_with_many_groups_and_a_chaotic_caller(emu, seed):
    fz.play_chaotic(seed, CHECKER, emu)


@pytest.mark.parametrize("seed", list(range(9000, 9006)))
def test_three_emulated_engines_interleaved_with_chaotic_callers(emu, seed):
    fz.play_interleaved_engines(seed, CHECKER, emu)


# the randomised callers again with EVERY host-buffer observation forced through the wire records + host expansion
# (MAGENT_B200_HOST_PATH=wire; small observations normally take the dense copy): all modes, many groups, late adds, resets
@pytest.mark.parametrize("seed", list(range(40000, 40010)) + [47002, 110000])
def test_chaotic_caller_with_wire_records_forced(emu, seed, monkeypatch):
    monkeypatch.setenv("MAGENT_B200_HOST_PATH", "wire")
    fz.play_chaotic(seed, CHECKER, emu)


@pytest.mark.parametrize("seed", [60000, 60003, 115000])
def test_chaotic_arena_batch_with_wire_records_forced(emu, seed, monkeypatch):
    monkeypatch.setenv("MAGENT_B200_HOST_PATH", "wire")
    fz.play_batch_chaotic(seed, CHECKER, emu, n_arenas=1 + seed % 4)
