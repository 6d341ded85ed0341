"""Destroying a solver handle releases every CUDA event it created, in both solver families and for single-device as well
as sharded construction.  An updateSolution from host arrays creates the event that orders the caller's q / v uploads.

CPU: the SIMT-emulator build, whose cudaEventCreate / cudaEventDestroy keep a live count (idocp_b200_emu_live_events)."""
import gc

import pytest

import idocp_b200 as I
from conftest import make_states
from idocp_b200.capi import SOLVER_UNOCP, SOLVER_UNPARNMPC


def _live_events(lib):
    return lib.L.idocp_b200_emu_live_events()


@pytest.mark.parametrize("devices", [None, [0, 0]])
@pytest.mark.parametrize("kind", [SOLVER_UNOCP, SOLVER_UNPARNMPC])
def test_fixed_base_solver_releases_its_events(emu_lib, kind, devices):
    before = _live_events(emu_lib)
    s = I.ShardedSolver(I.benchmark_problem(emu_lib, N=4), 4, devices, kind=kind, lib=emu_lib) if devices else \
        (I.UnOCPSolver if kind == SOLVER_UNOCP else I.UnParNMPCSolver)(I.benchmark_problem(emu_lib, N=4), 4, lib=emu_lib)
    q, v = make_states(4, 5)
    s.updateSolution(0.0, q, v)
    assert _live_events(emu_lib) > before
    s.close()
    assert _live_events(emu_lib) == before


@pytest.mark.parametrize("devices", [None, [0, 0]])
def test_floating_base_solver_releases_its_events(emu_lib, devices):
    import anymal_problems as ap
    import fb_py
    fb_py.lib()
    pr = ap.TrottingProblem()
    before = _live_events(emu_lib)
    s = ap.make_product_solver(pr, emu_lib, fb_py, batch=2, devices=devices)
    s.updateSolution(0.0, pr.q0, pr.v0)
    assert _live_events(emu_lib) > before
    del s
    gc.collect()
    assert _live_events(emu_lib) == before
