"""SURVEY 8b / appendix C: demo scripts run UNMODIFIED under scripts/run_demo.py (module resolution controlled by the
launcher, headless pygame, scripted QUIT).  The scripts are tests/demos/, stand-ins with the structure of the
reference's two demos (the reference itself is not part of this repository).  What is checked here is the launcher's
mechanics: a stand-in gicp module backed by the CPU oracle takes the engine's place (same 7-tuple).  The engine itself
in the demos' process layout - first gicp() call inside a forked worker, lists of tuples in, pickled numpy out - is
checked on the GPU by tests/test_gpu_fork.py."""
import os
import sys
import types

import pytest

from conftest import ROOT

REF = os.path.join(ROOT, "tests", "demos")


def _oracle_backed_module():
    from oracle import gicp_oracle as O
    import gicp as shim

    def gicp(source_points, target_points, max_iterations=100, tolerance=1e-6, max_distance_correspondence=150,
             max_distance_nearest_neighbors=50):
        r = O.gicp_oracle(source_points, target_points, max_iterations=max_iterations, tolerance=tolerance,
                          max_distance_correspondence=max_distance_correspondence,
                          max_distance_nearest_neighbors=max_distance_nearest_neighbors, inner="newton",
                          recompute_src_cov=False, record=False)
        if r["converged_at"] is not None:
            print("Converged at iteration", r["converged_at"])
        return (r["T"], r["all_T"], r["src_cov0"], r["tgt_cov"], r["hw_src"], r["hw_tgt"], r["all_src_cov"])

    m = types.ModuleType("gicp_standin")
    m.gicp = gicp
    m.apply_transformation = shim.apply_transformation      # the product's own numpy implementation (UI process)
    return m


def _launcher():
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import run_demo
    return run_demo


def test_static_viewer_runs_unmodified(capsys):
    """The static viewer builds its pair, calls gicp(source, target) once, steps through the result."""
    before = open(os.path.join(REF, "visualization.py"), "rb").read()
    r = _launcher().run(os.path.join(REF, "visualization.py"), frames=25, headless=True,
                        gicp_module=_oracle_backed_module(), seed=0, tick=0.0)
    assert r["exit"] == 0 and r["gicp_calls"] == 1
    assert r["pygame_calls"]["flip"] >= 20 and r["pygame_calls"]["draw"] > 100 and r["pygame_calls"]["quit"] == 1
    assert "Converged at iteration" in capsys.readouterr().out
    assert open(os.path.join(REF, "visualization.py"), "rb").read() == before


def test_robot_demo_runs_unmodified_with_forked_worker():
    """The robot demo: UI loop at 10 fps, GICP worker in a forked process fed through queues, each call padded to
    0.5 s.  40 frames of 0.1 s leave time for several results."""
    r = _launcher().run(os.path.join(REF, "robot-visualization.py"), frames=40, headless=True,
                        gicp_module=_oracle_backed_module(), seed=1, tick=0.1)
    assert r["exit"] == 0
    assert r["gicp_calls"] >= 1            # counted inside the forked worker, after gicp() returned
    assert r["pygame_calls"]["flip"] >= 30


def test_launcher_registers_the_repo_module_by_default():
    """Without a stand-in the launcher binds the demos to THIS repo's drop-in (which needs a GPU at call time):
    without a GPU the static viewer must fail loudly inside gicp(), not fall back to a gicp.py lying beside the
    script."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _launcher().run(os.path.join(REF, "visualization.py"), frames=3, headless=True, seed=0, tick=0.0)
