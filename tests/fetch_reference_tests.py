"""Copy the reference's own hot-path test files into baseline/_ref_tests/ (git-ignored, like baseline/_ref) so that they
travel to the GPU box with the tree, where tests/test_gpu_reference_suite.py runs them unmodified against this repository's
classes through the keisei -> shogidrl_b200 alias package (tests/ref_alias).  Run where a checkout of the reference is at hand:

    python tests/fetch_reference_tests.py [reference checkout, default $SHOGIDRL_REFERENCE]

The mock-driven tests of the two training-side callers of the path (tests/training/test_step_manager.py and
test_env_manager.py, with the reference's conftest.py for their fixtures) and two CPU-only files of tests/shogi
(test_move_formatting.py, test_shogi_core_definitions.py) go to baseline/_ref_tests/host/; they need no
GPU and run in the CPU suite too (tests/test_reference_host_suite_cpu.py).

The copies are never committed (the reference's sources do not belong in this repository)."""
import os
import shutil
import sys

FILES = ["test_legal_mask_generation.py", "test_shogi_rules_and_validation.py", "test_shogi_game_core_logic.py",
         "test_shogi_engine_integration.py", "test_shogi_game_rewards.py", "test_shogi_utils.py",
         "test_observation_constants.py", "test_reward_with_flipped_perspective.py",
         "test_shogi_game_io.py", "test_shogi_game_mock_comprehensive.py"]
# the last two import tests.utils.mock_utilities (a context manager that hides torch from NEW imports while a game is
# built): the reference's helper module is copied next to them as a `tests` package of its own
PKG_FILES = [("", "__init__.py"), ("utils", "__init__.py"), ("utils", "mock_utilities.py")]
HOST_FILES = [("", "conftest.py"), ("training", "test_step_manager.py"), ("training", "test_env_manager.py"),
              ("shogi", "test_move_formatting.py"), ("shogi", "test_shogi_core_definitions.py")]


def main() -> int:
    ref = sys.argv[1] if len(sys.argv) > 1 else os.environ.get("SHOGIDRL_REFERENCE")
    if not ref:
        sys.exit("usage: python tests/fetch_reference_tests.py <reference checkout> (or set SHOGIDRL_REFERENCE)")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dst = os.path.join(root, "baseline", "_ref_tests")
    os.makedirs(dst, exist_ok=True)
    for f in FILES:
        shutil.copyfile(os.path.join(ref, "tests", "shogi", f), os.path.join(dst, f))
    for sub, f in PKG_FILES:
        d = os.path.join(dst, "_pkg", "tests", sub)
        os.makedirs(d, exist_ok=True)
        shutil.copyfile(os.path.join(ref, "tests", sub, f), os.path.join(d, f))
    host = os.path.join(dst, "host")
    os.makedirs(host, exist_ok=True)
    for sub, f in HOST_FILES:
        shutil.copyfile(os.path.join(ref, "tests", sub, f), os.path.join(host, f))
    print(f"copied {len(FILES)} + {len(HOST_FILES)} files to {dst}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
