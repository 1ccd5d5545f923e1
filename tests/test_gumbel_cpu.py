"""CPU checks of the Gumbel MuZero search: the glibc logf restatement its softmax needs, the committed gumbel_*.npz fixtures
against the compiled reference (when oracle/_ref/gmz_tree is built), the no-device error and the reference class config."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN_DIR, ROOT

sys.path.insert(0, GOLDEN_DIR)
import make_gumbel_golden as mg  # noqa: E402


def gumbel_cases():
    return sorted(f[:-4] for f in os.listdir(GOLDEN_DIR) if f.startswith("gumbel_") and f.endswith(".npz"))


def test_logf_matches_libm(tmp_path):
    """Every float in [1, 64] (a softmax sum over at most 64 children); LZ_EXHAUSTIVE=1: every positive finite float."""
    exe = str(tmp_path / "check_logf")
    subprocess.check_call(["gcc", "-O2", "-o", exe, os.path.join(ROOT, "tests", "csrc", "check_logf.c"), "-lm"])
    args = [exe, "1", "all"] if os.environ.get("LZ_EXHAUSTIVE") else [exe, "1"]
    out = subprocess.run(args, capture_output=True, text=True)
    assert out.returncode == 0, out.stdout
    assert "mismatches 0" in out.stdout


def test_gumbel_fixtures_present():
    assert len(gumbel_cases()) >= 7


@pytest.mark.parametrize("case", gumbel_cases())
def test_reference_reproduces_fixture(case):
    gmz = mg.load_reference()
    if gmz is None:
        pytest.skip("oracle/_ref/gmz_tree not built")
    inp, m, exp = mg.load_fixture(os.path.join(GOLDEN_DIR, case + ".npz"))
    got = mg.run_reference(gmz, inp, m)
    for k in ("ix", "iy", "last_action", "vtp", "search_len", "value_bits", "children_value_bits", "policy_bits"):
        assert np.array_equal(np.asarray(got[k]), exp[k]), k
    assert got["dist"] == exp["dist"]
    assert got["traj"] == exp["traj"]


def test_no_device_is_a_loud_error():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    from lightzero_b200 import cabi, gmz_tree
    lib = cabi.load()
    h = ctypes.c_void_p()
    assert lib.lz_tree_create(4, 6, 10, h) == -2 and lib.lz_last_error()      # LZ_ECUDA
    assert lib.lz_tree_set_gumbel(None, 10, 4) == -1                           # LZ_EINVAL
    with pytest.raises(RuntimeError):
        gmz_tree.Roots(4, [[0, 1]] * 4)


def test_default_config_is_the_reference_class_config():
    from lightzero_b200 import GumbelMuZeroMCTSCtree
    cfg = GumbelMuZeroMCTSCtree.default_config()
    # lzero/mcts/tree_search/mcts_ctree.py:1018-1027 + default_config()
    assert dict(cfg) == dict(num_simulations=50, root_dirichlet_alpha=0.3, root_noise_weight=0.25, value_delta_max=0.01,
                             cfg_type="GumbelMuZeroMCTSCtreeDict")
