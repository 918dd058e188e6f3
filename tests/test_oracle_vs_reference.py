"""Re-check the oracle and the index paths against outputs of the reference beyond the seed-0 golden files: fresh seeds,
configurations without a golden file, and arange tensors.  The reference's outputs were recorded by
oracle/record_reference.py into tests/golden/reference/fresh_seeds.npz and tests/golden/reference/cswin_windows.npz."""
import json
import os

import numpy as np
import pytest
import torch

from _util import GOLDEN_DIR, load_golden
from oracle.cases import EXTRA_SPECS, GOLDEN_CASES, BVIT_QKV_CTORS, make_inputs, round_fp16_, run_oracle_case, sample_index, \
    shuffled_case, synth_linear_params
from oracle import cswin_window_table

FRESH = np.load(os.path.join(GOLDEN_DIR, "reference", "fresh_seeds.npz"))


def _assert_matches_recorded(y, key):
    """y against the recorded reference output `key` within 5e-6 * max(1, max|y_ref|): shape, the stored sample of elements,
    and max|y| (which moves by no more than the largest elementwise difference)."""
    assert tuple(y.shape) == tuple(FRESH[key + ".shape"])
    got = y.reshape(-1)[torch.from_numpy(sample_index(y.numel()))]
    ymax = float(FRESH[key + ".ymax"])
    tol = 5e-6 * max(1.0, ymax)
    assert (got - torch.from_numpy(FRESH[key + ".y"])).abs().max().item() <= tol
    assert abs(y.abs().max().item() - ymax) <= tol


@pytest.mark.parametrize("name", sorted(GOLDEN_CASES))
@pytest.mark.parametrize("seed", [1, 2])
def test_oracle_vs_live_reference(name, seed):
    spec = GOLDEN_CASES[name]
    inputs, params, _ = load_golden(name)
    inputs, params = shuffled_case(inputs, params, seed)
    _assert_matches_recorded(run_oracle_case(spec, inputs, params), f"{name}.s{seed}")


WINDOWS = np.load(os.path.join(GOLDEN_DIR, "reference", "cswin_windows.npz"))


@pytest.mark.parametrize("reso,idx,split", [(14, 0, 7), (14, 1, 7), (7, -1, 7), (28, 0, 2)])
def test_window_table_vs_reference_img2windows(reso, idx, split):
    """The reference's img2windows of an arange image: bit-exact index table; its windows2img of that table: the scatter
    through the table."""
    key = f"r{reso}_i{idx}_s{split}"
    table = cswin_window_table(reso, idx, split)
    assert np.array_equal(WINDOWS[key + ".img2windows"], table)
    back = np.empty(reso * reso, dtype=np.int64)
    back[table.reshape(-1)] = table.reshape(-1)
    assert np.array_equal(WINDOWS[key + ".windows2img"], back)
    assert np.array_equal(back, np.arange(reso * reso))


@pytest.mark.parametrize("name", sorted(EXTRA_SPECS))
def test_oracle_vs_live_reference_extra_configs(name):
    spec = EXTRA_SPECS[name]
    params = synth_linear_params(json.loads(str(FRESH[name + ".params"])), 7)
    _assert_matches_recorded(run_oracle_case(spec, make_inputs(spec, 7), params), name)


@pytest.mark.parametrize("ctor", BVIT_QKV_CTORS)
def test_bvit_q_k_v_and_identity_projection_vs_live_reference(ctor):
    """Broad_Attention returns (out, q, k, v) (bvit.py:76); with heads == 1 and dim_head == dim there is no output projection
    (bvit.py:52, 61-64).  All four outputs of the restatement against the recorded outputs of the reference module."""
    from oracle import attention as A
    key = f"bvit_qkv{BVIT_QKV_CTORS.index(ctor)}"
    sd = synth_linear_params(json.loads(str(FRESH[key + ".params"])), 3)
    assert ("to_out.0.weight" in sd) == (ctor["heads"] != 1 or ctor["dim_head"] != ctor["dim"])
    x = round_fp16_(torch.randn(2, 37, ctor["dim"], generator=torch.Generator().manual_seed(3)))
    got = A.bvit_broad_attention(x, sd["to_qkv.weight"], sd.get("to_out.0.weight"), sd.get("to_out.0.bias"), ctor["heads"],
                                 ctor["dim_head"])
    assert len(got) == 4
    for j, g in enumerate(got):
        _assert_matches_recorded(g, f"{key}.out{j}")
