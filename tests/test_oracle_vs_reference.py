"""CPU: pins the oracle restatement and the weight packer's helpers against what the unmodified reference modules
computed (tests/golden/reference_model.npz, written by oracle/make_golden_reference.py from the reference tree)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import vits_oracle as vo
from oracle.make_golden_reference import infer_inputs, spline_inputs


@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(GOLDEN, "reference_model.npz"))


def test_fold_equals_remove_weight_norm(ref, folded):
    """Every folded tensor exists in the reference's state dict after remove_weight_norm and agrees within 1e-6 on a seeded
    sample of its elements; its sum agrees within what 1e-6 per element allows."""
    keys = [str(k) for k in ref["state_keys"]]
    ends = np.cumsum(ref["state_sample_count"])
    for k, v in folded.items():
        assert k in keys, k
        i = keys.index(k)
        sl = slice(ends[i] - ref["state_sample_count"][i], ends[i])
        flat = v.reshape(-1).numpy()
        assert np.abs(flat[ref["state_sample_idx"][sl]] - ref["state_sample_val"][sl]).max() <= 1e-6, k
        assert abs(float(v.double().sum()) - float(ref["state_sum"][i])) <= 1e-6 * flat.size, k


def test_istft_basis_and_pqmf_match_reference(ref):
    from vosk_tts_b200 import weights
    assert np.abs(weights.istft_inverse_basis(16, 4) - ref["istft_inverse_basis"]).max() < 1e-7
    assert np.abs(weights.pqmf_synthesis_filter(4) - ref["pqmf_synthesis_filter"]).max() < 1e-7


def test_spline_inverse_matches_reference_transforms(ref):
    x, uw, uh, ud = spline_inputs()
    assert float(x.double().sum()) == float(ref["spline_x_sum"]), "seeded spline inputs drifted from the fixture"
    got = vo.rq_spline_inverse(x.clone(), uw.clone(), uh.clone(), ud.clone(), bound=5.0)
    assert torch.equal(torch.from_numpy(ref["spline_inverse"]), got)


@pytest.mark.parametrize("T,seed", [(24, 101), (77, 102)])
def test_oracle_equals_reference_infer(ref, folded, cfg, T, seed):
    tok, eps_dp, eps_z = infer_inputs(T, seed)
    scales = [0.667, 1.0, 0.8]
    with torch.no_grad():
        o = vo.infer(folded, cfg, tok, torch.tensor([T]), torch.tensor([3]), scales, eps_dp, eps_z, return_all=True)
    pre = "infer_t%d_" % T
    assert ref[pre + "o"].shape == tuple(o["o"].shape)
    assert np.array_equal(ref[pre + "attn"], o["attn"].numpy().astype(np.int8))
    assert np.abs(ref[pre + "o"] - o["o"].numpy()).max() < 1e-5
    assert np.abs(ref[pre + "z"] - o["z"].numpy()).max() < 5e-5
