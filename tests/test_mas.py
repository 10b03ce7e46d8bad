"""Monotonic Alignment Search: oracle (numpy restatement of training/vits2/monotonic_align/core.pyx) against fixtures generated
by the reference's own compiled Cython kernel (oracle/make_golden_mas.py), and the CUDA kernel (csrc/mas.cuh, through the C ABI)
against both -- bit-exact, it is integer/index work."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import mas_oracle as O  # noqa: E402
from oracle.make_golden_mas import LARGE, large_case  # noqa: E402
from oracle.make_golden_reference import mas_trials  # noqa: E402

G = np.load(os.path.join(ROOT, "tests", "golden", "mas_cases.npz"))


def _small():
    for i in range(int(G["n_small"])):
        yield G["s%d_nc" % i], G["s%d_ty" % i], G["s%d_tx" % i], G["s%d_path" % i]


def _token_of_frame(path):
    return np.where(path.sum(2) > 0, path.argmax(2), -1).astype(np.int16)


def _check_path_properties(path, t_ys, t_xs):
    """Size-independent properties: one token per valid frame, none beyond, starts at token 0, ends at t_x - 1, index moves by 0 or +1."""
    for b in range(path.shape[0]):
        ty, tx = int(t_ys[b]), int(t_xs[b])
        rows = path[b].sum(1)
        assert (rows[:ty] == 1).all() and (rows[ty:] == 0).all()
        idx = path[b, :ty].argmax(1)
        assert idx[0] == 0 and idx[-1] == tx - 1
        d = np.diff(idx)
        assert ((d == 0) | (d == 1)).all()


def test_oracle_matches_reference_fixtures():
    for nc, ty, tx, want in _small():
        assert np.array_equal(O.maximum_path(nc, ty, tx), want)
        assert np.array_equal(O.maximum_path_vectorised(nc, ty, tx), want)
        _check_path_properties(want, ty, tx)
    for i, (seed, B, Ty, Tx) in enumerate(LARGE):
        assert list(G["l%d_meta" % i]) == [seed, B, Ty, Tx]
        nc, ty, tx = large_case(seed, B, Ty, Tx)
        got = O.maximum_path_vectorised(nc, ty, tx)
        assert np.array_equal(_token_of_frame(got), G["l%d_token_of_frame" % i])
        _check_path_properties(got, ty, tx)


def test_oracle_matches_compiled_reference_when_present():
    """40 random ragged trials (every fourth with ties) against the paths the reference's compiled maximum_path_c returned
    (tests/golden/mas_reference_trials.npz, written by oracle/make_golden_reference.py)."""
    ref = np.load(os.path.join(ROOT, "tests", "golden", "mas_reference_trials.npz"))
    trials = list(mas_trials())
    assert len(trials) == len(ref.files) == 40
    for i, (nc, ty, tx) in enumerate(trials):
        assert np.array_equal(O.maximum_path(nc, ty, tx), ref["t%d_path" % i]), i


def test_abi_exports_mas():
    from vosk_tts_b200 import engine
    hdr = open(os.path.join(ROOT, "include", "vtts.h")).read()
    assert "vtts_maximum_path(" in hdr and "vtts_maximum_path_dev(" in hdr
    lib = engine.load_library()
    assert hasattr(lib, "vtts_maximum_path") and hasattr(lib, "vtts_maximum_path_dev")


@pytest.mark.gpu
def test_cuda_kernel_matches_fixtures_and_oracle():
    import torch
    from vosk_tts_b200 import monotonic_align as MA
    for nc, ty, tx, want in _small():
        assert np.array_equal(MA.maximum_path_numpy(nc, ty, tx), want)
    for i, (seed, B, Ty, Tx) in enumerate(LARGE):
        nc, ty, tx = large_case(seed, B, Ty, Tx)
        got = MA.maximum_path_numpy(nc, ty, tx)
        assert np.array_equal(_token_of_frame(got), G["l%d_token_of_frame" % i])
        _check_path_properties(got, ty, tx)
    # the reference's calling convention: torch tensors + mask, result on the same device, scores untouched
    nc, ty, tx = large_case(LARGE[0][0], *LARGE[0][1:])
    B, Ty, Tx = nc.shape
    mask = np.zeros((B, Ty, Tx), np.float32)
    for b in range(B):
        mask[b, : ty[b], : tx[b]] = 1
    d_nc = torch.as_tensor(nc, device="cuda")
    keep = d_nc.clone()
    attn = MA.maximum_path(d_nc, torch.as_tensor(mask, device="cuda"))
    assert attn.is_cuda and attn.dtype == d_nc.dtype and torch.equal(d_nc, keep)
    assert np.array_equal(_token_of_frame(attn.cpu().numpy().astype(np.int32)), G["l0_token_of_frame"])
    # ragged random cases incl. ties, full-size property check at a training-like shape (batch 32, 1000 frames, 200 tokens)
    rng = np.random.RandomState(5)
    for trial in range(10):
        B, Ty, Tx = rng.randint(1, 6), rng.randint(1, 300), rng.randint(1, 120)
        nc = (rng.randn(B, Ty, Tx) * 3).astype(np.float32)
        if trial % 3 == 0:
            nc = np.round(nc)
        ty = np.array([rng.randint(1, Ty + 1) for _ in range(B)], np.int32)
        tx = np.array([rng.randint(1, min(Tx, t) + 1) for t in ty], np.int32)
        assert np.array_equal(MA.maximum_path_numpy(nc, ty, tx), O.maximum_path_vectorised(nc, ty, tx))
    nc = (rng.randn(32, 1000, 200) * 4).astype(np.float32)
    ty = rng.randint(500, 1001, size=32).astype(np.int32)
    tx = rng.randint(60, 201, size=32).astype(np.int32)
    _check_path_properties(MA.maximum_path_numpy(nc, ty, tx), ty, tx)
    # error behaviour: more tokens than frames is refused, nothing is written
    from vosk_tts_b200.engine import VttsError
    with pytest.raises(VttsError):
        MA.maximum_path_numpy(nc[:1, :4, :8], [4], [8])
