"""SURVEY.md section 8f rank 3: the other inverse-STFT decoders of the reference (Multistream_iSTFT_Generator,
iSTFT_Generator).  The oracle restatement and the weight packing are pinned on CPU against what the UNMODIFIED reference
computed and exported (tests/golden/decoder_variants.npz, *_model_onnx.npz, written by oracle/make_golden_reference.py);
the CUDA engine's parity run for them is tests/test_gpu_parity.py::test_istft_decoder_variants_vs_oracle."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import onnx_fixture
from oracle import vits_oracle as vo
from oracle.make_golden_reference import VARIANT_SEED, VARIANT_T, VARIANT_VOCAB as N_VOCAB, variant_inputs, variant_training_json
from vosk_tts_b200 import config as C, synthetic, weights


def _training_json(flag):
    with open(os.path.join(GOLDEN, "reference_config.json")) as f:
        return variant_training_json(json.load(f), flag)


@pytest.mark.parametrize("flag,kind", [("ms_istft_vits", "ms_istft"), ("istft_vits", "istft"), ("mb_istft_vits", "mb_istft")])
def test_oracle_matches_reference_for_decoder_variant(flag, kind):
    tj = _training_json(flag)
    cfg = C.from_training_json(tj, n_vocab=N_VOCAB)
    assert cfg["decoder"] == kind and C.hop_total(cfg) == (64 if kind == "istft" else 256)
    folded = weights.fold_weight_norm(synthetic.make_random_checkpoint(cfg, VARIANT_SEED))
    tok, eps_dp, eps_z = variant_inputs(cfg)
    T = VARIANT_T
    scales = [0.8, 1.0, 0.8]
    torch.set_num_threads(1)
    with torch.no_grad():
        o = vo.infer(folded, cfg, tok, torch.tensor([T]), torch.tensor([2]), scales, eps_dp, eps_z, return_all=True)
    ref = np.load(os.path.join(GOLDEN, "decoder_variants.npz"))
    assert np.array_equal(o["w_ceil"][0, 0].numpy().astype(np.int32), ref[kind + "_w_ceil"])
    assert np.array_equal(o["idx"][0].numpy(), ref[kind + "_idx"])
    wav = o["o"][0, 0].numpy()
    assert o["o"].shape[:2] == (1, 1) and wav.size == int(ref[kind + "_wav_length"]) == int(o["y_lengths"][0]) * C.hop_total(cfg)
    assert float(np.abs(wav[ref[kind + "_wav_idx"]] - ref[kind + "_wav_val"]).max()) < 1e-5


@pytest.mark.parametrize("flag", ["ms_istft_vits", "istft_vits"])
def test_packed_tail_filter_is_what_the_decoder_applies(flag):
    """pack() hands the CUDA tail kernel one 63-tap filter per band: the learned multistream filter, or a unit impulse."""
    tj = _training_json(flag)
    cfg = C.from_training_json(tj, n_vocab=N_VOCAB)
    folded = weights.fold_weight_norm(synthetic.make_random_checkpoint(cfg, VARIANT_SEED))
    blob, man = weights.pack(folded, cfg, tc=False)
    ent = {}
    for line in man.strip().splitlines():
        parts = line.split()
        ent[parts[0]] = [int(x) for x in parts[1:]]
    off, n = ent["dec.pqmf"][0], ent["dec.pqmf"][1]
    bank = blob[off:off + n].reshape(-1, 63)
    if flag == "ms_istft_vits":
        assert np.array_equal(bank, folded["dec.multistream_conv_post.weight"][0].numpy())
        assert "dec.post.b" in ent            # models.py:1095: this conv_post has a bias
    else:
        assert bank.shape == (1, 63) and bank[0, 31] == 1.0 and np.count_nonzero(bank) == 1


def test_engine_config_accepts_every_istft_decoder():
    """All three inverse-STFT decoders map onto the same engine decoder type (the tail kernel takes the filter bank from
    the blob); the GPU parity runs are tests/test_gpu_parity.py::test_istft_decoder_variants_vs_oracle."""
    from vosk_tts_b200 import engine
    for flag in ("ms_istft_vits", "istft_vits", "mb_istft_vits"):
        cfg = C.from_training_json(_training_json(flag), n_vocab=N_VOCAB)
        cc = engine.make_c_config(cfg)
        assert cc.decoder_type == 0 and cc.subbands == (1 if flag == "istft_vits" else 4)


@pytest.mark.parametrize("flag,kind", [("ms_istft_vits", "ms_istft"), ("istft_vits", "istft")])
def test_variant_is_recognised_in_an_exported_graph(flag, kind, tmp_path):
    """model.onnx of the other decoders (exported with the reference recipe): configuration and every tensor pack() needs."""
    from vosk_tts_b200 import onnx_weights as ow
    tj = _training_json(flag)
    cfg = C.from_training_json(tj, n_vocab=N_VOCAB)
    path, _ = onnx_fixture.unpack(os.path.join(GOLDEN, kind + "_model_onnx.npz"), str(tmp_path / "model.onnx"))
    got = ow.config_from_onnx(path)
    assert got == cfg
    blob, man = weights.pack(ow.state_dict_from_onnx(path), got, tc=False)
    b2, m2 = weights.pack(weights.fold_weight_norm(synthetic.make_random_checkpoint(cfg, VARIANT_SEED)), cfg, tc=False)
    assert man == m2 and float(np.abs(blob - b2).max()) < 1e-6
