"""Weights and configuration straight from a ``model.onnx`` written by the reference's own export path
(training/vits2/onnx_export.py:60-104, run on the seeded reference model; stored as tests/golden/*_onnx.npz by
oracle/make_golden_reference.py and oracle/make_tiny_onnx.py, see oracle/onnx_fixture.py)."""
import os

import numpy as np
import pytest

from oracle import onnx_fixture
from vosk_tts_b200 import config as C, onnx_weights as ow, synthetic, weights

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def onnx_path(tmp_path_factory):
    """model.onnx of the full-size model from the seed-1234 synthetic checkpoint."""
    return onnx_fixture.unpack(os.path.join(GOLDEN, "model_onnx.npz"), str(tmp_path_factory.mktemp("onnx") / "model.onnx"))[0]


def test_state_dict_from_onnx_matches_folded_checkpoint(onnx_path):
    sd = ow.state_dict_from_onnx(onnx_path)
    ref = weights.fold_weight_norm(synthetic.make_random_checkpoint(C.DEFAULT_CONFIG, 1234))
    unused = {k for k in ref if k.startswith("dp.flows.1.")}          # the flow the reverse pass drops (models.py:94-96)
    for k, v in ref.items():
        v = v.detach().cpu().numpy() if hasattr(v, "detach") else np.asarray(v)
        if k in unused:
            assert k not in sd
            continue
        assert k in sd, k
        assert sd[k].shape == v.shape, k
        assert float(np.abs(sd[k] - v).max()) <= 1e-7, k               # 1-ulp differences of the weight-norm fold
    assert set(sd) <= set(ref)
    # the three anonymous constants: Linear weight (transposed), -logs of the ElementwiseAffine, the iSTFT basis
    assert sd["enc_p.encoder.spk_emb_linear.weight"].shape == (192, 256)
    assert sd["dp.flows.0.logs"].shape == (2, 1)


def test_config_from_onnx_recovers_the_training_configuration(onnx_path):
    cfg = ow.config_from_onnx(onnx_path)
    assert cfg == C.DEFAULT_CONFIG


def test_packed_blob_from_onnx_has_the_same_layout(onnx_path):
    sd = ow.state_dict_from_onnx(onnx_path)
    cfg = ow.config_from_onnx(onnx_path)
    ref = weights.fold_weight_norm(synthetic.make_random_checkpoint(C.DEFAULT_CONFIG, 1234))
    b1, m1 = weights.pack(sd, cfg)
    b2, m2 = weights.pack(ref, C.DEFAULT_CONFIG)
    assert m1 == m2 and b1.shape == b2.shape


def test_reader_rejects_non_onnx(tmp_path):
    p = tmp_path / "junk.onnx"
    p.write_bytes(b"\x08\x01")
    with pytest.raises(ValueError):
        ow.read_graph(str(p))


# ---- reduced-width model (tests/golden/tiny_model_onnx.npz + tiny_onnx.npz, oracle/make_tiny_onnx.py)
@pytest.fixture(scope="module")
def tiny_path(tmp_path_factory):
    return onnx_fixture.unpack(os.path.join(GOLDEN, "tiny_model_onnx.npz"), str(tmp_path_factory.mktemp("tiny") / "model.onnx"))[0]


def _tiny(path):
    g = np.load(os.path.join(GOLDEN, "tiny_onnx.npz"))
    return ow.state_dict_from_onnx(path), ow.config_from_onnx(path), g


def test_tiny_onnx_config_is_recovered(tiny_path):
    cfg = ow.config_from_onnx(tiny_path)
    assert (cfg["hidden_channels"], cfg["inter_channels"], cfg["filter_channels"], cfg["n_layers"], cfg["n_heads"]) == (64, 64, 128, 3, 2)
    assert (cfg["n_vocab"], cfg["n_speakers"], cfg["gin_channels"]) == (40, 4, 32)
    assert cfg["resblock_kernel_sizes"] == [3, 5] and cfg["resblock_dilation_sizes"] == [[1, 3, 5], [1, 3, 5]]
    assert cfg["upsample_rates"] == [4, 4] and cfg["upsample_kernel_sizes"] == [16, 16] and cfg["upsample_initial_channel"] == 64
    assert (cfg["subbands"], cfg["gen_istft_n_fft"], cfg["gen_istft_hop_size"]) == (4, 16, 4)
    assert (cfg["dp_filter_channels"], cfg["dp_n_flows"], cfg["dp_num_bins"], cfg["dp_kernel_size"]) == (256, 4, 10, 3)
    assert (cfg["flow_n_flows"], cfg["flow_wn_layers"], cfg["flow_kernel_size"]) == (4, 4, 5)


def test_oracle_on_onnx_weights_reproduces_the_reference_output(tiny_path):
    """model.onnx initializers -> oracle == the waveform the reference produced from the same module (CPU)."""
    import torch
    from oracle import vits_oracle as vo
    sd, cfg, g = _tiny(tiny_path)
    w = {k: torch.from_numpy(np.array(v)) for k, v in sd.items()}
    tok = torch.as_tensor(g["tokens"])[None]
    T = tok.shape[1]
    torch.set_num_threads(1)
    with torch.no_grad():
        o = vo.infer(w, cfg, tok, torch.tensor([T]), torch.tensor([int(g["sid"])]), g["scales"],
                     torch.as_tensor(g["eps_dp"])[None], torch.as_tensor(g["eps_z"])[None], return_all=True)
    assert int(o["y_lengths"][0]) == int(g["y_length"])
    assert np.array_equal(o["w_ceil"][0, 0].numpy().astype(np.int32), g["w_ceil"])
    assert np.array_equal(o["idx"][0].numpy().astype(np.int32), g["idx"])
    assert np.abs(o["o"][0, 0].numpy() - g["wav"]).max() < 1e-5


def test_session_packing_accepts_the_numpy_state_dict(tiny_path):
    """VitsSession folds + packs whatever Model hands it; for model.onnx that is a dict of numpy arrays."""
    sd, cfg, _ = _tiny(tiny_path)
    folded = weights.fold_weight_norm(sd)
    assert not weights.tc_supported(cfg)
    blob, man = weights.pack(folded, cfg)
    b2, m2 = weights.pack(sd, cfg, tc=False)
    assert man == m2 and np.array_equal(blob, b2)


@pytest.mark.gpu
def test_engine_from_onnx_initializers_reproduces_the_reference_output(tiny_path):
    """The deployment path end to end on the GPU: model.onnx -> initializers -> packed weights -> CUDA engine (fp32 mode:
    the reduced-width fixture has 64/32/16-channel convs, below the 64-multiple the tensor-core path packs)."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from vosk_tts_b200.engine import Engine
    sd, cfg, g = _tiny(tiny_path)
    blob, man = weights.pack(sd, cfg, tc=False)
    e = Engine(cfg, blob, man, device=0, precision=0)
    try:
        T = len(g["tokens"])
        for rep in range(3):          # eager, capture, replay
            ylen, dur = e.durations(g["tokens"][None], [T], [int(g["sid"])], g["scales"], g["eps_dp"][None], want_durations=True)
            assert int(ylen[0]) == int(g["y_length"])
            assert np.array_equal(dur[0], g["w_ceil"])
            wav = e.synthesize(ylen, g["eps_z"][None])
            assert np.abs(wav[0][: len(g["wav"])] - g["wav"]).max() < 1e-3
    finally:
        e.close()


@pytest.mark.gpu
def test_model_directory_in_deployed_layout_synthesizes(tmp_path, tiny_path):
    """What a vosk-tts user has on disk -- model.onnx + config.json + dictionary (vosk_tts/model.py:40-55) -- is all that
    `Model` / `Synth` need: text in, 22.05 kHz 16-bit WAV out, no checkpoint, no training json."""
    import json
    import shutil
    import wave
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from vosk_tts_b200.model import Model
    from vosk_tts_b200.synth import Synth
    phones = ["_", "^", "$", " ", ",", ".", "p", "rj", "i0", "i1", "v", "vj", "e0", "e1", "t", "j", "a0", "a1", "m", "mj", "r", "o0", "o1"]
    cfg = {"phoneme_id_map": {p: [i] for i, p in enumerate(phones)}, "inference": {"noise_level": 0.7, "speech_rate": 1.25},
           "model_type": "vits", "audio": {"sample_rate": 22050}}
    (tmp_path / "config.json").write_text(json.dumps(cfg), encoding="utf-8")
    (tmp_path / "dictionary").write_text("привет 1.0 p rj i0 vj e1 t\n", encoding="utf-8")
    shutil.copy(tiny_path, tmp_path / "model.onnx")
    m = Model(model_path=tmp_path)
    assert m.onnx.cfg["hidden_channels"] == 64 and m.onnx.cfg["n_speakers"] == 4
    s = Synth(m)
    out = tmp_path / "o.wav"
    s.synth("Привет, мир", str(out), speaker_id=3)
    with wave.open(str(out)) as w:
        assert (w.getnchannels(), w.getsampwidth(), w.getframerate()) == (1, 2, 22050)
        pcm = np.frombuffer(w.readframes(w.getnframes()), dtype=np.int16)
    assert len(pcm) > 0 and len(pcm) % 256 == 0 and int(m.onnx.last_y_lengths[0]) * 256 == len(pcm)
    assert pcm.std() > 10


def test_reader_rejects_external_data(tmp_path):
    """A TensorProto with data_location = EXTERNAL (field 14 = 1) cannot be served from the file alone: loud error."""
    def varint(n):
        out = b""
        while True:
            b7 = n & 0x7F
            n >>= 7
            out += bytes([b7 | (0x80 if n else 0)])
            if not n:
                return out
    def field(no, wt, payload):
        return varint((no << 3) | wt) + (varint(len(payload)) + payload if wt == 2 else payload)
    tensor = field(1, 0, varint(4)) + field(2, 0, varint(1)) + field(8, 2, b"w") + field(14, 0, varint(1))
    graph = field(5, 2, tensor)
    model = field(7, 2, graph)
    p = tmp_path / "ext.onnx"
    p.write_bytes(model)
    with pytest.raises(ValueError, match="external data"):
        ow.read_graph(str(p))
