"""CPU: host-side logic -- weight packing layouts, config mapping, C-ABI surface, sharding."""
import os
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import ROOT
from vosk_tts_b200 import config as C
from vosk_tts_b200 import parallel, weights


def _manifest(man):
    out = {}
    for line in man.splitlines():
        n, o, c = line.split()
        out[n] = (int(o), int(c))
    return out


def _get(blob, man, name):
    o, c = man[name]
    return blob[o:o + c]


def test_library_exports_every_declared_symbol():
    from vosk_tts_b200 import engine
    hdr = open(os.path.join(ROOT, "include", "vtts.h")).read()
    declared = sorted(set(re.findall(r"\b(vtts_[a-z_0-9]+)\s*\(", hdr)))
    assert declared, "no prototypes parsed"
    lib = engine.load_library()
    for name in declared:
        assert hasattr(lib, name), "libvtts.so does not export %s" % name
    assert sorted(engine.EXPORTS) == declared


def test_engine_fails_loudly_without_gpu(packed, cfg):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from vosk_tts_b200.engine import Engine, VttsError
    with pytest.raises(VttsError):
        Engine(cfg, packed[0], packed[1], device=0)


def test_conv_pack_layout(folded, packed, cfg):
    blob, man = packed
    man = _manifest(man)
    w = folded["enc_p.encoder.ffn_layers.3.conv_1.weight"].numpy()       # [768,192,3]
    p = _get(blob, man, "enc.3.ffn1.w").reshape(3, 192, 768)
    assert np.array_equal(p, np.transpose(w, (2, 1, 0)))
    # Cout = 29 is padded to 32 columns of zeros
    w = folded["dp.flows.7.proj.weight"].numpy()
    p = _get(blob, man, "dp.cf4.proj.w").reshape(1, 256, 32)
    assert np.array_equal(p[0, :, :29], w[:, :, 0].T) and not p[0, :, 29:].any()


def test_gate_interleave_and_cond_rows(folded, packed, cfg):
    blob, man = packed
    man = _manifest(man)
    H = cfg["hidden_channels"]
    w = folded["flow.flows.2.enc.in_layers.1.weight"].numpy()            # [384,192,5]
    p = _get(blob, man, "flow.1.in1.w").reshape(5, H, 2 * H)
    assert np.array_equal(p[:, :, 0::2], np.transpose(w[:H], (2, 1, 0)))     # tanh half -> even columns
    assert np.array_equal(p[:, :, 1::2], np.transpose(w[H:], (2, 1, 0)))     # sigmoid half -> odd columns
    cw = _get(blob, man, "cond.w").reshape(-1, cfg["gin_channels"])
    r0 = H + cfg["dp_filter_channels"] + (1 * 4 + 1) * 2 * H                  # flow 1, layer 1
    ref = folded["flow.flows.2.enc.cond_layer.weight"].numpy()[2 * H:4 * H, :, 0]
    assert np.array_equal(cw[r0:r0 + 2 * H][0::2], ref[:H]) and np.array_equal(cw[r0:r0 + 2 * H][1::2], ref[H:])


def test_flip_folding(folded, packed, cfg):
    blob, man = packed
    man = _manifest(man)
    # flow 3 (processed first, after one Flip) is "flipped": pre reads reversed inputs, post writes reversed rows
    w = folded["flow.flows.6.pre.weight"].numpy()[:, :, 0]               # [192,96]
    p = _get(blob, man, "flow.3.pre.w").reshape(96, 192)
    assert np.array_equal(p, w[:, ::-1].T)
    w = folded["flow.flows.4.pre.weight"].numpy()[:, :, 0]
    p = _get(blob, man, "flow.2.pre.w").reshape(96, 192)
    assert np.array_equal(p, w.T)
    w = folded["flow.flows.6.post.weight"].numpy()[:, :, 0]              # [96,192]
    p = _get(blob, man, "flow.3.post.w").reshape(192, 96)
    assert np.array_equal(p, w[::-1].T)


@pytest.mark.parametrize("u,K", [(4, 16), (8, 16), (2, 4)])
def test_convt_polyphase_equals_conv_transpose(u, K):
    g = torch.Generator().manual_seed(u * 100 + K)
    ci, co, L = 6, 5, 19
    x = torch.randn(1, ci, L, generator=g)
    w = torch.randn(ci, co, K, generator=g)
    ref = F.conv_transpose1d(x, w, stride=u, padding=(K - u) // 2)[0].numpy()     # [co, u*L]
    out = np.zeros_like(ref)
    xn, wn = x[0].numpy(), w.numpy()
    for r, (pad, js) in enumerate(weights.convt_phases(u, K)):
        for t in range(L):
            acc = np.zeros(co)
            for m, j in enumerate(js):
                q = t - pad + m
                if 0 <= q < L:
                    acc += xn[:, q] @ wn[:, :, j]
            out[:, u * t + r] = acc
    assert np.abs(out - ref).max() < 1e-4


def test_config_mapping_from_reference_json():
    """The reference's training/vits2/configs/mb_istft_vits2_multi.json (tests/golden/reference_config.json)."""
    path = os.path.join(ROOT, "tests", "golden", "reference_config.json")
    assert C.from_training_json(path) == C.DEFAULT_CONFIG
    assert C.hop_total(C.DEFAULT_CONFIG) == 256


def test_lpt_sharding_balanced_and_complete():
    rng = np.random.RandomState(1)
    lens = rng.randint(64, 257, size=64)
    shards = parallel.lpt_shards(lens, 8)
    assert sorted(i for s in shards for i in s) == list(range(64))
    loads = [int(lens[s].sum()) for s in shards]
    assert max(loads) - min(loads) <= 256
    assert parallel.lpt_shards(lens, 8) == shards


def test_session_rejects_non_vits_feeds():
    from vosk_tts_b200.session import VitsSession
    s = VitsSession.__new__(VitsSession)    # no engine needed for feed validation
    with pytest.raises(ValueError):
        VitsSession.run(s, None, {"input": np.zeros((1, 4), np.int64), "input_lengths": [4], "scales": [0, 1, 0],
                                   "sid": [0], "bert": np.zeros((1, 768, 4), np.float32), "phone_duration_extra": None})
    with pytest.raises(ValueError):
        VitsSession.run(s, None, {"input": np.zeros((1, 5, 4), np.int64), "input_lengths": [4], "scales": [0, 1, 0],
                                   "sid": [0], "bert": None, "phone_duration_extra": None})


def test_training_json_selects_the_decoder_like_the_reference():
    """SynthesizerTrn.__init__ picks the decoder by flag precedence mb > ms > istft > plain (models.py:1585-1606)."""
    from vosk_tts_b200 import config as C
    base = {"data": {"n_speakers": 3, "sampling_rate": 22050},
            "model": {"inter_channels": 64, "hidden_channels": 64, "filter_channels": 128, "n_heads": 2, "n_layers": 3,
                      "kernel_size": 3, "resblock": "1", "resblock_kernel_sizes": [3], "resblock_dilation_sizes": [[1, 3, 5]],
                      "upsample_rates": [4, 4], "upsample_initial_channel": 64, "upsample_kernel_sizes": [16, 16],
                      "subbands": 4, "gen_istft_n_fft": 16, "gen_istft_hop_size": 4, "gin_channels": 32,
                      "use_transformer_flows": True, "transformer_flow_type": "pre_conv2"}}
    import copy
    def cfg(**flags):
        j = copy.deepcopy(base)
        j["model"].update(flags)
        return C.from_training_json(j, n_vocab=10)
    assert cfg(mb_istft_vits=True, ms_istft_vits=True)["decoder"] == "mb_istft"
    assert cfg(ms_istft_vits=True, istft_vits=True)["decoder"] == "ms_istft"
    c = cfg(istft_vits=True)
    assert c["decoder"] == "istft" and c["subbands"] == 1 and C.hop_total(c) == 4 * 4 * 4
    assert cfg()["decoder"] == "hifigan" and C.hop_total(cfg()) == 16
    assert C.hop_total(cfg(mb_istft_vits=True)) == 256
