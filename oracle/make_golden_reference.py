"""TEST INFRASTRUCTURE ONLY -- stores what the CPU tests compare against when they pin this project to the UNMODIFIED
reference, so that they run from the repository alone.  Needs the reference tree (VTTS_REFERENCE_ROOT) and, for the
Monotonic Alignment Search trials, oracle/_ref built by oracle/build_ref_mas.py.

    python oracle/build_ref_mas.py && python oracle/make_golden_reference.py

Writes under tests/golden/:
  reference_config.json        training/vits2/configs/mb_istft_vits2_multi.json as the reference loads it
  g2p_reference.json           [word, vosk_tts.g2p.convert(word)] for the words of tests/test_frontend.py
  mas_reference_trials.npz     the compiled reference maximum_path_c on the random trials of tests/test_mas.py
  reference_model.npz          reference model built from the seed-1234 synthetic checkpoint: a seeded sample (and the sum)
                               of every tensor of its state dict after remove_weight_norm, the iSTFT basis and PQMF filter,
                               the inverse spline on seeded inputs, and ``infer`` on two seeded utterances
  decoder_variants.npz         ``infer`` of the reduced-width model with each inverse-STFT decoder (durations, and the
                               waveform at a seeded sample of positions)
  model_onnx.npz, {ms_istft,istft}_model_onnx.npz
                               model.onnx exported with the reference recipe (oracle/onnx_fixture.py format)
"""
import copy
import glob
import importlib.util
import json
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import onnx_fixture, ref_harness as rh  # noqa: E402
from vosk_tts_b200 import config as C, synthetic  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
WEIGHT_SEED = 1234
SAMPLES_PER_TENSOR = 16
WAV_SAMPLES = 4096

# tests/test_decoder_variants.py: reduced-width model, one decoder flag set at a time
VARIANT_VOCAB, VARIANT_SEED, VARIANT_T = 40, 11, 19
VARIANTS = [("ms_istft_vits", "ms_istft"), ("istft_vits", "istft"), ("mb_istft_vits", "mb_istft")]


def variant_training_json(ref_json, flag):
    j = copy.deepcopy(ref_json)
    m = j["model"]
    m.update(inter_channels=64, hidden_channels=64, filter_channels=128, n_heads=2, n_layers=3, kernel_size=3,
             resblock_kernel_sizes=[3, 5], resblock_dilation_sizes=[[1, 3, 5], [1, 3, 5]], upsample_rates=[4, 4],
             upsample_initial_channel=64, upsample_kernel_sizes=[16, 16], gin_channels=32,
             mb_istft_vits=False, ms_istft_vits=False, istft_vits=False)
    m[flag] = True
    j["data"]["n_speakers"] = 4
    return j


def g2p_words():
    words = ["прив+ет", "абстр+акция", "+ёлка", "подъ+езд", "семь+я", "чащ+а", "й+од", "объявл+ение", "в+ьюга", "съ+ёмка",
             "по-р+усски", "+я", "мышь", "компь+ютер", "ш+ёлк", "Гог+оль"]
    letters = "абвгдеёжзийклмнопрстуфхцчшщъыьэюя"
    rng = np.random.RandomState(0)
    for _ in range(300):
        n = rng.randint(1, 9)
        w = "".join(letters[i] for i in rng.randint(0, len(letters), n))
        p = rng.randint(0, n)
        words.append(w[:p] + "+" + w[p:])
    return words


def mas_trials():
    """(neg_cent, t_ys, t_xs) of the random trials, ties included (every fourth trial is rounded)."""
    rng = np.random.RandomState(3)
    for trial in range(40):
        B, Ty, Tx = rng.randint(1, 4), rng.randint(1, 80), rng.randint(1, 30)
        nc = (rng.randn(B, Ty, Tx) * 3).astype(np.float32)
        if trial % 4 == 0:
            nc = np.round(nc)
        ty = np.array([rng.randint(1, Ty + 1) for _ in range(B)], np.int32)
        tx = np.array([rng.randint(1, min(Tx, t) + 1) for t in ty], np.int32)
        yield nc, ty, tx


def spline_inputs(n=4000):
    g = torch.Generator().manual_seed(5)
    x = torch.randn(n, generator=g) * 3.0
    return x, torch.randn(n, 10, generator=g), torch.randn(n, 10, generator=g), torch.randn(n, 9, generator=g)


def infer_inputs(T, seed):
    g = torch.Generator().manual_seed(seed)
    tok = torch.randint(0, 62, (1, T), generator=g)
    return tok, torch.randn(1, 2, T, generator=g), torch.randn(1, 192, 24 * T, generator=g)


def variant_inputs(cfg):
    g = torch.Generator().manual_seed(3)
    T = VARIANT_T
    tok = torch.randint(0, VARIANT_VOCAB, (1, T), generator=g)
    eps_dp = torch.randn(1, 2, T, generator=g)
    eps_z = torch.randn(1, cfg["inter_channels"], 400 * T, generator=g)     # the random SDP of this seed is slow-spoken
    return tok, eps_dp, eps_z


def sample_positions(size, n, seed):
    """Sorted flat indices of a seeded sample of n positions out of size (all of them when size <= n)."""
    return np.sort(np.random.RandomState(seed).choice(size, min(n, size), replace=False)).astype(np.int32)


def load_ref_mas():
    so = glob.glob(os.path.join(ROOT, "oracle", "_ref", "ref_mas_core*.so"))
    if not so:
        raise SystemExit("run oracle/build_ref_mas.py first")
    spec = importlib.util.spec_from_file_location("ref_mas_core", so[0])
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def main():
    torch.set_num_threads(1)
    os.makedirs(OUT, exist_ok=True)
    ref_json = rh.load_ref_config()
    with open(os.path.join(OUT, "reference_config.json"), "w") as f:
        json.dump(ref_json, f, indent=1)

    spec = importlib.util.spec_from_file_location("ref_g2p", os.path.join(rh.REF_ROOT, "vosk_tts", "g2p.py"))
    ref_g2p = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_g2p)
    with open(os.path.join(OUT, "g2p_reference.json"), "w", encoding="utf-8") as f:
        json.dump([[w, ref_g2p.convert(w)] for w in g2p_words()], f, ensure_ascii=False, indent=0)

    ref_mas = load_ref_mas()
    paths = {}
    for i, (nc, ty, tx) in enumerate(mas_trials()):
        p = np.zeros(nc.shape, np.int32)
        ref_mas.maximum_path_c(p, nc.copy(), ty, tx)
        paths["t%d_path" % i] = p.astype(np.int8)
    np.savez_compressed(os.path.join(OUT, "mas_reference_trials.npz"), **paths)

    cfg = C.from_training_json(rh.REF_CONFIG)
    sd = synthetic.make_random_checkpoint(cfg, WEIGHT_SEED)
    net = rh.build_reference_model(sd)
    out = {}
    keys = sorted(net.state_dict())
    out["state_keys"] = np.asarray(keys)
    idx, val, count, total = [], [], [], []
    for i, k in enumerate(keys):
        v = net.state_dict()[k].detach().float().reshape(-1)
        pos = sample_positions(v.numel(), SAMPLES_PER_TENSOR, i)
        idx.append(pos)
        val.append(v.numpy()[pos])
        count.append(len(pos))
        total.append(float(v.double().sum()))
    out["state_sample_idx"], out["state_sample_val"] = np.concatenate(idx), np.concatenate(val)
    out["state_sample_count"], out["state_sum"] = np.asarray(count, np.int32), np.asarray(total, np.float64)
    out["istft_inverse_basis"] = net.state_dict()["dec.stft.inverse_basis"][:, 0].numpy()
    out["pqmf_synthesis_filter"] = sys.modules["pqmf"].PQMF("cpu").synthesis_filter[0].numpy()
    x, uw, uh, ud = spline_inputs()
    out["spline_x_sum"] = np.float64(x.double().sum())
    out["spline_inverse"], _ = [t.numpy() for t in sys.modules["transforms"].piecewise_rational_quadratic_transform(
        x.clone(), uw.clone(), uh.clone(), ud.clone(), inverse=True, tails="linear", tail_bound=5.0)]
    for T, seed in [(24, 101), (77, 102)]:
        tok, eps_dp, eps_z = infer_inputs(T, seed)
        r = rh.reference_infer(net, tok, torch.tensor([T]), torch.tensor([3]), [0.667, 1.0, 0.8], eps_dp, lambda s: eps_z[:, :, : s[2]])
        pre = "infer_t%d_" % T
        out[pre + "o"], out[pre + "z"] = r["o"].numpy(), r["z"].numpy()
        out[pre + "attn"] = r["attn"].numpy().astype(np.int8)
    np.savez_compressed(os.path.join(OUT, "reference_model.npz"), **out)
    with tempfile.TemporaryDirectory() as tmp:
        path = rh.export_reference_onnx(os.path.join(tmp, "model.onnx"), net)
        onnx_fixture.pack(path, os.path.join(OUT, "model_onnx.npz"), cfg, WEIGHT_SEED)

    var = {}
    for flag, kind in VARIANTS:
        tj = variant_training_json(ref_json, flag)
        vcfg = C.from_training_json(tj, n_vocab=VARIANT_VOCAB)
        vnet = rh.build_reference_model(synthetic.make_random_checkpoint(vcfg, VARIANT_SEED), cfg=tj, n_vocab=VARIANT_VOCAB)
        tok, eps_dp, eps_z = variant_inputs(vcfg)
        r = rh.reference_infer(vnet, tok, torch.tensor([VARIANT_T]), torch.tensor([2]), [0.8, 1.0, 0.8], eps_dp,
                               lambda s: eps_z[:, :, :s[2]])
        attn = r["attn"][0, 0]
        var[kind + "_w_ceil"] = attn.sum(0).numpy().astype(np.int32)
        var[kind + "_idx"] = attn.argmax(1).numpy().astype(np.int32)
        wav = r["o"][0, 0].numpy()
        var[kind + "_wav_length"] = np.int64(wav.size)
        var[kind + "_wav_idx"] = sample_positions(wav.size, WAV_SAMPLES, 0)
        var[kind + "_wav_val"] = wav[var[kind + "_wav_idx"]]
        print(kind, "T_y", attn.shape[0], "samples", r["o"].shape[-1])
        if kind != "mb_istft":
            with tempfile.TemporaryDirectory() as tmp:
                path = rh.export_reference_onnx(os.path.join(tmp, "model.onnx"), vnet, n_vocab=VARIANT_VOCAB)
                onnx_fixture.pack(path, os.path.join(OUT, kind + "_model_onnx.npz"), vcfg, VARIANT_SEED)
    np.savez_compressed(os.path.join(OUT, "decoder_variants.npz"), **var)


if __name__ == "__main__":
    main()
