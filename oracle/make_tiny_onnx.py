"""TEST INFRASTRUCTURE ONLY -- writes tests/golden/tiny_model_onnx.npz + tests/golden/tiny_onnx.npz.

A reduced-width VITS2 / MB-iSTFT model (same topology as the reference configuration, 64 instead of 192 channels, three
encoder layers, two resblock kernels) is built from the UNMODIFIED reference classes, exported with the reference's own
export recipe (training/vits2/onnx_export.py:60-104 via oracle/ref_harness.export_reference_onnx) and run once through
``SynthesizerTrn.infer`` with injected noise.  The exported file is stored in the compact form of oracle/onnx_fixture.py
(weights regenerated from the seed, exact bytes checked).  The fixture lets the GPU box (no reference tree there) prove the
deployment path end to end: model.onnx -> initializers -> packed weights -> engine == reference output.

Run in the build container:  python oracle/make_tiny_onnx.py
"""
import copy
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
N_VOCAB = 40


def tiny_training_json():
    j = copy.deepcopy(rh.load_ref_config())
    m = j["model"]
    m.update(inter_channels=64, hidden_channels=64, filter_channels=128, n_heads=2, n_layers=3, kernel_size=3,
             resblock_kernel_sizes=[3, 5], resblock_dilation_sizes=[[1, 3, 5], [1, 3, 5]], upsample_rates=[4, 4],
             upsample_initial_channel=64, upsample_kernel_sizes=[16, 16], gin_channels=32)
    j["data"]["n_speakers"] = 4
    return j


def main():
    torch.set_num_threads(1)
    tj = tiny_training_json()
    cfg = C.from_training_json(tj, n_vocab=N_VOCAB)
    sd = synthetic.make_random_checkpoint(cfg, 77)
    net = rh.build_reference_model(sd, cfg=tj, n_vocab=N_VOCAB)
    os.makedirs(OUT, exist_ok=True)
    with tempfile.TemporaryDirectory() as tmp:
        path = rh.export_reference_onnx(os.path.join(tmp, "model.onnx"), net, n_vocab=N_VOCAB)
        onnx_bytes = os.path.getsize(path)
        onnx_fixture.pack(path, os.path.join(OUT, "tiny_model_onnx.npz"), cfg, 77)
    g = torch.Generator().manual_seed(5)
    T, sid, scales = 23, 3, [0.8, 1.0, 0.8]
    tok = torch.randint(0, N_VOCAB, (1, T), generator=g)
    eps_dp = torch.randn(1, 2, T, generator=g)
    eps_z = torch.randn(1, cfg["inter_channels"], 24 * T + 8, generator=g)
    r = rh.reference_infer(net, tok, torch.tensor([T]), torch.tensor([sid]), scales, eps_dp, lambda s: eps_z[:, :, :s[2]])
    Ty = r["o"].shape[-1] // C.hop_total(cfg)
    attn = r["attn"][0, 0]
    np.savez_compressed(os.path.join(OUT, "tiny_onnx.npz"), tokens=tok[0].numpy().astype(np.int64), sid=np.int64(sid),
                        scales=np.asarray(scales, np.float32), eps_dp=eps_dp[0].numpy(), eps_z=eps_z[0, :, :Ty].numpy().copy(),
                        w_ceil=attn.sum(0).numpy().astype(np.int32), idx=attn.argmax(1).numpy().astype(np.int32),
                        y_length=np.int64(Ty), wav=r["o"][0, 0].numpy())
    print("tiny model: T_x", T, "T_y", Ty, "onnx bytes", onnx_bytes, "wav absmax %.3f" % float(r["o"].abs().max()))


if __name__ == "__main__":
    main()
