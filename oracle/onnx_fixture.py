"""TEST INFRASTRUCTURE ONLY -- stores a ``model.onnx`` written by the reference exporter as a small fixture.

An exported graph is mostly float32 initializers, and those are the weight-norm-folded tensors of a seeded synthetic
checkpoint (``vosk_tts_b200.synthetic.make_random_checkpoint``).  ``pack`` XORs the raw bytes of every named float
initializer with the same tensor regenerated from the seed, folded with ``torch._weight_norm`` (the function the
reference's ``remove_weight_norm`` calls), so what is left is nearly all zero bits and compresses with lzma to a few
hundred KB.  ``unpack`` reverses it and checks the SHA-256 of the original file: the tests read byte for byte the file
the reference exported, or fail loudly if the seeded generator has drifted.  Anonymous initializers (``onnx::*``) and
everything that is not an initializer are stored as they are.
"""
import hashlib
import json
import lzma

import numpy as np
import torch


def _varint(buf, pos):
    out, shift = 0, 0
    while True:
        b = buf[pos]
        pos += 1
        out |= (b & 0x7F) << shift
        if not b & 0x80:
            return out, pos
        shift += 7


def _fields(buf, start, end):
    """(field number, wire type, value start, value end) of the message in buf[start:end]."""
    pos = start
    while pos < end:
        key, pos = _varint(buf, pos)
        fno, wt = key >> 3, key & 7
        if wt == 0:
            _, nxt = _varint(buf, pos)
        elif wt == 1:
            nxt = pos + 8
        elif wt == 2:
            ln, pos = _varint(buf, pos)
            nxt = pos + ln
        elif wt == 5:
            nxt = pos + 4
        else:
            raise ValueError("unsupported protobuf wire type %d" % wt)
        yield fno, wt, pos, nxt
        pos = nxt


def _float_initializers(buf):
    """(name, byte offset, byte length) of the raw_data of every float32 initializer of ModelProto.graph."""
    for fno, wt, gs, ge in _fields(buf, 0, len(buf)):
        if fno != 7 or wt != 2:
            continue
        for f2, w2, ts, te in _fields(buf, gs, ge):
            if f2 != 5 or w2 != 2:
                continue
            name, dtype, raw = "", 1, None
            for f3, w3, s, e in _fields(buf, ts, te):
                if f3 == 8:
                    name = bytes(buf[s:e]).decode()
                elif f3 == 2:
                    dtype = _varint(buf, s)[0]
                elif f3 == 9:
                    raw = (s, e - s)
            if dtype == 1 and raw is not None:
                yield name, raw[0], raw[1]


def _predicted(cfg, seed):
    from vosk_tts_b200 import synthetic
    sd = synthetic.make_random_checkpoint(cfg, seed)
    out = {}
    for k, v in sd.items():
        if k.endswith(".weight_v"):
            base = k[: -len("_v")]
            out[base] = torch._weight_norm(v.float(), sd[base + "_g"].float(), 0)
        elif not k.endswith(".weight_g") and torch.is_floating_point(v):
            out[k] = v.float()
    return {k: np.ascontiguousarray(v.detach().numpy()).view(np.uint8).ravel() for k, v in out.items()}


def _xor_predicted(buf, cfg, seed):
    pred = _predicted(cfg, seed)
    for name, off, n in _float_initializers(buf):
        p = pred.get(name)
        if p is not None and p.size == n:
            view = np.frombuffer(buf, np.uint8, n, off)
            view ^= p


def pack(onnx_path, out_path, cfg, seed):
    with open(onnx_path, "rb") as f:
        data = f.read()
    buf = bytearray(data)
    _xor_predicted(buf, cfg, seed)
    np.savez(out_path, onnx_xz=np.frombuffer(lzma.compress(bytes(buf), preset=9), np.uint8),
             cfg=np.asarray(json.dumps(cfg, sort_keys=True)), seed=np.int64(seed),
             sha256=np.asarray(hashlib.sha256(data).hexdigest()))
    return out_path


def unpack(fixture_path, onnx_path):
    """Writes the exported model.onnx stored in ``fixture_path`` to ``onnx_path``; returns (path, the model's config)."""
    g = np.load(fixture_path)
    cfg = json.loads(str(g["cfg"]))
    buf = bytearray(lzma.decompress(g["onnx_xz"].tobytes()))
    _xor_predicted(buf, cfg, int(g["seed"]))
    if hashlib.sha256(buf).hexdigest() != str(g["sha256"]):
        raise RuntimeError("%s: the seeded synthetic checkpoint no longer reproduces the exported weights" % fixture_path)
    with open(onnx_path, "wb") as f:
        f.write(buf)
    return onnx_path, cfg
