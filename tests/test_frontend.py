"""CPU: the vosk_tts-compatible Model/Synth front end (host logic) with a stub session in place of the GPU engine."""
import json
import os
import wave

import numpy as np
import pytest

from vosk_tts_b200 import g2p
from vosk_tts_b200.model import Model, load_dictionary
from vosk_tts_b200.synth import Synth


class _StubSession:
    def __init__(self):
        self.feeds = None

    def run(self, names, feeds):
        self.feeds = feeds
        n = 256 * 3 * feeds["input"].shape[1]
        t = np.arange(n, dtype=np.float32)
        return [(1.5 * np.sin(t * 0.01)).reshape(1, 1, 1, n)]     # beyond +-1: exercises the int16 clip


def _model_dir(tmp_path):
    phones = ["_", "^", "$", " ", ",", ".", "p", "rj", "i0", "i1", "v", "vj", "e0", "e1", "t", "j", "a0", "a1", "m", "mj", "r", "o0", "o1"]
    cfg = {"phoneme_id_map": {p: [i] for i, p in enumerate(phones)}, "inference": {"noise_level": 0.7, "speech_rate": 1.25},
           "model_type": "vits"}
    (tmp_path / "config.json").write_text(json.dumps(cfg), encoding="utf-8")
    (tmp_path / "dictionary").write_text("привет 0.5 p rj i0 vj e0 t\nпривет 1.0 p rj i0 vj e1 t\n", encoding="utf-8")
    return tmp_path


def test_dictionary_keeps_most_probable(tmp_path):
    d = load_dictionary(_model_dir(tmp_path) / "dictionary")
    assert d == {"привет": "p rj i0 vj e1 t"}


def test_synth_builds_reference_feeds_and_wav(tmp_path):
    sess = _StubSession()
    m = Model(model_path=_model_dir(tmp_path), session=sess)
    s = Synth(m)
    ids = s.g2p_noembed("Привет, мир")
    assert ids[0] == 1 and ids[-1] == 2 and ids[1::2] == [0] * (len(ids) // 2)       # ^ ... $, blanks interspersed
    out = tmp_path / "o.wav"
    s.synth("Привет, мир", str(out), speaker_id=3)
    f = sess.feeds
    assert f["input"].dtype == np.int64 and f["input"].shape == (1, len(ids)) and list(f["input_lengths"]) == [len(ids)]
    assert np.allclose(f["scales"], [0.7, 1 / 1.25, 0.8]) and list(f["sid"]) == [3]
    assert f["bert"] is None and f["phone_duration_extra"] is None
    with wave.open(str(out)) as w:
        assert (w.getnchannels(), w.getsampwidth(), w.getframerate()) == (1, 2, 22050)
        pcm = np.frombuffer(w.readframes(w.getnframes()), dtype=np.int16)
    assert pcm.max() == 32767 and pcm.min() == -32767


def test_unsupported_model_types_raise(tmp_path):
    d = _model_dir(tmp_path)
    cfg = json.loads((d / "config.json").read_text(encoding="utf-8"))
    cfg["model_type"] = "multistream_v2"
    (d / "config.json").write_text(json.dumps(cfg), encoding="utf-8")
    with pytest.raises(ValueError):
        Model(model_path=d, session=_StubSession())


def test_missing_model_is_an_error_not_a_download():
    with pytest.raises(FileNotFoundError):
        Model(model_name="vosk-model-tts-ru-0.9-multi")


def test_g2p_matches_reference_converter():
    """vosk_tts.g2p.convert of the reference on hand-picked and seeded random stressed words (tests/golden/g2p_reference.json,
    written by oracle/make_golden_reference.py)."""
    from oracle.make_golden_reference import g2p_words
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "g2p_reference.json"), encoding="utf-8") as f:
        ref = json.load(f)
    words = g2p_words()
    assert [w for w, _ in ref] == words and len(words) == 316
    for w, want in ref:
        assert g2p.convert(w) == want, w


class _StubEngine:
    hop = 256

    def __init__(self):
        self.calls = []

    def synthesize_stream(self, ids, sid, scales, chunk_frames=64, noise_dp=None, noise_z=None, seed=0):
        self.calls.append((ids.copy(), sid, np.array(scales), chunk_frames, seed))
        frames = 3 * ids.shape[1]
        for f0 in range(0, frames, chunk_frames):
            n = (min(frames, f0 + chunk_frames) - f0) * self.hop
            yield np.full(n, 0.5, np.float32)


def test_streaming_front_end_chunks_lock_and_lengths(tmp_path):
    """Synth.synth_audio_stream -> VitsSession.run_stream -> Engine.synthesize_stream: same feeds as synth_audio, int16 chunks,
    the session lock is held while a stream is open and released when it ends or is abandoned."""
    import threading
    from vosk_tts_b200.session import VitsSession
    sess = VitsSession.__new__(VitsSession)
    sess.cfg, sess.engine, sess._lock, sess._seed, sess._calls = {}, _StubEngine(), threading.Lock(), 7, 0
    sess.last_y_lengths = sess.last_wav_lengths = None
    m = Model(model_path=_model_dir(tmp_path), session=sess)
    s = Synth(m)
    ids = s.g2p_noembed("Привет, мир")
    chunks = list(s.synth_audio_stream("Привет, мир", speaker_id=3, chunk_frames=10))
    frames = 3 * len(ids)
    assert len(chunks) == -(-frames // 10) and all(c.dtype == np.int16 for c in chunks)
    assert sum(c.size for c in chunks) == frames * 256 and int(chunks[0][0]) == int(0.5 * 32767)
    got_ids, sid, scales, cf, seed = sess.engine.calls[-1]
    assert got_ids.tolist() == [ids] and sid == 3 and cf == 10 and np.allclose(scales, [0.7, 1 / 1.25, 0.8])
    assert list(sess.last_wav_lengths) == [frames * 256] and list(sess.last_y_lengths) == [frames]
    assert not sess._lock.locked()
    gen = s.synth_audio_stream("Привет", speaker_id=0, chunk_frames=4)
    next(gen)
    assert sess._lock.locked()                      # a second request would wait here until the stream is finished
    gen.close()
    assert not sess._lock.locked()
    # two consecutive streams draw different seeds (per-call Philox seed, like run())
    list(s.synth_audio_stream("Привет", chunk_frames=64))
    assert sess.engine.calls[-1][4] != sess.engine.calls[-2][4]
    with pytest.raises(ValueError):
        list(sess.run_stream({"input": np.zeros((2, 3), np.int64), "input_lengths": np.array([3, 3]), "scales": np.ones(3, np.float32)}))
