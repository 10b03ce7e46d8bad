"""gRPC service (vosk_tts_b200/server.py) against the wire contract of the reference's server/tts_service.proto.
CPU tests use a stub Synth; the GPU test serves the real engine (tiny exported model) to concurrent clients."""
import json
import threading
from pathlib import Path

import numpy as np
import pytest

grpc = pytest.importorskip("grpc")
from vosk_tts_b200 import server as S  # noqa: E402


def test_messages_have_the_reference_wire_format():
    M = S.messages()
    # hand-encoded proto3: text (field 2, LEN) = "hi"; hints (field 3, LEN) = {speaker_id (1, VARINT) = 3}; hints = {speech_rate (2, I64) = 1.5}
    wire = bytes.fromhex("12026869" "1a020803" "1a09" "11000000000000f83f")
    req = M["UtteranceSynthesisRequest"](text="hi", hints=[M["Hints"](speaker_id=3), M["Hints"](speech_rate=1.5)])
    assert req.SerializeToString() == wire
    back = M["UtteranceSynthesisRequest"].FromString(wire)
    assert back.text == "hi" and back.WhichOneof("Utterance") == "text"
    assert back.hints[0].WhichOneof("Hint") == "speaker_id" and back.hints[0].speaker_id == 3
    assert back.hints[1].WhichOneof("Hint") == "speech_rate" and back.hints[1].speech_rate == 1.5
    # response: audio_chunk (1, LEN) = {data (1, LEN) = 4 bytes}
    resp = M["UtteranceSynthesisResponse"](audio_chunk=M["AudioChunk"](data=b"\x01\x00\xff\x7f"))
    assert resp.SerializeToString() == bytes.fromhex("0a06" "0a04" "0100ff7f")
    # output_audio_spec parses (field 4) even though the server ignores it, as the reference does
    spec = M["AudioFormatOptions"](raw_audio=M["RawAudio"](audio_encoding=1, sample_rate_hertz=22050))
    assert M["UtteranceSynthesisRequest"].FromString(M["UtteranceSynthesisRequest"](text="x", output_audio_spec=spec).SerializeToString()).output_audio_spec.raw_audio.sample_rate_hertz == 22050


class _StubSynth:
    """Deterministic PCM per (text, speaker, rate): lets concurrent clients check they got their own stream, in order."""

    def __init__(self):
        self.calls = []
        self.lock = threading.Lock()

    def _pcm(self, text, speaker_id, speech_rate):
        n = 256 * (3 + len(text))
        return ((np.arange(n) * (speaker_id + 1) + int(10 * speech_rate)) % 30000).astype(np.int16)

    def synth_audio(self, text, speaker_id=0, speech_rate=1.0):
        with self.lock:
            self.calls.append(("whole", text, speaker_id, speech_rate))
        if text == "boom":
            raise KeyError("unknown phoneme")
        return self._pcm(text, speaker_id, speech_rate)

    def synth_audio_stream(self, text, speaker_id=0, speech_rate=1.0, chunk_frames=64):
        with self.lock:
            self.calls.append(("stream", text, speaker_id, speech_rate))
        if text == "boom":
            raise KeyError("unknown phoneme")
        pcm = self._pcm(text, speaker_id, speech_rate)
        for i in range(0, len(pcm), 256 * chunk_frames):
            yield pcm[i:i + 256 * chunk_frames]


def test_streaming_service_over_loopback_with_concurrent_clients():
    stub = _StubSynth()
    srv, port = S.make_server(stub, "127.0.0.1:0", threads=4, chunk_frames=2)
    srv.start()
    try:
        addr = "127.0.0.1:%d" % port
        out = {}

        def client(k):
            text = "utterance number %d" % k
            out[k] = list(S.synthesize(addr, text, speaker_id=k, speech_rate=1.0 + 0.5 * k))

        ts = [threading.Thread(target=client, args=(k,)) for k in range(6)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        for k in range(6):
            want = stub._pcm("utterance number %d" % k, k, 1.0 + 0.5 * k)
            assert len(out[k]) == -(-len(want) // 512) and all(len(c) <= 1024 for c in out[k])      # 2 frames x 256 samples x 2 bytes
            assert np.array_equal(np.frombuffer(b"".join(out[k]), dtype="<i2"), want)
        assert sorted(c[2] for c in stub.calls) == list(range(6)) and all(c[0] == "stream" for c in stub.calls)
        # defaults when no hints are sent (tts_server.py:42-43): speaker 0, rate 1.0
        list(S.synthesize(addr, "plain"))
        assert stub.calls[-1] == ("stream", "plain", 0, 1.0)
        # a front-end error reaches the client as INVALID_ARGUMENT, the server keeps serving
        with pytest.raises(grpc.RpcError) as ei:
            list(S.synthesize(addr, "boom"))
        assert ei.value.code() == grpc.StatusCode.INVALID_ARGUMENT
        with pytest.raises(grpc.RpcError) as ei:
            list(S.synthesize(addr, "x", speech_rate=0.0))
        assert ei.value.code() == grpc.StatusCode.INVALID_ARGUMENT
        assert b"".join(S.synthesize(addr, "still alive", speaker_id=1))
    finally:
        srv.stop(0)


def test_single_message_mode_matches_the_reference_server_shape():
    stub = _StubSynth()
    srv, port = S.make_server(stub, "127.0.0.1:0", threads=2, chunk_frames=0)
    srv.start()
    try:
        chunks = list(S.synthesize("127.0.0.1:%d" % port, "one message", speaker_id=2))
        assert len(chunks) == 1 and stub.calls[-1][0] == "whole"
        assert np.array_equal(np.frombuffer(chunks[0], dtype="<i2"), stub._pcm("one message", 2, 1.0))
    finally:
        srv.stop(0)


@pytest.mark.gpu
def test_real_engine_behind_the_service(tmp_path):
    """Model directory in the deployed layout (tiny exported model) -> Model/Synth -> gRPC service; three concurrent clients
    (the reference shares one Synth across its thread pool, server/tts_server.py:37-38,57) each receive a chunked stream whose
    length is what the engine reported, and the single-message mode returns the same number of samples for the same text."""
    from vosk_tts_b200.model import Model
    from vosk_tts_b200.synth import Synth
    phones = ["_", "^", "$", " ", ",", ".", "p", "rj", "i0", "i1", "v", "vj", "e0", "e1", "t", "j", "a0", "a1", "m", "mj", "r", "o0", "o1"]
    cfg = {"phoneme_id_map": {p: [i] for i, p in enumerate(phones)}, "inference": {"noise_level": 0.7, "speech_rate": 1.0},
           "model_type": "vits", "audio": {"sample_rate": 22050}}
    (tmp_path / "config.json").write_text(json.dumps(cfg), encoding="utf-8")
    (tmp_path / "dictionary").write_text("привет 1.0 p rj i0 vj e1 t\nмир 1.0 m i1 r\n", encoding="utf-8")
    from oracle import onnx_fixture
    onnx_fixture.unpack(str(Path(__file__).parent / "golden" / "tiny_model_onnx.npz"), str(tmp_path / "model.onnx"))
    synth = Synth(Model(model_path=tmp_path))
    srv, port = S.make_server(synth, "127.0.0.1:0", threads=3, chunk_frames=8)
    srv.start()
    try:
        addr = "127.0.0.1:%d" % port
        res = {}

        def client(k):
            res[k] = list(S.synthesize(addr, "Привет, мир. " * (k + 1), speaker_id=k))

        ts = [threading.Thread(target=client, args=(k,)) for k in range(3)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        for k in range(3):
            pcm = np.frombuffer(b"".join(res[k]), dtype="<i2")
            assert len(res[k]) >= 2 and all(len(c) <= 8 * 256 * 2 for c in res[k])
            assert len(pcm) % 256 == 0 and pcm.std() > 10
        assert len(b"".join(res[2])) > len(b"".join(res[0]))
    finally:
        srv.stop(0)


class _LockingStub(_StubSynth):
    """Holds a lock for the duration of a stream, like VitsSession.run_stream holds the session lock."""

    def __init__(self):
        super().__init__()
        self.engine_lock = threading.Lock()

    def synth_audio_stream(self, text, speaker_id=0, speech_rate=1.0, chunk_frames=64):
        with self.engine_lock:
            pcm = self._pcm(text, speaker_id, speech_rate)
            for i in range(0, len(pcm), 256 * chunk_frames):
                yield pcm[i:i + 256 * chunk_frames]


def test_cancelled_stream_releases_the_engine():
    """A client that goes away in the middle of a stream must not leave the (single, shared) engine locked: the servicer closes
    the generator chain, the next request is served."""
    import time
    stub = _LockingStub()
    srv, port = S.make_server(stub, "127.0.0.1:0", threads=2, chunk_frames=1)
    srv.start()
    try:
        addr = "127.0.0.1:%d" % port
        M = S.messages()
        with grpc.insecure_channel(addr) as channel:
            call = channel.unary_stream("/%s/%s" % (S.SERVICE, S.METHOD), request_serializer=lambda m: m.SerializeToString(),
                                        response_deserializer=M["UtteranceSynthesisResponse"].FromString)
            it = call(M["UtteranceSynthesisRequest"](text="a long utterance that will be abandoned " * 20))
            first = next(it)
            assert len(first.audio_chunk.data) == 512
            it.cancel()
        t0 = time.time()
        while stub.engine_lock.locked() and time.time() - t0 < 10:
            time.sleep(0.05)
        assert not stub.engine_lock.locked(), "the abandoned stream still holds the engine"
        assert b"".join(S.synthesize(addr, "next request", speaker_id=1, timeout=10))
    finally:
        srv.stop(0)
