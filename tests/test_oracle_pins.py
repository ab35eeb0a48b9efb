"""Pins the CPU oracle against every closed-form known answer the reference's own tests hold for
the hot path (SURVEY 8c).  Each test names the reference test (file:line) it reproduces.  No GPU.
"""
import math

import numpy as np

from oracle import gguf_synth, mel as omel, q4 as oq4, tokenizer as otok


# ------------------------------------------------------------------ src/audio/mel.rs
def test_hann_window_periodic():          # mel.rs:384-396
    w = omel.hann_window(400)
    assert w.shape == (400,)
    assert abs(w[0]) < 1e-6
    assert abs(w[1] - 6.1690807e-5) < 1e-8


def test_hann_window_small():             # mel.rs:398-406
    assert np.allclose(omel.hann_window(4), [0.0, 0.5, 1.0, 0.5], atol=1e-6)


def test_mel_config_and_shapes():         # mel.rs:356-381, 424-435
    ms = omel.MelSpectrogram()
    assert ms.mel_basis.shape == (128, 201)
    assert ms.window.shape == (400,)
    out = ms.compute_log(np.zeros(16000, np.float32))
    assert out.shape[1] == 128


def test_silence_power_is_tiny():         # mel.rs:409-421
    mel = omel.MelSpectrogram().compute(np.zeros(16000, np.float32))
    assert mel.size > 0 and np.all(mel < 1e-6)


def test_sine_log_mel_range():            # mel.rs:438-456
    s = (0.5 * np.sin(2 * math.pi * 440.0 * np.arange(16000) / 16000.0)).astype(np.float32)
    lm = omel.MelSpectrogram().compute_log(s)
    assert lm.min() >= -2.0 and lm.max() <= 3.0


def test_num_frames():                    # mel.rs:459-465, SURVEY F5
    assert 99 <= omel.num_frames(16000) <= 101
    assert omel.num_frames(375040) == 2344
    assert omel.MelSpectrogram().compute_log(np.zeros(1600, np.float32)).shape[0] == omel.num_frames(1600)


def test_hz_mel_roundtrip():              # mel.rs:468-483
    for hz in (0.0, 100.0, 440.0, 1000.0, 4000.0, 8000.0):
        back = omel.mel_to_hz(omel.hz_to_mel(hz))
        assert abs(back - hz) < max(0.01, hz * 1e-4)
    assert abs(omel.hz_to_mel(1000.0) - 15.0) < 1e-4


def test_c_mel_matches_numpy_mel():       # the timed C port agrees with the numpy restatement
    lib = oq4._lib()
    x = omel.noise_chirp(2.0)
    out = np.empty((omel.num_frames(x.size), 128), np.float32)
    assert lib.oracle_mel_compute_log(x.ctypes.data, x.size, out.ctypes.data) == out.shape[0]
    assert np.abs(out - omel.MelSpectrogram().compute_log(x)).max() < 2e-4


# ------------------------------------------------------------------ src/audio/pad.rs, io.rs, chunk.rs
def test_pad_config_defaults():           # pad.rs:114-137
    c = omel.PadConfig()
    assert c.samples_per_token() == 1280
    assert c.left_pad_samples() == 76 * 1280 == 97280


def test_pad_exact_counts():              # pad.rs:139-218
    n = 255168                            # mary_had_lamb.wav, pad.rs:145
    left = 97280
    total = left + n
    right = omel.PadConfig().right_pad_samples(total)
    assert (total + right) % 1280 == 0
    padded = omel.pad_audio(np.ones(n, np.float32))
    assert padded.size == 375040
    assert omel.num_audio_tokens(padded.size) == 293
    assert np.all(padded[:left] == 0) and np.all(padded[left:left + n] == 1) and np.all(padded[left + n:] == 0)
    assert omel.pad_audio(np.zeros(256000, np.float32)).size == 375040   # 16 s (SURVEY 8d)


def test_peak_normalize():                # io.rs:59-68 (+ io.rs tests)
    s = np.array([0.1, -0.5, 0.25], np.float32)
    out = omel.peak_normalize(s, 0.95)
    assert abs(np.abs(out).max() - 0.95) < 1e-6
    z = np.zeros(8, np.float32)
    assert np.array_equal(omel.peak_normalize(z), z)


def test_chunk_plan():                    # chunk.rs tests
    assert not omel.needs_chunking(1500 * 160)
    assert omel.needs_chunking(1500 * 160 + 1)
    plan = omel.chunk_plan(500000, max_mel_frames=1200)
    assert [p[:2] for p in plan] == [(0, 192000), (192000, 384000), (384000, 500000)]
    assert [p[3] for p in plan] == [False, False, True]
    ov = omel.chunk_plan(1000 * 160, max_mel_frames=400, overlap_frames=100)
    assert ov[1][0] == 300 * 160
    assert omel.chunk_plan(0) == []


# ------------------------------------------------------------------ src/models/time_embedding.rs
def test_time_embedding_dim4():           # time_embedding.rs:91-128
    e = omel.time_embedding(1.0, 4)
    assert np.allclose(e, [math.cos(1.0), math.cos(0.01), math.sin(1.0), math.sin(0.01)], atol=1e-6)
    assert omel.time_embedding(6.0, 3072).shape == (3072,)
    z = omel.time_embedding(0.0, 8)
    assert np.allclose(z[:4], 1.0) and np.allclose(z[4:], 0.0)


# ------------------------------------------------------------------ src/gguf/tests.rs
def test_q4_block_dequant():              # tests.rs:190-227
    orig = ((np.arange(32, dtype=np.float32) - 15.5) / 15.5).astype(np.float32)
    raw = oq4.quantize_f32_to_q4_0(orig)
    assert raw.size == 18
    d = raw[:2].view(np.float16)[0]
    assert abs(float(d) - np.abs(orig).max() / 7.0) < 0.01
    assert np.abs(oq4.dequantize_q4_0(raw, 32) - orig).max() < 0.08


def test_q4_block_edge_cases():           # tests.rs:229-274
    assert np.all(oq4.dequantize_q4_0(oq4.quantize_f32_to_q4_0(np.zeros(32, np.float32))) == 0.0)
    u = np.full(32, 0.5, np.float32)
    assert np.abs(oq4.dequantize_q4_0(oq4.quantize_f32_to_q4_0(u)) - u).max() < 0.08
    large = ((np.arange(32, dtype=np.float32) - 15.5) * 100.0).astype(np.float32)
    dl = np.abs(large).max() / 7.0
    assert np.abs(oq4.dequantize_q4_0(oq4.quantize_f32_to_q4_0(large)) - large).max() < dl / 2 + 1.0


def test_test_quantiser_nibble_range():   # SURVEY quantiser note: never emits nibble 0
    rng = np.random.default_rng(0)
    raw = oq4.quantize_f32_to_q4_0(rng.standard_normal(32 * 64).astype(np.float32)).reshape(-1, 18)[:, 2:]
    assert (raw & 0xF).min() >= 1 and (raw >> 4).min() >= 1 and (raw & 0xF).max() <= 15


def test_q4_matmul_orders_agree():        # tests.rs:371-411 pattern, oracle-internal consistency
    k = n = 32
    wf = (np.sin(np.arange(n * k, dtype=np.float32) * np.float32(0.1)) * np.float32(0.5)).astype(np.float32)
    raw = oq4.quantize_f32_to_q4_0(wf)
    act = (np.arange(k, dtype=np.float32) * np.float32(0.1)).reshape(1, k)
    ref = oq4.reference_matmul(act, oq4.dequantize_q4_0(raw), 1, k, n)
    assert np.abs(oq4.q4_matmul_c(act, raw, n, k) - ref).max() < 1e-3
    assert np.array_equal(oq4.q4_matmul_c(act, raw, n, k), oq4.q4_matmul_shader_order(act, raw, n, k))
    assert np.array_equal(oq4.dequantize_c(raw), oq4.dequantize_q4_0(raw))


def test_gguf_reader_parse_header():      # tests.rs:281-306
    n = 32 * 64
    orig = np.sin(np.arange(n, dtype=np.float32) * np.float32(0.001) - np.float32(1.0)).astype(np.float32)
    raw = oq4.quantize_f32_to_q4_0(orig)
    data = gguf_synth.build_gguf_bytes([("test.weight", 2, (64, 32), raw)])  # GGUF dims [32, 64]
    g = gguf_synth.GgufFile(data)
    assert g.version == 3 and g.tensor_count() == 1
    dt, shape, _ = g.info("test.weight")
    assert dt == 2 and tuple(reversed(shape)) == (32, 64)
    assert np.array_equal(g.raw("test.weight"), raw)


def test_gguf_multiple_tensors():         # tests.rs:308-325
    a = oq4.quantize_f32_to_q4_0(np.full(1024, 0.1, np.float32))
    b = oq4.quantize_f32_to_q4_0(np.full(2048, 0.2, np.float32))
    c = oq4.quantize_f32_to_q4_0(np.full(2048, -0.1, np.float32))
    g = gguf_synth.GgufFile(gguf_synth.build_gguf_bytes(
        [("weight_a", 2, (32, 32), a), ("weight_b", 2, (32, 64), b), ("weight_c", 2, (64, 32), c)]))
    assert g.tensor_count() == 3
    assert g.info("weight_b") is not None and g.info("nonexistent") is None
    assert np.array_equal(g.raw("weight_c"), c)


def test_manifest_matches_reference_counts():   # SURVEY Appendix A: 711 tensors, Q4 payload 2 488 393 728 B
    man = gguf_synth.tensor_manifest(gguf_synth.VoxtralConfig())
    assert len(man) == 711
    q4b = sum(gguf_synth._nbytes(dt, sh) for _, dt, sh in man if dt == 2)
    assert q4b == 2_488_393_728
    dec = sum(gguf_synth._nbytes(dt, sh) for n, dt, sh in man if dt == 2 and n.startswith("layers."))
    emb = gguf_synth._nbytes(2, (131072, 3072))
    assert dec == 1_705_107_456 and emb == 226_492_416 and dec + emb == 1_931_599_872   # BASELINE.md §2


# ------------------------------------------------------------------ src/tokenizer/mod.rs
def test_tokenizer_semantics():           # mod.rs:170-208 (+ tests 216-270 without the real tekken.json)
    t = otok.VoxtralTokenizer.from_json(otok.synthetic_tekken_json(300, 8))
    assert t.vocab_size == 308
    assert t.decode([]) == ""
    assert t.decode([1, 2, 999]) == ""                      # control ids skipped
    # id-1000 indexes the vocab *position*: position 8+65 holds byte 65 ('A')
    assert t.decode([1000 + 8 + 65, 1000 + 8 + 66]) == "AB"
    assert t.decode([1000 + 8 + 0xC3, 1000 + 8 + 0xA9]) == "é"   # multi-token UTF-8 sequence
    assert t.decode([1000 + 8 + 0xC3]) == "�"                    # lossy
    assert t.decode([1000 + 5]) == ""                       # control entry has no bytes -> skipped
    assert t.decode([1000 + 100000]) == ""                  # unknown id silently skipped
    assert t.decode_token(3) == "<ctl3>" and t.decode_token(900) is None
    assert t.decode_token(1000 + 8 + 262) == " s262"        # token_str fallback (262 % 7 == 3)
    assert t.decode_token(1000 + 8 + 259) == " w259"        # base64 token_bytes


def test_tokenizer_reference_golden_if_available():        # mod.rs:255-268
    """The reference's golden on the real vocabulary: tests/golden/tekken_excerpt.json holds the config and the eight
    entries these ids index of the public Tekken vocabulary (mistral_common's tekken_240911.json); every other
    position of the 131072-entry vocabulary is left empty."""
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "tekken_excerpt.json")) as f:
        doc = json.load(f)
    vocab = [{"rank": r, "token_bytes": None, "token_str": None} for r in range(doc["config"]["default_vocab_size"])]
    for e in doc["vocab"]:
        vocab[e["rank"]] = e
    t = otok.VoxtralTokenizer({"config": doc["config"], "vocab": vocab})
    assert t.decode([1362, 19135, 1294, 1278, 4618, 40307, 3910, 1046]) == " I spoke in the original phonograph."


def test_vectorised_port_agrees_with_strict_order_port():
    """oracle/q4_fast.c (the timed CPU baseline of bench.py) against oracle/q4_ref.c (the checker's strict
    shader-order arithmetic): same result to f32 re-association noise, for matvec and small-M shapes, odd
    block counts and a bias."""
    rng = np.random.default_rng(11)
    for (m, n, k) in [(1, 96, 3072), (3, 50, 160), (8, 33, 96)]:
        raw = np.empty((n * k // 32, 18), np.uint8)
        raw[:, :2] = rng.uniform(0.002, 0.02, n * k // 32).astype(np.float16).view(np.uint8).reshape(-1, 2)
        raw[:, 2:] = rng.integers(0, 256, (n * k // 32, 16), dtype=np.uint8)
        raw = raw.reshape(-1)
        x = rng.standard_normal((m, k)).astype(np.float32)
        bias = rng.standard_normal(n).astype(np.float32)
        strict = oq4.q4_matmul_c(x, raw, n, k, bias, threads=2)
        oq4.FAST = True
        try:
            fast = oq4.q4_matmul_c(x, raw, n, k, bias, threads=2)
        finally:
            oq4.FAST = False
        assert np.abs(fast - strict).max() < 2e-5 * max(1.0, np.abs(strict).max())
