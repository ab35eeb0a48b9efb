"""CUDA path == the REFERENCE'S OWN torch scripts (fixtures tests/golden/ref_*.npz, generator
tests/golden/make_reference_fixtures.py: the reference's scripts/{reference_forward,generate_padded_reference,
compare_full_forward}.py run unmodified on our synthetic weights).  Everything through the C ABI.

Bounds: north_star -- encoder hidden states / audio embeddings within 1e-3 abs; logits of O(1) within 2e-3
(f32 summation order over K = 3072 and 26 layers); greedy ids exact wherever the reference's own top-2 margin
exceeds twice that; mel 1e-2 is what the reference accepts against this very file (mel.rs:534-614), we hold 5e-4.
"""
import os

import numpy as np
import pytest

from voxtral_mini_realtime_rs_b200 import synth

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")
FULL_GGUF = os.environ.get("VOX_BENCH_GGUF", "/dev/shm/voxtral_synth_s42.gguf")
ENC0 = f"{synth.ENC}.transformer.layers.0"


def maxdiff(a, b):
    return float(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max())


def _check_chain(vx, model, fx, what):
    audio = synth.speechlike(float(fx["seconds"]), seed=int(fx["audio_seed"]))
    # --- mel: peak-normalise + pad + GPU STFT/filterbank vs torch.stft + mistral_common filterbank
    ms = vx.MelSpectrogram.voxtral(0)
    padded = vx.pad_audio(vx.peak_normalize(audio))      # product host plumbing (vox_peak_normalize, vox_pad_audio)
    mel_gpu = ms.compute_log(padded).T        # [128, T]
    d_mel = maxdiff(mel_gpu, fx["mel"])
    assert mel_gpu.shape == fx["mel"].shape and d_mel < 5e-4, d_mel
    # --- encoder on the REFERENCE mel: conv stem, 32 layers, adapter
    model.debug("capture_on")
    try:
        emb = model.encode_audio(fx["mel"][None])[0]
        conv = model.debug("conv").reshape(-1, model.info["enc_dim"])
    finally:
        model.debug("capture_off")
    d_conv, d_emb = maxdiff(conv[fx["conv_rows"]], fx["conv"]), maxdiff(emb[fx["rows"]], fx["audio_embeds"])
    assert d_conv < 1e-3, d_conv
    assert d_emb < 1e-3, d_emb
    assert maxdiff(emb.astype(np.float64).sum(1), fx["emb_row_sums"]) < 2e-2
    # --- decoder + ADA + tied lm_head, teacher-forced with [STREAMING_PAD]*S like compare_full_forward.py:262-361
    s4 = emb.shape[0]
    lg = model.forward_streaming(fx["mel"][None], np.full((1, s4), 32, np.int32))[0]
    d_lg = maxdiff(lg[:, fx["cols"]], fx["logit_cols"])
    top_val = np.take_along_axis(lg, fx["top_idx"].astype(np.int64), axis=1)
    d_top = maxdiff(top_val, fx["top_val"])
    assert d_lg < 2e-3 and d_top < 2e-3, (d_lg, d_top)
    margin = fx["top_val"][:, 0] - fx["top_val"][:, 1]
    ids = lg.argmax(1)
    clear = margin > 4e-3
    assert clear.sum() >= 0.8 * s4
    assert np.array_equal(ids[clear], fx["predicted"][clear])
    n_eq = int((ids == fx["predicted"]).sum())
    print(f"\n[ref-py parity] {what}: mel {d_mel:.2e} conv {d_conv:.2e} audio_embeds {d_emb:.2e} logits {max(d_lg, d_top):.2e} "
          f"ids {n_eq}/{s4} (min reference margin {margin.min():.2e})")
    assert n_eq >= s4 - int((~clear).sum())


def test_chain_small_vs_reference_py(vx):
    fx = np.load(os.path.join(GOLD, "ref_chain_small.npz"))
    data = synth.build_aliased_gguf_bytes(synth.refshape_config(), seed=11)
    model = vx.Q4ModelLoader.from_bytes(data).load(0, max_batch=1, max_mel_frames=1000)
    try:
        _check_chain(vx, model, fx, "reference-shaped small model")
    finally:
        model.close()


@pytest.mark.slow
def test_chain_full_vs_reference_py(vx):
    fx = np.load(os.path.join(GOLD, "ref_chain_full.npz"))
    if not os.path.exists(FULL_GGUF):
        synth.write_synthetic_gguf(FULL_GGUF, synth.VoxtralConfig(), seed=42)
    model = vx.Q4ModelLoader.from_file(FULL_GGUF).load(0, max_batch=1, max_mel_frames=1000)
    try:
        _check_chain(vx, model, fx, "full-size seed-42 model")
    finally:
        model.close()


def test_swiglu_op_vs_reference_py(vx):
    """reference_forward.py:146-176 (the fixture swiglu.rs:100-187 loads) through the Q4 operator seam: three
    vox_q4_matmul calls on the layer-0 seed-42 weights, SiLU*up on the host."""
    ops = np.load(os.path.join(GOLD, "ref_ops.npz"))
    x = ops["swiglu_input"][0]                                   # [10, 1280]
    w = {}
    for n, shape in (("w1", (5120, 1280)), ("w3", (5120, 1280)), ("w2", (1280, 5120))):
        raw = synth.synth_tensor_bytes(f"{ENC0}.feed_forward.{n}.weight", synth.Q4_0_T, shape, 42)
        w[n] = vx.Q4Tensor.from_q4_bytes(raw, shape, 0)
    g = vx.q4_matmul(x[None], w["w1"])[0]
    u = vx.q4_matmul(x[None], w["w3"])[0]
    act = (g / (1.0 + np.exp(-g.astype(np.float64)))).astype(np.float32) * u
    out = vx.q4_matmul(act[None], w["w2"])[0]
    ref = ops["swiglu_output"][0]
    assert maxdiff(out, ref) < 1e-3 * max(1.0, float(np.abs(ref).max())), maxdiff(out, ref)   # swiglu.rs:183 accepts 1e-3
    del w
