"""oracle/ == the REFERENCE'S OWN torch scripts (CPU; no GPU, no reference checkout needed at run time).

The fixtures under tests/golden/ref_*.npz were produced by tests/golden/make_reference_fixtures.py, which imports,
unmodified, the reference's scripts/{reference_forward,generate_padded_reference,compare_full_forward}.py -- the scripts
that write the `.npy` files the reference's Rust layer tests load (rms_norm.rs:156-211, rope.rs:168-253,
swiglu.rs:100-187, conv.rs:113-215, rms_norm.rs:214-291, attention.rs:476-619, mel.rs:486-614) -- and runs them on
our synthetic weights.  The Rust tests accept 1e-3 (mel: 1e-2) against those files; the oracle is held to 1e-5 per op
(chains: 2e-4 on O(1) activations), i.e. it differs from the reference Python by f32 summation order only.

Weights are regenerated from (seed, tensor name); a checksum stored with the fixtures guards against generator drift.
"""
import os

import numpy as np
import pytest
import torch

from oracle import gguf_synth, mel as omel
from oracle.model import OracleModel, apply_rope, rms_norm, rope_tables
from voxtral_mini_realtime_rs_b200 import synth

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")
ENC0 = f"{synth.ENC}.transformer.layers.0"
FULL_GGUF = os.environ.get("VOX_BENCH_GGUF", "/dev/shm/voxtral_synth_s42.gguf")


def maxdiff(a, b):
    return float(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max())


@pytest.fixture(scope="module")
def ops():
    return np.load(os.path.join(GOLD, "ref_ops.npz"))


@pytest.fixture(scope="module")
def layer0_oracle():
    """Oracle over a GGUF holding the full-size seed-42 tensors the per-op fixtures use (layer 0 only aliased to
    every layer, tiny vocabulary: nothing else is touched by these tests)."""
    cfg = synth.VoxtralConfig(vocab=32)
    return OracleModel(gguf_synth.GgufFile(synth.build_aliased_gguf_bytes(cfg, seed=42, unique=1)))


def test_rms_norm_matches_reference_py(ops):               # reference_forward.py:91-115 -> rms_norm.rs:156-211
    out = rms_norm(torch.from_numpy(ops["rms_norm_input"][0]), torch.from_numpy(ops["rms_norm_weight"]), 1e-5)
    assert maxdiff(out.numpy(), ops["rms_norm_output"][0]) < 1e-5
    w = synth.synth_tensor_bytes(f"{ENC0}.attention_norm.weight", synth.F32_T, (1280,), 42).view(np.float32)
    assert np.array_equal(w, ops["rms_norm_weight"])           # the fixture really is the seed-42 tensor


def test_rope_matches_reference_py(ops):                   # reference_forward.py:118-143 -> rope.rs:168-253
    cos, sin = rope_tables(64, 100, 1e6)
    # tables: torch computes theta ** (arange/dim) then outer; ours follows rope.rs:35-64 (f32 powf)
    assert maxdiff(cos.numpy(), ops["rope_cos"]) < 1e-5 and maxdiff(sin.numpy(), ops["rope_sin"]) < 1e-5
    out = apply_rope(torch.from_numpy(ops["rope_input"][0]), cos, sin, 0)
    assert maxdiff(out.numpy(), ops["rope_output"][0]) < 1e-5


def test_swiglu_matches_reference_py(ops, layer0_oracle):  # reference_forward.py:146-176 -> swiglu.rs:100-187
    om = layer0_oracle
    w1 = om.g.raw(f"{ENC0}.feed_forward.w1.weight")
    from oracle import q4 as oq4
    assert abs(float(oq4.dequantize_c(w1).astype(np.float64).sum()) - float(ops["swiglu_w1_sum"])) < 1e-6
    out = om.swiglu(torch.from_numpy(ops["swiglu_input"][0]), ENC0)      # the script's swiglu has no bias
    assert maxdiff(out.numpy(), ops["swiglu_output"][0]) < 1e-5 * max(1.0, float(np.abs(ops["swiglu_output"]).max()))


def test_conv_matches_reference_py(ops, layer0_oracle):    # reference_forward.py:179-215 -> conv.rs:113-215
    out = layer0_oracle.conv_downsample(torch.from_numpy(ops["conv_input"]))
    assert out.shape == ops["conv_output"].shape == (1, 1280, 25)
    assert maxdiff(out.numpy(), ops["conv_output"]) < 1e-5 * max(1.0, float(np.abs(ops["conv_output"]).max()))


def test_attention_matches_reference_py(ops, layer0_oracle):   # reference_forward.py:218-281 -> attention.rs:476-619
    out = layer0_oracle.encoder_attention_block(torch.from_numpy(ops["attn_input"][0]), 0)
    assert maxdiff(out.numpy(), ops["attn_output"][0]) < 1e-5 * max(1.0, float(np.abs(ops["attn_output"]).max()))


def test_ada_modulation_matches_reference_py(ops, layer0_oracle):  # reference_forward.py:284-333 -> rms_norm.rs:214-291
    scale1 = layer0_oracle.ada_scales(ops["ada_rms_norm_t_embed"].reshape(-1))[0]        # 1 + w2 gelu(w0 t)
    assert maxdiff(scale1.numpy() - 1.0, ops["ada_rms_norm_scale"].reshape(-1)) < 1e-5
    out = torch.from_numpy(ops["ada_rms_norm_input"][0]) * scale1
    assert maxdiff(out.numpy(), ops["ada_rms_norm_output"][0]) < 1e-5


# ------------------------------------------------------------------ whole chain
def _check_chain(om: OracleModel, fx, tol_mel, tol_act, tol_logit):
    audio = omel.peak_normalize(synth.speechlike(float(fx["seconds"]), seed=int(fx["audio_seed"])))
    mel = omel.mel_tensor_from_audio(audio)                      # [1,128,T] via oracle pad + STFT + filterbank
    # generate_padded_reference.py:37-75 (torch.stft + mistral_common mel_filter_bank); mel.rs:534-614 accepts 1e-2
    d_mel = maxdiff(mel[0], fx["mel"])
    assert mel[0].shape == fx["mel"].shape and d_mel < tol_mel, d_mel
    # from here on feed the REFERENCE mel so that each stage is compared on identical inputs
    cap = {}
    emb = om.encode_audio(fx["mel"][None], cap)
    conv = cap["conv"].numpy()
    d_conv = maxdiff(conv[fx["conv_rows"]], fx["conv"])
    d_emb = maxdiff(emb.numpy()[fx["rows"]], fx["audio_embeds"])
    assert d_conv < tol_act, d_conv
    assert maxdiff(conv.astype(np.float64).sum(1), fx["conv_row_sums"]) < 100 * tol_act
    assert d_emb < tol_act, d_emb
    assert maxdiff(emb.numpy().astype(np.float64).sum(1), fx["emb_row_sums"]) < 100 * tol_act
    s4 = emb.shape[0]
    logits, hidden = om.forward_streaming(None, [32] * s4, omel.time_embedding(6.0, 3072), audio_embeds=emb, return_hidden=True)
    h = hidden.numpy()[fx["rows"]]
    d_h = maxdiff(h, fx["hidden"])
    assert d_h < tol_act * 5, d_h
    lg = logits.numpy()
    d_lg = maxdiff(lg[:, fx["cols"]], fx["logit_cols"])
    assert d_lg < tol_logit, d_lg
    top_val = np.take_along_axis(lg, fx["top_idx"].astype(np.int64), axis=1)
    assert maxdiff(top_val, fx["top_val"]) < tol_logit
    # greedy ids: exact wherever the reference's own top-2 margin exceeds the logit tolerance
    margin = fx["top_val"][:, 0] - fx["top_val"][:, 1]
    ids = lg.argmax(1)
    clear = margin > 2 * tol_logit
    assert clear.sum() >= 0.8 * s4
    assert np.array_equal(ids[clear], fx["predicted"][clear])
    return dict(mel=d_mel, conv=d_conv, emb=d_emb, hidden=d_h, logits=d_lg, ids=f"{int((ids == fx['predicted']).sum())}/{s4}")


def test_chain_small_matches_reference_py():
    """compute_mel + run_encoder (generate_padded_reference.py:37-187) + decoder/ADA/lm_head
    (compare_full_forward.py:262-361) on the reference-shaped small model."""
    fx = np.load(os.path.join(GOLD, "ref_chain_small.npz"))
    om = OracleModel(gguf_synth.GgufFile(synth.build_aliased_gguf_bytes(synth.refshape_config(), seed=11)))
    r = _check_chain(om, fx, tol_mel=2e-4, tol_act=2e-4, tol_logit=1e-3)
    print("oracle vs reference python (small):", r)


@pytest.mark.slow
def test_chain_full_matches_reference_py():
    fx = np.load(os.path.join(GOLD, "ref_chain_full.npz"))
    if not os.path.exists(FULL_GGUF):
        synth.write_synthetic_gguf(FULL_GGUF, synth.VoxtralConfig(), seed=42)
    om = OracleModel(FULL_GGUF)
    r = _check_chain(om, fx, tol_mel=2e-4, tol_act=2e-4, tol_logit=1e-3)
    print("oracle vs reference python (full):", r)
