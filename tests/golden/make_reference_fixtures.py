"""Pins the oracle to the REFERENCE'S OWN Python (needs a checkout of the reference repository):

    python tests/golden/make_reference_fixtures.py <reference checkout>/scripts [--full]

The reference validates its Rust layers against `.npy` files produced by its torch scripts
(rms_norm.rs:156-211, rope.rs:168-253, swiglu.rs:100-187, conv.rs:113-215, rms_norm.rs:214-291,
attention.rs:476-619, mel.rs:486-614).  Those scripts are imported here UNMODIFIED from
the reference's scripts/ directory and run on our synthetic weights (dequantised to f32, served through a
`get_tensor` shim in place of `safe_open(consolidated.safetensors)`):

  A  ref_ops.npz       reference_forward.py  test_rms_norm / test_rope / test_swiglu / test_conv /
                       test_attention / test_ada_rms_norm  -- exactly the fixtures the Rust tests load;
                       weights = layer 0 of the full-size seed-42 synthetic model.
  B  ref_chain_small.npz
                       generate_padded_reference.py  compute_mel (torch.stft + mistral_common.audio.mel_filter_bank,
                       the real upstream package, importable here) and run_encoder(mel, f); then the body of
                       compare_full_forward.py main() (conv -> encoder -> adapter -> 26-layer decoder with ADA ->
                       tied lm_head; lifted by `ast` without editing the file) on a reference-SHAPED model:
                       every hard-coded dimension of the scripts is kept (1280 / 32x64 / 32 layers, 3072 / 32:8x128 /
                       26 layers) while ffn = 512, vocab = 4096 and layers i >= 2 alias the bytes of layer i % 2 in
                       the GGUF tensor index, so the file is 100 MB and the CPU test stays fast.
  C  ref_chain_full.npz (--full)  the same chain on the full-size seed-42 model (2.5 GB GGUF in /dev/shm).

Stored: inputs, reference outputs (row subsets of the [positions, dim] activations, plus per-row sums of the conv
output, audio embeddings and logits, so that each fixture stays below 1 MB).  Consumers: tests/test_oracle_vs_reference_py.py (CPU: oracle == reference Python)
and tests/test_reference_py_gpu.py (-m gpu: CUDA == reference Python).  The reference is NOT needed to run those tests.
"""
import ast
import contextlib
import importlib.util
import os
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import gguf_synth, mel as omel, q4 as oq4  # noqa: E402
from voxtral_mini_realtime_rs_b200 import synth       # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
REF_SCRIPTS = None       # the reference's scripts/ directory (first command-line argument)
SEED_FULL = 42
SEED_SMALL = 11
AUDIO_SECONDS = 1.0
AUDIO_SEED = 7
FULL_GGUF = os.environ.get("VOX_BENCH_GGUF", "/dev/shm/voxtral_synth_s42.gguf")
LOGIT_COLS = 64          # evenly spaced vocabulary columns stored per position
TOPK = 8


def load_ref_module(fname):
    spec = importlib.util.spec_from_file_location("ref_" + fname[:-3], os.path.join(REF_SCRIPTS, fname))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


class TensorShim:
    """Stands in for `safe_open(...)`: get_tensor(name) -> torch f32 (Q4 tensors dequantised by the rule of
    tensor.rs:83-113 as restated in oracle/q4.py).  Source: a GgufFile or per-tensor synthesis."""

    def __init__(self, gguf=None, cfg=None, seed=None):
        self.g, self.cfg, self.seed = gguf, cfg, seed
        self.man = {n: (dt, sh) for n, dt, sh in synth.tensor_manifest(cfg)} if cfg is not None else None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False

    def raw(self, name):
        if self.g is not None:
            dt, shape, _ = self.g.info(name)
            return dt, shape, self.g.raw(name)
        dt, shape = self.man[name]
        return dt, shape, synth.synth_tensor_bytes(name, dt, shape, self.seed)

    def get_tensor(self, name):
        dt, shape, raw = self.raw(name)
        if dt == synth.Q4_0_T:
            return torch.from_numpy(oq4.dequantize_c(np.ascontiguousarray(raw))).reshape(shape)
        if dt == synth.F16_T:
            return torch.from_numpy(raw.view(np.float16).astype(np.float32).reshape(shape))
        return torch.from_numpy(raw.view(np.float32).reshape(shape).copy())


@contextlib.contextmanager
def in_tmp_cwd():
    old = os.getcwd()
    with tempfile.TemporaryDirectory() as d:
        os.makedirs(os.path.join(d, "test_data"))
        os.chdir(d)
        try:
            yield d
        finally:
            os.chdir(old)


# ------------------------------------------------------------------ A: per-op fixtures
def make_ops():
    rf = load_ref_module("reference_forward.py")
    shim = TensorShim(cfg=synth.VoxtralConfig(), seed=SEED_FULL)
    rf.safe_open = lambda *a, **k: shim          # the scripts' `with safe_open(MODEL_PATH, ...) as f`
    out = {}
    with in_tmp_cwd() as d:
        for fn in (rf.test_rms_norm, rf.test_rope, rf.test_swiglu, rf.test_conv, rf.test_attention, rf.test_ada_rms_norm):
            fn()
        td = os.path.join(d, "test_data")
        ld = lambda n: np.load(os.path.join(td, n + ".npy"))  # noqa: E731
        for n in ("rms_norm_input", "rms_norm_weight", "rms_norm_output", "rope_cos", "rope_sin",
                  "swiglu_input", "swiglu_output", "conv_input", "conv_output", "attn_input", "attn_output",
                  "ada_rms_norm_input", "ada_rms_norm_t_embed", "ada_rms_norm_scale", "ada_rms_norm_output"):
            out[n] = ld(n)
        # RoPE is per head: 4 of the 32 heads keep the file small
        out["rope_input"] = ld("rope_input")[:, :, :4, :]
        out["rope_output"] = ld("rope_output")[:, :, :4, :]
        # weights are NOT stored: they are the seed-42 layer-0 tensors, regenerated by name in the tests;
        # a checksum guards against generator drift
        out["swiglu_w1_sum"] = np.float64(ld("swiglu_w1").astype(np.float64).sum())
        out["attn_wq_sum"] = np.float64(ld("attn_wq").astype(np.float64).sum())
    np.savez_compressed(os.path.join(HERE, "ref_ops.npz"), **out)
    print("ref_ops.npz:", {k: v.shape for k, v in out.items()})


# ------------------------------------------------------------------ B/C: the whole chain
def lift_full_forward(cf):
    """compare_full_forward.py main(): the body of `with safe_open(...) as f:` (conv .. logits) as a function of
    (mel [1,128,T], f), by AST -- the file itself is not edited.  Stops after `predicted = ...`."""
    src = open(os.path.join(REF_SCRIPTS, "compare_full_forward.py")).read()
    tree = ast.parse(src)
    main = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "main")
    w = next(n for n in main.body if isinstance(n, ast.With))
    body = []
    for st in w.body:
        body.append(st)
        if isinstance(st, ast.Assign) and isinstance(st.targets[0], ast.Name) and st.targets[0].id == "predicted":
            break
    ret = ast.parse("return dict(audio_embeds=audio_embeds_out, hidden=hidden, logits=logits, predicted=predicted)").body[0]
    # `x` is overwritten by the decoder: remember the adapter output where the script saves it
    for i, st in enumerate(body):
        if isinstance(st, ast.Expr) and "python_audio_embeds" in ast.unparse(st):
            body.insert(i, ast.parse("audio_embeds_out = x.clone()").body[0])
            break
    fn = ast.FunctionDef(name="lifted_forward", args=ast.arguments(posonlyargs=[], args=[ast.arg("mel"), ast.arg("f")],
                                                                   kwonlyargs=[], kw_defaults=[], defaults=[]),
                         body=body + [ret], decorator_list=[])
    mod = ast.Module(body=[fn], type_ignores=[])
    ast.fix_missing_locations(mod)
    ns = cf.__dict__
    exec(compile(mod, "compare_full_forward.py<lifted>", "exec"), ns)
    return ns["lifted_forward"]


def make_chain(gguf: gguf_synth.GgufFile, out_name: str, dense: bool):
    gp = load_ref_module("generate_padded_reference.py")
    cf = load_ref_module("compare_full_forward.py")
    audio = omel.peak_normalize(synth.speechlike(AUDIO_SECONDS, seed=AUDIO_SEED))
    padded = omel.pad_audio(audio)
    shim = TensorShim(gguf=gguf)
    t0 = time.time()
    mel = gp.compute_mel(padded)                              # [128, T] torch
    emb_a = gp.run_encoder(mel, shim)[0]                      # [S4, 3072]
    print(f"  run_encoder {time.time() - t0:.1f}s", tuple(mel.shape), tuple(emb_a.shape))
    fwd = lift_full_forward(cf)
    t0 = time.time()
    with in_tmp_cwd() as d, torch.no_grad():
        r = fwd(mel.unsqueeze(0), shim)
        conv = np.load(os.path.join(d, "test_data", "python_conv_output.npy"))[0]     # [S, 1280]
    print(f"  full forward {time.time() - t0:.1f}s")
    emb_b = r["audio_embeds"][0]
    # the two scripts implement the same encoder; they must agree before either is used as a pin
    assert float((emb_a - emb_b).abs().max()) < 1e-4, float((emb_a - emb_b).abs().max())
    logits = r["logits"][0]                                   # [S4, V]
    S4, V = logits.shape
    top = torch.topk(logits, TOPK, dim=-1)
    cols = np.linspace(0, V - 1, LOGIT_COLS).astype(np.int64)
    e = emb_a.numpy().astype(np.float32)
    h = r["hidden"][0].numpy().astype(np.float32)
    out = dict(seconds=np.float32(AUDIO_SECONDS), audio_seed=np.int32(AUDIO_SEED), mel=mel.numpy().astype(np.float32),
               predicted=np.array(r["predicted"], np.int32), top_idx=top.indices.numpy().astype(np.int32),
               top_val=top.values.numpy().astype(np.float32), cols=cols.astype(np.int32),
               logit_cols=logits[:, cols].numpy().astype(np.float32),
               logit_row_sums=logits.numpy().astype(np.float64).sum(1),
               emb_row_sums=e.astype(np.float64).sum(1), emb_row_abs_sums=np.abs(e).astype(np.float64).sum(1),
               conv_row_sums=conv.astype(np.float64).sum(1))
    if dense:       # every conv row, every other embedding / hidden row and the last one
        rows = np.array(sorted(set(range(0, S4, 2)) | {S4 - 1}), np.int32)
        crow = np.arange(conv.shape[0], dtype=np.int32)
    else:
        rows = np.array(sorted(set([0, 1, 2, S4 // 2, S4 - 2, S4 - 1])), np.int32)
        crow = np.array(sorted(set([0, 1, conv.shape[0] // 2, conv.shape[0] - 1])), np.int32)
    out.update(rows=rows, audio_embeds=e[rows], hidden=h[rows], conv_rows=crow, conv=conv[crow].astype(np.float32))
    np.savez_compressed(os.path.join(HERE, out_name), **out)
    marg = (top.values[:, 0] - top.values[:, 1]).numpy()
    print(f"{out_name}: S4={S4} V={V} distinct ids {len(set(r['predicted']))} min top-2 margin {marg.min():.3e}")


if __name__ == "__main__":
    if len(sys.argv) < 2 or not os.path.isdir(sys.argv[1]):
        sys.exit(__doc__.splitlines()[2])
    REF_SCRIPTS = sys.argv[1]
    torch.set_num_threads(os.cpu_count() or 8)
    make_ops()
    make_chain(gguf_synth.GgufFile(synth.build_aliased_gguf_bytes(synth.refshape_config(), SEED_SMALL)), "ref_chain_small.npz", dense=True)
    if "--full" in sys.argv:
        if not os.path.exists(FULL_GGUF):
            synth.write_synthetic_gguf(FULL_GGUF, synth.VoxtralConfig(), seed=SEED_FULL)
        make_chain(gguf_synth.GgufFile(FULL_GGUF), "ref_chain_full.npz", dense=False)
