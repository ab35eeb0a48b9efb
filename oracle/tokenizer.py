"""Tekken decode-only tokenizer oracle (test infrastructure, see oracle/__init__.py).

Restates src/tokenizer/mod.rs: from_json 125-164 (per-vocab-index bytes: base64
`token_bytes`, else UTF-8 of `token_str`; `is_control` entries go to a rank->str map),
decode 170-191 (ids < 1000 skipped; id-1000 indexes the vocab *position*; unknown ids
skipped; bytes joined then lossy UTF-8), decode_token 194-208.

Pinned: the reference's golden (`[1362,19135,1294,1278,4618,40307,3910,1046]` ->
" I spoke in the original phonograph.", mod.rs:255-268) on the entries of the public Tekken
vocabulary it uses (tests/golden/tekken_excerpt.json); behaviour is otherwise pinned on
synthetic vocabularies.
"""
from __future__ import annotations

import base64
import json

TEXT_TOKEN_OFFSET = 1000


class VoxtralTokenizer:
    def __init__(self, obj: dict):
        self.vocab_size = int(obj["config"]["default_vocab_size"])
        vocab = obj["vocab"]
        self.vocab_bytes = [None] * len(vocab)
        self.special_tokens = {}
        for idx, e in enumerate(vocab):
            if e.get("is_control", False):
                if e.get("token_str") is not None:
                    self.special_tokens[int(e["rank"])] = e["token_str"]
                continue
            tb = e.get("token_bytes")
            if tb is not None:
                try:
                    self.vocab_bytes[idx] = base64.b64decode(tb, validate=True)
                    continue
                except Exception:
                    pass
            if e.get("token_str") is not None:
                self.vocab_bytes[idx] = e["token_str"].encode("utf-8")

    @staticmethod
    def from_json(s: str) -> "VoxtralTokenizer":
        return VoxtralTokenizer(json.loads(s))

    @staticmethod
    def from_file(path: str) -> "VoxtralTokenizer":
        with open(path, "r", encoding="utf-8") as f:
            return VoxtralTokenizer(json.load(f))

    def decode(self, ids) -> str:
        out = bytearray()
        for i in ids:
            if i < TEXT_TOKEN_OFFSET:
                continue
            v = i - TEXT_TOKEN_OFFSET
            if v < len(self.vocab_bytes) and self.vocab_bytes[v] is not None:
                out += self.vocab_bytes[v]
        return out.decode("utf-8", errors="replace")

    def decode_token(self, i: int):
        if i < TEXT_TOKEN_OFFSET:
            return self.special_tokens.get(i)
        v = i - TEXT_TOKEN_OFFSET
        if v < len(self.vocab_bytes) and self.vocab_bytes[v] is not None:
            return self.vocab_bytes[v].decode("utf-8", errors="replace")
        return None


def synthetic_tekken_json(n_vocab: int = 300, n_special: int = 8) -> str:
    """A small tekken.json-shaped document for tests (no real file is available offline)."""
    vocab = []
    for r in range(n_special):
        vocab.append({"rank": r, "token_bytes": None, "token_str": f"<ctl{r}>", "is_control": True})
    for r in range(n_vocab):
        if r < 256:
            b = bytes([r])
        else:
            b = (" w%d" % r).encode()
        e = {"rank": n_special + r, "token_bytes": base64.b64encode(b).decode(), "token_str": None}
        if r % 7 == 3 and r >= 256:  # exercise the token_str fallback
            e = {"rank": n_special + r, "token_bytes": None, "token_str": " s%d" % r}
        vocab.append(e)
    doc = {"config": {"pattern": "", "num_vocab_tokens": n_vocab, "default_vocab_size": n_vocab + n_special,
                      "default_num_special_tokens": n_special, "version": "v7"},
           "vocab": vocab}
    return json.dumps(doc)
