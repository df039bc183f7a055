"""Shared test helpers (golden loading, CSR flattening, wheel access)."""
import gzip, hashlib, json, os
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
ASSETS = os.path.join(ROOT, "assets")

GOLDEN_NAMES = ["gpt2", "gpt2_prefix", "llama3", "wordpiece", "bytes_only", "nonmonotone", "ignore_merges"]


def asset_json(name):
    return gzip.open(os.path.join(ASSETS, name + ".json.gz")).read().decode("utf-8")


def _set_path(d, dotted, value):
    ks = dotted.split(".")
    for k in ks[:-1]:
        d = d[k]
    d[ks[-1]] = value


def load_golden(name):
    """-> (tokenizer_json_str, cases)"""
    g = json.loads(gzip.open(os.path.join(GOLDEN, f"golden_{name}.json.gz")).read().decode("utf-8"))
    t = g["tokenizer"]
    if isinstance(t, str) and t.startswith("asset:"):
        tj = asset_json(t[6:])
    elif isinstance(t, dict) and "asset" in t:
        j = json.loads(asset_json(t["asset"]))
        for k, v in t["patch"].items():
            _set_path(j, k, v)
        tj = json.dumps(j)
    else:
        tj = json.dumps(t)
    return tj, g["cases"]


def cases_to_csr(cases):
    ids = np.array([i for c in cases for i in c["ids"]], dtype=np.uint32)
    offs = np.array([o for c in cases for o in c["offsets"]], dtype=np.uint32).reshape(-1, 2)
    wid = np.array([w for c in cases for w in c["word_ids"]], dtype=np.uint32)
    rp = np.zeros(len(cases) + 1, dtype=np.uint64)
    if cases:
        np.cumsum([len(c["ids"]) for c in cases], out=rp[1:])
    return ids, offs, wid, rp


def pack_docs(docs):
    bs = [d.encode("utf-8") for d in docs]
    off = np.zeros(len(bs) + 1, dtype=np.uint64)
    if bs:
        np.cumsum([len(b) for b in bs], out=off[1:])
    return np.frombuffer(b"".join(bs), dtype=np.uint8).copy(), off


def assert_csr_equal(got, exp, docs=None, what=""):
    names = ["ids", "offsets", "word_ids", "row_ptr"]
    for g, e, nm in zip(got, exp, names):
        if g is None:
            continue
        if not np.array_equal(np.asarray(g).reshape(-1), np.asarray(e).reshape(-1)):
            msg = f"{what}: {nm} differ"
            if docs is not None:
                grp, erp = np.asarray(got[3]), np.asarray(exp[3])
                for d in range(len(docs)):
                    a, b = int(erp[d]), int(erp[d + 1])
                    ga, gb = (int(grp[d]), int(grp[d + 1])) if d + 1 < len(grp) else (0, 0)
                    same = (gb - ga == b - a) and all(
                        x is None or np.array_equal(np.asarray(x)[ga:gb], np.asarray(y)[a:b]) for x, y in zip(got[:3], exp[:3]))
                    if not same:
                        msg += f"\n first differing doc {d}: {docs[d]!r}\n  exp ids {np.asarray(exp[0])[a:b].tolist()} off {np.asarray(exp[1])[a:b].tolist()}" \
                               f"\n  got ids {np.asarray(got[0])[ga:gb].tolist()} off {None if got[1] is None else np.asarray(got[1])[ga:gb].tolist()}"
                        break
            raise AssertionError(msg)


def wheel():
    """The reference implementation, if importable here (it is in the dev container and on the GPU image)."""
    try:
        import tokenizers
        return tokenizers
    except Exception:
        return None


def wheel_csr(tok, docs):
    encs = tok.encode_batch(docs, add_special_tokens=False)
    return cases_to_csr([{"ids": e.ids, "offsets": e.offsets, "word_ids": e.word_ids} for e in encs])


# ---------------------------------------------------------------------------------------------- recorded reference outputs
# What the reference implementation (the `tokenizers` wheel) returned for the tests' seeded inputs, kept as truncated SHA-256
# digests of a canonical JSON form, so that every comparison with it runs without the wheel and the file stays small.
# To record them again (the wheel importable): B2T_RECORD_REFERENCE=1 python -m pytest tests -k <tests>.  Every
# reference() call then runs the wheel and rewrites its entry.  The GPU tests record before they create the engine, so a
# machine without a GPU records their entries too (and then fails their engine part).
REFERENCE_DIGESTS = os.path.join(GOLDEN, "reference_digests.json")
RECORDING = os.environ.get("B2T_RECORD_REFERENCE") == "1"
_digests = None


def _plain(x):
    if isinstance(x, np.ndarray):
        return x.tolist()
    if isinstance(x, np.generic):
        return x.item()
    if isinstance(x, dict):
        return {str(k): _plain(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [_plain(v) for v in x]
    return x


def digest(x):
    js = json.dumps(_plain(x), sort_keys=True, separators=(",", ":"), ensure_ascii=False)
    return hashlib.sha256(js.encode("utf-8")).hexdigest()[:16]


def csr_plain(csr):
    """(ids, offsets, word_ids, row_ptr) in the form assert_csr_equal compares: flat, whatever the integer type"""
    return [np.asarray(a).reshape(-1).astype(np.int64) for a in csr]


def reference(key, fn):
    """The recorded digest of what the reference returned for `key`; when recording, fn() runs the wheel and replaces it."""
    global _digests
    if _digests is None:
        _digests = json.load(open(REFERENCE_DIGESTS))["digests"] if os.path.exists(REFERENCE_DIGESTS) else {}
    if RECORDING:
        _digests[key] = digest(fn())
        with open(REFERENCE_DIGESTS, "w") as f:
            json.dump({"generator": "B2T_RECORD_REFERENCE=1 python -m pytest tests (see tests/helpers.py)",
                       "tokenizers": wheel().__version__, "digests": dict(sorted(_digests.items()))}, f, indent=0)
            f.write("\n")
    assert key in _digests, f"no recorded reference output for {key}"
    return _digests[key]


def assert_reference(key, got, fn, what=""):
    """got must equal what the reference returned for `key` (fn() computes that with the wheel, only when recording)"""
    assert digest(got) == reference(key, fn), f"{what or key}: differs from the reference implementation's recorded output ({key})"


def wheel_tokenizer(tokenizer_json):
    """the reference's Tokenizer when recording, else None (the tests then compare with the recorded digests only)"""
    return wheel().Tokenizer.from_str(tokenizer_json) if RECORDING else None


# ---------------------------------------------------------------------------------------------- host-logic harness
def oracle_backed_tokenizer(tokenizer_json):
    """TEST ONLY: tokenizers_b200.Tokenizer's host logic (added tokens, templates, CSR stitching) in front of the ORACLE
    instead of the GPU engine, so that the host side can be checked on a box without a GPU.  The product class has no
    such switch: it always creates the CUDA engine."""
    import sys
    sys.path.insert(0, ROOT)
    from tokenizers_b200 import _lib
    from tokenizers_b200.tokenizer import Tokenizer
    from oracle.oracle import Oracle, OFF_CHAR, OFF_BYTE

    class OracleBacked(Tokenizer):
        def _create_engine(self, device):
            self._h = None
            self._orc = Oracle(tokenizer_json)

        def _engine_rows(self, data, row_off, flags, zero_copy=False):
            ids, offs, wid, rp = self._orc.encode_batch_csr(data, row_off, OFF_BYTE if flags & _lib.OFFSETS_BYTES else OFF_CHAR)
            return ids, (offs if flags & _lib.WANT_OFFSETS else None), (wid if flags & _lib.WANT_WORD_IDS else None), rp

    return OracleBacked(tokenizer_json)


ADDED_TOKEN_SPECS = [  # (content, single_word, lstrip, rstrip, normalized, special)
    ("<|endoftext|>", False, False, False, False, True),
    ("<mask>", False, True, False, False, True),
    ("[SEP2]", False, False, True, False, True),
    ("<both>", False, True, True, False, True),
    ("tok", True, False, False, True, False),
    ("Zürich", False, False, False, True, False),
    ("<a>", False, False, False, False, True),
    ("<a><b>", False, False, False, False, True),
    ("<|end", False, False, False, True, False),
    ("wörd", True, True, False, False, False),
]


def added_token_entries(vocab, specs):
    """ids the way the reference assigns them (added_vocabulary.rs:281-310): the model's id when the content is already
    in its vocabulary, else the next free id -- what a tokenizer.json written by the reference would contain"""
    nxt, out = len(vocab), []   # get_vocab_size of the model (the assets' vocabularies are dense, so this is also max id + 1)
    for c, sw, ls, rs, nm, sp in specs:
        if c in vocab:
            i = vocab[c]
        else:
            i, nxt = nxt, nxt + 1
        out.append({"id": i, "content": c, "single_word": sw, "lstrip": ls, "rstrip": rs, "normalized": nm, "special": sp})
    return out


def with_added_tokens(tokenizer_json, template=False):
    """asset tokenizer.json + the added tokens above (ids continue after the vocabulary) [+ a TemplateProcessing]"""
    js = json.loads(tokenizer_json)
    n = max(js["model"]["vocab"].values()) + 1
    js["added_tokens"] = added_token_entries(js["model"]["vocab"], ADDED_TOKEN_SPECS)
    if template:
        by = {e["content"]: e["id"] for e in js["added_tokens"]}
        bos, eos = by["<|endoftext|>"], by["<mask>"]
        js["post_processor"] = {"type": "TemplateProcessing",
                                "single": [{"SpecialToken": {"id": "<|endoftext|>", "type_id": 0}}, {"Sequence": {"id": "A", "type_id": 0}},
                                           {"SpecialToken": {"id": "<mask>", "type_id": 0}}],
                                "pair": [{"Sequence": {"id": "A", "type_id": 0}}, {"Sequence": {"id": "B", "type_id": 1}}],
                                "special_tokens": {"<|endoftext|>": {"id": "<|endoftext|>", "ids": [bos], "tokens": ["<|endoftext|>"]},
                                                   "<mask>": {"id": "<mask>", "ids": [eos], "tokens": ["<mask>"]}}}
    return json.dumps(js)


def added_token_docs(seed, n):
    """fuzz documents with the added tokens spliced in: glued to words, surrounded by spaces, back to back, truncated"""
    import random
    from fuzzgen import rand_doc
    rng = random.Random(seed)
    toks = [s[0] for s in ADDED_TOKEN_SPECS]
    docs = ["", "<|endoftext|>", "<|endoftext|><|endoftext|>", "a<|endoftext|>b", "x  <mask>  y", "x [SEP2] \n y", " \t<both>\n ",
            "tok", "a tok b", "atok", "tok.", "toktok", "tok tok", "Zürich", "inZürichx", "<a><b>", "<a><a><b>", "<a", "<|end", "<|endoftext",
            "<|endoftext|", "wörd", " wörd", "xwörd", "wörd!", "  <mask><both>  ", "<mask> tok <both>", "é<mask>é", "toké", "étok", "tok_", "tok1 1tok"]
    while len(docs) < n:
        parts = []
        for _ in range(rng.randint(1, 5)):
            parts.append(rand_doc(rng, 12))
            u = rng.random()
            if u < 0.75:
                t = rng.choice(toks)
                if rng.random() < 0.15:
                    t = t[:rng.randint(1, len(t))]
                parts.append(rng.choice(["", "", " ", "  ", "\n", " "]) + t + rng.choice(["", "", " ", "  ", "\t", "x", "1", "_"]))
        docs.append("".join(parts))
    return docs[:n]
