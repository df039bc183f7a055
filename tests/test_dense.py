"""Dense mode (b2t_encode_batch_dense*): special-token template + truncation + padding on the device.
CPU: the oracle-side restatement (oracle.dense_rows) against the reference wheel's recorded outputs.  GPU: the engine against both."""
import ctypes, json, os
import numpy as np
import pytest
import helpers, fuzzgen, corpus
from oracle import oracle as orc

TEMPLATES = {
    "gpt2_style": lambda v: {"type": "TemplateProcessing",
                             "single": [{"SpecialToken": {"id": "<s>", "type_id": 0}}, {"Sequence": {"id": "A", "type_id": 0}},
                                        {"SpecialToken": {"id": "</s>", "type_id": 0}}, {"SpecialToken": {"id": "<s>", "type_id": 0}}],
                             "pair": [{"Sequence": {"id": "A", "type_id": 0}}, {"Sequence": {"id": "B", "type_id": 1}}],
                             "special_tokens": {"<s>": {"id": "<s>", "ids": [v["a"]], "tokens": ["a"]},
                                                "</s>": {"id": "</s>", "ids": [v["b"], v["c"]], "tokens": ["b", "c"]}}},
    "wordpiece": lambda v: {"type": "BertProcessing", "sep": ["[SEP]", v["[SEP]"]], "cls": ["[CLS]", v["[CLS]"]]},
    "llama3_style": lambda v: None,
}
# (truncation | None, padding)
SETTINGS = [
    (dict(max_length=16, direction="right"), dict(length=16, direction="right", pad_id=0)),
    (dict(max_length=12, direction="left"), dict(length=None, direction="left", pad_id=3)),
    (dict(max_length=40, direction="right"), dict(length=None, direction="right", pad_id=1, pad_to_multiple_of=8)),
    (None, dict(length=None, direction="right", pad_id=2)),
    (dict(max_length=7, direction="right"), dict(length=20, direction="left", pad_id=5, pad_to_multiple_of=16)),
]


def tokenizer_json(name):
    js = json.loads(helpers.asset_json(name))
    pp = TEMPLATES[name](js["model"]["vocab"])
    js["post_processor"] = pp
    return json.dumps(js)


def docs_for(seed):
    return fuzzgen.rand_docs(seed, 600, max_len=120) + ["", " ", "a", "hello world " * 30]


def spec_of(js, tr, pd):
    """the tokenizer's template as (pre ids, post ids) + the settings, for oracle.dense_rows"""
    from tokenizers_b200.tokenizer import parse_post_processor
    tp = parse_post_processor(json.loads(js).get("post_processor"))
    pre = [t for t, _ in tp["pre"]] if tp else []
    post = [t for t, _ in tp["post"]] if tp else []
    return dict(length=pd["length"] or 0, pad_to_multiple_of=pd.get("pad_to_multiple_of") or 0, max_length=tr["max_length"] if tr else 0,
                pad_id=pd["pad_id"], truncate_left=bool(tr and tr["direction"] == "left"), pad_left=pd["direction"] == "left", pre=pre, post=post)


def wheel_dense(js, docs, tr, pd):
    tok = helpers.wheel_tokenizer(js)
    if tr:
        tok.enable_truncation(tr["max_length"], direction=tr["direction"])
    tok.enable_padding(direction=pd["direction"], pad_id=pd["pad_id"], length=pd["length"], pad_to_multiple_of=pd.get("pad_to_multiple_of"))
    encs = tok.encode_batch(docs)
    return (np.array([e.ids for e in encs], dtype=np.uint32).reshape(len(docs), -1),
            np.array([e.attention_mask for e in encs], dtype=np.uint8).reshape(len(docs), -1))


@pytest.mark.parametrize("name", list(TEMPLATES))
def test_oracle_dense_matches_wheel(name):
    js = tokenizer_json(name)
    o = orc.Oracle(js)
    docs = docs_for(11)
    helpers.assert_reference("dense/docs11", docs, lambda: docs)
    ids, _, _, rp = o.encode_batch(docs)
    for k, (tr, pd) in enumerate(SETTINGS):
        got = orc.dense_rows(ids, rp, **spec_of(js, tr, pd))
        helpers.assert_reference(f"dense/{name}/{k}/docs11", got[:2], lambda: wheel_dense(js, docs, tr, pd), f"{name} {tr} {pd}")
        assert np.array_equal(got[2], got[1].sum(axis=1))


def _golden():
    import gzip
    return json.loads(gzip.open(os.path.join(helpers.GOLDEN, "golden_dense.json.gz")).read().decode("utf-8"))


@pytest.mark.parametrize("name", list(TEMPLATES))
def test_oracle_dense_matches_golden(name):
    """the same restatement against committed vectors of the wheel (no wheel needed)"""
    g = _golden()
    js = tokenizer_json(name)
    ids, _, _, rp = orc.Oracle(js).encode_batch(g["docs"])
    for k, (tr, pd) in enumerate(SETTINGS):
        c = g["cases"][f"{name}/{k}"]
        got = orc.dense_rows(ids, rp, **spec_of(js, tr, pd))
        assert list(got[0].shape) == c["shape"] and got[0].reshape(-1).tolist() == c["ids"] and got[2].tolist() == c["lengths"], (name, k)


def _apply(tok, tr, pd):
    tok.no_truncation(); tok.no_padding()
    if tr:
        tok.enable_truncation(tr["max_length"], direction=tr["direction"])
    tok.enable_padding(direction=pd["direction"], pad_id=pd["pad_id"], length=pd["length"], pad_to_multiple_of=pd.get("pad_to_multiple_of"))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TEMPLATES))
def test_gpu_dense_matches_oracle_and_wheel(name):
    from tokenizers_b200 import Tokenizer
    js = tokenizer_json(name)
    docs = docs_for(12)
    helpers.assert_reference("dense/docs12", docs, lambda: docs)
    # the reference's outputs first, so that recording them needs no GPU
    wheel = [helpers.reference(f"dense/{name}/{k}/docs12", lambda: wheel_dense(js, docs, tr, pd)) for k, (tr, pd) in enumerate(SETTINGS)]
    tok, o = Tokenizer.from_str(js), orc.Oracle(js)
    ids, _, _, rp = o.encode_batch(docs)
    for k, (tr, pd) in enumerate(SETTINGS):
        _apply(tok, tr, pd)
        got = tok.encode_batch_dense(docs)
        exp = orc.dense_rows(ids, rp, **spec_of(js, tr, pd))
        assert got["input_ids"].shape == exp[0].shape, (name, tr, pd)
        assert np.array_equal(got["input_ids"], exp[0]) and np.array_equal(got["attention_mask"], exp[1]) and np.array_equal(got["lengths"], exp[2]), (name, tr, pd)
        assert helpers.digest((got["input_ids"], got["attention_mask"])) == wheel[k], (name, tr, pd, "wheel")
    g = _golden()   # and the committed vectors of the wheel
    for k, (tr, pd) in enumerate(SETTINGS):
        _apply(tok, tr, pd)
        got = tok.encode_batch_dense(g["docs"])
        c = g["cases"][f"{name}/{k}"]
        assert list(got["input_ids"].shape) == c["shape"] and got["input_ids"].reshape(-1).tolist() == c["ids"] and got["lengths"].tolist() == c["lengths"], (name, k, "golden")
    # without special tokens
    _apply(tok, *SETTINGS[0])
    got = tok.encode_batch_dense(docs, add_special_tokens=False, want_mask=False)
    sp = spec_of(js, *SETTINGS[0]); sp["pre"], sp["post"] = [], []
    exp = orc.dense_rows(ids, rp, **sp)
    assert np.array_equal(got["input_ids"], exp[0]) and got["attention_mask"] is None and np.array_equal(got["lengths"], exp[2])


@pytest.mark.gpu
def test_gpu_dense_multi_chunk_device_entry_and_errors(monkeypatch):
    from tokenizers_b200 import Tokenizer, _lib
    import torch
    js = tokenizer_json("gpt2_style")
    o = orc.Oracle(js)
    data, off = corpus.generate(2, 31, 0, 3000)
    ids, _, _, rp = o.encode_batch_csr(data, off)[0], None, None, o.encode_batch_csr(data, off)[3]
    tr, pd = dict(max_length=64, direction="right"), dict(length=64, direction="right", pad_id=9)
    exp = orc.dense_rows(ids, rp, **spec_of(js, tr, pd))
    monkeypatch.setenv("B2T_CHUNK_BYTES", "65536")   # many chunks through the host pipeline
    tok = Tokenizer.from_str(js)
    _apply(tok, tr, pd)
    got = tok.encode_batch_dense(data, off)
    assert np.array_equal(got["input_ids"], exp[0]) and np.array_equal(got["attention_mask"], exp[1])
    # BatchLongest runs as one device pass whatever the chunk size
    tr2, pd2 = dict(max_length=100, direction="left"), dict(length=None, direction="right", pad_id=9)
    _apply(tok, tr2, pd2)
    got = tok.encode_batch_dense(data, off)
    exp2 = orc.dense_rows(ids, rp, **spec_of(js, tr2, pd2))
    assert np.array_equal(got["input_ids"], exp2[0]) and np.array_equal(got["attention_mask"], exp2[1])
    # device entry point
    L = _lib.lib()
    for trd, pdd, e in ((tr, pd, exp), (tr2, pd2, exp2)):
        _apply(tok, trd, pdd)
        sp, keep = tok.dense_spec()
        d_bytes = torch.from_numpy(np.concatenate([data, np.zeros(64, np.uint8)])).cuda()
        d_off = torch.from_numpy(off.astype(np.int64)).cuda()
        res = ctypes.c_void_p()
        _lib.check(L.b2t_encode_batch_dense_device(tok.handle, d_bytes.data_ptr(), len(data), d_off.data_ptr(), len(off) - 1, ctypes.byref(sp), None, ctypes.byref(res)))
        torch.cuda.synchronize()
        W, n = L.b2t_result_dense_length(res), len(off) - 1
        assert L.b2t_result_on_device(res) == 1 and W == e[0].shape[1]
        out = torch.empty(n * W, dtype=torch.int32, device="cuda")
        ctypes.CDLL("libcudart.so").cudaMemcpy(ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(L.b2t_result_dense_ids(res)), ctypes.c_size_t(n * W * 4), 3)
        L.b2t_result_free(res)
        assert np.array_equal(out.cpu().numpy().view(np.uint32).reshape(n, W), e[0])
    # a row that does not fit a fixed length is an error, not a silently cut row
    _apply(tok, None, dict(length=8, direction="right", pad_id=0))
    with pytest.raises(_lib.B2TError):
        tok.encode_batch_dense(data, off)
    # empty batch
    _apply(tok, tr, pd)
    got = tok.encode_batch_dense([])
    assert got["input_ids"].shape == (0, 64)
