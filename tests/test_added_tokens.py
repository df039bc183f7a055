"""Host steps either side of the hot path: added-token extraction (added_vocabulary.rs:430-564) and the single-sequence
special-token template (processors/template.rs).  CPU: tokenizers_b200's host logic in front of the oracle, against the
reference wheel's recorded outputs and against committed golden vectors.  GPU: the same through the real engine."""
import gzip, json, os, types
import numpy as np
import pytest
from helpers import GOLDEN, asset_json, with_added_tokens, added_token_docs, oracle_backed_tokenizer, assert_reference, wheel, wheel_tokenizer

CONFIGS = [("gpt2_style", False), ("gpt2_style", True), ("llama3_style", False), ("wordpiece", True)]


def _patched(asset, prefix_space=None):
    js = json.loads(asset_json(asset))
    if prefix_space is not None and js["pre_tokenizer"]["type"] == "ByteLevel":
        js["pre_tokenizer"]["add_prefix_space"] = prefix_space
    return json.dumps(js)


def _flat(encs, tokens=True):
    return [{"ids": list(e.ids), "offsets": [list(o) for o in e.offsets], "word_ids": list(e.word_ids),
             "type_ids": list(e.type_ids), "special": list(e.special_tokens_mask), "tokens": list(e.tokens) if tokens else None} for e in encs]


def _compare(got, exp, docs, what):
    assert len(got) == len(exp)
    for d, (g, e) in enumerate(zip(got, exp)):
        assert g == e, f"{what}: doc {d} {docs[d]!r}\n exp {e}\n got {g}"


@pytest.mark.parametrize("asset,template", CONFIGS)
@pytest.mark.parametrize("prefix_space", [False, True])
def test_host_logic_vs_wheel(asset, template, prefix_space):
    if prefix_space and asset != "gpt2_style":
        pytest.skip("add_prefix_space only varies for the ByteLevel pre-tokenizer")
    tj = with_added_tokens(_patched(asset, prefix_space), template)
    ref = wheel_tokenizer(tj)
    mine = oracle_backed_tokenizer(tj)
    docs = added_token_docs(7, 1500)
    assert_reference("added/docs/7_1500", docs, lambda: docs)
    key = f"added/host_logic/{asset}/template={template}/prefix_space={prefix_space}"
    for special in (False, True):
        assert_reference(f"{key}/special={special}", _flat(mine.encode_batch(docs, add_special_tokens=special)),
                         lambda: _flat(ref.encode_batch(docs, add_special_tokens=special)), f"{asset} template={template} add_special_tokens={special}")
    assert_reference(f"{key}/mask_id", mine.token_to_id("<mask>"), lambda: ref.token_to_id("<mask>"))
    assert mine.id_to_token(mine.token_to_id("<a><b>")) == "<a><b>"
    assert_reference(f"{key}/vocab_size", [mine.get_vocab_size(), mine.get_vocab_size(False)], lambda: [ref.get_vocab_size(), ref.get_vocab_size(False)])


def test_byte_offsets_and_fast_vs_wheel():
    tj = with_added_tokens(asset_json("gpt2_style"), True)
    mine = oracle_backed_tokenizer(tj)
    docs = added_token_docs(11, 400)
    assert_reference("added/docs/11_400", docs, lambda: docs)
    full = mine.encode_batch(docs, add_special_tokens=True)
    fast = mine.encode_batch_fast(docs, add_special_tokens=True)
    assert [e.ids for e in full] == [e.ids for e in fast]
    # (token texts are not compared: without offsets the reference reports '' for added tokens found in the text)
    assert_reference("added/encode_batch_fast", _flat(fast, False), lambda: _flat(wheel_tokenizer(tj).encode_batch_fast(docs, add_special_tokens=True), False),
                     "encode_batch_fast")
    # byte offsets of the CSR entry point == char offsets mapped through the document's UTF-8 encoding
    data = np.frombuffer("".join(docs).encode("utf-8"), dtype=np.uint8)
    off = np.zeros(len(docs) + 1, dtype=np.uint64)
    np.cumsum([len(d.encode("utf-8")) for d in docs], out=off[1:])
    be_c = mine.encode_batch_csr(data, off)
    be_b = mine.encode_batch_csr(data, off, byte_offsets=True)
    assert np.array_equal(be_c.ids, be_b.ids) and np.array_equal(be_c.row_ptr, be_b.row_ptr)
    for d, doc in enumerate(docs):
        a, b = int(be_c.row_ptr[d]), int(be_c.row_ptr[d + 1])
        for (c0, c1), (b0, b1) in zip(be_c.offsets[a:b].tolist(), be_b.offsets[a:b].tolist()):
            assert len(doc[:c0].encode("utf-8")) == b0 and len(doc[:c1].encode("utf-8")) == b1, (doc, c0, c1, b0, b1)


def _post_processors(js):
    by = {e["content"]: e["id"] for e in js["added_tokens"]}
    cls, sep = ["<|endoftext|>", by["<|endoftext|>"]], ["<mask>", by["<mask>"]]
    tmpl = {"type": "TemplateProcessing", "single": [{"SpecialToken": {"id": "<a>", "type_id": 0}}, {"Sequence": {"id": "A", "type_id": 0}}],
            "pair": [{"Sequence": {"id": "A", "type_id": 0}}, {"Sequence": {"id": "B", "type_id": 1}}],
            "special_tokens": {"<a>": {"id": "<a>", "ids": [by["<a>"]], "tokens": ["<a>"]}}}
    return [{"type": "ByteLevel", "add_prefix_space": True, "trim_offsets": True, "use_regex": True},
            {"type": "ByteLevel", "add_prefix_space": False, "trim_offsets": True, "use_regex": True},
            {"type": "RobertaProcessing", "sep": sep, "cls": cls, "trim_offsets": True, "add_prefix_space": True},
            {"type": "RobertaProcessing", "sep": sep, "cls": cls, "trim_offsets": False, "add_prefix_space": False},
            {"type": "BertProcessing", "sep": sep, "cls": cls},
            {"type": "Sequence", "processors": [{"type": "ByteLevel", "add_prefix_space": True, "trim_offsets": True, "use_regex": True}, tmpl]}]


@pytest.mark.parametrize("asset,prefix_space", [("gpt2_style", False), ("gpt2_style", True), ("llama3_style", None)])
def test_post_processors_vs_wheel(asset, prefix_space):
    """offset trimming (byte_level.rs:202-234) and the Bert / Roberta / Template / Sequence processors for single sequences"""
    base = json.loads(with_added_tokens(_patched(asset, prefix_space)))
    docs = added_token_docs(13, 300) + ["  two  spaces  ", " x", "x ", "   ", " <mask> y", "a  <both>  b"]
    assert_reference("added/docs/13_300", docs, lambda: docs)
    for i, pp in enumerate(_post_processors(base)):
        js = dict(base, post_processor=pp)
        tj = json.dumps(js)
        ref, mine = wheel_tokenizer(tj), oracle_backed_tokenizer(tj)
        for special in (False, True):
            assert_reference(f"added/post_processors/{asset}/prefix_space={prefix_space}/{i}/special={special}",
                             _flat(mine.encode_batch(docs, add_special_tokens=special)), lambda: _flat(ref.encode_batch(docs, add_special_tokens=special)),
                             f"{asset} {pp['type']} trim={pp.get('trim_offsets')} aps={pp.get('add_prefix_space')} special={special}")


def test_candidate_start_inside_a_run_across_documents():
    """the batch-wide prefilter must report EVERY candidate start: with the added token "  " and a document that ends
    in a space, the next document's leading "  " is the second candidate of the run "   " (regression)"""
    from helpers import added_token_entries
    js = json.loads(asset_json("gpt2_style"))
    js["added_tokens"] = added_token_entries(js["model"]["vocab"], [("  ", False, False, False, False, True)])
    tid = js["added_tokens"][0]["id"]
    mine = oracle_backed_tokenizer(json.dumps(js))
    encs = mine.encode_batch(["a ", "  x>", "b", "   "], add_special_tokens=False)
    assert encs[1].ids[0] == tid and encs[1].offsets[0] == (0, 2)
    assert encs[3].ids[0] == tid and encs[3].offsets[:2] == [(0, 2), (2, 3)]
    assert_reference("added/boundary_run", _flat(encs),
                     lambda: _flat(wheel_tokenizer(json.dumps(js)).encode_batch(["a ", "  x>", "b", "   "], add_special_tokens=False)), "boundary run")


def _flat_full(encs):
    def one(e):
        return {"ids": list(e.ids), "offsets": [list(o) for o in e.offsets], "word_ids": list(e.word_ids), "type_ids": list(e.type_ids),
                "special": list(e.special_tokens_mask), "attention": list(e.attention_mask), "tokens": list(e.tokens),
                "overflowing": [one(o) for o in e.overflowing]}
    return [one(e) for e in encs]


@pytest.mark.parametrize("asset,template", [("gpt2_style", True), ("wordpiece", False)])
def test_truncation_and_padding_vs_wheel(asset, template):
    """TokenizerImpl::post_process steps 1 and 3 (utils/truncation.rs, Encoding::truncate, utils/padding.rs) for single sequences"""
    tj = with_added_tokens(asset_json(asset), template)
    ref, mine = wheel_tokenizer(tj), oracle_backed_tokenizer(tj)
    docs = added_token_docs(17, 150) + ["", "a", "a b c d e f g h i j k l m n o p q r s t u v w x y z " * 3]
    assert_reference("added/docs/17_150", docs, lambda: docs)
    key = f"added/truncation/{asset}/template={template}"
    cases = [dict(max_length=8, stride=0, direction="right"), dict(max_length=8, stride=3, direction="right"),
             dict(max_length=7, stride=2, direction="left"), dict(max_length=3, stride=0, direction="left"),
             dict(max_length=16, stride=5, direction="right", strategy="only_first")]
    pads = [None, dict(direction="left", pad_id=3, pad_type_id=1, pad_token="<pad>"), dict(length=12), dict(pad_to_multiple_of=8)]
    for ci, tc in enumerate(cases):
        for pi, pc in enumerate(pads):
            for t in filter(None, (ref, mine)):
                t.enable_truncation(**tc)
                t.no_padding() if pc is None else t.enable_padding(**pc)
            for special in (False, True):
                assert_reference(f"{key}/{ci}/{pi}/special={special}", _flat_full(mine.encode_batch(docs, add_special_tokens=special)),
                                 lambda: _flat_full(ref.encode_batch(docs, add_special_tokens=special)), f"{asset} trunc={tc} pad={pc} special={special}")
    # padding without truncation, settings read from tokenizer.json
    js = json.loads(tj)
    js["truncation"] = {"direction": "Right", "max_length": 10, "strategy": "LongestFirst", "stride": 2}
    js["padding"] = {"strategy": {"Fixed": 14}, "direction": "Right", "pad_to_multiple_of": None, "pad_id": 1, "pad_type_id": 0, "pad_token": "[PAD]"}
    ref, mine = wheel_tokenizer(json.dumps(js)), oracle_backed_tokenizer(json.dumps(js))
    assert_reference(f"{key}/json_settings", mine.truncation, lambda: ref.truncation)
    assert mine.padding["length"] == 14
    assert_reference(f"{key}/json_settings/encodings", _flat_full(mine.encode_batch(docs)), lambda: _flat_full(ref.encode_batch(docs)), "settings from tokenizer.json")
    def toks(encs):  # the text of an lstrip / rstrip token is its matched span (Token::new(id, value, ..), added_vocabulary.rs:508)
        return [(e.tokens, [o.tokens for o in e.overflowing]) for e in encs]
    assert_reference(f"{key}/json_settings/tokens", toks(mine.encode_batch(docs)), lambda: toks(ref.encode_batch(docs)))
    for t in filter(None, (ref, mine)):
        t.no_truncation()
    assert_reference(f"{key}/padding_only", _flat_full(mine.encode_batch(docs)), lambda: _flat_full(ref.encode_batch(docs)), "padding only")


def test_unsupported_post_processors():
    from tokenizers_b200.tokenizer import parse_tokenizer_json, UnsupportedConfig
    js = json.loads(asset_json("wordpiece"))
    js["post_processor"] = {"type": "ByteLevel", "add_prefix_space": True, "trim_offsets": True, "use_regex": True}
    with pytest.raises(UnsupportedConfig):
        parse_tokenizer_json(js)  # offset trimming is defined on the byte-level alphabet
    js = json.loads(asset_json("gpt2_style"))
    js["post_processor"] = {"type": "RobertaProcessing", "sep": ["</s>", 2], "cls": ["<s>", 0], "trim_offsets": False, "add_prefix_space": False}
    t = parse_tokenizer_json(js)["template"]
    assert (t["pre"], t["post"], t["type_id"], t["trim"]) == ([(0, 0)], [(2, 0)], 0, None)
    assert t["pair"] == [("special", 0, 0), ("seq", 0, 0), ("special", 2, 0), ("special", 2, 0), ("seq", 1, 0), ("special", 2, 0)]
    js["post_processor"] = {"type": "Sequence", "processors": [{"type": "ByteLevel", "trim_offsets": False},
                                                               {"type": "BertProcessing", "sep": ["[SEP]", 102], "cls": ["[CLS]", 101]}]}
    assert parse_tokenizer_json(js)["template"]["pre"] == [(101, 0)]


def _golden_cases():
    g = json.loads(gzip.open(os.path.join(GOLDEN, "golden_added_tokens.json.gz")).read().decode("utf-8"))
    return g


@pytest.mark.parametrize("idx", range(4))
def test_host_logic_vs_golden(idx):
    g = _golden_cases()["configs"][idx]
    tj = with_added_tokens(_patched(g["asset"], g["prefix_space"]), g["template"])
    mine = oracle_backed_tokenizer(tj)
    docs = g["docs"]
    for special in (False, True):
        _compare(_flat(mine.encode_batch(docs, add_special_tokens=special)), g["expected"][str(special)], docs, f"golden {g['asset']}")


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(4))
def test_gpu_added_tokens_vs_golden(idx):
    from tokenizers_b200 import Tokenizer
    g = _golden_cases()["configs"][idx]
    tok = Tokenizer.from_str(with_added_tokens(_patched(g["asset"], g["prefix_space"]), g["template"]))
    assert tok._dev_added == (not g["prefix_space"])   # add_prefix_space: the prefix goes in front of every piece, the host splits
    docs = g["docs"]
    for special in (False, True):
        _compare(_flat(tok.encode_batch(docs, add_special_tokens=special)), g["expected"][str(special)], docs, f"gpu golden {g['asset']}")
    ids_fast = [e.ids for e in tok.encode_batch_fast(docs, add_special_tokens=True)]
    assert ids_fast == [c["ids"] for c in g["expected"]["True"]]


@pytest.mark.gpu
@pytest.mark.parametrize("asset,template", CONFIGS)
def test_gpu_device_extraction_matches_host_logic(asset, template):
    """Added-token extraction ON THE DEVICE (b2t_engine_set_added_tokens: candidates, per-document resolution, spans as hard
    boundaries of the scan) against the host logic in front of the oracle (itself pinned to the wheel above)."""
    from tokenizers_b200 import Tokenizer
    from helpers import pack_docs
    tj = with_added_tokens(_patched(asset, False), template)
    tok, ref = Tokenizer.from_str(tj), oracle_backed_tokenizer(tj)
    assert tok._dev_added and not ref._dev_added
    docs = added_token_docs(99, 1500) + ["x" + " " * 40 + "<mask>" + " " * 50 + "[SEP2]" + "\t" * 30 + "y", "<a>" * 7 + "<a><b>" * 3, "tok" * 5]
    for special in (False, True):
        _compare(_flat(tok.encode_batch(docs, add_special_tokens=special)), _flat(ref.encode_batch(docs, add_special_tokens=special)), docs, f"device {asset}")
    assert [e.ids for e in tok.encode_batch_fast(docs)] == [e.ids for e in ref.encode_batch_fast(docs)]
    data, off = pack_docs(docs)
    for kw in (dict(byte_offsets=True), dict(offsets=False, word_ids=False), dict(add_special_tokens=True)):
        a, b = tok.encode_batch_csr(data, off, **kw), ref.encode_batch_csr(data, off, **kw)
        for x, y in ((a.ids, b.ids), (a.offsets, b.offsets), (a.word_ids, b.word_ids), (a.row_ptr, b.row_ptr)):
            assert (x is None and y is None) or np.array_equal(x, y), (asset, kw)
    # beyond the device limits (a span over 256 bytes after lstrip) the shim splits on the host: same result
    hard = ["a" + " " * 300 + "<mask> b", "<a>" * 40 + " z", "q " + "<|endoftext|>" * 12]
    _compare(_flat(tok.encode_batch(hard)), _flat(ref.encode_batch(hard)), hard, f"fallback {asset}")
    # many documents, many chunks
    os.environ["B2T_CHUNK_BYTES"] = "32768"
    try:
        tok2 = Tokenizer.from_str(tj)
        many = added_token_docs(7, 6000)
        _compare(_flat(tok2.encode_batch(many)), _flat(ref.encode_batch(many)), many, f"chunks {asset}")
    finally:
        del os.environ["B2T_CHUNK_BYTES"]


@pytest.mark.gpu
def test_gpu_dense_with_added_tokens():
    """dense mode runs the device extraction too"""
    from tokenizers_b200 import Tokenizer
    tj = with_added_tokens(_patched("gpt2_style", False), True)
    tok, ref = Tokenizer.from_str(tj), oracle_backed_tokenizer(tj)
    docs = added_token_docs(5, 400)
    tok.enable_truncation(24); tok.enable_padding(length=24, pad_id=7)
    ref.enable_truncation(24); ref.enable_padding(length=24, pad_id=7)
    got = tok.encode_batch_dense(docs)
    exp = ref.encode_batch(docs)
    assert np.array_equal(got["input_ids"], np.array([e.ids for e in exp], dtype=np.uint32))
    assert np.array_equal(got["attention_mask"], np.array([e.attention_mask for e in exp], dtype=np.uint8))


@pytest.mark.gpu
def test_gpu_decreasing_doc_off_is_rejected():
    """rows handed to the kernels must be ordered: the C ABI refuses anything else instead of indexing out of bounds"""
    import ctypes
    from tokenizers_b200 import Tokenizer, _lib
    tok = Tokenizer.from_str(asset_json("gpt2_style"))
    data = np.frombuffer(b"hello world, hello", dtype=np.uint8)
    off = np.array([0, 11, 5, 18], dtype=np.uint64)
    res = ctypes.c_void_p()
    rc = _lib.lib().b2t_encode_batch(tok.handle, data.ctypes.data, off.ctypes.data, 3, _lib.WANT_OFFSETS, ctypes.byref(res))
    assert rc == _lib.B2T_ERR_INVALID and b"non-decreasing" in _lib.lib().b2t_last_error()


@pytest.mark.parametrize("asset", ["gpt2_style", "wordpiece"])
def test_pretokenized_input_vs_wheel(asset):
    """is_pretokenized=True (tokenizer/mod.rs:762-805): words are encoded one by one, offsets stay relative to the word,
    word ids are the word's index -- with added tokens, a template, truncation and padding on top"""
    import random
    from fuzzgen import rand_doc
    rng = random.Random(3)
    tj = with_added_tokens(_patched(asset, True if asset == "gpt2_style" else None), True)
    ref, mine = wheel_tokenizer(tj), oracle_backed_tokenizer(tj)
    pool = ["hello", "world", "don't", "<mask>", " x", "", "a<|endoftext|>b", "tok", "Zürich", "  ", "multi word item", "日本語", "1234567", "wörd"]
    seqs = [[]] + [[rng.choice(pool) if rng.random() < 0.6 else rand_doc(rng, 5) for _ in range(rng.randint(0, 9))] for _ in range(300)]
    assert_reference("added/docs/pretokenized", seqs, lambda: seqs)
    key = f"added/pretokenized/{asset}"
    for special in (False, True):
        assert_reference(f"{key}/special={special}", _flat(mine.encode_batch(seqs, is_pretokenized=True, add_special_tokens=special)),
                         lambda: _flat(ref.encode_batch(seqs, is_pretokenized=True, add_special_tokens=special)), f"{asset} pretokenized special={special}")
    for t in filter(None, (ref, mine)):
        t.enable_truncation(max_length=6, stride=2)
        t.enable_padding(pad_to_multiple_of=4)
    assert_reference(f"{key}/truncation_padding", _flat_full(mine.encode_batch(seqs, is_pretokenized=True)),
                     lambda: _flat_full(ref.encode_batch(seqs, is_pretokenized=True)), f"{asset} pretokenized + truncation + padding")
    e = mine.encode(["hello", "world"], is_pretokenized=True)
    assert_reference(f"{key}/hello_world", list(e.ids), lambda: list(ref.encode(["hello", "world"], is_pretokenized=True).ids))
    with pytest.raises(TypeError):
        mine.encode_batch(["not a list of words"], is_pretokenized=True)


def _pair_processors(js):
    by = {e["content"]: e["id"] for e in js["added_tokens"]}
    cls, sep = ["<|endoftext|>", by["<|endoftext|>"]], ["<mask>", by["<mask>"]]
    sp = {"<a>": {"id": "<a>", "ids": [by["<a>"]], "tokens": ["<a>"]}, "<b>": {"id": "<b>", "ids": [by["<a><b>"], by["<a>"]], "tokens": ["<a><b>", "<a>"]}}
    tmpl = {"type": "TemplateProcessing",
            "single": [{"SpecialToken": {"id": "<a>", "type_id": 0}}, {"Sequence": {"id": "A", "type_id": 0}}],
            "pair": [{"SpecialToken": {"id": "<a>", "type_id": 0}}, {"Sequence": {"id": "A", "type_id": 0}}, {"SpecialToken": {"id": "<b>", "type_id": 1}},
                     {"Sequence": {"id": "B", "type_id": 1}}, {"SpecialToken": {"id": "<a>", "type_id": 1}}],
            "special_tokens": sp}
    return [None, {"type": "ByteLevel", "add_prefix_space": True, "trim_offsets": True, "use_regex": True},
            {"type": "BertProcessing", "sep": sep, "cls": cls}, {"type": "RobertaProcessing", "sep": sep, "cls": cls, "trim_offsets": True, "add_prefix_space": False},
            tmpl, {"type": "Sequence", "processors": [{"type": "ByteLevel", "add_prefix_space": False, "trim_offsets": True, "use_regex": True}, tmpl]}]


def test_pairs_vs_wheel():
    """EncodeInput::Dual: both sequences through the engine, then truncation strategies, the pair templates and the merge
    with every combination of overflowing parts (pairs.py), padding -- against the reference, mixed with single inputs"""
    import random
    rng = random.Random(8)
    base = json.loads(with_added_tokens(_patched("gpt2_style", True)))
    texts = added_token_docs(31, 120) + ["", "a", "a b c d e f g h i j k l m n o p", "  x  "]
    inputs = [(rng.choice(texts), rng.choice(texts)) if rng.random() < 0.7 else rng.choice(texts) for _ in range(45)] + [("", ""), ("a", ""), ("", "b")]
    truncs = [None, dict(max_length=12, stride=0), dict(max_length=9, stride=2, direction="left"), dict(max_length=11, stride=3, strategy="only_first"),
              dict(max_length=14, stride=1, strategy="only_second"), dict(max_length=7, stride=1, strategy="longest_first")]
    assert_reference("added/docs/pairs", inputs, lambda: inputs)

    def refused(tok, special, error):
        """indices of the inputs the tokenizer refuses (one by one only when the whole batch is refused)"""
        try:
            tok.encode_batch(inputs, add_special_tokens=special)
            return []
        except error:
            out = []
            for i, x in enumerate(inputs):
                try:
                    tok.encode(*((x,) if isinstance(x, str) else x), add_special_tokens=special)
                except error:
                    out.append(i)
            return out
    for pi, pp in enumerate(_pair_processors(base)):
        tj = json.dumps(dict(base, post_processor=pp))
        ref, mine = wheel_tokenizer(tj), oracle_backed_tokenizer(tj)
        for ti, tc in enumerate(truncs):
            for t in filter(None, (ref, mine)):
                t.no_truncation() if tc is None else t.enable_truncation(**tc)
                t.enable_padding(pad_to_multiple_of=4) if (ti + pi) % 3 == 0 else t.no_padding()
            for special in (False, True):
                # some (input, setting) combinations are errors in the reference (a strategy that cannot shorten the input
                # enough, a stride that no longer fits once the special tokens are subtracted): they must be errors here too
                key, what = f"added/pairs/{pi}/{ti}/special={special}", f"pairs pp={pp and pp['type']} trunc={tc} special={special}"
                bad = refused(mine, special, ValueError)
                assert_reference(f"{key}/refused", bad, lambda: refused(ref, special, BaseException), what)
                batch = [x for i, x in enumerate(inputs) if i not in bad]
                assert_reference(key, _flat_full(mine.encode_batch(batch, add_special_tokens=special)),
                                 lambda: _flat_full(ref.encode_batch(batch, add_special_tokens=special)), what)
        for t in filter(None, (ref, mine)):
            t.no_truncation(); t.no_padding()

        def seqs(e):
            return [e.sequence_ids, e.n_sequences, e.type_ids]
        assert_reference(f"added/pairs/{pi}/sequence_ids", seqs(mine.encode("hello world", "x <mask> y")), lambda: seqs(ref.encode("hello world", "x <mask> y")))


def test_decode_vs_wheel():
    for i, (asset, dec) in enumerate((("gpt2_style", {"type": "ByteLevel", "add_prefix_space": True, "trim_offsets": True, "use_regex": True}),
                                      ("wordpiece", {"type": "WordPiece", "prefix": "##", "cleanup": True}), ("wordpiece", None))):
        js = json.loads(with_added_tokens(asset_json(asset), True))
        js["decoder"] = dec
        tj = json.dumps(js)
        ref, mine = wheel_tokenizer(tj), oracle_backed_tokenizer(tj)
        docs = added_token_docs(5, 300) + ["I do not know , it 's fine . don't you ?"]
        ids = [list(e.ids) for e in mine.encode_batch(docs)]
        assert_reference(f"added/decode/{i}/ids", ids, lambda: [e.ids for e in ref.encode_batch(docs)])
        for skip in (True, False):
            assert_reference(f"added/decode/{i}/skip={skip}", mine.decode_batch(ids, skip_special_tokens=skip), lambda: ref.decode_batch(ids, skip_special_tokens=skip))
        assert_reference(f"added/decode/{i}/unknown", mine.decode([10 ** 9, 5]), lambda: ref.decode([10 ** 9, 5]))  # unknown ids are dropped


def test_add_tokens_vs_wheel():
    """Tokenizer.add_tokens / add_special_tokens after loading: id assignment and extraction follow the reference"""
    tj = asset_json("gpt2_style")
    ref, mine = wheel_tokenizer(tj), oracle_backed_tokenizer(tj)

    def at(t, content, **kw):   # the reference's AddedToken(content, **kw), or what it carries for a token that is not special
        if t is ref:
            return wheel().AddedToken(content, **kw)
        return types.SimpleNamespace(**dict(dict(content=content, single_word=False, lstrip=False, rstrip=False, normalized=True), **kw))
    for t in filter(None, (ref, mine)):
        assert t.add_special_tokens(["<|endoftext|>", "<pad>"]) == 2
        assert t.add_tokens(["hello", "newword", at(t, "tok", single_word=True), at(t, "<x>", lstrip=True, rstrip=True)]) == 4
        assert t.add_tokens(["newword"]) == 0
    assert_reference("added/add_tokens/vocab", [mine.get_vocab_size(), mine.get_vocab()], lambda: [ref.get_vocab_size(), ref.get_vocab()])
    assert mine.num_special_tokens_to_add(False) == 0
    assert_reference("added/add_tokens/num_special_tokens_to_add", mine.num_special_tokens_to_add(False), lambda: ref.num_special_tokens_to_add(False))
    docs = ["hello newword <|endoftext|> x  <x>  y tok atok <pad>", "newwordnewword", ""] + added_token_docs(4, 200)
    assert_reference("added/docs/4_200", docs, lambda: docs)
    assert_reference("added/add_tokens/encodings", _flat(mine.encode_batch(docs)), lambda: _flat(ref.encode_batch(docs)), "after add_tokens")
