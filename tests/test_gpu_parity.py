"""GPU (-m gpu): the CUDA path through the C ABI against the committed golden vectors, the oracle, and -- where it is
importable -- the reference implementation itself.  Bit-exact: ids, (char_start, char_end) offsets, word ids, row_ptr."""
import ctypes, json, os
import numpy as np
import pytest
import helpers, fuzzgen, corpus

pytestmark = pytest.mark.gpu

from tokenizers_b200 import Tokenizer, UnsupportedConfig, _lib  # noqa: E402
from oracle import oracle as orc  # noqa: E402

ASSET_NAMES = ["gpt2_style", "llama3_style", "wordpiece"]
_engines = {}


def engine(name_or_json):
    if name_or_json not in _engines:
        js = helpers.asset_json(name_or_json) if name_or_json in ASSET_NAMES else name_or_json
        _engines[name_or_json] = (Tokenizer.from_str(js), orc.Oracle(js), js)
    return _engines[name_or_json]


def gpu_csr(tok, docs, **kw):
    data, off = helpers.pack_docs(docs)
    be = tok.encode_batch_csr(data, off, **kw)
    return be.ids, be.offsets, be.word_ids, be.row_ptr


@pytest.mark.parametrize("name", helpers.GOLDEN_NAMES)
def test_gpu_matches_reference_golden(name):
    tj, cases = helpers.load_golden(name)
    tok = Tokenizer.from_str(tj)
    docs = [c["input"] for c in cases]
    helpers.assert_csr_equal(gpu_csr(tok, docs), helpers.cases_to_csr(cases), docs, f"gpu vs golden_{name}")


def test_add_prefix_space_variants():
    """ByteLevel(add_prefix_space=True): the device re-packs the batch with the space inserted and maps offsets back."""
    for patch in ({"add_prefix_space": True}, {"add_prefix_space": True, "use_regex": False}):
        j = json.loads(helpers.asset_json("gpt2_style"))
        j["pre_tokenizer"].update(patch)
        js = json.dumps(j)
        tok, o = Tokenizer.from_str(js), orc.Oracle(js)
        docs = fuzzgen.rand_docs(321, 1200, max_len=50) + ["", " x", "x", "é", "\n", "  ", "中文 text"]
        helpers.assert_csr_equal(gpu_csr(tok, docs), o.encode_batch(docs), docs, f"prefix {patch}")
        helpers.assert_csr_equal(gpu_csr(tok, docs, byte_offsets=True), o.encode_batch(docs, offset_type=orc.OFF_BYTE), docs, f"prefix bytes {patch}")
        got = tok.pre_tokenize_batch(docs[:400])
        for d, g in zip(docs[:400], got):
            assert g == o.pre_tokenize(d), repr(d)
    # the Llama-3 pipeline applies ByteLevel per split; a prefix space there is refused, not approximated
    j = json.loads(helpers.asset_json("llama3_style")); j["pre_tokenizer"]["pretokenizers"][1]["add_prefix_space"] = True
    with pytest.raises(UnsupportedConfig):
        Tokenizer.from_str(json.dumps(j))


@pytest.mark.parametrize("name", ASSET_NAMES)
def test_gpu_matches_oracle_fuzz(name):
    tok, o, _ = engine(name)
    for seed in range(6):
        docs = fuzzgen.rand_docs(5000 + seed, 1500, max_len=60 if seed % 2 else 300)
        helpers.assert_csr_equal(gpu_csr(tok, docs), o.encode_batch(docs), docs, f"{name} fuzz seed {seed}")


@pytest.mark.parametrize("name", ASSET_NAMES)
@pytest.mark.parametrize("kind", [1, 2, 4, 5])
def test_gpu_matches_oracle_corpus(name, kind):
    tok, o, _ = engine(name)
    data, off = corpus.generate(kind, 10 + kind, 0, 4000 if kind != 5 else 6000)
    be = tok.encode_batch_csr(data, off)
    exp = o.encode_batch_csr(data, off)
    helpers.assert_csr_equal((be.ids, be.offsets, be.word_ids, be.row_ptr), exp, corpus.to_strings(data, off), f"{name} corpus {kind}")


@pytest.mark.parametrize("name", ASSET_NAMES)
def test_pre_tokenize_matches_oracle(name):
    tok, o, _ = engine(name)
    docs = fuzzgen.rand_docs(77, 800, max_len=80)
    got = tok.pre_tokenize_batch(docs)
    for d, g in zip(docs, got):
        assert g == o.pre_tokenize(d), repr(d)


@pytest.mark.parametrize("name", ASSET_NAMES)
def test_flags_ids_only_and_byte_offsets(name):
    tok, o, _ = engine(name)
    docs = fuzzgen.rand_docs(91, 700, max_len=80)
    exp_c = o.encode_batch(docs)
    exp_b = o.encode_batch(docs, offset_type=orc.OFF_BYTE)
    ids, offs, wid, rp = gpu_csr(tok, docs, offsets=False, word_ids=False)
    assert offs is None and wid is None
    assert np.array_equal(ids, exp_c[0]) and np.array_equal(rp, exp_c[3])
    helpers.assert_csr_equal(gpu_csr(tok, docs, byte_offsets=True), exp_b, docs, f"{name} byte offsets")


@pytest.mark.parametrize("name", ASSET_NAMES)
def test_multi_chunk_host_pipeline(name):
    """Tiny chunks force many in-flight chunks through the 3-slot pipeline; the result must not change."""
    _, o, js = engine(name)
    os.environ["B2T_CHUNK_BYTES"] = "3000"
    try:
        tok = Tokenizer.from_str(js)
    finally:
        del os.environ["B2T_CHUNK_BYTES"]
    data, off = corpus.generate(2, 5, 0, 700)
    docs = corpus.to_strings(data, off) + ["", "", "x"]
    helpers.assert_csr_equal(gpu_csr(tok, docs), o.encode_batch(docs), docs, f"{name} multi-chunk")


def test_long_pretokens_monotone_and_not():
    """Pre-tokens longer than 256 bytes take the long path (pre-pass); hand-written NON-monotone merges force its
    one-merge-per-round mode, trained vocabularies the all-occurrences mode."""
    import random
    tj, _ = helpers.load_golden("nonmonotone")
    tok, o = Tokenizer.from_str(tj), orc.Oracle(tj)
    rng = random.Random(5)
    docs = ["ab" * 400, "a" * 1000, "aab" * 300 + " " + "ba" * 200, "x" + "ab" * 129, "ab" * 128, "ab" * 128 + "a",
            "".join(rng.choice("ab") for _ in range(5000)), "".join(rng.choice("ab ") for _ in range(3000)), "b" * 257 + " " + "a" * 2500]
    helpers.assert_csr_equal(gpu_csr(tok, docs), o.encode_batch(docs), docs, "nonmonotone long")
    helpers.assert_csr_equal(gpu_csr(tok, docs, byte_offsets=True), o.encode_batch(docs, offset_type=orc.OFF_BYTE), docs, "nonmonotone long bytes")
    for name in ("gpt2_style", "llama3_style"):
        tok, o, _ = engine(name)
        docs = ["a" * 70000, " " * 66000 + "x", "é" * 5000, "".join(rng.choice("abcdefghijklmnopqrstuvwxyz") for _ in range(40000)),
                "the" * 1000 + " and " + "1" * 3000, "\n" * 3000 + "x" * 300, "z" * 257, "z" * 256, "hello " + "q" * 2047 + " world",
                "".join(rng.choice("etaoinshr") for _ in range(300)) + " end", "中" * 2000, "😀" * 700]
        helpers.assert_csr_equal(gpu_csr(tok, docs), o.encode_batch(docs), docs, f"{name} long")


def test_edge_batches():
    tok, o, _ = engine("gpt2_style")
    for docs in ([], [""], ["", "", ""], ["a"], ["", "a", ""], ["é" * 700], [" " * 2047, "b"], ["a" * 2048, "b" * 2049, "c"],
                 ["x" * 31 + "é", "\n" * 40], ["ab " * 1000]):
        helpers.assert_csr_equal(gpu_csr(tok, docs), o.encode_batch(docs), docs, f"edge {[len(d) for d in docs]}")


def test_device_resident_entry_point():
    import torch
    tok, o, _ = engine("gpt2_style")
    data, off = corpus.generate(2, 21, 0, 3000)
    d_bytes = torch.from_numpy(data.copy()).cuda()
    d_off = torch.from_numpy(off.astype(np.int64)).cuda()
    L = _lib.lib()
    res = ctypes.c_void_p()
    flags = _lib.WANT_OFFSETS | _lib.WANT_WORD_IDS
    _lib.check(L.b2t_encode_batch_device(tok.handle, d_bytes.data_ptr(), int(off[-1]), d_off.data_ptr(), len(off) - 1, flags, None, ctypes.byref(res)))
    assert L.b2t_result_on_device(res) == 1
    T = L.b2t_result_n_tokens(res)

    def dev(ptr, count, dtype):
        out = torch.empty(count, dtype=dtype, device="cuda")
        torch.cuda.synchronize()
        ctypes.CDLL("libcudart.so").cudaMemcpy(ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(ptr), ctypes.c_size_t(count * out.element_size()), 3)
        return out.cpu().numpy()
    ids = dev(L.b2t_result_ids(res), T, torch.int32).view(np.uint32)
    offs = dev(L.b2t_result_offsets(res), 2 * T, torch.int32).view(np.uint32).reshape(-1, 2)
    wid = dev(L.b2t_result_word_ids(res), T, torch.int32).view(np.uint32)
    rp = dev(L.b2t_result_row_ptr(res), len(off), torch.int64).view(np.uint64)
    L.b2t_result_free(res)
    helpers.assert_csr_equal((ids, offs, wid, rp), o.encode_batch_csr(data, off), None, "device entry point")


@pytest.mark.parametrize("name", ASSET_NAMES)
def test_gpu_matches_reference_wheel_large(name):
    data, off = corpus.generate(4 if name == "wordpiece" else 2, 99, 0, 40000)
    docs = corpus.to_strings(data, off)
    # the reference's output first, so that recording it needs no GPU
    helpers.assert_reference(f"gpu_parity/wheel_large/{name}/docs", docs, lambda: docs)
    exp = helpers.reference(f"gpu_parity/wheel_large/{name}",
                            lambda: helpers.csr_plain(helpers.wheel_csr(helpers.wheel_tokenizer(helpers.asset_json(name)), docs)))
    tok, _, _ = engine(name)
    be = tok.encode_batch_csr(data, off)
    assert helpers.digest(helpers.csr_plain((be.ids, be.offsets, be.word_ids, be.row_ptr))) == exp, f"{name}: differs from the reference's recorded output"


def test_full_size_properties():
    """256 MB of the config-2 corpus: size-independent properties + oracle parity on a sampled slice."""
    tok, o, _ = engine("gpt2_style")
    data, off = corpus.generate(2, 2, 0, 1 << 19, max_bytes=256 << 20)
    be = tok.encode_batch_csr(data, off)
    rp = be.row_ptr
    assert rp[0] == 0 and np.all(np.diff(rp.astype(np.int64)) >= 0) and int(rp[-1]) == len(be.ids)
    assert be.ids.max() < tok.get_vocab_size()
    # offsets: within a doc, starts are non-decreasing, end >= start, and the last token ends at the doc's char count
    st, en = be.offsets[:, 0].astype(np.int64), be.offsets[:, 1].astype(np.int64)
    assert np.all(en >= st)
    lead = (data & 0xC0) != 0x80
    cum = np.concatenate([[0], np.cumsum(lead)])
    nchar = cum[off[1:].astype(np.int64)] - cum[off[:-1].astype(np.int64)]
    last = rp[1:].astype(np.int64) - 1
    nonempty = rp[1:] > rp[:-1]
    assert np.array_equal(en[last[nonempty]], nchar[nonempty])
    # sampled oracle parity: 3 slices of 2000 docs
    n = len(off) - 1
    for a in (0, n // 2, n - 2000):
        sl_off = (off[a:a + 2001] - off[a]).astype(np.uint64)
        sl = data[int(off[a]):int(off[a + 2000])]
        exp = o.encode_batch_csr(sl, sl_off)
        t0, t1 = int(rp[a]), int(rp[a + 2000])
        got = (be.ids[t0:t1], be.offsets[t0:t1], be.word_ids[t0:t1], rp[a:a + 2001] - rp[a])
        helpers.assert_csr_equal(got, exp, None, f"slice at doc {a}")


def test_concurrent_callers_share_one_engine():
    """encode_batch is callable from many host threads (the reference: &self + Send/Sync, mod.rs:1328-1335)."""
    import threading
    tok, o, _ = engine("gpt2_style")
    batches = [fuzzgen.rand_docs(900 + i, 600, max_len=80) for i in range(6)]
    exp = [o.encode_batch(b) for b in batches]
    out, errs = [None] * 6, []

    def work(i):
        try:
            for _ in range(3):
                out[i] = gpu_csr(tok, batches[i])
        except Exception as ex:  # pragma: no cover
            errs.append(ex)
    ts = [threading.Thread(target=work, args=(i,)) for i in range(6)]
    [t.start() for t in ts]; [t.join() for t in ts]
    assert not errs, errs
    for i in range(6):
        helpers.assert_csr_equal(out[i], exp[i], batches[i], f"thread {i}")


def test_document_larger_than_a_chunk_and_many_empty_docs():
    _, o, js = engine("gpt2_style")
    os.environ["B2T_CHUNK_BYTES"] = str(1 << 20)
    try:
        tok = Tokenizer.from_str(js)
    finally:
        del os.environ["B2T_CHUNK_BYTES"]
    data, off = corpus.generate(2, 77, 0, 9000)
    big = data.tobytes()[: 3 << 20].decode("utf-8", "ignore")
    docs = [""] * 3000 + [big] + ["tail doc"] + [""] * 5000 + ["x"]
    helpers.assert_csr_equal(gpu_csr(tok, docs), o.encode_batch(docs), None, "big doc + empties")


def test_invalid_utf8_does_not_fault():
    """The ABI takes bytes; Rust's &str can never be invalid UTF-8, so the result is unspecified -- but it must not crash,
    hang, or write out of bounds (row_ptr stays a valid CSR over ids)."""
    tok, _, _ = engine("gpt2_style")
    rng = np.random.default_rng(7)
    data = rng.integers(0, 256, size=200000, dtype=np.uint8)
    off = np.arange(0, 200001, 1000, dtype=np.uint64)
    be = tok.encode_batch_csr(data, off)
    assert be.row_ptr[0] == 0 and int(be.row_ptr[-1]) == len(be.ids) and np.all(np.diff(be.row_ptr.astype(np.int64)) >= 0)
    assert be.ids.max() < tok.get_vocab_size()


def test_multi_gpu_sharded_equals_single():
    """N ranks (one process per GPU, NCCL) encode byte-balanced shards of one batch and gather the CSR in place: the result
    must equal what one GPU produces for the whole batch (tests/mgpu_check.py).  Needs >= 2 visible GPUs."""
    import subprocess, sys, torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("one GPU visible")
    n = min(n, 4)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--local-addr", "127.0.0.1", "--nproc-per-node", str(n),
                        os.path.join(helpers.ROOT, "tests", "mgpu_check.py")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
