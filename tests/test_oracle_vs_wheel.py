"""CPU: differential fuzz of the oracle against the reference implementation itself (the `tokenizers` wheel, its outputs
recorded as digests: tests/helpers.py).  Keeps the oracle honest beyond the committed golden vectors."""
import json
import pytest
import helpers, fuzzgen, corpus
from oracle import oracle as orc


def _variants():
    out = []
    for name in ("gpt2_style", "llama3_style", "wordpiece"):
        js = helpers.asset_json(name)
        out.append((name, js))
        if name == "gpt2_style":
            j = json.loads(js); j["pre_tokenizer"]["add_prefix_space"] = True; out.append((name + "+prefix", json.dumps(j)))
            j = json.loads(js); j["pre_tokenizer"]["use_regex"] = False; out.append((name + "+noregex", json.dumps(j)))
    return out


@pytest.mark.parametrize("name,js", _variants(), ids=[v[0] for v in _variants()])
def test_oracle_vs_wheel_fuzz(name, js):
    tok = helpers.wheel_tokenizer(js)
    o = orc.Oracle(js)
    for seed in range(4):
        docs = fuzzgen.rand_docs(1000 + seed, 800, max_len=60 if seed % 2 else 300)
        helpers.assert_reference(f"oracle_vs_wheel/{name}/seed{seed}/docs", docs, lambda: docs)
        helpers.assert_reference(f"oracle_vs_wheel/{name}/seed{seed}", helpers.csr_plain(o.encode_batch(docs)),
                                 lambda: helpers.csr_plain(helpers.wheel_csr(tok, docs)), f"{name} seed {seed}")
    for kind in (1, 2, 4, 5):
        data, off = corpus.generate(kind, 70 + kind, 0, 150)
        docs = corpus.to_strings(data, off)
        helpers.assert_reference(f"oracle_vs_wheel/{name}/corpus{kind}/docs", docs, lambda: docs)
        helpers.assert_reference(f"oracle_vs_wheel/{name}/corpus{kind}", helpers.csr_plain(o.encode_batch(docs)),
                                 lambda: helpers.csr_plain(helpers.wheel_csr(tok, docs)), f"{name} corpus {kind}")
