#!/usr/bin/env python
"""bench.py -- encode_batch throughput of the B200 engine on BASELINE.json's headline config.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--mb 1024] [--config gpt2|llama3|wordpiece]
                    [--dump-outputs DIR]

One step = one pass of the whole hot path (doc_mark -> pretok_scan -> page_scan -> long_find -> bpe_tile -> compaction)
over one batch of the synthetic corpus of SURVEY.md 8(d) config 2 ("GPT-2 ByteLevel BPE, 1 GB synthetic UTF-8 docs avg
512 B").  Prints ONE JSON line (rank 0):
  value         device-resident: input already in HBM, CUDA events (N > 1: see below)
  e2e           the C-ABI call b2t_encode_batch with pinned HOST buffers, H2D + kernels + D2H inside the timed region
                (ids + char offsets); e2e_ids_only = the encode_batch_fast analogue (4 B per token back instead of 12)
  roofline      the pre-tokenization scan kernel, CUDA events on its launch stream, against MEASURED_PEAKS.json
  configs       the other BASELINE configs (Llama-3 style, Whitespace + WordPiece, length-skew corpus) at 512 MB, fewer steps
  cpu_baseline  the reference's own Rust encode_batch (the `tokenizers` wheel) on this box's host cores, >= 256 MB sample

N > 1 (torchrun, one rank per GPU): every rank encodes its own byte-balanced shard of an N x 1 GB batch (weak scaling)
through tokenizers_b200.parallel.encode_batch_sharded -- counts exchanged, every rank's compaction kernel writes at its
displacement of the gathered CSR, one NCCL send / recv group completes it on every rank.  The exchange of step i overlaps
the kernels of step i + 1 (it runs on its own stream), all exchanges complete inside the timed region; `value` = all
ranks' bytes / max-over-ranks time of that loop.  `sharded_no_collective` is the same loop without the exchange.
"""
import argparse, ctypes, gzip, json, os, subprocess, sys, threading, time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

ASSET = {"gpt2": "gpt2_style", "llama3": "llama3_style", "wordpiece": "wordpiece", "bert": "wordpiece"}
KIND = {"gpt2": 2, "llama3": 2, "wordpiece": 4, "bert": 2}
SEED = {"gpt2": 2, "llama3": 3, "wordpiece": 4, "bert": 2}


def tokenizer_json(cfg):
    js = gzip.open(os.path.join(ROOT, "assets", ASSET[cfg] + ".json.gz")).read().decode("utf-8")
    if cfg == "bert":   # the bert-base-uncased pipeline: BertNormalizer (lowercase, strip accents, CJK spacing) + BertPreTokenizer + WordPiece
        j = json.loads(js)
        j["normalizer"] = {"type": "BertNormalizer", "clean_text": True, "handle_chinese_chars": True, "strip_accents": None, "lowercase": True}
        j["pre_tokenizer"] = {"type": "BertPreTokenizer"}
        js = json.dumps(j)
    return js


def gen_corpus(kind, seed, first_doc, n_docs, max_bytes, out):
    """Generate docs [first_doc, ...) into `out` (np.uint8 view of pinned memory) with 8 host threads."""
    import corpus
    corpus.build()
    nthr = 8
    per = (n_docs + nthr - 1) // nthr
    parts = [None] * nthr
    cap_each = max_bytes // nthr

    def work(i):
        buf = np.empty(cap_each + 200000, dtype=np.uint8)
        d, o = corpus.generate(kind, seed, first_doc + i * per, per, max_bytes=cap_each, out=buf)
        parts[i] = (d, o)
    ts = [threading.Thread(target=work, args=(i,)) for i in range(nthr)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    pos, offs = 0, [np.zeros(1, dtype=np.uint64)]
    for d, o in parts:
        out[pos:pos + len(d)] = d
        offs.append(o[1:] + np.uint64(pos))
        pos += len(d)
    return pos, np.concatenate(offs)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpus):
        self.gpus, self.p, self.lines = list(gpus), None, []

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", ",".join(map(str, self.gpus)), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for ln in self.p.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except Exception:
            self.p.kill()
        sm, mx, reasons = {}, [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.setdefault(f[0], []).append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        med = {g: float(np.median(v)) for g, v in sorted(sm.items(), key=lambda kv: (len(kv[0]), kv[0]))}
        # sm_mhz: the slowest GPU's median under load (every rank's GPU is sampled, not only rank 0's)
        return {"sm_mhz": min(med.values()) if med else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": min((len(v) for v in sm.values()), default=0), "per_gpu_sm_mhz": list(med.values())}


def cpu_reference_worker(cfg, threads, budget_s, min_mb):
    """Runs in a fresh process (rayon's pool size is fixed at first use): the reference's own Rust encode_batch
    (tokenizers wheel, bindings/python/src/tokenizer.rs:1312-1340) over a bounded sample of the bench corpus."""
    os.environ["TOKENIZERS_PARALLELISM"] = "true"
    os.environ["RAYON_NUM_THREADS"] = str(threads)
    import tokenizers
    tok = tokenizers.Tokenizer.from_str(tokenizer_json(cfg))
    cap = max(int(min_mb) + 8, 40) << 20
    buf = np.empty(cap + (1 << 20), dtype=np.uint8)
    n, off = gen_corpus(KIND[cfg], SEED[cfg], 0, cap // 300, cap, buf)
    raw = buf[:n].tobytes()
    n_avail = len(off) - 1

    def docs(k):
        return [raw[int(off[i]):int(off[i + 1])].decode("utf-8") for i in range(k)]
    probe_n = min(n_avail, 16384)
    d = docs(probe_n)
    tok.encode_batch(d[:2048], add_special_tokens=False)  # warm-up (rayon pool)
    t0 = time.perf_counter(); tok.encode_batch(d, add_special_tokens=False); t1 = time.perf_counter()
    rate = int(off[probe_n]) / (t1 - t0)
    want = max(rate * budget_s, float(min_mb) * (1 << 20))
    k = int(min(n_avail, max(probe_n, np.searchsorted(off, want))))
    d = docs(k)
    best = None
    for _ in range(2 if min_mb <= 0 else 1):
        t0 = time.perf_counter(); enc = tok.encode_batch(d, add_special_tokens=False); dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    nbytes = int(off[k]); ntok = sum(len(e.ids) for e in enc)
    return {"value": nbytes / best / 1e9, "unit": "GB/s", "tokens_per_s": ntok / best, "cores": threads, "kind": "reference",
            "sample": f"tokenizers wheel {tokenizers.__version__} Tokenizer.encode_batch (char offsets), RAYON_NUM_THREADS={threads}, "
                      f"first {k} docs / {nbytes / 1e6:.1f} MB of the bench corpus",
            "seconds": best, "sample_bytes": nbytes}


def host_facts():
    """What explains the reference's thread scaling on this box: cgroup CPU quota, affinity, NUMA layout."""
    f = {"affinity_cpus": len(os.sched_getaffinity(0))}
    for path, key in (("/sys/fs/cgroup/cpu.max", "cgroup_cpu_max"), ("/sys/fs/cgroup/cpu/cpu.cfs_quota_us", "cgroup_cfs_quota_us")):
        try:
            f[key] = open(path).read().strip()
        except Exception:
            pass
    try:
        nodes = sorted(d for d in os.listdir("/sys/devices/system/node") if d.startswith("node"))
        f["numa_nodes"] = {d: open(f"/sys/devices/system/node/{d}/cpulist").read().strip() for d in nodes}
    except Exception:
        pass
    return f


def cpu_reference(cfg, budget_s=4.0, min_mb=256):
    """Thread sweep (all visible cores, 32, 16, 8, 4) on a few-second sample, each in its own process; then the best
    thread count once more on >= min_mb MB of the corpus (BASELINE.md 3)."""
    cores = len(os.sched_getaffinity(0))
    tried = []

    def run(th, bud, mb):
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-worker", cfg, str(th), str(bud), str(mb)],
                             capture_output=True, text=True, timeout=900)
        return json.loads(out.stdout.strip().splitlines()[-1])
    for th in sorted({cores, min(cores, 32), min(cores, 16), min(cores, 8), min(cores, 4)}, reverse=True):
        try:
            tried.append(run(th, budget_s, 0))
        except Exception as ex:
            tried.append({"value": 0.0, "cores": th, "error": str(ex)[:200]})
    best = dict(max(tried, key=lambda r: r.get("value") or 0.0))
    if min_mb > 0 and best.get("value"):
        try:
            big = run(best["cores"], 1.0, min_mb)
            big["sweep_value"] = best["value"]
            best = big
        except Exception as ex:
            best["big_sample_error"] = str(ex)[:200]
    best["host_cores"] = cores
    best["sweep"] = {str(r["cores"]): round(r.get("value") or 0.0, 5) for r in tried}
    best["host"] = host_facts()
    return best


class DevArr:  # zero-copy torch view of an engine-owned device buffer
    def __init__(self, ptr, count, typestr):
        self.__cuda_array_interface__ = {"shape": (count,), "typestr": typestr, "data": (ptr, False), "version": 3}


DUMP_BYTES = 64 << 20
DUMP_DOCS = 1 << 15


def dump_outputs(out_dir, L, res, n_docs):
    """Writes what a caller of b2t_encode_batch_device received from one step, as .npy files of at most DUMP_BYTES in all:
    row_ptr.npy  float64, every stride-th entry of the CSR row pointer (every entry up to 4M documents);
    docs.npy     float64, a fixed seeded sample of DUMP_DOCS documents (ascending; trimmed to the byte budget);
    ids.npy      float32, the token ids of those documents, one after the other (exact: ids < 2^24);
    offsets.npy  float32 [n, 2], their (start, end) char offsets (exact: documents of fewer than 2^24 characters).
    The same arguments give the same inputs, so two builds can be compared file by file."""
    import torch
    T = int(L.b2t_result_n_tokens(res))
    row_ptr = torch.as_tensor(DevArr(L.b2t_result_row_ptr(res), n_docs + 1, "<i8"), device="cuda").cpu().numpy()
    stride = max(1, -(-(n_docs + 1) * 8 // (DUMP_BYTES // 2)))
    docs = np.sort(np.random.default_rng(0).choice(n_docs, size=min(n_docs, DUMP_DOCS), replace=False))
    lens = row_ptr[docs + 1] - row_ptr[docs]
    budget = (DUMP_BYTES - row_ptr[::stride].nbytes - docs.nbytes) // 12    # 4 B of id + 8 B of offsets per token
    docs, lens = docs[np.cumsum(lens) <= budget], lens[np.cumsum(lens) <= budget]
    tok = np.repeat(row_ptr[docs] - (np.cumsum(lens) - lens), lens) + np.arange(int(lens.sum()))
    ids, offs = np.zeros(0, np.float32), np.zeros((0, 2), np.float32)
    if tok.size:
        idx = torch.from_numpy(tok).cuda()
        ids = torch.as_tensor(DevArr(L.b2t_result_ids(res), T, "<i4"), device="cuda")[idx].cpu().numpy().astype(np.float32)
        offs = torch.as_tensor(DevArr(L.b2t_result_offsets(res), 2 * T, "<i4"), device="cuda").view(-1, 2)[idx].cpu().numpy().astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in (("row_ptr", row_ptr[::stride].astype(np.float64)), ("docs", docs.astype(np.float64)), ("ids", ids), ("offsets", offs)):
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def measure(ctx, cfg, kind, mb, steps, warmup, sharded=False, special=None, dump=None):
    """Device-resident and end-to-end numbers of one configuration on this rank.  Returns a dict of raw measurements.
    dump: a directory that receives what the last timed device-resident step computed (dump_outputs)."""
    import torch
    from tokenizers_b200 import Tokenizer, _lib
    L, rank, world, local = ctx["L"], ctx["rank"], ctx["world"], ctx["local"]
    dist = ctx.get("dist")
    tok = Tokenizer.from_str(tokenizer_json(cfg), device=local)
    if special:   # AddedVocabulary::add_special_tokens: the extraction then runs in front of the scan, on the device
        tok.add_special_tokens(special)
        assert tok._dev_added
    max_bytes = mb << 20
    n_docs_target = max_bytes // (200 if kind == 5 else 300)
    hptr = ctypes.c_void_p()
    _lib.check(L.b2t_host_alloc(max_bytes + (1 << 20), ctypes.byref(hptr)))
    hbuf = np.ctypeslib.as_array(ctypes.cast(hptr, ctypes.POINTER(ctypes.c_uint8)), shape=(max_bytes + (1 << 20),))
    n, off = gen_corpus(kind, 5 if kind == 5 else SEED[cfg], rank * n_docs_target, n_docs_target, max_bytes, hbuf)
    n_docs = len(off) - 1
    hoff_ptr = ctypes.c_void_p()
    _lib.check(L.b2t_host_alloc((n_docs + 1) * 8, ctypes.byref(hoff_ptr)))
    hoff = np.ctypeslib.as_array(ctypes.cast(hoff_ptr, ctypes.POINTER(ctypes.c_uint64)), shape=(n_docs + 1,))
    hoff[:] = off
    d_bytes = torch.empty(n + 64, dtype=torch.uint8, device="cuda")
    d_bytes[:n].copy_(torch.from_numpy(hbuf[:n]))
    d_off = torch.from_numpy(off.astype(np.int64)).cuda()
    torch.cuda.synchronize()
    flags = _lib.WANT_OFFSETS
    stream = torch.cuda.current_stream()
    _lib.check(L.b2t_engine_set_profiling(tok.handle, 1))

    def step_device(keep=False):
        res = ctypes.c_void_p()
        _lib.check(L.b2t_encode_batch_device(tok.handle, d_bytes.data_ptr(), n, d_off.data_ptr(), n_docs, flags, ctypes.c_void_p(stream.cuda_stream), ctypes.byref(res)))
        T = L.b2t_result_n_tokens(res)
        if keep:   # the result stays valid until the next call on the engine or b2t_result_free
            return T, res
        L.b2t_result_free(res)
        return T

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    names = (ctypes.c_char_p * 16)(); ms = (ctypes.c_float * 16)()
    for _ in range(warmup):
        T = step_device()
    barrier()
    kern_ms, launches = {}, 0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for i in range(steps):
        if dump and i == steps - 1:
            T, kept = step_device(keep=True)
        else:
            T = step_device()
        launches += L.b2t_engine_last_kernels(tok.handle, names, ms, 16)
        for i in range(16):
            if names[i] is None:
                break
            kern_ms.setdefault(names[i].decode(), []).append(ms[i])
        for i in range(16):
            names[i] = None
    ev1.record(stream)
    barrier()
    dev_ms = ev0.elapsed_time(ev1)
    if dump:
        if rank == 0:
            dump_outputs(dump, L, kept, n_docs)
        L.b2t_result_free(kept)
    _lib.check(L.b2t_engine_set_profiling(tok.handle, 0))

    # ---- N > 1: the sharded product path, exchange of step i overlapping the kernels of step i + 1
    shard_ms = None
    if sharded and world > 1:
        from tokenizers_b200.parallel import encode_batch_sharded
        gs = torch.cuda.Stream()
        out = None
        for _ in range(2):
            r = encode_batch_sharded(tok, d_bytes, n, d_off, n_docs, True, out=out, stream=stream, gather_stream=gs)
            out = (r.ids, r.offsets, r.row_ptr)
        stream.wait_stream(gs); barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record(stream)
        for _ in range(steps):
            r = encode_batch_sharded(tok, d_bytes, n, d_off, n_docs, True, out=out, stream=stream, gather_stream=gs)
        stream.wait_stream(gs)     # every exchange has completed inside the timed region
        g1.record(stream)
        barrier()
        shard_ms = g0.elapsed_time(g1)
        del r, out

    # ---- end to end through the C ABI with pinned host buffers (H2D + kernels + D2H inside the call)
    def step_e2e(fl):
        res = ctypes.c_void_p()
        _lib.check(L.b2t_encode_batch(tok.handle, hptr, hoff_ptr, n_docs, fl, ctypes.byref(res)))
        Tt = L.b2t_result_n_tokens(res)
        L.b2t_result_free(res)
        return Tt
    e2e = {}
    for key, fl in (("e2e", flags), ("e2e_ids_only", 0)):
        for _ in range(warmup):
            step_e2e(fl)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            Te = step_e2e(fl)
        torch.cuda.synchronize()
        e2e[key] = (time.perf_counter() - t0) * 1e3
        assert Te == T
    # dense mode: truncation to 128 + padding to 128 on the device, [n_docs, 128] ids + row lengths come back (no CSR, no mask)
    sp = _lib.DenseSpec()
    sp.struct_size = ctypes.sizeof(_lib.DenseSpec); sp.length = 128; sp.max_length = 128; sp.pad_id = 0; sp.want_mask = 0

    def step_dense():
        res = ctypes.c_void_p()
        _lib.check(L.b2t_encode_batch_dense(tok.handle, hptr, hoff_ptr, n_docs, ctypes.byref(sp), ctypes.byref(res)))
        L.b2t_result_free(res)
    for _ in range(warmup):
        step_dense()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step_dense()
    torch.cuda.synchronize()
    e2e["e2e_dense"] = (time.perf_counter() - t0) * 1e3
    L.b2t_host_free(hptr); L.b2t_host_free(hoff_ptr)
    del d_bytes, d_off, tok
    torch.cuda.empty_cache()
    return {"n": n, "n_docs": n_docs, "T": int(T), "dev_ms": dev_ms, "shard_ms": shard_ms, "e2e_ms": e2e["e2e"], "e2e_ids_ms": e2e["e2e_ids_only"], "e2e_dense_ms": e2e["e2e_dense"],
            "kern_ms": {k: float(np.mean(v)) for k, v in kern_ms.items()}, "launches": int(launches), "steps": steps}


def measure_api(ctx, cfg, mb=128):
    """The drop-in surface a user calls (tokenizers_b200.Tokenizer, the mirror of bindings/python/src/tokenizer.rs:1312-1340),
    wall clock, inputs in ordinary (pageable) host memory, results read back: what the Python layer costs on top of the C ABI."""
    import torch
    from tokenizers_b200 import Tokenizer
    tok = Tokenizer.from_str(tokenizer_json(cfg), device=ctx["local"])
    buf = np.empty((mb << 20) + (1 << 20), dtype=np.uint8)
    n, off = gen_corpus(KIND[cfg], SEED[cfg], 0, (mb << 20) // 300, mb << 20, buf)
    data, off = buf[:n].copy(), np.ascontiguousarray(off, dtype=np.uint64)
    n_docs = len(off) - 1

    def timed(fn, reps=3):
        fn()
        best = 1e30
        for _ in range(reps):
            t0 = time.perf_counter(); r = fn(); torch.cuda.synchronize(); best = min(best, time.perf_counter() - t0)
        return best, r
    res = {"sample": f"{n / 1e6:.0f} MB / {n_docs} docs of the bench corpus, pageable numpy input, best of 3"}
    t, be = timed(lambda: tok.encode_batch_csr(data, off))
    res["encode_batch_csr"] = {"GBps": n / t / 1e9, "tokens_per_s": be.n_tokens / t, "what": "ids + char offsets + word ids copied out of the pinned result"}
    t, be = timed(lambda: tok.encode_batch_csr(data, off, zero_copy=True))
    res["encode_batch_csr_zero_copy"] = {"GBps": n / t / 1e9, "what": "the arrays are views of the result's pinned buffers"}
    t, be = timed(lambda: tok.encode_batch_csr(data, off, offsets=False, word_ids=False, zero_copy=True))
    res["encode_batch_csr_ids_only_zero_copy"] = {"GBps": n / t / 1e9}
    k = min(n_docs, 200000)
    raw = data.tobytes()
    docs = [raw[int(off[i]):int(off[i + 1])].decode("utf-8") for i in range(k)]
    nb = int(off[k])
    t, encs = timed(lambda: tok.encode_batch(docs, add_special_tokens=False), reps=2)
    res["encode_batch_list_of_str"] = {"GBps": nb / t / 1e9, "docs_per_s": k / t, "docs": k, "what": "list[str] in, list of lazy Encoding views out (UTF-8 encode + join on the host)"}
    t, encs = timed(lambda: tok.encode_batch_fast(docs, add_special_tokens=False), reps=2)
    res["encode_batch_fast_list_of_str"] = {"GBps": nb / t / 1e9, "docs_per_s": k / t}
    tok.enable_truncation(128); tok.enable_padding(length=128, pad_id=0)
    t, dn = timed(lambda: tok.encode_batch_dense(data, off, want_mask=False))
    res["encode_batch_dense_128"] = {"GBps": n / t / 1e9, "rows_per_s": n_docs / t, "what": "truncation to 128 + padding to 128 on the device, [n_docs, 128] ids + row lengths back"}
    return res


def roofline_of(m, peaks, cfg):
    peak = peaks.get("hbm_gbs", 6650.0)
    k1 = m["kern_ms"].get("pretok_scan", float("nan"))
    n = m["n"]
    k1_bytes = n * 1.25 + (n / 2048) * 8  # bytes + doc_bits in, start_bits + page summaries out (DESIGN.md)
    traffic, src = None, None
    try:  # dram bytes of one launch from the committed ncu --set full capture (profiles/), scaled by input size
        tj = json.load(open(os.path.join(ROOT, "profiles", "k1_traffic.json")))
        if tj.get("config") == cfg:
            traffic, src = tj["dram_bytes_per_input_byte"] * n, tj.get("source", "profiles/k1_traffic.json")
    except Exception:
        pass
    return {"kernel": "pretok_lean_kernel" if cfg != "llama3" else "pretok_stream_kernel", "bound": "hbm", "achieved": k1_bytes / (k1 * 1e-3) / 1e9, "peak": peak,
            "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "B200_PROFILING.md fallback (of fallback)",
            "unit": "GB/s", "frac": k1_bytes / (k1 * 1e-3) / 1e9 / peak, "traffic": traffic,
            "traffic_source": (f"ncu capture {src}, dram bytes per input byte x this launch's input bytes (not re-measured in this run)" if traffic else None),
            "algorithmic_bytes_per_launch": k1_bytes, "ms_per_launch": k1, "input_GBps": n / (k1 * 1e-3) / 1e9,
            "frac_survey_8d_accounting": (n * 1.75) / (k1 * 1e-3) / 1e9 / peak,
            "note": "achieved uses THIS kernel's layout (bytes + doc bitmap in, split bitmap + page summaries out = 1.25 B per input byte); "
                    "frac_survey_8d_accounting is the same time with SURVEY.md 8(d)'s u32-start-list accounting (N + 4*N_pretok ~ 1.75 B/B)"}


def main():
    if len(sys.argv) >= 6 and sys.argv[1] == "--cpu-worker":
        print(json.dumps(cpu_reference_worker(sys.argv[2], int(sys.argv[3]), float(sys.argv[4]), float(sys.argv[5]))))
        return
    # Only the JSON line may reach stdout (NCCL and others print there): park the real stdout, send fd 1 to stderr.
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--mb", type=int, default=1024, help="corpus size per GPU in MiB")
    ap.add_argument("--config", default="gpt2", choices=list(ASSET))
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the secondary configs (llama3 / wordpiece / skew)")
    ap.add_argument("--kind", type=int, default=0, help="corpus kind override (5 = length-skew stress of BASELINE configs[4])")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed device-resident step computed to DIR/<name>.npy "
                    "(rank 0's batch; a seeded sample, at most 64 MiB: see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    a.warmup = max(a.warmup, 3) if a.impl != "reference" else a.warmup
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = a.config
    WORK = {"gpt2": "GPT-2 ByteLevel BPE (50257 vocab trained offline by the reference trainer), synthetic UTF-8 docs avg ~480 B",
            "llama3": "Llama-3-style BPE (tiktoken regex, 128k vocab, ignore_merges)", "wordpiece": "Whitespace + WordPiece 30522",
            "bert": "bert-base-uncased pipeline: BertNormalizer + BertPreTokenizer + WordPiece 30522, mixed-case multilingual corpus"}
    SKEW = " [length-skew corpus: Zipf doc lengths 8 B-64 KB, 0.1 % docs hold a 4-64 KB letter/space run]"
    workload = WORK[cfg] + (SKEW if a.kind == 5 else "")

    if a.impl == "reference":
        # the reference's CPU implementation, all host threads, bounded sample per step; rank 0 only
        if rank != 0:
            return
        per_step = []
        for s_i in range(a.warmup + a.steps):
            r = cpu_reference(cfg, budget_s=max(1.5, 30.0 / (3 * (a.warmup + a.steps))), min_mb=256 if s_i == a.warmup else 0)
            if s_i >= a.warmup:
                per_step.append(r)
        r = max(per_step, key=lambda x: (x.get("sample_bytes", 0) >= (200 << 20), x["value"]))
        out = {"impl": "reference", "metric": "encode_batch input throughput", "value": r["value"], "unit": "GB/s", "tokens_per_s": r["tokens_per_s"],
               "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": r["seconds"] * 1e3, "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": {"workload": workload, "bytes_per_step": r.get("sample_bytes"), "sample": r["sample"]},
               "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "host_cores", "sweep", "host") if k in r},
               "e2e": {"value": r["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        real_stdout.write(json.dumps(out) + "\n"); real_stdout.flush()
        return

    import torch
    from tokenizers_b200 import _lib
    from tokenizers_b200.parallel import bind_to_gpu_numa_node
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local)   # before any pinned allocation
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = {"L": _lib.lib(), "rank": rank, "world": world, "local": local, "dist": dist}
    # one node: local rank r runs on the r-th visible GPU (nvidia-smi does not honour CUDA_VISIBLE_DEVICES, so map it)
    vis = [v.strip() for v in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if v.strip()]
    sampler = ClockSampler(vis[:world] if len(vis) >= world else range(world))
    if rank == 0:
        sampler.start()  # samples every 50 ms from the warm-up through the timed device and e2e regions
    kind = a.kind or KIND[cfg]
    m = measure(ctx, cfg, kind, a.mb, a.steps, a.warmup, sharded=True, dump=a.dump_outputs)
    clocks = sampler.stop() if rank == 0 else None

    # ---- reduce over ranks: time = max, work = sum
    if world > 1:
        v = torch.tensor([m["dev_ms"], m["e2e_ms"], m["e2e_ids_ms"], m["shard_ms"], m["e2e_dense_ms"]], dtype=torch.float64, device="cuda")
        dist.all_reduce(v, op=dist.ReduceOp.MAX)
        w = torch.tensor([float(m["n"]), float(m["T"])], dtype=torch.float64, device="cuda")
        dist.all_reduce(w, op=dist.ReduceOp.SUM)
        mine = torch.tensor([m["dev_ms"] / a.steps, sum(m["kern_ms"].values()), m["e2e_ms"] / a.steps, float(numa if numa is not None else -1)], dtype=torch.float64, device="cuda")
        allr = torch.empty(4 * world, dtype=torch.float64, device="cuda")
        dist.all_gather_into_tensor(allr, mine)
        allr = allr.reshape(world, 4).tolist()
        dev_ms, e2e_ms, e2e_ids_ms, shard_ms, e2e_dense_ms = v.tolist(); tot_bytes, tot_tok = w.tolist()
        # BASELINE configs[4]: the length-skew corpus across the ranks (Zipf doc lengths 8 B-64 KB, 0.1 % of the documents hold a
        # 4-64 KB run), same sharded step; what the load balance looks like is in the per-rank times
        skew = None
        if cfg == "gpt2" and a.kind == 0 and not a.no_configs:
            try:
                ms = measure(ctx, "gpt2", 5, 512, 3, 3, sharded=True)
                sv = torch.tensor([ms["shard_ms"], ms["dev_ms"]], dtype=torch.float64, device="cuda")
                dist.all_reduce(sv, op=dist.ReduceOp.MAX)
                sw = torch.tensor([float(ms["n"])], dtype=torch.float64, device="cuda")
                dist.all_reduce(sw, op=dist.ReduceOp.SUM)
                smine = torch.tensor([ms["dev_ms"] / ms["steps"], ms["kern_ms"].get("bpe_long", 0.0) + ms["kern_ms"].get("long_find", 0.0)], dtype=torch.float64, device="cuda")
                sall = torch.empty(2 * world, dtype=torch.float64, device="cuda")
                dist.all_gather_into_tensor(sall, smine)
                sall = sall.reshape(world, 2).tolist()
                per = [x[0] for x in sall]
                skew = {"workload": "length-skew corpus, 512 MB per GPU, 3 timed steps, the sharded step with its exchange",
                        "value": sw.item() / (sv[0].item() / ms["steps"] * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": sv[0].item() / ms["steps"],
                        "no_collective_GBps": sw.item() / (sv[1].item() / ms["steps"] * 1e-3) / 1e9,
                        "per_rank_ms_per_step": [round(x, 3) for x in per], "imbalance_max_over_mean": max(per) / (sum(per) / len(per)),
                        "per_rank_long_pretoken_kernels_ms": [round(x[1], 3) for x in sall]}
            except Exception as ex:
                skew = {"error": str(ex)[:300]}
    else:
        dev_ms, e2e_ms, e2e_ids_ms, shard_ms, e2e_dense_ms = m["dev_ms"], m["e2e_ms"], m["e2e_ids_ms"], None, m["e2e_dense_ms"]
        tot_bytes, tot_tok = float(m["n"]), float(m["T"])
        allr = [[m["dev_ms"] / a.steps, sum(m["kern_ms"].values()), m["e2e_ms"] / a.steps, float(numa if numa is not None else -1)]]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    n, n_docs, T = m["n"], m["n_docs"], m["T"]
    dev_step = dev_ms / a.steps
    head_step = (shard_ms / a.steps) if world > 1 else dev_step     # N > 1: the sharded path with its exchange is the headline
    gbps = lambda ms_: tot_bytes / (ms_ * 1e-3) / 1e9
    out = {"metric": "encode_batch input throughput", "value": gbps(head_step), "unit": "GB/s",
           "tokens_per_s": tot_tok / (head_step * 1e-3), "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": head_step,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
           "config": {"workload": workload + f", {n / 1e6:.0f} MB / {n_docs} docs per GPU, ids + char offsets", "bytes_per_gpu": n, "docs_per_gpu": n_docs,
                      "tokens_per_gpu": int(T), "l2": "inputs larger than L2 (no flush needed)",
                      "parallelism": ("one GPU" if world == 1 else
                                      f"one batch of {world} shards (contiguous, one per rank); every rank ends with the whole CSR: counts exchanged, compaction "
                                      f"writes at the rank's displacement, one NCCL send/recv group; the exchange of a step overlaps the next step's kernels")},
           "kernels_ms": m["kern_ms"], "per_rank_ms_per_step": [round(x[0], 3) for x in allr], "per_rank_kernel_ms_per_step": [round(x[1], 3) for x in allr],
           "roofline": roofline_of(m, peaks, cfg),
           "e2e": {"value": gbps(e2e_ms / a.steps), "unit": "GB/s", "tokens_per_s": tot_tok / (e2e_ms / a.steps * 1e-3), "ms_per_step": e2e_ms / a.steps,
                   "h2d_bytes_per_step": int(n + (n_docs + 1) * 8), "d2h_bytes_per_step": int(T * 12 + (n_docs + 1) * 8 + 16 * ((n >> 26) + 1)),
                   "per_rank_ms_per_step": [round(x[2], 3) for x in allr], "numa_node_of_rank": [int(x[3]) for x in allr]},
           "e2e_ids_only": {"value": gbps(e2e_ids_ms / a.steps), "unit": "GB/s", "ms_per_step": e2e_ids_ms / a.steps,
                            "what": "b2t_encode_batch with flags = 0 (the encode_batch_fast analogue, tokenizer/mod.rs:1382): ids + row_ptr back, 4 B per token",
                            "h2d_bytes_per_step": int(n + (n_docs + 1) * 8), "d2h_bytes_per_step": int(T * 4 + (n_docs + 1) * 8 + 16 * ((n >> 26) + 1))},
           "e2e_dense_128": {"value": gbps(e2e_dense_ms / a.steps), "unit": "GB/s", "ms_per_step": e2e_dense_ms / a.steps,
                             "what": "b2t_encode_batch_dense, pinned host buffers: truncation to 128 tokens + padding to 128 on the device, [n_docs, 128] u32 ids + row lengths back",
                             "h2d_bytes_per_step": int(n + (n_docs + 1) * 8), "d2h_bytes_per_step": int(n_docs * 128 * 4 + n_docs * 4)},
           "gpu_launches": m["launches"], "clocks": clocks}
    if world > 1:
        out["sharded_no_collective"] = {"what": "the same shards, every rank keeps only its own slice of the CSR (no exchange)", "ms_per_step": dev_step,
                                        "value": gbps(dev_step), "unit": "GB/s"}
        out["exchange"] = {"what": "bytes of other ranks' CSR each rank receives per step", "bytes": int((tot_tok - T) * 12 + (world - 1) * (n_docs + 1) * 8)}
        if skew is not None:
            out["configs"] = {"skew_sharded": skew}
    if world == 1 and not a.no_configs and a.kind == 0 and cfg == "gpt2":
        # the other BASELINE configs on the same line: smaller corpora, fewer steps (stated), same measurement code
        out["configs"] = {}
        for name, c2, k2 in (("llama3", "llama3", 2), ("wordpiece", "wordpiece", 4), ("bert_uncased", "bert", 2), ("skew", "gpt2", 5)):
            try:
                mm = measure(ctx, c2, k2, 512, 3, 3)
                st = mm["dev_ms"] / mm["steps"]
                out["configs"][name] = {
                    "workload": WORK[c2] + (SKEW if k2 == 5 else "") + f", {mm['n'] / 1e6:.0f} MB / {mm['n_docs']} docs, 3 timed steps",
                    "value": mm["n"] / (st * 1e-3) / 1e9, "unit": "GB/s", "tokens_per_s": mm["T"] / (st * 1e-3), "ms_per_step": st, "kernels_ms": mm["kern_ms"],
                    "roofline_frac": roofline_of(mm, peaks, c2)["frac"], "roofline_kernel_ms": mm["kern_ms"].get("pretok_scan"),
                    "e2e": {"value": mm["n"] / (mm["e2e_ms"] / mm["steps"] * 1e-3) / 1e9, "unit": "GB/s"},
                    "e2e_ids_only": {"value": mm["n"] / (mm["e2e_ids_ms"] / mm["steps"] * 1e-3) / 1e9, "unit": "GB/s"}}
            except Exception as ex:
                out["configs"][name] = {"error": str(ex)[:300]}
        # added-token extraction on the device (added_vocabulary.rs:430-564): the same corpus with "<|endoftext|>" at the end of every document
        try:
            mm = measure(ctx, "gpt2", 6, 512, 3, 3, special=["<|endoftext|>"])
            st = mm["dev_ms"] / mm["steps"]
            out["configs"]["gpt2_special_token_in_every_doc"] = {
                "workload": WORK["gpt2"] + f" + the special token <|endoftext|> behind every document, extracted on the device, {mm['n'] / 1e6:.0f} MB / {mm['n_docs']} docs, 3 timed steps",
                "value": mm["n"] / (st * 1e-3) / 1e9, "unit": "GB/s", "tokens_per_s": mm["T"] / (st * 1e-3), "ms_per_step": st, "kernels_ms": mm["kern_ms"],
                "e2e": {"value": mm["n"] / (mm["e2e_ms"] / mm["steps"] * 1e-3) / 1e9, "unit": "GB/s"}}
        except Exception as ex:
            out["configs"]["gpt2_special_token_in_every_doc"] = {"error": str(ex)[:300]}
        # the reference benches BPE with its word cache off too (benches/bpe_benchmark.rs:59-71, cache_capacity(0)): same corpus, the
        # per-batch word cache of the page kernel switched off, so that every pre-token goes through the merge loop
        try:
            os.environ["B2T_WCACHE"] = "0"
            mm = measure(ctx, "gpt2", 2, 256, 2, 3)
            st = mm["dev_ms"] / mm["steps"]
            out["configs"]["gpt2_word_cache_off"] = {
                "workload": WORK["gpt2"] + f", {mm['n'] / 1e6:.0f} MB / {mm['n_docs']} docs, 2 timed steps, B2T_WCACHE=0 (no word cache: every pre-token is merged)",
                "value": mm["n"] / (st * 1e-3) / 1e9, "unit": "GB/s", "tokens_per_s": mm["T"] / (st * 1e-3), "ms_per_step": st, "kernels_ms": mm["kern_ms"]}
        except Exception as ex:
            out["configs"]["gpt2_word_cache_off"] = {"error": str(ex)[:300]}
        finally:
            os.environ.pop("B2T_WCACHE", None)
    if world == 1 and not a.no_configs and a.kind == 0 and cfg == "gpt2":
        try:
            out["api"] = measure_api(ctx, cfg)
        except Exception as ex:
            out["api"] = {"error": str(ex)[:300]}
    if not a.no_cpu and world == 1:
        try:
            cb = cpu_reference(cfg)
            out["cpu_baseline"] = {k: v for k, v in cb.items() if k != "seconds"}
            if cb.get("tokens_per_s"):
                out["cpu_baseline"]["gpu_over_cpu_tokens_per_s"] = {"device_resident": out["tokens_per_s"] / cb["tokens_per_s"],
                                                                    "e2e": out["e2e"]["tokens_per_s"] / cb["tokens_per_s"]}
        except Exception as ex:  # the wheel is part of the image; if it is missing say so instead of inventing a number
            out["cpu_baseline"] = {"value": None, "unit": "GB/s", "cores": len(os.sched_getaffinity(0)), "kind": "reference", "sample": f"unavailable: {ex}"}
    real_stdout.write(json.dumps(out) + "\n"); real_stdout.flush()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
