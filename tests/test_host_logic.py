"""CPU: host-side logic of the product — index construction, sdsl .fmi parsing, native container,
C-ABI surface — plus the per-thread device primitives compiled for the host (tests/hostcheck)."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from oracle.fm_oracle import PortFM

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
G = np.load(os.path.join(HERE, "golden", "fm_golden.npz"))


def test_abi_library_loads_and_exports_every_declared_symbol():
    from seal_b200 import _lib
    for hdr in sorted(os.listdir(os.path.join(ROOT, "include"))):
        text = open(os.path.join(ROOT, "include", hdr)).read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        names = set(re.findall(r"\b(seal(?:fm|dec|bart|ev)_[a-z0-9_]+)\s*\(", text))
        assert names, hdr
        for n in sorted(names):
            assert hasattr(_lib.lib, n), f"{n} declared in include/{hdr} but not exported"
    assert _lib.lib.sealfm_abi_version() >= 1


def test_queries_fail_loudly_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from seal_b200.cpp_modules.fm_index import FMIndex
    from seal_b200._lib import SealB200Error
    fm = FMIndex(); fm.initialize(G["toy.text"])
    with pytest.raises(SealB200Error) as e:
        fm.backward_search_step(11, 0, fm.size())
    assert e.value.code == -4


@pytest.mark.parametrize("name", ["keeper", "toy", "rand5k", "phrase"])
def test_builder_sections_equal_oracle_sections(name):
    """SA-IS + level-wise WT (product, C++) vs prefix-doubling + sdsl-style WT (oracle, C):
    tree bits, alphabet, C, SA/ISA samples must agree word for word."""
    from seal_b200.cpp_modules.fm_index import FMIndex
    text = G[f"{name}.text"]
    fm = FMIndex(); fm.initialize(text)
    p = PortFM(text)
    assert fm.size() == p.size()
    assert np.array_equal(fm.section(0), p.section("tree_words"))
    assert np.array_equal(fm.section(1), p.section("alphabet"))
    assert np.array_equal(fm.section(2), p.section("C"))
    assert np.array_equal(fm.section(3), p.section("sa_samples"))
    assert np.array_equal(fm.section(4), p.section("isa_samples"))


def test_sdsl_fmi_written_by_reference_parses_to_the_same_sections(tmp_path):
    """tests/golden/tiny_ref.fmi was written by the reference's FMIndex::save (sdsl store_to_file)."""
    from seal_b200.cpp_modules.fm_index import FMIndex, load_FMIndex
    ref = load_FMIndex(os.path.join(HERE, "golden", "tiny_ref.fmi"))
    own = FMIndex(); own.initialize(G["phrase.text"])
    assert ref.size() == own.size()
    for s in range(5):
        assert np.array_equal(ref.section(s), own.section(s)), s
    # native container round trip
    p = str(tmp_path / "x.fmi")
    own.save(p)
    back = load_FMIndex(p)
    for s in range(5):
        assert np.array_equal(back.section(s), own.section(s)), s


def test_build_from_file_matches_in_memory(tmp_path):
    from seal_b200.cpp_modules.fm_index import FMIndex
    text = G["rand5k.text"]
    p = tmp_path / "t.bin"
    text.astype("<i4").tofile(p)
    a = FMIndex(); a.initialize_from_file(str(p), 4)
    b = FMIndex(); b.initialize(text)
    for s in range(5):
        assert np.array_equal(a.section(s), b.section(s))


def test_bad_inputs_return_errors_not_aborts(tmp_path):
    from seal_b200.cpp_modules.fm_index import FMIndex, load_FMIndex
    from seal_b200._lib import SealB200Error
    with pytest.raises(SealB200Error):
        load_FMIndex(str(tmp_path / "missing.fmi"))
    junk = tmp_path / "junk.fmi"; junk.write_bytes(b"\x01" * 100)
    with pytest.raises(SealB200Error):
        load_FMIndex(str(junk))
    with pytest.raises(SealB200Error):
        FMIndex().initialize([5, 0, 7])          # 0 is the sentinel
    with pytest.raises(RuntimeError):
        FMIndex().size()


# ---- per-thread device primitives, compiled for the host -------------------------------------------
@pytest.fixture(scope="module")
def hostcheck():
    so = os.path.join(HERE, "hostcheck", "libhostcheck.so")
    srcs = [os.path.join(HERE, "hostcheck", "hostcheck.cpp"), os.path.join(ROOT, "seal_b200", "csrc", "fm_host.cpp")]
    deps = srcs + [os.path.join(ROOT, "seal_b200", "csrc", f) for f in ("fm_device.cuh", "fm_layout.hpp", "fm_host.hpp", "sais.hpp")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", so] + srcs +
                              ["-Wl,-Bsymbolic", "-Wl,--exclude-libs,ALL"])
    L = C.CDLL(so)
    u64, vp = C.c_uint64, C.c_void_p
    L.hc_build.restype = vp; L.hc_build.argtypes = [vp, u64]
    L.hc_load.restype = vp; L.hc_load.argtypes = [C.c_char_p]
    L.hc_free.argtypes = [vp]
    L.hc_size.restype = u64; L.hc_size.argtypes = [vp]
    L.hc_lf_step.argtypes = [vp, u64, vp, vp, vp, vp, vp]
    L.hc_distinct_count.restype = u64; L.hc_distinct_count.argtypes = [vp, u64, u64, vp, u64]
    L.hc_locate.restype = u64; L.hc_locate.argtypes = [vp, u64]
    L.hc_extract.argtypes = [vp, u64, u64, vp]
    return L


@pytest.mark.parametrize("name", ["keeper", "toy", "rand5k", "phrase"])
def test_device_primitives_on_host_match_goldens(hostcheck, name):
    L = hostcheck
    text = np.ascontiguousarray(G[f"{name}.text"])
    h = L.hc_build(text.ctypes.data, len(text))
    assert h
    size = int(G[f"{name}.size"])
    fl, fh = G[f"{name}.first_lo"], G[f"{name}.first_hi"]
    syms = np.arange(len(fl), dtype=np.uint64)
    lo = np.zeros_like(syms); hi = np.full_like(syms, size)
    ol = np.zeros_like(syms); oh = np.zeros_like(syms)
    L.hc_lf_step(h, len(syms), syms.ctypes.data, lo.ctypes.data, hi.ctypes.data, ol.ctypes.data, oh.ctypes.data)
    assert np.array_equal(ol, fl) and np.array_equal(oh, fh)
    wsym, wlo, whi = G[f"{name}.walk_sym"], G[f"{name}.walk_lo"], G[f"{name}.walk_hi"]
    dc_off, dc = G[f"{name}.dc_off"], G[f"{name}.dc"]
    W, D = wsym.shape
    cl = np.zeros(W, dtype=np.uint64); ch = np.full(W, size, dtype=np.uint64)
    buf = np.zeros(1 << 18, dtype=np.uint64)
    for d in range(D):
        sy = np.ascontiguousarray(wsym[:, d])
        a = np.zeros(W, dtype=np.uint64); b = np.zeros(W, dtype=np.uint64)
        L.hc_lf_step(h, W, sy.ctypes.data, cl.ctypes.data, ch.ctypes.data, a.ctypes.data, b.ctypes.data)
        assert np.array_equal(a, wlo[:, d]) and np.array_equal(b, whi[:, d])
        cl, ch = a, b
        for w in range(W):
            k = w * D + d
            got = L.hc_distinct_count(h, int(a[w]), int(b[w]) + 1, buf.ctypes.data, len(buf)) if int(b[w]) + 1 >= int(a[w]) else 0
            assert np.array_equal(buf[:got], dc[int(dc_off[k]):int(dc_off[k + 1])])
    for row, exp in zip(G[f"{name}.loc_rows"], G[f"{name}.loc"]):
        assert L.hc_locate(h, int(row)) == int(exp)
    eo, ex = G[f"{name}.ext_off"], G[f"{name}.ext"]
    for i, (b, e) in enumerate(zip(G[f"{name}.ext_b"], G[f"{name}.ext_e"])):
        o = np.zeros(max(int(e) - int(b), 1), dtype=np.uint64)
        L.hc_extract(h, int(b), int(e), o.ctypes.data)
        assert np.array_equal(o[: int(e) - int(b)], ex[int(eo[i]):int(eo[i + 1])])
    L.hc_free(h)


def test_gpu_index_builder_reports_missing_device():
    """sealfm_build_gpu must fail loudly (SEALFM_ENODEVICE), never fall back to the host builder, without a GPU."""
    import ctypes as C
    import numpy as np
    import torch
    from seal_b200 import _lib
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a CUDA device is present")
    a = np.array([5, 6, 7], dtype=np.uint64); out = C.c_void_p()
    assert _lib.lib.sealfm_build_gpu(a.ctypes.data, 3, 0, C.byref(out)) == -4
    assert out.value is None


def test_records_to_output_matches_the_reference_formula():
    """beam_search.py:555 / :752-755 restated literally vs the vectorised product conversion (every bit)."""
    import numpy as np
    from seal_b200.beam_search import records_to_output
    rng = np.random.default_rng(5)
    Q, H, T = 7, 40, 9
    rec = {"scores": (rng.standard_normal((Q, H)) * 5 - 20).astype(np.float32), "lens": rng.integers(1, T + 1, size=(Q, H)).astype(np.int32),
           "tokens": rng.integers(0, 50000, size=(Q, H, T)).astype(np.int32)}
    rec["scores"][rng.random((Q, H)) < 0.4] = -np.inf
    rec["scores"][2, :] = -np.inf                                    # a query whose hypotheses are all masked
    for lp in (0.0, 0.5, 1.0, 0.37):
        exp = []
        for q in range(Q):
            row = []
            for i in range(H):
                n = int(rec["lens"][q, i])
                sc = float(rec["scores"][q, i]) / (n ** lp)
                if sc > float("-inf"):
                    row.append((sc * n ** lp, rec["tokens"][q, i, :n].tolist()))
            exp.append(row)
        assert records_to_output(rec, lp) == exp


def _host_build(text):
    import ctypes as C
    import numpy as np
    from seal_b200._lib import lib, check
    from seal_b200.cpp_modules.fm_index import FMIndex as RawFM
    a = np.ascontiguousarray(np.asarray(text, dtype=np.uint64)); out = C.c_void_p()
    check(lib.sealfm_build(a.ctypes.data, len(a), C.byref(out)))
    fm = RawFM(); fm._adopt(out.value)
    return fm


def sdsl_writer_texts():
    """The texts of the .fmi writer test (both select_support_mcl construction paths, contiguous and sparse alphabets,
    long select blocks); tests/golden/make_fmi_golden.py saves each with the reference's FMIndex::save."""
    from seal_b200.synthetic import make_corpus, corpus_symbols
    rng = np.random.default_rng(1)
    return {"toy": [12, 13, 12, 14, 13, 12], "one": [5], "contiguous": rng.integers(1, 6, size=300),
            "rand5k": rng.integers(10, 300, size=5000), "wide": rng.integers(10, 50000, size=7000),
            "phrase 40k": corpus_symbols(make_corpus(n_docs=400, doc_len=100, n_phrases=600, seed=4)),   # tree > 100 000 bits
            "run": np.full(9000, 11), "sparse": np.array([2 ** 15] + [1] * 20000, dtype=np.uint64)}


def test_sdsl_format_writer_round_trip_and_reference_bytes(tmp_path):
    """FMIndex.save writes the reference's own .fmi format: (1) our loader reads it back to identical sections;
    (2) the file is byte-identical to the reference's FMIndex::save of the same text, whose length and SHA-256 are
    stored in tests/golden/fmi_golden.json."""
    import hashlib
    import json
    import numpy as np
    from seal_b200.cpp_modules.fm_index import load_FMIndex
    with open(os.path.join(HERE, "golden", "fmi_golden.json")) as f:
        ref_files = json.load(f)["files"]
    texts = sdsl_writer_texts()
    assert sorted(texts) == sorted(ref_files)
    for name, text in texts.items():
        fm = _host_build(text)
        ours = str(tmp_path / "ours.fmi")
        fm.save(ours)
        back = load_FMIndex(ours)
        for w in range(5):
            assert np.array_equal(fm.section(w), back.section(w)), (name, w)
        data = open(ours, "rb").read()
        assert {"bytes": len(data), "sha256": hashlib.sha256(data).hexdigest()} == ref_files[name], name
        nat = str(tmp_path / "ours.native")
        fm.save(nat, native=True)
        assert np.array_equal(load_FMIndex(nat).section(0), fm.section(0))


@pytest.mark.parametrize("lp,seed", [(0.0, 1), (1.0, 2), (0.7, 3), (1.0, 4)])
def test_stock_scorer_replay_equals_scorer_in_the_loop(lp, seed):
    """keep_history=False (seal/beam_search.py:505-515): the product replays transformers' stock BeamSearchScorer over
    the per-step candidate records of the keep_history=True kernels.  Here, on the CPU, with a synthetic logit model
    that ends hypotheses often: records rebuilt from the oracle's keep_history=True trace -> product replay, against
    the oracle running the stock scorer INSIDE the loop (done queries padded, early exit, finalize)."""
    import torch
    from oracle.decode_oracle import constrained_beam_search_oracle
    from seal_b200.beam_search import _replay_beam_search_scorer
    V, B, T, Q, EOS, PAD = 40, 3, 9, 4, 2, 1
    g = torch.Generator().manual_seed(seed)
    table = torch.randn(V, V, generator=g) * 2.0
    table[:, EOS] += 2.5                                         # hypotheses finish early and often

    def step_logits(dec):
        return table[dec[:, -1]] + 0.3 * table[dec[:, 0] * 0 + dec.shape[1] % V]

    kw = dict(batch_size=Q, index=None, num_beams=B, min_length=0, max_length=T, length_penalty=lp, eos_token_id=EOS,
              pad_token_id=PAD, decoder_start_token_id=EOS, model_eos_token_id=EOS, forced_eos_token_id=None,
              disable_fm_index=True)
    trace = []
    constrained_beam_search_oracle(step_logits, trace=trace, **kw)
    steps = [t for t in trace if "top_scores" in t]; fin = trace[-1]
    H = len(steps) * 2 * B + B
    rec = {"scores": np.zeros((Q, H), np.float32), "lens": np.zeros((Q, H), np.int32), "tokens": np.full((Q, H, T), PAD, np.int32)}
    for st, t in enumerate(steps):
        for q in range(Q):
            for k in range(2 * B):
                h = st * 2 * B + k
                par = t["input_ids"][q * B + int(t["top_beams"][q, k])].tolist()
                rec["scores"][q, h] = float(t["top_scores"][q, k]); rec["lens"][q, h] = len(par) + 1
                rec["tokens"][q, h, :len(par) + 1] = par + [int(t["top_tokens"][q, k])]
    for q in range(Q):
        for j in range(B):
            h = len(steps) * 2 * B + j
            row = fin["final_input_ids"][q * B + j].tolist()
            rec["scores"][q, h] = float(fin["final_beam_scores"][q * B + j]); rec["lens"][q, h] = len(row); rec["tokens"][q, h, :len(row)] = row
    beams, seq, seq_scores = _replay_beam_search_scorer(rec, B, lp, EOS, PAD, T)
    exp = constrained_beam_search_oracle(step_logits, keep_history=False, **kw)
    exp_seq = constrained_beam_search_oracle(step_logits, keep_history=False, transformers_output=True, **kw)
    got = [[(sc * (len(t) ** lp), t) for sc, t in b if sc > float("-inf")] for b in beams]
    assert any(len(t) < T for b in got for _, t in b), "the case must contain finished hypotheses"
    for qa, qb in zip(got, exp):
        assert [t for _, t in qa] == [t for _, t, _ in qb]
        assert all(abs(x[0] - y[0]) < 1e-5 for x, y in zip(qa, qb))
    assert np.array_equal(seq, exp_seq.numpy())
