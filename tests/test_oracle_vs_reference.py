"""Pin the oracle to the reference itself (CPU only).  The reference's outputs on these inputs are recorded in
tests/golden/reference_cpu.npz by tools/make_golden_reference.py from the UNMODIFIED reference CPU sources compiled by
oracle/Makefile; the inputs are regenerated here from the same seeds (the functions below are shared with the tool).

  * scans: oracle/crf_oracle.c vs the reference's inner::forward_scores / backward_scores / softmax
    (dorado/basecall/decode/CPUDecoder.cpp:43-92,130) on a fixed set of rows.  libtorch's vectorised exp/log and
    reduction order are not reproducible bit for bit, and the guides reach magnitudes of ~2 per block (fp32 ulp 2.4e-4
    at 4000), so the bound is 4 ulp of the largest guide.
  * beam search + sequence/qstring generation: the reference's own beam_search_decode
    (dorado/basecall/decode/beam_search.cpp:522-606) fed the ORACLE's guides must give bit-identical sequence and
    moves; the qstring may differ in isolated characters where libm's powf/log10f and the contract's differ in the
    last ulp (bound 1 %).
  * network forward: oracle/nn_oracle.py vs the reference's CRFModel / TxModel forward on the same weights, at a fixed
    sample of score positions (oracle.golden.sample_index).
"""
import pathlib

import numpy as np
import pytest

from conftest import model_dir, synthetic_scores
from oracle.golden import sample_index
from oracle.oracle import DecodeResult

GOLDEN = pathlib.Path(__file__).resolve().parent / "golden" / "reference_cpu.npz"
SCAN_CASES = [(3, 300), (4, 200), (5, 60)]
SCAN_ROWS = {3: 16, 4: 8, 5: 4}         # recorded rows of the guides per state_len (keeps the fixture small)
BEAM_CASES = [(3, 400), (3, 1666), (4, 250), (5, 80)]
BEAM_SEEDS = 6
BEAM_OPTIONS = [(32, 100.0), (8, 20.0), (32, 0.0)]
FORWARD_CASES = [("fast", 2, 1200), ("hac", 2, 900), ("sup", 1, 1536)]
FORWARD_SAMPLES = 2048


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


def _text(a):
    return bytes(a).decode("ascii")


def scan_scores(state_len, T):
    return np.clip(synthetic_scores(1, T, state_len, seed=state_len, dtype=np.float32)[0], -5, 5)


def scan_rows(state_len, T):
    return np.unique(np.linspace(0, T, SCAN_ROWS[state_len]).astype(np.int64))


def beam_scores(state_len, T, seed):
    return np.clip(synthetic_scores(1, T, state_len, seed=50 + seed, scale=1.5)[0].astype(np.float32), -5, 5)


def beam_option_scores():
    return np.clip(synthetic_scores(1, 200, 3, seed=9, scale=1.0, dtype=np.float32)[0], -5, 5)


def cpu_decoder_scores():
    return synthetic_scores(6, 300, 3, seed=3, scale=1.5)


def forward_inputs(kind, N, T):
    from dorado_b200.config import load_model_config
    from dorado_b200.weights import synthetic_weights
    cfg = load_model_config(model_dir(kind))
    sig = np.random.default_rng(7).standard_normal((N, cfg.normalise_chunk_size(T))).astype(np.float32)
    return cfg, synthetic_weights(cfg, 42), sig


@pytest.mark.parametrize("state_len,T", SCAN_CASES)
def test_scans_match_reference(crf_oracle, golden, state_len, T):
    f, b, p = crf_oracle.scans(scan_scores(state_len, T))
    k = f"scans_sl{state_len}_T{T}"
    rows = scan_rows(state_len, T)
    rf, rb, rp = golden[f"{k}_fwd"], golden[f"{k}_bwd"], golden[f"{k}_posts"]
    tol = 4 * np.spacing(np.float32(golden[f"{k}_bwd_absmax"]))
    assert np.abs(f[rows] - rf).max() <= tol and np.abs(b[rows] - rb).max() <= tol
    assert np.abs(p[rows] - rp).max() <= 2e-3 * golden[f"{k}_posts_max"] + 1e-6  # softmax of values carrying that noise
    np.testing.assert_allclose(p.sum(axis=1), 1.0, rtol=1e-5)


@pytest.mark.parametrize("state_len,T", BEAM_CASES)
def test_beam_search_matches_reference_on_same_guides(crf_oracle, golden, state_len, T):
    """The reference is fed the fp16 scores widened to fp32, i.e. its CPU path (CPUDecoder hands beam_search_decode
    float tensors).  Its beam_search<c10::Half, float> instantiation is not a usable oracle: the beam-init threshold
    there memcpy()s the float back-guides into a vector<Half> (beam_search.cpp:168-171), so the initial beam is
    chosen from reinterpreted bytes."""
    mism = total = 0
    for seed in range(BEAM_SEEDS):
        s = beam_scores(state_len, T, seed)
        _, b, p = crf_oracle.scans(s)
        k = f"beam_sl{state_len}_T{T}_{seed}"
        rs, rq, rm = _text(golden[f"{k}_seq"]), _text(golden[f"{k}_qstr"]), golden[f"{k}_moves"]
        os_, oq, om = crf_oracle.beam_search(s, b, p, q_shift=-1.1, q_scale=1.1)
        assert rs == os_
        np.testing.assert_array_equal(rm, om)
        assert len(rq) == len(oq)
        mism += sum(a != c for a, c in zip(rq, oq))
        total += len(rq)
    # glibc's powf differs from the correctly rounded value on 0.06 % of its arguments; a character only moves when that
    # last ulp also crosses a quantiser edge, so at most an isolated character may differ
    assert mism <= 1, f"{mism}/{total} qstring characters differ from the reference"


@pytest.mark.parametrize("beam_width,beam_cut", BEAM_OPTIONS)
def test_beam_options_match_reference(crf_oracle, golden, beam_width, beam_cut):
    s = beam_option_scores()
    _, b, p = crf_oracle.scans(s)
    k = f"beamopt_w{beam_width}_c{beam_cut:g}"
    rs, rq, rm = _text(golden[f"{k}_seq"]), _text(golden[f"{k}_qstr"]), golden[f"{k}_moves"]
    os_, oq, om = crf_oracle.beam_search(s, b, p, beam_width=beam_width, beam_cut=beam_cut)
    assert rs == os_ and (rm == om).all()
    assert sum(a != c for a, c in zip(rq, oq)) <= 1


def test_full_decode_matches_reference_cpu_decoder(crf_oracle, golden):
    """CPUDecoder::beam_search_part_2 end to end (its own libtorch scans) vs the oracle: guides differ by a few
    ulp, so the bound is statistical: all move tables / sequences equal on these inputs, qstrings >= 98 %."""
    s16 = cpu_decoder_scores()
    r = DecodeResult(*(golden[f"cpu_decoder_{n}"] for n in ("seq", "qstr", "moves", "n_bases")))
    o = crf_oracle.decode(s16, clamp_val=5.0)
    same_seq = sum(a == b for a, b in zip(r.sequences, o.sequences))
    assert same_seq >= 5
    q_tot = q_bad = 0
    for a, b, sa, sb in zip(r.qstrings, o.qstrings, r.sequences, o.sequences):
        if sa == sb:
            q_tot += len(a)
            q_bad += sum(x != y for x, y in zip(a, b))
    assert q_bad <= 0.002 * q_tot + 1


@pytest.mark.parametrize("kind,N,T", FORWARD_CASES)
def test_forward_matches_reference(golden, kind, N, T):
    from oracle import nn_oracle
    cfg, w, sig = forward_inputs(kind, N, T)
    k = f"forward_{kind}"
    stride, outsize, state_len, _is_tx, clamp, _nf = (int(v) for v in golden[f"{k}_info"])
    qscale, qbias = (float(v) for v in golden[f"{k}_q"])
    assert stride == cfg.stride and outsize == cfg.outsize and state_len == cfg.state_len
    assert bool(clamp) == cfg.clamp and abs(qscale - cfg.qscale) < 1e-6 and abs(qbias - cfg.qbias) < 1e-6
    mine = nn_oracle.forward(cfg, w, sig, cpu_split_quirk=True)  # the CPU fallback's 12-way key slicing
    assert mine.shape == tuple(golden[f"{k}_shape"])
    idx = sample_index(mine.size, FORWARD_SAMPLES)
    ref = golden[f"{k}_values"]
    np.testing.assert_allclose(mine.reshape(-1)[idx], ref, rtol=0, atol=5e-5)
    if kind == "sup":
        # the true window differs from the CPU fallback only through the one dropped key per split
        true_win = nn_oracle.forward(cfg, w, sig, cpu_split_quirk=False)
        d = np.abs(true_win.reshape(-1)[idx] - ref)
        assert d.max() <= 2e-2 and (d > 1e-3).mean() <= 5e-3


@pytest.mark.parametrize("kind", ["fast", "hac"])
def test_reference_model_runner_reproduces_full_length_fixture(reference, kind):
    """dorado::basecall::ModelRunner (accept_chunk / call_chunks, ModelRunner.cpp:32-49) driven through the shim gives
    exactly the strings committed in tests/golden/full_<kind>.npz for the same chunk, and keeps its model_ms / decode_ms
    accounting (:51-57).  One chunk per call, as the fixture was generated: libtorch's fp32 kernels are not batch-invariant
    (a different GEMM blocking at batch 2 changes last bits of the scores, and these ill-conditioned synthetic models then
    flip a base), so only equal batch shapes are comparable bit for bit."""
    import pathlib
    from conftest import unpack_rows
    from dorado_b200.config import load_model_config
    from dorado_b200.weights import synthetic_weights
    from oracle.oracle import ReferenceRunner
    g = np.load(pathlib.Path(__file__).resolve().parent / "golden" / f"full_{kind}.npz")
    cfg = load_model_config(model_dir(kind))
    reference.set_num_threads(1)
    r = ReferenceRunner(reference, model_dir(kind), synthetic_weights(cfg, int(g["weights_seed"])), 1, 10000)
    assert r.chunk_size == int(g["T"]) and r.t_out == int(g["T_out"]) and r.batch_size == 1
    sig = np.random.default_rng(int(g["signal_seed"])).standard_normal((int(g["M"]), r.chunk_size)).astype(np.float16)
    nb = g["ref_n_bases"]
    seqs, qs = unpack_rows(g["ref_seq"], nb), unpack_rows(g["ref_qstr"], nb)
    mv = np.unpackbits(g["ref_moves"], axis=1)[:, : r.t_out]
    for i in (3, 0):
        r.accept_chunk(0, sig[i])
        out = r.call_chunks(1)
        assert out.sequences[0].encode() == seqs[i] and out.qstrings[0].encode() == qs[i]
        np.testing.assert_array_equal(out.moves[0], mv[i])
    st = r.sample_stats()
    assert st["batches_called"] == 2 and st["model_ms"] > 0 and st["decode_ms"] > 0
    r.close()
