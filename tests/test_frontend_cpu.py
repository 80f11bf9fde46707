"""Front end of the hot path (SURVEY.md 8f rows 2-3) on the CPU: the product's host logic (generate_chunks,
stitch_chunks through the C ABI) and the numpy oracle of the device-side scaling, both pinned to
  * the golden vectors of the reference's own tests (tests/ChunkTest.cpp, tests/StitchTest.cpp), restated below,
  * the compiled reference (chunk.cpp, stitch.cpp, tensor_utils.cpp) on seeded random inputs, whose outputs
    tools/make_golden_reference.py records as digests in tests/golden/reference_cpu.npz (the *_cases functions below
    generate the inputs for both),
  * the committed fixture tests/golden/frontend.npz (generated from the compiled reference).
"""
import numpy as np
import pytest

from conftest import ROOT
from dorado_b200 import lib as L
from dorado_b200.frontend import generate_chunks, stitch_chunks
from oracle import frontend_oracle as fo
from oracle.golden import digest


@pytest.fixture(scope="module")
def golden():
    return np.load(ROOT / "tests" / "golden" / "reference_cpu.npz")


# ---- generate_chunks -------------------------------------------------------------------------------------------
def test_generate_chunks_invalid_input_like_ChunkTest():
    # tests/ChunkTest.cpp "Invalid input": every one of these throws in the reference
    for args in [(0, 9996, 6, 498), (12345, 0, 6, 498), (12345, 9996, 0, 498), (12345, 9996, 10, 498),
                 (12345, 9996, 7, 498), (12345, 9996, 6, 9996), (12345, 9996, 6, 9997)]:
        with pytest.raises(L.B200Error) as e:
            generate_chunks(*args)
        assert e.value.status == L.B200_ERR_INVALID
        with pytest.raises((RuntimeError, ValueError)):
            fo.generate_chunks(*args)


def test_generate_chunks_golden_vectors_of_ChunkTest():
    golden = [((9996 // 2, 9996, 6, 498), [0]), ((9996, 9996, 6, 498), [0]), ((9996 + 1, 9996, 6, 498), [0, 6]),
              ((9996 + 9996 // 2, 9996, 6, 498), [0, 4998]), ((2 * 9996 + 9996 // 2, 9996, 1, 0), [0, 9996, 14994]),
              ((3 * 9996, 9996, 6, 498), [0, 9498, 18996, 19992])]
    for args, want in golden:
        assert generate_chunks(*args) == want
        assert fo.generate_chunks(*args) == want


@pytest.mark.parametrize("chunk_size,stride,overlap", [(9996, 6, 498), (9996, 7, 497), (9996, 12, 492), (9996, 17, 510),
                                                       (555, 5, 25), (83, 1, 13), (123, 1, 0)])
def test_generate_chunks_properties_of_ChunkTest(chunk_size, stride, overlap):
    rng = np.random.default_rng(42)
    for num_samples in rng.integers(1024, 2097152, 16):
        offs = generate_chunks(int(num_samples), chunk_size, stride, overlap)
        assert offs and offs[0] == 0
        for i in range(1, len(offs) - 1):
            assert offs[i] % stride == 0 and offs[i] == i * (chunk_size - overlap)
        assert offs[-1] % stride == 0 and offs[-1] < num_samples
        if len(offs) > 1:
            assert chunk_size - stride <= num_samples - offs[-1] <= chunk_size
        assert offs == fo.generate_chunks(int(num_samples), chunk_size, stride, overlap)


def generate_chunks_cases():
    rng = np.random.default_rng(7)
    for _ in range(300):
        stride = int(rng.choice([1, 5, 6, 12]))
        chunk = stride * int(rng.integers(2, 400))
        overlap = stride * int(rng.integers(0, chunk // stride))
        n = int(rng.integers(1, 40 * chunk))
        yield n, chunk, stride, overlap


def test_generate_chunks_matches_compiled_reference(golden):
    want = golden["generate_chunks"]
    cases = list(generate_chunks_cases())
    assert len(cases) == len(want)
    for args, w in zip(cases, want):
        got = generate_chunks(*args)
        assert (digest(np.array(got, np.uint64)) == w).all(), args
        assert fo.generate_chunks(*args) == got
    assert golden["generate_chunks_zero_raises"]   # the reference throws on an empty read; so must the product
    with pytest.raises(L.B200Error):
        generate_chunks(0, 9996, 6, 498)


def test_generate_chunks_capacity_reports_full_count():
    import ctypes as C
    lib = L.load_library()
    n = C.c_uint64()
    buf = (C.c_uint64 * 2)()
    L.check(lib.b200_generate_chunks(3 * 9996, 9996, 6, 498, buf, 2, C.byref(n)))
    assert n.value == 4 and list(buf) == [0, 9498]
    L.check(lib.b200_generate_chunks(3 * 9996, 9996, 6, 498, None, 0, C.byref(n)))
    assert n.value == 4


# ---- stitch_chunks ---------------------------------------------------------------------------------------------
STITCH_MOVES = [[1, 0, 0, 1, 0, 0, 1, 0, 1, 0], [1, 0, 0, 1, 0, 0, 0, 1, 0, 1], [1, 0, 0, 1, 0, 1, 1, 0, 0, 0],
                [1, 0, 0, 1, 0, 0, 1, 0, 1, 0], [0, 1, 0, 1, 0, 0, 1, 0, 1, 0], [1, 0, 0, 0, 0, 0, 1, 0, 1, 1],
                [1, 0, 0, 1, 0, 0, 1, 0, 1, 0]]


def _stitch_test_chunks():
    # tests/StitchTest.cpp: RAW_SIGNAL_SIZE 50, CHUNK_SIZE 10, OVERLAP 3, seven chunks "ACGT" / "!&.-"
    offs, off = [0], 0
    while off + 10 < 50:
        off = min(off + 7, 40)
        offs.append(off)
    return [(o, 10, np.array(STITCH_MOVES[i], np.uint8), "ACGT", "!&.-") for i, o in enumerate(offs)]


def test_stitch_chunks_golden_vector_of_StitchTest():
    want_seq, want_q = "ACGTCGCGTCGTCGTCCGT", "!&.-&.&.-&.-&.-&&.-"
    want_moves = [1, 0, 0, 1, 0, 0, 1, 0, 1, 0, 1, 0, 0, 0, 1, 0, 0, 1, 0, 1, 1, 0, 0, 0, 1, 0, 0, 1, 0, 1, 0, 1, 0, 0,
                  1, 0, 1, 0, 0, 0, 0, 1, 0, 1, 0, 0, 1, 0, 1]
    # the reference test leaves raw_data empty (0 samples), which also exercises the overhang pop
    for impl in (stitch_chunks, fo.stitch_chunks):
        seq, q, moves = impl(_stitch_test_chunks(), 0, 1)
        assert seq == want_seq and q == want_q and moves.tolist() == want_moves


def _random_called_read(rng, n_samples, chunk, stride, overlap):
    chunks = []
    for off in fo.generate_chunks(n_samples, chunk, stride, overlap):
        moves = (rng.random(chunk // stride) < 0.45).astype(np.uint8)
        moves[0] = 1  # beam_search.cpp:447-455
        nb = int(moves.sum())
        seq = "".join(rng.choice(list("ACGT"), nb))
        q = "".join(chr(33 + int(v)) for v in rng.integers(1, 50, nb))
        chunks.append((off, chunk, moves, seq, q))
    return chunks


def stitch_cases():
    rng = np.random.default_rng(11)
    for _ in range(200):
        stride = int(rng.choice([1, 5, 6]))
        chunk = stride * int(rng.integers(8, 120))
        overlap = stride * int(rng.integers(0, max(1, chunk // stride // 2)))
        n = int(rng.integers(1, 12 * chunk))
        yield n, chunk, stride, overlap, _random_called_read(rng, n, chunk, stride, overlap)


def stitch_digest(seq, q, moves):
    return digest(seq, q, np.asarray(moves, np.uint8))


def test_stitch_chunks_matches_compiled_reference(golden):
    want = golden["stitch_chunks"]
    cases = list(stitch_cases())
    assert len(cases) == len(want)
    for it, ((n, chunk, stride, overlap, chunks), w) in enumerate(zip(cases, want)):
        for impl in (stitch_chunks, fo.stitch_chunks):
            seq, q, moves = impl(chunks, n, stride)
            assert (stitch_digest(seq, q, moves) == w).all(), (it, n, chunk, stride, overlap)
        assert len(moves) == n // stride or len(chunks) > 1
        assert int(moves.sum()) == len(seq)


def test_stitch_chunks_rejects_bad_input():
    with pytest.raises(L.B200Error):
        stitch_chunks([], 100, 6)
    a = (0, 60, np.ones(10, np.uint8), "A" * 10, "!" * 10)
    b = (120, 60, np.ones(10, np.uint8), "A" * 10, "!" * 10)  # gap instead of an overlap
    with pytest.raises(L.B200Error):
        stitch_chunks([a, b], 180, 6)
    c = (57, 60, np.ones(10, np.uint8), "A" * 10, "!" * 10)   # overlap not on a stride boundary
    with pytest.raises(L.B200Error):
        stitch_chunks([a, c], 117, 6)
    with pytest.raises(L.B200Error):
        stitch_chunks([a], 60, 0)


# ---- raw int16 -> scaled, repeat-padded fp16 rows (numpy oracle of the device kernel) -----------------------------
def scaling_cases():
    # tests/TensorUtilsTest.cpp:121-143: random sizes < 100, shift in [-100, 100], scale in [0.1, 100], zero tolerance
    rng = np.random.default_rng(42)
    for _ in range(40):
        n = int(rng.integers(1, 100))
        shift, scale = float(rng.uniform(-100, 100)), float(rng.uniform(0.1, 100))
        yield (rng.random(n) * 1000).astype(np.int16), shift, scale


def test_scaling_oracle_like_TensorUtilsTest(golden):
    want = golden["scaling"]
    cases = list(scaling_cases())
    assert len(cases) == len(want)
    for (raw, shift, scale), w in zip(cases, want):
        got = fo.scale_i16_to_f16(raw, np.float32(shift), np.float32(scale))
        assert (digest(got.view(np.uint16)) == w).all()


def chunk_input_cases():
    rng = np.random.default_rng(5)
    for _ in range(60):
        chunk = 6 * int(rng.integers(2, 300))
        n = int(rng.integers(1, 6 * chunk))
        raw = rng.integers(-32768, 32768, n).astype(np.int16)
        shift, scale = float(rng.uniform(-500, 900)), float(rng.uniform(0.5, 400))
        yield raw, fo.generate_chunks(n, chunk, 6, 6 * int(rng.integers(0, chunk // 12 + 1))), chunk, shift, scale


def test_chunk_input_oracle_matches_compiled_reference(golden):
    want = golden["chunk_input"]
    cases = list(chunk_input_cases())
    assert len(cases) == len(want)
    for (raw, offs, chunk, shift, scale), w in zip(cases, want):
        rows = [fo.chunk_input(raw, off, chunk, shift, scale).view(np.uint16) for off in offs]
        assert (digest(*rows) == w).all()


def test_frontend_golden_fixture_matches_oracle():
    g = np.load(ROOT / "tests" / "golden" / "frontend.npz")
    chunk, stride, overlap = int(g["chunk_size"]), int(g["stride"]), int(g["overlap"])
    row = 0
    for r, n in enumerate(g["read_lens"]):
        raw = g[f"raw_{r}"]
        shift, scale = g[f"shift_scale_{r}"]
        offs = generate_chunks(int(n), chunk, stride, overlap)
        assert offs == g[f"offsets_{r}"].tolist() == fo.generate_chunks(int(n), chunk, stride, overlap)
        for o in offs:
            assert g["row_read_offset"][row].tolist() == [r, o]
            got = fo.chunk_input(raw, o, chunk, shift, scale)
            assert (got.view(np.uint16) == g["input_rows_f16_bits"][row]).all()
            row += 1
    assert row == g["input_rows_f16_bits"].shape[0]


# ---- batch-size selection rule (CudaCaller::determine_batch_dims, CudaCaller.cpp:487-631) -----------------------------
def _select_like_reference(table, max_size, granularity, penalty):
    """Restatement of the reference's loop: `times_and_batch_sizes` keeps entries that improve on best_time (:585-589),
    the first entry under best * (1 + penalty) bounds the search (:604-607), the last kept batch size <= max_size up to it
    wins (:619-631), starting from the granularity (:405)."""
    best, kept = float("inf"), []
    for bs, t in table:
        if t < best:
            best = t
            kept.append((t, bs))
    thr = np.float32(best) * (np.float32(1) + np.float32(penalty))
    idx = next(i for i, (t, _) in enumerate(kept) if np.float32(t) <= thr)
    final = granularity
    for t, bs in kept[: idx + 1]:
        if bs <= max_size:
            final = bs
    return final


def test_select_batch_size_matches_reference_rule():
    from dorado_b200.batching import select_batch_size
    t = [(64, 1.0), (128, 0.6), (192, 0.65), (256, 0.5), (320, 0.49), (384, 0.495)]
    assert select_batch_size(t, 10240, 64, 0.0) == 320          # the best time itself
    assert select_batch_size(t, 10240, 64, 0.05) == 256         # first entry within 5 % of the best
    assert select_batch_size(t, 200, 64, 0.0) == 128            # memory cap
    assert select_batch_size(t, 32, 64, 0.0) == 64              # nothing fits: the granularity
    rng = np.random.default_rng(3)
    for _ in range(300):
        n = int(rng.integers(1, 40))
        g = int(rng.choice([16, 32, 64]))
        table = [(g * (i + 1), float(np.float32(rng.uniform(0.05, 2.0) / (1 + 0.1 * i)))) for i in range(n)]
        cap = int(rng.integers(1, g * (n + 2)))
        pen = float(rng.choice([0.0, 0.05, 0.1, 0.5]))
        assert select_batch_size(table, cap, g, pen) == _select_like_reference(table, cap, g, pen)


def test_select_batch_size_rejects_bad_tables():
    from dorado_b200.batching import select_batch_size
    with pytest.raises(L.B200Error):
        select_batch_size([], 512, 64, 0.0)
    with pytest.raises(L.B200Error):
        select_batch_size([(128, 1.0), (64, 0.5)], 512, 64, 0.0)   # not ascending
    with pytest.raises(L.B200Error):
        select_batch_size([(64, 1.0)], 512, 64, -0.1)


# ---- generate_variable_chunks (first piece of SURVEY 8f row 1) -------------------------------------------------------
VARIABLE_CHUNKS_INVALID = [(0, 9996, 6, 498), (12345, 0, 6, 498), (12345, 9996, 0, 498), (12345, 9996, 10, 498),
                           (12345, 6, 6, 498), (12345, 9996, 7, 498), (12345, 9996, 7, 0), (12345, 9996, 6, 9996),
                           (12345, 9996, 6, 9997)]
VARIABLE_CHUNKS_GOLDEN = [((9996 // 2, 9996, 6, 498), [(0, 4998)]), ((9996, 9996, 6, 498), [(0, 9996)]),
                          ((9996 + 1, 9996, 6, 498), [(0, 5244), (4752, 9997)]),
                          ((9996 + 9996 // 2, 9996, 6, 498), [(0, 7746), (7248, 14994)]),
                          ((2 * 9996 + 9996 // 2, 9996, 1, 0), [(0, 8330), (8330, 16660), (16660, 24990)]),
                          ((3 * 9996, 9996, 6, 498), [(0, 7866), (7374, 15240), (14748, 22614), (22122, 29988)])]


def variable_chunks_cases():
    rng = np.random.default_rng(42)
    for chunk_size, stride, overlap in [(9996, 6, 498), (9996, 7, 497), (9996, 12, 492), (9996, 17, 510), (555, 5, 25),
                                        (83, 1, 13), (123, 1, 0)]:
        for n in rng.integers(1024, 2097152, 16):
            yield int(n), chunk_size, stride, overlap


def intervals_digest(iv):
    return digest(np.array(iv, np.uint64).reshape(-1, 2))


def test_generate_variable_chunks_like_ChunkTest(golden):
    from dorado_b200.frontend import generate_variable_chunks
    assert golden["variable_chunks_invalid_raises"].all()   # the reference throws on every one of these
    for args in VARIABLE_CHUNKS_INVALID:
        with pytest.raises(L.B200Error):
            generate_variable_chunks(*args)
    assert len(golden["variable_chunks_golden"]) == len(VARIABLE_CHUNKS_GOLDEN)
    for (args, want), w in zip(VARIABLE_CHUNKS_GOLDEN, golden["variable_chunks_golden"]):
        assert generate_variable_chunks(*args) == want == fo.generate_variable_chunks(*args)
        assert (intervals_digest(want) == w).all()
    want = golden["variable_chunks"]
    cases = list(variable_chunks_cases())
    assert len(cases) == len(want)
    for (n, chunk_size, stride, overlap), w in zip(cases, want):
        iv = generate_variable_chunks(n, chunk_size, stride, overlap)
        assert (intervals_digest(iv) == w).all(), (n, chunk_size, stride, overlap)
        assert iv == fo.generate_variable_chunks(n, chunk_size, stride, overlap)
        assert iv[0][0] == 0 and iv[-1][1] == n
        assert all(a % stride == 0 for a, _ in iv[1:]) and all(b % stride == 0 for _, b in iv[:-1])
        assert all(0 < b - a <= chunk_size for a, b in iv)
        assert all(iv[i - 1][1] - iv[i][0] <= overlap for i in range(1, len(iv)))


def test_batch_size_granularity_like_the_reference():
    from conftest import model_dir
    from dorado_b200.batching import batch_size_granularity
    from dorado_b200.config import load_model_config
    assert batch_size_granularity(load_model_config(model_dir("fast"))) == 64   # CudaCaller.h:60-63
    assert batch_size_granularity(load_model_config(model_dir("hac"))) == 64
    assert batch_size_granularity(load_model_config(model_dir("sup"))) == 32
