"""Generate tests/golden/reference_cpu.npz: the outputs of the reference's own CPU code (oracle/_ref/libdorado_ref.so,
the unmodified reference sources built by oracle/Makefile) on the inputs of tests/test_oracle_vs_reference.py and
tests/test_frontend_cpu.py.  The inputs come from those test modules' case functions, so the tests regenerate exactly
what was recorded.  Exact outputs too large to store whole are recorded as digests (oracle/golden.py).

Run where the reference tree is available:  make -C oracle ref && python tools/make_golden_reference.py
"""
import pathlib
import sys
import tempfile

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import test_frontend_cpu as tf  # noqa: E402
import test_oracle_vs_reference as tr  # noqa: E402
from conftest import model_dir  # noqa: E402
from dorado_b200.weights import save_b2w  # noqa: E402
from oracle.golden import digest, sample_index  # noqa: E402
from oracle.oracle import CrfOracle, Reference  # noqa: E402

OUT = ROOT / "tests" / "golden" / "reference_cpu.npz"


def _raises(fn, *args):
    try:
        fn(*args)
    except RuntimeError:
        return True
    return False


def frontend(ref, out):
    out["generate_chunks"] = np.stack([digest(np.array(ref.generate_chunks(*a), np.uint64))
                                       for a in tf.generate_chunks_cases()])
    out["generate_chunks_zero_raises"] = _raises(ref.generate_chunks, 0, 9996, 6, 498)
    out["stitch_chunks"] = np.stack([tf.stitch_digest(*ref.stitch_chunks(chunks, n, stride))
                                     for n, _, stride, _, chunks in tf.stitch_cases()])
    out["scaling"] = np.stack([digest(ref.make_chunk_input(raw, 0, raw.size, shift, scale).view(np.uint16))
                               for raw, shift, scale in tf.scaling_cases()])
    out["chunk_input"] = np.stack([digest(*[ref.make_chunk_input(raw, off, chunk, shift, scale).view(np.uint16) for off in offs])
                                   for raw, offs, chunk, shift, scale in tf.chunk_input_cases()])
    out["variable_chunks_invalid_raises"] = np.array([_raises(ref.generate_variable_chunks, *a)
                                                      for a in tf.VARIABLE_CHUNKS_INVALID])
    out["variable_chunks_golden"] = np.stack([tf.intervals_digest(ref.generate_variable_chunks(*a))
                                              for a, _ in tf.VARIABLE_CHUNKS_GOLDEN])
    out["variable_chunks"] = np.stack([tf.intervals_digest(ref.generate_variable_chunks(*a))
                                       for a in tf.variable_chunks_cases()])


def decoder(ref, orc, out):
    for sl, T in tr.SCAN_CASES:
        f, b, p = ref.scans(tr.scan_scores(sl, T))
        k, rows = f"scans_sl{sl}_T{T}", tr.scan_rows(sl, T)
        out[f"{k}_fwd"], out[f"{k}_bwd"], out[f"{k}_posts"] = f[rows], b[rows], p[rows]
        out[f"{k}_bwd_absmax"], out[f"{k}_posts_max"] = np.abs(b).max(), p.max()
    for sl, T in tr.BEAM_CASES:
        for seed in range(tr.BEAM_SEEDS):
            s = tr.beam_scores(sl, T, seed)
            _, b, p = orc.scans(s)      # the reference is fed the oracle's guides
            seq, qstr, moves = ref.beam_search_decode(s, b, p, q_shift=-1.1, q_scale=1.1)
            k = f"beam_sl{sl}_T{T}_{seed}"
            out[f"{k}_seq"], out[f"{k}_qstr"], out[f"{k}_moves"] = np.frombuffer(seq.encode(), np.uint8), \
                np.frombuffer(qstr.encode(), np.uint8), moves
    s = tr.beam_option_scores()
    _, b, p = orc.scans(s)
    for w, c in tr.BEAM_OPTIONS:
        seq, qstr, moves = ref.beam_search_decode(s, b, p, beam_width=w, beam_cut=c)
        k = f"beamopt_w{w}_c{c:g}"
        out[f"{k}_seq"], out[f"{k}_qstr"], out[f"{k}_moves"] = np.frombuffer(seq.encode(), np.uint8), \
            np.frombuffer(qstr.encode(), np.uint8), moves
    r = ref.decode(np.clip(tr.cpu_decoder_scores().astype(np.float32), -5, 5))
    out["cpu_decoder_seq"], out["cpu_decoder_qstr"], out["cpu_decoder_moves"], out["cpu_decoder_n_bases"] = \
        r.seq_buf, r.qstr_buf, r.moves, r.n_bases


def forward(ref, out):
    for kind, N, T in tr.FORWARD_CASES:
        cfg, w, sig = tr.forward_inputs(kind, N, T)
        with tempfile.TemporaryDirectory() as td:
            save_b2w(f"{td}/w.b2w", w)
            h = ref.load_model(model_dir(kind), f"{td}/w.b2w")
        info = ref.model_info(h)
        scores = ref.forward(h, sig)
        ref.free_model(h)
        k = f"forward_{kind}"
        out[f"{k}_info"] = np.array([info[n] for n in ("stride", "outsize", "state_len", "is_tx", "clamp", "num_features")],
                                    np.int32)
        out[f"{k}_q"] = np.array([info["qscale"], info["qbias"]], np.float32)
        out[f"{k}_shape"] = np.array(scores.shape, np.int64)
        out[f"{k}_values"] = scores.reshape(-1)[sample_index(scores.size, tr.FORWARD_SAMPLES)]


def main():
    ref, orc = Reference(), CrfOracle()
    out = {}
    frontend(ref, out)
    decoder(ref, orc, out)
    forward(ref, out)
    np.savez_compressed(OUT, **out)
    print(f"{OUT.relative_to(ROOT)}: {len(out)} arrays, {OUT.stat().st_size} bytes")


if __name__ == "__main__":
    main()
