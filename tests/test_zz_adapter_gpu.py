"""The reference-side binding EXECUTED: oracle/_ref/adapter_host is include/B200ModelRunner.h compiled against the reference's
own headers (ModelRunnerBase, BasecallModelConfig, crf_utils) and libtorch (oracle/Makefile, built where the reference tree
is available).  It drives the engine only through dorado::basecall::ModelRunnerBase -- accept_chunk(at::Tensor),
call_chunks(), sample_stats(), terminate()/restart() -- and must return exactly what the ctypes path returns for the same
chunks.  The test runs the host whenever it is built and holds its output, header lines included, to the ctypes path.
Its output on a B200 for these inputs is also recorded in tests/golden/adapter_<kind>.txt by tools/make_golden_adapter.py;
the ctypes path is held to that recording in every case, so a checkout without the reference tree still pins the chunks
the adapter returned."""
import pathlib
import subprocess

import numpy as np
import pytest

from conftest import model_dir

pytestmark = pytest.mark.gpu
ROOT = pathlib.Path(__file__).resolve().parents[1]
HOST = ROOT / "oracle" / "_ref" / "adapter_host"
CASES = [("fast", 16, 1200, 40), ("sup", 4, 1536, 6)]


def adapter_inputs(kind, chunk, n):
    from dorado_b200.config import load_model_config
    from dorado_b200.weights import synthetic_weights
    cfg = load_model_config(model_dir(kind))
    sig = np.random.default_rng(11).standard_normal((n, cfg.normalise_chunk_size(chunk))).astype(np.float16)
    return cfg, synthetic_weights(cfg, 42), sig


def run_adapter_host(work, kind, batch, chunk, n) -> str:
    """Run oracle/_ref/adapter_host on the inputs of one case in the directory `work`; returns its output text."""
    from dorado_b200.weights import save_b2w
    _, w, sig = adapter_inputs(kind, chunk, n)
    work = pathlib.Path(work)
    save_b2w(work / "w.b2w", w)
    sig.tofile(work / "sig.f16")
    out = work / "out.txt"
    r = subprocess.run([str(HOST), str(model_dir(kind)), str(work / "w.b2w"), str(work / "work"), str(batch), str(chunk),
                        str(work / "sig.f16"), str(n), str(out)], capture_output=True, text=True, timeout=600)
    if r.returncode != 0:
        raise RuntimeError(r.stderr[-2000:])
    return out.read_text()


def ctypes_chunks(cfg, w, sig, batch, chunk):
    """The same chunks through the Python ctypes path: [(sequence, qstring, moves as a 0/1 string), ...]."""
    from dorado_b200.runner import B200Caller, B200ModelRunner
    runner = B200ModelRunner(B200Caller(cfg, w), batch, chunk)
    out = []
    for start in range(0, len(sig), batch):
        cnt = min(batch, len(sig) - start)
        for i in range(cnt):
            runner.accept_chunk(i, sig[start + i])
        out += [[c.sequence, c.qstring, "".join("1" if m else "0" for m in c.moves)] for c in runner.call_chunks(cnt)]
    return out


@pytest.mark.parametrize("kind,batch,chunk,n", CASES)
def test_cpp_adapter_matches_ctypes_path(tmp_path, kind, batch, chunk, n):
    cfg, w, sig = adapter_inputs(kind, chunk, n)
    T = cfg.normalise_chunk_size(chunk)
    want = ctypes_chunks(cfg, w, sig, batch, chunk)
    assert len(want) == n
    recorded = (ROOT / "tests" / "golden" / f"adapter_{kind}.txt").read_text().splitlines()
    # the recorded run pins the engine's output for these chunks whether or not the host is built here
    assert [l.split()[1:] for l in recorded if l.startswith("chunk")] == want
    if not HOST.exists():
        return   # the host needs the reference tree to build (`make -C oracle ref`); the recorded run stands in for it
    lines = run_adapter_host(tmp_path, kind, batch, chunk, n).splitlines()
    head = {l.split()[0]: l.split()[1:] for l in lines if not l.startswith("chunk")}
    assert head["name"][0].startswith("B200ModelRunner_0_")
    assert [int(x) for x in head["dims"]] == [batch, T, cfg.stride]
    assert head["timeouts"][:2] == ["300000", "30000"] and head["timeouts"][3] == "0"
    assert head["stats"][0] == "batches_called" and float(head["stats"][1]) == (n + batch - 1) // batch
    assert float(head["stats"][3]) > 0                      # model_decode_ms
    assert head["terminate_refuses"] == ["1", "restart_ok", "1"]
    assert [l.split()[1:] for l in lines if l.startswith("chunk")] == want
