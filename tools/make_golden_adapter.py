"""Generate tests/golden/adapter_<kind>.txt: the output of oracle/_ref/adapter_host (include/B200ModelRunner.h built
against the reference's headers by `make -C oracle ref`) on the inputs of tests/test_zz_adapter_gpu.py.

Needs a B200 and the built host:  python tools/make_golden_adapter.py [OUT_DIR]   (default tests/golden)
"""
import pathlib
import sys
import tempfile

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import test_zz_adapter_gpu as ta  # noqa: E402


def main():
    out_dir = pathlib.Path(sys.argv[1]) if len(sys.argv) > 1 else ROOT / "tests" / "golden"
    out_dir.mkdir(parents=True, exist_ok=True)
    for kind, batch, chunk, n in ta.CASES:
        with tempfile.TemporaryDirectory() as td:
            text = ta.run_adapter_host(td, kind, batch, chunk, n)
        (out_dir / f"adapter_{kind}.txt").write_text(text)
        print(f"adapter_{kind}.txt: {len(text.splitlines())} lines")


if __name__ == "__main__":
    main()
