"""CPU-only checks of the host side: C ABI symbols, loud failure without a GPU, config parsing, weight container,
the numerics contract, and the multi-process sharding helpers (gloo, world_size 2)."""
import ctypes as C
import math
import os
import pathlib
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import MODELS, ROOT, model_dir


def test_library_exports_every_declared_symbol():
    from dorado_b200 import lib as L
    header = (ROOT / "include" / "b200call.h").read_text()
    declared = set(re.findall(r"B200_API\s+[\w\s\*]+?\b(b200_\w+)\s*\(", header))
    assert declared, "no B200_API declarations parsed"
    lib = L.load_library()
    for name in sorted(declared):
        assert hasattr(lib, name), f"libb200call.so does not export {name}"
    assert set(L.EXPORTS) == declared
    assert b"sm_100a" in lib.b200_version()


def test_fails_loudly_without_a_gpu():
    from dorado_b200 import lib as L
    lib = L.load_library()
    if lib.b200_device_count() > 0:
        pytest.skip("a CUDA device is visible")
    with pytest.raises(L.B200Error) as e:
        L.decode_scores(np.zeros((1, 4, 256), np.float16))
    assert e.value.status == L.B200_ERR_CUDA and "no CPU fallback" in str(e.value)
    from dorado_b200.config import load_model_config
    from dorado_b200.runner import B200Caller
    from dorado_b200.weights import synthetic_weights
    cfg = load_model_config(model_dir("fast"))
    with pytest.raises(L.B200Error) as e:
        B200Caller(cfg, synthetic_weights(cfg, 1))
    assert e.value.status == L.B200_ERR_CUDA


def test_null_arguments_return_invalid():
    from dorado_b200 import lib as L
    lib = L.load_library()
    assert lib.b200_engine_create(None, None, 0, 0, None) == L.B200_ERR_INVALID
    assert b"null" in lib.b200_last_error()
    assert lib.b200_runner_batch_size(None) == 0


def test_model_configs_parse_like_the_reference():
    """Expected values follow dorado/config/BasecallModelConfig.cpp (and its tests/BasecallModelConfigTest.cpp)."""
    from dorado_b200.config import ACT_SWISH, ACT_TANH, load_model_config
    fast, hac, sup = (load_model_config(model_dir(k)) for k in ("fast", "hac", "sup"))
    assert (fast.stride, fast.lstm_size, fast.lstm_layers, fast.state_len, fast.outsize) == (6, 96, 5, 3, 256)
    assert (hac.stride, hac.lstm_size, hac.state_len, hac.outsize, hac.clamp) == (6, 384, 4, 1024, True)
    assert [c.activation for c in hac.convs] == [ACT_SWISH, ACT_SWISH, ACT_TANH]
    assert hac.bias is False and hac.out_features is None
    assert (hac.qscale, hac.qbias) == (1.1, -1.1)
    assert sup.is_tx_model and sup.stride == 6 and sup.stride_inner() == 12 and sup.outsize == 4096
    assert sup.tx.attn_window == (127, 128) and sup.tx.depth == 18 and abs(sup.tx.deepnorm_alpha - 2.4494897) < 1e-6
    assert sup.chunk_size_granularity() == 192 and sup.normalise_chunk_size(10000) == 9984
    assert fast.normalise_chunk_size(10000) == 9996 and fast.out_len(9996) == 1666


def test_weight_names_follow_reference_file_list(tmp_path):
    from dorado_b200.config import load_model_config
    from dorado_b200.weights import load_b2w, save_b2w, synthetic_weights, tensor_specs
    hac = load_model_config(model_dir("hac"))
    names = list(tensor_specs(hac))
    # dorado/basecall/crf_utils.cpp:34-95
    assert names[:2] == ["0.conv.weight.tensor", "0.conv.bias.tensor"]
    assert "4.rnn.weight_ih_l0.tensor" in names and "8.rnn.bias_hh_l0.tensor" in names
    assert names[-1] == "9.linear.weight.tensor"
    sup = load_model_config(model_dir("sup"))
    sn = list(tensor_specs(sup))
    assert sn[10] == "transformer_encoder.0.self_attn.Wqkv.weight.tensor" and sn[-1] == "crf.linear.weight.tensor"
    assert len(sn) == 10 + 18 * 7 + 3
    w = synthetic_weights(hac, 3)
    save_b2w(tmp_path / "w.b2w", w)
    back = load_b2w(tmp_path / "w.b2w")
    assert list(back) == list(w) and all(np.array_equal(back[k], w[k]) for k in w)
    assert not np.any(w["4.rnn.bias_hh_l0.tensor"])


def test_numerics_contract_accuracy(crf_oracle):
    lib = crf_oracle.lib
    xs = np.concatenate([-np.logspace(-6, 1.9, 4000), [0.0]]).astype(np.float32)
    got = np.array([lib.crf_math_expf(float(x)) for x in xs], np.float32)
    ref = np.exp(xs.astype(np.float64))
    assert np.max(np.abs(got - ref) / np.maximum(ref, 1e-37)) < 3e-7
    ys = np.logspace(-6, 3, 4000).astype(np.float32)
    gl = np.array([lib.crf_math_logf(float(y)) for y in ys], np.float32)
    rl = np.log(ys.astype(np.float64))
    assert np.max(np.abs(gl - rl) / np.maximum(np.abs(rl), 1e-3)) < 3e-7
    ps = np.linspace(0, 1, 1001).astype(np.float32)
    gp = np.array([lib.crf_math_pow0p4f(float(p)) for p in ps], np.float32)
    assert np.max(np.abs(gp - ps.astype(np.float64) ** 0.4)) < 2e-7
    assert lib.crf_math_lse2(1.0, 1.0) == pytest.approx(1.0 + math.log(2.0), rel=2e-7)
    assert lib.crf_math_lse2(30.0, 1.0) == 30.0  # 17.0 cut-off of beam_search.cpp:44
    halfs = np.arange(0, 65536, 7, dtype=np.uint16)
    halfs = halfs[~np.isnan(halfs.view(np.float16))]  # NaN payload quieting is implementation-defined
    conv = np.array([lib.crf_half_to_float(int(h)) for h in halfs], np.float32)
    np.testing.assert_array_equal(conv.view(np.uint32), halfs.view(np.float16).astype(np.float32).view(np.uint32))


def test_expf_variants_are_bit_identical(crf_oracle):
    """b200_expf_nonpos (what the max-shifted sums of the scans call: no upper clamp) equals b200_expf bit for bit on every
    sampled x <= 0 (all of [-0, -inf) in steps of 4099 bit patterns, plus a dense window around the -86 cut-off), and the
    integer form of the 2^n scale equals the float -> int conversion it replaced."""
    import ctypes as C
    lib = crf_oracle.lib
    lib.crf_expf_audit.restype = C.c_long
    lib.crf_expf_audit.argtypes = [C.c_uint32, C.c_uint32, C.c_long, C.POINTER(C.c_long)]
    sb = C.c_long()
    n = (0xff800000 - 0x80000000) // 4099 + 1
    assert lib.crf_expf_audit(0x80000000, 4099, n, C.byref(sb)) == 0 and sb.value == 0
    cut = int(np.float32(-86.0).view(np.uint32))
    assert lib.crf_expf_audit(cut - 200000, 1, 400000, C.byref(sb)) == 0 and sb.value == 0
    assert lib.crf_math_expf_nonpos(0.0) == 1.0 and lib.crf_math_expf_nonpos(-87.0) == 0.0


def test_pow0p4_against_libm(crf_oracle):
    """The contract's pow(p, 0.4f) (binary64 exp(0.4f * log p), one rounding) is the correctly rounded powf on every
    sampled argument; the host libm's powf is within 1 ulp of it and differs on < 0.2 % of the arguments."""
    import ctypes as C
    n, a, b, m = C.c_long(), C.c_long(), C.c_long(), C.c_long()
    crf_oracle.lib.crf_pow0p4_audit(C.c_uint32(61), C.byref(n), C.byref(a), C.byref(b), C.byref(m))
    assert n.value > 5_000_000
    assert b.value == 0, f"{b.value} of {n.value} differ from the correctly rounded powf"
    assert m.value <= 1 and a.value <= 2e-3 * n.value, (a.value, m.value)
    lib = crf_oracle.lib
    assert lib.crf_math_pow0p4f(0.0) == 0.0 and lib.crf_math_pow0p4f(1.0) == 1.0 and lib.crf_math_pow0p4f(-0.0) == 0.0
    tiny = float(np.float32(1e-42))  # subnormal argument: handled exactly
    assert lib.crf_math_pow0p4f(tiny) == pytest.approx(tiny ** float(np.float32(0.4)), rel=1e-6)


@pytest.mark.parametrize("scale,shift", [(1.0, 0.0), (0.97, -0.05), (1.04, 0.4), (0.9, -0.2), (0.5, 3.0), (1.1, -1.1)])
def test_quality_character_quantiser_is_exact(crf_oracle, scale, shift):
    """b200_qtable (bin edges bisected on the host libm) reproduces the reference expression
    char(33.5 + clamp(-10 log10(err) * scale + shift, 1, 50)) on every 29th float of (0, 1] and on +-4096 ulp around
    every edge -- the engine's traceback kernel looks characters up in this table."""
    import ctypes as C
    lib = crf_oracle.lib
    lib.crf_qtable_audit.restype = C.c_long
    lib.crf_qtable_audit.argtypes = [C.c_float, C.c_float, C.c_uint32, C.c_uint32]
    assert lib.crf_qtable_audit(scale, shift, 29, 4096) == 0
    lib.crf_qchar_libm.restype = C.c_char
    lib.crf_qchar_libm.argtypes = [C.c_float, C.c_float, C.c_float]
    assert lib.crf_qchar_libm(0.0, scale, shift) == bytes([33 + 50])   # err = 0 -> +inf -> clamps to 50
    assert lib.crf_qchar_libm(1.0, scale, shift) == bytes([int(33.5 + min(50.0, max(1.0, shift)))])


def test_oracle_decode_edge_cases(crf_oracle):
    """T = 1, ties everywhere, saturated scores, narrow beams: the reference's edge behaviour, restated."""
    r = crf_oracle.decode(np.zeros((2, 1, 256), np.float16))
    assert r.n_bases.tolist() == [1, 1] and (r.moves[:, 0] == 1).all()
    r = crf_oracle.decode(np.full((1, 50, 256), 5.0, np.float16), clamp_val=5.0)
    assert r.n_bases[0] == 50  # every step beats the fixed stay score 2.0
    r = crf_oracle.decode(np.full((1, 50, 256), -5.0, np.float16), clamp_val=5.0)
    assert r.n_bases[0] == 1   # stays win everywhere; the first block always emits
    r1 = crf_oracle.decode(np.random.default_rng(0).standard_normal((1, 80, 1024)).astype(np.float16), beam_width=1)
    assert 1 <= r1.n_bases[0] <= 80 and set(r1.sequences[0]) <= set("ACGT")


_WORKER = r"""
import os, sys
sys.path.insert(0, os.environ["B200_ROOT"])
import torch, torch.distributed as dist
from dorado_b200 import parallel as P
dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{os.environ['B200_PORT']}",
                        rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
rank, world = dist.get_rank(), dist.get_world_size()
mine = P.shard_reads(103, world, rank)
sizes = P.all_gather_int(len(mine))
assert sum(sizes) == 103 and max(sizes) - min(sizes) <= 1, sizes
t = P.max_over_ranks(1.0 + rank)
assert t == float(world), t
total = P.sum_over_ranks(len(mine))
assert total == 103
P.barrier()
print("ok", rank, len(mine), t)
"""


def test_multi_rank_sharding_with_gloo(tmp_path):
    port = 29500 + (os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", B200_ROOT=str(ROOT), B200_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, "-c", _WORKER], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=240)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert all("ok" in o for o in outs)


def test_adapter_header_compiles_against_reference_headers():
    """include/B200ModelRunner.h implements dorado::basecall::ModelRunnerBase; type-check it against the
    reference's own headers where the reference tree is available (not on the GPU box)."""
    d = pathlib.Path("/root/reference/dorado")
    if not os.path.isdir(d):   # also False where the tree exists but this user may not read it
        pytest.skip("reference tree not present")
    import torch
    t = pathlib.Path(torch.__file__).parent
    src = ROOT / "tests" / "data" / "adapter_check.cpp"
    inc = [ROOT / "include", d, d / "basecall", d / "basecall/include", d / "nn/include", d / "config/include",
           d / "torch_utils/include", d / "utils/include", d / "models/include", d / "3rdparty/spdlog/include",
           d / "3rdparty/NVTX/c/include", d / "3rdparty/toml11/include"]
    cmd = ["/usr/bin/g++", "-std=c++23", "-fsyntax-only", "-w", "-D_GLIBCXX_USE_CXX11_ABI=1", "-DDORADO_CUDA_BUILD=0",
           "-DDORADO_METAL_BUILD=0", "-DDORADO_ORIN=0"] + [f"-I{p}" for p in inc] + \
          ["-isystem", str(t / "include"), "-isystem", str(t / "include/torch/csrc/api/include"), str(src)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]


def test_c_abi_from_a_plain_c_client(tmp_path):
    """include/b200call.h is a C header: a C11 program built with gcc links libb200call.so, exercises the host-side entry
    points (golden vectors of the reference's ChunkTest) and sees the device entry points fail loudly without a GPU."""
    exe = tmp_path / "abi_smoke"
    lib_dir = ROOT / "dorado_b200"
    cmd = ["/usr/bin/gcc", "-std=c11", "-Wall", "-Wextra", "-Werror", "-pedantic", f"-I{ROOT / 'include'}",
           str(ROOT / "tests" / "data" / "abi_smoke.c"), "-o", str(exe), f"-L{lib_dir}", "-lb200call",
           f"-Wl,-rpath,{lib_dir}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and "abi_smoke ok" in r.stdout, r.stdout + r.stderr


def test_chunk_size_buckets_and_benchmark_table_lookup():
    """CudaCaller.cpp:379-414: the requested chunk size plus half of it (simplex), normalised; CudaChunkBenchmarks lookup by
    (GPU name, model name) with the alias list, empty for unknown pairs."""
    from dorado_b200 import batching
    from dorado_b200.config import load_model_config
    from conftest import MODELS
    hac = load_model_config(model_dir("hac"))
    sup = load_model_config(model_dir("sup"))
    assert batching.chunk_size_buckets(hac, 10000) == [9996, 4998]
    assert batching.chunk_size_buckets(hac, 10000, pipeline="duplex") == [9996]
    assert batching.chunk_size_buckets(sup, 10000) == [9984, 4992]
    assert batching.chunk_size_buckets(hac, 600) == [600, 504]          # never below overlap + 1, rounded up to the granularity
    assert batching.lookup_chunk_benchmarks("NVIDIA GeForce 256", MODELS["hac"]) == []
    assert batching.lookup_chunk_benchmarks("NVIDIA B200", "no_such_model@v0") == []
    for kind in ("fast", "hac", "sup"):
        t = batching.lookup_chunk_benchmarks("NVIDIA B200", MODELS[kind])
        assert t == batching.lookup_chunk_benchmarks("NVIDIA HGX B200", MODELS[kind])
        if t:   # measured table committed: ascending batch sizes, strictly improving times
            assert all(a[0] < b[0] and a[1] > b[1] for a, b in zip(t, t[1:]))
            gran = batching.batch_size_granularity(load_model_config(model_dir(kind)))
            assert all(b % gran == 0 for b, _ in t)


def test_flstm_config_and_weight_folding():
    """FLSTM models (BasecallModelConfig.cpp:257-279, nn/FLSTMStack.cpp): config parsing, tensor list (crf_utils.cpp:36-41) and
    the fold up @ dn that lets the LSTM kernels serve them: the oracle's FLSTM forward equals its LSTM forward on the folded
    tensors."""
    from conftest import model_dir
    from dorado_b200.config import load_model_config
    from dorado_b200.weights import fold_flstm_weights, synthetic_weights, tensor_specs
    from oracle import nn_oracle
    cfg = load_model_config(model_dir("flstm"))
    plain = load_model_config(model_dir("fast"))
    assert cfg.is_flstm_model and not plain.is_flstm_model
    assert cfg.lstm_inner_dim == 32 and cfg.lstm_layers == 5 and cfg.lstm_size == 96
    names = list(tensor_specs(cfg))
    assert names[6:12] == [f"4.rnn.{k}.tensor" for k in ("dn_weight_ih", "dn_weight_hh", "up_weight_ih", "up_weight_hh",
                                                         "up_bias_ih", "up_bias_hh")]
    w = synthetic_weights(cfg, 3)
    folded = fold_flstm_weights(cfg, w)
    assert list(folded) == list(tensor_specs(plain))
    assert folded["4.rnn.weight_ih_l0.tensor"].shape == (384, 96)
    sig = np.random.default_rng(0).standard_normal((2, cfg.normalise_chunk_size(1200))).astype(np.float32)
    a = nn_oracle.forward(cfg, w, sig)
    b = nn_oracle.forward(plain, folded, sig)
    np.testing.assert_allclose(a, b, rtol=0, atol=1e-5)
    assert np.abs(a).max() > 1.0
