"""CPU tests of the C-ABI library: it loads, exports every symbol include/kgb200.h declares, parses model files
identically to the oracle loader, reports errors like the reference, and refuses to run without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import kg_nn_oracle as orc
from conftest import ROOT, has_gpu
from katago_b200 import KGBError, NeuralNet, modelgen, nn_backend


def header_symbols():
    text = open(os.path.join(ROOT, "include", "kgb200.h")).read()
    return sorted(set(re.findall(r"KGB_API\s+[\w\s\*]+?\b(kgb_\w+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = nn_backend.load_library()
    syms = header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"libkgb200.so does not export {s}"
    assert sorted(nn_backend.ABI_SYMBOLS) == syms


def test_library_is_sm100a_native():
    """SASS carries tcgen05 MMA, TMA and TMEM loads (B200_PROFILING.md 'What proves a Blackwell-native kernel')."""
    import shutil, subprocess
    # the toolkit that built the library (katago_b200/csrc/build.sh) need not be on PATH
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not found")
    sass = subprocess.run([cuobjdump, "-sass", nn_backend.library_path()], capture_output=True, text=True).stdout
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in sass
    assert "sm_100a" in sass


@pytest.mark.parametrize("key", ["tiny_reg", "tiny_nbt", "tiny_nbt_gz", "tiny_relu_v8"])
def test_model_info_matches_oracle_loader(tmp_models, key):
    lm = NeuralNet.loadModelFile(tmp_models[key])
    m = orc.load_model(tmp_models[key])
    d = NeuralNet.getModelDesc(lm)
    assert d["model_version"] == m.version
    assert d["num_input_channels"] == 22 and d["num_input_global_channels"] == 19
    assert d["trunk_num_channels"] == m.trunk_c and d["num_blocks"] == len(m.blocks)
    assert d["num_policy_channels"] == m.policy_out_channels
    assert d["num_score_value_channels"] == m.sv3_mul.cout
    assert d["conv_macs_per_position"] == orc.conv_macs_per_position(m)
    assert d["name"] == m.name


def test_real_net_and_sha256(golden_dir):
    import hashlib
    path = os.path.join(golden_dir, "models", "g170-b6c96-s175395328-d26788732.bin.gz")
    sha = hashlib.sha256(open(path, "rb").read()).hexdigest()
    lm = NeuralNet.loadModelFile(path, sha)
    assert lm.desc["sha256"] == sha and lm.desc["model_version"] == 8 and lm.desc["conv_macs_per_position"] == 1002112
    with pytest.raises(KGBError, match="sha256"):
        NeuralNet.loadModelFile(path, "0" * 64)


def test_loader_errors(tmp_path, tmp_models):
    with pytest.raises(KGBError, match="could not open"):
        NeuralNet.loadModelFile(str(tmp_path / "missing.bin.gz"))
    bad = tmp_path / "bad.bin"
    bad.write_bytes(b"name 15 22 19 garbage")
    with pytest.raises(KGBError):
        NeuralNet.loadModelFile(str(bad))
    trunc = tmp_path / "trunc.bin"
    trunc.write_bytes(open(tmp_models["tiny_reg"], "rb").read()[:5000])
    with pytest.raises(KGBError):
        NeuralNet.loadModelFile(str(trunc))
    # a header that announces far more weights than the file holds must fail on the size check, not by allocating them
    # (3 x 3 x 16000 x 16000 floats = 9 GB; 1 x 1 x 2^30 x 2^30 would wrap a size_t)
    for conv, what in (("conv1 3 3 16000 16000 1 1 @BIN@", "too short"), ("conv1 1 1 1073741824 1073741824 1 1 @BIN@", "unreasonable size")):
        huge = tmp_path / "huge.bin"
        huge.write_bytes(("m 8 22 19 trunk 2 16 16 16 16 16 " + conv).encode() + b"\0" * 64)
        with pytest.raises(KGBError, match=what):
            NeuralNet.loadModelFile(str(huge))
    wrong = tmp_path / "model.weights"
    wrong.write_bytes(b"x")
    with pytest.raises(KGBError, match="should end with"):
        NeuralNet.loadModelFile(str(wrong))


def test_no_silent_cpu_fallback(tmp_models):
    if has_gpu():
        pytest.skip("a GPU is present")
    lm = NeuralNet.loadModelFile(tmp_models["tiny_reg"])
    ctx = NeuralNet.createComputeContext([0], 9, 9, True, lm)
    with pytest.raises(KGBError, match="no CUDA device|CUDA"):
        NeuralNet.createComputeHandle(ctx, lm, 4, False, True, 0)
    with pytest.raises(KGBError):
        NeuralNet.testEvaluateConv(1, 1, 8, 8, np.zeros((1, 1, 8, 8), np.float32), 1, 9, 9, True, np.zeros((1, 9, 9, 8), np.float32))


def test_context_argument_checks(tmp_models):
    lm = NeuralNet.loadModelFile(tmp_models["tiny_reg"])
    with pytest.raises(KGBError):
        NeuralNet.createComputeContext([0], 1, 19, True, lm)
    with pytest.raises(KGBError):
        NeuralNet.createComputeContext([0], 19, 50, True, lm)


def test_synthetic_file_roundtrip_weights(tmp_models):
    """modelgen -> file -> oracle loader keeps the weights (format check incl. the @BIN@ blocks)."""
    a = orc.load_model(tmp_models["tiny_nbt"], apply_transform=False)
    b = orc.load_model(tmp_models["tiny_nbt_gz"], apply_transform=False)
    assert np.array_equal(a.initial_conv.w, b.initial_conv.w)
    assert np.array_equal(a.blocks[1].blocks[0].gpool_to_bias.w, b.blocks[1].blocks[0].gpool_to_bias.w)


def test_zobrist_tables_reproduce_reference_pos_hash(golden_dir):
    """Row a25: the backend's restatement of Rand (MD5 + SHA-256 seeding, XorShift1024* + PCG32) and of Board::initHash's draw
    order regenerates the reference's Zobrist tables: XOR over the stones of fixture positions == the reference's pos_hash."""
    from katago_b200 import zobrist_tables
    for name in ("boardstream_19x19_multisuicide", "boardstream_9x9_multisuicide", "boardstream_13x7_nosuicide", "boardstream_5x5_multisuicide"):
        d = np.load(os.path.join(golden_dir, name + ".npz"))
        bh, sh = zobrist_tables(int(d["X"]), int(d["Y"]))
        for m in range(0, len(d["moves"]), 11):
            col = d["colors"][m]
            h = sh.copy()
            for yy, xx in zip(*np.nonzero(col)):
                h ^= bh[yy, xx, col[yy, xx] - 1]
            assert np.array_equal(h, d["pos_hash"][m]), (name, m)


def test_score_value_table_is_bit_exact_vs_reference(golden_dir):
    """Row a21: ScoreValue::expectedWhiteScoreValue (table built by the reference's quadrature, bilinear lookup) on 3000 argument
    tuples incl. clamped means, zero and huge stdevs, static (0, 2) and dynamic centres/scales, four board areas.
    Fixture: tests/golden/make_scorevalue_fixture.py (the reference's own function)."""
    from katago_b200.nn_backend import expected_white_score_value
    d = np.load(os.path.join(golden_dir, "scorevalue_samples.npz"))
    a = d["args"]
    got = expected_white_score_value(a[:, 0], a[:, 1], a[:, 2], a[:, 3], a[:, 4])
    assert np.array_equal(got, d["value"])


def test_value_weight_cdf_table_is_bit_exact_vs_reference(golden_dir):
    """Row a20: the t-distribution (3 dof) CDF table of the value weighting, as Search's constructor builds it from
    FancyMath::tdistcdf (fixture: the reference's own DistributionTable, tests/golden/make_scorevalue_fixture.py)."""
    from katago_b200.nn_backend import value_weight_cdf_table
    assert np.array_equal(value_weight_cdf_table(), np.load(os.path.join(golden_dir, "value_weight_cdf_table.npy")))


def test_search_shaped_facade_compiles_against_the_abi(tmp_path):
    """integration/b200selfplay.h (boundary 2: the Search-shaped C++ facade over the device game slots) is plain C++17 over
    include/kgb200.h; it must compile and link against the library (no GPU needed for that)."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "facade.cpp"
    src.write_text('#include "integration/b200selfplay.h"\nint main(int argc, char**) { if(argc > 100) { kgb_selfplay_config c = {}; b200::GameSlots s(nullptr, c, 19, 19); s.runWaves(1); return (int)s.getRootVisits(0); } return 0; }\n')
    exe = tmp_path / "facade"
    subprocess.run(["g++", "-std=c++17", "-Wall", "-I", root, str(src), "-o", str(exe), "-L", os.path.join(root, "katago_b200"), "-lkgb200",
                    "-Wl,-rpath," + os.path.join(root, "katago_b200")], check=True)
    assert subprocess.run([str(exe)]).returncode == 0


def test_rand_reproduces_the_reference_self_test_vector():
    """Row a25: the reference's own known-answer test for its generator (core/rand.cpp:386-415: Rand("abc"), 24 outputs)."""
    from katago_b200.nn_backend import rand_uint32_stream
    expected = [0x1C6B83BD, 0xFB7677DB, 0x698688D5, 0xA3CD21C3, 0xD0AD5B77, 0x8F889E6E, 0x22852278, 0xD71A114D, 0x295EF301, 0xAA0CCA48, 0x0B7271BB,
                0x4FE798FB, 0x26B4DD4B, 0x78B77C1B, 0x231C4DFB, 0x17FB87C6, 0x9CC23870, 0x1C2C2CF7, 0x62D51240, 0xF1D1A7FF, 0x44C45C0A, 0xF93ACFCE,
                0x42B1D236, 0xC1069B75]
    assert rand_uint32_stream("abc", 24).tolist() == expected


def test_product_code_never_touches_the_oracle():
    """oracle/ is test infrastructure: nothing under katago_b200/ or integration/ may import, execute, link or open it (only tests/,
    __graft_entry__.smoke() and bench.py's CPU legs do), and the product has no CPU fallback to route through."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    offenders = []
    for base in ("katago_b200", "integration"):
        for dirpath, _, files in os.walk(os.path.join(root, base)):
            if "_build" in dirpath:
                continue
            for f in files:
                if not f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".sh")):
                    continue
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                for m in re.finditer(r"(import\s+kg_nn_oracle|from\s+oracle|kg_nn_oracle\.|[\"'/]oracle/[\w./]*\.(py|so|a)\b|kgref_driver|libkgref)", text):
                    line = text[:m.start()].count("\n") + 1
                    src_line = text.splitlines()[line - 1].strip()
                    if src_line.startswith(("//", "#", "*")):       # mentions in comments (where a file is built from) are fine
                        continue
                    offenders.append((os.path.join(base, f), line, src_line[:120]))
    assert not offenders, offenders
