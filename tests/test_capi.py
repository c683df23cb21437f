"""CPU suite for the boundary: the shared library loads and exports exactly what include/ofdm_b200.h
declares, fails loudly without a GPU, and its host-side writers produce the files the reference's own
scripts (compare_double.py, compare_complex.py, OFDM_Plotting.py) parse."""
import ast
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

REF_ROOT = os.environ.get("REF_ROOT", "")          # a checkout of the original simulator, as for oracle/Makefile
REF_SCRIPTS = os.path.join(REF_ROOT, "scripts")


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "ofdm_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ofdm_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(pkg, lib):
    syms = declared_symbols()
    assert len(syms) >= 38
    for s in syms:
        assert hasattr(lib, s), "declared in ofdm_b200.h but not exported: " + s
    assert set(syms) == set(pkg.binding.SIGNATURES), set(syms) ^ set(pkg.binding.SIGNATURES)
    assert lib.ofdm_version() == 100
    assert C.sizeof(pkg.Counters) == 64


def test_no_cpu_fallback(pkg, lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    h = C.c_void_p()
    st = lib.ofdm_ctx_create(C.byref(h), 0)
    assert st == 5 and b"no CPU fallback" in lib.ofdm_strerror(st)
    with pytest.raises(pkg.OfdmError):
        pkg.Ofdm(0, lib=lib)
    # every entry point refuses a null context instead of computing anything
    assert lib.ofdm_fft64(None, None, None, 1, 0) == 1
    assert lib.ofdm_sweep_inject_host(None, None, None, 1, 2, None, 0, 0, None) == 1


def test_product_never_touches_the_oracle():
    """the oracle is test infrastructure: nothing under the product package may mention it"""
    pkg_dir = os.path.join(ROOT, "ieee-802.11-ofdm-qpsk-simulator_b200")
    for dirpath, _, files in os.walk(pkg_dir):
        for f in files:
            if f.endswith((".py", ".c", ".cu", ".cuh", ".h")) or f == "Makefile":
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "pyoracle" not in text and "libofdm_oracle" not in text and "libofdm_ref" not in text, f
    out = subprocess.run(["ldd", os.path.join(pkg_dir, "libofdm_b200.so")], capture_output=True, text=True).stdout
    assert "oracle" not in out and "torch" not in out


def test_float_writer_format(pkg, lib, tmp_path):
    a = np.array([6, 7.5, -3.7, 0, 1e-7, -np.inf, 3.65e-2], np.float32)
    p = str(tmp_path / "Output_BER.txt")
    assert pkg.write_float_array_to_file(lib, a, p) == 0
    text = open(p).read()
    assert text == "\t".join("%.2e" % float(x) for x in a) + "\n"
    assert pkg.write_float_array_to_file(lib, a, str(tmp_path / "nodir" / "x.txt")) == 4          # OFDM_ERR_IO, no exit()


def test_writers_match_reference_writers(pkg, lib, ref, tmp_path):
    rng = np.random.default_rng(0)
    a = rng.standard_normal(35).astype(np.float32)
    iq = rng.standard_normal((96, 2)).astype(np.float32)
    ref.write_float(a, str(tmp_path / "r.txt")); pkg.write_float_array_to_file(lib, a, str(tmp_path / "m.txt"))
    assert open(tmp_path / "r.txt").read() == open(tmp_path / "m.txt").read()
    ref.write_complex(iq, str(tmp_path / "rc.txt")); pkg.write_complex_array_to_file(lib, iq, str(tmp_path / "mc.txt"), 0)
    assert open(tmp_path / "rc.txt").read() == open(tmp_path / "mc.txt").read()


@pytest.mark.skipif(not REF_ROOT or not os.path.isdir(REF_SCRIPTS), reason="REF_ROOT (the original simulator's scripts) not set")
def test_reference_scripts_consume_outputs_unchanged(pkg, lib, port, golden, tmp_path):
    # compare_double.py: demodulated bits of the golden payload, dumped in the live (real-part) format, vs data/Matlab_Output.txt
    b96 = golden["matlab_output_bits"]
    bits = np.concatenate([b96, b96])[None, :]
    rx = port.rx_frames(port.tx_frames(bits, 2), bits, 2)["bits"][0, :96]
    iq = np.stack([rx.astype(np.float32), np.zeros(96, np.float32)], axis=1)
    assert pkg.write_complex_array_to_file(lib, iq, str(tmp_path / "Code_Output.txt"), 0) == 0
    with open(tmp_path / "Matlab_Output.txt", "w") as f:
        f.write(open(os.path.join(REF_ROOT, "data", "Matlab_Output.txt")).read())
    out = subprocess.run([sys.executable, os.path.join(REF_SCRIPTS, "compare_double.py")], cwd=tmp_path, capture_output=True, text=True)
    assert out.returncode == 0 and "Extracted 96 numbers" in out.stdout and "Max Error: 0.000000e+00" in out.stdout, out.stdout + out.stderr
    # compare_complex.py: IQ in the "re + imi" triple format on both sides
    tx = port.tx_frames(bits, 2)[0]
    assert pkg.write_complex_array_to_file(lib, tx, str(tmp_path / "Code_Output.txt"), 1) == 0
    assert pkg.write_complex_array_to_file(lib, tx, str(tmp_path / "Matlab_Output.txt"), 1) == 0
    out = subprocess.run([sys.executable, os.path.join(REF_SCRIPTS, "compare_complex.py")], cwd=tmp_path, capture_output=True, text=True)
    assert out.returncode == 0 and "Extracted 320 complex numbers" in out.stdout and "No Mismatch Found!" in out.stdout, out.stdout + out.stderr
    # OFDM_Plotting.py: its parser (the module itself plots at import time and matplotlib is not installed)
    src = open(os.path.join(REF_SCRIPTS, "OFDM_Plotting.py")).read()
    fn = [n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "read_double_file"][0]
    ns = {}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), "OFDM_Plotting.py", "exec"), ns)
    vals = np.array([-3.7, 12.8, -np.inf, 0.0, 41.3], np.float32)
    p = str(tmp_path / "Output_EVM_AGC_DB.txt")
    assert pkg.write_float_array_to_file(lib, vals, p) == 0
    got = ns["read_double_file"](p)
    assert got[2] == float("-inf") and np.allclose([got[0], got[1], got[3], got[4]], [-3.7, 12.8, 0.0, 41.3], rtol=1e-2)


def test_shard_range_and_counter_packing(pkg):
    sw = pkg.sweep
    for n, w in ((10, 3), (1000000, 8), (5, 8), (0, 2)):
        edges = [sw.shard_range(n, r, w) for r in range(w)]
        assert edges[0][0] == 0 and edges[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(edges, edges[1:]))
        sizes = [b - a for a, b in edges]
        assert max(sizes) - min(sizes) <= 1
    c = pkg.Counters(); c.bit_errors = 7; c.bits = 192; c.frames = 1; c.sum_err2 = 0.5; c.sum_ref2 = 96.0
    i, d = sw.counters_to_arrays([c, c])
    back = sw.arrays_to_counters(i, d)
    assert back[1].as_dict() == c.as_dict()


def test_every_documented_option_is_handled_and_vice_versa():
    """include/ofdm_b200.h documents the knobs of ofdm_ctx_set_option; csrc/ofdm_b200.cu handles them: the two lists must agree"""
    import re
    header = open(os.path.join(ROOT, "include", "ofdm_b200.h")).read()
    source = open(os.path.join(ROOT, "ieee-802.11-ofdm-qpsk-simulator_b200", "csrc", "ofdm_b200.cu")).read()
    block = header[header.index("int ofdm_ctx_set_option") - 4000:header.index("int ofdm_ctx_set_option")]
    documented = set(re.findall(r'\*\s+"([a-z_]+)"\s+=', block))
    handled = set(re.findall(r'!strcmp\(name, "([a-z_]+)"\)', source))
    assert handled and documented == handled, (sorted(documented - handled), sorted(handled - documented))
