"""CPU-side checks: the C-ABI library loads and exports every symbol include/b200pir.h declares,
the cooperative-NTT index logic (emulated thread by thread) equals the oracle, and the product path
fails loudly without a GPU instead of falling back."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from sdk_b200 import build
    build.build()
    import sdk_b200._lib as L
    header = open(os.path.join(ROOT, "include", "b200pir.h")).read()
    declared = set(re.findall(r"\b(b200pir_[a-z0-9_]+)\s*\(", header))
    nm = subprocess.check_output(["nm", "-D", "--defined-only", L.SO_PATH], text=True)
    exported = set(re.findall(r" T (b200pir_[a-z0-9_]+)", nm))
    assert declared <= exported, sorted(declared - exported)
    assert declared == set(L.EXPORTED), sorted(declared ^ set(L.EXPORTED))


def test_header_is_plain_c_and_links_from_c(tmp_path):
    """The boundary is a C ABI: include/b200pir.h must compile as C99 (no C++-isms, no torch or CUDA types) and a C program must
    link against the library (the native callers in tests/cpp compile the same way on the GPU box)."""
    src = tmp_path / "abi.c"
    src.write_text('#include "b200pir.h"\n#include <stdio.h>\n'
                   'int main(void) { b200pir_params p; (void)p; printf("%d %s\\n", b200pir_device_count() >= 0, '
                   'b200pir_last_error() ? "ok" : "null"); return 0; }\n')
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.check_call([cc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I" + os.path.join(ROOT, "include"), "-o",
                           str(tmp_path / "abi"), str(src), "-L" + os.path.join(ROOT, "sdk_b200"), "-lb200pir",
                           "-Wl,-rpath," + os.path.join(ROOT, "sdk_b200")])
    out = subprocess.check_output([str(tmp_path / "abi")], text=True).split()
    assert out == ["1", "ok"]
    for cpp in ("concurrent_callers.cpp", "host_mirror_smoke.cpp"):          # the native test programs at least compile here
        gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([gxx, "-std=c++17", "-O1", "-pthread", "-Wall", "-o", str(tmp_path / cpp[:-4]),
                               os.path.join(ROOT, "tests", "cpp", cpp), "-L" + os.path.join(ROOT, "sdk_b200"), "-lb200pir",
                               "-Wl,-rpath," + os.path.join(ROOT, "sdk_b200")])


def test_no_cpu_fallback_without_gpu():
    import sdk_b200.spiral as S
    import sdk_b200._lib as L
    if L.LIB.b200pir_device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(S.B200PirError):
        S.Params(n=2, nu_1=6, nu_2=2, p=256, q2_bits=20, t_gsw=8, t_conv=4, t_exp_left=8, t_exp_right=8,
                 instances=1, db_item_size=8192, version=0)


def test_product_never_imports_the_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may touch oracle/: not the package, not the public
    headers, not the scripts."""
    for top in ("sdk_b200", "include", "scripts"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, top)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".sh")):
                    src = open(os.path.join(dirpath, f)).read()
                    assert "oracle_lib" not in src and "liboracle" not in src and "spiral_oracle" not in src, (top, f)


def test_cooperative_ntt_emulation_matches_oracle(tmp_path):
    exe = str(tmp_path / "ntt_core_emul")
    subprocess.check_call(["/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++", "-O2", "-std=c++17", "-o", exe,
                           os.path.join(ROOT, "tests", "cpp", "ntt_core_emul.cpp")])
    out = subprocess.check_output([exe], text=True)
    assert out.strip() == "OK", out


def test_tcgen05_operand_images_and_epilogue_emulation(tmp_path):
    """tests/cpp/tc5_emul.cpp: the per-thread image builders and the epilogue lane arithmetic of the tcgen05 first
    dimension, run on the CPU against the canonical UMMA K-major layout definition and 128-bit reference sums."""
    exe = str(tmp_path / "tc5_emul")
    subprocess.check_call(["/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++", "-O2", "-std=c++17", "-o", exe,
                           os.path.join(ROOT, "tests", "cpp", "tc5_emul.cpp")])
    out = subprocess.check_output([exe], text=True)
    assert out.strip() == "tc5 emulation ok", out


def test_tcgen05_descriptors_match_cutlass_bitfields(tmp_path):
    """tests/cpp/tc5_desc_check.cu: our hand-packed instruction / shared-memory descriptors vs the same fields packed by CUTLASS's
    bit-field structs (cute/arch/mma_sm100_desc.hpp), frozen in tests/golden/tc5_descriptors.json by
    tests/golden/make_tc5_descriptors.cu."""
    import json
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    exe = str(tmp_path / "tc5_desc_check")
    subprocess.check_call([nvcc if os.path.exists(nvcc) else "nvcc", "-std=c++17", "-o", exe,
                           os.path.join(ROOT, "tests", "cpp", "tc5_desc_check.cu"), "-ccbin",
                           "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"])
    got = json.loads(subprocess.check_output([exe], text=True))
    with open(os.path.join(ROOT, "tests", "golden", "tc5_descriptors.json")) as f:
        gold = json.load(f)
    assert got == {k: gold[k] for k in ("instr_desc", "smem_desc")}, (got, gold)


def test_cooperative_ntt4096_emulation_matches_oracle(tmp_path):
    exe = str(tmp_path / "ntt_core4096_emul")
    subprocess.check_call(["/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++", "-O2", "-std=c++17", "-o", exe,
                           os.path.join(ROOT, "tests", "cpp", "ntt_core4096_emul.cpp")])
    out = subprocess.check_output([exe], text=True)
    assert out.strip() == "OK", out
