"""The C-ABI shared library loads without a GPU and exports every symbol the headers in include/ declare
(no compute calls here)."""
import ctypes as C
import os
import re
import subprocess

import pytest

import ffi
import refgold

INC = os.path.join(ffi.ROOT, "include")


def _declared_c_symbols():
    txt = open(os.path.join(INC, "voldor_b200.h")).read()
    return sorted(set(re.findall(r"\b(vb_[a-z0-9_]+)\s*\(", txt)))


def _declared_cpp_symbols():
    txt = open(os.path.join(INC, "gpu_kernels.h")).read() + open(os.path.join(INC, "py_export.h")).read()
    return sorted(set(re.findall(r"(?:DLL_EXPORT|VB_EXPORT) int ([a-z0-9_]+)\s*\(", txt)))


@pytest.mark.skipif(not os.path.exists(ffi.OURS), reason="libvoldor_b200.so not built (make lib)")
def test_library_exports_every_declared_symbol():
    lib = C.CDLL(ffi.OURS)
    names = _declared_c_symbols()
    assert len(names) >= 14
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/voldor_b200.h but not exported"
    # C++-linkage entry points keep the reference's mangled names (drop-in for voldor/*.cpp, pyvoldor_vo.pyx)
    out = subprocess.check_output(["nm", "-D", "--defined-only", ffi.OURS], text=True)
    for n in _declared_cpp_symbols():
        assert re.search(rf"\b_Z\d+{n}", out), f"C++ symbol {n} missing"
    lib.vb_version.restype = C.c_char_p
    assert b"sm_100a" in lib.vb_version()


@pytest.mark.skipif(not os.path.exists(ffi.OURS), reason="libvoldor_b200.so not built (make lib)")
def test_mangled_names_match_the_reference_build():
    """the reference's own objects and ours export byte-identical mangled names for the 8 entry points"""
    def syms(path):
        out = subprocess.check_output(["nm", "-D", "--defined-only", path], text=True)
        return {l.split()[-1] for l in out.splitlines() if " T " in l and l.split()[-1].startswith("_Z")}
    ours, ref = syms(ffi.OURS), set(refgold.reference(lambda: sorted(syms(ffi.REF))))
    wanted = {s for s in ref if re.match(r"_Z\d+(meanshift_gpu|fit_robust_gaussian|collect_p3p_instances|"
                                        r"solve_batch_p3p_ap3p_gpu|solve_batch_p3p_lambdatwist_gpu|"
                                        r"optimize_depth_gpu|align_frame_init_gpu|align_frame_eval_gpu)", s)}
    assert len(wanted) == 8
    missing = wanted - ours
    assert not missing, missing


def test_python_binding_fails_loudly_without_library(tmp_path, monkeypatch):
    import voldor_b200.pyvoldor_vo as pv

    monkeypatch.setattr(pv, "_lib", None)
    monkeypatch.setattr(pv, "_LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(ImportError):
        pv.load_library()


def test_library_binds_its_own_symbols():
    """The library exports the reference's mangled names; -Bsymbolic keeps its internal calls bound to itself when
    a second library with the same names (the reference build, oracle/_ref) lives in the same process."""
    import subprocess
    dyn = subprocess.run(["readelf", "-d", ffi.OURS], capture_output=True, text=True).stdout
    assert "SYMBOLIC" in dyn
    if os.path.exists(ffi.REF):
        assert "SYMBOLIC" in subprocess.run(["readelf", "-d", ffi.REF], capture_output=True, text=True).stdout


def test_libc_rand_speculation_is_invisible():
    """fused mean-shift start-sample selection (csrc/libc_rand.h): after snapshot / 20 draws / rewind / k draws the
    process-wide rand() stream is exactly k draws further — the consumption the reference's loop would show."""
    lib = C.CDLL(ffi.OURS)
    libc = C.CDLL(None)
    for seed, keep in ((5, 3), (77, 0), (123, 20)):
        libc.srand(seed)
        want = [libc.rand() for _ in range(keep + 4)]
        libc.srand(seed)
        assert lib.vb_debug_rand_speculate(20, keep) == 0
        got = [libc.rand() for _ in range(4)]
        assert got == want[keep:], (seed, keep)
    # and without any srand: the stream simply continues
    a = libc.rand()
    assert lib.vb_debug_rand_speculate(7, 0) == 0
    libc.srand(1)


def test_caller_compiled_against_the_reference_headers_links_against_this_library(tmp_path):
    """library-level drop-in (INTEGRATION.md §3): a translation unit that includes the REFERENCE's own
    gpu-kernels/gpu_kernels.h and voldor/py_export.h (where the checkout lies) and uses every entry point — with
    the header's default arguments where it has them — links against libvoldor_b200.so with nothing else."""
    ref = os.environ.get("VOLDOR_REFERENCE", "/root/reference")
    hdr = os.path.join(ref, "gpu-kernels", "gpu_kernels.h")
    if not os.path.exists(hdr):
        pytest.skip("reference checkout not present")
    src = tmp_path / "caller.cpp"
    src.write_text(
        '#include "%s"\n#include "%s"\n' % (hdr, os.path.join(ref, "voldor", "py_export.h")) +
        "int main(int argc, char**) {\n"
        "  if (argc < 1000) return 0;  // only has to link\n"
        "  float f = 0; int i = 0; float* t[1] = {&f};\n"
        "  i += meanshift_gpu(&f, 1.f, &f, &f, &i, false, 1, 1);              // default epsilon .. good_init\n"
        "  i += fit_robust_gaussian(&f, &f, &f, 3.f, 0.f, &f, &i, 1, 1, 1e-5f, 1);\n"
        "  i += collect_p3p_instances(t, t, &f, &f, t, t, &f, &f, 1, 1, 1, 0, .5f, 1.f, .1f, 1.f, 3);\n"
        "  i += solve_batch_p3p_ap3p_gpu(&f, &f, &f, &f, &f, 1, 1);\n"
        "  i += solve_batch_p3p_lambdatwist_gpu(&f, &f, &f, &f, &f, 1, 1);\n"
        "  i += optimize_depth_gpu(t, t, t, t, t, t, t, &f, &f, &f, t, t, t, t, 1.f, 1, 0, 1, 1, 0.f, 1, 1, 1,\n"
        "                          .1f, .1f, 1.f, 1.f, true, .5f, .9f, 1.f, false);\n"
        "  i += align_frame_init_gpu(t, t, t, &f, 1.f, 1.f, 1, 1, 1);\n"
        "  i += align_frame_eval_gpu(0, 0, &f, &f, &f, &f);                     // default apply_weights\n"
        "  i += py_voldor_wrapper(&f, 0, 0, 0, 0, 0, 1, 1, 0, 0, 0, 1, 0, 1, 1, \"\", i, &f, &f, &f, &f);\n"
        "  return i;\n}\n")
    exe = tmp_path / "caller"
    libdir = os.path.dirname(ffi.OURS)
    r = subprocess.run(["g++", "-std=c++17", str(src), "-o", str(exe), "-L" + libdir, "-lvoldor_b200",
                        "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    # and it starts (loads the library, resolves every symbol eagerly) without a GPU
    r = subprocess.run([str(exe)], capture_output=True, text=True, env=dict(os.environ, LD_BIND_NOW="1"))
    assert r.returncode == 0, r.stderr
