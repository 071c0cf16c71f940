"""The drop-in boundary exercised on the CUDA library itself (SURVEY.md 8(b)): user programs written against
<nlopt.h> -- a plain C one and a C++ one over a wrapper in the style of the reference's nlopt.hpp -- are compiled on
the GPU box with `-lnlopt`, resolve libnlopt.so.1 (this repository's build under the reference's SONAME,
reference CMakeLists.txt:31-33) and run the tutorial problem of test/t_tutorial.cxx on the B200 for LD_MMA (24),
LD_CCSAQ (41) and LD_AUGLAG (31).  The not-gpu half checks that the programs compile and link here and that the
SONAME / NEEDED entries are the reference's."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COMPAT = os.path.join(ROOT, "nlopt_b200", "compat")
OUT = os.path.join(ROOT, "tests", "_build", "dropin")


def _build(kind):
    os.makedirs(OUT, exist_ok=True)
    src = os.path.join(ROOT, "tests", "cpp", "dropin_tutorial." + ("c" if kind == "c" else "cpp"))
    exe = os.path.join(OUT, "dropin_" + kind)
    cc = ["gcc", "-O1", "-std=c99"] if kind == "c" else ["g++", "-O1", "-std=c++11"]
    cmd = cc + [f"-I{os.path.join(ROOT, 'include')}", src, "-o", exe, f"-L{COMPAT}", "-lnlopt", f"-Wl,-rpath,{COMPAT}", "-lm"]
    subprocess.check_call(cmd)
    return exe


@pytest.mark.parametrize("kind", ["c", "cxx"])
def test_user_programs_link_against_the_reference_soname(built, kind):
    exe = _build(kind)
    dyn = subprocess.run(["readelf", "-d", exe], capture_output=True, text=True).stdout
    assert "libnlopt.so.1" in dyn and "libnlopt_b200" not in dyn
    so = subprocess.run(["readelf", "-d", os.path.join(COMPAT, "libnlopt.so.1")], capture_output=True, text=True).stdout
    assert "SONAME" in so and "libnlopt.so.1" in so
    # every symbol the programs import from the library is exported by it
    need = {l.split()[-1] for l in subprocess.run(["nm", "-u", exe], capture_output=True, text=True).stdout.splitlines()
            if " nlopt_" in l}
    have = {l.split()[-1] for l in subprocess.run(["nm", "-D", "--defined-only", os.path.join(COMPAT, "libnlopt.so.1")],
                                                   capture_output=True, text=True).stdout.splitlines()}
    assert need and need <= have, need - have


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["c", "cxx"])
@pytest.mark.parametrize("alg", ["24", "41", "31"])
def test_user_programs_run_on_the_cuda_library(built, kind, alg):
    exe = _build(kind)
    r = subprocess.run([exe, alg], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "found minimum" in r.stdout
    maps_probe = subprocess.run(["ldd", exe], capture_output=True, text=True).stdout
    assert os.path.join("nlopt_b200", "compat", "libnlopt.so.1") in maps_probe


# ---- the reference's own test programs on the CUDA library -------------------------------------------------------
REFPROG = os.path.join(ROOT, "oracle", "_ref", "refprog")


def _refprog(name):
    exe = os.path.join(REFPROG, name)
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/refprog not built (make -C oracle refprog needs the reference's sources at build time)")
    return exe


@pytest.mark.gpu
@pytest.mark.parametrize("arg", [None, "24", "41", "31"])      # ctest t_tutorial, t_tutorial_24/41/31 (test/CMakeLists.txt:19)
def test_reference_t_tutorial_on_the_cuda_library(built, arg):
    r = subprocess.run([_refprog("t_tutorial")] + ([arg] if arg else []), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "found minimum" in r.stdout


@pytest.mark.gpu
def test_reference_cpp_functor_on_the_cuda_library(built):
    r = subprocess.run([_refprog("cpp_functor")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("alg", [24, 41])
@pytest.mark.parametrize("obj", [0, 1])
def test_reference_testopt_on_the_cuda_library(built, alg, obj):
    """ctest testopt_algo{24,41}_obj{0,1} (test/CMakeLists.txt:39-60): the reference's benchmark driver must report
    success (exit status 0 = it found the known optimum to its own tolerance)."""
    r = subprocess.run([_refprog("testopt"), "-r", "0", "-a", str(alg), "-o", str(obj)], stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:]
