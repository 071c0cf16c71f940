"""The reference's own test programs against a library of ours.  build() compiles them, unmodified, into
oracle/_ref/refprog (`make refprog`, oracle/Makefile); here their objects are linked against a given library exporting
the NLopt C ABI.  The reference tree itself is only needed by test/t_python.py, a script that is run in place."""
import os
import subprocess

REF = os.environ.get("NLOPT_REFERENCE_DIR", "/root/reference")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROG = os.path.join(ROOT, "oracle", "_ref", "refprog")
NOT_BUILT = "oracle/_ref/refprog not built (make -C oracle refprog needs the reference's sources at build time)"


def available():
    return os.path.isfile(os.path.join(REF, "test", "t_python.py"))


def built():
    return all(os.path.exists(os.path.join(PROG, f)) for f in
               ("t_tutorial_refhdr.o", "t_tutorial_ourhdr.o", "cpp_functor_refhdr.o", "testopt.o", "testfuncs.o", "timer.o",
                "mt19937ar.o"))


def _link(compiler, objs, libpath, exe, extra=()):
    libdir, libfile = os.path.split(libpath)
    subprocess.check_call([compiler, *[os.path.join(PROG, o) for o in objs], "-o", exe, f"-L{libdir}", f"-l:{libfile}",
                           f"-Wl,-rpath,{libdir}", *extra])
    return exe


def reference_test(name, libpath, outdir, use_our_header):
    """test/<name>.cxx compiled over the reference-generated nlopt.hpp and the reference's nlopt.h (or ours, include/),
    linked against `libpath`; returns the executable path."""
    os.makedirs(outdir, exist_ok=True)
    hdr = "ourhdr" if use_our_header else "refhdr"
    return _link("g++", [f"{name}_{hdr}.o"], libpath, os.path.join(outdir, f"{name}_{hdr}"))


def reference_testopt(libpath, outdir):
    """The reference's benchmark driver test/testopt.c (+ testfuncs.c and, as test/CMakeLists.txt:26 does, the two util
    sources whose symbols it uses directly) linked against `libpath`."""
    os.makedirs(outdir, exist_ok=True)
    exe = os.path.join(outdir, "testopt_" + os.path.splitext(os.path.basename(libpath))[0])
    return _link("gcc", ["testopt.o", "testfuncs.o", "timer.o", "mt19937ar.o"], libpath, exe, ["-lm"])
