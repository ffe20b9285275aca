#!/usr/bin/env python
"""Build the reference's own example / test programs UNMODIFIED against this library (SURVEY.md 8(f)3).

The programs reach the reference implementation through relative includes ("../../../src/JPEGDEC.h", "../../../src/jpeg.inl",
"../../../src/JPEGDEC.cpp").  A shadow tree under oracle/_ref/examples/shadow/ holds *symlinks* to the reference's program
sources and test images at their original relative places, and a src/ directory whose three files forward to
include/JPEGDEC.h (the C entry points and the C++ class live in libjpegdec_b200.so / the header).  Nothing from the
reference is copied; the binaries land in oracle/_ref/examples/ (git-ignored, next to the other reference builds) and find
libjpegdec_b200.so relative to themselves, so the tree can be moved to another machine after the build.

  ref_c_cmdline   <- linux/examples/c_cmdline/main.c          (C, includes JPEGDEC.h + jpeg.inl)
  ref_perf_test   <- linux/examples/jpeg_perf_test/main.cpp   (C++, #include <JPEGDEC.h>)
  ref_jpegdec_test<- MacOS/JPEGDEC_Test/JPEGDEC_Test/main.cpp (C++, includes JPEGDEC.cpp; the reference's 12 tests)

With --with-reference it also builds the same three programs against the real reference sources (CPU) as
*_refimpl: their output is what ours is compared with (tests/golden/make_golden.py records the digests).
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("JPEGDEC_REFERENCE", "/root/reference")
OUT = os.path.join(HERE, "_ref", "examples")
SHADOW = os.path.join(OUT, "shadow")
LIBDIR = os.path.join(ROOT, "jpegdec_b200")

PROGRAMS = {
    "ref_c_cmdline": ("gcc", "linux/examples/c_cmdline/main.c"),
    "ref_perf_test": ("g++", "linux/examples/jpeg_perf_test/main.cpp"),
    "ref_jpegdec_test": ("g++", "MacOS/JPEGDEC_Test/JPEGDEC_Test/main.cpp"),
}
LINKS = ["linux/examples/c_cmdline/main.c", "linux/examples/jpeg_perf_test/main.cpp",
         "MacOS/JPEGDEC_Test/JPEGDEC_Test/main.cpp", "test_images"] + \
        ["MacOS/JPEGDEC_Test/JPEGDEC_Test/corrupt%d.h" % i for i in range(1, 6)]


def available():
    return os.path.isdir(os.path.join(REF, "src"))


def _shadow():
    for rel in LINKS:
        dst = os.path.join(SHADOW, rel)
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        if os.path.islink(dst):
            os.unlink(dst)
        os.symlink(os.path.join(REF, rel), dst)
    src = os.path.join(SHADOW, "src")
    os.makedirs(src, exist_ok=True)
    fwd = '#include "%s"\n' % os.path.join(ROOT, "include", "JPEGDEC.h")
    for name, body in (("JPEGDEC.h", fwd), ("JPEGDEC.cpp", fwd), ("jpeg.inl", "/* the JPEG_* entry points come from libjpegdec_b200.so */\n")):
        with open(os.path.join(src, name), "w") as f:
            f.write(body)


def build(with_reference=False):
    if not available():
        raise RuntimeError("reference sources not present at %s" % REF)
    _shadow()
    built = []
    for name, (cc, rel) in PROGRAMS.items():
        out = os.path.join(OUT, name)
        cmd = [cc, "-O2", "-w", "-I" + os.path.join(ROOT, "include"), os.path.join(SHADOW, rel), "-o", out,
               "-L" + LIBDIR, "-ljpegdec_b200", "-Wl,-rpath,$ORIGIN/" + os.path.relpath(LIBDIR, OUT)]
        subprocess.run(cmd, check=True)
        built.append(out)
        if with_reference:
            out2 = out + "_refimpl"
            extra = [os.path.join(REF, "src", "JPEGDEC.cpp")] if name == "ref_perf_test" else []   # as linux/examples/jpeg_perf_test/Makefile does
            subprocess.run([cc, "-O2", "-w", "-D__LINUX__", "-I" + os.path.join(REF, "src"), os.path.join(REF, rel)] + extra + ["-o", out2], check=True)
            built.append(out2)
    return built


if __name__ == "__main__":
    for b in build("--with-reference" in sys.argv):
        print(b)
