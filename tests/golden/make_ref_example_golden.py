#!/usr/bin/env python
"""Golden outputs of the reference's own example programs, built against the REAL reference here (CPU):
tests/golden/ref_examples.json <- sha256 of the BMP that linux/examples/c_cmdline/main.c writes for each fixture.
Run in the container that has /root/reference:  python tests/golden/make_ref_example_golden.py"""
import hashlib, json, os, subprocess, sys, tempfile
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import ref_examples as B

FIXTURES = ["tulips", "croptest", "ncc1701", "sciopero", "batman"]


def main():
    B.build(with_reference=True)
    exe = os.path.join(B.OUT, "ref_c_cmdline_refimpl")
    out = {}
    with tempfile.TemporaryDirectory() as td:
        for n in FIXTURES:
            bmp = os.path.join(td, n + ".bmp")
            r = subprocess.run([exe, os.path.join(HERE, "images", n + ".jpg"), bmp], stdout=subprocess.PIPE, text=True)
            assert r.returncode == 0 and os.path.exists(bmp), (n, r.stdout)
            data = open(bmp, "rb").read()
            out[n] = {"bmp_sha256": hashlib.sha256(data).hexdigest(), "bmp_bytes": len(data)}
    json.dump({"program": "linux/examples/c_cmdline/main.c <in.jpg> <out.bmp> (RGB565_LITTLE_ENDIAN framebuffer -> BMP), default (SSE2) build",
               "fixtures": out}, open(os.path.join(HERE, "ref_examples.json"), "w"), indent=1, sort_keys=True)
    print(json.dumps(out, indent=1))


main()
