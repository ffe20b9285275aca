#!/usr/bin/env python
"""Record what the compiled reference returns for the calls the tests compare with -> tests/golden/reference/<name>.json.

Each test module that compares with the reference defines a record_* function next to its test: it makes the same calls
on the reference (oracle/_ref, both arithmetic builds) and returns digests of exactly what the test compares (pixels,
callback logs, return codes), so that the tests run without the reference.  Needs the reference build and
libjpegdec_b200.so (host-side calls only, no GPU):

    make -C oracle ref && python -m jpegdec_b200.build && python tests/golden/make_reference_golden.py
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import refdrv  # noqa: E402
from tests import test_gpu_parity, test_host, test_idct_blocks, test_oracle  # noqa: E402

RECORDS = {
    "oracle_dither": test_oracle.record_dither,
    "oracle_synthetic": test_oracle.record_synthetic_formats,
    "oracle_sweep": test_oracle.record_seeded_sweep,
    "idct_blocks": test_idct_blocks.record_idct_blocks,
    "host_schedule": test_host.record_schedule,
    "gpu_callbacks": test_gpu_parity.record_callbacks,
    "gpu_framebuffer_crop_thumb_dither": test_gpu_parity.record_framebuffer_crop_thumb_dither,
    "gpu_sweep": test_gpu_parity.record_gpu_sweep,
    "gpu_crop_scale": test_gpu_parity.record_crop_scale,
}


def main(names):
    refs = {m: refdrv.Ref(m) for m in ("sse", "scalar")}
    os.makedirs(os.path.join(HERE, "reference"), exist_ok=True)
    for name in names or RECORDS:
        rec = RECORDS[name](refs)
        lines = ["%s: %s" % (json.dumps(k), json.dumps(rec[k], separators=(",", ":"))) for k in sorted(rec)]
        with open(os.path.join(HERE, "reference", name + ".json"), "w") as f:
            f.write("{\n" + ",\n".join(lines) + "\n}\n")
        print(name, len(rec))


if __name__ == "__main__":
    main(sys.argv[1:])
