"""The reference build's outputs on the seeded cases of the `ref` tests, stored as CRC-32 in
tests/golden/reference_records.json, so that those tests run where oracle/_ref/libdmc_ref.so cannot be built.

RecordedReference stands in for oracle_py.Reference.  Every call is answered by a source library (the reference build
where it exists, else the C port, oracle/dmc_oracle.c) and its output must hash to the record of that exact call
(method, arguments, input bytes); a call without a record fails.  With the reference build present the records are
therefore checked against it as well.  The reference sources are not part of the repository; where they are absent
the records may come from the C port, which these very tests found bit-equal to the reference build on every one of
these cases (DESIGN.md, oracle table), and the file names its source.

Re-record (overwrites the file; the source is noted in it) with
    DMC_RECORD_REFERENCE=1 python -m pytest tests/test_oracle_vs_reference.py tests/test_pointcloud.py \
        tests/test_joint_bwrf.py tests/test_refshim_vs_cv2.py -m "not gpu"
"""
import hashlib
import json
import os
import zlib

import numpy as np
import pytest

from _util import GOLDEN_DIR

RECORDS = os.path.join(GOLDEN_DIR, "reference_records.json")
# the reference projects with _mm_rcp_ps, whose table differs between CPU vendors (see oracle/dmc_oracle.c)
HOST_DEPENDENT = {"project_points", "project_image"}
SHIM_CALLS = {"median_blur", "gaussian_kernel32f", "gaussian_blur32f", "morph", "copy_make_border", "convert_to"}


def _enc(v):
    if isinstance(v, np.ndarray):
        return "%s%s:%08x" % (v.dtype.str, v.shape, zlib.crc32(np.ascontiguousarray(v).tobytes()) & 0xFFFFFFFF)
    if isinstance(v, (float, np.floating)):
        return float(v).hex()
    return repr(v)


def call_key(name, args, kwargs):
    s = "|".join([name] + [_enc(a) for a in args] + ["%s=%s" % (k, _enc(v)) for k, v in sorted(kwargs.items())])
    return hashlib.sha1(s.encode()).hexdigest()[:12]


def output_crc(out):
    """CRC-32 of the output bytes, NaNs canonicalised (the tests compare NaN-aware)."""
    c = 0
    for a in (out if isinstance(out, tuple) else (out,)):
        a = np.ascontiguousarray(a)
        if a.dtype.kind == "f" and np.isnan(a).any():
            a = a.copy(); a[np.isnan(a)] = np.nan
        c = zlib.crc32(a.tobytes(), c)
    return "%08x" % (c & 0xFFFFFFFF)


def intel_host():
    try:
        return "GenuineIntel" in open("/proc/cpuinfo").read()
    except OSError:
        return False


class RecordedReference:
    def __init__(self, port, shim, live=None, record=False):
        self.port, self.shim, self.live, self.record = port, shim, live, record
        if record:
            self.records = {}
        else:
            with open(RECORDS) as f:
                self.records = json.load(f)["records"]

    def source(self):
        return "the reference build (oracle/_ref/libdmc_ref.so)" if self.live else "the C port (oracle/dmc_oracle.c)"

    def set_num_threads(self, n):
        (self.live or self.port).set_num_threads(n)

    def _call(self, name, args, kwargs):
        if self.live is not None:
            return getattr(self.live, name)(*args, **kwargs)
        if name in SHIM_CALLS:
            return getattr(self.shim, name)(*args, **kwargs)
        kw = {k: v for k, v in kwargs.items() if k != "inplace"}     # in place or not, the reference's result is the same
        return getattr(self.port, "blur_remove_minmax" if name == "blur_remove_minmax_base" else name)(*args, **kw)

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)

        def call(*args, **kwargs):
            if name in HOST_DEPENDENT and not intel_host():
                pytest.skip("the reference's rcp projection was recorded on an Intel host")
            out = self._call(name, args, kwargs)
            key, got = call_key(name, args, kwargs), output_crc(out)
            if self.record:
                self.records[key] = got
            else:
                want = self.records.get(key)
                assert want is not None, "no recorded reference output for %s%r" % (name, tuple(_enc(a) for a in args))
                assert got == want, "%s: output of %s differs from the recorded reference output" % (name, self.source())
            return out
        return call

    def save(self):
        with open(RECORDS, "w") as f:
            json.dump({"_doc": "CRC-32 of the reference build's output for each call the ref tests make (tests/_recorded_ref.py)",
                       "_recorded_from": self.source(), "records": self.records}, f, indent=0, sort_keys=True)
            f.write("\n")
