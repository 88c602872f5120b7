"""The library reads its environment knobs and never writes them: a self-check that forces a layout, a key width or a pair
window through its arguments leaves the caller's own setting of that knob in place.  Each case runs in a child process,
whose environment it changes through libc (os.environ is only Python's copy of it)."""
import subprocess
import sys

import pytest

from conftest import ROOT

_CHILD = r"""
import ctypes as C, os, sys
import numpy as np
sys.path.insert(0, %r)
import rowbowt_b200 as rb
from oracle import rbformats as F
libc = C.CDLL(None)
libc.getenv.restype = C.c_char_p
lib, case, knob = rb.lib(), sys.argv[1], sys.argv[2].encode()
pre = os.path.join(%r, "tests", "golden", "tiny", "tiny")
libc.setenv(knob, sys.argv[3].encode(), 1)
a, b, c = C.c_uint64(), C.c_uint64(), C.c_uint64()
if case == "layout":
    rc = lib.rbg_selftest_layout(pre.encode(), 0 | (5 << 16), 1, C.byref(a), C.byref(b), C.byref(c))
elif case == "toehold":
    rc = lib.rbg_selftest_toehold(pre.encode(), 3, C.byref(a), C.byref(b))
else:
    bwt = F.read_rbwt(pre + ".rbwt")
    heads = np.ascontiguousarray(bwt.heads, np.uint8)
    lens = np.ascontiguousarray(bwt.lens, np.uint64)
    rc = lib.rbg_selftest_pair(int(lens.sum()), heads.ctypes.data, lens.ctypes.data, len(heads), 64, 7, None,
                               C.byref(a), C.byref(b), C.byref(c))
print(rc, a.value, (libc.getenv(knob) or b"<unset>").decode())
"""


@pytest.mark.parametrize("case,knob,value", [
    ("layout", "RBG_LAYOUT", "4"),              # the self-check forces layout 5
    ("toehold", "RBG_TOEHOLD_SHIFT", "5"),      # ... forces buckets of 2^3 rows
    ("pair", "RBG_LAYOUT", "4"),                # ... builds layout 5 under the pair directory
])
def test_selftests_leave_the_callers_knobs_alone(case, knob, value):
    p = subprocess.run([sys.executable, "-c", _CHILD % (ROOT, ROOT), case, knob, value], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    rc, checked, after = p.stdout.split()
    assert rc == "0" and int(checked) > 0
    assert after == value
