"""Every environment switch the library reads is documented in DESIGN §8a and has a parity entry in test_gpu_switches.SWITCHES, so a new
kernel variant cannot land reachable but unchecked.  No GPU needed: this reads the sources."""
import glob
import os
import re

from test_gpu_switches import SWITCHES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# read by the library but not kernel variants
NOT_VARIANTS = {
    "SVA_DEBUG": "prints launch shapes to stderr; changes no launch",
    "SVA_NCCL_LIB": "path of the NCCL library to load; no kernel of this library",
    "SVA_ROWS_TIMEOUT_MS": "the row pipeline's hand-off time-out; its validation is tested in test_gpu_switches::test_bad_rows_timeout_is_refused",
}


def _read_by_library():
    names = set()
    for path in glob.glob(os.path.join(ROOT, "stereovisionarray_b200", "csrc", "*.cu")):
        src = open(path).read()
        names |= set(re.findall(r'getenv\("(SVA_[A-Z0-9_]+)"\)', src))
        names |= set(re.findall(r'read_switch\("(SVA_[A-Z0-9_]+)"', src))  # sva_create's validated reads (sva_ctx.cu)
    return names


def _design_8a():
    text = open(os.path.join(ROOT, "DESIGN.md")).read()
    start = text.index("## 8a.")
    end = text.index("\n## ", start + 1)
    return text[start:end]


def test_every_switch_is_documented_and_checked():
    read = _read_by_library()
    assert "SVA_BOX_OCC" in read and "SVA_SGM_PACE" in read, "the source scan found nothing: %s" % sorted(read)
    doc = _design_8a()
    undocumented = sorted(n for n in read - set(NOT_VARIANTS) if "`%s`" % n not in doc)
    assert not undocumented, "read by the library, missing from DESIGN §8a: %s" % undocumented
    covered = {k for e in SWITCHES for k in e.env}
    unchecked = sorted(n for n in read - set(NOT_VARIANTS) if n not in covered)
    assert not unchecked, "switches without an entry in test_gpu_switches.SWITCHES: %s" % unchecked


def test_documented_switches_exist():
    """the reverse: §8a and the table name nothing the library no longer reads"""
    read = _read_by_library()
    stale = sorted(n for n in set(re.findall(r"`(SVA_[A-Z0-9_]+)", _design_8a())) - read if not n.startswith("SVA_ERR_"))
    assert not stale, "DESIGN §8a documents switches the library does not read: %s" % stale
    assert {k for e in SWITCHES for k in e.env} <= read
    assert set(NOT_VARIANTS) <= read


def test_every_entry_reaches_its_variant_somewhere():
    from test_gpu_switches import GEOM, ROWS
    for e in SWITCHES:
        assert e.cases and all(c in GEOM or c in ROWS for c in e.cases), e
        assert e.witness is not None or e.why, "an entry without a witness says why its cases reach the variant: %s" % (e.env,)
        assert e.stages in ("K1a", "K1b", "K2", "K3", "stream"), e
