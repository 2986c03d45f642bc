"""CPU tests of the bf16x3 precision mode's host side: mode names, the FMT_MODE variable, the node widgets and the C-ABI mode id."""
import os
import re
import sys

import pytest

from __graft_entry__ import ROOT, load_package


@pytest.fixture(scope="module")
def pkg():
    return load_package()


def test_bf16x3_mode_resolution(pkg, monkeypatch):
    monkeypatch.delenv("FMT_MODE", raising=False)
    assert "bf16x3" in pkg.PRECISION_MODES
    assert pkg.resolve_mode("bf16x3") == "bf16x3" and pkg.resolve_mode("BF16X3") == "bf16x3"
    monkeypatch.setenv("FMT_MODE", "bf16x3")
    assert pkg.resolve_mode(None) == "bf16x3" and pkg.resolve_mode("default") == "bf16x3" and pkg.resolve_mode("bf16") == "bf16"
    with pytest.raises(ValueError):
        pkg.resolve_mode("bf16x2")


def test_precision_widgets_offer_bf16x3(pkg):
    for cls in (pkg.FloatSampleMotionSequenceRD_VA, pkg.FloatSampleMotionSequenceRD, pkg.FloatProcess):
        choices, opts = cls.INPUT_TYPES()["optional"]["precision"]
        assert list(choices) == ["default", "bf16", "fp32", "bf16x3"] and opts["default"] == "default"
        assert "bf16x3" in opts["tooltip"]
    assert "precision" not in pkg.FloatApplyAudioProjection.INPUT_TYPES()["optional"]   # reachable through _mode only


def test_bf16x3_maps_to_mode_id_2(pkg):
    cabi = sys.modules[pkg.__name__ + "._cabi"]
    audio = sys.modules[pkg.__name__ + ".audio"]
    hdr = open(os.path.join(ROOT, "include", "fmt_b200.h")).read()
    assert re.search(r"FMT_MODE_BF16X3\s*=\s*2\b", hdr)
    assert re.search(r"#define FMT_ABI_VERSION 2\b", hdr) and cabi.FMT_ABI_VERSION == 2
    assert cabi.FMT_MODE_BF16X3 == 2 and cabi.MODE_IDS == {"bf16": 0, "fp32": 1, "bf16x3": 2}
    assert set(cabi.MODE_IDS) == set(pkg.PRECISION_MODES) and audio._MODES["bf16x3"] == 2
