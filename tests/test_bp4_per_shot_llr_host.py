"""Host-side pieces of bp4_osd per-shot priors (no GPU): the C-ABI declarations and the Python bindings' export list."""
import os

from conftest import ROOT

BP4_LLR_SYMBOLS = ("swd_bp4_decode_batch_host_llr", "swd_bp4_decode_batch_device_llr", "swd_bp4_camel_decode_batch_host_llr",
                   "swd_bp4_camel_decode_batch_device_llr")


def test_bp4_per_shot_entry_points_declared():
    header = open(os.path.join(ROOT, "include", "swd_b200.h")).read()
    for sym in BP4_LLR_SYMBOLS:
        assert sym + "(" in header, sym
        decl = header[header.index(sym + "("):]
        decl = decl[:decl.index(";")]
        assert "const double *" in decl and "channel_llr" in decl, sym       # the five prior planes


def test_bp4_per_shot_entry_points_exported():
    from slidingwindowdecoder_b200 import _lib
    for sym in BP4_LLR_SYMBOLS:
        assert sym in _lib.EXPORTS, sym
