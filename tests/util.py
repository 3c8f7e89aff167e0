import hashlib

import numpy as np

from fdreadoutlibs_b200 import frames as F

FIELDS = ("time_start", "time_peak", "time_over_threshold", "adc_integral", "adc_peak", "channel", "link")


def assert_same_tps(got: np.ndarray, want: np.ndarray, what: str = ""):
    """Bit-exact comparison of two TP lists as sorted field tuples."""
    g, w = F.sort_tps(np.asarray(got, dtype=F.TP_DTYPE)), F.sort_tps(np.asarray(want, dtype=F.TP_DTYPE))
    assert g.size == w.size, f"{what}: {g.size} TPs, expected {w.size}"
    for f in FIELDS:
        bad = np.nonzero(g[f] != w[f])[0]
        assert bad.size == 0, f"{what}: field {f} differs at sorted index {bad[0]}: got {g[bad[0]]}, want {w[bad[0]]}"


def digest(name: str, a: np.ndarray) -> np.ndarray:
    """SHA-256 of an output array, a TP list in canonical order."""
    if name == "tps":
        a = F.sort_tps(np.asarray(a, dtype=F.TP_DTYPE))
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), dtype=np.uint8)


def assert_same_as_reference(got: dict, ref, key: str):
    """got: {name: array} for the input `key` of tests/cases.py:reference_runs; ref: tests/golden/reference_outputs.npz, which
    holds each array either as it is ("<key>__<name>") or, when it is large, as its length and digest."""
    for name, a in got.items():
        k = f"{key}__{name}"
        if k in ref.files:
            if name == "tps":
                assert_same_tps(a, ref[k], key)
            else:
                assert a.shape == ref[k].shape and (a == ref[k]).all(), f"{key}: {name} differs from the reference"
        else:
            assert a.size == ref[k + "_count"][0], f"{key}: {a.size} {name}, the reference has {ref[k + '_count'][0]}"
            assert (digest(name, a) == ref[k + "_sha256"]).all(), f"{key}: {name} differs from the reference (digest)"


def oracle_config(case, B):
    from fdreadoutlibs_b200.api import ALGORITHMS

    return B.make_config(fmt=case["fmt"], algorithm=ALGORITHMS[case["algorithm"]], threshold=case["threshold"],
                         acc_limit=case.get("acc_limit", 10), rs_memory_factor=case.get("rs_memory_factor", 8),
                         rs_scale_factor=case.get("rs_scale_factor", 5))
