"""CIF timestamps (funasr_b200/timestamps.py) against golden vectors produced by the reference's own
ts_prediction_lfr6_standard (oracle/make_timestamp_golden.py), and against the live reference when it is present."""
import copy
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN

from funasr_b200 import timestamps as TS


def _cases():
    with open(os.path.join(GOLDEN, "timestamps.json")) as f:
        return json.load(f)


def test_timestamps_match_reference_golden():
    cases = _cases()
    assert len(cases) >= 100
    n_nonempty = 0
    for c in cases:
        first, second = np.array(c["first"], np.float32), np.array(c["second"], np.float32)
        txt, res = TS.ts_prediction_lfr6_standard(first, second, c["chars"], vad_offset=c["vad_offset"], upsample_rate=c["upsample_rate"])
        assert res == c["res"]              # integer milliseconds: exact
        assert txt == c["txt"]
        # the model classes ask for the stamps only (want_text=False): same stamps, no string
        assert TS.ts_prediction_lfr6_standard(first, second, c["chars"], vad_offset=c["vad_offset"], upsample_rate=c["upsample_rate"],
                                              want_text=False) == ("", c["res"])
        n_nonempty += bool(res)
    assert n_nonempty > len(cases) // 2


def test_cif_wo_hidden_is_the_running_integral():
    a = np.array([0.4, 0.7, 0.2, 0.9, 0.05], np.float32)
    f = TS.cif_wo_hidden(a, 1.0)
    assert np.allclose(f, [0.4, 1.1, 0.3, 1.2, 0.25], atol=1e-6)
    assert TS.ts_prediction_lfr6_standard(a, a, []) == ("", [])


def test_timestamps_against_live_reference_if_available():
    """The Paraformer call of the reference's ts_prediction_lfr6_standard on 50 seeded cases: its outputs as stored in
    tests/golden/live_host.json (oracle/make_live_golden.py) and, when the reference is importable, a fresh run of it."""
    import make_live_golden as mk
    import ref_shim
    with open(os.path.join(GOLDEN, "live_host.json"), encoding="utf8") as f:
        runs = [json.load(f)["timestamps"]]
    if ref_shim.reference_available():
        ref_shim.import_reference()
        runs.append(mk.run_timestamps())
    for want in runs:
        assert len(want) == 50
        for (a, peaks, chars), (w_txt, w_stamps) in zip(mk.timestamp_inputs(), want):
            got = TS.paraformer_timestamps(peaks, a, copy.copy(chars))
            assert got[1] == w_stamps and got[0] == w_txt


def test_stamps_only_path_equals_the_labelled_walk():
    """want_text=False takes a vectorised route; it must return the labelled walk's stamps in every regime: fire count equal to /
    above / below the token count (re-integration), tokens cut at 12 frames (incl. the last one), leading / trailing silence or none,
    a vocabulary entry spelled "<sil>", a VAD offset, upsampled (x3) and plain frames, a single fire, no fire at all."""
    rng = np.random.default_rng(5)
    n_checked = n_cut_last = 0
    for trial in range(600):
        T = int(rng.integers(4, 400))
        dens = rng.choice([0.05, 0.15, 0.3, 0.6])
        a = (rng.random(T).astype(np.float32) * np.float32(2 * dens)).astype(np.float32)
        if trial % 7 == 0:
            a[: T // 3] = 0                                      # long leading silence
        if trial % 5 == 0:
            a[-(T // 4):] = 0                                    # long trailing silence
        if trial % 11 == 0:
            a[T // 2: T // 2 + 20] = 0                           # a gap: the token before it is cut at 12 frames
        peaks = TS.cif_wo_hidden(a, 1.0)
        n_fire = int((peaks >= np.float32(1 - 1e-4)).sum())
        n_tok = max(0, n_fire - 1 + int(rng.integers(-2, 3)))
        chars = ["c%d" % i for i in range(n_tok)]
        if chars and trial % 13 == 0:
            chars[int(rng.integers(0, len(chars)))] = "<sil>"
        for kw in ({"upsample_rate": 1}, {"upsample_rate": 3, "vad_offset": 12340}, {"upsample_rate": 1, "vad_offset": 250.5}):
            for first, second in ((peaks, a), (a, peaks)):       # the Paraformer call order and the BiCif one
                want = TS.ts_prediction_lfr6_standard(first, second, list(chars), **kw)
                got = TS.ts_prediction_lfr6_standard(first, second, list(chars), want_text=False, **kw)
                assert got == ("", want[1]), (trial, kw)
                n_checked += 1
        tr = peaks
        fires = np.flatnonzero(tr >= np.float32(1 - 1e-4))
        n_cut_last += int(fires.size >= 2 and fires[-1] - fires[-2] > 12)
    assert n_checked == 3600 and n_cut_last > 5


def test_native_cif_wo_hidden_equals_the_python_loop_bit_for_bit():
    """fa_cif_wo_hidden_host (the library's host code) against the numpy-scalar loop it replaces: identical fp32 traces."""
    rng = np.random.default_rng(9)
    for trial in range(500):
        n = int(rng.integers(0, 600))
        a = (rng.random(n) ** int(rng.choice([1, 2, 3])) * float(rng.choice([0.3, 1.0, 2.5]))).astype(np.float32)
        for thr in (1.0, 1.0 - 1e-4, 0.5):
            assert np.array_equal(TS.cif_wo_hidden(a, thr), TS.cif_wo_hidden_py(a, thr))
    assert TS.cif_wo_hidden(np.zeros(0, np.float32), 1.0).shape == (0,)
    nan = TS.cif_wo_hidden(np.array([0.5, np.nan, 0.7], np.float32), 1.0)
    assert nan[0] == np.float32(0.5) and np.isnan(nan[1:]).all()


@pytest.mark.parametrize("name", ["bicif_large_single", "bicif_tiny_ragged3"])
def test_model_class_route_reproduces_the_bicif_golden_timestamps(name):
    """The route BiCifParaformerB200.inference takes on the host (stamps only, native re-integration) over the REFERENCE's own
    upsampled weights / fires: the reference's timestamps (bicif_paraformer/model.py:402-407), integer milliseconds exact."""
    from conftest import gold_stamps
    d = np.load(os.path.join(GOLDEN, name + ".npz"))
    want, pos = gold_stamps(d), 0
    for b in range(d["us_alphas"].shape[0]):
        k = int(d["ids_len"][b])
        ids = d["ids_flat"][pos: pos + k]
        pos += k
        n = int(d["enc_lens"][b]) * 3
        got = TS.ts_prediction_lfr6_standard(d["us_alphas"][b][:n], d["us_peaks"][b][:n], [str(t) for t in ids], want_text=False)
        assert got == ("", want[b])
