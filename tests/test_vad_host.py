"""CPU: the FSMN-VAD host logic (funasr_b200/vad.py: end-point detector, the reference's chunked frame delivery, the dynamic
end-silence schedule) and the oracle restatement of the VAD scores (oracle/vad_oracle.py) against golden vectors produced by the
UNMODIFIED reference (oracle/make_vad_golden.py: FsmnVADStreaming + WavFrontendOnline through AutoModel.generate)."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN

import vad_oracle as VO
from funasr_b200 import synth, vad

# must match oracle/make_vad_golden.py:VAD_CASES
VAD_CASES = {
    "vad_30s": (30.0, 1, [(3.0, 2.5), (1.5, 0.4), (4.0, 3.0), (2.0, 2.2)], {}),
    "vad_130s": (130.0, 2, [(70.0, 2.5), (5.0, 0.3), (20.0, 2.1), (10.0, 3.0)], {}),
    "vad_fixed800": (30.0, 3, [(2.0, 1.0), (3.0, 0.5), (1.0, 1.5)], {"max_end_silence_time": 800}),
    "vad_random45": (45.0, 4, None, {}),
    "vad_short": (1.2, 5, [(5.0, 0.1)], {}),
    "vad_silence": (3.0, 6, [(0.0, 9.0)], {}),
}


def _gold(name):
    return dict(np.load(os.path.join(GOLDEN, name + ".npz")))


@pytest.mark.parametrize("name", list(VAD_CASES))
def test_detector_reproduces_reference_segments_from_reference_scores(name):
    """Given the reference's OWN per-frame silence posteriors and frame energies, the restated detector returns the reference's
    segments exactly (integer milliseconds) — incl. the 130 s case that crosses two 60 s chunk boundaries (frame delivery per
    chunk, dynamic end-silence schedule, the 60 s maximum segment length) and the fixed-threshold case."""
    g = _gold(name)
    kw = VAD_CASES[name][3]
    got = vad.detect_segments(g["sil_prob"].tolist(), g["decibel"].tolist(), int(g["n_samples"]), **kw)
    assert got == g["segments"].tolist()
    assert [c for c in vad.chunk_frame_counts(int(g["n_samples"])) if c > 0] == g["chunk_frames"].tolist()


@pytest.mark.parametrize("name", ["vad_30s", "vad_130s", "vad_short"])
def test_vad_oracle_scores_match_reference(name):
    """The whole-waveform restatement of frontend + FSMN equals what the reference computed chunk by chunk through its stateful
    online frontend and encoder caches."""
    g = _gold(name)
    seconds, seed, pattern, _ = VAD_CASES[name]
    wav = synth.make_vad_wav(seconds, seed, pattern)
    assert wav.numel() == int(g["n_samples"])
    o = VO.vad_scores(wav, synth.make_vad_state_dict(synth.VAD_DEFAULT, 0), synth.make_vad_cmvn(0))
    assert o["sil_prob"].numel() == g["sil_prob"].shape[0]
    assert np.abs(o["sil_prob"].numpy() - g["sil_prob"]).max() <= 2e-5
    assert np.abs(o["scores"][g["score_rows"].tolist()].numpy() - g["score_sel"]).max() <= 2e-5
    assert np.abs(o["decibel"].numpy() - g["decibel"]).max() <= 1e-3
    # and the end-to-end CPU chain oracle scores -> detector reproduces the reference's segments
    got = vad.detect_segments(o["sil_prob"].tolist(), o["decibel"].tolist(), wav.numel(), **VAD_CASES[name][3])
    assert got == g["segments"].tolist()


def test_chunk_frame_counts_cover_every_frame():
    for n in [399, 400, 559, 560, 1200, 16000, 959999, 960000, 960001, 960399, 960400, 1919999, 1920000, 2080000, 5000000]:
        c = vad.chunk_frame_counts(n)
        assert len(c) == n // 960000 + 1
        total = vad.num_frames(n)
        assert sum(c) == (total if total >= 3 else 0), (n, c, total)      # fewer than lfr_m - 2 frames: the online LFR never emits


def test_merge_vad_matches_reference_function():
    segs = [[0, 2450], [2990, 7940], [8970, 11440], [11990, 16920], [17970, 20440], [21030, 25940], [27000, 40000]]
    assert vad.merge_vad(segs, 15000) == [[0, 11990], [11990, 25940], [25940, 40000]]
    assert vad.merge_vad([[5, 9]], 15000) == [[5, 9]]
    # the reference's funasr.utils.vad_utils.merge_vad on 50 seeded segment lists (tests/golden/live_host.json, oracle/make_live_golden.py)
    import make_live_golden as mk
    want = _live_host()["merge_vad"]
    assert len(want) == 50
    for t, w in zip(mk.merge_vad_inputs(), want):
        assert vad.merge_vad([list(x) for x in t], 15000) == w


def _live_host():
    with open(os.path.join(GOLDEN, "live_host.json"), encoding="utf8") as f:
        return json.load(f)


def _flat_decibels(n_samples):
    """Frame energies of make_vad_cpp_golden.flat_wave: every 400-sample frame holds 400 x 0.05^2."""
    frames = vad.num_frames(n_samples)
    return [10.0 * float(np.log10(np.float32(400 * np.float32(0.05) ** 2) + 1e-6))] * frames


def test_detector_matches_the_reference_runtimes_compiled_cpp_detector():
    """Second, independent pin of the end-point state machine: the reference's C++ runtime carries its own implementation
    (runtime/onnxruntime/src/e2e-vad.h, header-only; compiled from the reference tree by oracle/knf/Makefile and called like
    fsmn-vad.cpp:245-249).  It has no dynamic end-silence schedule, so funasr_b200/vad.py is run with a fixed max_end_silence_time.
    Checked against the committed outputs of that detector (tests/golden/vad_cpp_detector.npz, oracle/make_vad_cpp_golden.py), on
    seeded random posteriors (incl. recordings beyond the 60 s chunk / segment limit) against its stored segments
    (tests/golden/live_host.json, oracle/make_live_golden.py) and — when the compiled library is present — against a live run, and on the
    Python reference's own scores of the fixed-schedule golden cases."""
    import knf_ref
    import make_live_golden as mk
    g = np.load(os.path.join(GOLDEN, "vad_cpp_detector.npz"))
    for i, (n, mes, thr10) in enumerate(g["meta"].tolist()):
        sp = (g["sil_prob_%d" % i].astype(np.float32) / 1024).tolist()
        got = vad.detect_segments(sp, _flat_decibels(n), n, max_end_silence_time=mes, speech_noise_thres=thr10 / 10)
        assert got == g["segments_%d" % i].tolist(), i
    stored = _live_host()["vad_cpp"]
    have = knf_ref.build()
    for it, (n, sp, wav, mes, thr) in enumerate(mk.vad_cpp_random_inputs()):
        want = stored["random"][it]
        if have:
            assert knf_ref.vad_segments(sp, wav, mes, 60000, thr) == want, it
        db = VO.frame_decibels(torch.from_numpy(wav)).double().tolist()
        assert vad.detect_segments(sp.tolist(), db, n, max_end_silence_time=mes, speech_noise_thres=thr) == want, it
    for name in mk.VAD_GOLDEN_CASES:                                 # the Python reference's scores through the C++ detector
        seconds, seed, pattern, _ = VAD_CASES[name]
        gg = _gold(name)
        assert stored["golden_scores"][name] == gg["segments"].tolist()
        if have:
            wav = synth.make_vad_wav(seconds, seed, pattern).numpy()
            assert knf_ref.vad_segments(gg["sil_prob"], wav, 800, 60000, 0.6) == gg["segments"].tolist()


@pytest.mark.parametrize("name", list(VAD_CASES))
def test_native_detector_reproduces_reference_segments(name):
    """fa_vad_detect_segments (csrc/vad_detector.cpp, the state machine the product runs) on the reference's own scores: the
    reference's segments, and the same as the Python restatement — fp64 and fp32 inputs (the GPU delivers fp32)."""
    g = _gold(name)
    kw = VAD_CASES[name][3]
    n = int(g["n_samples"])
    assert vad.detect_segments_native(g["sil_prob"], g["decibel"], n, **kw) == g["segments"].tolist()
    both = np.stack([g["sil_prob"].astype(np.float32), g["decibel"].astype(np.float32)])
    assert vad.detect_segments_native(both[0], both[1], n, **kw) == vad.detect_segments(both[0].tolist(), both[1].tolist(), n, **kw)


def test_native_detector_equals_the_python_walk_on_random_recordings():
    """Dynamic and fixed end-silence schedules, explicit thresholds, option changes, recordings past several 60 s chunks, empty input;
    posteriors outside (0, 1) are an error in both (math.log raises in the reference)."""
    import make_vad_cpp_golden as mk
    rng = np.random.default_rng(11)
    opts = [None, vad.VadOptions(do_extend=0), vad.VadOptions(detect_mode=0, max_start_silence_time=500), vad.VadOptions(max_single_segment_time=5000),
            vad.VadOptions(window_size_ms=300, sil_to_speech_time_thres=200, speech_to_sil_time_thres=100), vad.VadOptions(decibel_thres=-1.0, snr_thres=-3.0)]
    for it in range(120):
        n, sp, wav, mes, thr = mk.random_case(rng, 200.0 if it % 10 == 0 else 30.0)
        wav = (wav * rng.uniform(0.2, 2.0, size=wav.size).astype(np.float32)) if it % 3 == 0 else wav      # varying frame energies
        db = VO.frame_decibels(torch.from_numpy(wav)).double().numpy()
        o = opts[it % len(opts)]
        for kw in ({}, {"max_end_silence_time": mes, "speech_noise_thres": thr}, {"dynamic_silence": True, "speech_noise_thres": thr},
                   {"chunk_ms": 20000}):
            assert vad.detect_segments_native(sp, db, n, o, **kw) == vad.detect_segments(sp.tolist(), db.tolist(), n, o, **kw), (it, kw)
    assert vad.detect_segments_native(np.zeros(0), np.zeros(0), 300) == [] == vad.detect_segments([], [], 300)
    from funasr_b200._abi import FunasrB200Error
    with pytest.raises(FunasrB200Error):
        vad.detect_segments_native(np.array([0.5, 0.0, 0.5]), np.zeros(3), 400 + 160 * 4)
    with pytest.raises(ValueError):
        vad.detect_segments([0.5, 0.0, 0.5], [0.0] * 3, 400 + 160 * 4)
