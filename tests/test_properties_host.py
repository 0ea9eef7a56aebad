"""Property tests (hypothesis) of the host-side logic around the hot path: utterance sharding, length bucketing, frame
arithmetic and the CIF timestamp routine.  CPU only."""
import json
import os

import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

from conftest import GOLDEN

from funasr_b200.batching import bucket_by_length, padding_efficiency, run_bucketed
from funasr_b200.engine import num_lfr_frames
from funasr_b200.sharding import shard_utterances
from funasr_b200 import timestamps as TS

durs = st.lists(st.floats(min_value=0.03, max_value=120.0, allow_nan=False), min_size=0, max_size=200)


@settings(max_examples=200, deadline=None)
@given(durs, st.integers(min_value=1, max_value=8))
def test_sharding_is_a_balanced_partition(d, world):
    shards = shard_utterances(d, world)
    flat = sorted(i for s in shards for i in s)
    assert flat == list(range(len(d)))                               # every utterance exactly once
    sizes = [len(s) for s in shards]
    assert max(sizes) - min(sizes) <= 1                              # snake deal: sizes differ by at most one
    if len(d) >= 2 * world:                                          # work is balanced to within the longest utterance
        load = [sum(d[i] for i in s) for s in shards]
        assert max(load) - min(load) <= max(d) + 1e-9


@settings(max_examples=200, deadline=None)
@given(st.lists(st.integers(min_value=400, max_value=16000 * 90), min_size=1, max_size=300),
       st.integers(min_value=1, max_value=64), st.integers(min_value=1500, max_value=64 * 500))
def test_bucketing_respects_caps_and_covers_everything(ns, max_batch, max_frames):
    batches = bucket_by_length(ns, max_batch, max_frames)
    assert sorted(i for b in batches for i in b) == list(range(len(ns)))
    for b in batches:
        assert 1 <= len(b) <= max_batch
        t_max = max(num_lfr_frames(ns[i]) for i in b)
        assert len(b) == 1 or len(b) * t_max <= max_frames           # a single over-long utterance still gets its own batch
    assert 0.0 < padding_efficiency(ns, batches) <= 1.0
    out = run_bucketed([np.zeros(n, np.float32) for n in ns], lambda ws: [[len(w)] for w in ws], max_batch, max_frames)
    assert out == [[n] for n in ns]                                  # results come back in input order


@given(st.integers(min_value=0, max_value=16000 * 600))
def test_frame_arithmetic_matches_the_reference_formulas(n):
    win = min(400, n)                                                # wav_frontend.py:174: frame_length = min(25 ms, len / fs)
    m = 1 + (n - win) // 160 if n >= 2 else 0                        # kaldi.py _get_strided, snip_edges (window_size >= 2 asserted)
    t = int(np.ceil(m / 6))                                          # wav_frontend.py:73
    assert num_lfr_frames(n) == t


@settings(max_examples=150, deadline=None)
@given(st.lists(st.floats(min_value=0.0, max_value=0.9375, allow_nan=False, width=32), min_size=8, max_size=300), st.integers(1, 40),
       st.sampled_from([1, 3]), st.sampled_from([0.0, 250.0]))
def test_timestamps_are_ordered_and_inside_the_utterance(alphas, n_tok, rate, offset):
    a = np.array(alphas, dtype=np.float32)
    peaks = TS.cif_wo_hidden(a, 1.0)
    txt, res = TS.ts_prediction_lfr6_standard(a, peaks, ["t%d" % i for i in range(n_tok)], vad_offset=offset, upsample_rate=rate)
    end_ms = (len(a) * 60.0 / rate) + offset
    prev = -10**9
    for s, e in res:
        assert s <= e and s >= prev - 1                                # monotone up to the 1 ms integer truncation
        assert e <= end_ms + 1
        prev = s
    assert len(res) <= max(n_tok, 1) + 1


def test_hotword_list_follows_reference_seg_dict_rules(tmp_path):
    """funasr_b200.hotwords.generate_hotwords_list against hand-derived expectations and the stored outputs of the reference's own
    function (contextual_paraformer/model.py:528-660): seg_dict lookup (lower-cased), per-character
    fallback for CJK / digit words, <unk> for the rest, [sos] terminator; .txt files and plain strings."""
    from funasr_b200.hotwords import generate_hotwords_list, seg_tokenize

    class Tok:
        vocab = {"<unk>": 9, "he@@": 3, "llo": 4, "你": 5, "好": 6, "7": 7, "gpu": 8}

        def tokens2ids(self, toks):
            return [self.vocab.get(t, self.vocab["<unk>"]) for t in toks]

    class Fe:
        cmvn_file = None

    mvn = tmp_path / "am.mvn"
    mvn.write_text("x")
    (tmp_path / "seg_dict").write_text("hello he@@ llo\n你 你\n好 好\n7 7\ngpu gpu\n", encoding="utf8")
    fe = Fe()
    fe.cmvn_file = str(mvn)
    sd = {"hello": "he@@ llo", "你": "你", "好": "好", "7": "7", "gpu": "gpu"}
    assert seg_tokenize(["Hello", "你好7", "wörld", "你坏"], sd) == ["he@@", "llo", "你", "好", "7", "<unk>", "你", "<unk>"]
    got = generate_hotwords_list("Hello 你好 GPU xyz", Tok(), fe, sos=1)
    assert got == [[3, 4], [5, 6], [8], [9], [1]]
    txt = tmp_path / "hw.txt"
    txt.write_text("hello 你好\ngpu\n", encoding="utf8")
    assert generate_hotwords_list(str(txt), Tok(), fe, sos=1) == [[3, 4, 5, 6], [8], [1]]
    assert generate_hotwords_list(None, Tok(), fe, sos=1) is None
    # without a seg_dict beside the cmvn file the words go to the tokenizer unchanged
    assert generate_hotwords_list("gpu Hello", Tok(), Fe(), sos=1) == [[8], [9], [1]]
    with pytest.raises(ValueError):
        generate_hotwords_list("http://example.com/hw.txt", Tok(), fe, sos=1)
    # the reference's own function on the same string and file (tests/golden/live_host.json, oracle/make_live_golden.py)
    import make_live_golden as mk
    assert Tok.vocab == mk.HotwordTokenizer.vocab
    assert ((tmp_path / "seg_dict").read_text(encoding="utf8"), txt.read_text(encoding="utf8")) == (mk.HOTWORD_SEG_DICT, mk.HOTWORD_FILE)
    with open(os.path.join(GOLDEN, "live_host.json"), encoding="utf8") as f:
        want = json.load(f)["hotwords"]
    assert generate_hotwords_list(mk.HOTWORD_STRING, Tok(), fe, sos=1) == want["string"]
    assert generate_hotwords_list(str(txt), Tok(), fe, sos=1) == want["file"]


def test_bench_flop_model_matches_the_survey_figures():
    """bench.py's roofline numerators are SURVEY.md §8(d)'s algorithmic FLOPs: encoder 183.2 + predictor 0.787 + decoder
    8.389 + 0.1132 N GFLOP per 30 s utterance (T = 500) = 206 GFLOP at N = 120; SenseVoiceSmall (T = 504) = 272 GFLOP."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    assert abs(bench.flops_paraformer(500, 0) / 1e9 - (183.2 + 0.787 + 8.389)) < 0.1
    assert abs((bench.flops_paraformer(500, 1) - bench.flops_paraformer(500, 0)) / 1e9 - 0.1132) < 1e-3
    assert abs(bench.flops_paraformer(500, 120) / 1e9 - 206.0) < 0.5
    assert abs(bench.flops_sensevoice(504) / 1e9 - 272.0) < 1.0
    # every bucket limit is a whole number of 30 s utterances of 500 frames
    assert all(mf % 500 == 0 and mb >= mf // 500 for mb, mf in bench.BUCKET_LIMITS.values())


def test_bench_stage_tap_comparison():
    """bench.py's parity block also compares the stage taps (BASELINE.md §3.4): the GPU tensors are subsampled like the oracle's dump,
    the acoustic rows cut at the largest token count, bars as in the GPU parity tests; missing taps (config 5 has no feats / alphas in
    its oracle output) are skipped, a shape disagreement is reported instead of raised."""
    import importlib.util
    import os
    import torch
    spec = importlib.util.spec_from_file_location("bench_mod2", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    g = torch.Generator().manual_seed(0)
    full = {"feats": torch.randn(2, 50, 560, generator=g), "enc": torch.randn(2, 50, 512, generator=g), "alphas": torch.rand(2, 51, generator=g),
            "acoustic": torch.randn(2, 17, 512, generator=g)}
    dump = {"tap_" + k: (v[:, ::bench.TAP_STRIDES[k]] if bench.TAP_STRIDES[k] > 1 else v).numpy() for k, v in full.items()}
    dump["token_num"] = np.array([17, 9])
    got = dict(full)
    got["acoustic"] = torch.cat([full["acoustic"], torch.zeros(2, 34, 512)], 1)            # the device buffer is [B, T + 1, 512]
    r = bench.compare_taps(dump, got)
    assert set(r) == {"feats", "enc", "alphas", "acoustic"} and all(v["within"] and v["max_abs"] == 0.0 for v in r.values())
    got["enc"] = full["enc"] * 1.01
    got["alphas"] = full["alphas"] + 2e-4
    r = bench.compare_taps(dump, got)
    assert not r["enc"]["within"] and not r["alphas"]["within"] and r["feats"]["within"]
    del dump["tap_feats"], dump["tap_alphas"]
    assert set(bench.compare_taps(dump, dict(full, acoustic=got["acoustic"]))) == {"enc", "acoustic"}
    assert "error" in bench.compare_taps(dump, dict(full, enc=full["enc"][:, :40], acoustic=got["acoustic"]))["enc"]


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: every utterance's ids in input order, padded with -1, lengths beside them, float64 (ids exact)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod3", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    bench.dump_outputs(str(tmp_path / "out"), [[5, 8404, 3], [], [7]])
    ids, lens = np.load(tmp_path / "out" / "token_ids.npy"), np.load(tmp_path / "out" / "token_lens.npy")
    assert ids.dtype == np.float64 and lens.dtype == np.float64
    assert ids.tolist() == [[5, 8404, 3], [-1, -1, -1], [7, -1, -1]] and lens.tolist() == [3, 0, 1]
