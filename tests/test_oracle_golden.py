"""CPU: the oracle restatement against the golden vectors produced by the UNMODIFIED reference
(oracle/make_golden.py), and — when /root/reference is present — against the live reference itself."""
import os

import numpy as np
import pytest
import torch

from conftest import (BICIF_CASES, CTX_CASES, GOLDEN, GOLDEN_CASES, SEACO_CASES, SV_CASES, gold_stamps, load_bicif_case, load_case, load_ctx_case,
                      load_seaco_case, load_sv_case,
                      rel_err, state_dict_for)

import paraformer_oracle as O
import ref_shim


def _sub(cfg, t, step):
    return t[:, ::step] if cfg.enc_layers > 10 else t


@pytest.mark.parametrize("name", list(GOLDEN_CASES))
def test_oracle_matches_reference_golden(name):
    cfg, wseed, wavs, cmvn, g = load_case(name)
    p = state_dict_for(cfg, wseed)
    o = O.paraformer_forward(wavs, p, cmvn, cfg.enc_layers, cfg.dec_layers, tail_threshold=cfg.tail_threshold)
    assert o["feat_lens"].tolist() == g["feat_lens"].tolist()
    # same machine class + same torch ops: frontend and encoder are (near) bit-identical to the reference
    assert np.abs(_sub(cfg, o["feats"], 7).numpy() - g["feats"]).max() <= 1e-5
    assert rel_err(_sub(cfg, o["enc"], 7).numpy(), g["enc"]) <= 1e-5
    assert np.abs(o["alphas"].numpy() - g["alphas"]).max() <= 1e-5
    assert o["token_num"].tolist() == g["token_num"].tolist()            # integer outcome: exact
    assert rel_err(_sub(cfg, o["acoustic"], 5).numpy(), g["acoustic"]) <= 1e-4
    lp = o["logp"][:, g["logp_rows"].tolist(), :].numpy()
    assert rel_err(lp, g["logp_sel"]) <= 1e-3                            # contract: logits within 1e-3 rel fp32
    valid = np.arange(g["argmax"].shape[1])[None, :] < g["token_num"][:, None]
    assert (o["logp"].argmax(-1).numpy()[valid] == g["argmax"][valid]).all()
    ids_flat = [t for r in o["ids"] for t in r]
    assert ids_flat == g["ids_flat"].tolist() and [len(r) for r in o["ids"]] == g["ids_len"].tolist()   # bit-exact ids
    assert abs(float(g["batch_data_time"]) - sum(int(x) for x in o["feat_lens"]) * 0.06) < 1e-6


def test_fbank_matches_pinned_torchaudio():
    """Third-party pin: torchaudio.compliance.kaldi.fbank (2.11.0) as WavFrontend calls it (wav_frontend.py:171-181)."""
    ta = pytest.importorskip("torchaudio")
    import torchaudio.compliance.kaldi as kaldi
    from funasr_b200 import synth
    for n, seed, kind in [(16000, 7, "speechlike"), (400, 8, "noise"), (8123, 9, "noise")]:
        w = synth.make_wav(n, seed, kind) * (1 << 15)
        ref = kaldi.fbank(w.unsqueeze(0), num_mel_bins=80, frame_length=25, frame_shift=10, dither=0.0, energy_floor=0.0,
                          window_type="hamming", sample_frequency=16000, snip_edges=True)
        assert torch.equal(ref, O.kaldi_fbank(w))


def test_fbank_matches_the_reference_runtimes_compiled_kaldi_native_fbank():
    """Second, independent pin of the Fbank arithmetic: the reference's vendored kaldi-native-fbank, compiled from the reference
    tree (oracle/knf/Makefile) and driven like its C++ runtime (paraformer.cpp:24-31, :298-312).  Different FFT (Ooura), same
    definition: frame counts equal, log-mel inside the two FFTs' rounding floor.  Checked against the committed fixture and,
    when the compiled library is here, against a live run (which must also reproduce the fixture bit for bit)."""
    from conftest import knf_bound, knf_logmel_cases
    for w, gold, live in knf_logmel_cases():
        mine = O.kaldi_fbank(w * (1 << 15)).double().numpy()
        assert mine.shape == gold.shape                                   # integer: frame count exact
        d = np.abs(mine - gold.astype(np.float64))
        assert (d <= knf_bound(mine)).all(), float((d / knf_bound(mine)).max())
        assert d.mean() <= 2e-5
        if live is not None:
            assert np.array_equal(live, gold)


def test_lfr_equals_reference_formula():
    """apply_lfr restated as a clamped gather == the reference's pad+as_strided construction (wav_frontend.py:63-86)."""
    def ref_lfr(inputs, m, n):
        T = inputs.shape[0]
        T_lfr = int(np.ceil(T / n))
        inputs = torch.vstack((inputs[0].repeat((m - 1) // 2, 1), inputs))
        T = T + (m - 1) // 2
        d = inputs.shape[-1]
        last_idx = (T - m) // n + 1
        num_padding = m - (T - last_idx * n)
        if num_padding > 0:
            num_padding = (2 * m - 2 * T + (T_lfr - 1 + last_idx) * n) / 2 * (T_lfr - last_idx)
            inputs = torch.vstack([inputs] + [inputs[-1:]] * int(num_padding))
        return inputs.as_strided((T_lfr, m * d), (n * d, 1)).clone()
    g = torch.Generator().manual_seed(0)
    for T in list(range(1, 40)) + [499, 2998, 3000]:
        x = torch.randn(T, 5, generator=g)
        assert torch.equal(ref_lfr(x, 7, 6), O.apply_lfr(x, 7, 6)), T


def test_oracle_matches_live_reference_components():
    """The reference's own SANMEncoder and CifPredictorV2 on seeded random inputs, compared stage by stage: their outputs as stored
    in tests/golden/live_components.npz (oracle/make_live_golden.py) and, when the reference is importable, a fresh run of them."""
    import make_live_golden as mk
    from funasr_b200 import synth
    cfg = synth.PARAFORMER_TINY
    p, feats, lens = mk.component_inputs()
    runs = [{k: torch.from_numpy(v) for k, v in mk.load_components(os.path.join(GOLDEN, "live_components.npz")).items()}]
    if ref_shim.reference_available():
        ref_shim.import_reference()
        runs.append({k: torch.from_numpy(v) for k, v in mk.run_components().items()})
    with torch.no_grad():
        o_enc, o_len = O.encoder(feats, lens, p, cfg.enc_layers)
        for r in runs:
            assert torch.allclose(r["enc"], o_enc, rtol=0, atol=1e-5) and r["enc_lens"].tolist() == o_len.tolist()
            o_emb, o_tok, o_al, o_pk = O.predictor(r["enc"], lens, p)
            assert r["token_num"].tolist() == o_tok.tolist()
            assert torch.allclose(r["alphas"], o_al, atol=1e-6) and torch.allclose(r["peaks"], o_pk, atol=1e-5)
            assert torch.allclose(r["acoustic"], o_emb, atol=1e-4)


@pytest.mark.parametrize("name", list(SV_CASES))
def test_sensevoice_oracle_matches_reference_golden(name):
    """SenseVoiceSmall (BASELINE config 4): oracle vs outputs of the unmodified reference SenseVoiceSmall.inference."""
    from funasr_b200 import synth
    cfg, wseed, wavs, cmvn, g = load_sv_case(name)
    o = O.sensevoice_forward(wavs, synth.make_sensevoice_state_dict(cfg, wseed), cmvn, cfg.enc_layers, cfg.tp_layers)
    step = 7 if cfg.enc_layers > 10 else 1
    assert o["enc_lens"].tolist() == g["enc_lens"].tolist()
    assert rel_err(o["enc"][:, ::step].numpy(), g["enc"]) <= 1e-5
    assert rel_err(o["logp"][:, g["logp_rows"].tolist()].numpy(), g["logp_sel"]) <= 1e-4
    assert [t for r in o["ids"] for t in r] == g["ids_flat"].tolist() and [len(r) for r in o["ids"]] == g["ids_len"].tolist()


@pytest.mark.parametrize("name", list(CTX_CASES))
def test_contextual_oracle_matches_reference_golden(name):
    """ContextualParaformer (BASELINE config 5): hotword LSTM memory + bias decoder vs the unmodified reference."""
    from funasr_b200 import synth
    cfg, wseed, wavs, cmvn, hw, g = load_ctx_case(name)
    o = O.contextual_forward(wavs, synth.make_contextual_state_dict(cfg, wseed), cmvn, cfg.enc_layers, cfg.dec_layers, hw)
    assert o["token_num"].tolist() == g["token_num"].tolist()
    assert rel_err(o["hw_embed"].numpy(), g["hw_embed"]) <= 1e-5
    assert rel_err(o["logp"][:, g["logp_rows"].tolist()].numpy(), g["logp_sel"]) <= 1e-4
    assert [t for r in o["ids"] for t in r] == g["ids_flat"].tolist() and [len(r) for r in o["ids"]] == g["ids_len"].tolist()


@pytest.mark.parametrize("name", list(BICIF_CASES))
def test_bicif_oracle_matches_reference_golden(name):
    """BiCifParaformer (SURVEY §8f rank 1): sequential fp32 `cif`, upsampled CIF timestamp head (ConvTranspose + BLSTM) and the
    timestamps the reference's ts_prediction_lfr6_standard derives, vs the unmodified reference."""
    from funasr_b200 import synth
    from funasr_b200.timestamps import ts_prediction_lfr6_standard
    cfg, wseed, wavs, cmvn, g = load_bicif_case(name)
    o = O.bicif_forward(wavs, synth.make_bicif_state_dict(cfg, wseed), cmvn, cfg.enc_layers, cfg.dec_layers)
    assert o["token_num"].tolist() == g["token_num"].tolist()
    assert np.abs(o["alphas"].numpy() - g["alphas"]).max() <= 1e-5
    assert np.abs(o["peaks"].numpy() - g["peaks"]).max() <= 1e-4
    assert rel_err(o["acoustic"][:, :, ::5].numpy(), g["acoustic"]) <= 1e-5
    assert rel_err(o["us_alphas"].numpy(), g["us_alphas"]) <= 1e-4
    assert np.abs(o["us_peaks"].numpy() - g["us_peaks"]).max() <= 1e-3
    assert [t for r in o["ids"] for t in r] == g["ids_flat"].tolist() and [len(r) for r in o["ids"]] == g["ids_len"].tolist()
    want = gold_stamps(g)
    for i, ids in enumerate(o["ids"]):
        n = int(o["enc_lens"][i]) * 3
        got = ts_prediction_lfr6_standard(o["us_alphas"][i][:n].numpy(), o["us_peaks"][i][:n].numpy(), ["t%d" % (t - 3) for t in ids])[1]
        assert got == want[i]


@pytest.mark.parametrize("name", list(SEACO_CASES))
def test_seaco_oracle_matches_reference_golden(name):
    """SeacoParaformer (SURVEY §8f rank 1, second half): 2-layer hotword LSTM, the seaco decoder over the hotword memory, attention-
    score filtering (second case: 25 hotwords, nfilter 8) and the NO_BIAS merge, vs the unmodified reference's
    `_seaco_decode_with_ASF`.  Oracle only — the CUDA path for this row is round-2 work."""
    from funasr_b200 import synth
    cfg, wseed, wavs, cmvn, hw, nfilter, g = load_seaco_case(name)
    o = O.seaco_forward(wavs, synth.make_seaco_state_dict(cfg, wseed), cmvn, cfg.enc_layers, cfg.dec_layers, hw, synth.seaco_no_bias_id(cfg),
                        nfilter=nfilter)
    assert o["token_num"].tolist() == g["token_num"].tolist()
    assert rel_err(seaco_sel(o, hw), g["hw_selected"]) <= 1e-5
    assert rel_err(o["merged"][:, g["logp_rows"].tolist()].numpy(), g["merged_sel"]) <= 1e-4
    assert [t for r in o["ids"] for t in r] == g["ids_flat"].tolist() and [len(r) for r in o["ids"]] == g["ids_len"].tolist()
    if nfilter < len(hw):
        assert o["asf_picked"] is not None and len(o["asf_picked"]) == nfilter + 1


def seaco_sel(o, hw):
    """the golden file stores the UNFILTERED hotword representations; recompute them when ASF filtered the oracle's copy"""
    return o["hw_selected_all"].numpy()


def test_torch_row_sum_emulation():
    """The step-by-step restatement of torch's CPU fp32 row sum (oracle torch_row_sum_f32, mirrored by csrc/cif.cu) equals
    torch.sum bit for bit — row lengths around every structural boundary (8-lane vectors, 4 ILP accumulators, 16-vector cascade
    flushes), the CIF row lengths (T+1 = 84..1001, 3T = 1500) and rows whose sum sits within an ulp of an integer."""
    g = np.random.default_rng(0)
    for n in [1, 2, 3, 7, 8, 9, 15, 16, 31, 32, 33, 63, 64, 84, 101, 255, 256, 257, 500, 501, 502, 511, 512, 513, 1001, 1500, 3001, 9001]:
        for trial in range(6):
            x = (g.random(n) * (1.0 if trial % 2 else 0.4)).astype(np.float32)
            want = torch.from_numpy(np.stack([x, x]))[1:].sum(-1).numpy()[0]
            assert O.torch_row_sum_f32(x) == want, (n, trial)
    # near-integer sums: scale a row so that its exact sum is an integer +- a few fp32 ulps; floor() then depends on the order
    flips = 0
    for trial in range(200):
        n = 501
        x = (g.random(n) * 0.5).astype(np.float32)
        target = np.round(x.astype(np.float64).sum())
        x = (x.astype(np.float64) * (target / x.astype(np.float64).sum())).astype(np.float32)
        want = torch.from_numpy(x[None]).sum(-1).numpy()[0]
        got = O.torch_row_sum_f32(x)
        assert got == want
        flips += int(np.floor(want) != np.floor(np.float32(x.astype(np.float64).sum())))
    assert flips > 0      # the cases exist: an order-agnostic (fp64, rounded once) sum disagrees with torch on the integer part
