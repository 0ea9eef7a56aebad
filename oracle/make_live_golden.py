"""Writes tests/golden/live_components.npz and tests/golden/live_host.json: what the tests used to compare with only where the
unmodified reference itself could be imported (or its C++ end-point detector compiled), stored so that every checkout runs those
comparisons.
  * live_components.npz — the reference's SANMEncoder and CifPredictorV2 on seeded random features (tiny config, weight seed 11);
  * live_host.json — ts_prediction_lfr6_standard on seeded CIF weights, merge_vad on seeded segment lists,
    ContextualParaformer.generate_hotwords_list on a seg_dict case, and the segments of the C++ runtime's end-point detector
    (runtime/onnxruntime/src/e2e-vad.h via oracle/_ref/libvad_ref.so) on seeded posteriors and on the golden VAD cases' scores.
The inputs are rebuilt from the same seeds by the tests (tests/test_oracle_golden.py, tests/test_timestamps.py, tests/test_vad_host.py,
tests/test_properties_host.py).  TEST INFRASTRUCTURE ONLY; needs the reference tree.  Usage: python oracle/make_live_golden.py"""
import copy
import json
import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLD = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)

import knf_ref  # noqa: E402
import make_vad_cpp_golden as mk  # noqa: E402
import ref_shim  # noqa: E402
from funasr_b200 import synth  # noqa: E402
from funasr_b200 import timestamps as TS  # noqa: E402


def component_inputs():
    """-> (state dict, feats [3, 41, 560], lens) of the encoder / predictor comparison."""
    p = synth.make_state_dict(synth.PARAFORMER_TINY, 11)
    g = torch.Generator().manual_seed(5)
    feats = torch.randn(3, 41, 560, generator=g)
    lens = torch.tensor([41, 17, 30], dtype=torch.int32)
    for b in range(3):
        feats[b, lens[b]:] = 0
    return p, feats, lens


def run_components():
    """The reference's own encoder and predictor -> {enc, enc_lens, token_num, alphas, peaks, acoustic}."""
    from funasr.register import tables
    cfg = synth.PARAFORMER_TINY
    p, feats, lens = component_inputs()
    enc = tables.encoder_classes["SANMEncoder"](input_size=560, output_size=512, attention_heads=4, linear_units=2048,
                                                num_blocks=cfg.enc_layers, input_layer="pe", kernel_size=11, sanm_shfit=0,
                                                selfattention_layer_type="sanm").eval()
    enc.load_state_dict({k[len("encoder."):]: v for k, v in p.items() if k.startswith("encoder.")}, strict=True)
    pred = tables.predictor_classes["CifPredictorV2"](idim=512, threshold=1.0, l_order=1, r_order=1, tail_threshold=0.45).eval()
    pred.load_state_dict({k[len("predictor."):]: v for k, v in p.items() if k.startswith("predictor.")}, strict=True)
    with torch.no_grad():
        r_enc, r_len, _ = enc(feats, lens)
        mask = (torch.arange(feats.shape[1])[None, :] < lens[:, None])[:, None, :]
        r_emb, r_tok, r_al, r_pk = pred(r_enc, None, mask, ignore_id=-1)
    return {"enc": r_enc.numpy(), "enc_lens": r_len.numpy(), "token_num": r_tok.numpy(), "alphas": r_al.numpy(), "peaks": r_pk.numpy(),
            "acoustic": r_emb.numpy()}


def save_components(path, comp):
    """np.savez_compressed with every float32 array split into its four byte planes (lossless; the plane of sign and exponent bytes
    compresses, which keeps the fixture small)."""
    out = {}
    for k, v in comp.items():
        if v.dtype == np.float32:
            out[k + "_planes"] = np.ascontiguousarray(np.ascontiguousarray(v).view(np.uint8).reshape(-1, 4).T)
            out[k + "_shape"] = np.array(v.shape)
        else:
            out[k] = v
    np.savez_compressed(path, **out)


def load_components(path):
    """Inverse of save_components -> {enc, enc_lens, token_num, alphas, peaks, acoustic} as numpy arrays."""
    d = dict(np.load(path))
    for k in [k[: -len("_planes")] for k in d if k.endswith("_planes")]:
        d[k] = np.ascontiguousarray(d.pop(k + "_planes").T).view(np.float32).reshape(d.pop(k + "_shape").tolist())
    return d


def timestamp_inputs():
    """-> [(CIF weights, fires, chars)] of the 50 seeded timestamp cases."""
    rng = np.random.default_rng(7)
    out = []
    for trial in range(50):
        T = int(rng.integers(6, 120))
        a = (rng.random(T).astype(np.float32) ** 2 * 0.8).astype(np.float32)
        peaks = TS.cif_wo_hidden(a, 1.0)
        chars = ["c%d" % i for i in range(max(1, int((peaks >= 1 - 1e-4).sum()) - 1 + trial % 2))]
        out.append((a, peaks, chars))
    return out


def run_timestamps():
    from funasr.utils.timestamp_tools import ts_prediction_lfr6_standard as ref_fn
    res = []
    for a, peaks, chars in timestamp_inputs():
        try:
            txt, stamps = ref_fn(torch.tensor(peaks.copy()), torch.tensor(a.copy()), copy.copy(chars), upsample_rate=1)
        except IndexError:
            txt, stamps = "", []
        res.append([txt, stamps])
    return res


def merge_vad_inputs():
    g = np.random.default_rng(0)
    return [np.sort(g.integers(0, 200000, size=2 * int(g.integers(1, 12)))).reshape(-1, 2).tolist() for _ in range(50)]


def run_merge_vad():
    from funasr.utils.vad_utils import merge_vad as ref_merge
    return [ref_merge([list(x) for x in t], 15000) for t in merge_vad_inputs()]


class HotwordTokenizer:
    vocab = {"<unk>": 9, "he@@": 3, "llo": 4, "你": 5, "好": 6, "7": 7, "gpu": 8}

    def tokens2ids(self, toks):
        return [self.vocab.get(t, self.vocab["<unk>"]) for t in toks]


HOTWORD_SEG_DICT = "hello he@@ llo\n你 你\n好 好\n7 7\ngpu gpu\n"
HOTWORD_STRING = "Hello 你好 GPU xyz"
HOTWORD_FILE = "hello 你好\ngpu\n"


def run_hotwords():
    """generate_hotwords_list for the plain string and for the same words in a .txt file, seg_dict beside the cmvn file."""
    from funasr.models.contextual_paraformer.model import ContextualParaformer

    class Model:
        sos = 1

    class Frontend:
        cmvn_file = None

    with tempfile.TemporaryDirectory() as d:
        fe = Frontend()
        fe.cmvn_file = os.path.join(d, "am.mvn")
        with open(fe.cmvn_file, "w") as f:
            f.write("x")
        with open(os.path.join(d, "seg_dict"), "w", encoding="utf8") as f:
            f.write(HOTWORD_SEG_DICT)
        txt = os.path.join(d, "hw.txt")
        with open(txt, "w", encoding="utf8") as f:
            f.write(HOTWORD_FILE)
        return {"string": ContextualParaformer.generate_hotwords_list(Model(), HOTWORD_STRING, tokenizer=HotwordTokenizer(), frontend=fe),
                "file": ContextualParaformer.generate_hotwords_list(Model(), txt, tokenizer=HotwordTokenizer(), frontend=fe)}


def vad_cpp_random_inputs():
    """-> [(n_samples, sil_prob, waveform, max_end_silence_ms, speech_noise_thres)]: 50 recordings up to 40 s, 10 up to 150 s."""
    rng = np.random.default_rng(7)
    return [mk.random_case(rng, 40.0 if it < 50 else 150.0) for it in range(60)]


VAD_GOLDEN_CASES = ("vad_fixed800", "vad_short", "vad_silence")


def run_vad_cpp():
    """The C++ detector on the seeded posteriors and on the Python reference's own scores of three golden VAD cases."""
    from make_vad_golden import VAD_CASES
    rand = [knf_ref.vad_segments(sp, wav, mes, 60000, thr) for n, sp, wav, mes, thr in vad_cpp_random_inputs()]
    gold = {}
    for name in VAD_GOLDEN_CASES:
        seconds, seed, pattern, _ = VAD_CASES[name]
        sil = np.load(os.path.join(GOLD, name + ".npz"))["sil_prob"]
        gold[name] = knf_ref.vad_segments(sil, synth.make_vad_wav(seconds, seed, pattern).numpy(), 800, 60000, 0.6)
    return {"random": rand, "golden_scores": gold}


def main():
    assert knf_ref.build(), "needs the reference tree (oracle/knf/Makefile)"
    ref_shim.import_reference()
    comp = run_components()
    path = os.path.join(GOLD, "live_components.npz")
    save_components(path, comp)
    assert all(np.array_equal(v, comp[k]) for k, v in load_components(path).items())
    print("wrote", path, os.path.getsize(path), "bytes")
    host = {"timestamps": run_timestamps(), "merge_vad": run_merge_vad(), "hotwords": run_hotwords(), "vad_cpp": run_vad_cpp()}
    path = os.path.join(GOLD, "live_host.json")
    with open(path, "w", encoding="utf8") as f:
        json.dump(host, f, ensure_ascii=False, separators=(",", ":"))
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
