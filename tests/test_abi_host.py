"""CPU: the C-ABI library loads and exports every symbol include/funasr_b200.h declares; host-side logic
(registry drop-in surface, parameter names, cmvn parsing, sharding + all-gather over gloo with 2 ranks)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT

import funasr_b200
import ref_shim
from funasr_b200 import _abi, synth
from funasr_b200.engine import kaldi_mel_banks, num_lfr_frames
from funasr_b200.sharding import shard_utterances


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "funasr_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(fa_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    assert os.path.exists(_abi.LIB_PATH), "build first: python -c 'import __graft_entry__ as g; g.build()'"
    lib = ctypes.CDLL(_abi.LIB_PATH)
    syms = _header_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(lib, s), "library does not export %s" % s
        assert s in _abi.SIGNATURES, "ctypes mirror lacks %s" % s
    assert set(_abi.SIGNATURES) == set(syms)
    lib.fa_version.restype = ctypes.c_char_p
    assert b"sm_100a" in lib.fa_version()


def test_no_cpu_fallback():
    m = _tiny_model()
    with pytest.raises(_abi.FunasrB200Error):
        m.inference([np.zeros(16000, dtype=np.float32)], key=["a"], frontend=None, device="cpu")
    with pytest.raises(_abi.FunasrB200Error):
        m.encoder(torch.zeros(1, 4, 560), torch.tensor([4]))


def _tiny_conf():
    cfg = synth.PARAFORMER_TINY
    return dict(
        encoder="SANMEncoderB200",
        encoder_conf=dict(output_size=512, attention_heads=4, linear_units=2048, num_blocks=cfg.enc_layers, dropout_rate=0.1,
                          input_layer="pe", pos_enc_class="SinusoidalPositionEncoder", normalize_before=True, kernel_size=11,
                          sanm_shfit=0, selfattention_layer_type="sanm"),
        decoder="ParaformerSANMDecoderB200",
        decoder_conf=dict(attention_heads=4, linear_units=2048, num_blocks=cfg.dec_layers, att_layer_num=cfg.dec_layers,
                          kernel_size=11, sanm_shfit=0),
        predictor="CifPredictorV2B200",
        predictor_conf=dict(idim=512, threshold=1.0, l_order=1, r_order=1, tail_threshold=0.45),
        input_size=560, vocab_size=cfg.vocab)


def _tiny_model():
    return funasr_b200.ParaformerB200(**_tiny_conf())


def test_state_dict_names_match_reference_layout():
    """SURVEY §8 a21: the synthetic dict uses the reference's names; strict load must accept it unchanged."""
    m = _tiny_model()
    sd = synth.make_state_dict(synth.PARAFORMER_TINY, 3)
    assert set(m.state_dict().keys()) == set(sd.keys())
    for k, v in m.state_dict().items():
        assert tuple(v.shape) == tuple(sd[k].shape), k
    m.load_state_dict(sd, strict=True)
    full = synth.ParaformerConfig()
    assert full.feat_dim == 560


def test_registry_surface():
    # install() = the documented step after `import funasr` (another test of this session may have imported the live reference after
    # funasr_b200, which switches get_tables() to the reference's own tables); without funasr it returns the local tables unchanged
    t = funasr_b200.install()
    assert t is funasr_b200.get_tables()
    for table, key in [("model_classes", "ParaformerB200"), ("frontend_classes", "WavFrontendB200"),
                       ("encoder_classes", "SANMEncoderB200"), ("predictor_classes", "CifPredictorV2B200"),
                       ("decoder_classes", "ParaformerSANMDecoderB200")]:
        assert key in getattr(t, table)


def test_cmvn_file_parse():
    cm = funasr_b200.load_cmvn(os.path.join(GOLDEN, "am_synth.mvn"))
    ref = synth.make_cmvn(synth.PARAFORMER_LARGE, seed=1)
    assert cm.shape == (2, 560) and torch.allclose(cm, ref, rtol=0, atol=0)


def test_frame_count_and_mel_banks():
    assert num_lfr_frames(480000) == 500 and num_lfr_frames(80000) == 83 and num_lfr_frames(400) == 1
    # below one 25 ms window the reference shrinks the window to the utterance: still one frame, down to 2 samples (wav_frontend.py:174)
    assert num_lfr_frames(399) == 1 and num_lfr_frames(2) == 1 and num_lfr_frames(1) == 0
    import paraformer_oracle as O
    banks = torch.nn.functional.pad(O.get_mel_banks(), (0, 1))
    assert torch.equal(kaldi_mel_banks(), banks.float())
    for nfft in (256, 128, 32, 2):                                  # the FFT sizes of sub-frame utterances
        assert torch.equal(kaldi_mel_banks(n_fft=nfft), torch.nn.functional.pad(O.get_mel_banks(80, nfft, 16000.0), (0, 1)).float())
    for n in (399, 200, 17, 2):                                     # oracle frontend row count for such inputs
        f_, l_ = O.frontend([synth.make_wav(n, 3)], None)
        assert l_.tolist() == [1] and f_.shape == (1, 1, 560)
    assert torch.equal(synth.sinusoid_inv_timescales(560), torch.exp(torch.arange(280.0) * -(torch.log(torch.tensor([10000.0])) / 279)))


def test_shard_utterances_partition():
    g = torch.Generator().manual_seed(1234)
    dur = (5 + 25 * torch.rand(512, generator=g)).tolist()
    for w in (1, 2, 4, 8):
        sh = shard_utterances(dur, w)
        assert sorted(i for s in sh for i in s) == list(range(512))
        assert max(len(s) for s in sh) - min(len(s) for s in sh) <= 1
        loads = [sum(dur[i] for i in s) for s in sh]
        assert max(loads) / min(loads) < 1.02


_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from funasr_b200.sharding import shard_utterances, gather_token_ids
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % sys.argv[2], rank=int(sys.argv[3]), world_size=2)
n = 11
dur = [float((7 * i) % 13 + 1) for i in range(n)]
shards = shard_utterances(dur, 2)
mine = shards[dist.get_rank()]
fake = lambda i: [100 * i + k for k in range(i % 5)]       # utterance i "decodes" to a known id list
res = gather_token_ids([fake(i) for i in mine], mine, n, width=16)
assert res == [fake(i) for i in range(n)], res
assert gather_token_ids([fake(i) for i in mine], mine, n) == res            # width=None: sized by an all_reduce(MAX)
try:
    gather_token_ids([fake(i) for i in mine], mine, n, width=2)              # too narrow: raises, never truncates
    raise SystemExit("expected ValueError")
except ValueError:
    pass
# ShardedRunner: shard -> bucket -> infer -> (device-side rows) -> one all_gather, every rank gets every result in input order
from funasr_b200.sharding import ShardedRunner
lens = [400 + 160 * 6 * ((5 * i) % 9 + 1) for i in range(13)]                # 1..9 LFR frames... ragged
wavs = [torch.full((k,), float(i)) for i, k in enumerate(lens)]
def infer(batch):                                                            # "decodes" utterance i (read back from its samples) to [i, i+1, ...]
    idx = [int(w[0]) for w in batch]
    n = max(i % 4 for i in idx) or 1
    ids = torch.full((len(batch), n), -1, dtype=torch.int32)
    for r, i in enumerate(idx):
        for k in range(i % 4):
            ids[r, k] = i + k
    return ids, torch.tensor([i % 4 for i in idx], dtype=torch.int32)
run = ShardedRunner(infer, "cpu", max_batch=3, max_frames=3 * 10)
got = run.run(wavs)
assert got == [[i + k for k in range(i % 4)] for i in range(13)], got
plan = run.plan(lens)
assert sorted(i for b in plan["buckets"] for i in b) == sorted(plan["mine"]) and all(len(b) <= 3 for b in plan["buckets"])
dist.barrier(); dist.destroy_process_group(); print("ok")
'''


def test_gather_token_ids_two_ranks_gloo(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(_WORKER)
    port = str(29500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, port, str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    outs = [p.communicate(timeout=180)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert all("ok" in o for o in outs)


@pytest.mark.skipif(not ref_shim.reference_available(), reason="needs the FunASR package itself (the unmodified reference)")
def test_plugs_into_reference_tables_and_automodel_build():
    """Drop-in surface against the real FunASR: classes land in funasr.register.tables and AutoModel.build_model
    constructs ParaformerB200 + WavFrontendB200 and strict-loads a checkpoint via load_pretrained_model (CPU build
    only — running it needs a GPU)."""
    ref_shim.import_reference()
    from funasr.register import tables
    funasr_b200.install()
    assert tables.model_classes["ParaformerB200"] is funasr_b200.ParaformerB200
    assert tables.frontend_classes["WavFrontendB200"] is funasr_b200.WavFrontendB200
    from funasr import AutoModel
    import tempfile
    cfg = synth.PARAFORMER_TINY
    conf = _tiny_conf()
    tokens = ["<blank>", "<s>", "</s>"] + ["t%d" % i for i in range(cfg.vocab - 4)] + ["<unk>"]
    with tempfile.TemporaryDirectory() as tmp:
        pt = os.path.join(tmp, "model.pt")
        torch.save(synth.make_state_dict(cfg, 3), pt)
        am = AutoModel(model="ParaformerB200", model_conf={}, encoder=conf["encoder"], encoder_conf=conf["encoder_conf"],
                       decoder=conf["decoder"], decoder_conf=conf["decoder_conf"], predictor=conf["predictor"],
                       predictor_conf=conf["predictor_conf"], frontend="WavFrontendB200",
                       frontend_conf=dict(fs=16000, window="hamming", n_mels=80, frame_length=25, frame_shift=10, lfr_m=7, lfr_n=6,
                                          dither=0.0, cmvn_file=os.path.join(GOLDEN, "am_synth.mvn")),
                       tokenizer="CharTokenizer", tokenizer_conf=dict(token_list=tokens, unk_symbol="<unk>", split_with_space=True),
                       device="cpu", disable_update=True, disable_pbar=True, init_param=pt)
    assert isinstance(am.model, funasr_b200.ParaformerB200)
    assert isinstance(am.kwargs["frontend"], funasr_b200.WavFrontendB200)
    sd = synth.make_state_dict(cfg, 3)
    assert torch.equal(am.model.state_dict()["encoder.encoders.0.feed_forward.w_1.weight"], sd["encoder.encoders.0.feed_forward.w_1.weight"])
    # override mode: the reference's own keys now resolve to this backend
    saved = {k: getattr(tables, k[0]).get(k[1]) for k in funasr_b200.registry.DROP_IN_KEYS}
    try:
        funasr_b200.install(override_reference_keys=True)
        assert tables.model_classes["Paraformer"] is funasr_b200.ParaformerB200
    finally:
        for (tb, key), cls in saved.items():
            if cls is not None:
                getattr(tables, tb)[key] = cls


def test_bucket_by_length_config3():
    """BASELINE config 3: 512 utterances, durations ~U[5,30] s (seed 1234): buckets are a partition, respect the caps,
    and waste little padding; run_bucketed restores the input order."""
    from funasr_b200.batching import bucket_by_length, padding_efficiency, run_bucketed
    g = torch.Generator().manual_seed(1234)
    n = [int(x) for x in ((5 + 25 * torch.rand(512, generator=g)) * 16000).tolist()]
    for shard, mb, eff in ((n, 64, 0.9), (n[::8], 16, 0.85)):      # whole job / one GPU's shard of 64
        bk = bucket_by_length(shard, max_batch=mb, max_frames=mb * 500)
        assert sorted(i for b in bk for i in b) == list(range(len(shard)))
        for b in bk:
            t = [num_lfr_frames(shard[i]) for i in b]
            assert len(b) <= mb and len(b) * max(t) <= mb * 500
        assert padding_efficiency(shard, bk) > eff
    fake = lambda batch: [[int(w.shape[-1]) % 97] for w in batch]
    wavs = [torch.zeros(k) for k in n[:50]]
    assert run_bucketed(wavs, fake, max_batch=8) == [[k % 97] for k in n[:50]]


def test_model_file_roundtrip(tmp_path):
    """pack.py writes exactly what csrc/offline.cu:load_file parses: FunASR state_dict names + derived tables."""
    from funasr_b200 import pack, synth
    cfg = synth.PARAFORMER_TINY
    st = synth.make_state_dict(cfg, 3)
    cmvn = synth.make_cmvn(cfg, 1)
    path = str(tmp_path / "tiny.fab2")
    n = pack.write_model_file(path, st, cfg, cmvn)
    back = pack.read_model_file(path)
    assert len(back) == n
    assert back["__config__"].tolist()[:7] == [cfg.enc_layers, cfg.dec_layers, cfg.d_model, cfg.heads, cfg.kernel, cfg.vocab, cfg.feat_dim]
    for k in ("encoder.encoders0.0.self_attn.linear_q_k_v.weight", "decoder.output_layer.weight", "predictor.cif_output.bias"):
        assert np.array_equal(back[k], st[k].numpy())
    cw = st["predictor.cif_conv1d.weight"]
    assert np.array_equal(back["predictor.cif_conv1d.gemm_weight"][:, 512:1024], cw[:, :, 1].numpy())   # W[n, k*512+c] = w[n,c,k]
    assert back["frontend.mel_banks"].shape == (80, 257) and back["frontend.cmvn"].shape == (2, 560)
    with open(path, "rb") as f:
        assert f.read(8) == b"FAB2MDL1"


def test_offline_api_rejects_bad_arguments_without_a_gpu():
    """The handle API fails loudly (NULL + message), never falls back: missing file / no CUDA device."""
    from funasr_b200 import _abi
    lib = _abi.load()
    h = lib.fa_offline_init(b"/nonexistent/model.fab2", 0, 3)
    assert not h
    assert lib.fa_offline_last_error() != b""
    assert not lib.fa_offline_init(None, 0, 3)
    assert lib.fa_offline_result_count(None) == 0


def test_resample_table_matches_torchaudio():
    """funasr_b200.resample restates torchaudio's _get_sinc_resample_kernel (the resampler behind load_utils.py:176-178)."""
    import math
    taf = pytest.importorskip("torchaudio.functional.functional")
    from funasr_b200.resample import sinc_resample_table
    for o, n in [(8000, 16000), (48000, 16000), (44100, 16000), (22050, 16000), (32000, 16000), (16000, 8000)]:
        tab, orig, new, width = sinc_resample_table(o, n)
        ref, w = taf._get_sinc_resample_kernel(o, n, math.gcd(o, n))
        assert (orig, new, width) == (o // math.gcd(o, n), n // math.gcd(o, n), w)
        assert np.array_equal(tab, ref[:, 0, :].numpy())


def test_header_is_plain_c_and_links(tmp_path):
    """include/funasr_b200.h is a C header (not just C++): a C99 client compiles with -pedantic, links against the library and
    runs; without a GPU / model file the handle API reports an error instead of falling back."""
    exe = str(tmp_path / "offline_demo")
    libdir = os.path.join(ROOT, "funasr_b200")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I" + os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "examples", "offline_demo.c"), "-L" + libdir, "-lfunasr_b200", "-Wl,-rpath," + libdir, "-o", exe],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    run = subprocess.run([exe], capture_output=True, text=True)
    assert run.returncode == 0 and "library: funasr_b200" in run.stdout
    if not torch.cuda.is_available():
        assert "init failed" in run.stdout


def test_funoffline_client_links_against_the_reference_header(tmp_path):
    """Link compatibility of the C++ runtime surface: the client of examples/offline_runtime_client.cpp (the call sequence of
    runtime/onnxruntime/bin/funasr-onnx-offline.cpp) compiled against the REFERENCE's own funasrruntime.h needs the mangled entry
    points stored in tests/golden/funasrruntime_client_symbols.txt (oracle/make_runtime_symbols_golden.py): libfunasr_b200.so
    defines every one of them — same names, same C++ argument types — and this repo's copy of the declarations asks for exactly
    that set.  The client built against this repo's header (and, when the reference tree is present, against its header too)
    links and fails cleanly (no CPU path, no model) when run without a GPU."""
    import shutil
    import make_runtime_symbols_golden as mk
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    with open(os.path.join(GOLDEN, "funasrruntime_client_symbols.txt")) as f:
        want = f.read().split()
    assert len(want) == 15
    lib = ctypes.CDLL(_abi.LIB_PATH)
    assert [s for s in want if not hasattr(lib, s)] == []
    assert mk.client_runtime_symbols('"funasrruntime_b200.h"', os.path.join(ROOT, "include")) == want
    exe = str(tmp_path / "client")
    headers = [('"funasrruntime_b200.h"', os.path.join(ROOT, "include"))]
    if os.path.exists(os.path.join(mk.reference_header_dir(), "funasrruntime.h")):
        headers.append(('"funasrruntime.h"', mk.reference_header_dir()))
    for hdr, inc in headers:
        cmd = ["g++", "-std=c++17", "-DFUNASR_RUNTIME_HEADER=" + hdr, "-I" + inc, "-I" + os.path.join(ROOT, "include"),
               os.path.join(ROOT, "examples", "offline_runtime_client.cpp"), "-L" + os.path.join(ROOT, "funasr_b200"), "-lfunasr_b200",
               "-Wl,-rpath," + os.path.join(ROOT, "funasr_b200"), "-o", exe]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert r.returncode == 0, r.stdout[-2000:]
        r = subprocess.run([exe, str(tmp_path), str(tmp_path / "none.wav")], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert r.returncode == 1 and "init failed" in r.stdout


def test_product_never_touches_the_oracle_or_the_reference_tree():
    """The oracle is test infrastructure: nothing under funasr_b200/ (Python or native sources) or include/ may import, open, link or
    name it, nor read /root/reference; missing the CUDA library must raise instead of falling back."""
    bad = []
    for base in (os.path.join(ROOT, "funasr_b200"), os.path.join(ROOT, "include"), os.path.join(ROOT, "examples")):
        for dirpath, _, files in os.walk(base):
            if "_build" in dirpath or "__pycache__" in dirpath:
                continue
            for fn in files:
                if not fn.endswith((".py", ".cu", ".cuh", ".h", ".cpp", ".c", ".sh")):
                    continue
                text = open(os.path.join(dirpath, fn), errors="ignore").read()
                for needle in ("paraformer_oracle", "vad_oracle", "punc_oracle", "ref_shim", "ref_runner", "knf_ref", "import oracle", "from oracle",
                               "/root/reference", "baseline/_ref", "oracle/"):
                    if needle in text:
                        bad.append((os.path.relpath(os.path.join(dirpath, fn), ROOT), needle))
    assert not bad, bad
    src = open(os.path.join(ROOT, "funasr_b200", "_abi.py")).read()
    assert "FunasrB200Error" in src and "LIB_PATH" in src


def test_host_side_entry_points_from_plain_c(tmp_path):
    """The two host-only routines of the ABI (no GPU needed) called from a C99 program: the integrate-and-fire trace and the VAD
    end-point walk give the values the Python specifications give."""
    src = tmp_path / "host_calls.c"
    src.write_text(r'''
#include <math.h>
#include <stdio.h>
#include <string.h>
#include "funasr_b200.h"
int main(void) {
  const float a[5] = {0.4f, 0.7f, 0.2f, 0.9f, 0.05f};
  float tr[5];
  if (fa_cif_wo_hidden_host(a, 5, 1.0f, tr) != FA_OK) return 1;
  printf("trace %.6f %.6f %.6f %.6f %.6f\n", tr[0], tr[1], tr[2], tr[3], tr[4]);
  enum { F = 300 };
  double sil[F], db[F];
  for (int i = 0; i < F; ++i) { sil[i] = (i >= 60 && i < 200) ? 0.05 : 0.95; db[i] = 0.0; }
  FaVadOptions o;
  memset(&o, 0, sizeof o);
  o.sample_rate = 16000; o.detect_mode = 1; o.max_end_silence_time = 800; o.max_start_silence_time = 3000; o.window_size_ms = 200;
  o.sil_to_speech_time_thres = 150; o.speech_to_sil_time_thres = 150; o.do_extend = 1; o.lookback_time_start_point = 200;
  o.lookahead_time_end_point = 100; o.max_single_segment_time = 60000; o.noise_frame_num_used_for_snr = 100; o.frame_in_ms = 10;
  o.frame_length_ms = 25; o.speech_2_noise_ratio = 1.0; o.snr_thres = -100.0; o.decibel_thres = -100.0; o.speech_noise_thres = 0.6;
  o.fe_prior_thres = 1e-4;
  int32_t seg[16];
  const int64_t n = fa_vad_detect_segments(sil, db, F, 400 + 160 * (F - 1), &o, 60000, 0, NULL, 0, NAN, seg, 8);
  printf("segments %lld", (long long)n);
  for (int i = 0; i < n && i < 8; ++i) printf(" [%d,%d]", seg[2 * i], seg[2 * i + 1]);
  printf("\n");
  printf("bad %lld\n", (long long)fa_vad_detect_segments(sil, db, F, 48000, NULL, 60000, 0, NULL, 0, NAN, seg, 8));
  return 0;
}
''')
    exe = str(tmp_path / "host_calls")
    libdir = os.path.join(ROOT, "funasr_b200")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I" + os.path.join(ROOT, "include"), str(src),
                        "-L" + libdir, "-lfunasr_b200", "-Wl,-rpath," + libdir, "-lm", "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    run = subprocess.run([exe], capture_output=True, text=True)
    assert run.returncode == 0, run.stdout + run.stderr
    lines = run.stdout.strip().splitlines()
    from funasr_b200 import timestamps as TS, vad
    want_tr = TS.cif_wo_hidden_py(np.array([0.4, 0.7, 0.2, 0.9, 0.05], np.float32), 1.0)
    assert lines[0] == "trace " + " ".join("%.6f" % v for v in want_tr)
    sil = [0.05 if 60 <= i < 200 else 0.95 for i in range(300)]
    want = vad.detect_segments(sil, [0.0] * 300, 400 + 160 * 299, max_end_silence_time=800)
    assert want and lines[1] == "segments %d" % len(want) + "".join(" [%d,%d]" % (s, e) for s, e in want)
    assert lines[2] == "bad -1"
