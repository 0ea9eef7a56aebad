#!/usr/bin/env python
"""Benchmark of the offline Paraformer hot path (BASELINE.json metric: RTFx = audio-seconds / second).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config 2|3|4|5] [--mode fp32|fp16x3|fp16x6|fp16] [--impl reference]
                  [--dump-outputs DIR]

One step = one pass of the hot path over one job of synthetic 16 kHz utterances (BASELINE.json `configs`):
  --config 2 (default, the configuration the metric is quoted on): Paraformer-large, 64 x 30 s per GPU, weak scaling
  --config 3: Paraformer-large, 512 utterances of U[5,30] s (seed 1234), duration-sharded over the ranks, length-bucketed
              (<= 64 utterances / <= 32000 padded frames per batch), strong scaling
  --config 4: SenseVoiceSmall (50 + 20 SAN-M blocks, CTC greedy), 128 x 30 s per GPU, weak scaling
  --config 5: ContextualParaformer (hotword bias decoder, 32 hotwords seed 7), 256 x 30 s sharded over the ranks, strong scaling
Every rank decodes its shard (funasr_b200.sharding.ShardedRunner: shard -> bucket -> infer -> rows on the device) and ONE
all-gather of the token-id rows per job returns every result to every rank; the collective is issued asynchronously so it
overlaps the next job's kernels.  Prints ONE JSON line (rank 0).

`value` times the job with the waveforms already resident in HBM; `e2e` times the same job through the plugin call
(ParaformerB200.inference / infer_ids_device) with HOST (pinned) waveforms in and token ids on the host out, copies inside the
timed region.  `parity` compares the ids of the TIMED job (and the log-probabilities and stage taps — features, encoder output, CIF
weights, acoustic embeddings — of an untimed taps pass over the same utterances) with the CPU oracle's output for a bounded sample,
computed by the CPU leg of the same run.
`--impl reference` times the unmodified reference on the host cores (AutoModel(device="cpu").generate() from the offline
install under baseline/_ref, kind "reference"; the CPU restatement oracle/, kind "port", when that cannot be imported).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "RTFx (audio-sec/s) Paraformer-large 30s utts"
UTT_SECONDS = 30.0
UTT_SAMPLES = 480000
_T0 = time.perf_counter()


def log(msg):
    print("[bench %6.1fs] %s" % (time.perf_counter() - _T0, msg), file=sys.stderr, flush=True)


# algorithmic FLOPs (SURVEY.md §8d), per utterance with T LFR frames and n tokens
def flops_paraformer(T, ntok):
    enc = 2 * T * 560 * 1536 + 49 * 2 * T * 512 * 1536 + 50 * (4 * T * T * 512) + 50 * 2 * T * 512 * 512 + 50 * 4 * T * 512 * 2048 + 50 * 2 * T * 512 * 11
    pred = 2 * T * 512 * 512 * 3 + 2 * T * 512
    dec = 16 * (2 * T * 512 * 1024 + ntok * (4 * 512 * 2048 + 2 * 512 * 512 + 4 * T * 512 + 2 * 512 * 512 + 2 * 512 * 11)) + ntok * 4 * 512 * 2048 + ntok * 2 * 512 * 8404
    return float(enc + pred + dec)


def flops_sensevoice(T):
    layer = 2 * T * 512 * 1536 + 4 * T * T * 512 + 2 * T * 512 * 512 + 4 * T * 512 * 2048 + 2 * T * 512 * 11
    return float(2 * T * 560 * 1536 - 2 * T * 512 * 1536 + 70 * layer + 2 * T * 512 * 25055)


def usable_cpus() -> int:
    """CPUs this process may actually use: affinity mask, capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, n)


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (profiling recipe's clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, pw, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1]))
                out["sm_max_mhz"] = float(r[2])
                pw.append(float(r[3]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.strip().lower() == "active":
                        reasons.add(name)
            except Exception:
                pass
        if sm:
            out["sm_mhz"] = statistics.median(sm)
            out["samples"] = len(sm)
        if pw:
            out["power_w_median"] = statistics.median(pw)
        out["reasons"] = sorted(reasons)
        return out


# ------------------------------------------------------------------------------------------------------------ workloads
def _base_waves(seed0, n=8):
    from funasr_b200 import synth
    return [synth.make_wav(UTT_SAMPLES, seed0 + i, "speechlike") for i in range(n)]


def job_waveforms(config, rank, world):
    """-> (wavs: {global index: 1-D fp32 tensor} for THIS rank's utterances, n_samples of ALL utterances [global order]).
    Deterministic from seeds, so the CPU leg rebuilds exactly the utterances of the timed job."""
    from funasr_b200.sharding import shard_utterances
    if config in (2, 4):                               # weak scaling: `per` identical-length utterances per rank
        per = 64 if config == 2 else 128
        n_all = [UTT_SAMPLES] * (per * world)
        mine = shard_utterances([float(n) for n in n_all], world)[rank]
        base = _base_waves(1000 + 16 * rank)
        g = torch.Generator().manual_seed(4242 + rank)
        gains = 0.4 + 0.6 * torch.rand(per, generator=g)
        local = [(base[i % 8].roll(1601 * i) * gains[i]).contiguous() for i in range(per)]
        return {gi: local[j] for j, gi in enumerate(mine)}, n_all
    if config == 3:                                    # 512 utterances, U[5,30] s, seed 1234 (SURVEY §8d)
        g = torch.Generator().manual_seed(1234)
        n_all = [int(x) for x in ((5 + 25 * torch.rand(512, generator=g)) * 16000).tolist()]
    else:                                              # config 5: 256 x 30 s
        n_all = [UTT_SAMPLES] * 256
    mine = shard_utterances([float(n) for n in n_all], world)[rank]
    base = _base_waves(2000)
    g = torch.Generator().manual_seed(777)
    gains = 0.4 + 0.6 * torch.rand(len(n_all), generator=g)
    return {gi: (base[gi % 8].roll(1601 * gi)[: n_all[gi]] * gains[gi]).contiguous() for gi in mine}, n_all


HOTWORDS_SEED, N_HOTWORDS = 7, 32


class Job:
    """One config's engines, plugin objects and the two step functions (device-resident / end-to-end)."""

    def __init__(self, config, mode, dev, rank, world):
        import funasr_b200
        from funasr_b200 import synth
        from funasr_b200.engine import FrontendEngine, ParaformerEngine, SenseVoiceEngine, num_lfr_frames
        from funasr_b200.sharding import ShardedRunner
        self.config, self.mode, self.dev, self.rank, self.world = config, mode, dev, rank, world
        self.num_lfr_frames = num_lfr_frames
        self.cmvn = synth.make_cmvn(synth.PARAFORMER_LARGE, 1)
        self.wavs, self.n_all = job_waveforms(config, rank, world)
        self.audio_seconds = sum(self.n_all) / 16000.0                      # whole job, all ranks
        self.frontend = funasr_b200.WavFrontendB200(fs=16000, window="hamming", n_mels=80, frame_length=25, frame_shift=10, lfr_m=7,
                                                    lfr_n=6, dither=0.0, cmvn=self.cmvn)
        self.fe = FrontendEngine(self.cmvn, dev)
        self.frontend._engine = self.fe
        self.hotwords = None
        if config == 4:
            self.cfg = synth.SENSEVOICE_SMALL
            self.model = funasr_b200.SenseVoiceSmallB200(
                encoder="SenseVoiceEncoderSmallB200",
                encoder_conf=dict(output_size=512, attention_heads=4, linear_units=2048, num_blocks=self.cfg.enc_layers, tp_blocks=self.cfg.tp_layers,
                                  input_layer="pe", kernel_size=11, sanm_shfit=0, selfattention_layer_type="sanm"),
                input_size=560, vocab_size=self.cfg.vocab, gemm_mode=mode)
            self.eng = SenseVoiceEngine(synth.make_sensevoice_state_dict(self.cfg, 0), self.cfg, dev, gemm_mode=mode, cmvn=self.cmvn)
            self.eng.frontend = self.fe
        else:
            self.cfg = synth.PARAFORMER_LARGE
            conf = dict(encoder="SANMEncoderB200",
                        encoder_conf=dict(output_size=512, attention_heads=4, linear_units=2048, num_blocks=self.cfg.enc_layers, input_layer="pe",
                                          kernel_size=11, sanm_shfit=0, selfattention_layer_type="sanm"),
                        decoder="ParaformerSANMDecoderB200",
                        decoder_conf=dict(attention_heads=4, linear_units=2048, num_blocks=self.cfg.dec_layers, att_layer_num=self.cfg.dec_layers,
                                          kernel_size=11, sanm_shfit=0),
                        predictor="CifPredictorV2B200", predictor_conf=dict(idim=512, threshold=1.0, l_order=1, r_order=1, tail_threshold=0.45),
                        input_size=560, vocab_size=self.cfg.vocab, gemm_mode=mode)
            if config == 5:
                conf["decoder"] = "ContextualParaformerDecoderB200"
                self.model = funasr_b200.ContextualParaformerB200(**conf)
                state = synth.make_contextual_state_dict(self.cfg, 0)
                self.model.load_state_dict(state, strict=True)             # the hotword LSTM / embedding run in torch (O(#hotwords))
                self.model.bias_encoder.to(dev)
                self.model.bias_embed.to(dev)
                self.eng = ParaformerEngine(state, self.cfg, dev, gemm_mode=mode, contextual=True)
                self.hotwords = synth.make_hotwords(N_HOTWORDS, self.cfg.vocab, seed=HOTWORDS_SEED)
                self.eng.set_hotwords(self.model.encode_hotwords(self.hotwords))
            else:
                self.model = funasr_b200.ParaformerB200(**conf)
                self.eng = ParaformerEngine(synth.make_state_dict(self.cfg, 0), self.cfg, dev, gemm_mode=mode)
            self.model.cfg = self.cfg
        self.model._engine = self.eng                                       # the plugin object drives the very same packed weights
        mb, mf = BUCKET_LIMITS[config]
        self.runner_dev = ShardedRunner(self._infer_resident, dev, max_batch=mb, max_frames=mf, extra_ids=4 if config == 4 else 1)
        self.runner_e2e = ShardedRunner(self._infer_plugin, dev, max_batch=self.runner_dev.max_batch, max_frames=self.runner_dev.max_frames,
                                        extra_ids=self.runner_dev.extra_ids)
        self.plan = self.runner_dev.plan(self.n_all)
        # device-resident inputs: one padded [b, Nmax] tensor + lengths per bucket; pinned host copies for the e2e path
        self.resident = {}
        for b in self.plan["buckets"]:
            ws = [self.wavs[i] for i in b]
            pad = torch.nn.utils.rnn.pad_sequence(ws, batch_first=True).to(dev)
            ln = [int(w.numel()) for w in ws]
            self.resident[tuple(b)] = (pad, torch.tensor(ln, dtype=torch.int32, device=dev), ln)
        self.host = {i: w.pin_memory() for i, w in self.wavs.items()}
        self.tok_stats = []
        self._slot = 0
        self._pending = [None, None]

    # ---- one padded batch, inputs resident in HBM
    def _infer_resident(self, batch):
        pad, lens_dev, ln = self.resident[tuple(batch)]
        if self.config == 4:
            out = self.eng.forward_wav(pad, lens_dev, ln, host_lists=False)
            return out["ids_dev"], out["ids_lens_dev"]
        feats, fl = self.fe(pad, lens_dev, max(self.num_lfr_frames(n) for n in ln))
        out = self.eng.forward_feats(feats, fl, host_lists=False)
        self.tok_stats.append(out["token_num"])
        if "ids_dev" not in out:
            return torch.full((len(ln), 1), -1, dtype=torch.int32, device=self.dev), torch.zeros((len(ln),), dtype=torch.int32, device=self.dev)
        return out["ids_dev"], out["ids_lens_dev"]

    # ---- one padded batch through the plugin call: pinned host waveforms in
    def _infer_plugin(self, batch):
        kw = {"hotword_ids": self.hotwords} if self.config == 5 else {}
        return self.model.infer_ids_device([self.host[i] for i in batch], frontend=self.frontend, device=self.dev, **kw)

    def _run(self, runner, key_of):
        slot = self._slot
        self._slot ^= 1
        if self._pending[slot] is not None and self._pending[slot][1] is not None:
            self._pending[slot][1].wait()                                   # the gather that last used this slot's buffers
        rows = runner._rows_buffer(self.plan["per"], self.plan["width"], slot)
        rows.fill_(-1)
        at = 0
        for b in self.plan["buckets"]:
            ids, lens = runner.infer_batch(key_of(b))
            at = runner.pack_rows(rows, at, b, ids, lens)
        self._pending[slot] = runner.gather_async(rows, slot)
        return self._pending[slot]

    def step_device(self):
        return self._run(self.runner_dev, lambda b: b)

    def step_e2e(self):
        if self.world == 1 and self.config == 2:                            # the plain plugin call a single-GPU user makes
            b = self.plan["buckets"][0]
            res, _ = self.model.inference([self.host[i] for i in b], key=["utt%d" % i for i in b], tokenizer=None, frontend=self.frontend,
                                          device=self.dev)
            return res
        h = self._run(self.runner_e2e, lambda b: b)
        return self.runner_e2e.finish(h, self.plan["n_total"])              # waits for the gather, D2H, id lists in input order

    def workload_name(self):
        return {2: "Paraformer-large (50 enc + 16 dec layers, vocab 8404, 220 M params, seeded synthetic weights), batch=64 synthetic 30 s 16 kHz "
                   "utterances per GPU, fused Fbank+encoder+CIF+decoder+greedy",
                3: "Paraformer-large, 512 synthetic utterances of U[5,30] s (seed 1234), duration-sharded over the GPUs, length-bucketed "
                   "(<= 64 utterances and <= 32000 padded frames per batch)",
                4: "SenseVoiceSmall (50 + 20 SAN-M blocks, CTC vocab 25055, seeded synthetic weights), batch=128 synthetic 30 s utterances per GPU, "
                   "fused Fbank + query prepend + encoder + CTC greedy",
                5: "ContextualParaformer-large (hotword bias decoder, 32 hotwords seed 7), 256 synthetic 30 s utterances sharded over the GPUs "
                   "in batches of 64"}[self.config]

    def flops_whole_job(self, ntok_mean):
        tot = 0.0
        for n in self.n_all:
            T = self.num_lfr_frames(n)
            tot += flops_sensevoice(T + 4) if self.config == 4 else flops_paraformer(T, ntok_mean * T / 500.0)
        return tot


# (max utterances, max padded LFR frames) of one bucket: every config works on at most 32 000 padded frames (64 x 30 s) at a time
# (128 x 30 s for the lighter SenseVoice encoder); the ragged config 3 lets short utterances fill that budget (up to 512 per bucket)
# instead of stopping at 64, which keeps the GEMMs of the 5-10 s buckets as large as those of the 30 s ones
BUCKET_LIMITS = {2: (64, 64 * 500), 3: (512, 64 * 500), 4: (128, 128 * 500), 5: (64, 64 * 500)}


# ------------------------------------------------------------------------------------------------------------ CPU arm
def parity_sample(config):
    """Global utterance indices whose ids / log-probs the CPU leg computes with the oracle, as ONE padded batch (the reference's
    padded-batch semantics matter for ragged lengths: the CIF conv reads the first padded frame)."""
    from funasr_b200.sharding import ShardedRunner
    if config == 3:
        plan = ShardedRunner(None, "cpu", max_batch=BUCKET_LIMITS[3][0], max_frames=BUCKET_LIMITS[3][1]).plan(_n_all_cfg3())
        return list(plan["buckets"][-1])                                   # the last (shortest) bucket
    return [0, 1]


def _n_all_cfg3():
    g = torch.Generator().manual_seed(1234)
    return [int(x) for x in ((5 + 25 * torch.rand(512, generator=g)) * 16000).tolist()]


def sample_waveforms(config):
    """The parity / CPU-arm sample of the N=1 job: its utterances (rank 0 of world 1) in sample order."""
    idx = parity_sample(config)
    if config == 3:
        n_all = _n_all_cfg3()
        base = _base_waves(2000)
        g = torch.Generator().manual_seed(777)
        gains = 0.4 + 0.6 * torch.rand(len(n_all), generator=g)
        return idx, [(base[gi % 8].roll(1601 * gi)[: n_all[gi]] * gains[gi]).contiguous() for gi in idx]
    wavs, _ = job_waveforms(config, 0, 1)
    return idx, [wavs[i] for i in idx]


def oracle_on_sample(config, wavs, want_logp=True):
    """CPU oracle (kind 'port') on the sample as one padded batch -> ids (+ selected log-prob rows for the parity block)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import paraformer_oracle as O
    from funasr_b200 import synth
    cmvn = synth.make_cmvn(synth.PARAFORMER_LARGE, 1)
    if config == 4:
        cfg = synth.SENSEVOICE_SMALL
        o = O.sensevoice_forward(wavs, synth.make_sensevoice_state_dict(cfg, 0), cmvn, cfg.enc_layers, cfg.tp_layers)
    elif config == 5:
        cfg = synth.PARAFORMER_LARGE
        o = O.contextual_forward(wavs, synth.make_contextual_state_dict(cfg, 0), cmvn, cfg.enc_layers, cfg.dec_layers,
                                 synth.make_hotwords(N_HOTWORDS, cfg.vocab, seed=HOTWORDS_SEED))
    else:
        cfg = synth.PARAFORMER_LARGE
        o = O.paraformer_forward(wavs, synth.make_state_dict(cfg, 0), cmvn, cfg.enc_layers, cfg.dec_layers)
    return o


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path, timed on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from funasr_b200 import synth
    threads = usable_cpus()
    torch.set_num_threads(threads)
    config = args.config
    idx, wavs = sample_waveforms(config)
    audio = sum(w.numel() for w in wavs) / 16000.0
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    kind, report, ref_ids, err = "port", {}, None, None
    batch = len(wavs) if config == 3 else 1                                # config 3's sample is one padded bucket
    sample = ("each step = the %d utterances (%.0f audio-s) of the job's shortest bucket as one padded batch" % (len(wavs), audio)) if config == 3 else \
        ("each step = %d x 30 s utterances of the job at batch 1 (the reference's CPU default, auto_model.py:785)" % len(wavs))
    am = None
    if not args.port:
        try:
            import ref_runner
            import ref_shim
            tmp = tempfile.mkdtemp(prefix="fa_ref_")
            cm = synth.make_cmvn(synth.PARAFORMER_LARGE, 1)
            ref_kind = {2: "paraformer", 3: "paraformer", 4: "sensevoice", 5: "contextual"}[config]
            cfg = synth.SENSEVOICE_SMALL if config == 4 else synth.PARAFORMER_LARGE
            log("reference arm: building AutoModel(%s, device=cpu) from %s" % (ref_kind, ref_shim.REFERENCE_ROOT))
            am = ref_runner.build_automodel(ref_kind, cfg, 0, cm, tmp, threads)
            kind = "reference"
        except Exception as e:  # pragma: no cover
            err = repr(e)[:300]
            log("reference import/build failed (%s): falling back to the oracle port" % err)
            am = None
    gen_kw = {}
    if am is not None and config == 4:
        gen_kw = dict(language="auto", use_itn=False)
    if am is not None and config == 5:
        hw = synth.make_hotwords(N_HOTWORDS, synth.PARAFORMER_LARGE.vocab, seed=HOTWORDS_SEED)[:-1]      # the reference appends [sos] itself
        hw_file = os.path.join(tmp, "hotwords.txt")
        with open(hw_file, "w") as f:
            for h in hw:
                f.write(" ".join("t%d" % (t - 3) for t in h) + "\n")
        gen_kw = dict(hotword=hw_file)

    def one_pass():
        if am is None:
            if config == 3:
                return oracle_on_sample(config, wavs)["ids"]
            return [oracle_on_sample(config, [w])["ids"][0] for w in wavs]
        if config == 2 or config == 3:
            return ref_runner.generate_ids(am, wavs, batch_size=batch)
        tok = ref_runner.IdTokenizer() if config == 4 else None
        kw = dict(gen_kw)
        if tok is not None:
            kw["tokenizer"] = tok
        res = am.generate(input=[w.numpy() for w in wavs], batch_size=batch, disable_pbar=True, **kw)
        return [r.get("token_int", r.get("text")) for r in res]

    for _ in range(max(1, args.warmup)):
        ref_ids = one_pass()
    ts = []
    for _ in range(max(1, args.steps)):
        t0 = time.perf_counter()
        ref_ids = one_pass()
        ts.append(time.perf_counter() - t0)
    dt = sum(ts)
    val = len(ts) * audio / dt
    cb = {"value": val, "unit": "audio-sec/s", "cores": threads, "kind": kind, "sample": sample, "runs_s": ts, "min_s": min(ts),
          "median_s": statistics.median(ts), "rtfx_best_run": audio / min(ts), "rtfx_median_run": audio / statistics.median(ts)}
    try:
        import ref_runner
        cb["cpu_model"] = ref_runner.cpu_model_string()
    except Exception:
        pass
    if err:
        cb["reference_unavailable"] = err
    if am is not None and config in (2, 3) and not args.no_extras:
        try:
            import ref_runner
            rep = ref_runner.paraformer_report(am, wavs[:2], threads, runs=1)
            cb.update({k: rep[k] for k in ("stages_ms", "batch8_rtfx", "one_thread_rtfx") if k in rep})
        except Exception as e:  # pragma: no cover
            cb["extras_error"] = repr(e)[:200]
    # ---- parity dump for the GPU arm: the ORACLE (always present, pinned to the reference by tests/golden) on the same sample
    if args.parity_out:
        o = oracle_on_sample(config, wavs)
        lp = o["logp"]
        dump = {"ids_flat": np.array([t for r in o["ids"] for t in r], dtype=np.int64), "ids_len": np.array([len(r) for r in o["ids"]], dtype=np.int64),
                "idx": np.array(idx, dtype=np.int64)}
        if lp is not None:
            rows = sorted(set([0, 1, lp.shape[1] // 2, lp.shape[1] - 1]))
            dump["logp_rows"] = np.array(rows, dtype=np.int64)
            dump["logp_sel"] = lp[:, rows, :].numpy()
            dump["logp_absmax"] = np.float64(lp.abs().max() if config != 4 else lp[:, rows, :].abs().max())
        if lp is not None:                                  # per-token top-2 of the oracle: classifies arg-max differences as near-ties
            t2 = torch.topk(lp, 2, dim=-1)
            dump["top2_idx"] = t2.indices.numpy().astype(np.int64)
            dump["top2_val"] = t2.values.numpy().astype(np.float64)
            dump["valid_len"] = (o["token_num"] if "token_num" in o else o["enc_lens"]).numpy().astype(np.int64)
        if "token_num" in o:
            dump["token_num"] = o["token_num"].numpy()
        for k, step in TAP_STRIDES.items():                 # stage taps (BASELINE.md §3.4): subsampled along time to keep the file small
            if k in o and o[k] is not None:
                dump["tap_" + k] = o[k][:, ::step].numpy() if step > 1 else o[k].numpy()
        if isinstance(ref_ids, list) and ref_ids and isinstance(ref_ids[0], list):
            dump["ref_equals_oracle"] = np.int64(int([list(map(int, r)) for r in ref_ids] == [list(map(int, r)) for r in o["ids"]]))
        np.savez(args.parity_out, **dump)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "audio-sec/s", "n_gpus": args.gpus, "steps": len(ts),
            "warmup": args.warmup, "ms_per_step": dt / len(ts) * 1000, "higher_is_better": True, "scaling": "weak" if config in (2, 4) else "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "BASELINE config %d (bounded CPU sample of the same job)" % config, "sample": sample, "bench_config": config},
            "cpu_baseline": cb,
            "e2e": {"value": val, "unit": "audio-sec/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def cpu_baseline(config, parity_path, time_cap_s=420):
    """This script's --impl reference leg in a subprocess with a hard time cap (rank 0, N=1 only)."""
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--config", str(config), "--steps", "5", "--warmup", "1",
                            "--parity-out", parity_path],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, timeout=time_cap_s, text=True,
                           env={**os.environ, "RANK": "0", "WORLD_SIZE": "1", "CUDA_VISIBLE_DEVICES": ""})
        for ln in r.stdout.splitlines():
            if ln.startswith("{"):
                return json.loads(ln)["cpu_baseline"]
        return {"error": "reference leg printed no JSON (rc=%d)" % r.returncode}
    except subprocess.TimeoutExpired:
        return {"error": "CPU leg exceeded %d s" % time_cap_s}


# stage taps compared in the parity block: oracle tensor -> stride along the time / token axis
TAP_STRIDES = {"feats": 7, "enc": 7, "alphas": 1, "acoustic": 5}
TAP_BARS = {"feats": ("mean_abs", 2e-5), "enc": ("rel", 1e-3), "alphas": ("max_abs", 1e-4), "acoustic": ("rel", 1e-3)}


def compare_taps(dump, got):
    """Stage taps of the GPU path (dict of tensors: feats [b,T,560], enc [b,T,512], alphas [b,T+1], acoustic [b,>=n,512]) against the
    oracle's (`tap_*` arrays of the parity dump, subsampled by TAP_STRIDES) -> {name: {max_abs, mean_abs, rel, within}} with the bars the
    GPU parity tests use (tests/test_gpu_parity.py: log-mel mean 2e-5, encoder / acoustic 1e-3 relative, alpha 1e-4 absolute)."""
    out = {}
    for k, step in TAP_STRIDES.items():
        if "tap_" + k not in dump or k not in got or got[k] is None:
            continue
        ref = np.asarray(dump["tap_" + k], dtype=np.float64)
        g = got[k].detach().float().cpu().numpy().astype(np.float64)
        if k == "acoustic":
            g = g[:, : int(np.asarray(dump["token_num"]).max())] if "token_num" in dump else g
        g = g[:, ::step] if step > 1 else g
        if g.shape != ref.shape:
            out[k] = {"error": "shape %s vs oracle %s" % (list(g.shape), list(ref.shape))}
            continue
        d = np.abs(g - ref)
        r = {"max_abs": float(d.max()) if d.size else 0.0, "mean_abs": float(d.mean()) if d.size else 0.0,
             "rel": float(d.max() / max(float(np.abs(ref).max()), 1e-30)) if d.size else 0.0}
        kind, bar = TAP_BARS[k]
        r["bar"] = "%s <= %g" % (kind, bar)
        r["within"] = bool(r[kind] <= bar)
        out[k] = r
    return out


def parity_block(job, parity_path, last_ids):
    """ids of the TIMED job vs the oracle's for the sample; log-probs of an untimed taps pass over the same utterances."""
    d = dict(np.load(parity_path))
    idx = [int(i) for i in d["idx"]]
    want, pos = [], 0
    for n in d["ids_len"].tolist():
        want.append(d["ids_flat"][pos: pos + n].tolist())
        pos += n
    got = [list(map(int, last_ids[i])) for i in idx]
    out = {"oracle": "oracle/paraformer_oracle.py (CPU fp32 restatement, pinned to the unmodified reference by tests/golden)",
           "utterances": len(idx), "ids_equal": got == want, "ids_compared": int(sum(len(w) for w in want)),
           "source": "ids of the timed job (last timed step)"}
    if not out["ids_equal"]:
        out["first_mismatch"] = next(({"utt": idx[k], "got": g[:12], "want": w[:12]} for k, (g, w) in enumerate(zip(got, want)) if g != w), None)
    if "ref_equals_oracle" in d:
        out["reference_ids_equal_oracle"] = bool(int(d["ref_equals_oracle"]))
    if "logp_sel" in d:
        ws = [job.wavs[i] for i in idx]
        ln = [int(w.numel()) for w in ws]
        pad = torch.nn.utils.rnn.pad_sequence(ws, batch_first=True).to(job.dev)
        lens_dev = torch.tensor(ln, dtype=torch.int32, device=job.dev)
        rows = d["logp_rows"].tolist()
        if job.config == 4:
            o = job.eng.forward_wav(pad, lens_dev, ln, want_taps=True)
            lp = o["logp"][:, rows, :].cpu().numpy()
        else:
            feats, fl = job.fe(pad, lens_dev, max(job.num_lfr_frames(n) for n in ln))
            o = job.eng.forward_feats(feats, fl, want_taps=True)
            lp = o["logp"][:, rows, :].cpu().numpy()
            if "token_num" in d:
                out["token_num_equal"] = o["token_num"].tolist() == d["token_num"].tolist()
        if job.config != 4:
            try:
                out["taps"] = compare_taps(d, {"feats": feats, "enc": o.get("enc"), "alphas": o.get("alphas"), "acoustic": o.get("acoustic")})
            except Exception as e:  # pragma: no cover
                out["taps"] = {"error": repr(e)[:200]}
        ref = d["logp_sel"]
        out["logp_rel_err"] = float(np.abs(lp.astype(np.float64) - ref).max() / max(float(np.abs(ref).max()), 1e-30))
        out["logp_tolerance"] = 1e-3
        out["taps_ids_equal"] = [list(map(int, r)) for r in o["ids"]] == want
        if "top2_idx" in d:
            # every arg-max over the sample, token by token: a difference is a NEAR-TIE when the oracle's own top-2 margin is inside
            # twice the allowed log-prob deviation (1e-3 of max |logp|, the north star's tolerance) and the GPU picked the oracle's
            # runner-up — there the greedy id is not a well-defined function of the input at the stated floating-point tolerance
            am = o["argmax"].cpu().numpy()
            full = o["logp"].double().cpu().numpy()
            n_c = min(am.shape[1], d["top2_idx"].shape[1])
            valid = np.arange(n_c)[None, :] < d["valid_len"][:, None]
            t1, t2 = d["top2_idx"][:, :n_c, 0], d["top2_idx"][:, :n_c, 1]
            margin = d["top2_val"][:, :n_c, 0] - d["top2_val"][:, :n_c, 1]
            diff = (am[:, :n_c] != t1) & valid
            tol_abs = 2e-3 * float(d["logp_absmax"])
            near = diff & (am[:, :n_c] == t2) & (margin <= tol_abs)
            bi, ti = np.nonzero(valid)
            noise = np.abs(full[bi, ti, t1[valid]] - d["top2_val"][:, :n_c, 0][valid])
            out.update(argmax_tokens=int(valid.sum()), argmax_mismatches=int(diff.sum()), near_tie_mismatches=int(near.sum()),
                       mismatch_margins=[float(x) for x in margin[diff][:16]], near_tie_margin_bound=tol_abs,
                       min_top2_margin=float(margin[valid].min()), abs_err_at_top1_max=float(noise.max()),
                       ids_equal_outside_near_ties=bool(int(diff.sum()) == int(near.sum())))
    return out


def dump_outputs(out_dir, ids):
    """--dump-outputs: what a caller of the timed path receives from its last step, the greedy token ids of every utterance of the
    job in input order, so that two builds can be compared output for output on the same seeded inputs.  float64 (ids are exact):
    token_ids.npy [utterances, longest] padded with -1, token_lens.npy [utterances]; under 1 MB for every config."""
    os.makedirs(out_dir, exist_ok=True)
    rows = [[int(t) for t in r] for r in ids]
    out = np.full((len(rows), max((len(r) for r in rows), default=0)), -1.0, dtype=np.float64)
    for i, r in enumerate(rows):
        out[i, :len(r)] = r
    np.save(os.path.join(out_dir, "token_ids.npy"), out)
    np.save(os.path.join(out_dir, "token_lens.npy"), np.array([len(r) for r in rows], dtype=np.float64))


# ------------------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", type=int, default=int(os.environ.get("FA_BENCH_CONFIG", "2")), choices=[2, 3, 4, 5])
    ap.add_argument("--mode", default=os.environ.get("FA_GEMM_MODE", "fp16x3"))
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--parity-out", default=None, help="(reference leg) write the oracle's ids / log-probs of the sample here")
    ap.add_argument("--port", action="store_true", help="(reference leg) time the oracle port even when the reference imports")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the token ids of the last timed step to DIR/token_ids.npy and DIR/token_lens.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the timed GPU path's outputs; --impl reference times a CPU sample of the job instead")
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist
    from funasr_b200 import _abi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":   # NCCL would print its banner to stdout ahead of the one JSON line
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    lib = _abi.load()
    args.warmup = max(args.warmup, 3)
    job = Job(args.config, args.mode, dev, rank, world)
    log("config %d ready (mode %s, %d local utterances in %d buckets), warm-up" % (args.config, args.mode, len(job.wavs), len(job.plan["buckets"])))

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        h = job.step_device()
    torch.cuda.synchronize(dev)
    job.tok_stats.clear()
    log("timed region")
    sync_all()
    sampler = ClockSampler(local) if rank == 0 else None
    l0 = lib.fa_launch_count()
    r0 = getattr(job.eng, "replayed_launches", 0)       # kernels replayed from the decoder's CUDA graph are not seen by the C-side counter
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        h = job.step_device()
    for p in job._pending:                               # the (asynchronous) gathers of the last jobs are part of the timed work
        if p is not None and p[1] is not None:
            p[1].wait()
    e1.record()
    sync_all()
    launches = int(lib.fa_launch_count() - l0) + int(getattr(job.eng, "replayed_launches", 0) - r0)
    my_ms = e0.elapsed_time(e1)
    ms = torch.tensor([my_ms], device=dev)
    per_rank = [my_ms]
    if world > 1:
        allms = torch.empty(world, device=dev)
        dist.all_gather_into_tensor(allms, ms)
        per_rank = [float(x) for x in allms.tolist()]
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    last_ids = job.runner_dev.finish(h, job.plan["n_total"])       # id lists of the last timed job, all utterances, input order
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_ids)
    toks = torch.cat([t.float() for t in job.tok_stats]) if job.tok_stats else torch.zeros(1)
    ntok_mean, n_max = float(toks.mean()), int(toks.max())
    log("device-resident: %.2f ms/step" % (ms_total / args.steps))

    # ---- e2e: plugin call(s), host (pinned) waveforms in -> token ids on the host out
    for _ in range(2):
        res = job.step_e2e()
    sync_all()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = job.step_e2e()
    torch.cuda.synchronize(dev)
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_s = float(e2e_s.item())
    clocks = sampler.stop() if sampler else None
    log("e2e done: %.2f ms/step" % (e2e_s / args.steps * 1e3))

    if rank == 0:
        pk, pk_src = peaks()
        value = job.audio_seconds * args.steps / (ms_total / 1000)
        flops_job = job.flops_whole_job(ntok_mean)
        ach = flops_job * args.steps / (ms_total / 1000) / 1e12
        roof = None
        try:
            roof = dominant_gemm_roofline(lib, job, dev, args.mode, pk, pk_src)
        except Exception as e:  # pragma: no cover
            roof = {"error": str(e)}
        local_samples = sum(int(w.numel()) for w in job.wavs.values())
        rows_bytes = job.plan["per"] * (job.plan["width"] + 2) * 4
        if world == 1 and args.config == 2:
            d2h = 64 * 4 + 64 * n_max * 4 + 64 * 4
        else:
            d2h = world * rows_bytes
        line = {"metric": METRIC, "value": value, "unit": "audio-sec/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak" if args.config in (2, 4) else "strong",
                "vs_baseline": None,
                "dtype": {"fp32": "f32", "fp16x3": "fp16x3->f32", "fp16x6": "fp16x6->f32", "fp16": "fp16"}[args.mode],
                "data": "synthetic",
                "config": {"workload": job.workload_name(), "bench_config": args.config, "utterances_total": len(job.n_all),
                           "utterances_this_gpu": len(job.wavs), "batches_this_gpu": len(job.plan["buckets"]),
                           "audio_seconds_total": job.audio_seconds, "gemm_mode": args.mode, "tokens_per_utt_mean": ntok_mean, "n_max": n_max,
                           "parallelism": "utterance-sharded dp%d, one asynchronous all-gather of id rows per job" % world,
                           "l2": "per-step working set (0.9 GB weights + >1 GB activations) exceeds the 126 MB L2; no flush needed",
                           "algorithmic_gflop_per_job": flops_job / 1e9},
                "clocks": clocks,
                "e2e": {"value": job.audio_seconds * args.steps / e2e_s, "unit": "audio-sec/s", "h2d_bytes_per_step": local_samples * 4 + len(job.wavs) * 4,
                        "d2h_bytes_per_step": d2h,
                        "api": "ParaformerB200.inference(list of pinned host waveforms)" if (world == 1 and args.config == 2) else
                               "ShardedRunner over %s.infer_ids_device(list of pinned host waveforms) + all-gather + D2H of id rows" % type(job.model).__name__},
                "gpu_launches": launches,
                "per_rank_ms_per_step": [x / args.steps for x in per_rank],
                "achieved_tflops_algorithmic": ach,
                "step_frac_of_sustained_peak": ach / world / pk.get("bf16_tflops_sustained", 1400.0),
                "roofline": roof}
        if world == 1 and not args.no_cpu_baseline:
            try:
                log("cpu baseline leg + parity")
                with tempfile.TemporaryDirectory() as td:
                    pp = os.path.join(td, "parity.npz")
                    line["cpu_baseline"] = cpu_baseline(args.config, pp)
                    if os.path.exists(pp):
                        line["parity"] = parity_block(job, pp, last_ids)
            except Exception as e:  # pragma: no cover
                line["cpu_baseline"] = {"error": str(e)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def dominant_gemm_roofline(lib, job, dev, mode, pk, pk_src):
    """The dominant kernel = the tcgen05 GEMM.  Timed ALONE — exactly the launch the encoder makes for FFN w_1 (A operand = the
    fp16 planes LayerNorm wrote, plane-emitting epilogue: gemm_tc2_kernel<3,2,EPI_PLANES>) at this job's largest batch — with CUDA
    events on the launching stream, L2 flushed between launches; algorithmic flops 2MNK vs the measured fp16 burst peak."""
    import ctypes as C
    from funasr_b200 import _abi
    eng = job.eng
    b0 = max(job.plan["buckets"], key=lambda b: len(b) * max(job.n_all[i] for i in b))
    T = max(job.num_lfr_frames(job.n_all[i]) for i in b0) + (4 if job.config == 4 else 0)
    M, K, N = len(b0) * T, 512, 2048
    lin = (eng._keep_structs[0] if job.config == 4 else eng.enc_layers)[1].w1
    x = torch.randn(M, K, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    passes = {"fp32": 1, "fp16": 1, "fp16x3": 3, "fp16x6": 6}[mode]
    algo = 2.0 * M * N * K
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    gm = _abi.GEMM_MODES[mode]
    npl = {"fp16": 1, "fp16x3": 2, "fp16x6": 3}.get(mode, 0)
    if not npl:
        return {"bound": "fp32-simt", "kernel": "gemm_f32_kernel", "achieved": None, "peak": None, "unit": "TFLOP/s", "frac": None, "traffic": None}
    planes = torch.empty(npl, M, K, dtype=torch.float16, device=dev)
    outp = torch.empty(npl, M, N, dtype=torch.float16, device=dev)
    _abi.check(lib.fa_split_rows(x.data_ptr(), K, M, K, K, npl, planes.data_ptr(), st), "fa_split_rows")
    times = []
    for i in range(9):
        flush.zero_()                                      # L2 flush between timed launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _abi.check(lib.fa_linear_planes_to_planes(planes.data_ptr(), M, C.byref(lin), 1, outp.data_ptr(), N, gm, st), "fa_linear_planes_to_planes")
        e1.record()
        torch.cuda.synchronize(dev)
        if i >= 3:
            times.append(e0.elapsed_time(e1))
    ms = sum(times) / len(times)
    ach = algo / (ms / 1e3) / 1e12
    peak = pk.get("bf16_tflops", 1590.0)
    traffic, tsrc = None, "no ncu capture of this build committed (profiles/r2_ncu_w1_traffic.json)"
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_w1_traffic.json")))
        if int(t.get("M", 0)) == M:
            traffic, tsrc = float(t["dram_read_bytes"]) + float(t["dram_write_bytes"]), "profiles/r2_ncu_w1_traffic.json (%s)" % t.get("source", "ncu --set full")
        else:
            tsrc = "profiles/r2_ncu_w1_traffic.json was captured at M=%s, this launch has M=%d" % (t.get("M"), M)
    except Exception:
        pass
    return {"bound": "tensor", "kernel": "gemm_tc2_kernel<3,2,EPI_PLANES> (FFN w_1 as the encoder launches it: M=%d N=2048 K=512, %s, cta_group::2, "
                                         "fp16 planes in, ReLU fp16 planes out)" % (M, mode),
            "achieved": ach, "peak": peak, "peak_source": pk_src + " fp16 burst (MEASURED_PEAKS.json)", "unit": "TFLOP/s", "frac": ach / peak,
            "traffic": traffic, "traffic_source": tsrc,
            "algorithmic_bytes": float(npl * M * K * 2 + 2 * N * K * 2 + npl * M * N * 2),
            "ms": ms, "tensor_passes": passes, "tensor_issue_tflops": ach * passes, "tensor_issue_frac": ach * passes / peak,
            "note": "achieved = ALGORITHMIC fp32-equivalent flops (2MNK) / event time; the fp16x3 split issues 3 fp16 MMAs per product for "
                    "~2^-17 relative accuracy, so the tensor pipe runs at tensor_issue_frac of the measured peak"}


if __name__ == "__main__":
    main()
