#!/usr/bin/env python
"""bench.py -- utterances/sec of the Speech2Text hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # espnet_b200 CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU Speech2Text (oracle/_ref) on the host cores
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's hypotheses as DIR/*.npy

A "step" is one pass of the hot path over one batch of synthetic 16 kHz waveforms: BASELINE.json configs[1],
Conformer-large (12L/512d/8h, ff 2048, conv2d, macaron, rel-pos latest, kernel 31) + 6L Transformer decoder,
V=5000, joint CTC/attention decoding (ctc_weight 0.3, beam 10, maxlenratio -64), batch 64 x 30 s per GPU.
`value` times encode+search with the waveforms resident in HBM; `e2e` times Speech2Text.batch_decode_padded from
pinned host memory to host-side hypotheses (H2D + D2H inside the timed region).  Multi-GPU: utterances are
sharded (weak scaling, one batch per rank, no data-path collective) and the final hypotheses are all-gathered.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    # name: (model cfg, seconds, batch per GPU, beam, ctc_weight, maxlenratio)
    "conformer_large_joint_64x30s": (dict(d_model=512, heads=8, ff=2048, enc_layers=12, dec_layers=6, vocab=5000, kernel=31), 30, 64, 10, 0.3, -64.0),
    "conformer_large_joint_32x15s": (dict(d_model=512, heads=8, ff=2048, enc_layers=12, dec_layers=6, vocab=5000, kernel=31), 15, 32, 10, 0.3, -64.0),
    "conformer_4l256_joint_8x5s": (dict(d_model=256, heads=4, ff=2048, enc_layers=4, dec_layers=2, vocab=5000, kernel=31), 5, 8, 10, 0.3, -16.0),
    # next scope row (SURVEY.md 8f-1 / BASELINE configs[4]): Transformer 24L/1024d/16h enc + 6L dec, attention-only beam 5; 64 utterances per GPU
    # keep the conv1 planes within HBM (measured line: profiles/r02_bench_transformer_24l1024_att_64x30s_n1.json).
    "transformer_24l1024_att_64x30s": (dict(d_model=1024, heads=16, ff=4096, enc_layers=24, dec_layers=6, vocab=5000, encoder="transformer"),
                                       30, 64, 5, 0.0, -64.0),
}
# The one decoding setup the reference publishes an RTF for (BASELINE.md section 1: egs2/librispeech/asr1/conf/decode_asr.yaml:1-3, beam 60 / ctc 0.3 /
# lm 0.6 with a Transformer LM): the same Conformer-large + the Librispeech LM shape (16L / 512d / 8h / 2048 units, embed 128), 16 utterances per GPU.
WORKLOADS["conformer_large_lm_beam60_16x30s"] = (WORKLOADS["conformer_large_joint_64x30s"][0], 30, 16, 60, 0.3, -64.0)
LM_FUSION = {"conformer_large_lm_beam60_16x30s": dict(weight=0.6, conf=dict(pos_enc="sinusoidal", embed_unit=128, att_unit=512, head=8, unit=2048, layer=16))}
METRIC = "utterances/sec (RTF) Conformer-large ASR inference at 1/2/4/8 B200 vs CPU ref"
# BASELINE.json configs[3] (next row 8f-2): contextual-block Conformer (12L/512d/8h, block 40 / hop 16 / look-ahead 16), 128 live streams per GPU,
# 40-ms pushes (640 samples).  One "step" = 64 pushes (2.56 s of audio per stream); value = audio seconds processed per second (all streams).
STREAMING = {"streaming_cbconformer_128x40ms": dict(streams=128, push=640, pushes_per_step=64, d_model=512, heads=8, ff=2048, layers=12, vocab=5000)}


def waveforms(n, nsamples, offset=0):
    out = torch.empty(n, nsamples)
    for i in range(n):
        g = torch.Generator().manual_seed(1234 + offset + i)
        out[i] = 0.1 * torch.randn(nsamples, generator=g)
    return out


_WEIGHTS = {}


def model_weights(cfg):
    """Random-init (PyTorch default init, seed 0) weights with the reference's parameter names; built once per process."""
    from gpu_util import random_weights

    key = tuple(sorted(cfg.items()))
    if key not in _WEIGHTS:
        _WEIGHTS[key] = random_weights(cfg, seed=0)
    return _WEIGHTS[key]


def lm_weights(workload, vocab):
    """Random-init (seed 1) TransformerLM weights with the reference's parameter names (espnet2/lm/transformer_lm.py), or None."""
    spec = LM_FUSION.get(workload)
    if spec is None:
        return None
    key = ("lm", workload)
    if key not in _WEIGHTS:
        import espnet_b200

        torch.manual_seed(1)
        _WEIGHTS[key] = {k: v.detach().clone() for k, v in espnet_b200.TransformerLM(vocab, **spec["conf"]).state_dict().items()}
    return _WEIGHTS[key]


# ----------------------------------------------------------------------------------------------- reference CPU path
# The reference's own espnet2.bin.asr_inference.Speech2Text (unmodified files under oracle/_ref, made by oracle/install_ref.py where
# /root/reference is mounted; it travels to the GPU box with the snapshot), batch-1 as the reference decodes, FULL search (all
# |maxlenratio| steps) -- no extrapolation.  The reference parallelises decoding by running independent processes over slices of the key
# file (egs2/TEMPLATE/asr1/asr.sh:1591-1618, `inference_nj`): the CPU arm does the same with REF_WORKERS processes x REF_THREADS torch
# threads (fixed numbers, stated in the line; one process with all host threads is far slower: the search is thousands of tiny ops).
REF_THREADS = 8


def ref_workers():
    """Decoding processes of the CPU arm.  Default 1: the reference decodes batch-1 in one process, and one 30-s utterance takes ~13 s on 8 threads,
    which lets the arm honour the driver's --steps within a few minutes.  ESPB_REF_WORKERS=8 (8 x 8 threads) was measured on the 128-thread GPU host:
    51 s per step of 8 utterances = 0.156 utt/s, i.e. 2x the single process -- the processes slow each other down 4x."""
    return int(os.environ.get("ESPB_REF_WORKERS", 1))


def ref_kind():
    from oracle import install_ref

    return "reference" if install_ref.available() else "port"


def _ref_worker(rank, cfg, wfile, beam, ctcw, mlr, inq, outq, lm_spec=None):
    """One decoding process: builds the CPU Speech2Text once, then decodes the waveforms it is sent."""
    import torch as _t

    _t.set_num_threads(REF_THREADS)
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    weights = _t.load(wfile)
    from oracle import install_ref

    if install_ref.available():
        install_ref.activate()
        import logging

        import refbuild

        logging.disable(logging.WARNING)
        kw = {}
        if lm_spec is not None:      # LM shallow fusion exactly as a user passes it: lm_train_config (asr_inference.py:178-191)
            import tempfile

            import yaml

            lm_yaml = os.path.join(tempfile.mkdtemp(prefix="espb_ref_lm_"), "lm.yaml")
            with open(lm_yaml, "w") as f:
                yaml.safe_dump(dict(token_list=refbuild.token_list(cfg["vocab"]), lm="transformer", model_conf={}, init=None, use_preprocessor=False,
                                    lm_conf=dict(dropout_rate=0.1, positional_dropout_rate=0.1, attention_dropout_rate=0.1, **lm_spec["conf"])), f)
            kw = dict(lm_train_config=lm_yaml, lm_file=None, lm_weight=lm_spec["weight"])
        s2t = refbuild.build_reference(cfg, seed=0, beam_size=beam, ctc_weight=ctcw, maxlenratio=mlr, nbest=1, **kw)
        s2t.asr_model.load_state_dict(weights["asr"] if "asr" in weights else weights, strict=True)   # same weights as the CUDA arm (parity check of the bench)
        s2t.asr_model.eval()
        if lm_spec is not None:
            s2t.beam_search.full_scorers["lm"].load_state_dict(weights["lm"], strict=True)
        run = lambda w: s2t(w.numpy())  # noqa: E731
    else:
        import oracle

        if lm_spec is not None:
            raise RuntimeError("the LM-fusion workload needs the real reference (oracle/_ref) on the CPU arm")
        o = oracle.OracleSpeech2Text(cfg, weights, beam_size=beam, ctc_weight=ctcw, maxlenratio=mlr, nbest=1)
        run = lambda w: o(w)  # noqa: E731
    outq.put(("ready", rank))
    while True:
        item = inq.get()
        if item is None:
            return
        idx, wave = item
        t0 = time.perf_counter()
        res = run(wave)
        dt = time.perf_counter() - t0
        outq.put((idx, dt, res[0][3].yseq.tolist() if res else None, float(res[0][3].score) if res else None))


class RefPool:
    """REF_WORKERS reference decoders; decode(waves) runs one utterance per worker concurrently and returns the wall time."""

    def __init__(self, cfg, beam, ctcw, mlr, workers, workload=None):
        import tempfile

        import torch.multiprocessing as mp

        self.n = workers
        ctx = mp.get_context("spawn")
        self.wfile = os.path.join(tempfile.mkdtemp(prefix="espb_ref_"), "weights.pt")
        lm_spec, lmw = LM_FUSION.get(workload), lm_weights(workload, cfg["vocab"])
        torch.save(model_weights(cfg) if lmw is None else {"asr": model_weights(cfg), "lm": lmw}, self.wfile)
        self.inq = [ctx.Queue() for _ in range(workers)]
        self.outq = ctx.Queue()
        self.procs = [ctx.Process(target=_ref_worker, args=(r, cfg, self.wfile, beam, ctcw, mlr, self.inq[r], self.outq, lm_spec), daemon=True)
                      for r in range(workers)]
        for p in self.procs:
            p.start()
        for _ in range(workers):
            assert self.outq.get(timeout=900)[0] == "ready"

    def decode(self, waves):
        assert len(waves) <= self.n
        t0 = time.perf_counter()
        for r, w in enumerate(waves):
            self.inq[r].put((r, w))
        out = [self.outq.get(timeout=3600) for _ in range(len(waves))]
        wall = time.perf_counter() - t0
        return wall, sorted(out)

    def close(self):
        for q in self.inq:
            q.put(None)
        for p in self.procs:
            p.join(timeout=30)


def ref_sample_desc(secs, mlr, workers, beam, workload=None):
    return (f"{workers} utterance(s) of {secs} s decoded concurrently, one per process ({workers} processes x {REF_THREADS} torch threads of "
            f"{os.cpu_count()} host threads), each batch-1 through {'espnet2.bin.asr_inference.Speech2Text (oracle/_ref)' if ref_kind() == 'reference' else 'the oracle port'}: "
            f"encoder + the full {int(-mlr)}-step joint beam-{beam} search"
            + (f" with TransformerLM shallow fusion (lm_weight {LM_FUSION[workload]['weight']})" if workload in LM_FUSION else "") + ", no extrapolation")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json, bf16 sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------- reference arm (CPU)
def run_reference(args, rank, world):
    """Reference arm: one step = REF_WORKERS utterances of the workload decoded concurrently by the reference's own CPU Speech2Text
    (a bounded sample of the 64-utterance batch).  value = utterances / wall time over exactly --steps timed steps.  A CPU decode needs
    one warm-up, not W: min(W, 1) are run."""
    if rank != 0:
        return
    cfg, secs, batch, beam, ctcw, mlr = WORKLOADS[args.workload]
    workers = ref_workers()
    pool = RefPool(cfg, beam, ctcw, mlr, workers, args.workload)
    warm = min(args.warmup, 1)
    waves = waveforms((warm + args.steps) * workers, secs * 16000)
    k = 0
    for i in range(warm):
        pool.decode(list(waves[k:k + workers])); k += workers
    walls = []
    for i in range(args.steps):
        w, _ = pool.decode(list(waves[k:k + workers])); k += workers
        walls.append(w)
    pool.close()
    done = len(walls)
    dt = sum(walls)
    ups = done * workers / dt
    desc = ref_sample_desc(secs, mlr, workers, beam, args.workload)
    line = {
        "impl": "reference", "metric": METRIC, "value": ups, "unit": "utterances/s", "n_gpus": args.gpus, "steps": done,
        "warmup": warm, "ms_per_step": 1000.0 * dt / done, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "rtf": (dt / (done * workers)) / secs,
        "config": {"workload": args.workload, "sample": "per step: " + desc, "beam": beam, "global_batch": batch,
                   "ctc_weight": ctcw, "maxlenratio": mlr, "utt_seconds": secs, "vocab": cfg["vocab"],
                   "steps_requested": args.steps, "warmup_requested": args.warmup,
                   "note": "a CPU decode needs no more than one warm-up"},
        "cpu_baseline": {"value": ups, "unit": "utterances/s", "cores": workers * REF_THREADS, "kind": ref_kind(),
                         "sample": f"{done} steps, each: {desc}; {warm} warm-up"},
        "e2e": {"value": ups, "unit": "utterances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- espnet_b200 arm
# DRAM traffic of ONE launch of the dominant kernel, from the committed `ncu --set full` capture (scripts/gpu_ncu_micro.sh ffn 2cta):
# the encoder feed-forward w_1 GEMM of this workload (M 59968, N 2048, K 512, Swish, hi/lo split output).  dram__bytes_read.sum +
# dram__bytes_write.sum; the algorithmic bytes are the hi/lo A and B planes read once and the hi/lo C planes written once.
NCU_TRAFFIC = {"launch": "gemm_tf32x3_2cta_kernel<256,3,swish,split> M59968 N2048 K512", "dram_bytes": 275.803136e6 + 959.088128e6,
               "algorithmic_bytes": (2 * 59968 * 512 + 2 * 2048 * 512 + 2 * 59968 * 2048) * 4.0, "gpu_time_us_under_ncu": 627.264,
               "tensor_pipe_active_pct": 61.13, "source": "profiles/r01_ncu_gemm_2cta_ffn_w1_summary.txt"}


def _load_ncu_traffic():
    """Prefer the round-2 capture of the same launch (16-warp epilogue) when its summary is committed: profiles/r02_ncu_gemm_2cta_ffn_w1_ew16_summary.txt,
    written by scripts/ncu_summary.py from `ncu --set full` of scripts/gemm_enc_microbench.py (scripts/gpu_final.sh)."""
    path = os.path.join(ROOT, "profiles", "r02_ncu_gemm_2cta_ffn_w1_ew16_summary.txt")
    if not os.path.exists(path):
        return
    vals = {}
    with open(path) as f:
        for ln in f:
            parts = ln.split()
            if len(parts) >= 3 and parts[0] in ("gpu__time_duration.sum", "dram__bytes_read.sum", "dram__bytes_write.sum",
                                                "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active"):
                scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0, "us": 1.0, "ms": 1e3, "ns": 1e-3, "%": 1.0}.get(parts[2], 1.0)
                vals.setdefault(parts[0], float(parts[1].replace(",", "")) * scale)
    if len(vals) == 4:
        NCU_TRAFFIC.update(dram_bytes=vals["dram__bytes_read.sum"] + vals["dram__bytes_write.sum"], gpu_time_us_under_ncu=vals["gpu__time_duration.sum"],
                           tensor_pipe_active_pct=vals["sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active"],
                           source="profiles/r02_ncu_gemm_2cta_ffn_w1_ew16_summary.txt")


_load_ncu_traffic()


def run_streaming(args, rank, local_rank, world):
    """Streaming workload: frontend chunking -> ContextualBlockConformerEncoder.forward_infer -> CTC greedy, N streams in lock step."""
    import argparse as _ap

    import torch.distributed as dist

    import espnet_b200
    from espnet_b200 import ops
    from gpu_util import refbuild

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    w = STREAMING[args.workload]
    y = refbuild.model_yaml(dict(d_model=w["d_model"], heads=w["heads"], ff=w["ff"], enc_layers=w["layers"], dec_layers=1, vocab=w["vocab"], kernel=31))
    y.update(encoder="contextual_block_conformer", normalize=None, normalize_conf={}, decoder=None,
             encoder_conf=dict(output_size=w["d_model"], attention_heads=w["heads"], linear_units=w["ff"], num_blocks=w["layers"], macaron_style=True,
                               cnn_module_kernel=31, block_size=40, hop_size=16, look_ahead=16))
    torch.manual_seed(0)
    model = espnet_b200.build_model(_ap.Namespace(**y)).to(dev).eval()
    s2t = espnet_b200.Speech2TextStreaming(model, n_streams=w["streams"], device=str(dev), greedy=True)
    host = waveforms(w["streams"], w["push"] * w["pushes_per_step"], offset=rank * w["streams"]).pin_memory()

    def step():
        n_tok = 0
        for p in range(w["pushes_per_step"]):
            new = s2t(host[:, p * w["push"]:(p + 1) * w["push"]], is_final=False)     # pinned host chunk -> device inside the call
            n_tok += sum(len(t) for t in new)
        return n_tok

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local_rank)
    barrier(); sampler.start(); ops.launch_counter[0] = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    if rank != 0:
        return
    audio_s = world * w["streams"] * w["pushes_per_step"] * args.steps * w["push"] / 16000.0
    val = audio_s / (ms / 1000.0)
    line = {"metric": "audio seconds per second, streaming contextual-block Conformer + CTC greedy (BASELINE configs[3] shape)", "value": val,
            "unit": "audio-s/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "streams_per_gpu": w["streams"], "push_ms": 1000.0 * w["push"] / 16000.0,
                       "pushes_per_step": w["pushes_per_step"], "real_time_streams_sustained": val, "ms_per_push": ms / args.steps / w["pushes_per_step"],
                       "model": "contextual-block Conformer 12L/512d/8h block 40 hop 16 look-ahead 16, V=5000, CTC greedy",
                       "note": "next-row workload (SURVEY 8f-2): host chunks are copied inside the timed region; no beam search"},
            "e2e": {"value": val, "unit": "audio-s/s", "h2d_bytes_per_step": w["streams"] * w["push"] * w["pushes_per_step"] * 4, "d2h_bytes_per_step": 0},
            "gpu_launches": ops.launch_counter[0], "clocks": clocks}
    print(json.dumps(line), flush=True)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, results, nbest):
    """Write what BatchBeamSearch.forward_batch returned (per utterance, its hypotheses sorted best first) as float64 arrays, the top
    `nbest` of each utterance: hyp_yseq (U, nbest, L) padded with -1, hyp_score (U, nbest) and hyp_score_<scorer> per scorer, NaN where an
    utterance has fewer hypotheses.  Inputs are seeded, so two builds run with the same arguments can be compared array by array."""
    import numpy as np

    U = len(results)
    L = max((len(h.yseq) for hyps in results for h in hyps[:nbest]), default=0)
    keys = sorted({k for hyps in results for h in hyps[:nbest] for k in h.scores})
    arrays = {"hyp_yseq": np.full((U, nbest, L), -1.0), "hyp_score": np.full((U, nbest), np.nan)}
    arrays.update({f"hyp_score_{k}": np.full((U, nbest), np.nan) for k in keys})
    for u, hyps in enumerate(results):
        for j, h in enumerate(hyps[:nbest]):
            y = h.yseq.tolist()
            arrays["hyp_yseq"][u, j, :len(y)] = y
            arrays["hyp_score"][u, j] = float(h.score)
            for k, v in h.scores.items():
                arrays[f"hyp_score_{k}"][u, j] = float(v)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return sorted(arrays)


def run_b200(args, rank, local_rank, world):
    import torch.distributed as dist

    import espnet_b200
    from espnet_b200 import ops
    from gpu_util import speech2text

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    cfg, secs, batch, beam, ctcw, mlr = WORKLOADS[args.workload]
    nsamp = secs * 16000
    kw = {}
    if args.workload in LM_FUSION:
        import espnet_b200 as _eb

        spec = LM_FUSION[args.workload]
        lm = _eb.TransformerLM(cfg["vocab"], **spec["conf"])
        lm.load_state_dict(lm_weights(args.workload, cfg["vocab"]), strict=True)
        kw = dict(lm=lm, lm_weight=spec["weight"])
    s2t = speech2text(cfg, model_weights(cfg), beam_size=beam, ctc_weight=ctcw, maxlenratio=mlr, nbest=1, **kw)
    host = waveforms(batch, nsamp, offset=rank * batch).pin_memory()      # utterances sharded by rank
    lens = torch.full((batch,), nsamp, dtype=torch.long)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident(speech_dev):
        enc, enc_lens = s2t.asr_model.encode(speech_dev, lens)
        return s2t.beam_search.forward_batch(enc, enc_lens, s2t.asr_model.enc_split(enc), mlr, 0.0)

    def run_e2e(k, workload_host=None, workload_lens=None, engine=None):
        """k end-to-end steps through the public API: Speech2Text.decode_stream over pinned host batches (the H2D copy of step i+1 runs on a copy
        stream under the computation of step i), each step ending in host-side hypotheses; with several ranks every step also all-gathers the
        n-best records (Speech2Text.batch_decode_sharded, the single exchange of the path, SURVEY.md 8e).  Returns the last step's local results."""
        eng = engine or s2t
        hb, hl = (host, lens) if workload_host is None else (workload_host, workload_lens)

        def batches():
            for _ in range(k):
                flush.zero_()          # L2 flush between steps (inside the timed region: ~0.1 ms)
                yield hb, hl
        res, t_prev = None, time.perf_counter()
        for out in eng.decode_stream(batches(), sharded=world > 1):
            res = out[0] if world > 1 else out
            if os.environ.get("ESPB_BENCH_DEBUG"):
                torch.cuda.synchronize()
                print(f"[bench debug] rank {rank} e2e step wall {1e3 * (time.perf_counter() - t_prev):.1f} ms", file=sys.stderr, flush=True)
                t_prev = time.perf_counter()
        return res

    speech_dev = host.to(dev)
    for _ in range(args.warmup):
        step_resident(speech_dev)
    if args.breakdown:   # per-launch CUDA-event timing of one step, aggregated by kernel (and GEMM shape) -> stderr
        from espnet_b200 import lib as _lib
        import collections

        _lib.profile = []
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        step_resident(speech_dev)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        prof, _lib.profile = _lib.profile, None
        agg = collections.defaultdict(lambda: [0, 0.0])
        for name, tag, e0, e1 in prof:
            k = name.replace("espb_", "") + (" " + tag if tag else "")
            agg[k][0] += 1
            agg[k][1] += e0.elapsed_time(e1)
        tot = sum(v[1] for v in agg.values())
        print(f"[breakdown] {args.workload}: {len(prof)} launches, sum of kernel times {tot:.1f} ms, wall {wall * 1e3:.1f} ms", file=sys.stderr)
        for k, (c, ms) in sorted(agg.items(), key=lambda kv: -kv[1][1])[:60]:
            print(f"[breakdown] {100 * ms / tot:6.2f}%  {ms:9.3f} ms  {c:5d}x  avg {1e3 * ms / c:9.1f} us  {k}", file=sys.stderr)
        return
    if args.trace:   # CUPTI activity trace (torch.profiler) of one step: in-situ kernel durations inside the replayed CUDA graphs
        import collections
        import re as _re

        from torch.profiler import ProfilerActivity, profile

        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step_resident(speech_dev)
            torch.cuda.synchronize()
        evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and e.time_range.end > e.time_range.start]
        evs.sort(key=lambda e: e.time_range.start)
        agg = collections.defaultdict(lambda: [0, 0.0])
        for e in evs:
            name = _re.sub(r"^void |\(anonymous namespace\)::|<unnamed>::", "", e.name)
            name = _re.sub(r"\(.*", "", name)
            agg[name][0] += 1
            agg[name][1] += (e.time_range.end - e.time_range.start)
        t_first, t_last = evs[0].time_range.start, max(e.time_range.end for e in evs)
        busy, cur_end = 0.0, t_first           # union of kernel intervals (streams overlap)
        for e in evs:
            st, en = max(e.time_range.start, cur_end), e.time_range.end
            if en > st:
                busy += en - st
                cur_end = en
        # exclusive time per kernel name: the part of each interval during which no other kernel runs (what the kernel adds to the critical
        # path when branches of the step graph overlap, e.g. the CTC state recursion under the decoder pass)
        pts = sorted([(e.time_range.start, 1, i) for i, e in enumerate(evs)] + [(e.time_range.end, 0, i) for i, e in enumerate(evs)])
        excl = collections.defaultdict(float)
        live, last_t = set(), pts[0][0]
        for t, kind, i in pts:
            if len(live) == 1 and t > last_t:
                excl[next(iter(live))] += t - last_t
            last_t = t
            (live.add if kind == 1 else live.discard)(i)
        excl_by_name = collections.defaultdict(float)
        for i, v in excl.items():
            nm = _re.sub(r"\(.*", "", _re.sub(r"^void |\(anonymous namespace\)::|<unnamed>::", "", evs[i].name))
            excl_by_name[nm] += v
        if os.environ.get("ESPB_TRACE_DUMP"):   # timeline around the k-th CTC state recursion: which kernels overlap it
            adv = [i for i, e in enumerate(evs) if "ctc_advance" in e.name]
            if len(adv) > 10:
                i0 = adv[10]
                t0 = evs[i0].time_range.start
                for e in evs[max(0, i0 - 3): i0 + int(os.environ["ESPB_TRACE_DUMP"])]:
                    print(f"[timeline] {e.time_range.start - t0:9.1f} .. {e.time_range.end - t0:9.1f} us  {_re.sub(r"[(].*", "", _re.sub(r"^void |[(]anonymous namespace[)]::|<unnamed>::", "", e.name))[:60]}", file=sys.stderr)
        tot = sum(v[1] for v in agg.values())
        print(f"[trace] {args.workload}: {len(evs)} device activities, span {(t_last - t_first) / 1e3:.2f} ms, device busy (union) {busy / 1e3:.2f} ms, "
              f"sum of durations {tot / 1e3:.2f} ms", file=sys.stderr)
        for k, (c, us) in sorted(agg.items(), key=lambda kv: -kv[1][1])[:50]:
            print(f"[trace] {100 * us / tot:6.2f}%  {us / 1e3:9.3f} ms  {c:5d}x  avg {us / c:9.1f} us  exclusive {excl_by_name.get(k, 0.0) / 1e3:8.3f} ms  {k[:120]}",
                  file=sys.stderr)
        return
    if args.profile_one_step:   # for ncu --profile-from-start off: exactly one resident step inside the profiler range
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step_resident(speech_dev)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        if rank == 0:
            print(json.dumps({"profiled_one_step": True, "workload": args.workload, "launches_per_step": ops.launch_counter[0] // (args.warmup + 1)}))
        return
    run_e2e(max(1, min(args.warmup, 2)))

    # ---- timed: K resident steps (per-step CUDA events, L2 flushed between steps, not timed)
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    ops.launch_counter[0] = 0
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    wall0 = time.perf_counter()
    for a, b in ev:
        flush.zero_()
        a.record()
        res = step_resident(speech_dev)
        b.record()
    barrier()
    wall = time.perf_counter() - wall0
    launches = ops.launch_counter[0]
    res_resident = res
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    # ---- timed: K end-to-end steps (one event pair around all of them: consecutive steps overlap copy and compute)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    res = run_e2e(args.steps)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    n_hyp_tokens = sum(len(r[0][2]) for r in res if r)
    dumped = dump_outputs(args.dump_outputs, res_resident, beam) if args.dump_outputs and rank == 0 else None

    # ---- roofline of the dominant kernel (tcgen05 3xTF32 GEMM): per-launch CUDA events over one extra step
    ops.gemm_profile = []
    step_resident(speech_dev)
    torch.cuda.synchronize()
    prof = ops.gemm_profile
    ops.gemm_profile = None
    big = [p for p in prof if p[3]]          # gemm_tf32x3_2cta_kernel launches (the dominant kernel)
    small = [p for p in prof if not p[3]]    # gemm_tf32x3_kernel (1-CTA tiles, decode-step problems)
    g_flops = sum(p[0] for p in big)
    g_ms = sum(p[1].elapsed_time(p[2]) for p in big)
    s_flops = sum(p[0] for p in small)
    s_ms = sum(p[1].elapsed_time(p[2]) for p in small)
    peak_tf, hbm_gbs, peak_src = measured_peaks()
    # ---- the other kernels the north star names, timed live (CUDA events around every C-ABI call of one un-graphed step)
    from espnet_b200 import lib as _lib

    _lib.profile = []
    step_resident(speech_dev)
    torch.cuda.synchronize()
    calls, _lib.profile = _lib.profile, None
    tsum = {}
    for name, tag, a, b in calls:
        c = tsum.setdefault(name, [0, 0.0])
        c[0] += 1; c[1] += a.elapsed_time(b)
    Tf = 1 + nsamp // 128
    Tenc = ((Tf - 1) // 2 - 1) // 2
    H, dk = cfg["heads"], cfg["d_model"] // cfg["heads"]
    other = []

    def add(name, bound, work_per_launch, unit_scale, unit, peak, what):
        if name in tsum and tsum[name][1] > 0:
            n, ms = tsum[name]
            ach = work_per_launch * n / (ms / 1000.0) / unit_scale
            other.append({"kernel": name, "what": what, "bound": bound, "launches": n, "ms_per_step": ms, "achieved": ach, "peak": peak, "unit": unit,
                          "frac": ach / peak if peak else None})
    add("espb_stft_logmel_f32", "hbm", batch * (4.0 * nsamp + 320.0 * Tf), 1e9, "GB/s", hbm_gbs, "fused STFT + log-mel: waveform read + log-mel write")
    add("espb_flash_attn_f32", "tensor", 2 * 2.0 * batch * H * Tenc * Tenc * dk, 1e12, "TFLOP/s", peak_tf,
        "fused encoder self-attention: q k^T and p v (algorithmic FLOPs; executed as 3 tf32 MMAs each)")
    add("espb_dec_src_attn_f32", "hbm", 2.0 * batch * H * Tenc * dk * 4, 1e9, "GB/s", hbm_gbs, "decoder cross-attention: K / V memory read once per launch")

    # ---- BASELINE.json configs[2] (beam 10, 15-s utterances, 32 per GPU: 256 x 15 s on 8 GPUs), measured end to end in multi-GPU runs
    extra_ms, extra_name = 0.0, "conformer_large_joint_32x15s"
    if world > 1 and args.workload == "conformer_large_joint_64x30s":
        xcfg, xsecs, xbatch, xbeam, xctcw, xmlr = WORKLOADS[extra_name]
        xs2t = speech2text(xcfg, model_weights(xcfg), beam_size=xbeam, ctc_weight=xctcw, maxlenratio=xmlr, nbest=1)
        xhost = waveforms(xbatch, xsecs * 16000, offset=rank * xbatch).pin_memory()
        xlens = torch.full((xbatch,), xsecs * 16000, dtype=torch.long)
        run_e2e(2, xhost, xlens, xs2t)
        x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        x0.record()
        run_e2e(args.steps, xhost, xlens, xs2t)
        x1.record()
        barrier()
        extra_ms = x0.elapsed_time(x1)

    t = torch.tensor([dev_ms, e2e_ms, extra_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, extra_ms = t.tolist()
    if rank != 0:
        return
    utts = world * batch * args.steps
    value = utts / (dev_ms / 1000.0)
    e2e = utts / (e2e_ms / 1000.0)
    ach = g_flops / (g_ms / 1000.0) / 1e12 if g_ms > 0 else 0.0
    line = {
        "metric": METRIC, "value": value, "unit": "utterances/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "rtf": (dev_ms / 1000.0) / (utts * secs),
        "config": {"workload": args.workload, "global_batch": world * batch, "utt_seconds": secs, "beam": beam, "ctc_weight": ctcw,
                   "maxlenratio": mlr, "vocab": cfg["vocab"], "parallelism": f"utterance-sharded x{world}", "l2": "flushed between steps (256 MiB write)",
                   "gemm": "tcgen05 kind::tf32 x3 (error-compensated fp32), mode " + ops.gemm_mode(), "attention": ops.attn_mode(),
                   "wall_s_timed_region": wall,
                   **({"lm": {"type": "TransformerLM", "weight": LM_FUSION[args.workload]["weight"], **LM_FUSION[args.workload]["conf"]},
                       "decode_setup": "egs2/librispeech/asr1/conf/decode_asr.yaml:1-3 (beam 60, ctc 0.3, lm 0.6)"} if args.workload in LM_FUSION else {})},
        "e2e": {"value": e2e, "unit": "utterances/s", "h2d_bytes_per_step": batch * nsamp * 4,
                "d2h_bytes_per_step": int(2 * 4 * 64 * batch * beam + 6 * 4 * batch * beam * 64), "ms_per_step": e2e_ms / args.steps,
                "api": "Speech2Text.decode_stream (double-buffered pinned H2D)" + (" + batch_decode_sharded (all-gather of n-best records)" if world > 1 else ""),
                "hyp_tokens_last_step": n_hyp_tokens},
        "gpu_launches": launches,
        "clocks": clocks,
        **({"dumped_outputs": {"dir": args.dump_outputs, "arrays": dumped, "step": "last timed resident step (encode + search)"}} if dumped else {}),
        "roofline": {"bound": "tensor", "kernel": "gemm_tf32x3_2cta_kernel (all its launches in one step: encoder, CTC head, decoder memory)", "achieved": ach, "peak": peak_tf,
                     "unit": "TFLOP/s", "frac": ach / peak_tf if peak_tf else None, "traffic": NCU_TRAFFIC["dram_bytes"], "traffic_launch": NCU_TRAFFIC,
                     "peak_source": peak_src,
                     "launches": len(big), "gemm_ms_per_step": g_ms, "algorithmic_tflop_per_step": g_flops / 1e12,
                     "frac_of_3xtf32_ceiling": (ach / (peak_tf / 6.0)) if peak_tf else None,
                     "decode_gemm_1cta": {"kernel": "gemm_tf32x3_sk_kernel / gemm_tf32x3_mc_kernel / gemm_tf32x3_kernel (128-row 1-CTA tiles)", "launches": len(small), "ms_per_step_ungraphed": s_ms,
                                          "achieved": (s_flops / (s_ms / 1000.0) / 1e12) if s_ms > 0 else None},
                     "note": "algorithmic FLOPs (2MNK); each is executed as 3 tf32 MMAs at half the bf16 rate, so 1/6 of the bf16 peak is the ceiling of this formulation",
                     "other_kernels": other},
    }
    if extra_ms > 0:
        xb = WORKLOADS[extra_name][2]
        line["config"]["extra"] = {"workload": extra_name, "what": "BASELINE.json configs[2]: beam 10, 15-s utterances, 32 per GPU, end to end "
                                   "(pinned host waveforms -> all-gathered hypotheses)", "global_batch": world * xb, "steps": args.steps,
                                   "value": world * xb * args.steps / (extra_ms / 1000.0), "unit": "utterances/s", "ms_per_step": extra_ms / args.steps}
    print("[bench] gpu arm done: " + json.dumps(line), file=sys.stderr, flush=True)
    if args.cpu_baseline and world == 1:   # the host-core baseline is reported by the single-GPU run only
        workers = ref_workers()
        n_par = 1 if args.workload in LM_FUSION else 4   # parity is checked on more utterances than the timed sample (those run concurrently, untimed)
        pool = RefPool(cfg, beam, ctcw, mlr, max(workers, n_par), args.workload)
        wall, out = pool.decode([host[i] for i in range(workers)])      # the first `workers` utterances of this rank's batch, no warm-up
        _, more = pool.decode([host[workers + i] for i in range(n_par)])
        out = out + [(workers + i, dt, ys, sc) for i, dt, ys, sc in more]
        pool.close()
        line["cpu_baseline"] = {"value": workers / wall, "unit": "utterances/s", "cores": workers * REF_THREADS, "kind": ref_kind(),
                                "sample": ref_sample_desc(secs, mlr, workers, beam, args.workload) + "; one step, no warm-up"}
        # parity of the benchmarked configuration, enforced by the bench itself: the CUDA n-best of the same utterances (from the last timed
        # end-to-end step) against the reference CPU result -- identical token sequences, scores within rtol 2e-4
        eq, rel = True, 0.0
        for idx, _, yseq, score in out:
            g = res[idx][0][3] if res[idx] else None
            if g is None or yseq is None:
                eq = eq and (g is None and yseq is None)
                continue
            eq = eq and (g.yseq.tolist() == yseq)
            rel = max(rel, abs(float(g.score) - score) / max(1.0, abs(score)))
        line["parity_check"] = {"against": ref_kind(), "utterances": len(out), "search_steps": int(-mlr), "yseq_equal": bool(eq), "score_rel_err": rel,
                                "tolerance": "identical yseq, score rtol 2e-4"}
        if not eq or rel > 2e-4:
            print(json.dumps(line), flush=True)
            print("[bench] PARITY CHECK FAILED: " + json.dumps(line["parity_check"]), file=sys.stderr, flush=True)
            sys.exit(3)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="conformer_large_joint_64x30s", choices=sorted(WORKLOADS) + sorted(STREAMING))
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--trace", action="store_true", help="CUPTI activity trace of one step (kernel durations inside the CUDA graphs) -> stderr")
    ap.add_argument("--breakdown", action="store_true", help="time every launch of one step with CUDA events and print a per-kernel table")
    ap.add_argument("--profile-one-step", action="store_true", help="warm up, then run one step inside cudaProfilerStart/Stop and exit")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the hypotheses of the last timed step (rank 0's "
                    "utterances, top `beam` per utterance) as DIR/<name>.npy in float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload in STREAMING):
        ap.error("--dump-outputs is implemented for the espnet_b200 arm of the non-streaming workloads")
    rank, local_rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        (run_streaming if args.workload in STREAMING else run_b200)(args, rank, local_rank, world)
    finally:
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()


if __name__ == "__main__":
    main()
