#!/usr/bin/env python
"""bench.py -- RTFx (audio-seconds / second) of the ASR inference hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # our sm_100a path
    python bench.py --impl reference --gpus N --steps K ...   # the UNMODIFIED reference (baseline/_ref) on host CPU cores
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py ... --dump-outputs DIR                    # + the last timed step's outputs as DIR/<name>.npy

Default workload = BASELINE.json configs[2], the configuration the metric is quoted on: Conformer-L (conformer_large.yaml:
12L/512d/8h RoPEMHA encoder, 6L decoder, vocab 5000, n_fft=512), random init, batch = 32 x 10 s @ 16 kHz synthetic per GPU,
Fbank -> global CMVN -> CNN front-end -> encoder -> greedy search pinned to 48 decode steps (random weights never emit EOS;
SURVEY.md 8d).  One "step" = one pass of the whole path over one 32 x 10 s batch.  Weak scaling: every GPU gets its own
batches; the one exchange is an all-gather of the token ids (speechbrain_b200.parallel.gather_hypotheses, once per group
call, inside the timed region).

Other BASELINE configs (not the driver's line; run by hand, results in profiles/ and DESIGN.md):
    --config small_enc     configs[1]: Conformer-small (12L/144d/4h RelPosMHAXL) encoder-only, 8 x 5 s
    --config beam10_lm     configs[3]: Conformer-L, beam 10 + TransformerLM (0.6) + CTC (0.4) scorers, 16 x 10 s, 48 steps
    --config beam10_shard  configs[4]: Conformer-L, beam 10 (no scorer), 32 x 10 s per GPU, NCCL gather of the hypotheses

value  : device-timed throughput, wav already resident in HBM.  The K-step region is repeated --repeats times (>= 7 by
         default); the line reports the MEDIAN (max over ranks per repeat) and min / max beside it.
e2e    : the same K steps through the host-buffer C-ABI call EncoderDecoderASR.transcribe_batches_async ->
         sbk_asr_transcribe_greedy_group_host_async: pinned host wav -> H2D -> pipeline -> D2H token ids, all inside the
         timed region.
roofline: the dominant kernel (gemm_tc2_kernel, 2-CTA tcgen05) timed live per launch with CUDA events in a separate pass.
cpu_baseline / --impl reference: the reference's own modules (pip-installed copy under baseline/_ref) on the host cores.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SAMPLE_RATE = 16000
DECODE_STEPS = 48
BOS, EOS = 1, 2
METRIC = "audio-sec/sec (RTFx) Conformer-L ASR, batch=32x10s@16kHz"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), d.get("bf16_tflops", 1590.0), "measured"
    return 6650.0, 1400.0, 1590.0, "fallback"


def encoder_flops_per_utt(cfg, T):
    """SURVEY.md 8(d): per frame per layer 8*d*ffn + 6d^2 + 2d^2 + 4*T*d + 4d^2 + 2*K*d + 2d^2, x T x layers,
    + CNN + input linear."""
    d, f, K = cfg["d_model"], cfg["d_ffn"], cfg["kernel_size"]
    per = 8 * d * f + 6 * d * d + 2 * d * d + 4 * T * d + 4 * d * d + 2 * K * d + 2 * d * d
    if cfg["attention_type"] == "RelPosMHAXL":
        per += 2 * (2 * T - 1) * d
    return per * T * cfg["num_encoder_layers"] + (23.1e6 + 185.0e6) * T / 251.0 + 2 * T * cfg["input_size"] * d


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed regions (started before the warm-up so that NVML
    initialisation is over when the first timed region begins)."""

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def mark(self):
        return time.perf_counter()

    def stop(self, windows):
        """Keep the samples taken inside any of the (t0, t1) host-time windows (the timed regions)."""
        if self.proc:
            self.proc.terminate()
        rows = [r for t, r in self.rows if any(a <= t <= b for a, b in windows)] or [r for _, r in self.rows]
        sm = [float(r[0]) for r in rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in rows if len(r) >= 7 for i in range(4) if r[3 + i] == "Active"})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": reasons, "samples": len(sm)}


def usable_threads(cap=None):
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return max(1, min(n, cap) if cap else n)


def synth_batch(B, seconds, seed):
    import torch
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, int(SAMPLE_RATE * seconds), generator=g), torch.ones(B)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: {name: tensor} -> out_dir/<name>.npy, floating tensors as float32 and integer ones (token ids) as
    float64, so that the outputs of two builds on the same seeded inputs can be compared array by array."""
    import numpy as np
    arrs = {k: v.detach().cpu().float().numpy() if v.is_floating_point() else v.detach().cpu().double().numpy()
            for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrs.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {DUMP_LIMIT_BYTES})")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrs.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


# =============================================================================================== reference arm
def import_reference():
    """The pip-installed, unmodified reference (baseline/_ref; `python -m pip install --no-index --no-build-isolation
    --no-deps --target baseline/_ref <copy of /root/reference>`, see DESIGN.md section 8) + the 2-function hyperpyyaml
    import shim (baseline/stubs).  Returns None when it is not there."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref, "speechbrain")):
        return None
    for p in (ref, os.path.join(ROOT, "baseline", "stubs")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import speechbrain  # noqa: F401
    return speechbrain


def build_reference_asr(cfg, sd, device="cpu", beam=None, lm_sd=None):
    """The reference's own modules with the recipe's kwargs (conformer_large.yaml / conformer_small.yaml), loaded with the
    same seeded state the product gets.  Returns a callable wav, lens -> token lists (greedy or beam)."""
    import torch
    from speechbrain.decoders.seq2seq import S2STransformerBeamSearcher, S2STransformerGreedySearcher
    from speechbrain.lobes.features import Fbank
    from speechbrain.lobes.models.convolution import ConvolutionFrontEnd
    from speechbrain.lobes.models.transformer.TransformerASR import TransformerASR
    from speechbrain.nnet.linear import Linear
    from speechbrain.processing.features import InputNormalization

    fb = Fbank(n_fft=cfg["n_fft"], n_mels=cfg["n_mels"], win_length=int(cfg["win"] * 1000 / SAMPLE_RATE))
    norm = InputNormalization(norm_type="global", update_until_epoch=4)
    cnn = ConvolutionFrontEnd(input_shape=(8, 10, 80), num_blocks=2, num_layers_per_block=1, out_channels=cfg["cnn_channels"],
                              kernel_sizes=(3, 3), strides=(2, 2), residuals=(False, False))
    tr = TransformerASR(input_size=cfg["input_size"], tgt_vocab=cfg["vocab"], d_model=cfg["d_model"], nhead=cfg["nhead"],
                        num_encoder_layers=cfg["num_encoder_layers"], num_decoder_layers=cfg["num_decoder_layers"],
                        d_ffn=cfg["d_ffn"], dropout=0.1, activation=torch.nn.GELU, encoder_module="conformer",
                        attention_type=cfg["attention_type"], normalize_before=True, causal=False)
    seq_lin = Linear(input_size=cfg["d_model"], n_neurons=cfg["vocab"])
    mods = torch.nn.ModuleDict(dict(CNN=cnn, Transformer=tr, seq_lin=seq_lin))
    own = mods.state_dict()
    mods.load_state_dict({k: sd[k] if k in sd else v for k, v in own.items()})
    norm.glob_mean, norm.glob_std, norm.count = sd["normalize.glob_mean"], sd["normalize.glob_std"], 1
    for m in (fb, norm, mods):
        m.eval()
        m.to(device)
    norm.to(device)

    def run(wav, lens, steps, encode_only=False):
        with torch.no_grad():
            wav, lens = wav.to(device), lens.to(device)
            enc = tr.encode(cnn(norm(fb(wav), lens)), lens)
            if encode_only:
                return enc
            T = enc.shape[1]
            if beam:
                s = S2STransformerBeamSearcher(modules=[tr, seq_lin], bos_index=BOS, eos_index=EOS, min_decode_ratio=0.0,
                                               max_decode_ratio=(steps + 0.5) / T, beam_size=beam, temperature=1.15,
                                               using_eos_threshold=False, length_normalization=True)
            else:
                s = S2STransformerGreedySearcher(modules=[tr, seq_lin], bos_index=BOS, eos_index=EOS, min_decode_ratio=0.0,
                                                 max_decode_ratio=(steps + 0.5) / T)
            return s(enc, lens)[0]
    return run


def best_thread_count(run, seconds, encode_only=False):
    """The reference's decode loop is thousands of small ops per step: more threads than it can use make it slower (measured
    on the 128-core GPU box in round 1: 16 threads 60x faster than 128).  Give it the count that is fastest on a quick probe
    (4 utterances, encode + 4 greedy steps) among {8, 16, 32, 64, all}."""
    import torch
    n_all = usable_threads()
    wav, lens = synth_batch(4, seconds, 99)
    best, best_t = n_all, None
    for n in sorted({min(n_all, c) for c in (8, 16, 32, 64, n_all)}):
        torch.set_num_threads(n)
        run(wav, lens, 2, encode_only)
        t0 = time.perf_counter()
        run(wav, lens, 4, encode_only)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


def time_reference(cfg, sd, B, seconds, steps, device, n_steps, warmup, budget_s, encode_only=False, beam=None, tune_threads=False):
    """`n_steps` timed passes of the reference over one B x `seconds` batch (stops early when `budget_s` is spent)."""
    import torch
    run = build_reference_asr(cfg, sd, device, beam=beam)
    if tune_threads and device == "cpu":
        best_thread_count(run, seconds, encode_only)
    wav, lens = synth_batch(B, seconds, 1234)
    times = []
    t_start = time.perf_counter()
    for i in range(warmup + n_steps):
        if device != "cpu":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        run(wav, lens, steps, encode_only)
        if device != "cpu":
            torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
        if times and time.perf_counter() - t_start > budget_s:
            break
    return times


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (its nn.Modules, fp32, no KV cache) on this
    box's host cores, the SAME config: every step is one full batch."""
    import torch

    from speechbrain_b200.utils.seeded_init import CONFORMER_LARGE, CONFORMER_SMALL, seeded_asr_state
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = workload(args)
    kind = "reference"
    if import_reference() is None:
        print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref (pip-installed reference) is missing"}))
        return
    cfg = dict(CONFORMER_SMALL if args.config == "small_enc" else CONFORMER_LARGE, attention_type=wl["attention"])
    sd = seeded_asr_state(cfg, 0)
    device = args.device
    torch.set_num_threads(usable_threads(args.ref_threads))
    if device != "cpu":
        torch.backends.cuda.matmul.allow_tf32 = True  # what speechbrain/utils/quirks.py:50-63 enables on import
        torch.backends.cudnn.allow_tf32 = True
    times = time_reference(cfg, sd, wl["B"], wl["seconds"], DECODE_STEPS, device, max(1, args.steps), 1 if args.warmup > 0 else 0,
                           args.ref_budget_s, encode_only=wl["encode_only"], beam=wl["beam"], tune_threads=args.ref_threads is None)
    audio = wl["B"] * wl["seconds"]
    value = audio * len(times) / sum(times)
    sample = (f"{len(times)} full steps of {wl['B']} x {wl['seconds']:g} s ({wl['name']}), 1 warm-up; time budget "
              f"{args.ref_budget_s:g} s" + (f"; device {device} (eager PyTorch, TF32 on)" if device != "cpu" else ""))
    line = {"metric": METRIC, "impl": "reference", "value": value, "unit": "audio-sec/sec", "n_gpus": args.gpus,
            "steps": len(times), "warmup": 1 if args.warmup > 0 else 0, "ms_per_step": 1e3 * statistics.median(times),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32" if device == "cpu" else "tf32",
            "data": "synthetic",
            "config": {"workload": wl["desc"], "global_batch": wl["B"], "timing": "host wall clock around each full step",
                       "device": device, "torch_threads": torch.get_num_threads(), "host_cpus": os.cpu_count()},
            "cpu_baseline": {"value": value, "unit": "audio-sec/sec", "cores": torch.get_num_threads(), "kind": kind,
                             "sample": sample},
            "e2e": {"value": value, "unit": "audio-sec/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# =============================================================================================== workloads
def workload(args):
    c = args.config
    if c == "greedy32":
        return dict(name=c, B=32, seconds=10.0, attention=args.attention, encode_only=False, beam=None,
                    desc=f"conformer_large.yaml ({args.attention}) random init: Fbank+CMVN+CNN+12L Conformer encode + greedy "
                         f"{DECODE_STEPS} steps (6L decoder), 32 x 10 s per GPU")
    if c == "small_enc":
        return dict(name=c, B=8, seconds=5.0, attention="RelPosMHAXL", encode_only=True, beam=None,
                    desc="conformer_small.yaml (12L/144d/4h RelPosMHAXL) random init: Fbank+CMVN+CNN+encode only, 8 x 5 s")
    if c == "beam10_lm":
        return dict(name=c, B=16, seconds=10.0, attention=args.attention, encode_only=False, beam=10, lm=True, ctc=True,
                    desc=f"conformer_large.yaml ({args.attention}) random init: encode + S2STransformerBeamSearcher beam 10, "
                         f"TransformerLM 12x768 (0.6, T 1.15) + CTC (0.4) full scorers, {DECODE_STEPS} steps, 16 x 10 s")
    if c == "beam10_shard":
        return dict(name=c, B=32, seconds=10.0, attention=args.attention, encode_only=False, beam=10, lm=False, ctc=False,
                    desc=f"conformer_large.yaml ({args.attention}) random init: encode + beam 10 (no scorer), {DECODE_STEPS} "
                         f"steps, 32 x 10 s per GPU, all-gather of the hypotheses")
    raise SystemExit(f"unknown --config {c}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=7, help="timed repetitions of the K-step region (median reported)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="greedy32", choices=["greedy32", "small_enc", "beam10_lm", "beam10_shard"])
    ap.add_argument("--attention", default="RoPEMHA", choices=["RoPEMHA", "RelPosMHAXL"])
    ap.add_argument("--device", default="cpu", help="--impl reference only: cpu (the contract's arm) or cuda (eager PyTorch leg)")
    ap.add_argument("--ref-threads", type=int, default=0, help="--impl reference: torch threads (0 = all usable cores)")
    ap.add_argument("--ref-budget-s", type=float, default=170.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-eager", action="store_true", help="skip the informational eager-PyTorch-on-GPU reference leg")
    ap.add_argument("--lanes", type=int, default=3, help="groups in flight per GPU (engine clones on their own streams)")
    ap.add_argument("--group", type=int, default=16, help="max batches whose decode is coalesced into one greedy loop")
    ap.add_argument("--decode-steps", type=int, default=48, help="diagnostic: override the pinned 48 decode steps")
    ap.add_argument("--fuse-dec-ln", type=int, default=1)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the outputs of the last timed step "
                    "as DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.ref_threads = args.ref_threads or None
    global DECODE_STEPS
    DECODE_STEPS = args.decode_steps
    if args.impl == "reference":
        return run_reference(args)
    if args.config == "greedy32":
        return run_greedy32(args)
    return run_other(args)


# =============================================================================================== the headline workload
def run_greedy32(args):
    import torch
    import torch.distributed as dist

    from speechbrain_b200 import _lib
    from speechbrain_b200.parallel import gather_hypotheses
    from speechbrain_b200.utils.seeded_init import CONFORMER_LARGE, seeded_asr_state

    wl = workload(args)
    BATCH, UTT_SECONDS = wl["B"], wl["seconds"]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # before anything else: NVML start-up must not fall into a timed region
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W = max(args.warmup, 3)
    K = args.steps
    R = max(1, args.repeats)

    cfg = dict(CONFORMER_LARGE, attention_type=args.attention)
    sd = seeded_asr_state(cfg, 0)
    asr = build_product_asr(cfg, sd, dev)       # the module mirrors + EncoderDecoderASR: the public API the e2e leg calls
    eng = asr.engine()                          # ... and the C-ABI engine they share (device-resident leg)
    wav_host, lens_host = synth_batch(BATCH, UTT_SECONDS, 1234 + rank)
    wav_host, lens_host = wav_host.pin_memory(), lens_host.pin_memory()
    wav_dev, lens_dev = wav_host.to(dev), lens_host.to(dev)
    L = wav_host.shape[1]
    T_f, T = eng.num_frames(L)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    lib = _lib.lib()

    # ---- schedule: K steps = n_calls group calls (G <= --group batches each, balanced), NL groups in flight on NL streams.
    # A group = G batches of 32 x 10 s: each batch is encoded on its own, the G*32 hypotheses are decoded together.
    NLmax = max(1, args.lanes)
    n_calls = max(-(-K // args.group), min(NLmax, K))
    sizes = [K // n_calls + (1 if i < K % n_calls else 0) for i in range(n_calls)]  # exactly K batches
    G = max(sizes)
    NL = min(NLmax, n_calls)
    lanes = [eng] + [eng.clone() for _ in range(NL - 1)]
    for e in lanes:
        e.set_decoder_ln_fusion(args.fuse_dec_ln)
        e.set_poll_interval(0)  # exactly DECODE_STEPS steps, never block the host (random weights never emit EOS)
    streams = [torch.cuda.Stream(device=dev) for _ in range(NL)]
    wavs = [[wav_dev.clone() for _ in range(G)] for _ in range(NL)]
    lens = [[lens_dev.clone() for _ in range(G)] for _ in range(NL)]
    # token ids of one group: ONE [G*32, steps] tensor per lane (views per batch) so the final gather is one collective
    pred_all = [torch.full((G * BATCH, DECODE_STEPS), -1, dtype=torch.int32, device=dev) for _ in range(NL)]
    preds = [[pred_all[ln][g * BATCH:(g + 1) * BATCH] for g in range(G)] for ln in range(NL)]
    wavs_host = [[wav_host.clone().pin_memory() for _ in range(G)] for _ in range(NL)]
    lens_host_l = [[lens_host.clone().pin_memory() for _ in range(G)] for _ in range(NL)]
    preds_host = [[torch.empty(BATCH, DECODE_STEPS, dtype=torch.int32).pin_memory() for _ in range(G)] for _ in range(NL)]
    gathered = {}

    def gather(ln, g):
        if world > 1:  # the path's only collective: every rank ends up with all ranks' hypotheses of this group
            key = (ln, g)
            if key not in gathered:
                gathered[key] = torch.empty(world * g * BATCH, DECODE_STEPS, dtype=torch.int32, device=dev)
            # max_len = the decode limit: a static width, so the helper needs no width-agreeing all-reduce (whose .item() would
            # block the host until this lane's group has finished and serialise the lanes)
            gather_hypotheses(pred_all[ln][: g * BATCH], world * g * BATCH, world, max_len=DECODE_STEPS, out=gathered[key])

    def step_dev(i):
        ln, g = i % NL, sizes[i]
        with torch.cuda.stream(streams[ln]):
            lanes[ln].transcribe_greedy_group_dev(wavs[ln][:g], lens[ln][:g], DECODE_STEPS, BOS, EOS, preds[ln][:g])
            gather(ln, g)

    def step_host(i):
        ln, g = i % NL, sizes[i]
        with torch.cuda.stream(streams[ln]):
            # public API: pinned host wav in, pinned host token ids out; H2D + pipeline + D2H are enqueued by the C ABI
            asr_lanes[ln].transcribe_batches_async(wavs_host[ln][:g], lens_host_l[ln][:g], preds_host[ln][:g],
                                                   preds[ln][:g] if world > 1 else None)
            gather(ln, g)

    class _Lane:  # EncoderDecoderASR front of a lane: same modules, the lane's engine clone
        def __init__(self, e):
            self.e = e

        def transcribe_batches_async(self, w, l_, p, pd):
            return self.e.transcribe_greedy_group_host_async(w, l_, DECODE_STEPS, BOS, EOS, p, pd)
    asr_lanes = [asr] + [_Lane(e) for e in lanes[1:]]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    windows = []

    def timed(fn):
        """One repetition: K steps between ONE pair of CUDA events; every lane stream starts after the start event and the
        stop event is recorded after all lane streams have drained."""
        barrier()
        cur = torch.cuda.current_stream(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_a = time.perf_counter()
        e0.record(cur)
        for s_ in streams:
            s_.wait_event(e0)
        t_host = time.perf_counter()
        for i in range(n_calls):
            fn(i)
        host_ms = (time.perf_counter() - t_host) * 1e3 / K
        for s_ in streams:
            cur.wait_stream(s_)
        e1.record(cur)
        e1.synchronize()
        windows.append((t_a, time.perf_counter()))
        return e0.elapsed_time(e1), host_ms

    def repeat(fn):
        """R repetitions -> per-repeat ms (max over ranks), so the median is a median of whole-job times."""
        ms, host = [], []
        for _ in range(R):
            m, h = timed(fn)
            ms.append(m)
            host.append(h)
        t = torch.tensor(ms, device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t], statistics.median(host)

    for rep in range(max(1, -(-W // K))):  # warm-up = the timed schedule itself (captures every (lane, group size) graph)
        for i in range(n_calls):
            step_dev(i)
        for i in range(n_calls):
            step_host(i)
    barrier()
    launches0 = lib.sbk_launch_count()
    ms_dev_all, host_enqueue_ms = repeat(step_dev)
    launches = (lib.sbk_launch_count() - launches0) // R  # libsbk kernels inside one K-step region (graph nodes included)
    ms_host_all, _ = repeat(step_host)
    barrier()
    # parity of the two legs: same inputs -> same token ids
    e2e_matches_dev = all(bool(torch.equal(preds_host[0][g], preds[0][g].cpu())) for g in range(sizes[0])) if world == 1 else None

    # single batch in flight (latency view) through EncoderDecoderASR.transcribe_batch on HOST tensors, L2 flushed per step
    lat = []
    eng.set_poll_interval(0)
    for i in range(5):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        words, toks = asr.transcribe_batch(wav_host, lens_host)
        lat.append((time.perf_counter() - t0) * 1e3)
    ms_single = statistics.median(lat)
    clocks = sampler.stop(windows) if rank == 0 else None

    ms_dev, ms_host = statistics.median(ms_dev_all), statistics.median(ms_host_all)
    audio = world * BATCH * UTT_SECONDS * K
    value = audio / (ms_dev / 1e3)
    e2e = audio / (ms_host / 1e3)

    # ---- roofline leg: dominant kernel = the 2-CTA tcgen05 GEMM, timed live per launch with CUDA events (rank 0)
    roof = None
    if rank == 0:
        import ctypes
        hbm, tf_sus, tf_burst, src = peaks()
        pred1 = torch.empty(BATCH, DECODE_STEPS, dtype=torch.int32, device=dev)
        eng.set_poll_interval(8)  # per-kernel launches (no whole-pipeline graph) so the GEMM launches can be event-timed
        eng.transcribe_greedy_dev(wav_dev, lens_dev, DECODE_STEPS, BOS, EOS, pred=pred1)
        torch.cuda.synchronize()
        lib.sbk_gemm_profile_enable(1)
        eng.transcribe_greedy_dev(wav_dev, lens_dev, DECODE_STEPS, BOS, EOS, pred=pred1)
        torch.cuda.synchronize()
        n, ms, fl = ctypes.c_int(), ctypes.c_double(), ctypes.c_double()
        _lib.check(lib.sbk_gemm_profile_read(ctypes.byref(n), ctypes.byref(ms), ctypes.byref(fl)), "gemm_profile_read")
        lib.sbk_gemm_profile_enable(0)
        eng.set_poll_interval(0)
        ach = fl.value / (ms.value * 1e-3) / 1e12 if ms.value > 0 else 0.0
        enc_fl = BATCH * encoder_flops_per_utt(cfg, T)
        roof = {"bound": "tensor",
                "kernel": "gemm_tc2_kernel (2-CTA tcgen05.mma cta_group::2 kind::f16, 256x256x64 tiles, fp16 in / fp32 acc in "
                          "TMEM) -- all encoder / cross-K,V GEMM launches of one 32 x 10 s batch",
                "achieved": ach, "peak": tf_sus, "unit": "TFLOP/s", "frac": ach / tf_sus,
                "traffic": None,  # dram__bytes per launch is only available under ncu: see profiles/ (not hard-coded here)
                "peak_source": f"{src} bf16_tflops_sustained (kernel timed inside a long step)",
                "launches_per_step": n.value, "gemm_ms_per_step": ms.value, "gemm_flops_per_step": fl.value,
                "gemm_share_of_gpu_time_per_step": ms.value / (ms_dev / K),
                "encoder_flops_per_step": enc_fl,
                "encoder_roofline_rtfx": BATCH * UTT_SECONDS / (enc_fl / (tf_sus * 1e12)),
                "frac_of_encoder_roofline": (value / world) / (BATCH * UTT_SECONDS / (enc_fl / (tf_sus * 1e12)))}
    # ---- the reference beside it (rank 0): its CPU path on the host cores, and eager PyTorch on this GPU (informational)
    cpu_base = gpu_eager = None
    if rank == 0 and import_reference() is not None:
        if not args.no_cpu_baseline:
            torch.set_num_threads(usable_threads())
            times = time_reference(cfg, sd, BATCH, UTT_SECONDS, DECODE_STEPS, "cpu", 2, 0, 45.0, tune_threads=True)
            v = BATCH * UTT_SECONDS * len(times) / sum(times)
            cpu_base = {"value": v, "unit": "audio-sec/sec", "cores": torch.get_num_threads(), "kind": "reference",
                        "sample": f"{len(times)} full step(s) of 32 x 10 s (encode + {DECODE_STEPS} greedy steps) with the "
                                  f"reference's own modules from baseline/_ref, fp32, {sum(times):.1f} s wall"}
        if not args.no_gpu_eager:
            torch.backends.cuda.matmul.allow_tf32 = True
            torch.backends.cudnn.allow_tf32 = True
            times = time_reference(cfg, sd, BATCH, UTT_SECONDS, DECODE_STEPS, str(dev), 3, 1, 60.0)
            gpu_eager = {"value": BATCH * UTT_SECONDS / statistics.median(times), "unit": "audio-sec/sec",
                         "ms_per_step": 1e3 * statistics.median(times),
                         "what": "the reference's own nn.Modules in eager PyTorch on this same B200 (TF32 on, as "
                                 "speechbrain/utils/quirks.py enables), wav on the device; informational competitor (SURVEY 2.3)"}
    if rank == 0:
        def spread(xs):
            return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "n": len(xs)}
        line = {"metric": METRIC, "value": value, "unit": "audio-sec/sec", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "fp16 operands, fp32 accumulate/residual/softmax", "data": "synthetic",
                "config": {"workload": wl["desc"], "global_batch": world * BATCH, "utt_seconds": UTT_SECONDS, "enc_frames": T,
                           "parallelism": f"dp{world} (utterance shards, one all-gather of token ids per group call)",
                           "lanes": NL, "decode_group": G, "group_sizes": sizes, "decoder_ln_fused": bool(args.fuse_dec_ln),
                           "repeats": R, "ms_per_region": spread(ms_dev_all), "host_enqueue_ms_per_step": host_enqueue_ms,
                           "l2": "no flush inside the K-step bracket: per-step working set (0.25 GB weights + 0.3 GB "
                                 "activations/KV per lane) exceeds the 126 MB L2; single_batch is flushed (256 MiB) per step",
                           "timing": f"median of {R} repetitions; each = one CUDA-event pair around K steps (= {n_calls} group "
                                     f"calls, sizes {sizes}), {NL} groups in flight on {NL} streams; max over ranks per repetition"},
                "e2e": {"value": e2e, "unit": "audio-sec/sec", "ms_per_step": ms_host / K, "ms_per_region": spread(ms_host_all),
                        "h2d_bytes_per_step": BATCH * L * 4 + BATCH * 4, "d2h_bytes_per_step": BATCH * DECODE_STEPS * 4,
                        "api": "EncoderDecoderASR.transcribe_batches_async -> sbk_asr_transcribe_greedy_group_host_async "
                               "(pinned host buffers; H2D, pipeline and D2H enqueued by the C ABI)",
                        "ids_equal_device_leg": e2e_matches_dev},
                "single_batch": {"value": BATCH * UTT_SECONDS / (ms_single / 1e3), "unit": "audio-sec/sec", "ms_per_step": ms_single,
                                 "note": "EncoderDecoderASR.transcribe_batch(host wav, lens) -> words: one batch in flight, no "
                                         "decode coalescing, L2 flushed before every call, host wall clock (latency view)"},
                "gpu_launches": int(launches), "gpu_launches_per_step": int(launches) // max(K, 1), "clocks": clocks,
                "roofline": roof, "cpu_baseline": cpu_base, "gpu_eager_reference": gpu_eager}
        print(json.dumps(line))
        if args.dump_outputs:  # the token ids of the last batch of the device-resident leg's last group call
            dump_outputs(args.dump_outputs, {"token_ids": preds[(n_calls - 1) % NL][sizes[-1] - 1]})
    if world > 1:
        dist.destroy_process_group()


def build_product_asr(cfg, sd, dev, decoder="greedy", beam=10, lm=False, ctc=False, coverage=None):
    """speechbrain_b200 module mirrors wired like the recipe, loaded with the seeded state through load_state_dict."""
    import torch

    from speechbrain_b200.decoders.scorer import CoverageScorer, CTCScorer, ScorerBuilder, TransformerLMScorer
    from speechbrain_b200.decoders.seq2seq import S2STransformerBeamSearcher, S2STransformerGreedySearcher
    from speechbrain_b200.inference.ASR import EncoderDecoderASR
    from speechbrain_b200.lobes.features import Fbank
    from speechbrain_b200.lobes.models.convolution import ConvolutionFrontEnd
    from speechbrain_b200.lobes.models.transformer.TransformerASR import TransformerASR
    from speechbrain_b200.lobes.models.transformer.TransformerLM import TransformerLM
    from speechbrain_b200.nnet.containers import LengthsCapableSequential
    from speechbrain_b200.nnet.linear import Linear
    from speechbrain_b200.processing.features import InputNormalization
    from speechbrain_b200.utils.seeded_init import seeded_state_dict

    fb = Fbank(n_fft=cfg["n_fft"], n_mels=cfg["n_mels"], win_length=int(cfg["win"] * 1000 / SAMPLE_RATE))
    norm = InputNormalization(norm_type="global", update_until_epoch=4)
    norm.glob_mean, norm.glob_std, norm.count = sd["normalize.glob_mean"], sd["normalize.glob_std"], 1
    norm.eval()
    cnn = ConvolutionFrontEnd(input_shape=(8, 10, 80), num_blocks=2, num_layers_per_block=1, out_channels=cfg["cnn_channels"],
                              kernel_sizes=(3, 3), strides=(2, 2), residuals=(False, False))
    cnn.load_state_dict({k[4:]: v for k, v in sd.items() if k.startswith("CNN.")})
    tr = TransformerASR(input_size=cfg["input_size"], tgt_vocab=cfg["vocab"], d_model=cfg["d_model"], nhead=cfg["nhead"],
                        num_encoder_layers=cfg["num_encoder_layers"], num_decoder_layers=cfg["num_decoder_layers"],
                        d_ffn=cfg["d_ffn"], activation=torch.nn.GELU, encoder_module="conformer",
                        attention_type=cfg["attention_type"], normalize_before=True, causal=False)
    tr.load_state_dict({k[len("Transformer."):]: v for k, v in sd.items() if k.startswith("Transformer.")}, strict=False)
    lin = Linear(input_size=cfg["d_model"], n_neurons=cfg["vocab"])
    lin.load_state_dict({"w.weight": sd["seq_lin.w.weight"], "w.bias": sd["seq_lin.w.bias"]})
    if decoder == "greedy":
        dec = S2STransformerGreedySearcher(modules=[tr, lin], bos_index=BOS, eos_index=EOS, min_decode_ratio=0.0,
                                           max_decode_ratio=(DECODE_STEPS + 0.5) / 251.0, return_log_probs=False)
    else:
        full, weights = [], {}
        if lm:
            lm_m = TransformerLM(vocab=cfg["vocab"], d_model=768, nhead=12, num_encoder_layers=12, num_decoder_layers=0,
                                 d_ffn=3072, dropout=0.0, activation=torch.nn.GELU, normalize_before=False)
            lm_m.load_state_dict(seeded_state_dict(lm_m, seed=1))
            full.append(TransformerLMScorer(language_model=lm_m, temperature=1.15))
            weights["transformerlm"] = 0.6
        if ctc:
            ctc_lin = Linear(input_size=cfg["d_model"], n_neurons=cfg["vocab"])
            ctc_lin.load_state_dict({"w.weight": sd["ctc_lin.w.weight"], "w.bias": sd["ctc_lin.w.bias"]})
            full.append(CTCScorer(eos_index=EOS, blank_index=0, ctc_fc=ctc_lin))
            weights["ctc"] = 0.4
        if coverage is not None:  # (weight, threshold)
            full.append(CoverageScorer(cfg["vocab"], threshold=coverage[1]))
            weights["coverage"] = coverage[0]
        scorer = ScorerBuilder(full_scorers=full, weights=weights) if full else None
        dec = S2STransformerBeamSearcher(modules=[tr, lin], bos_index=BOS, eos_index=EOS, min_decode_ratio=0.0,
                                         max_decode_ratio=(DECODE_STEPS + 0.5) / 251.0, beam_size=beam, temperature=1.15,
                                         using_eos_threshold=False, length_normalization=True, scorer=scorer)
    enc = LengthsCapableSequential(compute_features=fb, normalize=norm, cnn=cnn)
    return EncoderDecoderASR(modules=dict(encoder=enc, transformer=tr, decoder=dec),
                             hparams=dict(tokenizer=None, transformer_beam_search=True), run_opts={"device": str(dev)})


# =============================================================================================== the other BASELINE configs
def run_other(args):
    import torch
    import torch.distributed as dist

    from speechbrain_b200 import _lib
    from speechbrain_b200.engine import AsrEngine
    from speechbrain_b200.parallel import gather_hypotheses
    from speechbrain_b200.utils.seeded_init import CONFORMER_LARGE, CONFORMER_SMALL, seeded_asr_state

    wl = workload(args)
    B, seconds = wl["B"], wl["seconds"]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    K, R, W = args.steps, max(1, args.repeats), max(args.warmup, 3)
    small = args.config == "small_enc"
    cfg = dict(CONFORMER_SMALL if small else CONFORMER_LARGE, attention_type=wl["attention"])
    sd = seeded_asr_state(cfg, 0)
    wav_host, lens_host = synth_batch(B, seconds, 1234 + rank)
    wav_host, lens_host = wav_host.pin_memory(), lens_host.pin_memory()
    wav_dev, lens_dev = wav_host.to(dev), lens_host.to(dev)
    L = wav_host.shape[1]
    lib = _lib.lib()
    windows = []
    if small:
        eng = AsrEngine(cfg, sd, device=dev, parts=("fbank", "cnn", "encoder"))
        eng.set_poll_interval(0)
        T = eng.num_frames(L)[1]
        enc_out = torch.empty(B, T, cfg["d_model"], device=dev)
        enc_host = torch.empty(B, T, cfg["d_model"]).pin_memory()

        def step(host):
            if host:
                wav_dev.copy_(wav_host, non_blocking=True)
                lens_dev.copy_(lens_host, non_blocking=True)
            eng.encode_wav(wav_dev, lens_dev, out=enc_out)
            if host:
                enc_host.copy_(enc_out, non_blocking=True)
        d2h = B * T * cfg["d_model"] * 4
    else:
        asr = build_product_asr(cfg, sd, dev, decoder="beam", beam=wl["beam"], lm=wl.get("lm", False), ctc=wl.get("ctc", False))
        dec = asr.mods["decoder"]
        T = asr.engine().num_frames(L)[1]
        hyp_buf = torch.full((B, DECODE_STEPS), -1, dtype=torch.int32, device=dev)
        last_hyps = []

        def step(host):
            w, l_ = (wav_host, lens_host) if host else (wav_dev, lens_dev)
            words, hyps = asr.transcribe_batch(w, l_)  # public API: encode (fused pipeline) + beam search + host replay
            last_hyps[:] = hyps
            if world > 1:
                hyp_buf.fill_(-1)
                for b, h in enumerate(hyps):
                    hyp_buf[b, : len(h)] = torch.tensor(h, dtype=torch.int32)
                gather_hypotheses(hyp_buf, world * B, world, max_len=DECODE_STEPS)
        d2h = B * wl["beam"] * DECODE_STEPS * 16

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def region(host):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_a = time.perf_counter()
        e0.record()
        for _ in range(K):
            step(host)
        e1.record()
        e1.synchronize()
        windows.append((t_a, time.perf_counter()))
        return e0.elapsed_time(e1)

    for _ in range(W):
        step(False)
        step(True)
    barrier()
    l0 = lib.sbk_launch_count()
    dev_ms = [region(False) for _ in range(R)]
    launches = (lib.sbk_launch_count() - l0) // R
    host_ms = [region(True) for _ in range(R)]
    t = torch.tensor([dev_ms, host_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, host_ms = [float(x) for x in t[0]], [float(x) for x in t[1]]
    clocks = sampler.stop(windows) if rank == 0 else None
    if rank == 0:
        hbm, tf_sus, tf_burst, src = peaks()
        audio = world * B * seconds * K
        md, mh = statistics.median(dev_ms), statistics.median(host_ms)
        enc_fl = B * encoder_flops_per_utt(cfg, T)
        line = {"metric": METRIC + f" [{args.config}]", "value": audio / (md / 1e3), "unit": "audio-sec/sec", "n_gpus": world,
                "steps": K, "warmup": W, "ms_per_step": md / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "fp16 operands, fp32 accumulate/residual/softmax", "data": "synthetic",
                "config": {"workload": wl["desc"], "global_batch": world * B, "utt_seconds": seconds, "enc_frames": T,
                           "repeats": R, "ms_per_region": {"median": md, "min": min(dev_ms), "max": max(dev_ms)},
                           "timing": f"median of {R} repetitions of one CUDA-event pair around K sequential steps; max over ranks"},
                "e2e": {"value": audio / (mh / 1e3), "unit": "audio-sec/sec", "ms_per_step": mh / K,
                        "h2d_bytes_per_step": B * L * 4 + B * 4, "d2h_bytes_per_step": d2h},
                "gpu_launches": int(launches), "clocks": clocks,
                "roofline": {"bound": "tensor", "unit": "TFLOP/s", "peak": tf_sus, "achieved": enc_fl / (md / K * 1e-3) / 1e12,
                             "frac": enc_fl / (md / K * 1e-3) / 1e12 / tf_sus, "traffic": None,
                             "note": "whole step vs the encoder FLOP roofline (SURVEY 8d); the decode loop of the beam configs "
                                     "is weight-bandwidth / latency bound, see DESIGN.md"}}
        print(json.dumps(line))
        if args.dump_outputs:  # the last timed step: encoder states, or the best hypotheses padded with -1
            if small:
                out = {"encoder_out": enc_out}
            else:
                ids = torch.full((B, max(map(len, last_hyps), default=0)), -1, dtype=torch.int32)
                for b, h in enumerate(last_hyps):
                    ids[b, : len(h)] = torch.tensor(h, dtype=torch.int32)
                out = {"token_ids": ids}
            dump_outputs(args.dump_outputs, out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
