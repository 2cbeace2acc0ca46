#!/usr/bin/env python
"""bench.py -- mel-frames/s and RTF of JETSGenerator.forward (PromptTTS AM + HiFi-GAN) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--precision fp32|tf32|bf16|fp32_ffma] [--lean]
                    [--dump-outputs DIR]
    torchrun --nproc-per-node N ... bench.py --gpus N ...        (one rank per GPU, NCCL)

Headline workload (BASELINE.json configs[1], the configuration `metric` is quoted on): batch = 1, one 100-phoneme utterance
per step, fp32, full acoustic model + vocoder, seeded synthetic weights of the released architecture.  The steps walk a
seeded corpus of DISTINCT utterances (synth.corpus_utterance: utterance i is the same whatever the corpus size or world
size) that runner.plan_shards deals over the ranks, so every rank synthesises different audio; there is no data-path
collective, only the one-time NCCL weight broadcast (raw parameters + the packed blob rank 0 built).  Weak scaling: K steps
per rank.

* `value`: mel-frames/s with each step's inputs already resident in HBM; per-step CUDA-event pairs on the launching stream,
  L2 flushed (256 MiB write) between steps outside the pairs; whole job = sum of frames over ranks / max over ranks of time.
* `e2e`: the same steps through the public API from HOST data: collate -> pinned host tensors -> H2D -> forward ->
  fp32 waveform D2H into pinned memory, all inside the timed region (host preparation included: the start event is
  recorded before it).
* `b1`, `b32`, `voc`, `cfg5`: compact secondary measurements of the other BASELINE.json configurations, taken after the
  headline numbers are final (each guarded: a failure there costs a sub-object, never the line):
    b1   = configs[1] on the committed fixture utterance (latency, parity against the UNMODIFIED reference's output)
    b32  = configs[2]: one batch of 32 mixed EN/ZH utterances, 20-200 phonemes, bf16 (and the headline precision)
    voc  = configs[3]: vocoder-only points, layer-granular HBM fraction (SURVEY.md s8d accounting)
    cfg5 = configs[4]: a fixed 256-utterance-per-GPU... see `cfg5_block` -- corpus sharded over the ranks in B=32
           buckets, wall-clock end to end (pinned int16 D2H), with a digest that is identical for every world size iff
           every utterance's PCM is bit-identical.
    cfg5_strong = the same pipeline on a FIXED 2048-utterance corpus (strong scaling 1 -> N; digest over all of it).
* --impl reference: the reference's algorithm on the host CPU (oracle/jets_oracle.py, the torch-CPU restatement pinned
  bit-exactly to the unmodified reference, which is Python and cannot travel to the GPU box), all usable host threads,
  same corpus, same unit (B=1 per step as every reference caller runs), rank 0 only.

The LAST stdout line is ONE compact JSON object (< 4 KB, checked by tests/test_bench_contract.py); everything longer goes
to stderr.

--dump-outputs DIR: after the timed steps, rank 0 writes every array its last `value` step returned (the forward's output dict;
with --impl reference, the last timed oracle forward's) as DIR/<key>.npy, float32 or float64.  The steps' inputs depend only on
the arguments (seeded corpus), so two builds of the project can be compared output for output.

bench.py writes nothing into the tree, which may be read-only: it needs the library build() left there and compiles nothing.
"""
import argparse
import atexit
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True         # no __pycache__ in the tree either

import torch  # noqa: E402

N_PHONEMES = 100
SR, HOP = 16000, 256
WORKLOAD = ("cfg2: batch=1, one 100-phoneme utterance per step (distinct seeded utterances, LPT-sharded over ranks), fp32, "
            "PromptTTS AM + HiFi-GAN")
# identical on both arms (the driver compares it): everything arm-specific lives in `detail`
CONFIG = {"workload": WORKLOAD, "batch": 1, "phonemes_per_utterance": N_PHONEMES, "corpus_seed": 1234,
          "l2": "flushed between timed steps", "timing": "per-step CUDA events, max over ranks",
          "workspace": "arena reserved at start-up for 1 x 1024 frames (JETSGenerator.reserve), grow-only afterwards"}
VOC_FLOP_PER_FRAME = 614105088.0       # SURVEY.md s8d
VOC_BYTES_PER_FRAME = 5010752.0        # layer-granular fp32 activation traffic per mel frame
MAX_LINE = 4096
MAX_DUMP_BYTES = 64 << 20


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=float(d["hbm_gbs"]), bf16_tflops=float(d["bf16_tflops"]),
                    bf16_tflops_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


def _r(x, n=4):
    """round to n significant digits (keeps the JSON line short)"""
    if x is None or isinstance(x, (bool, int, str)):
        return x
    if x == 0 or not math.isfinite(x):
        return x
    return float("%.*g" % (n, x))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
            atexit.register(self.proc.kill)         # also when bench.py fails before stop(); a no-op once stop() has reaped it
        except Exception:
            self.proc = None
        # nvidia-smi's own start-up (driver handshake, ~100 ms) should not overlap the timed region: wait for the first sample line
        # (at most 3 s); the samples that follow come at the recipe's 200 ms interval
        t0 = time.perf_counter()
        while self.proc is not None and time.perf_counter() - t0 < 3.0:
            try:
                if os.path.getsize(self.path) > 0:
                    break
            except OSError:
                break
            time.sleep(0.02)

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        try:
            sm, smax, reasons = [], [], set()
            with open(self.path) as f:
                for line in f:
                    p = [x.strip() for x in line.split(",")]
                    if len(p) < 9:
                        continue
                    try:
                        sm.append(float(p[1]))
                        smax.append(float(p[2]))
                    except ValueError:
                        continue
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                        if v.lower().startswith("active"):
                            reasons.add(name)
            if sm:
                load = [x for x in sm if x > 0.5 * max(sm)] or sm
                out = dict(sm_mhz=statistics.median(load), sm_max_mhz=max(smax), reasons=sorted(reasons), samples=len(sm))
            os.unlink(self.path)
        except Exception:
            pass
        return out


def usable_cpus():
    """CPUs this process may actually run on: affinity mask capped by the cgroup CPU quota
    (os.cpu_count() reports the whole host and oversubscribes a quota-limited container)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, per = f.read().split()
        if q != "max":
            n = min(n, max(1, int(math.ceil(float(q) / float(per)))))
    except Exception:
        pass
    return max(1, n)


def pick_cpu_threads(sd, conf):
    """The reference's own hint is `torch.set_num_threads(4)  # faster` (inference_tts.py:186): more threads is not
    monotonically better for these small convolutions.  Calibrate on a short vocoder-only sample and keep the fastest
    thread count <= the usable CPUs, so the CPU baseline is the best the host can do, not an oversubscribed one."""
    from emotivoice_b200 import synth
    from oracle import jets_oracle as O
    n = usable_cpus()
    cands = sorted({c for c in (4, 8, 16, 32, 64, n) if c <= n} or {n})
    mel = synth.make_mel(1, 48, seed=3)
    best, best_t, log = cands[0], float("inf"), {}
    for c in cands:
        torch.set_num_threads(c)
        O.vocoder(sd, conf.model, mel)
        t0 = time.perf_counter()
        O.vocoder(sd, conf.model, mel)
        dt = time.perf_counter() - t0
        log[c] = round(dt * 1e3, 1)
        if dt < best_t:
            best, best_t = c, dt
        if dt > 3 * best_t:
            break
    torch.set_num_threads(best)
    return best, n, log


def cpu_reference_run(steps, warmup, first_index=0):
    """The reference's algorithm on the host CPU (oracle port): `steps` utterances of the bench corpus, B=1 each (how every
    reference caller runs), best thread count <= usable CPUs.  Returns (stats, output dict of the last timed forward)."""
    from emotivoice_b200.config import default_config
    from emotivoice_b200 import synth
    from oracle import jets_oracle as O
    conf = default_config()
    sd = synth.make_state_dict(conf)
    cores, usable, calib = pick_cpu_threads(sd, conf)
    utt = lambda i: synth.collate_utterances([synth.corpus_utterance(i, n_phonemes=N_PHONEMES)])
    for w in range(max(1, warmup)):
        O.jets_forward(sd, conf, **utt(first_index + w))
    frames, t = 0, 0.0
    for s in range(steps):
        batch = utt(first_index + warmup + s)
        t0 = time.perf_counter()
        out = O.jets_forward(sd, conf, **batch)
        t += time.perf_counter() - t0
        frames += int(out["dec_outputs"].shape[1])
    return dict(frames=frames, seconds=t, fps=frames / t, cores=cores, usable=usable, calib=calib, steps=steps), out


def emit(line, detail=None):
    """ONE compact JSON line on stdout (readers parse the last line); the long form to stderr."""
    s = json.dumps(line, separators=(",", ":"))
    if len(s) >= MAX_LINE:       # never let a secondary block cost the headline: drop the optional sub-objects, largest first
        for k in sorted(("cfg5_strong", "cfg5", "voc", "b32", "b1", "parity"), key=lambda k: -len(json.dumps(line.get(k, None)))):
            if k in line:
                line[k] = {"dropped": "line too long; see bench_detail"}
                s = json.dumps(line, separators=(",", ":"))
                if len(s) < MAX_LINE:
                    break
    if detail is not None:
        sys.stderr.write("[bench detail] " + json.dumps(detail) + "\n")
        sys.stderr.flush()
    sys.stdout.write(s + "\n")
    sys.stdout.flush()


def reference_arm(args, rank):
    if rank != 0:
        return
    steps, warm = max(1, args.steps), max(1, args.warmup)   # ~0.3 s of host CPU work per step
    r, last = cpu_reference_run(steps, warm)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    audio_s = r["frames"] * HOP / SR
    line = {
        "impl": "reference", "metric": "mel_frames_per_sec", "value": r["fps"], "unit": "mel-frames/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": r["seconds"] / steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": CONFIG,
        "rtf": _r(r["seconds"] / audio_s), "x_realtime": _r(audio_s / r["seconds"]),
        "cpu_baseline": {"value": r["fps"], "unit": "mel-frames/s", "cores": r["cores"], "kind": "port",
                         "sample": "%d B=1 forwards over corpus utterances %d.. (oracle/jets_oracle.py, torch %s CPU, %d threads of %d usable)"
                                   % (steps, warm, torch.__version__, r["cores"], r["usable"])},
        "e2e": {"value": r["fps"], "unit": "mel-frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "detail": {"device": "host CPU", "frames": r["frames"], "thread_calibration_ms": r["calib"]},
    }
    emit(line)


def dump_outputs(out_dir, outputs):
    """Every tensor of one forward's output dict -> out_dir/<key>.npy: floating point as float32 (float64 stays float64),
    integers as float64 (exact)."""
    import numpy as np
    arrays = {}
    for k, v in outputs.items():
        if torch.is_tensor(v):
            v = v.detach().cpu()
            arrays[k] = (v.float() if v.is_floating_point() and v.dtype != torch.float64 else v.double()).numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > MAX_DUMP_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes of outputs, more than the %d allowed" % (total, MAX_DUMP_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def parity_vs_fixture(model, dev):
    """tests/golden/b1_t100.npz holds inputs + outputs of the UNMODIFIED reference (oracle/make_golden.py) for the cfg2
    utterance: the engine's distance from it, with the tolerance this precision is held to."""
    import numpy as np
    path = os.path.join(ROOT, "tests", "golden", "b1_t100.npz")
    if not os.path.exists(path):
        return None
    z = np.load(path)
    keys = ("inputs_ling", "input_lengths", "inputs_speaker", "inputs_style_embedding", "inputs_content_embedding")
    out = model(**{k: torch.from_numpy(z[k]).to(dev) for k in keys})
    mel, wav, dur = torch.from_numpy(z["mel"]), torch.from_numpy(z["wav"]), torch.from_numpy(z["durations"])
    m, w = out["dec_outputs"].cpu(), out["wav_predictions"].cpu()
    ok = bool(torch.equal(out["log_duration_predictions"].cpu(), dur))
    res = {"vs": "reference fixture b1_t100", "dur_equal": ok}
    if ok and m.shape == mel.shape:
        res["mel_relmax"] = _r(float((m - mel).abs().max() / mel.abs().max()), 3)
        res["wav_relrms"] = _r(float((w - wav).double().pow(2).mean().sqrt() / wav.double().pow(2).mean().sqrt()), 3)
    return res


def timed_forwards(fn, n, flush, keep_last=False):
    """n x (flush; event; fn(i); event) -> list of seconds; synchronises once at the end.  keep_last: only the last result is kept
    (results that hold device tensors would otherwise pile up and force fresh cudaMallocs inside the timed steps)."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    outs = []
    for i, (a, b) in enumerate(ev):
        flush()
        a.record()
        r = fn(i)
        b.record()
        if keep_last:
            outs = [r]
        else:
            outs.append(r)
    torch.cuda.synchronize()
    return [a.elapsed_time(b) * 1e-3 for a, b in ev], outs


def dominant_launch(lib, dev, frames, precision="fp32"):
    """The most expensive launch of the batch-1 step, as the engine issues it: the k = 3 / 7 / 11 convolutions of the three parallel
    ResBlocks of HiFi-GAN stage 2 (C = 128, L = 64 F; about 42 % of the step's FLOPs sit in this stage) as ONE grouped launch (conv1d_gp: bf16x3
    in the "fp32" precision, tf32, or bf16 with bf16 activations), here the c2 step with its residual.  Returns the launch closure
    and its algorithmic work; tools/profile_dominant.py runs the same closure under ncu."""
    import ctypes
    from emotivoice_b200 import _abi, layout, packing
    C, Ks, L = 128, (11, 7, 3), 64 * frames
    g = torch.Generator().manual_seed(0)
    xs = [torch.randn(1, L, C, generator=g) for _ in Ks]
    ws = [torch.randn(K, C, C, generator=g) / math.sqrt(C * K) for K in Ks]
    bs = [torch.randn(C, generator=g).to(dev) for _ in Ks]
    res = [torch.randn(1, L, C, generator=g) for _ in Ks]
    st = torch.cuda.current_stream().cuda_stream
    keep = []
    if precision == "fp32_ffma":
        K = 11
        xd, wd, rd, out = xs[0].to(dev), ws[0].to(dev), res[0].to(dev), torch.empty(1, L, C, device=dev)
        keep = [xd, wd, rd, out, bs]
        call = lambda: lib.ev_op_conv1d(xd.data_ptr(), wd.data_ptr(), bs[0].data_ptr(), 0, rd.data_ptr(), out.data_ptr(), 1, L, C, C, K, 1, None, 1,
                                        _abi.ACT_LRELU, 0.1, _abi.ACT_NONE, _abi.ACC_STORE, 1.0, st)
        return dict(call=call, keep=keep, kname="conv1d_tm (fp32 FFMA), C=128 k=11 L=%d" % L, flops=2.0 * L * C * C * K,
                    alg_bytes=4.0 * (L * C * 3) + 4.0 * K * C * C, mma_mult=1, rate=None, L=L)
    gmode = {"fp32": 3, "tf32": 0, "bf16": 2}[precision]
    bf = precision == "bf16"
    pack = packing.to_tc16x2_layout if gmode == 3 else (packing.to_tc16_layout if bf else packing.to_tc_layout)
    wd = [pack(w).to(dev) for w in ws]
    xd = [layout.to_gp(x, bf).to(dev) for x in xs]
    od = [layout.to_gp(r, bf).to(dev) for r in res]          # residual and output (in place, as the engine's x_j += c2_j(...))
    n = len(Ks)
    VP, IA = ctypes.c_void_p * n, ctypes.c_int * n
    tabs = dict(x=VP(*[t.data_ptr() for t in xd]), w=VP(*[t.data_ptr() for t in wd]), b=VP(*[t.data_ptr() for t in bs]),
                o=VP(*[t.data_ptr() for t in od]), K=IA(*Ks), d=IA(*([1] * n)))
    keep = [wd, xd, od, bs, tabs]
    call = lambda: lib.ev_op_conv1d_gp_group(n, tabs["x"], tabs["w"], gmode, tabs["b"], tabs["o"], tabs["o"], tabs["K"], tabs["d"], 1, L, C, C, None, 1,
                                             _abi.ACT_LRELU, 0.1, st)
    esize = 2 if bf else 4
    kname = "conv1d_gp grouped launch (3 ResBlock convolutions k=11,7,3; %s), C=128 L=%d" % (
        {3: "bf16x3: fp32 activations, 3 bf16 MMAs per K=16", 0: "tf32", 2: "bf16 activations"}[gmode], L)
    return dict(call=call, keep=keep, kname=kname, flops=2.0 * L * C * C * sum(Ks), alg_bytes=float(esize) * (L * C * 3) * n + 4.0 * sum(Ks) * C * C,
                mma_mult=3 if gmode == 3 else 1, rate="tf32 = half the bf16 rate" if gmode == 0 else "bf16 rate", L=L)


def dominant_kernel_roofline(lib, dev, frames, peaks, flush, precision="fp32"):
    """`roofline` of the bench line: dominant_launch() timed live with CUDA events on the launching stream, L2 flushed before every launch."""
    from emotivoice_b200 import _abi
    d = dominant_launch(lib, dev, frames, precision)
    times = []
    for i in range(13):
        flush()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _abi.check(d["call"]())
        e1.record()
        e1.synchronize()
        if i >= 3:
            times.append(e0.elapsed_time(e1) * 1e-3)
    t = statistics.mean(times)
    achieved = d["flops"] / t / 1e12
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")   # dram bytes/launch from the committed ncu --set full capture
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(precision, {}).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    exec_frac = d["mma_mult"] * (2 if precision == "tf32" else 1) * achieved / peaks["bf16_tflops"]
    roof = {"bound": "tensor", "achieved": _r(achieved), "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
            "frac": achieved / peaks["bf16_tflops"], "traffic": traffic,
            "kernel": d["kname"], "ms": _r(t * 1e3),
            "peak_is": "%s bf16 burst (cuBLAS); `achieved` counts ALGORITHMIC flops, the mode executes %dx of them at the %s"
                       % (peaks["source"], d["mma_mult"], d["rate"]),
            "tensor_pipe_frac_est": _r(exec_frac), "alg_gbs": _r(d["alg_bytes"] / t / 1e9)}
    full = dict(roof, flops_per_launch=d["flops"], algorithmic_bytes_per_launch=d["alg_bytes"], times_ms=[x * 1e3 for x in times])
    return roof, full


def b32_block(model, dev, flush, headline_precision, conf, sd_cpu):
    """BASELINE.json configs[2]: batch 32, mixed EN/ZH, 20-200 phonemes, bf16.  Device-timed; parity of 3 items against the
    CPU oracle's B=1 fp32 runs (the batch-invariant contract: every item equals the reference's B=1 call)."""
    from emotivoice_b200 import synth
    utts = [synth.corpus_utterance(10_000 + i) for i in range(32)]
    utts.sort(key=lambda u: -len(u["ids"]))
    batch = {k: v.to(dev) for k, v in synth.collate_utterances(utts).items()}
    res = {"phonemes": "U{20..200}, 16 EN + 16 ZH"}
    for prec in ("bf16", headline_precision):
        model.precision = prec
        for _ in range(2):
            out = model(**batch)
        ts, outs = timed_forwards(lambda i: model(**batch), 5, flush, keep_last=True)
        out = outs[-1]
        t = statistics.median(ts)
        valid = int(out["mel_lengths_host"].sum())
        padded = int(32 * out["dec_outputs"].shape[1])
        res[prec] = {"ms": _r(t * 1e3), "valid_fps": _r(valid / t), "x_rt": _r(valid * HOP / SR / t)}
        res["valid_frames"], res["padded_frames"] = valid, padded
        if prec == "bf16":
            from oracle import jets_oracle as O
            errs, dur_ok = [], True
            for b in (0, 15, 31):
                ref = O.jets_forward(sd_cpu, conf, **synth.collate_utterances([utts[b]]))
                Fb = int(ref["dec_outputs"].shape[1])
                dur_ok = dur_ok and bool(torch.equal(out["log_duration_predictions"][b, :len(utts[b]["ids"])].cpu(), ref["log_duration_predictions"][0]))
                if int(out["mel_lengths_host"][b]) == Fb:
                    w, rw = out["wav_predictions"][b, 0, :Fb * HOP].cpu(), ref["wav_predictions"][0, 0]
                    errs.append(float((w - rw).double().pow(2).mean().sqrt() / rw.double().pow(2).mean().sqrt()))
            res["parity_bf16_vs_oracle_b1"] = {"items": 3, "dur_equal": dur_ok, "wav_relrms_max": _r(max(errs), 3) if errs else None, "tol": 2e-2}
    model.precision = headline_precision
    return res


def voc_block(model, dev, flush, peaks, headline_precision, lean):
    """BASELINE.json configs[3]: vocoder-only points with the layer-granular traffic accounting of SURVEY.md s8d."""
    from emotivoice_b200 import synth
    res = {}
    points = [(8, 1024)] if lean else [(1, 1024), (8, 1024), (32, 1024)]
    for prec in dict.fromkeys((headline_precision, "tf32", "bf16")):
        model.precision = prec
        for (B, F) in points:
            mel = synth.make_mel(B, F, seed=B * 7 + F).to(dev)
            model.generator(mel)
            ts, _ = timed_forwards(lambda i: model.generator(mel), 3, flush, keep_last=True)
            t = statistics.median(ts)
            res["%s_b%d_f%d" % (prec, B, F)] = {"ms": _r(t * 1e3), "fps": _r(B * F / t), "tflops": _r(B * F * VOC_FLOP_PER_FRAME / t / 1e12),
                                               "hbm_frac": _r(B * F * VOC_BYTES_PER_FRAME / t / 1e9 / peaks["hbm_gbs"], 3)}
            del mel
    model.precision = headline_precision
    res["hbm_frac_is"] = "5,010,752 B/frame (fp32 layer-granular) / time / %s GB/s" % peaks["hbm_gbs"]
    return res


def cfg5_block(model, dev, rank, world, dist, per_gpu=256, total_fixed=None):
    """BASELINE.json configs[4] (offline batch over the GPUs), scaled to fit a bench run: the first `world * per_gpu`
    utterances of the seeded 20-200-phoneme corpus (weak scaling; utterance i is the same at every world size), dealt to the
    ranks by runner.plan_shards (LPT), synthesised in B=32 length buckets with pinned int16 D2H; wall clock per rank over
    its whole shard (host collate, H2D, forward with its length sync, PCM conversion, D2H, trimming + hashing).
    `digest_first` covers utterances 0..per_gpu-1, present at every world size: equal digests across N = bit-identical PCM."""
    from emotivoice_b200 import synth, runner
    n = total_fixed or world * per_gpu
    lens = synth.corpus_lengths(n)
    mine = runner.plan_shards(lens, world)[rank]
    utts = {i: synth.corpus_utterance(i) for i in mine}
    ulist = [utts.get(i) or {"ids": [0] * lens[i]} for i in range(n)]        # placeholders keep global indices
    # warm-up: two buckets (allocator, pinned pools)
    runner.synthesize_corpus(model, ulist, dev, batch_size=32, indices=mine[:64], keep_pcm=False)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    st = {}
    t0 = time.perf_counter()
    res = runner.synthesize_corpus(model, ulist, dev, batch_size=32, indices=mine, keep_pcm=False, stats=st)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    frames = sum(v[1] for v in res.values())
    pairs = [(i, v[2]) for i, v in res.items() if i < per_gpu]
    rec = dict(rank=rank, wall_s=wall, frames=frames, utts=len(res), pairs=pairs, stats=st)
    if dist is not None:
        allrec = [None] * world
        dist.all_gather_object(allrec, rec)
    else:
        allrec = [rec]
    if rank != 0:
        return None, None
    tmax = max(r["wall_s"] for r in allrec)
    tot_frames = sum(r["frames"] for r in allrec)
    tot_utts = sum(r["utts"] for r in allrec)
    digest = runner.combine_digests([tuple(p) for r in allrec for p in r["pairs"]])
    slow = max(allrec, key=lambda r: r["wall_s"])["stats"]
    out = {"utts": tot_utts, "per_gpu": per_gpu, "batch": 32, "wall_s": _r(tmax), "utt_per_s": _r(tot_utts / tmax),
           "fps": _r(tot_frames / tmax), "x_rt": _r(tot_frames * HOP / SR / tmax), "rank_wall_min_s": _r(min(r["wall_s"] for r in allrec)),
           "host_collate_s": _r(slow["collate_s"], 3), "host_finish_s": _r(slow["finish_s"], 3),
           "digest_first%d" % per_gpu: digest[:16]}
    return out, allrec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--precision", default=os.environ.get("EV_PRECISION", "fp32"), choices=["fp32", "tf32", "bf16", "fp32_ffma"])
    ap.add_argument("--lean", action="store_true", help="headline + roofline + cpu_baseline only (no b32 / voc / cfg5 blocks)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "engine":
        args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        reference_arm(args, rank)
        return

    import __graft_entry__  # noqa: F401  (sys.path)
    from emotivoice_b200 import build as _build
    if not _build.up_to_date():
        sys.exit("bench.py: %s is missing or older than its sources; build it first (python -m emotivoice_b200.build)" % _build.LIB_PATH)
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"      # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        dist.init_process_group("nccl", device_id=dev)
        dist.barrier()                              # also creates the communicator, so the broadcast below times the copy only

    from emotivoice_b200.config import default_config
    from emotivoice_b200 import synth, _abi, runner
    from emotivoice_b200.modules import JETSGenerator

    conf = default_config()
    sd_cpu = synth.make_state_dict(conf) if rank == 0 else None
    t_setup0 = time.perf_counter()
    model = JETSGenerator(conf).to(dev)
    bcast = None
    if world > 1:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sd = runner.broadcast_state_dict(sd_cpu, conf, dev, src=0)     # raw parameters (213 MB), one NCCL broadcast
        model.load_state_dict(sd)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        nbytes = runner.broadcast_engine(model, dev, src=0)            # rank 0 packs once; the packed blob, one NCCL broadcast
        torch.cuda.synchronize()
        bcast = {"raw_ms": _r((t1 - t0) * 1e3), "pack_and_blob_ms": _r((time.perf_counter() - t1) * 1e3), "blob_mb": _r(nbytes / 1e6)}
    else:
        model.load_state_dict(sd_cpu)
    model.eval()
    model.precision = args.precision
    lib = _abi.load()
    setup_s = time.perf_counter() - t_setup0

    # ---- this rank's shard of the corpus ------------------------------------------------------------
    n_steps = args.warmup + args.steps
    total = world * n_steps
    shard = runner.plan_shards(synth.corpus_lengths(total, n_phonemes=N_PHONEMES), world)[rank]
    assert len(shard) == n_steps
    utts = [synth.corpus_utterance(i, n_phonemes=N_PHONEMES) for i in shard]
    dev_batches = [{k: v.to(dev) for k, v in synth.collate_utterances([u]).items()} for u in utts]
    h2d_bytes = sum(v.numel() * v.element_size() for v in dev_batches[0].values())

    flush_buf = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # 256 MiB > 126 MB L2

    def flush():
        flush_buf.zero_()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # serving set-up: size the workspace arena once (no device allocation inside the timed steps when a longer utterance arrives)
    model.reserve(batch=1, phonemes=N_PHONEMES + 28, frames=1024)

    # ---- warm-up -----------------------------------------------------------------------
    for s in range(args.warmup):
        out = model(**dev_batches[s])
    torch.cuda.synchronize()
    parity = parity_vs_fixture(model, dev) if rank == 0 else None

    # ---- timed: inputs resident in HBM -------------------------------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    l0 = _abi.launch_count()
    wall0 = time.perf_counter()
    last = {}

    def value_step(s):      # the outputs are dropped at once (only their shapes are kept): holding 20 waveforms would make torch's allocator
        o = model(**dev_batches[args.warmup + s])      # cudaMalloc fresh segments inside the timed region (a device-synchronising call)
        if args.dump_outputs and s == args.steps - 1:
            last.update(o)
        return int(o["dec_outputs"].shape[1]), int(o["wav_predictions"].shape[-1])

    ts, outs = timed_forwards(value_step, args.steps, flush)
    barrier()
    wall = time.perf_counter() - wall0
    launches = _abi.launch_count() - l0
    dev_s = sum(ts)
    frames = sum(o[0] for o in outs)
    n_samples = sum(o[1] for o in outs)
    del outs

    # ---- timed: end to end from host data (collate -> pinned -> H2D -> forward -> wav D2H pinned) --------
    max_samples = 1 << 20
    wav_pin = torch.empty((max_samples,), dtype=torch.float32).pin_memory()

    def e2e_step(s):
        batch = synth.collate_utterances([utts[args.warmup + s]], pin=True)
        o = model(**{k: v.to(dev, non_blocking=True) for k, v in batch.items()})
        w = o["wav_predictions"].reshape(-1)
        wav_pin[:w.numel()].copy_(w, non_blocking=True)
        torch.cuda.current_stream().synchronize()      # the caller holds the waveform on the host before the next request starts
        return int(o["dec_outputs"].shape[1])

    for s in range(2):
        e2e_step(s)
    barrier()
    ts2, fr2 = timed_forwards(e2e_step, args.steps, flush)
    barrier()
    e2e_s, e2e_frames = sum(ts2), sum(fr2)
    clocks = sampler.stop() if rank == 0 else None
    if last and rank == 0:
        dump_outputs(args.dump_outputs, last)
    last.clear()

    # ---- whole job: sum of frames over ranks / max over ranks of time ------------------------------------------
    t = torch.tensor([dev_s, e2e_s, float(frames), float(e2e_frames), float(launches)], dtype=torch.float64, device=dev)
    if dist is not None:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        dev_s, e2e_s = float(tmax[0]), float(tmax[1])
        total_frames, total_e2e_frames, total_launches = float(tsum[2]), float(tsum[3]), int(tsum[4])
    else:
        total_frames, total_e2e_frames, total_launches = float(frames), float(e2e_frames), int(launches)

    line, detail = None, {}
    if rank == 0:
        peaks = _peaks()
        value = total_frames / dev_s
        audio_s = frames * HOP / SR
        line = {
            "metric": "mel_frames_per_sec", "value": _r(value, 6), "unit": "mel-frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": _r(dev_s / args.steps * 1e3, 5), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None,
            "dtype": {"fp32": "fp32 (fp32 storage + accumulate; tcgen05 fp32 emulation: 3xTF32 prefix, bf16x3 after it)", "tf32": "tf32",
                      "bf16": "bf16 (fp32 accumulate)", "fp32_ffma": "fp32 (FFMA)"}[args.precision],
            "data": "synthetic", "config": CONFIG,
            "rtf": _r(dev_s / audio_s), "x_realtime": _r(audio_s / dev_s),
            "clocks": clocks,
            "e2e": {"value": _r(total_e2e_frames / e2e_s, 6), "unit": "mel-frames/s", "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": int(n_samples * 4 // args.steps), "ms_per_step": _r(e2e_s / args.steps * 1e3, 5),
                    "x_realtime": _r(audio_s / e2e_s)},
            "gpu_launches": total_launches,
            "parity": parity,
        }
        detail.update(precision=args.precision, frames_rank0=frames, audio_seconds_rank0=audio_s, wall_ms_per_step_incl_flush=wall / args.steps * 1e3,
                      weight_broadcast=bcast, setup_s=setup_s, step_ms_rank0=[x * 1e3 for x in ts], e2e_step_ms_rank0=[x * 1e3 for x in ts2],
                      launches_per_step=total_launches / (args.steps * world), peaks=peaks)
        if bcast:
            line["weights"] = bcast
        try:
            roof, roof_full = dominant_kernel_roofline(lib, dev, frames // args.steps, peaks, flush, args.precision)
            line["roofline"] = roof
            detail["roofline"] = roof_full
        except Exception as e:
            line["roofline"] = {"bound": "tensor", "achieved": None, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": None,
                                "traffic": None, "error": repr(e)[:200]}

    # ---- secondary blocks (the headline numbers above are final) ---------------------------------------
    if not args.lean:
        if rank == 0:
            for name, fn in (("b1", lambda: b1_block(model, dev, flush, line["parity"])),
                             ("b32", lambda: b32_block(model, dev, flush, args.precision, conf, sd_cpu)),
                             ("voc", lambda: voc_block(model, dev, flush, peaks, args.precision, world > 1))):
                try:
                    line[name] = fn()
                except Exception as e:
                    line[name] = {"error": repr(e)[:200]}
                torch.cuda.empty_cache()
        try:
            c5, recs = cfg5_block(model, dev, rank, world, dist)
            if rank == 0:
                line["cfg5"] = c5
                detail["cfg5_ranks"] = [{k: v for k, v in r.items() if k != "pairs"} for r in recs]
        except Exception as e:
            if rank == 0:
                line["cfg5"] = {"error": repr(e)[:200]}
        try:
            # the same pipeline on a FIXED 2048-utterance corpus (strong scaling: the shard shrinks as N grows); the digest
            # covers every utterance, so equal digests across world sizes = the whole corpus is bit-identical
            c5s, recs = cfg5_block(model, dev, rank, world, dist, per_gpu=2048, total_fixed=2048)
            if rank == 0:
                line["cfg5_strong"] = {"utts": c5s["utts"], "wall_s": c5s["wall_s"], "utt_per_s": c5s["utt_per_s"], "fps": c5s["fps"],
                                       "rank_wall_min_s": c5s["rank_wall_min_s"], "digest": c5s["digest_first2048"]}
                detail["cfg5_strong_ranks"] = [{k: v for k, v in r.items() if k != "pairs"} for r in recs]
        except Exception as e:
            if rank == 0:
                line["cfg5_strong"] = {"error": repr(e)[:200]}

    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    # the other ranks have left: the host cores are free for the CPU baseline
    if not args.no_cpu_baseline:
        try:
            r, _ = cpu_reference_run(steps=12, warmup=1)
            line["cpu_baseline"] = {"value": _r(r["fps"], 5), "unit": "mel-frames/s", "cores": r["cores"], "kind": "port",
                                    "sample": "12 B=1 forwards over corpus utterances (oracle/jets_oracle.py, torch CPU, %d threads of %d usable), %.0f ms each"
                                              % (r["cores"], r["usable"], r["seconds"] / r["steps"] * 1e3)}
            detail["cpu_baseline"] = r
        except Exception as e:
            line["cpu_baseline"] = {"value": None, "unit": "mel-frames/s", "cores": 0, "kind": "port", "sample": "failed: " + repr(e)[:120]}
    emit(line, detail)


def b1_block(model, dev, flush, parity):
    """configs[1] on the committed fixture utterance (537 frames): device and end-to-end latency of ONE fixed utterance."""
    import numpy as np
    z = np.load(os.path.join(ROOT, "tests", "golden", "b1_t100.npz"))
    keys = ("inputs_ling", "input_lengths", "inputs_speaker", "inputs_style_embedding", "inputs_content_embedding")
    batch = {k: torch.from_numpy(z[k]).to(dev) for k in keys}
    for _ in range(2):
        out = model(**batch)
    ts, outs = timed_forwards(lambda i: model(**batch), 10, flush, keep_last=True)
    frames = int(outs[-1]["dec_outputs"].shape[1])
    t = statistics.median(ts)
    return {"frames": frames, "ms": _r(t * 1e3), "x_rt": _r(frames * HOP / SR / t), "ms_min": _r(min(ts) * 1e3)}


if __name__ == "__main__":
    main()
