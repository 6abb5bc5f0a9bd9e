#!/usr/bin/env python
"""Benchmark of the Tortoise `preset='standard'` hot path (BASELINE.json metric: audio-seconds per wall-second).

  python bench.py --gpus N --steps K --warmup W            # this engine (one rank per GPU under torchrun for N>1)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port) on the host cores
  python bench.py ... --dump-outputs DIR                   # + the last timed step's waveform(s) as DIR/<name>.npy

A step = one `TextToSpeech.tts_with_preset(preset='standard')` call (256 AR candidates, 200 diffusion iterations,
k=1) on the 53-word paragraph of SURVEY §8d config 3 (T=169 BPE tokens, N=430 mel tokens => S=1872 mel frames,
19.97 s of 24 kHz audio), synthetic seeded checkpoint in the reference layout (EOS suppressed so that every candidate
runs exactly N steps), synthetic conditioning latents. Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "audio-seconds/sec at preset='standard'"
UNIT = "audio-s/s"


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the probed kernels, parsed from the committed ncu
    --set full captures by tools/ncu_traffic.py into profiles/ncu_traffic.json ({probe-name prefix: {bytes, source}})."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return {}
    with open(p) as f:
        return json.load(f)


def load_tokens(name="para53"):
    with open(os.path.join(ROOT, "tests", "golden", "bench_text_tokens.json")) as f:
        return json.load(f)[name]["tokens"]


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [v.strip() for v in out.strip().split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for n, v in zip(names, f[2:6]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


_T0 = time.perf_counter()


def progress(msg):
    """stderr breadcrumbs (stdout carries only the JSON line): a run cut off by a timeout still says where it was."""
    if os.environ.get("RANK", "0") == "0":
        sys.stderr.write("[bench %7.1fs] %s\n" % (time.perf_counter() - _T0, msg))
        sys.stderr.flush()


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["hbm_gbs"], d.get("bf16_tflops_sustained", d["bf16_tflops"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1400.0, "fallback (B200_PROFILING.md)"


def kernel_probes(tts, cfg, n_mel, B, P, iters=200):
    """Times the candidate dominant kernels live, in isolation at the workload's shapes, with CUDA events on the
    launching stream; returns per-kernel dicts with achieved throughput against the roofline that bounds each."""
    import torch
    from tortoise_tts_b200 import lib
    dev = tts.device
    hbm, tfl, how = peaks()
    out = []

    def timeit(fn, reps=10, flush=None):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            if flush is not None:
                flush.zero_()          # > L2 (126 MB) write between timed launches
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return sum(ts) / len(ts)

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    S = n_mel * 4 * 24000 // 22050
    C, H = cfg.diff_dim, cfg.diff_heads
    # (1) diffusion attention: B=2 (cond+uncond), 16 heads, S x S, relative-position bias
    qkv = torch.randn(2 * S, 3 * C, device=dev).to(torch.bfloat16)
    o = torch.empty(2 * S, C, device=dev, dtype=torch.bfloat16)
    from tortoise_tts_b200.diffusion_engine import _rel_pos_table
    bias = _rel_pos_table(torch.randn(32, H, device=dev), S, 8.0)      # T5 table as the denoiser uses it
    ms = timeit(lambda: lib.attention(qkv, o, nseq=2, T=S, H=H, ld=3 * C, ldo=C, k_off=C, v_off=2 * C, scale=0.125, bias=bias,
                                      bias_sat=64), flush=flush)
    flops = 2 * H * 4.0 * S * S * 64
    out.append(dict(kernel="diffusion attention (2x16 heads, S=%d)" % S, bound="tensor", ms=ms, count=13 * iters,
                    achieved=flops / ms / 1e9, peak=tfl, unit="TFLOP/s"))
    # (2) diffusion conv k=3 as GEMM: [2, S, 1024] x [1024, 3*1024]
    a = torch.randn(2, S, C, device=dev).to(torch.bfloat16)
    w = (torch.randn(C, 3 * C, device=dev) * 0.02).to(torch.bfloat16)
    x = torch.zeros(2, S, C, device=dev)
    bb = torch.zeros(C, device=dev)
    ms = timeit(lambda: lib.gemm(a, w, M=S, N=C, K=C, taps=3, pad=1, bias=bb, residual=x, out_f32=x, batch=2, a_bstride=S * C,
                                 res_bstride=S * C, outf_bstride=S * C), flush=flush)
    flops = 2 * 2.0 * S * C * 3 * C
    out.append(dict(kernel="diffusion conv k=3 GEMM (tcgen05, M=2x%d N=1024 K=3072)" % S, bound="tensor", ms=ms,
                    count=16 * iters, achieved=flops / ms / 1e9, peak=tfl, unit="TFLOP/s"))
    # (3) the AR decode step at the mean context (step n_mel/2): ONE kernel = all 30 layers + mel_head for every candidate
    # of this GPU. Algorithmic bytes per launch (DESIGN §4): every weight once (bf16) + the shared prompt K/V once per layer
    # + every candidate's own K/V (bf16) of the n_mel/2 positions decoded so far.
    eng = tts.autoregressive
    st = eng._decode_state(B, P, n_mel)
    Hh, D, L = cfg.ar_heads, cfg.ar_dim, cfg.ar_layers
    mode = st["mode"]
    if st["fused"]:
        # the decode workspace may be split into chains (TTB_AR_CHAINS): each chain launches these kernels on its own
        # half of the candidates, so the probe times one chain's launch and counts it once per chain
        ch = st["chains"][0]
        nch, Bc = len(st["chains"]), ch["B"]
        hd = eng._step_handle(ch, 1)
        ch["state"].zero_()
        ch["state"][0] = n_mel // 2
        ch["codes"].zero_()
        ms = timeit(lambda: hd.step(), flush=flush)
        assert int(ch["state"][2].item()) == 0, "ar_step_kernel timed out internally"
        w_bytes = (L * 12 * D * D + cfg.number_mel_codes * D) * 2
        kv_bytes = L * Hh * P * 128 * 2 + Bc * L * Hh * (n_mel // 2) * 128 * 2
        out.append(dict(kernel="AR decode step kernel (B=%d, ctx=%d+%d, 30 layers + mel_head)" % (Bc, P, n_mel // 2),
                        bound="hbm", ms=ms, count=(n_mel - 1) if mode == "fused" else 0,
                        achieved=(w_bytes + kv_bytes) / ms / 1e6, peak=hbm, unit="GB/s", algorithmic_bytes=w_bytes + kv_bytes))
        # the attention kernel as the mixed mode launches it: all L layers back to back (every layer streams its own
        # slice of the 13.5 GB cache, so nothing is reused from the 126 MB L2 between launches), per-launch = / L
        def all_layers():
            for l in range(L):
                hd.step(phase_mask=4, layer_begin=l, layer_end=l + 1)
        ms_a = timeit(all_layers, flush=flush) / L
        nbytes = Bc * Hh * (n_mel // 2) * 128 * 2 + Hh * P * 128 * 2
        kname = "ar_attn_compact_kernel" if ch.get("compact") else "ar_attn_only_kernel"
        out.append(dict(kernel="AR decode attention kernel (%s, one layer, B=%d, ctx=%d+%d; mean of %d "
                               "back-to-back layers)" % (kname, Bc, P, n_mel // 2, L), bound="hbm", ms=ms_a,
                        count=nch * L * (n_mel - 1) if mode == "mixed" else 0,
                        achieved=nbytes / ms_a / 1e6, peak=hbm, unit="GB/s", algorithmic_bytes=nbytes))
    else:
        ck = torch.zeros(B, Hh, n_mel, 64, device=dev, dtype=torch.bfloat16)
        cv = torch.zeros_like(ck)
        pk = torch.zeros(Hh, P, 64, device=dev, dtype=torch.bfloat16)
        pv = torch.zeros_like(pk)
        qkv2 = torch.randn(B, 3 * D, device=dev).to(torch.bfloat16)
        o2 = torch.empty(B, D, device=dev, dtype=torch.bfloat16)
        state = torch.zeros(64, dtype=torch.int32, device=dev)
        state[0] = n_mel // 2
        so = torch.zeros(2, B, D, device=dev)
        sl = torch.zeros(2, B, Hh, device=dev)
        ms = timeit(lambda: lib.ar_decode_attention(qkv2, pk, pv, ck, cv, state, B, Hh, P, n_mel, o2, so, sl), flush=flush)
        nbytes = B * Hh * (n_mel // 2) * 64 * 2 * 2 + Hh * P * 64 * 2 * 2
        out.append(dict(kernel="AR decode attention (B=%d, ctx=%d+%d)" % (B, P, n_mel // 2), bound="hbm", ms=ms,
                        count=30 * (n_mel - 1), achieved=nbytes / ms / 1e6, peak=hbm, unit="GB/s", algorithmic_bytes=nbytes))
    for d in out:
        d["frac"] = d["achieved"] / d["peak"]
        d["total_ms_per_utterance"] = d["ms"] * d["count"]
    return out, how


def config5_tokens(base):
    """BASELINE configs[4]: 8 long utterances. Token lists of growing length built by cycling the 169-token paragraph
    (T = 169 ... 337; SURVEY quotes T up to ~380, capped here so that the prompt fits the one-kernel decode step)."""
    return [[base[i % len(base)] for i in range(n)] for n in (169, 193, 217, 241, 265, 289, 313, 337)]


DUMP_BYTES = 63 << 20          # --dump-outputs: at most 64 MB on disk, .npy headers included


def dump_outputs(d, wav):
    """Writes what the timed call returned (the waveform, or one per candidate for k > 1) as float32 DIR/<name>.npy, so
    that two builds can be compared output for output. Beyond DUMP_BYTES in all, every array is cut to the same fixed,
    seeded share of its elements."""
    import numpy as np
    wavs = wav if isinstance(wav, list) else [wav]
    arrays = {"wav" if len(wavs) == 1 else "wav_%d" % i: w.float().numpy() for i, w in enumerate(wavs)}
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            keep = np.random.default_rng(0).permutation(a.size)[:a.size * DUMP_BYTES // total]
            a = a.reshape(-1)[np.sort(keep)]
        np.save(os.path.join(d, name + ".npy"), a)


ITERS = {"standard": 200, "fast": 80, "ultra_fast": 30, "high_quality": 400}
NCAND = {"standard": 256, "high_quality": 256, "fast": 96, "ultra_fast": 16}


def run_engine(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=300))
    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    from tortoise_tts_b200.config import ModelConfig
    from tortoise_tts_b200.synth import synth_all
    from tortoise_tts_b200.api import TextToSpeech
    from tortoise_tts_b200 import lib
    progress("extension built; synthesising the full-size checkpoint")
    cfg = ModelConfig.full()
    sds = synth_all(cfg, seed=0, suppress_stop=True)
    progress("checkpoint ready; loading engines")
    tts = TextToSpeech(state_dicts=sds, config=cfg, kv_cache=True, device="cuda:%d" % local)
    progress("engines ready")
    tokens = load_tokens(args.text)
    config5 = args.workload == "config5"
    preset = "high_quality" if config5 else args.preset
    n_mel = 500 if config5 else args.mel_tokens
    g = torch.Generator().manual_seed(0)
    cl_host = ((torch.randn(1, cfg.ar_dim, generator=g) * 0.5).pin_memory(),
               (torch.randn(1, 2 * cfg.diff_dim, generator=g) * 0.3).pin_memory())
    kw = dict(conditioning_latents=cl_host, max_mel_tokens=n_mel, verbose=False, k=1)
    if args.preset_override:
        kw.update(json.loads(args.preset_override))
    utt = config5_tokens(tokens) if config5 else [tokens]

    def step(i):
        if config5:
            # read.py loop: 8 utterances, one whole utterance per GPU (no collective inside an utterance)
            return tts.tts_long("|".join("u%d" % u for u in range(len(utt))), preset=preset, text_tokens_list=utt,
                                use_deterministic_seed=1000 + i, **kw)
        return tts.tts_with_preset("", preset=preset, text_tokens=tokens, use_deterministic_seed=1000 + i, **kw)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        wav = step(i)
        progress("warm-up %d done: %s" % (i, {k_: round(v, 1) for k_, v in tts.last_timings.items()}))
    sampler = ClockSampler(local)
    sampler.start()
    sync()
    c0 = lib.CALLS
    dev_ms = []
    stage = {}
    t0 = time.perf_counter()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(args.steps):
        ev0.record()
        wav = step(args.warmup + i)
        ev1.record()
        torch.cuda.synchronize()
        # device time of the step: CUDA events on the launching stream around the whole call (config5: the sum of this
        # rank's utterances); for one utterance this equals the stage events inside tts()
        dev_ms.append(ev0.elapsed_time(ev1) if config5 else tts.last_timings["device_total_ms"])
        progress("timed step %d: %.1f ms on device" % (i, dev_ms[-1]))
        for k_, v in tts.last_timings.items():
            stage[k_] = stage.get(k_, 0.0) + v / args.steps
    sync()
    wall = time.perf_counter() - t0
    sampler.stop_flag = True
    launches = lib.CALLS - c0
    audio_s = wav.shape[-1] / 24000.0
    ms_per_step = wall / args.steps * 1e3
    dev_step = sum(dev_ms) / len(dev_ms)
    if world > 1:
        t = torch.tensor([ms_per_step, dev_step], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_per_step, dev_step = float(t[0]), float(t[1])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, wav)
    B = NCAND[preset]
    iters = ITERS[preset]
    h2d = sum(t.numel() * 4 for t in cl_host) * len(utt) + sum(4 * (len(u) + 1) for u in utt)
    if config5:
        workload = ("configs[4]: preset='high_quality' (256 AR samples, 400 diffusion iters), 8 utterances of %s BPE tokens, "
                    "N=%d mel tokens each -> %.1f s audio, k=1" % ("/".join(str(len(u)) for u in utt), n_mel, audio_s))
        par = "whole utterances sharded %d/GPU (read.py loop), no collective inside an utterance" % ((len(utt) + world - 1) // world)
    else:
        workload = ("configs[2]: preset='%s' (%d AR samples, %d diffusion iters), %d-token paragraph, N=%d mel tokens -> "
                    "%.2f s audio, k=1" % (preset, B, iters, len(tokens), n_mel, audio_s))
        par = "candidates sharded %d/GPU; CFG branch pair on 2 GPUs for the k=1 diffusion tail" % ((B + world - 1) // world)
        dec = getattr(tts.autoregressive, "_dec", None)       # how the decode step of this run was organised
        if dec is not None:
            par += "; decode step: %s, %d chain(s) per GPU" % (dec["mode"], len(dec["chains"]))
    line = {
        "metric": METRIC if not config5 else "audio-seconds/sec at preset='high_quality' (8 utterances)",
        "value": audio_s / (dev_step / 1e3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "bf16 tensor-core operands, fp32 accumulate/residual/norm/softmax/scheduler",
        "data": "synthetic (seeded random checkpoint in the reference .pth layout, EOS suppressed; synthetic latents)",
        "config": {"workload": workload,
                   "l2": "working set (1.9 GB weights + %.1f GB KV cache) >> 126 MB L2; no flush between steps" %
                         (2 * 30 * ((B + world - 1) // world if not config5 else B) * 16 * n_mel * 64 * 2 / 1e9),
                   "parallelism": par},
        "e2e": {"value": audio_s / (ms_per_step / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": int(wav.numel() * 4)},
        "gpu_launches": int(launches),
        "clocks": sampler.summary(),
        "stage_ms": {k_: round(v, 2) for k_, v in stage.items()},
    }
    if not config5:
        # the two phases scale differently (SURVEY §8e): candidates shard over all GPUs, the k=1 tail over a pair
        line["phase_ms"] = {"candidate_sharded (ar+clvp)": round(stage.get("ar_ms", 0) + stage.get("clvp_ms", 0), 2),
                            "tail (latents+diffusion+vocoder)": round(stage.get("latents_ms", 0) + stage.get("diffusion_ms", 0)
                                                                      + stage.get("vocoder_ms", 0), 2)}
    if world == 1 and not config5:
        progress("kernel probes")
        probes, how = kernel_probes(tts, cfg, n_mel, B, len(tokens) + 5, iters)
        progress("probes done")
        dom = max(probes, key=lambda d: d["total_ms_per_utterance"])
        traffic, source = None, None
        best = ""
        for key, val in ncu_traffic().items():          # the most specific (longest) matching probe-name prefix
            if dom["kernel"].startswith(key) and len(key) > len(best):
                best, traffic, source = key, val["bytes"], val["source"]
        line["roofline"] = {"kernel": dom["kernel"], "bound": dom["bound"], "achieved": round(dom["achieved"], 2),
                            "peak": dom["peak"], "unit": dom["unit"], "frac": round(dom["frac"], 4), "traffic": traffic,
                            "traffic_source": source, "peak_source": how, "launch_ms": round(dom["ms"], 4),
                            "algorithmic": dom.get("algorithmic_bytes")}
        line["kernels"] = [{k_: (round(v, 4) if isinstance(v, float) else v) for k_, v in d.items()} for d in probes]
        if not args.no_cpu_baseline:
            progress("cpu baseline (reference modules on the host cores)")
            line["cpu_baseline"] = cpu_baseline(args, "cpu")
            progress("cpu baseline done")
        if not args.no_ref_gpu:
            progress("reference in PyTorch eager on this GPU (BASELINE.md: bar to beat)")
            line["reference_gpu"] = cpu_baseline(args, "cuda")
            progress("reference-on-GPU done")
    print(json.dumps(line))
    sys.stdout.flush()
    if world > 1:
        dist.destroy_process_group()


def _ref_available():
    from oracle.ref_shims import reference_available
    return reference_available()


def _baseline_cmd(args, device, repeat=1):
    """The unmodified reference modules when they are importable (oracle/_ref or /root/reference), else the oracle port."""
    mod = "oracle.ref_baseline" if _ref_available() else "oracle.cpu_baseline"
    cmd = [sys.executable, "-m", mod, "--preset", args.preset, "--mel-tokens", str(args.mel_tokens),
           "--tokens-json", os.path.join(ROOT, "tests", "golden", "bench_text_tokens.json"), "--text", args.text,
           "--repeat", str(repeat)]
    if mod == "oracle.ref_baseline":
        cmd += ["--device", device]
    elif device != "cpu":
        return None
    return cmd


def cpu_baseline(args, device):
    # child process under a timeout: the baseline's thread pool must not inherit this process's CUDA-side state, and a
    # host whose CPU quota misbehaves must not take the GPU arm's JSON line down with it
    cmd = _baseline_cmd(args, device)
    if cmd is None:
        return {"value": None, "unit": UNIT, "kind": "port", "sample": "the oracle port has no %s mode" % device}
    try:
        out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=args.cpu_timeout)
        r = json.loads(out.stdout.strip().splitlines()[-1])
    except subprocess.TimeoutExpired:
        return {"value": None, "unit": UNIT, "cores": None, "kind": "reference" if _ref_available() else "port",
                "sample": "not finished within %d s on this host" % args.cpu_timeout}
    except (ValueError, IndexError):
        return {"value": None, "unit": UNIT, "cores": None, "kind": "port", "sample": "failed: " + out.stderr[-300:]}
    return {"value": r["value"], "unit": UNIT, "cores": r["cores"], "cores_available": r.get("cores_available"),
            "kind": r.get("kind", "port"), "device": r.get("device", "cpu"), "sample": r["sample"],
            "total_s_extrapolated": round(r["total_s"], 1), "units_s": {k: round(v, 4) for k, v in r["units"].items()}}


def run_reference(args):
    """The reference arm: the reference's own implementation of the path (its unmodified PyTorch modules, copied next to
    the oracle by oracle/build_ref.py; the oracle port only if that copy is missing) timed on the host cores - or, with
    --device cuda, in PyTorch eager on the GPU."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    tokens = load_tokens(args.text)
    n = args.warmup + args.steps
    cmd = _baseline_cmd(args, args.device, repeat=n)
    t0 = time.perf_counter()
    samples = []
    try:
        out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=args.cpu_timeout * n)
        txt, err = out.stdout, out.stderr
    except subprocess.TimeoutExpired as e:
        txt = e.stdout.decode() if isinstance(e.stdout, bytes) else (e.stdout or "")
        err = "timeout after %d s" % (args.cpu_timeout * n)
    for ln in txt.strip().splitlines():
        try:
            samples.append(json.loads(ln))
        except ValueError:
            pass
    wall = time.perf_counter() - t0
    timed = samples[args.warmup:] if len(samples) > args.warmup else samples[-1:]
    if not timed:
        print(json.dumps({"impl": "reference", "unavailable": "reference produced no sample: " + err[-200:].replace("\n", " ")}))
        return
    last = timed[-1]
    v = sum(s["value"] for s in timed) / len(timed)
    audio_s = (args.mel_tokens * 4 * 24000 // 22050) * 256 / 24000.0
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": audio_s / v * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[2]: preset='%s', %d-token paragraph, N=%d mel tokens (%s on %s, unit costs "
                                   "extrapolated)" % (args.preset, len(tokens), args.mel_tokens,
                                                      "unmodified reference modules" if last.get("kind") == "reference"
                                                      else "CPU oracle port of the reference path", last.get("device", "cpu"))},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": last["cores"], "cores_available": last.get("cores_available"),
                             "kind": last.get("kind", "port"), "sample": last["sample"]},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "bench_wall_s": round(wall, 1)}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--workload", default="config3", choices=["config3", "config5"],
                    help="config3 = BASELINE configs[2] (the metric's configuration; configs[3] under torchrun); config5 = "
                         "configs[4]: high_quality, 8 utterances, one per GPU")
    ap.add_argument("--device", default="cpu", choices=["cpu", "cuda"], help="--impl reference: where the reference runs")
    ap.add_argument("--preset", default="standard")
    ap.add_argument("--text", default="para53")
    ap.add_argument("--mel-tokens", type=int, default=430)
    ap.add_argument("--preset-override", default=None, help="JSON dict of tts kwargs (debug)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true")
    ap.add_argument("--cpu-timeout", type=int, default=240, help="seconds allowed per baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the waveform(s) of the last timed step as float32 DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_engine(args)


if __name__ == "__main__":
    main()
