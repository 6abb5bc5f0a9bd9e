"""Pins oracle/*.py against the UNMODIFIED reference modules: their results on the inputs below are stored in
tests/golden/reference_v1.pt (tests/ref_golden.py, which also says how to record them again)."""
import os

import numpy as np
import pytest
import torch

import ref_golden as rg
from oracle.ref_shims import load_reference
from tortoise_tts_b200.config import ModelConfig
from tortoise_tts_b200.synth import synth_all


@pytest.fixture(scope="module")
def small():
    cfg = ModelConfig.small()
    sds = synth_all(cfg, seed=0, suppress_stop=False)
    models = None
    if rg.RECORD:
        from oracle.ref_build import build_reference_models
        with torch.no_grad():
            models = build_reference_models(cfg, sds, kv_cache=True)
    return cfg, sds, models


TEXT = [42, 2, 194, 91, 24, 2, 243, 190, 2, 182, 37, 2, 0]  # once zero-padded, as api.py:391 does


def test_ar_teacher_forced_logits_recompute_path(small):
    """oracle teacher_forced_logits(train_consistent) == GPT2InferenceModel full-recompute forward."""
    from oracle import ar
    cfg, sds, m = small
    sd = sds["autoregressive"]
    torch.manual_seed(1)
    cond = torch.randn(1, cfg.ar_dim)
    codes = torch.randint(0, 8192, (2, 7))

    def reference():
        # recompute path of the inference model (kv_cache off => whole sequence every call)
        uv = m["autoregressive"]
        inf = uv.inference_model
        inf.kv_cache = False
        text = torch.tensor(TEXT[:-1] + [0]).unsqueeze(0)  # tokens + api pad
        ti = torch.nn.functional.pad(text, (0, 1), value=0)
        ti = torch.nn.functional.pad(ti, (1, 0), value=cfg.start_text_token)
        emb = uv.text_embedding(ti) + uv.text_pos_embedding(ti)
        emb = torch.cat([cond.unsqueeze(1), emb], dim=1)
        inf.store_mel_emb(emb)
        fake = torch.full((2, emb.shape[1] + 1), 1, dtype=torch.long)
        fake[:, -1] = cfg.start_mel_token
        ids = torch.cat([fake, codes], dim=1)
        out = inf(input_ids=ids, attention_mask=torch.ones_like(ids), return_dict=True)
        inf.kv_cache = True
        return out.logits[:, emb.shape[1]:]
    with torch.no_grad():
        want = ar.teacher_forced_logits(sd, cfg, cond, TEXT, codes, pos_mode="train_consistent")
        idx, got, shape = rg.sampled("ar_logits_recompute", reference)
    assert shape == want.shape
    assert (got - want.reshape(-1)[idx]).abs().max().item() < 2e-4


def test_ar_generate_matches_reference_kv_path(small):
    """With identical forced samples, oracle KV decode (ref_kv_quirk) logits == reference cached logits."""
    from oracle import ar
    cfg, sds, m = small
    sd = sds["autoregressive"]
    torch.manual_seed(2)
    cond = torch.randn(1, cfg.ar_dim)
    codes = torch.randint(0, 8192, (1, 5))

    def reference():
        uv = m["autoregressive"]
        inf = uv.inference_model
        text = torch.tensor(TEXT).unsqueeze(0)
        ti = torch.nn.functional.pad(text, (0, 1), value=0)
        ti = torch.nn.functional.pad(ti, (1, 0), value=cfg.start_text_token)
        emb = uv.text_embedding(ti) + uv.text_pos_embedding(ti)
        emb = torch.cat([cond.unsqueeze(1), emb], dim=1)
        inf.store_mel_emb(emb)
        fake = torch.full((1, emb.shape[1] + 1), 1, dtype=torch.long)
        fake[:, -1] = cfg.start_mel_token
        ids = fake
        past = None
        got = []
        for j in range(codes.shape[1] + 1):
            am = torch.ones_like(ids)
            if past is None:
                out = inf(input_ids=ids, attention_mask=am, use_cache=True, return_dict=True)
            else:
                out = inf(input_ids=ids[:, -1:], past_key_values=past, attention_mask=am, use_cache=True,
                          return_dict=True)
            past = out.past_key_values
            got.append(out.logits[:, -1])
            if j < codes.shape[1]:
                ids = torch.cat([ids, codes[:, j:j + 1]], dim=1)
        return torch.stack(got, dim=1)
    with torch.no_grad():
        want = ar.teacher_forced_logits(sd, cfg, cond, TEXT, codes, pos_mode="ref_kv_quirk")
        idx, got, shape = rg.sampled("ar_logits_kv", reference)
    assert shape == want.shape
    assert (got - want.reshape(-1)[idx]).abs().max().item() < 2e-4


def test_stream_latents_match_reference_kv_path(small):
    """oracle.stream_latents == what `sample_stream` yields next to every token (stream_generator.py:982):
    `final_norm(outputs.hidden_states[-1][:, -1])` of the cached forward, fed the same forced tokens. (The generator
    itself is a transformers-4.31 `GenerationMixin` copy that does not run on the installed 5.x; the forward it calls and
    the expression it yields are exercised here directly.)"""
    from oracle import ar
    cfg, sds, m = small
    sd = sds["autoregressive"]
    torch.manual_seed(21)
    cond = torch.randn(1, cfg.ar_dim)
    codes = torch.randint(0, 8192, (1, 6))
    codes[0, -1] = cfg.stop_mel_token               # the stop token is yielded too

    def reference():
        uv = m["autoregressive"]
        inf = uv.inference_model
        text = torch.tensor(TEXT).unsqueeze(0)
        ids = uv.compute_embeddings(cond, text)      # stores the prompt embeddings, returns the fake input ids
        past = None
        got = []
        for j in range(codes.shape[1]):
            am = torch.ones_like(ids)
            kw = dict(attention_mask=am, use_cache=True, return_dict=True, output_hidden_states=True)
            out = inf(input_ids=ids, **kw) if past is None else inf(input_ids=ids[:, -1:], past_key_values=past, **kw)
            past = out.past_key_values
            got.append(inf.final_norm(out.hidden_states[-1][:, -1])[0])
            ids = torch.cat([ids, codes[:, j:j + 1]], dim=1)
        return torch.stack(got, dim=0)
    with torch.no_grad():
        want = ar.stream_latents(sd, cfg, cond, TEXT, codes[0], pos_mode="ref_kv_quirk")
        got = rg.value("stream_latents_kv", reference)
    assert got.shape == want.shape == (6, cfg.ar_dim)
    assert (got - want).abs().max().item() < 2e-4
    # without the KV cache the reference recomputes the sequence with positions 0..n (autoregressive.py:136-146):
    # the stream latents are then the rows of the teacher-forced latent pass
    with torch.no_grad():
        a = ar.stream_latents(sd, cfg, cond, TEXT, codes[0], pos_mode="train_consistent")
        b = ar.latents(sd, cfg, cond, TEXT, codes)[0]
    assert (a - b).abs().max().item() < 1e-5


def test_handle_chunks_matches_reference():
    """tortoise_tts_b200.api_fast.TextToSpeech.handle_chunks == api_fast.py:277-303 over a whole stream (growing decoder
    outputs, the short last chunk and the repeated flush at the end included)."""
    from tortoise_tts_b200.api_fast import TextToSpeech as Mine

    def reference(lens, ov):
        # the module itself pulls in wav2vec alignment etc.; the method is taken from the reference SOURCE
        import ast
        from oracle.ref_shims import REFERENCE_ROOT
        src = open(os.path.join(REFERENCE_ROOT, "tortoise", "api_fast.py")).read()
        fn = [n for n in ast.walk(ast.parse(src)) if isinstance(n, ast.FunctionDef) and n.name == "handle_chunks"][0]
        ns = {"torch": torch}
        exec(compile(ast.Module(body=[fn], type_ignores=[]), "api_fast.handle_chunks", "exec"), ns)
        ref = ns["handle_chunks"]
        st_r, out = (None, None), []
        for n in lens:
            w = base[:n] * 0.9 + 0.01 * n / 9000.0          # a new tensor per flush, like a decoder output
            cr, pr, orr = ref(None, w.clone(), st_r[0], st_r[1], ov)
            out.append((cr, orr))
            st_r = (pr, orr)
        return out
    torch.manual_seed(5)
    base = torch.randn(9000)
    for case, (lens, ov) in enumerate((((3000, 5200, 5200, 5300), 1024), ((2500, 2600, 9000), 512), ((4000,), 1024))):
        st_m, got = (None, None), []
        for n in lens:
            w = base[:n] * 0.9 + 0.01 * n / 9000.0
            cm, pm, om = Mine.handle_chunks(None, w.clone(), st_m[0], st_m[1], ov)
            got.append((cm, om))
            st_m = (pm, om)
        # every chunk and every kept-back tail (or None) equal to the reference's, bit for bit
        assert rg.hexdigest(got) == rg.digest("handle_chunks_%d" % case, lambda: reference(lens, ov)), (lens, ov)


def test_sampler_matches_hf_processors():
    """oracle.sample_step kept set / probabilities == HF processor chain (RepetitionPenalty ->
    Temperature -> TopK -> TopP) of the installed transformers (form identical to 4.31)."""
    from transformers.generation.logits_process import (RepetitionPenaltyLogitsProcessor, TemperatureLogitsWarper,
                                                        TopKLogitsWarper, TopPLogitsWarper)
    from oracle import ar
    torch.manual_seed(3)
    for trial in range(5):
        logits = torch.randn(1, 8194) * 3
        prev = torch.cat([torch.tensor([[1] * 10 + [8192]]), torch.randint(0, 8192, (1, 20))], dim=1)
        s = RepetitionPenaltyLogitsProcessor(2.0)(prev, logits.clone())
        s = TemperatureLogitsWarper(0.8)(prev, s)
        s = TopKLogitsWarper(50)(prev, s)
        s = TopPLogitsWarper(0.8)(prev, s)
        p = torch.softmax(s, dim=-1)[0]
        tok, kept, kp = ar.sample_step(logits[0], prev[0].tolist(), 0.5)
        ref_kept = (p > 0).nonzero().flatten()
        assert sorted(kept.tolist()) == sorted(ref_kept.tolist())
        assert (p[kept] - kp).abs().max().item() < 1e-6
        assert tok in kept.tolist()


def test_fix_autoregressive_output():
    from oracle import ar

    def reference(c):
        load_reference()
        from tortoise.api import fix_autoregressive_output
        return fix_autoregressive_output(c.clone(), 8193, complain=False)
    for i, row in enumerate(([5, 6, 7, 8193, 8193, 8193, 8193, 8193], [1, 2, 3, 4, 5, 6], [8193, 1, 2, 3],
                             [1, 2, 3, 4, 5, 8193])):
        c = torch.tensor(row)
        want = rg.value("fix_autoregressive_output_%d" % i, lambda: reference(c))
        got = ar.fix_autoregressive_output(c, 8193)
        assert torch.equal(want, got)


def test_ar_latents(small):
    from oracle import ar
    cfg, sds, m = small
    torch.manual_seed(4)
    cond = torch.randn(1, cfg.ar_dim)
    codes = torch.randint(0, 8192, (2, 12))
    text = torch.tensor(TEXT).unsqueeze(0)

    def reference():
        uv = m["autoregressive"]
        return uv(cond.repeat(2, 1), text.repeat(2, 1), torch.tensor([text.shape[-1]]), codes,
                  torch.tensor([codes.shape[-1] * uv.mel_length_compression]), return_latent=True, clip_inputs=False)
    with torch.no_grad():
        want = rg.value("ar_latents", reference)
        got = ar.latents(sds["autoregressive"], cfg, cond, TEXT, codes)
    assert got.shape == want.shape == (2, 12, cfg.ar_dim)
    assert (got - want).abs().max().item() < 2e-4


def test_clvp_scores(small):
    from oracle import clvp
    cfg, sds, m = small
    torch.manual_seed(5)
    codes = torch.randint(0, 8192, (3, 20))
    text = torch.tensor(TEXT)
    with torch.no_grad():
        want = rg.value("clvp_scores", lambda: m["clvp"](text.unsqueeze(0).repeat(3, 1), codes, return_loss=False))
        got = clvp.scores(sds["clvp"], cfg, text, codes)
    assert (got - want).abs().max().item() < 1e-5


def test_cvvp_scores(small):
    """oracle/cvvp.py == CVVP.forward(mel_cond, codes, return_loss=False) accumulated over the conditioning clips as
    api.py:464-468 does (strict=True load of the synthetic cvvp.pth checks the key layout too)."""
    from oracle import cvvp
    cfg, sds, m = small
    torch.manual_seed(15)
    codes = torch.randint(0, 8192, (3, 23))
    auto_conds = torch.randn(1, 2, 80, 131) * 2 - 4           # [1, n_clips, 80, T] as get_conditioning_latents returns

    def reference():
        acc = 0
        for cl in range(auto_conds.shape[1]):
            acc = acc + m["cvvp"](auto_conds[:, cl].repeat(3, 1, 1), codes, return_loss=False)
        return acc / auto_conds.shape[1]
    with torch.no_grad():
        want = rg.value("cvvp_scores", reference)
        got = cvvp.scores(sds["cvvp"], cfg, auto_conds, codes)
    assert (got - want).abs().max().item() < 1e-5


def test_hifigan(small):
    """oracle/hifigan.py == HifiganGenerator.inference(gpt_latents, g=speaker latent) of the api_fast path
    (hifigan_decoder.py:270-294); strict=True load of the synthetic hifidecoder.pth checks the key layout."""
    from oracle import hifigan as oh
    cfg, sds, m = small
    torch.manual_seed(16)
    lat = torch.randn(1, 9, cfg.ar_dim)
    spk = torch.randn(1, cfg.ar_dim)
    with torch.no_grad():
        idx, want, shape = rg.sampled("hifigan", lambda: m["hifigan"].inference(lat, spk))
        got = oh.inference(sds["hifigan"], lat, spk)
    assert got.shape == shape and got.shape[-1] == 256 * int(int(9 * 4) * 24000 / 22050)
    assert (got.reshape(-1)[idx] - want).abs().max().item() < 1e-5
    assert want.abs().max().item() > 0.05          # a meaningful waveform, not a saturated / vanishing one


def test_diffusion_forward_and_loop(small):
    from oracle import diffusion as od
    cfg, sds, m = small
    sd = sds["diffusion"]
    torch.manual_seed(6)
    N = 10
    lat = torch.randn(1, N, cfg.ar_dim)
    cond = torch.randn(1, 2 * cfg.diff_dim)
    S = od.output_seq_len(N)
    with torch.no_grad():
        ce_ref = rg.value("diffusion_code_emb", lambda: m["diffusion"].timestep_independent(lat, cond, S, False))
        ce = od.timestep_independent(sd, cfg, lat, cond, S)
        assert (ce - ce_ref).abs().max().item() < 1e-4
        x = torch.randn(1, 100, S)
        t = torch.tensor([3979])
        for cf in (False, True):
            idx, want, shape = rg.sampled("diffusion_forward_cf%d" % cf, lambda: m["diffusion"](
                x, t, precomputed_aligned_embeddings=ce_ref, conditioning_free=cf))
            got = od.forward(sd, cfg, x, t, code_emb=ce, conditioning_free=cf)
            assert got.shape == shape
            assert (got.reshape(-1)[idx] - want).abs().max().item() < 1e-4

        # full sampling loop with the same torch RNG stream
        iters = 5

        def loop():
            from tortoise.api import load_discrete_vocoder_diffuser, do_spectrogram_diffusion
            diffuser = load_discrete_vocoder_diffuser(desired_diffusion_steps=iters, cond_free=True, cond_free_k=2.0)
            torch.manual_seed(7)
            return do_spectrogram_diffusion(m["diffusion"], diffuser, lat, cond, temperature=1.0, verbose=False)
        want = rg.value("diffusion_loop", loop)
        torch.manual_seed(7)
        noise0 = torch.randn(1, 100, S)
        step_noise = torch.stack([torch.randn(1, 100, S) for _ in range(iters)])
        got = od.spectrogram_diffusion(sd, cfg, lat, cond, noise0, step_noise, iters, True, 2.0)
    assert (got - want).abs().max().item() < 1e-3


def test_schedule_kats():
    """SURVEY App. A3 known-answer values, re-derived from the reference's SpacedDiffusion."""
    from oracle import diffusion as od
    names = ("timestep_map", "betas", "sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod",
             "posterior_log_variance_clipped", "posterior_mean_coef1", "posterior_mean_coef2")

    def reference(iters, name):
        load_reference()
        from tortoise.api import load_discrete_vocoder_diffuser
        d = load_discrete_vocoder_diffuser(desired_diffusion_steps=iters)
        return torch.from_numpy(np.asarray(getattr(d, name), dtype=np.int64 if name == "timestep_map" else np.float64))
    for iters in (30, 80, 200, 400):
        s = od.make_schedule(iters)
        for name in names:
            # bit for bit: the digest covers dtype, shape and every element
            mine = torch.from_numpy(np.asarray(s[name], dtype=np.int64 if name == "timestep_map" else np.float64))
            assert rg.hexdigest(mine) == rg.digest("schedule_%d_%s" % (iters, name), lambda: reference(iters, name)), name
        # the betas are the reference's, bit for bit (above)
        assert np.array_equal(s["log_betas"], np.log(s["betas"]))


def test_vocoder(small):
    from oracle import vocoder as ov
    cfg, sds, m = small
    torch.manual_seed(8)
    mel = torch.randn(1, 100, 12) * 2 - 5
    z = torch.randn(1, 64, 22)
    with torch.no_grad():
        want = rg.value("vocoder", lambda: m["vocoder"].inference(mel, z))
        got = ov.inference(sds["vocoder"], mel, z)
    assert got.shape == want.shape == (1, 1, 256 * 12)
    assert (got - want).abs().max().item() < 1e-4
