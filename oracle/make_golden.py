"""Generate tests/golden/*.pt by running the UNMODIFIED reference modules (authoring container only).

    python -m oracle.make_golden [t3] [s3gen] [variants] [turbo]

The reference ships no golden vectors, known-answer tests or fixtures for this path (SURVEY.md 4,
8c), so the fixtures are outputs of the reference itself: its own `T3.inference`,
`CausalMaskedDiffWithXvec.inference`, `UpsampleConformerEncoder`, `HiFTGenerator.inference` are
imported from /root/reference/src (oracle/ref_harness.py), loaded (strict) with the seeded synthetic
checkpoints of oracle/weights.py, and run on CPU fp32.  The files hold inputs + reference outputs only
(weights are regenerated from the seed).  tests/test_oracle_pinned.py then checks the CPU restatement
in oracle/ against these files on any machine; the GPU parity tests compare the CUDA path to the
restatement and to these same files.
"""
import os
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ref_harness as R, weights as W  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def text_pair(seed, n, vocab_hi=255):
    g = torch.Generator().manual_seed(seed)
    text = torch.randint(1, vocab_hi, (1, n), generator=g)
    text = torch.cat([text, text], 0)                      # CFG pair (tts.py:237-238)
    text = F.pad(text, (1, 0), value=255)                  # SOT (tts.py:242)
    return F.pad(text, (0, 1), value=0)                    # EOT (tts.py:243)


def golden_t3():
    R.install()
    from chatterbox.models.t3.modules.cond_enc import T3Cond
    sd = W.make_t3_weights(0)
    t3 = R.build_t3()
    t3.load_state_dict(sd, strict=True)
    c3, _ = W.make_conds()
    mk = lambda: T3Cond(speaker_emb=c3["speaker_emb"], cond_prompt_speech_tokens=c3["cond_prompt_speech_tokens"],
                        emotion_adv=c3["emotion_adv"])
    out = dict(weights_seed=0, conds_seed=1234)
    cases = []
    for (tseed, ntext, steps, rng_seed, min_p) in [(7, 24, 24, 11, 0.05), (7, 24, 24, 3, 1.0), (8, 61, 12, 5, 1.0)]:
        text = text_pair(tseed, ntext)
        torch.manual_seed(rng_seed)
        toks = t3.inference(t3_cond=mk(), text_tokens=text, max_new_tokens=steps, temperature=0.8, top_p=1.0,
                            min_p=min_p, repetition_penalty=1.2, cfg_weight=0.5)
        # prefill logits of the reference backbone for the same inputs (teacher-forcing anchor)
        embeds, _ = t3.prepare_input_embeds(t3_cond=mk(), text_tokens=text,
                                            speech_tokens=6561 * torch.ones_like(text[:, :1]), cfg_weight=0.5)
        bos = t3.speech_emb(torch.tensor([[6561]])) + t3.speech_pos_emb.get_fixed_embedding(0)
        x = torch.cat([embeds, torch.cat([bos, bos])], dim=1)
        with torch.inference_mode():
            o = t3.patched_model(inputs_embeds=x, past_key_values=None, use_cache=True, output_hidden_states=True,
                                 return_dict=True)
        cases.append(dict(text_seed=tseed, n_text=ntext, steps=steps, rng_seed=rng_seed, min_p=min_p,
                          text_tokens=text, tokens=toks.clone(), prefill_logits=o.logits[:, -1, :].clone(),
                          cond_emb=t3.prepare_conditioning(mk()).clone()))
        print("t3 case", tseed, ntext, steps, min_p, toks[0, :8].tolist())
    out["cases"] = cases
    torch.save(out, os.path.join(OUT, "t3_golden.pt"))


def golden_flow_hift():
    R.install()
    fsd = W.make_flow_weights(0)
    flow = R.build_flow()
    flow.load_state_dict(fsd, strict=True)
    hsd = W.make_hift_weights(0)
    hift = R.build_hift()
    hift.load_state_dict(hsd, strict=True)
    out = dict(weights_seed=0)
    cases = []
    for (np_, n, tok_seed, rng_seed) in [(40, 30, 5, 21), (17, 9, 6, 22)]:
        _, cg = W.make_conds(seed=1234, n_gen_prompt=np_)
        tok = torch.randint(0, 6561, (1, n), generator=torch.Generator().manual_seed(tok_seed))
        x = fsd["input_embedding.weight"][torch.cat([cg["prompt_token"], tok], 1)]
        with torch.inference_mode():
            h, _ = flow.encoder(x, torch.tensor([x.shape[1]]))
            mu = flow.encoder_proj(h)
        torch.manual_seed(rng_seed)
        z = torch.randn(1, 80, 2 * (np_ + n))             # what flow_matching.py:216 will draw
        torch.manual_seed(rng_seed)
        mel, _ = flow.inference(token=tok, token_len=torch.tensor([n]), prompt_token=cg["prompt_token"],
                                prompt_token_len=cg["prompt_token_len"], prompt_feat=cg["prompt_feat"],
                                prompt_feat_len=None, embedding=cg["embedding"], finalize=True, n_timesteps=10)
        # one NFE of the estimator on the CFG pair at t=t_span[1] (unit anchor)
        est = flow.decoder.estimator
        T = mu.shape[1]
        with torch.inference_mode():
            spk = flow.spk_embed_affine_layer(F.normalize(cg["embedding"], dim=1))
            cond = torch.zeros(1, 80, T)
            cond[:, :, :2 * np_] = cg["prompt_feat"].transpose(1, 2)
            t = torch.tensor([0.3])
            v = est(z, torch.ones(1, 1, T), mu.transpose(1, 2).contiguous(), t, spk, cond)
        # HiFT on the reference mel
        torch.manual_seed(rng_seed + 100)
        wav, s = hift.inference(speech_feat=mel)
        cases.append(dict(n_prompt=np_, n=n, tok_seed=tok_seed, rng_seed=rng_seed, tokens=tok, mu=mu.clone(),
                          z=z, mel=mel.clone(), nfe_t=0.3, nfe_v=v.clone(), wav=wav.clone(), source=s.clone()))
        print("flow case", np_, n, mel.shape, float(mel.std()), wav.shape, float(wav.std()))
    out["cases"] = cases
    torch.save(out, os.path.join(OUT, "s3gen_golden.pt"))


def golden_meanflow_and_mtl():
    """Variants (SURVEY.md 8 a14): meanflow 2-step estimator (Turbo's decoder, s3gen.py:313-317, flow_matching.py:235-246)
    and the multilingual T3 (text vocab 2454, t3_config.py:28-41)."""
    R.install()
    from chatterbox.models.t3.modules.cond_enc import T3Cond
    fsd = W.make_flow_weights(0, meanflow=True)
    flow = R.build_flow(meanflow=True)
    flow.load_state_dict(fsd, strict=True)
    out = dict(weights_seed=0)
    np_, n = 30, 21
    _, cg = W.make_conds(seed=1234, n_gen_prompt=np_)
    tok = torch.randint(0, 6561, (1, n), generator=torch.Generator().manual_seed(9))
    torch.manual_seed(77)
    noise = torch.randn(1, 80, 2 * n)                      # s3gen.py:316
    z = torch.randn(1, 80, 2 * (np_ + n))                  # flow_matching.py:216
    z[..., 2 * np_:] = noise                               # flow_matching.py:218-220
    torch.manual_seed(77)
    noise2 = torch.randn(1, 80, 2 * n)
    mel, _ = flow.inference(token=tok, token_len=torch.tensor([n]), prompt_token=cg["prompt_token"],
                            prompt_token_len=cg["prompt_token_len"], prompt_feat=cg["prompt_feat"], prompt_feat_len=None,
                            embedding=cg["embedding"], finalize=True, n_timesteps=2, noised_mels=noise2, meanflow=True)
    out["meanflow"] = dict(n_prompt=np_, n=n, tokens=tok, z=z, mel=mel.clone())
    print("meanflow", mel.shape, float(mel.std()))
    # multilingual T3
    sd = W.make_t3_weights(1, text_vocab=2454)
    t3 = R.build_t3(multilingual=True)
    t3.load_state_dict(sd, strict=True)
    c3, _ = W.make_conds()
    g = torch.Generator().manual_seed(31)
    text = torch.randint(1, 2454, (1, 33), generator=g)
    text[text == 255] = 256
    text = F.pad(F.pad(torch.cat([text, text], 0), (1, 0), value=255), (0, 1), value=0)
    torch.manual_seed(5)
    toks = t3.inference(t3_cond=T3Cond(speaker_emb=c3["speaker_emb"], cond_prompt_speech_tokens=c3["cond_prompt_speech_tokens"],
                                       emotion_adv=c3["emotion_adv"]),
                        text_tokens=text, max_new_tokens=10, temperature=0.8, top_p=1.0, min_p=1.0,
                        repetition_penalty=2.0, cfg_weight=0.5)
    out["mtl"] = dict(weights_seed=1, text_tokens=text, tokens=toks.clone())
    print("mtl", toks.tolist())
    torch.save(out, os.path.join(OUT, "variants_golden.pt"))


TURBO_TEXT_VOCAB = 2048      # fixture-sized gather table (shipped: 50276); see ref_harness.build_t3_turbo


def golden_turbo():
    """Turbo T3 (SURVEY.md 8 a14): the reference's own `T3(hp).inference_turbo` (t3.py:392-468) on the GPT2_medium
    backbone (24 layers), seeded weights, 375-token voice prompt (tts_turbo.py:157)."""
    R.install()
    from chatterbox.models.t3.modules.cond_enc import T3Cond
    sd = W.make_t3_turbo_weights(0, text_vocab=TURBO_TEXT_VOCAB)
    t3 = R.build_t3_turbo(text_vocab=TURBO_TEXT_VOCAB)
    res = t3.load_state_dict(sd, strict=False)
    assert res.missing_keys == ["tfmr.wte.weight"] and not res.unexpected_keys, res   # wte is deleted by the reference
    c3, _ = W.make_conds(seed=1234, n_t3_prompt=375)
    mk = lambda: T3Cond(speaker_emb=c3["speaker_emb"], cond_prompt_speech_tokens=c3["cond_prompt_speech_tokens"],
                        emotion_adv=c3["emotion_adv"])
    out = dict(weights_seed=0, conds_seed=1234, text_vocab=TURBO_TEXT_VOCAB, n_prompt=375)
    cases = []
    for (tseed, ntext, steps, rng_seed, top_k, top_p, rep) in [(21, 19, 16, 11, 1000, 0.95, 1.2), (21, 19, 16, 3, 1, 0.95, 1.2),
                                                               (22, 47, 10, 5, 1, 1.0, 2.0), (23, 30, 12, 9, 50, 0.8, 1.2)]:
        g = torch.Generator().manual_seed(tseed)
        text = torch.randint(0, TURBO_TEXT_VOCAB, (1, ntext), generator=g)
        torch.manual_seed(rng_seed)
        toks = t3.inference_turbo(mk(), text, temperature=0.8, top_k=top_k, top_p=top_p, repetition_penalty=rep,
                                  max_gen_len=steps)
        embeds, len_cond = t3.prepare_input_embeds(t3_cond=mk(), text_tokens=text,
                                                   speech_tokens=6561 * torch.ones_like(text[:, :1]), cfg_weight=0.0)
        with torch.inference_mode():
            hs = t3.tfmr(inputs_embeds=embeds, use_cache=True)[0]
            pl = t3.speech_head(hs[:, -1:])[:, -1, :]
        cases.append(dict(text_seed=tseed, n_text=ntext, steps=steps, rng_seed=rng_seed, top_k=top_k, top_p=top_p,
                          rep=rep, text_tokens=text, tokens=toks.clone(), prefill_logits=pl.clone(), len_cond=len_cond,
                          cond_emb_head=t3.prepare_conditioning(mk())[:, :4].clone()))   # [spkr | first prompt rows]
        print("turbo case", tseed, ntext, steps, top_k, top_p, toks[0, :8].tolist(), toks.shape)
    out["cases"] = cases
    torch.save(out, os.path.join(OUT, "turbo_golden.pt"))


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(min(16, len(os.sched_getaffinity(0))))
    which = [a for a in sys.argv[1:] if not a.startswith("long_")] or ([] if sys.argv[1:] else ["t3", "s3gen", "variants", "turbo"])
    if "t3" in which:
        golden_t3()
    if "s3gen" in which:
        golden_flow_hift()
    if "variants" in which:
        golden_meanflow_and_mtl()
    if "turbo" in which:
        golden_turbo()


# ------------------------------------------------------------------------------------------------------------------
# Round 2: fixtures at the benchmarked configuration (context >= 1000 tokens, CFM T >= 2000 frames).
#   python -m oracle.make_golden long_t3 long_flow
# ------------------------------------------------------------------------------------------------------------------
LONG_T3_STEPS = 900
LONG_T3_TAPS = (1, 64, 256, 512, 768, 900)      # logits kept after consuming this many generated tokens


def golden_t3_long():
    """The reference's own T3.inference for 900 greedy steps on a 150-token text (context 188 -> 1088 tokens, the
    bench regime), then a teacher-forced pass of the reference backbone (`t3.patched_model`, DynamicCache) over the
    reference's ids that keeps the logits of both CFG rows at LONG_T3_TAPS."""
    R.install()
    from chatterbox.models.t3.modules.cond_enc import T3Cond
    sd = W.make_t3_weights(0)
    t3 = R.build_t3()
    t3.load_state_dict(sd, strict=True)
    c3, _ = W.make_conds()
    mk = lambda: T3Cond(speaker_emb=c3["speaker_emb"], cond_prompt_speech_tokens=c3["cond_prompt_speech_tokens"],
                        emotion_adv=c3["emotion_adv"])
    text = text_pair(41, 150)
    torch.manual_seed(17)
    toks = t3.inference(t3_cond=mk(), text_tokens=text, max_new_tokens=LONG_T3_STEPS, temperature=0.8, top_p=1.0,
                        min_p=1.0, repetition_penalty=1.2, cfg_weight=0.5)
    ids = toks[0]
    print("t3 long: generated", ids.numel(), "ids, eos" if (ids == 6562).any() else "no eos", ids[:8].tolist())
    # teacher-forced pass: same call sequence as t3.py:320-386 (prefill with both BOS embeddings, then one token per step)
    embeds, _ = t3.prepare_input_embeds(t3_cond=mk(), text_tokens=text,
                                        speech_tokens=6561 * torch.ones_like(text[:, :1]), cfg_weight=0.5)
    bos = t3.speech_emb(torch.tensor([[6561]])) + t3.speech_pos_emb.get_fixed_embedding(0)
    x = torch.cat([embeds, torch.cat([bos, bos])], dim=1)
    taps = {}
    with torch.inference_mode():
        o = t3.patched_model(inputs_embeds=x, past_key_values=None, use_cache=True, output_hidden_states=True,
                             return_dict=True)
        past = o.past_key_values
        for i in range(ids.numel()):
            e = t3.speech_emb(ids[i].view(1, 1)) + t3.speech_pos_emb.get_fixed_embedding(i + 1)
            e = torch.cat([e, e])
            o = t3.patched_model(inputs_embeds=e, past_key_values=past, output_hidden_states=True, return_dict=True)
            past = o.past_key_values
            if (i + 1) in LONG_T3_TAPS:
                taps[i + 1] = o.logits[:, -1, :].clone()
                print("  tap", i + 1, float(taps[i + 1].abs().max()))
    torch.save(dict(weights_seed=0, conds_seed=1234, text_tokens=text, tokens=toks.clone(), taps=taps,
                    s0=int(x.shape[1])), os.path.join(OUT, "t3_long_golden.pt"))


def golden_flow_long():
    """CausalMaskedDiffWithXvec.inference at T = 2(250 + 770) = 2040 mel frames (the bench's long-utterance regime: 32
    query tiles / 32 key blocks per head in the tcgen05 attention)."""
    R.install()
    fsd = W.make_flow_weights(0)
    flow = R.build_flow()
    flow.load_state_dict(fsd, strict=True)
    np_, n, tok_seed, rng_seed = 250, 770, 15, 31
    _, cg = W.make_conds(seed=1234, n_gen_prompt=np_)
    tok = torch.randint(0, 6561, (1, n), generator=torch.Generator().manual_seed(tok_seed))
    x = fsd["input_embedding.weight"][torch.cat([cg["prompt_token"], tok], 1)]
    with torch.inference_mode():
        h, _ = flow.encoder(x, torch.tensor([x.shape[1]]))
        mu = flow.encoder_proj(h)
    torch.manual_seed(rng_seed)
    z = torch.randn(1, 80, 2 * (np_ + n))
    torch.manual_seed(rng_seed)
    mel, _ = flow.inference(token=tok, token_len=torch.tensor([n]), prompt_token=cg["prompt_token"],
                            prompt_token_len=cg["prompt_token_len"], prompt_feat=cg["prompt_feat"],
                            prompt_feat_len=None, embedding=cg["embedding"], finalize=True, n_timesteps=10)
    print("flow long", mel.shape, float(mel.std()))
    torch.save(dict(weights_seed=0, n_prompt=np_, n=n, tok_seed=tok_seed, rng_seed=rng_seed, tokens=tok,
                    mu_sample=mu[:, ::16].clone(), mel=mel.clone(),
                    # z is re-drawn from rng_seed by the test (torch CPU randn is reproducible); checksum to be sure
                    z_head=z[..., :8].clone(), z_sum=float(z.double().sum())),
               os.path.join(OUT, "flow_long_golden.pt"))


if __name__ == "__main__" and any(a.startswith("long_") for a in sys.argv[1:]):
    if "long_t3" in sys.argv[1:]:
        golden_t3_long()
    if "long_flow" in sys.argv[1:]:
        golden_flow_long()
