"""GPU (-m gpu): the CUDA path through the C ABI vs the CPU oracle on identical seeded inputs.

Tolerances (stated, SURVEY 8d): bf16 kernels vs the fp32 oracle on bf16-representable weights:
  rel-Frobenius <= 2e-2, and no worse than 1.5x the error of the same oracle run in torch-bf16 (floor 5e-3);
greedy token ids exact wherever the oracle's top-1/top-2 margin exceeds 2x the max logit error;
integer / index logic (splice plan, token rows) bit-exact."""
import os

import pytest
import torch

import helpers as Hh
from oracle import valley_oracle as O
from valley_b200 import _lib, synthetic as syn

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
_models = {}


def get(spec_name, seed=0):
    key = (spec_name, seed)
    if key not in _models:
        spec = syn.SPECS[spec_name]
        sd = Hh.bf16_weights(spec, seed)
        _models[key] = (spec, sd, Hh.build_model(spec, sd))
    return _models[key]


def bf16_sd(sd):
    return {k: v.bfloat16() for k, v in sd.items()}


def check_close(got, ref_fp32, ref_bf16=None, what=""):
    e = Hh.rel_fro(got, ref_fp32)
    assert not torch.isnan(got.float()).any(), what
    assert e <= 2e-2, (what, e)
    if ref_bf16 is not None:
        eb = Hh.rel_fro(ref_bf16, ref_fp32)
        assert e <= max(1.5 * eb, 5e-3), (what, e, eb)
    return e


@pytest.mark.parametrize("M,N,K,bn", [(128, 128, 64, 128), (300, 512, 256, 256), (1000, 1024, 640, 256), (77, 1032, 512, 128),
                                      (1, 256, 64, 256), (2056, 1024, 4096, 256)])
def test_gemm_bias_and_residual(M, N, K, bn):
    _, _, m = get("tiny")
    a = (torch.randn(M, K, device="cuda") * 0.5).bfloat16()
    w = (torch.randn(N, K, device="cuda") * 0.05).bfloat16()
    bias = torch.randn(N, device="cuda")
    out = torch.zeros(M, N, device="cuda", dtype=torch.bfloat16)
    _lib.check(m._lib.vly_test_gemm(m._ctx, a.data_ptr(), w.data_ptr(), M, N, K, 0, bias.data_ptr(), None, out.data_ptr(), bn, 0))
    ref = a.float() @ w.float().T + bias
    assert Hh.rel_fro(out, ref) < 4e-3
    if N % 32 == 0:
        res = torch.randn(M, N, device="cuda").bfloat16()
        out2 = res.clone()
        _lib.check(m._lib.vly_test_gemm(m._ctx, a.data_ptr(), w.data_ptr(), M, N, K, 3, bias.data_ptr(), out2.data_ptr(), out2.data_ptr(), bn, 0))
        assert Hh.rel_fro(out2, ref + res.float()) < 4e-3


@pytest.mark.parametrize("F", [1, 2, 37])
def test_vit_attention_kernel(F):
    _, _, m = get("tiny")
    qkv = torch.randn(F * 257, 3072, device="cuda").bfloat16()
    out = torch.zeros(F * 257, 1024, device="cuda", dtype=torch.bfloat16)
    _lib.check(m._lib.vly_test_vit_attention(m._ctx, qkv.data_ptr(), F, out.data_ptr(), 0))
    x = qkv.float().view(F, 257, 3, 16, 64)
    q, k, v = (x[:, :, i].transpose(1, 2) for i in range(3))
    ref = (torch.softmax(q @ k.transpose(-1, -2) * 0.125, -1) @ v).transpose(1, 2).reshape(F * 257, 1024)
    assert Hh.rel_fro(out, ref) < 6e-3


@pytest.mark.parametrize("spec_name,F,sel", [("tiny", 1, -2), ("tiny", 5, -1), ("tiny", 3, 0), ("tiny-wide", 8, -2)])
def test_vit_encode_vs_oracle(spec_name, F, sel):
    spec, sd, m = get(spec_name, 1 if spec_name == "tiny-wide" else 0)
    px = syn.make_pixels(1, F, 3)[0]
    got = m._vit_encode(px.cuda(), sel)
    with torch.no_grad():
        ref = O.vit_hidden_state(sd, px, sel, num_layers=spec.vit_layers)
        ref_bf = O.vit_hidden_state(bf16_sd(sd), px.bfloat16(), sel, num_layers=spec.vit_layers)
    check_close(got, ref, ref_bf, f"vit[{sel}]")
    # pixel dtype variants the callers send (fp16: valley_model.py:430)
    got16 = m._vit_encode(px.half().cuda(), sel)
    assert Hh.rel_fro(got16, got) < 1e-2


def test_vit_frames_are_independent_and_chunking_is_invisible():
    spec, sd, m = get("tiny")
    px = syn.make_pixels(1, 7, 9)[0].cuda()
    full = m.encode_frames(px)
    parts = torch.cat([m.encode_frames(px[:3]), m.encode_frames(px[3:])])
    assert torch.equal(full, parts)                      # same kernels, same tiles per frame -> bit-identical


def test_vit_rejects_wrong_image_size():
    _, _, m = get("tiny")
    with pytest.raises(ValueError):
        m.encode_frames(torch.zeros(1, 3, 196, 196, device="cuda"))


def test_encode_images_and_splice_vs_oracle():
    spec, sd, m = get("tiny")
    cfg, tok = Hh.oracle_cfg(spec), Hh.oracle_tok(spec)
    B, T = 2, 3
    ids, px = syn.make_prompt_ids(spec, B, T, 0), syn.make_pixels(B, T, 0)
    with torch.no_grad():
        ref_enc = O.encode_images(sd, px, cfg.mm_vision_select_layer, num_layers=cfg.vit_layers)
        ref_emb = O.prepare_inputs_embeds(sd, ids, ref_enc, tok)
    enc = m.encode_images(px.cuda())
    assert enc.shape == ref_enc.shape
    check_close(enc, ref_enc, None, "encode_images")
    r = m.prepare_inputs_labels_for_multimodal(ids.cuda(), None, None, None, px.cuda())
    assert r[0] is None and r[3].shape == ref_emb.shape
    check_close(r[3], ref_emb, None, "inputs_embeds")
    text = ids[0] < spec.vocab_size - 6
    assert torch.equal(r[3][0][text.cuda()].float().cpu(), ref_emb[0][text])     # gathered token rows: bit-exact
    # list-of-tensors input with different T per sample (valley_model.py:168-176)
    lst = [px[0, :2].cuda(), px[1].cuda()]
    ids2 = torch.stack([syn.make_prompt_ids(spec, 1, 3, 0)[0], syn.make_prompt_ids(spec, 1, 3, 1)[0]])
    ids2[0] = syn.make_prompt_ids(spec, 1, 3, 0)[0]
    r2 = m.prepare_inputs_labels_for_multimodal(ids2[1:].cuda(), None, None, None, [lst[1]])
    with torch.no_grad():
        e1 = O.prepare_inputs_embeds(sd, ids2[1:], O.encode_images(sd, [px[1]], cfg.mm_vision_select_layer, num_layers=cfg.vit_layers), tok)
    check_close(r2[3], e1, None, "list input")


def test_splice_golden_cases_and_errors_through_the_model():
    spec, sd, m = get("tiny")
    g = torch.load(os.path.join(GOLD, "ref_tiny.pt"))
    px = syn.make_pixels(g["B"], g["T"], g["seed"])
    fp32_sd = syn.make_state_dict(spec, g["seed"])
    for case, d in torch.load(os.path.join(GOLD, "ref_tiny_splice.pt")).items():
        if isinstance(d["n_frames"], list):          # images as a list of clips with different frame counts (valley_model.py:168-176)
            cpx = [px[i, :n].cuda() for i, n in enumerate(d["n_frames"])]
        else:
            cpx = px[:1, : d["n_frames"]].cuda()
        emb = m.prepare_inputs_labels_for_multimodal(d["ids"].cuda(), None, None, None, cpx)[3]
        ref = d["embeds_sub"]                       # the REFERENCE's own inputs_embeds (fp32 weights), sub-sampled
        assert Hh.rel_fro(emb[:, :, ::8], ref) < 2e-2, case
    for case, d in g["errors"].items():
        with pytest.raises(ValueError) as ei:
            m(input_ids=d["ids"].cuda(), images=px[:1].cuda())
        assert str(ei.value) == d["message"], case


@pytest.mark.parametrize("spec_name,B,T", [("tiny", 2, 3), ("tiny-wide", 1, 8), ("tiny", 5, 1)])
def test_prefill_logits_vs_oracle(spec_name, B, T):
    spec, sd, m = get(spec_name, 1 if spec_name == "tiny-wide" else 0)
    cfg, tok = Hh.oracle_cfg(spec), Hh.oracle_tok(spec)
    ids, px = syn.make_prompt_ids(spec, B, T, 0), syn.make_pixels(B, T, 0)
    with torch.no_grad():
        ref = O.causal_lm_forward(sd, cfg, tok, ids, px, None)
        ref_bf = O.causal_lm_forward(bf16_sd(sd), cfg, tok, ids, px.bfloat16(), None).float()
    out = m(input_ids=ids.cuda(), images=px.cuda())
    assert out.logits.shape == ref.shape and out.past_key_values.get_seq_length() == ids.shape[1]
    assert out.past_key_values[0][0].shape[-2] == ids.shape[1]            # model_worker.py:253 access pattern
    err = check_close(out.logits, ref, ref_bf, "prefill logits")
    # argmax must agree wherever the oracle's margin exceeds 2x the max logit error
    max_err = (out.logits.cpu() - ref).abs().max().item()
    top2 = ref.topk(2, -1).values
    safe = (top2[..., 0] - top2[..., 1]) > 2 * max_err
    assert safe.float().mean() > 0.5
    assert torch.equal(out.logits.argmax(-1).cpu()[safe], ref.argmax(-1)[safe])
    # KV cache contents (layer 0) vs the oracle's cache
    cache = O.KVCache(spec.num_hidden_layers)
    with torch.no_grad():
        O.causal_lm_forward(sd, cfg, tok, ids, px, cache)
    k, v = out.past_key_values.to_hf(0)
    assert Hh.rel_fro(k, cache.k[0]) < 2e-2 and Hh.rel_fro(v, cache.v[0]) < 2e-2


def test_golden_reference_logits_and_tokens():
    """Against the committed outputs of the reference itself (fp32 weights there, bf16 here)."""
    for name in ("tiny", "tiny-wide"):
        g = torch.load(os.path.join(GOLD, f"ref_{name}.pt"))
        spec, sd, m = get(name, g["seed"])
        ids, px = syn.make_prompt_ids(spec, g["B"], g["T"], g["seed"]), syn.make_pixels(g["B"], g["T"], g["seed"])
        out = m(input_ids=ids.cuda(), images=px.cuda())
        assert Hh.rel_fro(out.logits[:, -1], g["prefill_logits_last"]) < 2e-2
        n = g["greedy_tokens"].shape[1]
        gen = m.generate(input_ids=ids.cuda(), images=px.cuda(), max_new_tokens=n)[:, ids.shape[1]:].cpu()
        top2 = g["greedy_logits"].topk(2, -1).values
        margin = top2[..., 0] - top2[..., 1]
        for b in range(g["B"]):
            for i in range(n):
                if gen[b, i] != g["greedy_tokens"][b, i]:
                    assert margin[b, i] < 0.05, (name, b, i, margin[b, i].item())     # only near-ties may differ
                    break


@pytest.mark.parametrize("spec_name,B", [("tiny", 2), ("tiny", 1), ("tiny-wide", 1), ("tiny", 6)])
def test_greedy_decode_vs_oracle(spec_name, B):
    spec, sd, m = get(spec_name, 1 if spec_name == "tiny-wide" else 0)
    cfg, tok = Hh.oracle_cfg(spec), Hh.oracle_tok(spec)
    T, n = 3, 10
    ids, px = syn.make_prompt_ids(spec, B, T, 0), syn.make_pixels(B, T, 0)
    with torch.no_grad():
        r_tok, r_log = O.greedy_generate(sd, cfg, tok, ids, px, n, return_logits=True)
    # teacher-forced through forward(past_key_values=...) exactly like model_worker.py:380-391
    out = m(input_ids=ids.cuda(), images=px.cuda())
    cache, logs = out.past_key_values, [out.logits[:, -1].cpu()]
    for i in range(1, n):
        o = m(input_ids=r_tok[:, i - 1:i].cuda(), past_key_values=cache,
              attention_mask=torch.ones(B, cache[0][0].shape[-2] + 1, device="cuda"))
        logs.append(o.logits[:, -1].cpu())
        assert cache.get_seq_length() == ids.shape[1] + i
    logs = torch.stack(logs, 1)
    max_err = (logs - r_log).abs().max().item()
    assert Hh.rel_fro(logs, r_log) < 2e-2
    top2 = r_log.topk(2, -1).values
    safe = (top2[..., 0] - top2[..., 1]) > 2 * max_err
    assert torch.equal(logs.argmax(-1)[safe], r_tok[safe])
    # free-running device-side loop (CUDA graph): identical until the first unsafe (near-tie) position
    gen = m.generate(input_ids=ids.cuda(), images=px.cuda(), max_new_tokens=n)[:, ids.shape[1]:].cpu()
    for b in range(B):
        for i in range(n):
            if not safe[b, i]:
                break
            assert gen[b, i] == r_tok[b, i], (b, i)
    # determinism: the same request twice gives the same ids
    gen2 = m.generate(input_ids=ids.cuda(), images=px.cuda(), max_new_tokens=n)[:, ids.shape[1]:].cpu()
    assert torch.equal(gen, gen2)


def test_generate_host_loop_equals_device_loop_and_stops():
    spec, sd, m = get("tiny")
    ids, px = syn.make_prompt_ids(spec, 1, 2, 4), syn.make_pixels(1, 2, 4)
    a = m.generate(input_ids=ids.cuda(), images=px.cuda(), max_new_tokens=9)
    stop_after = lambda seq, scores: seq.shape[1] >= ids.shape[1] + 5
    b = m.generate(input_ids=ids.cuda(), images=px.cuda(), max_new_tokens=9, stopping_criteria=[stop_after])
    assert b.shape[1] == ids.shape[1] + 5 and torch.equal(a[:, : b.shape[1]], b)
    c = m.generate(input_ids=ids.cuda(), images=px.cuda(), max_new_tokens=4, do_sample=True, temperature=0.7)
    assert c.shape[1] == ids.shape[1] + 4 and int(c.max()) < spec.vocab_size
    inp = m.prepare_inputs_for_generation(a, past_key_values=None, images=px)
    assert inp["input_ids"].shape == a.shape and inp["images"] is px


@pytest.mark.parametrize("B,pads", [(2, (5, 0)), (1, (3,)), (3, (0, 130, 64)), (6, (0, 130, 1, 64, 7, 0))])
def test_left_padded_batch_vs_oracle(B, pads):
    """attention_mask with LEFT padding (build_inputs / tokenizer(padding=True), valley_model.py:402-403): padded keys are never
    attended, positions are not shifted.  Pads of 64 / 130 mask whole 64-key decode splits and a whole 128-key prefill tile.
    B = 1, 2, 3 run the persistent decode kernel (CUDA-core and tensor-core consumers), B = 6 the grouped per-op kernels."""
    spec, sd, m = get("tiny")
    cfg, tok = Hh.oracle_cfg(spec), Hh.oracle_tok(spec)
    T, n, P = 3, 6, max(pads)
    base, px = syn.make_prompt_ids(spec, B, T, 0), syn.make_pixels(B, T, 0)
    fill = torch.randint(3, spec.vocab_size - 8, (B, P), generator=torch.Generator().manual_seed(3))
    ids, am = torch.cat([fill, base], 1), torch.ones(B, P + base.shape[1], dtype=torch.int64)
    for b, p in enumerate(pads):
        ids[b, :p] = 0
        am[b, :p] = 0
    with torch.no_grad():
        r_tok, r_log = O.greedy_generate(sd, cfg, tok, ids, px, n, return_logits=True, attention_mask=am)
        u_log = O.causal_lm_forward(sd, cfg, tok, ids, px, None)[:, -1]      # the same batch with the mask ignored
    out = m(input_ids=ids.cuda(), attention_mask=am.cuda(), images=px.cuda())      # logits at every position
    assert torch.isfinite(out.logits).all()                     # fully masked (padding) query rows stay finite
    cache, logs, mask = out.past_key_values, [out.logits[:, -1].cpu()], am
    for b, p in enumerate(pads):     # every padded row must sit clearly on the masked side (a short pad moves logits by only ~1e-2)
        if p >= 3:                   # (a single masked key moves them by less than the bf16 noise)
            assert Hh.rel_fro(logs[0][b], r_log[b, 0]) < 0.5 * Hh.rel_fro(logs[0][b], u_log[b]), (b, p)
    for i in range(1, n):
        mask = torch.cat([mask, torch.ones(B, 1, dtype=mask.dtype)], 1)
        o = m(input_ids=r_tok[:, i - 1:i].cuda(), past_key_values=cache, attention_mask=mask)     # CPU mask on purpose
        logs.append(o.logits[:, -1].cpu())
    logs = torch.stack(logs, 1)
    max_err = (logs - r_log).abs().max().item()
    assert Hh.rel_fro(logs, r_log) < 2e-2, Hh.rel_fro(logs, r_log)
    top2 = r_log.topk(2, -1).values
    safe = (top2[..., 0] - top2[..., 1]) > 2 * max_err
    assert torch.equal(logs.argmax(-1)[safe], r_tok[safe])
    gen = m.generate(input_ids=ids.cuda(), images=px.cuda(), max_new_tokens=n, attention_mask=am.cuda())[:, ids.shape[1]:].cpu()
    for b in range(B):
        for i in range(n):
            if not safe[b, i]:
                break
            assert gen[b, i] == r_tok[b, i], (b, i)
    # a recycled cache must not remember the mask: the same unpadded request before and after gives the same ids
    plain = m.generate(input_ids=base.cuda(), images=px.cuda(), max_new_tokens=n)
    fresh = m._generate_with_cache(m.new_cache(B), base, m.prepare_inputs_labels_for_multimodal(base, None, None, None, px)[3],
                                   n, False, 1.0, None, None)
    assert torch.equal(plain, fresh)
    with pytest.raises(ValueError):
        m(input_ids=ids.cuda(), attention_mask=am[:, :-1].cuda(), images=px.cuda())


def test_left_padded_golden_reference_logits():
    """The REFERENCE's own fp32 outputs for a left-padded batch (tests/golden, oracle/make_golden.py)."""
    g = torch.load(os.path.join(GOLD, "ref_tiny.pt"))
    lp = g["leftpad"]
    spec = syn.SPECS["tiny"]
    sd = syn.make_state_dict(spec, g["seed"])
    m = Hh.build_model(spec, sd)
    px = syn.make_pixels(g["B"], g["T"], g["seed"])
    out = m(input_ids=lp["ids"].cuda(), attention_mask=lp["mask"].cuda(), images=px.cuda())
    assert Hh.rel_fro(out.logits[:, -1], lp["prefill_logits_last"]) < 2e-2
    cache, cur, mask = out.past_key_values, lp["first_token"], lp["mask"]
    for i in range(lp["decode_logits"].shape[1]):
        mask = torch.cat([mask, torch.ones(mask.shape[0], 1, dtype=mask.dtype)], 1)
        o = m(input_ids=cur.cuda(), past_key_values=cache, attention_mask=mask.cuda())
        assert Hh.rel_fro(o.logits[:, -1], lp["decode_logits"][:, i]) < 2e-2
        cur = lp["decode_logits"][:, i].argmax(-1)[:, None]


def _sample_direct(m, cache, logits, temperature, seed, eos=-1, pad=0):
    from valley_b200._lib import VlySampling, check
    import ctypes as C
    sp = VlySampling(float(temperature), int(seed), int(eos), int(pad))
    out = torch.empty(cache.batch, dtype=torch.int64, device="cuda")
    lg = logits.reshape(cache.batch, -1).float().contiguous()
    check(m._lib.vly_sample_logits(m._ctx, cache._h, lg.data_ptr(), C.byref(sp), out.data_ptr(), None))
    return out


def test_device_sampler_draws_softmax_of_logits_over_temperature():
    """model_worker.py:392-395: probs = softmax(logits / T); token = multinomial(probs).  The device draws it by Gumbel-max over
    Philox noise: goodness of fit of 6000 draws (one seed each) against the oracle's softmax, determinism per seed, and the
    temperature -> 0 limit (arg-max, :390-391)."""
    from scipy import stats
    spec, sd, m = get("tiny")
    V, T, N = spec.vocab_size, 0.7, 6000
    cache = m.new_cache(1, 128)
    logits = (torch.randn(1, V, generator=torch.Generator().manual_seed(11)) * 1.5).cuda()
    probs = torch.softmax(logits[0].double().cpu() / T, -1)
    draws = torch.stack([_sample_direct(m, cache, logits, T, 1000 + i) for i in range(N)]).cpu().reshape(-1)
    assert int(draws.min()) >= 0 and int(draws.max()) < V
    counts = torch.bincount(draws, minlength=V).double()
    big = probs * N >= 10                         # individual cells for likely tokens, one pooled cell for the tail
    obs = torch.cat([counts[big], counts[~big].sum()[None]])
    exp = torch.cat([probs[big] * N, (probs[~big].sum() * N)[None]])
    chi2 = float(((obs - exp) ** 2 / exp).sum())
    assert chi2 < stats.chi2.ppf(1 - 1e-6, df=len(obs) - 1), (chi2, len(obs))
    assert len(obs) > 50 and counts.max() < 0.5 * N          # a real spread, not one token
    a, b = _sample_direct(m, cache, logits, T, 77), _sample_direct(m, cache, logits, T, 77)
    assert torch.equal(a, b)
    assert int(_sample_direct(m, cache, logits, 1e-5, 5)) == int(logits.argmax())
    # a sharper temperature concentrates mass on the arg-max
    cold = torch.stack([_sample_direct(m, cache, logits, 0.05, 9000 + i) for i in range(200)]).cpu().reshape(-1)
    p_cold = torch.softmax(logits[0].double().cpu() / 0.05, -1)
    assert abs(float((cold == int(logits.argmax())).double().mean()) - float(p_cold.max())) < 0.15


@pytest.mark.parametrize("B", [1, 2, 6])
def test_fused_sampling_equals_standalone_selection_on_the_same_logits(B):
    """generate(do_sample=True) selects inside the decode step (persistent kernel epilogue for B <= 4, post-step kernel for the
    per-op path).  Teacher-forcing the drawn ids through forward() and selecting from each step's logits with the stand-alone
    kernel under the same (seed, row, position) counter must give the same ids: the fused path is the same distribution."""
    spec, sd, m = get("tiny")
    n, T = 7, 0.8
    ids, px = syn.make_prompt_ids(spec, B, 2, 5), syn.make_pixels(B, 2, 5)
    torch.manual_seed(4242)
    gen = m.generate(input_ids=ids.cuda(), images=px.cuda(), max_new_tokens=n, do_sample=True, temperature=T)[:, ids.shape[1]:]
    assert gen.shape == (B, n)
    torch.manual_seed(4242)
    seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    out = m(input_ids=ids.cuda(), images=px.cuda())
    cache, toks = out.past_key_values, []
    toks.append(_sample_direct(m, cache, out.logits[:, -1], T, seed))
    for i in range(1, n):
        o = m(input_ids=toks[-1][:, None], past_key_values=cache)
        toks.append(_sample_direct(m, cache, o.logits[:, -1], T, seed))
    assert torch.equal(torch.stack(toks, 1), gen)
    greedy = m.generate(input_ids=ids.cuda(), images=px.cuda(), max_new_tokens=n)[:, ids.shape[1]:]
    assert not torch.equal(greedy, gen)                      # T = 0.8 on ~flat random-init logits: not the arg-max path
    torch.manual_seed(4243)
    other = m.generate(input_ids=ids.cuda(), images=px.cuda(), max_new_tokens=n, do_sample=True, temperature=T)[:, ids.shape[1]:]
    assert not torch.equal(other, gen)                       # another seed, another draw


@pytest.mark.parametrize("B", [1, 2, 5])
def test_eos_stops_on_the_device_like_hf_generate(B):
    """model_worker.py:396-397 / HF generate: a row that emits eos is finished, finished rows are padded, generation ends when
    every row is finished.  Expected ids are derived from the free-running greedy ids (rows are independent)."""
    spec, sd, m = get("tiny")
    n, PAD = 9, 7
    ids, px = syn.make_prompt_ids(spec, B, 2, 6), syn.make_pixels(B, 2, 6)
    S = ids.shape[1]
    g = m.generate(input_ids=ids.cuda(), images=px.cuda(), max_new_tokens=n)[:, S:].cpu()
    i0 = next(i for i in range(2, n) if g[0, i] not in g[0, :i])
    eos = int(g[0, i0])
    exp, stop = g.clone(), []
    for b in range(B):
        hit = (g[b] == eos).nonzero()
        k = int(hit[0]) if len(hit) else n - 1
        exp[b, k + 1:] = PAD
        stop.append(k if len(hit) else n - 1)
    n_valid = max(stop) + 1
    got = m.generate(input_ids=ids.cuda(), images=px.cuda(), max_new_tokens=n, eos_token_id=eos, pad_token_id=PAD)
    assert got.shape[1] == S + n_valid, (got.shape, n_valid)
    assert torch.equal(got[:, S:].cpu(), exp[:, :n_valid])
    if B == 1:      # the host-visible loop (stopping criteria present) ends at the same place
        never = lambda seq, scores: False
        host = m.generate(input_ids=ids.cuda(), images=px.cuda(), max_new_tokens=n, eos_token_id=eos, stopping_criteria=[never])
        assert torch.equal(host, got)
    # the recycled cache is clean again: same greedy ids as before
    g2 = m.generate(input_ids=ids.cuda(), images=px.cuda(), max_new_tokens=n)[:, S:].cpu()
    assert torch.equal(g, g2)
    # and a cache used directly reports the true length after an early stop
    if B <= 4:      # (the per-op path of larger batches keeps stepping with pad tokens instead of skipping the steps)
        cache = m.new_cache(B)
        emb = m.prepare_inputs_labels_for_multimodal(ids, None, None, None, px)[3]
        full = m._generate_with_cache(cache, ids, emb, n, False, 1.0, None, eos, PAD)
        assert cache.get_seq_length() == S + (full.shape[1] - S) - 1


@pytest.mark.parametrize("h,w", [(360, 640), (640, 360), (256, 340), (300, 256), (200, 150), (224, 224), (720, 1280), (255, 257), (481, 853)])
def test_frame_preprocessing_is_bit_exact(h, w):
    """vly_preprocess_frames vs the oracle (same clip) and vs the REFERENCE's own output (tests/golden/ref_preprocess.pt, written
    by running valley/data/video_transform.py): integer stage and fp32 output bit for bit; fp16 / bf16 = RN of the fp32 result."""
    import hashlib
    import numpy as np
    from oracle import preprocess_oracle as P
    from valley_b200 import video
    from test_oracle_golden import _clip
    spec, sd, m = get("tiny")
    g = torch.load(os.path.join(GOLD, "ref_preprocess.pt"))[(h, w)]
    clip = _clip(h, w, g["seed"])
    ref = P.preprocess_frames(clip)
    out = video.preprocess_frames(m, torch.from_numpy(clip), torch.float32).cpu().numpy()
    assert np.array_equal(out.view(np.uint32), ref.view(np.uint32))
    assert hashlib.sha256(np.ascontiguousarray(out).tobytes()).hexdigest() == g["sha_f32"]
    for dt in (torch.float16, torch.bfloat16):
        lo = video.preprocess_frames(m, torch.from_numpy(clip).cuda(), dt).cpu()
        assert torch.equal(lo, torch.from_numpy(ref).to(dt))
    # T = 5 frames, device-resident input, through the reader-style entry point
    class Reader:
        def __init__(self, frames): self.f = frames
        def __len__(self): return len(self.f)
        def get_batch(self, idx): return torch.from_numpy(self.f[np.asarray(idx)])
        def get_avg_fps(self): return 2.2
    many = np.concatenate([clip] * 6)[:11]
    got = video.load_video(m, Reader(many), "fixed", 5, dtype=torch.float32).cpu().numpy()
    assert np.array_equal(got, P.preprocess_frames(many[P.fixed_frame_indices(11, 5)]))
    got = video.load_video(m, Reader(many), "fps", fps_number=0.5, dtype=torch.float32).cpu().numpy()
    assert np.array_equal(got, P.preprocess_frames(many[P.fps_frame_indices(11, 2.2, 0.5)]))


def test_preprocessed_frames_feed_the_vision_tower():
    """uint8 frames -> preprocess -> encode_images == oracle preprocessing -> oracle ViT (same tolerance as the ViT test)."""
    import numpy as np
    from oracle import preprocess_oracle as P
    from valley_b200 import video
    from test_oracle_golden import _clip
    spec, sd, m = get("tiny")
    clip = np.concatenate([_clip(360, 640, 3), _clip(360, 640, 4)])[:3]
    px = video.preprocess_frames(m, torch.from_numpy(clip), torch.float16)
    got = m.get_model().vision_tower(px).selected_hidden_state
    with torch.no_grad():
        want = O.vit_hidden_state(sd, torch.from_numpy(P.preprocess_frames(clip)).half().float(), spec.mm_vision_select_layer,
                                  num_layers=spec.vit_layers, heads=spec.vit_heads)
    check_close(got, want, what="ViT on device-preprocessed frames")


@pytest.mark.parametrize("spec_name,B,T", [("tiny-max", 2, 4), ("tiny-v2", 2, 4), ("tiny-v3", 2, 4), ("tiny-v2", 1, 8), ("tiny-v3", 3, 1),
                                            ("shape-7b-1l-v3", 1, 8)])
def test_pooling_variants_vs_oracle(spec_name, B, T):
    """patch_pooling_method = max / temporal_importance (v2) / temporal_transformer (v3), valley_model.py:205-213: the spliced
    inputs_embeds (pooled block + frame rows) and the prefill logits against the oracle; the pooled block must differ from mean pooling."""
    spec = syn.SPECS[spec_name]
    big = spec.hidden_size > 1024
    if big:
        sd = Hh.bf16_weights(spec, 3)
        m = Hh.build_model(spec, sd)
    else:
        spec, sd, m = get(spec_name, 3)
    assert m.get_model().patch_pooling_method == spec.patch_pooling_method
    cfg, tok = Hh.oracle_cfg(spec), Hh.oracle_tok(spec)
    ids, px = syn.make_prompt_ids(spec, B, T, 3, len_a=10, len_b=6), syn.make_pixels(B, T, 3)
    with torch.no_grad():
        feats = O.encode_images(sd, px, cfg.mm_vision_select_layer, num_layers=cfg.vit_layers)
        want = O.prepare_inputs_embeds(sd, ids, feats, tok, spec.patch_pooling_method)
        mean = O.prepare_inputs_embeds(sd, ids, feats, tok, "mean")
        want_logits = O.causal_lm_forward(sd, cfg, tok, ids, px, None)[:, -1]
    got = m.prepare_inputs_labels_for_multimodal(ids.cuda(), None, None, None, px.cuda())[3]
    p0 = int((ids[0] == tok.im_start_token).nonzero()[0, 0]) + 1
    blk = slice(p0, p0 + 256)
    e = check_close(got[:, blk], want[:, blk], what=f"{spec_name} pooled block")
    check_close(got, want, what=f"{spec_name} inputs_embeds")
    if T > 1:
        assert Hh.rel_fro(got[:, blk], mean[:, blk]) > max(5 * e, 2e-2)          # it is not mean pooling
    m.logits_all_positions = False
    try:
        out = m(input_ids=ids.cuda(), images=px.cuda())
    finally:
        m.logits_all_positions = True
    check_close(out.logits[:, -1], want_logits, what=f"{spec_name} prefill logits")
    if big:
        del m
        torch.cuda.empty_cache()


@pytest.mark.parametrize("spec_name", ["tiny-max", "tiny-v2", "tiny-v3"])
def test_pooling_variants_golden_reference(spec_name):
    """The REFERENCE's own outputs with config.use_patch_importance_pooling / use_delta_transformer / patch_pooling_method='max'
    (tests/golden/ref_tiny-*.pt, written by oracle/make_golden.py from the live valley_model.py)."""
    g = torch.load(os.path.join(GOLD, f"ref_{spec_name}.pt"))
    spec = syn.SPECS[spec_name]
    sd = syn.make_state_dict(spec, g["seed"])
    m = Hh.build_model(spec, sd)
    tok = Hh.oracle_tok(spec)
    ids, px = syn.make_prompt_ids(spec, g["B"], g["T"], g["seed"]), syn.make_pixels(g["B"], g["T"], g["seed"])
    emb = m.prepare_inputs_labels_for_multimodal(ids.cuda(), None, None, None, px.cuda())[3]
    p0 = int((ids[0] == tok.im_start_token).nonzero()[0, 0]) + 1
    assert Hh.rel_fro(emb[:, p0:p0 + 256][:, ::4, ::4], g["pooled_rows"]) < 2e-2
    assert Hh.rel_fro(emb[:, :, ::8], g["embeds_sub"]) < 2e-2
    m.logits_all_positions = False
    out = m(input_ids=ids.cuda(), images=px.cuda())
    assert Hh.rel_fro(out.logits[:, -1], g["prefill_logits_last"]) < 2e-2


def test_forward_with_labels_returns_the_reference_loss():
    """valley_model.py:308-318 through vly_cross_entropy: oracle on the same weights, and the REFERENCE's fp32 loss (golden)."""
    spec, sd, m = get("tiny")
    cfg, tok = Hh.oracle_cfg(spec), Hh.oracle_tok(spec)
    g = torch.load(os.path.join(GOLD, "ref_tiny.pt"))
    ids, px = syn.make_prompt_ids(spec, g["B"], g["T"], g["seed"]), syn.make_pixels(g["B"], g["T"], g["seed"])
    labels = g["loss"]["labels"]
    with torch.no_grad():
        want = O.causal_lm_loss(O.causal_lm_forward(sd, cfg, tok, ids, px, None), labels)
    out = m(input_ids=ids.cuda(), images=px.cuda(), labels=labels.cuda())
    assert abs(float(out.loss) - float(want)) < 2e-2 * float(want), (float(out.loss), float(want))
    assert abs(float(out.loss) - float(g["loss"]["loss"])) < 2e-2 * float(want)
    # exactly the mean of logsumexp - logit[label] over the counted labels of OUR logits (fp32 arithmetic check of the kernel)
    mine = torch.nn.functional.cross_entropy(out.logits[:, :-1].reshape(-1, spec.vocab_size).cpu().double(), labels[:, 1:].reshape(-1))
    assert abs(float(out.loss) - float(mine)) < 1e-5 * float(mine)
    tup = m(input_ids=ids.cuda(), images=px.cuda(), labels=labels.cuda(), return_dict=False)
    assert len(tup) == 3 and float(tup[0]) == float(out.loss)
    allign = m(input_ids=ids.cuda(), images=px.cuda(), labels=torch.full_like(labels, -100).cuda())
    assert torch.isnan(allign.loss)                                  # nothing counted: nan, like nn.CrossEntropyLoss


class _FakeTokenizer:
    """Word-level tokenizer over the model's id space: special strings -> the sentinel ids, 'w<id>' words -> id."""
    eos_token_id = 2

    def __init__(self, spec, add_bos=True):
        import re
        self.add_bos = add_bos
        t = syn.sentinel_ids(spec)
        self.special = {"<im_patch>": t["im_patch_token"], "<im_start>": t["im_start_token"], "<im_end>": t["im_end_token"],
                        "<vi_frame>": t["vi_frame_token"], "<vi_start>": t["vi_start_token"], "<vi_end>": t["vi_end_token"]}
        self.rx = re.compile(r"<[a-z_]+>|w\d+")

    def __call__(self, text):
        import types
        ids = ([1] if self.add_bos else []) + [self.special[m] if m in self.special else int(m[1:]) for m in self.rx.findall(text)]
        return types.SimpleNamespace(input_ids=ids)

    def decode(self, ids, skip_special_tokens=True):
        return "".join(f" w{int(i)}" for i in ids if int(i) not in (1, 2))


def _reference_worker_loop(m, tokenizer, params, stream_interval, context_len=2048):
    """model_worker.py:319-426 verbatim in structure (one forward per token, host sync per token), over OUR model."""
    from valley_b200 import serving
    prompt = params["prompt"]
    ori_prompt, video = prompt, params.get("video")
    prompt = serving.expand_video_prompt(prompt, video.shape[0], True)
    temperature, max_new_tokens = float(params.get("temperature", 1.0)), min(int(params.get("max_new_tokens", 256)), 1024)
    stop_str = params.get("stop")
    stop_idx = serving.stop_token_index(tokenizer, stop_str)
    input_ids = tokenizer(prompt).input_ids
    input_ids = input_ids[-(context_len - max_new_tokens - 8):]
    pred_ids, past, outs = [], None, []
    for i in range(max_new_tokens):
        if i == 0:
            out = m(torch.as_tensor([input_ids]).cuda(), use_cache=True, images=video.cuda().half().unsqueeze(0))
        else:
            out = m(input_ids=torch.as_tensor([[token]], device="cuda"), use_cache=True, past_key_values=past,
                    attention_mask=torch.ones(1, past[0][0].shape[-2] + 1, device="cuda"))
        past = out.past_key_values
        assert temperature < 1e-4
        token = int(torch.argmax(out.logits[0][-1]))
        pred_ids.append(token)
        stopped = (stop_idx is not None and token == stop_idx) or token == tokenizer.eos_token_id
        if i % stream_interval == 0 or i == max_new_tokens - 1 or stopped:
            cur_out = tokenizer.decode(pred_ids, skip_special_tokens=True)
            pos = cur_out.rfind(stop_str) if stop_str is not None else -1
            if pos != -1:
                cur_out, stopped = cur_out[:pos], True
            outs.append(ori_prompt + cur_out)
        if stopped:
            break
    return outs, pred_ids


@pytest.mark.parametrize("interval", [1, 2, 5])
def test_generate_stream_matches_the_reference_worker_loop(interval):
    """valley_b200.serving.generate_stream (device loop in chunks of stream_interval) yields the same texts at the same
    points as the reference worker's token-by-token loop: plain run, single-token stop id, multi-token stop string, eos."""
    from valley_b200 import serving
    spec, sd, m = get("tiny")
    tk = _FakeTokenizer(spec)
    video = syn.make_pixels(1, 3, 8)[0]
    words = " ".join(f"w{i}" for i in torch.randint(3, 900, (12,), generator=torch.Generator().manual_seed(1)).tolist())
    base = dict(prompt=f"{words} <video> w77 w78", video=video, temperature=0.0, max_new_tokens=11)
    ref_outs, ref_ids = _reference_worker_loop(m, tk, base, interval)
    got = [d["text"] for d in serving.generate_stream(m, tk, base, stream_interval=interval)]
    assert got == ref_outs and len(ref_ids) == 11
    assert all(d["error_code"] == 0 for d in serving.generate_stream(m, tk, base, stream_interval=interval))
    # single-token stop string -> stop id handled on the device (model_worker.py:354-360, :396-397)
    # (with a BOS-prepending tokenizer the stop string is never ONE id -- a quirk of the reference -- so: a tokenizer without BOS)
    tk1 = _FakeTokenizer(spec, add_bos=False)
    r1_plain, ids1 = _reference_worker_loop(m, tk1, base, interval)
    p1 = dict(base, stop=f" w{ids1[4]}")
    assert serving.stop_token_index(tk1, p1["stop"]) == ids1[4] and serving.stop_token_index(tk, p1["stop"]) is None
    r1, rid1 = _reference_worker_loop(m, tk1, p1, interval)
    g1 = [d["text"] for d in serving.generate_stream(m, tk1, p1, stream_interval=interval)]
    assert g1 == r1 and len(rid1) <= 5 and not r1[-1].endswith(p1["stop"])
    # multi-token stop string: only found at emission points (the text check), cut off the output
    p2 = dict(base, stop=f" w{ref_ids[5]} w{ref_ids[6]}")
    r2, _ = _reference_worker_loop(m, tk, p2, interval)
    g2 = [d["text"] for d in serving.generate_stream(m, tk, p2, stream_interval=interval)]
    assert g2 == r2 and p2["stop"] not in r2[-1]
    # eos
    tk3 = _FakeTokenizer(spec)
    tk3.eos_token_id = ref_ids[3]
    r3, ids3 = _reference_worker_loop(m, tk3, base, interval)
    g3 = [d["text"] for d in serving.generate_stream(m, tk3, base, stream_interval=interval)]
    assert g3 == r3 and len(ids3) == 4
    with pytest.raises(AssertionError):
        list(serving.generate_stream(m, tk, dict(base, prompt="w5 w6"), stream_interval=interval))


def test_from_pretrained_checkpoint_directory(tmp_path):
    """ValleyLlamaForCausalLM.from_pretrained(dir) (run_valley.py:39): same logits as loading the same tensors by hand."""
    from test_host_logic import _write_checkpoint
    from valley_b200.model import ValleyLlamaForCausalLM
    spec, sd, m = get("tiny")
    _write_checkpoint(str(tmp_path), spec, {k: v.bfloat16() for k, v in sd.items()}, "safetensors")
    m2 = ValleyLlamaForCausalLM.from_pretrained(str(tmp_path), torch_dtype=torch.float16)
    for k, v in syn.sentinel_ids(spec).items():
        setattr(m2.get_model().vision_tower.config, k, v)
    ids, px = syn.make_prompt_ids(spec, 1, 2, 0), syn.make_pixels(1, 2, 0)
    a = m(input_ids=ids.cuda(), images=px.cuda()).logits
    b = m2(input_ids=ids.cuda(), images=px.cuda()).logits
    assert torch.equal(a, b)


def test_long_prompt_near_the_context_limit():
    """S = 1 800 of the 2 048-position context: 15 query tiles x up to 15 key tiles in the prefill attention, 29 KV splits per head in
    the decode step; prefill last-token logits + teacher-forced decode steps vs the oracle, then generation up to the last position."""
    spec, sd, m = get("tiny")
    cfg, tok = Hh.oracle_cfg(spec), Hh.oracle_tok(spec)
    B, T, n = 2, 3, 4
    ids, px = syn.make_prompt_ids(spec, B, T, 2, len_a=900, len_b=636), syn.make_pixels(B, T, 2)
    assert ids.shape[1] == 1800
    with torch.no_grad():
        r_tok, r_log = O.greedy_generate(sd, cfg, tok, ids, px, n, return_logits=True)
    m.logits_all_positions = False
    try:
        out = m(input_ids=ids.cuda(), images=px.cuda())
    finally:
        m.logits_all_positions = True
    cache, logs = out.past_key_values, [out.logits[:, -1].cpu()]
    for i in range(1, n):
        o = m(input_ids=r_tok[:, i - 1:i].cuda(), past_key_values=cache)
        logs.append(o.logits[:, -1].cpu())
    logs = torch.stack(logs, 1)
    check_close(logs, r_log, what="long prompt logits")
    max_err = (logs - r_log).abs().max().item()
    top2 = r_log.topk(2, -1).values
    safe = (top2[..., 0] - top2[..., 1]) > 2 * max_err
    assert torch.equal(logs.argmax(-1)[safe], r_tok[safe])
    full = m.generate(input_ids=ids.cuda(), images=px.cuda(), max_new_tokens=1000)      # clipped to the room that is left
    assert full.shape[1] == spec.max_position_embeddings and int(full.max()) < spec.vocab_size


def test_cache_capacity_is_enforced():
    spec, sd, m = get("tiny")
    ids = syn.make_prompt_ids(spec, 1, 2, 0)
    cache = m.new_cache(1, 384)
    m(input_ids=ids.cuda(), past_key_values=cache)
    with pytest.raises(ValueError):
        m(input_ids=ids.cuda(), past_key_values=cache)            # 2 x 327 > 384


@pytest.mark.parametrize("spec_name,B", [("shape-13b-1l", 1), ("shape-13b-1l", 4), ("shape-7b-1l", 3)])
def test_production_shapes_one_layer(spec_name, B):
    """One decoder layer at the real 7B / 13B widths (H 4096/5120, I 11008/13824, 32/40 heads, V 32008): prefill logits and
    6 teacher-forced decode steps vs the oracle -- covers the K-tail slices of the CUDA-core (B = 1) and tensor-core (B > 1)
    decode consumers and the 256-wide / CTA-pair GEMM tilings."""
    spec = syn.SPECS[spec_name]
    sd = Hh.bf16_weights(spec, 2)
    m = Hh.build_model(spec, sd)
    cfg, tok = Hh.oracle_cfg(spec), Hh.oracle_tok(spec)
    T, n = 2, 6
    ids, px = syn.make_prompt_ids(spec, B, T, 0, len_a=12, len_b=7), syn.make_pixels(B, T, 0)
    with torch.no_grad():
        r_tok, r_log = O.greedy_generate(sd, cfg, tok, ids, px, n, return_logits=True)
    m.logits_all_positions = False
    out = m(input_ids=ids.cuda(), images=px.cuda())
    cache, logs = out.past_key_values, [out.logits[:, -1].cpu()]
    for i in range(1, n):
        o = m(input_ids=r_tok[:, i - 1:i].cuda(), past_key_values=cache)
        logs.append(o.logits[:, -1].cpu())
    logs = torch.stack(logs, 1)
    assert not torch.isnan(logs).any()
    assert Hh.rel_fro(logs, r_log) < 2e-2
    max_err = (logs - r_log).abs().max().item()
    top2 = r_log.topk(2, -1).values
    safe = (top2[..., 0] - top2[..., 1]) > 2 * max_err
    assert torch.equal(logs.argmax(-1)[safe], r_tok[safe])
    del m
    _models.pop((spec_name, 2), None)
    torch.cuda.empty_cache()


def _decode_parity(spec_name, B, n=8, seed=0, len_a=20, len_b=11):
    spec, sd, m = get(spec_name, seed)
    cfg, tok = Hh.oracle_cfg(spec), Hh.oracle_tok(spec)
    T = 2
    ids, px = syn.make_prompt_ids(spec, B, T, 0, len_a=len_a, len_b=len_b), syn.make_pixels(B, T, 0)
    with torch.no_grad():
        r_tok, r_log = O.greedy_generate(sd, cfg, tok, ids, px, n, return_logits=True)
    m.logits_all_positions = False
    try:
        out = m(input_ids=ids.cuda(), images=px.cuda())
    finally:
        m.logits_all_positions = True
    cache, logs = out.past_key_values, [out.logits[:, -1].cpu()]
    for i in range(1, n):
        o = m(input_ids=r_tok[:, i - 1:i].cuda(), past_key_values=cache)
        logs.append(o.logits[:, -1].cpu())
    logs = torch.stack(logs, 1)
    assert torch.isfinite(logs).all()
    assert Hh.rel_fro(logs, r_log) < 2e-2, Hh.rel_fro(logs, r_log)
    max_err = (logs - r_log).abs().max().item()
    top2 = r_log.topk(2, -1).values
    safe = (top2[..., 0] - top2[..., 1]) > 2 * max_err
    assert torch.equal(logs.argmax(-1)[safe], r_tok[safe])
    gen = m.generate(input_ids=ids.cuda(), images=px.cuda(), max_new_tokens=n)[:, ids.shape[1]:].cpu()
    gen2 = m.generate(input_ids=ids.cuda(), images=px.cuda(), max_new_tokens=n)[:, ids.shape[1]:].cpu()
    assert torch.equal(gen, gen2)
    for b in range(B):
        for i in range(n):
            if not safe[b, i]:
                break
            assert gen[b, i] == r_tok[b, i], (b, i)
    return Hh.rel_fro(logs, r_log)


@pytest.mark.parametrize("B", [2, 3, 4])
def test_tcgen05_decode_consumer_full_and_tail_stages(B):
    """decode_step_umma_kernel (B = 2..4, K multiples of 512): tiny-umma has intermediate_size 3584 = one 2560-column stage + a 1024-column
    tail stage per work unit of down_proj (two sub-phases on one staged activation block); prefill + 8 teacher-forced steps +
    free-running ids vs the oracle.  B = 1 on the same model runs decode_step_kernel<1> (the reference point)."""
    _decode_parity("tiny-umma", B)


@pytest.mark.parametrize("len_a,len_b", [(230, 120), (400, 250)])
def test_decode_attention_multi_pass_items_at_production_head_count(len_a, len_b):
    """B = 4 sequences x 40 heads (one LLaMA-13B-wide layer) at contexts of ~610 and ~910 keys: more 16- / 32-key items than the
    2368 warps of the decode kernel, so the attention phase runs 48- / 64-key items (3 - 4 passes per warp, mask bits fetched per
    pass, up to 5 % of the items in a second round) -- the regime the headline request spends its second half in.  Prefill logits,
    8 teacher-forced decode steps and free-running ids vs the oracle."""
    _decode_parity("shape-13b-1l", 4, len_a=len_a, len_b=len_b)


def _decode_parity_subprocess(env, calls):
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r); import test_gpu_parity as t; print('ERR', %s)"
            % (os.path.dirname(__file__), os.path.dirname(os.path.dirname(__file__)), ", ".join("t._decode_parity(%r, %d)" % c for c in calls)))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, env=dict(os.environ, **env))
    assert r.returncode == 0 and "ERR" in r.stdout, r.stdout[-1500:] + r.stderr[-1500:]


def test_tcgen05_decode_consumer_ragged_k():
    """intermediate_size = 3776 = 59 panels of 64 columns (Llama-2-7B: 11008 = 172): the K walk is rounded up to whole 512-column
    groups and the panels beyond the real K are out of bounds in both tensor maps (zero fill, no memory read).  Not the default for
    such shapes (measured slower than the mma.sync consumer on Llama-2-7B), so it is forced with VLY_DECODE_UMMA=2."""
    _decode_parity_subprocess({"VLY_DECODE_UMMA": "2"}, [("tiny-umma-ragged", 2), ("tiny-umma-ragged", 4)])


def test_tcgen05_decode_consumer_restaged_sub_phases():
    """The same with VLY_UMMA_XC=512: the activation block holds 512 columns, so down_proj (K = 3584) is walked in SEVEN sub-phases
    with the block re-staged behind a CTA-local barrier and the accumulators resident in TMEM in between -- the mechanism the 13B
    model uses for K = 13824 (3 pieces).  The switch is read once per process, hence the subprocess."""
    _decode_parity_subprocess({"VLY_UMMA_XC": "512"}, [("tiny-umma", 4), ("tiny-umma", 2)])
