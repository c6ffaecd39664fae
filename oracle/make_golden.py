"""Pin the oracle against the REFERENCE ITSELF and write golden fixtures (build container only).

Run:  python oracle/make_golden.py            (needs /root/reference; CPU, ~1-2 min)

What it does
  1. imports /root/reference/valley/model/valley_model.py unmodified (decord / skimage are
     stubbed: they are only needed by load_video, which synthetic inputs bypass) on top of the
     installed HuggingFace transformers (5.5.0; the reference's pin cae78c46 is not
     available offline -- SURVEY.md 8c);
  2. builds random-init reference models at the parity-test sizes, loads OUR synthetic
     state_dict into them, and runs ValleyLlamaForCausalLM.forward(images=...) plus the
     model_worker-style greedy loop (valley/serve/model_worker.py:371-397; HF generate() is
     not a valid oracle under HF 5.x, SURVEY Appendix C-1);
  3. asserts oracle/valley_oracle.py reproduces the reference (fp32, tight tolerance) --
     including the splice edge cases and the two ValueError paths;
  4. writes the REFERENCE's outputs to tests/golden/*.pt (small, sub-sampled where large).

/root/reference does not exist on the GPU box; nothing at test/bench time imports this file.
"""
from __future__ import annotations

import os
import sys
import tempfile
import types

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, "/root/reference")
for name in ("decord", "skimage", "skimage.transform"):
    sys.modules.setdefault(name, types.ModuleType(name))

import torch  # noqa: E402
from transformers import CLIPVisionConfig, CLIPVisionModel  # noqa: E402

from valley.model.valley_model import ValleyConfig, ValleyLlamaForCausalLM  # noqa: E402  (the reference)

from oracle import valley_oracle as O  # noqa: E402
from valley_b200 import synthetic as syn  # noqa: E402

GOLD = os.path.join(REPO, "tests", "golden")


def build_reference(spec: syn.ShapeSpec, sd, tmp):
    vc = CLIPVisionConfig(hidden_size=spec.vit_hidden, intermediate_size=spec.vit_mlp,
                          num_hidden_layers=spec.vit_layers, num_attention_heads=spec.vit_heads,
                          image_size=spec.vit_image, patch_size=spec.vit_patch, hidden_act="quick_gelu",
                          layer_norm_eps=spec.vit_eps)
    vc._attn_implementation = "eager"
    vdir = os.path.join(tmp, "vit_" + spec.name)
    CLIPVisionModel(vc).save_pretrained(vdir)
    cfg = ValleyConfig(hidden_size=spec.hidden_size, num_hidden_layers=spec.num_hidden_layers,
                       num_attention_heads=spec.num_attention_heads, num_key_value_heads=spec.num_attention_heads,
                       intermediate_size=spec.intermediate_size, vocab_size=spec.vocab_size,
                       rms_norm_eps=spec.rms_norm_eps, max_position_embeddings=spec.max_position_embeddings,
                       attention_bias=False, mlp_bias=False, tie_word_embeddings=False)
    cfg.mm_vision_tower = vdir
    cfg.use_mm_proj = True
    cfg.mm_hidden_size = spec.vit_hidden
    cfg.mm_vision_select_layer = spec.mm_vision_select_layer
    cfg._attn_implementation = "eager"
    if spec.patch_pooling_method == "temporal_importance":
        cfg.use_patch_importance_pooling = True                   # valley_model.py:40-43
    if spec.patch_pooling_method == "temporal_transformer":
        cfg.use_delta_transformer = True                          # valley_model.py:45-52
    model = ValleyLlamaForCausalLM(cfg).to(torch.float32).eval()
    if spec.patch_pooling_method == "max":
        model.model.patch_pooling_method = "max"                  # only reachable by setting the attribute (:208-209)
    model.model.vision_tower.config._attn_implementation = "eager"
    missing, unexpected = model.load_state_dict(sd, strict=False)
    # transforemr_adding_layer is the template nn.TransformerEncoder deep-copies: present in the state_dict, never executed
    bad = [m for m in missing if "post_layernorm" not in m and "position_ids" not in m and "inv_freq" not in m
           and "transforemr_adding_layer" not in m]
    assert not bad and not unexpected, (bad, unexpected)
    vcfg = model.get_model().vision_tower.config
    for k, v in syn.sentinel_ids(spec).items():
        setattr(vcfg, k, v)
    vcfg.use_im_start_end = True
    return model


def ref_greedy(model, input_ids, images, n):
    """model_worker.py:371-397 generalised to B rows, get_seq_length() instead of [0][0].shape[-2]."""
    toks, logs, past = [], [], None
    for i in range(n):
        if i == 0:
            out = model(input_ids, use_cache=True, images=images)
        else:
            am = torch.ones(input_ids.shape[0], past.get_seq_length() + 1)
            out = model(input_ids=cur, use_cache=True, attention_mask=am, past_key_values=past)
        past = out.past_key_values
        last = out.logits[:, -1, :]
        nxt = torch.argmax(last, dim=-1)
        toks.append(nxt)
        logs.append(last.float())
        cur = nxt[:, None]
    return torch.stack(toks, 1), torch.stack(logs, 1)


def oracle_cfg(spec):
    return O.OracleConfig(hidden_size=spec.hidden_size, num_hidden_layers=spec.num_hidden_layers,
                          num_attention_heads=spec.num_attention_heads, intermediate_size=spec.intermediate_size,
                          vocab_size=spec.vocab_size, rms_norm_eps=spec.rms_norm_eps, rope_theta=spec.rope_theta,
                          vit_layers=spec.vit_layers, vit_heads=spec.vit_heads, vit_patch=spec.vit_patch,
                          vit_eps=spec.vit_eps, mm_vision_select_layer=spec.mm_vision_select_layer,
                          patch_pooling_method=spec.patch_pooling_method)


def close(a, b, what, rtol=2e-5):
    err = (a - b).abs().max().item()
    scale = b.abs().max().item() + 1e-12
    print(f"  {what:48s} max|d|={err:.3e}  rel={err / scale:.3e}")
    assert err / scale < rtol, what


@torch.no_grad()
def main():
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count())
    os.makedirs(GOLD, exist_ok=True)
    with tempfile.TemporaryDirectory() as tmp:
        for spec, B, T, seed, ntok in ((syn.TINY, 2, 3, 0, 8), (syn.TINY_WIDE, 1, 8, 1, 6)):
            print(f"== {spec.name}: B={B} T={T}")
            sd = syn.make_state_dict(spec, seed)
            ref = build_reference(spec, sd, tmp)
            cfg, tok = oracle_cfg(spec), O.SentinelIds(*[syn.sentinel_ids(spec)[k] for k in (
                "im_patch_token", "im_start_token", "im_end_token", "vi_frame_token", "vi_start_token", "vi_end_token")])
            ids = syn.make_prompt_ids(spec, B, T, seed)
            px = syn.make_pixels(B, T, seed)

            # --- ViT hidden states straight from the reference's vision tower ------------------
            vt = ref.get_model().vision_tower
            hs = vt(px[0], output_hidden_states=True).hidden_states
            for sel in (-2, -1, 0):
                mine = O.vit_hidden_state(sd, px[0], sel, num_layers=spec.vit_layers, heads=spec.vit_heads)
                close(mine, hs[sel], f"vit hidden_states[{sel}]")

            # --- full forward + greedy loop ---------------------------------------------------
            out = ref(ids, images=px, use_cache=True)
            mine = O.causal_lm_forward(sd, cfg, tok, ids, px, O.KVCache(spec.num_hidden_layers))
            close(mine, out.logits, "prefill logits")
            r_tok, r_log = ref_greedy(ref, ids, px, ntok)
            o_tok, o_log = O.greedy_generate(sd, cfg, tok, ids, px, ntok, return_logits=True)
            close(o_log, r_log, "greedy last-token logits")
            assert torch.equal(o_tok, r_tok), "greedy token ids differ"
            print("  greedy token ids identical:", r_tok[0].tolist())

            # --- left-padded batch with a 2-D attention_mask (build_inputs pads left; HF masks the padded keys,
            #     positions are NOT shifted): prefill + 3 cached decode steps, compared at the non-pad positions -----
            pad = 5
            ids_p = torch.cat([ids[:, :pad], ids], 1)
            am = torch.ones_like(ids_p)
            am[0, :pad] = 0
            ids_p[0, :pad] = 0
            lp_out = ref(ids_p, attention_mask=am, images=px, use_cache=True)
            lp_cache = O.KVCache(spec.num_hidden_layers)
            mine = O.causal_lm_forward(sd, cfg, tok, ids_p, px, lp_cache, attention_mask=am)
            close(mine[am.bool()], lp_out.logits[am.bool()], "left-pad prefill logits (non-pad rows)")
            lp_steps, lp_mask, past = [], am, lp_out.past_key_values
            cur = lp_out.logits[:, -1].argmax(-1)[:, None]
            lp_first = cur.clone()
            for i in range(3):
                lp_mask = torch.cat([lp_mask, torch.ones(B, 1, dtype=am.dtype)], 1)
                o = ref(input_ids=cur, attention_mask=lp_mask, past_key_values=past, use_cache=True)
                mo = O.causal_lm_forward(sd, cfg, tok, cur, None, lp_cache, attention_mask=lp_mask)
                close(mo, o.logits, f"left-pad decode step {i} logits")
                lp_steps.append(o.logits[:, -1].clone())
                cur = o.logits[:, -1].argmax(-1)[:, None]
            # --- labels -> loss (valley_model.py:308-318), prompt part masked with IGNORE_INDEX like the data pipeline ------
            labels = ids.clone()
            labels[:, : ids.shape[1] // 2] = -100
            lo = ref(ids, images=px, labels=labels, use_cache=False)
            mine_loss = O.causal_lm_loss(O.causal_lm_forward(sd, cfg, tok, ids, px, None), labels)
            close(mine_loss[None], lo.loss[None], "cross-entropy loss (labels)")
            gold_loss = dict(labels=labels, loss=lo.loss.clone())
            gold_leftpad = dict(ids=ids_p, mask=am, prefill_logits_last=lp_out.logits[:, -1].clone(), first_token=lp_first,
                                decode_logits=torch.stack(lp_steps, 1))

            # --- inputs_embeds after splice: hook the reference's LlamaModel.forward -----------
            grabbed = {}
            import transformers
            orig = transformers.LlamaModel.forward

            def spy(self, *a, **k):
                grabbed["e"] = k["inputs_embeds"].clone()
                return orig(self, *a, **k)

            transformers.LlamaModel.forward = spy
            try:
                cases = {}
                V = spec.vocab_size
                t = syn.sentinel_ids(spec)
                base = ids[0].clone()
                # (a) row 1 has no image tokens at all (non-multimodal sample in a multimodal batch)
                plain = torch.randint(3, V - 8, base.shape, generator=torch.Generator().manual_seed(5))
                cases["mixed_batch"] = (torch.stack([base, plain]), px[:1])
                # (b) video frame count mismatch -> silent fallback to image-only splice (bare except)
                bad_vid = base.clone()
                bad_vid[(bad_vid == t["vi_frame_token"]).nonzero()[0]] = 5
                cases["video_fallback"] = (bad_vid[None], px[:1])
                # (c) two <im_start> blocks in one sample: both get the same pooled block
                mid = [t["im_start_token"]] + [t["im_patch_token"]] * 256 + [t["im_end_token"]]
                two = torch.cat([base, torch.tensor(mid), torch.tensor([9, 10])])
                cases["two_images"] = (two[None], px[:1])
                # (d) no vi_* tokens in the prompt at all (image-only prompt)
                only_img = torch.cat([torch.tensor([1, 11, 12]), torch.tensor(mid), torch.tensor([13, 14, 15])])
                cases["image_only"] = (only_img[None], px[:1, :1])
                gold_splice = {}
                for name, (cid, cpx) in cases.items():
                    ref(cid, images=cpx, use_cache=False)
                    feats = O.encode_images(sd, cpx, cfg.mm_vision_select_layer, num_layers=cfg.vit_layers)
                    mine = O.prepare_inputs_embeds(sd, cid, feats, tok)
                    close(mine, grabbed["e"], f"splice[{name}] inputs_embeds")
                    gold_splice[name] = dict(ids=cid, n_frames=cpx.shape[1], embeds_sub=grabbed["e"][:, :, ::8].clone())
                # (e) images as a Python LIST of clips with different frame counts (valley_model.py:168-176, :187-188):
                #     rows padded to one length with plain tokens; each sample's <vi_frame> count matches its own clip
                if B >= 2:
                    ra = syn.make_prompt_ids(spec, 1, 2, seed, len_b=25)[0]
                    rb = syn.make_prompt_ids(spec, 1, 3, seed + 1, len_b=24)[0]
                    lids = torch.stack([ra, rb])
                    limgs = [px[0, :2], px[1, :3]]
                    ref(lids, images=limgs, use_cache=False)
                    lfeats = O.encode_images(sd, limgs, cfg.mm_vision_select_layer, num_layers=cfg.vit_layers)
                    assert isinstance(lfeats, list) and lfeats[0].shape[0] == 2 and lfeats[1].shape[0] == 3
                    mine = O.prepare_inputs_embeds(sd, lids, lfeats, tok)
                    close(mine, grabbed["e"], "splice[list_images] inputs_embeds")
                    gold_splice["list_images"] = dict(ids=lids, n_frames=[2, 3], embeds_sub=grabbed["e"][:, :, ::8].clone())
                # error paths: same exception type + message from both
                errs = {}
                cut = base.clone()
                cut[(cut == t["im_end_token"]).nonzero()[0]] = 7
                cut2 = torch.cat([cut, torch.tensor([t["im_end_token"]])])     # counts match, position wrong
                unbalanced = base.clone()
                unbalanced[(unbalanced == t["im_end_token"]).nonzero()[0]] = 7
                for name, cid in (("image_cut", cut2[None]), ("unbalanced", unbalanced[None])):
                    msgs = []
                    for fn in (lambda: ref(cid, images=px[:1]),
                               lambda: O.causal_lm_forward(sd, cfg, tok, cid, px[:1], None)):
                        try:
                            fn()
                            msgs.append(None)
                        except ValueError as e:
                            msgs.append(str(e))
                    assert msgs[0] is not None and msgs[0] == msgs[1], msgs
                    errs[name] = dict(ids=cid, message=msgs[0])
                    print(f"  error[{name}]: {msgs[0]!r} (identical)")
            finally:
                transformers.LlamaModel.forward = orig

            torch.save(dict(
                spec=spec.name, seed=seed, B=B, T=T,
                vit_hidden_m2_sub=hs[-2][:, ::4, ::8].clone(), vit_hidden_m1_sub=hs[-1][:, ::4, ::8].clone(),
                prefill_logits_last=out.logits[:, -1, :].clone(), prefill_logits_sub=out.logits[:, ::16, ::8].clone(),
                greedy_tokens=r_tok, greedy_logits=r_log, errors=errs, leftpad=gold_leftpad, loss=gold_loss,
            ), os.path.join(GOLD, f"ref_{spec.name}.pt"))
            torch.save(gold_splice, os.path.join(GOLD, f"ref_{spec.name}_splice.pt"))       # own file: every fixture stays under 1 MB
            print("  wrote", f"tests/golden/ref_{spec.name}.pt", f"tests/golden/ref_{spec.name}_splice.pt")
        # --- pooling variants (valley_model.py:205-213): max, temporal_importance (v2), temporal_transformer (v3) -------
        import transformers
        for spec in (syn.TINY_MAX, syn.TINY_V2, syn.TINY_V3):
            print(f"== {spec.name}: patch_pooling_method = {spec.patch_pooling_method}")
            B, T, seed = 2, 4, 3
            sd = syn.make_state_dict(spec, seed)
            ref = build_reference(spec, sd, tmp)
            assert ref.get_model().patch_pooling_method == spec.patch_pooling_method
            cfg, tok = oracle_cfg(spec), O.SentinelIds(*[syn.sentinel_ids(spec)[k] for k in (
                "im_patch_token", "im_start_token", "im_end_token", "vi_frame_token", "vi_start_token", "vi_end_token")])
            ids, px = syn.make_prompt_ids(spec, B, T, seed), syn.make_pixels(B, T, seed)
            grabbed, orig = {}, transformers.LlamaModel.forward

            def spy(self, *a, **k):
                grabbed["e"] = k["inputs_embeds"].clone()
                return orig(self, *a, **k)

            transformers.LlamaModel.forward = spy
            try:
                out = ref(ids, images=px, use_cache=False)
            finally:
                transformers.LlamaModel.forward = orig
            feats = O.encode_images(sd, px, cfg.mm_vision_select_layer, num_layers=cfg.vit_layers)
            emb = O.prepare_inputs_embeds(sd, ids, feats, tok, spec.patch_pooling_method)
            close(emb, grabbed["e"], "inputs_embeds after splice")
            plain = O.prepare_inputs_embeds(sd, ids, feats, tok, "mean")
            assert (plain - grabbed["e"]).abs().max() > 1e-3          # the variant really differs from mean pooling
            close(O.causal_lm_forward(sd, cfg, tok, ids, px, None), out.logits, "prefill logits")
            p0 = (ids[0] == tok.im_start_token).nonzero()[0, 0] + 1
            torch.save(dict(spec=spec.name, seed=seed, B=B, T=T, pooled_rows=grabbed["e"][:, p0:p0 + 256, ::4][:, ::4].clone(),
                            embeds_sub=grabbed["e"][:, :, ::8].clone(), prefill_logits_last=out.logits[:, -1, :].clone()),
                       os.path.join(GOLD, f"ref_{spec.name}.pt"))
            print("  wrote", f"tests/golden/ref_{spec.name}.pt")
    print("oracle == reference on all cases; golden fixtures written")


if __name__ == "__main__":
    main()
