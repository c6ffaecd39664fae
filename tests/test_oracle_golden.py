"""CPU: the oracle must reproduce the REFERENCE's outputs stored in tests/golden/ (written by
oracle/make_golden.py from the live reference classes).  fp32, tight tolerance."""
import os

import pytest
import torch

import helpers as Hh
from oracle import valley_oracle as O
from valley_b200 import synthetic as syn

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("name", ["tiny", "tiny-wide"])
def test_oracle_matches_reference_fixture(name):
    g = torch.load(os.path.join(GOLD, f"ref_{name}.pt"))
    spec = syn.SPECS[name]
    sd = syn.make_state_dict(spec, g["seed"])
    cfg, tok = Hh.oracle_cfg(spec), Hh.oracle_tok(spec)
    ids, px = syn.make_prompt_ids(spec, g["B"], g["T"], g["seed"]), syn.make_pixels(g["B"], g["T"], g["seed"])
    with torch.no_grad():
        h2 = O.vit_hidden_state(sd, px[0], -2, num_layers=spec.vit_layers, heads=spec.vit_heads)
        h1 = O.vit_hidden_state(sd, px[0], -1, num_layers=spec.vit_layers, heads=spec.vit_heads)
        assert torch.allclose(h2[:, ::4, ::8], g["vit_hidden_m2_sub"], rtol=1e-5, atol=1e-5)
        assert torch.allclose(h1[:, ::4, ::8], g["vit_hidden_m1_sub"], rtol=1e-5, atol=1e-5)
        logits = O.causal_lm_forward(sd, cfg, tok, ids, px, None)
        assert torch.allclose(logits[:, -1], g["prefill_logits_last"], rtol=1e-4, atol=1e-5)
        assert torch.allclose(logits[:, ::16, ::8], g["prefill_logits_sub"], rtol=1e-4, atol=1e-5)
        n = g["greedy_tokens"].shape[1]
        toks, logs = O.greedy_generate(sd, cfg, tok, ids, px, n, return_logits=True)
        assert torch.equal(toks, g["greedy_tokens"])                       # token ids: exact
        assert torch.allclose(logs, g["greedy_logits"], rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("name", ["tiny"])
def test_oracle_splice_cases_match_reference(name):
    g = torch.load(os.path.join(GOLD, f"ref_{name}.pt"))
    splice = torch.load(os.path.join(GOLD, f"ref_{name}_splice.pt"))
    spec = syn.SPECS[name]
    sd = syn.make_state_dict(spec, g["seed"])
    cfg, tok = Hh.oracle_cfg(spec), Hh.oracle_tok(spec)
    px = syn.make_pixels(g["B"], g["T"], g["seed"])
    with torch.no_grad():
        for case, d in splice.items():
            if isinstance(d["n_frames"], list):          # images given as a list of clips with different frame counts
                cpx = [px[i, :n] for i, n in enumerate(d["n_frames"])]
            else:
                cpx = px[:1, : d["n_frames"]]
            feats = O.encode_images(sd, cpx, cfg.mm_vision_select_layer, num_layers=cfg.vit_layers)
            emb = O.prepare_inputs_embeds(sd, d["ids"], feats, tok)
            assert torch.allclose(emb[:, :, ::8], d["embeds_sub"], rtol=1e-5, atol=1e-6), case
        for case, d in g["errors"].items():
            with pytest.raises(ValueError) as ei:
                O.causal_lm_forward(sd, cfg, tok, d["ids"], px[:1], None)
            assert str(ei.value) == d["message"], case


@pytest.mark.parametrize("name", ["tiny", "tiny-wide"])
def test_oracle_left_padded_batch_matches_reference(name):
    """attention_mask with left padding (model_worker/build_inputs pad left): masked keys, unshifted positions."""
    g = torch.load(os.path.join(GOLD, f"ref_{name}.pt"))
    spec, lp = syn.SPECS[name], g["leftpad"]
    sd = syn.make_state_dict(spec, g["seed"])
    cfg, tok = Hh.oracle_cfg(spec), Hh.oracle_tok(spec)
    px = syn.make_pixels(g["B"], g["T"], g["seed"])
    with torch.no_grad():
        cache = O.KVCache(spec.num_hidden_layers)
        logits = O.causal_lm_forward(sd, cfg, tok, lp["ids"], px, cache, attention_mask=lp["mask"])
        assert torch.allclose(logits[:, -1], lp["prefill_logits_last"], rtol=1e-4, atol=1e-5)
        cur, mask = logits[:, -1].argmax(-1)[:, None], lp["mask"]
        assert torch.equal(cur, lp["first_token"])
        for i in range(lp["decode_logits"].shape[1]):
            mask = torch.cat([mask, torch.ones(mask.shape[0], 1, dtype=mask.dtype)], 1)
            lg = O.causal_lm_forward(sd, cfg, tok, cur, None, cache, attention_mask=mask)[:, -1]
            assert torch.allclose(lg, lp["decode_logits"][:, i], rtol=1e-4, atol=1e-5)
            cur = lg.argmax(-1)[:, None]


def _clip(h, w, seed):
    import numpy as np
    rs = np.random.RandomState(seed)
    a = rs.randint(0, 256, (h, w, 3)).astype(np.uint8)
    yy, xx = np.mgrid[0:h, 0:w]
    b = np.stack([(xx * 255 // max(w - 1, 1)), (yy * 255 // max(h - 1, 1)), ((xx + yy) % 256)], -1)
    b = np.clip(b + rs.randint(-3, 4, b.shape), 0, 255).astype(np.uint8)
    return np.stack([a, b])


def test_preprocess_oracle_matches_reference_fixture():
    """load_video's PIL pipeline (Resize(256) BILINEAR -> CenterCrop(224) -> /255 -> mean/std), bit for bit."""
    import hashlib
    import numpy as np
    from oracle import preprocess_oracle as P
    gold = torch.load(os.path.join(GOLD, "ref_preprocess.pt"))
    assert len(gold) >= 9
    for (h, w), g in gold.items():
        clip = _clip(h, w, g["seed"])
        u8 = P.preprocess_frames(clip, return_uint8=True)
        f = P.preprocess_frames(clip)
        assert hashlib.sha256(np.ascontiguousarray(u8).tobytes()).hexdigest() == g["sha_u8"], (h, w)
        assert hashlib.sha256(np.ascontiguousarray(f).tobytes()).hexdigest() == g["sha_f32"], (h, w)
        assert np.array_equal(f[:, :, ::9, ::7], g["sub_f32"].numpy())
        assert np.array_equal(P.pil_pipeline(clip), f)                # the Pillow-executed pipeline bench.py times as the CPU baseline


@pytest.mark.parametrize("name", ["tiny-max", "tiny-v2", "tiny-v3"])
def test_oracle_pooling_variants_match_reference_fixture(name):
    """patch_pooling_method max / temporal_importance / temporal_transformer (valley_model.py:113-133, :205-213)."""
    g = torch.load(os.path.join(GOLD, f"ref_{name}.pt"))
    spec = syn.SPECS[name]
    sd = syn.make_state_dict(spec, g["seed"])
    cfg, tok = Hh.oracle_cfg(spec), Hh.oracle_tok(spec)
    ids, px = syn.make_prompt_ids(spec, g["B"], g["T"], g["seed"]), syn.make_pixels(g["B"], g["T"], g["seed"])
    with torch.no_grad():
        feats = O.encode_images(sd, px, cfg.mm_vision_select_layer, num_layers=cfg.vit_layers)
        emb = O.prepare_inputs_embeds(sd, ids, feats, tok, spec.patch_pooling_method)
        assert torch.allclose(emb[:, :, ::8], g["embeds_sub"], rtol=1e-5, atol=1e-6)
        logits = O.causal_lm_forward(sd, cfg, tok, ids, px, None)
        assert torch.allclose(logits[:, -1], g["prefill_logits_last"], rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("name", ["tiny", "tiny-wide"])
def test_oracle_loss_matches_reference_fixture(name):
    """forward(labels=...) -> shifted cross-entropy with IGNORE_INDEX (valley_model.py:308-318)."""
    g = torch.load(os.path.join(GOLD, f"ref_{name}.pt"))
    spec = syn.SPECS[name]
    sd = syn.make_state_dict(spec, g["seed"])
    cfg, tok = Hh.oracle_cfg(spec), Hh.oracle_tok(spec)
    ids, px = syn.make_prompt_ids(spec, g["B"], g["T"], g["seed"]), syn.make_pixels(g["B"], g["T"], g["seed"])
    with torch.no_grad():
        loss = O.causal_lm_loss(O.causal_lm_forward(sd, cfg, tok, ids, px, None), g["loss"]["labels"])
    assert torch.allclose(loss, g["loss"]["loss"], rtol=1e-5, atol=1e-6)


def test_preprocess_oracle_equals_pillow_on_random_geometries():
    """The numpy restatement against Pillow itself (the library the reference calls) on 40 random frame sizes, including
    up-scaling, extreme aspect ratios and sizes next to the 256 / 224 thresholds: bit for bit, plus the host tables of the C ABI."""
    import numpy as np
    from oracle import preprocess_oracle as P
    from valley_b200 import video
    rs = np.random.RandomState(7)
    sizes = [(int(rs.randint(30, 700)), int(rs.randint(30, 700))) for _ in range(34)] + [(256, 256), (257, 256), (224, 1000), (1000, 225), (31, 640), (256, 31)]
    for h, w in sizes:
        clip = rs.randint(0, 256, (1, h, w, 3)).astype(np.uint8)
        a, b = P.preprocess_frames(clip), P.pil_pipeline(clip)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), (h, w)
        nh, nw, cy, cx = video.preprocess_plan(h, w)
        assert (nh, nw) == P.resize_sizes(h, w) and (cy, cx) == P.crop_origin(nh, nw), (h, w)
        for n_in, n_out in ((h, nh), (w, nw)):
            k, xmin, cnt, kk = video.resample_coeffs(n_in, n_out)
            ok, oxmin, ocnt, okk = P.bilinear_coeffs(n_in, n_out)
            assert k == ok and np.array_equal(xmin, oxmin) and np.array_equal(cnt, ocnt) and np.array_equal(kk, okk), (h, w)
