"""Differential fuzz of the splice logic (valley_model.py:192-247) against the LIVE reference -> tests/golden/ref_splice_fuzz.pt.

Random token rows with well-formed, corrupted, truncated, duplicated and misplaced <im_*> / <vi_*> blocks are pushed through the
reference model's forward (tiny LLaMA, 1-layer ViT).  For each row the fixture stores what the reference did: the exception type +
message, or the per-position SOURCE MAP recovered from the inputs_embeds it built (-1 = token embedding, j < 256 = pooled patch
row j, 256 + t = frame t's CLS row).  The oracle's splice and the C host plan (vly_build_splice_map) are checked against it here
and again, from the fixture, in tests/test_host_logic.py.  Run in the build container only.
"""
import os
import sys
import tempfile
import types

for n in ("decord", "skimage", "skimage.transform", "cv2"):
    sys.modules.setdefault(n, types.ModuleType(n))
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, "/root/reference")

import dataclasses

import torch
import transformers

import make_golden as G
from oracle import valley_oracle as O
from valley_b200 import synthetic as syn

N_CASES, T = 400, 3


def make_rows(spec, n, T, seed=0):
    """Deterministic case generator (shared with the test through the stored ids)."""
    g = torch.Generator().manual_seed(seed)
    t = syn.sentinel_ids(spec)
    ri = lambda lo, hi: int(torch.randint(lo, hi, (1,), generator=g))
    rnd = lambda: float(torch.rand(1, generator=g))
    rows = []
    img = [t["im_start_token"]] + [t["im_patch_token"]] * 256 + [t["im_end_token"]]
    plain = lambda k: torch.randint(3, spec.vocab_size - 8, (k,), generator=g).tolist()
    for _ in range(n):
        sc = rnd()
        if sc < 0.3:                                             # well-formed image block(s) + a video block in several states
            parts = plain(ri(1, 40))
            for _b in range(ri(1, 3)):
                parts += img + plain(ri(0, 10))
            r = rnd()
            k = T if r < 0.6 else T + ri(-1, 2)
            vid = [t["vi_start_token"]] + [t["vi_frame_token"]] * max(k, 0) + [t["vi_end_token"]]
            if r > 0.85:
                vid = vid[:-1] + [13, t["vi_end_token"]]        # <vi_end> misplaced -> silent image-only fallback
            if rnd() < 0.85:
                parts += vid
            if rnd() < 0.2:
                parts += vid                                     # two video blocks: every <vi_start> gets the frames
            rows.append(torch.tensor(parts + plain(ri(0, 30)), dtype=torch.int64))
            continue
        if sc < 0.4:                                             # balanced counts, but the block runs past the end of the row
            k = ri(2, 256)
            parts = plain(ri(0, 20)) + [t["im_end_token"]] + plain(ri(0, 20)) + [t["im_start_token"]] + [t["im_patch_token"]] * k
            rows.append(torch.tensor(parts, dtype=torch.int64))
            continue
        S = ri(40, 900)
        row = torch.randint(3, spec.vocab_size - 8, (S,), generator=g)
        for _b in range(ri(0, 3)):                               # image blocks
            blk = [t["im_start_token"]] + [t["im_patch_token"]] * 256 + [t["im_end_token"]]
            r = rnd()
            if r < 0.06:
                blk[-1] = 7                                      # missing <im_end>
            elif r < 0.1:
                blk = blk[:-1] + [9, t["im_end_token"]]         # <im_end> one position late
            elif r < 0.13:
                blk = blk[: ri(2, 200)]                          # truncated block
            elif r < 0.15:
                blk = blk[1:]                                    # missing <im_start>
            p = ri(0, max(1, S - 1))
            blk = blk[: max(0, S - p)]
            row[p: p + len(blk)] = torch.tensor(blk, dtype=row.dtype)
        if rnd() < 0.7:                                          # video block
            k = T + (0 if rnd() < 0.7 else ri(-1, 2))
            blk = [t["vi_start_token"]] + [t["vi_frame_token"]] * max(k, 0) + [t["vi_end_token"]]
            r = rnd()
            if r < 0.1:
                blk[-1] = 11
            elif r < 0.18:
                blk = blk[:-1] + [12, t["vi_end_token"]]
            p = ri(0, max(1, S - 1))
            blk = blk[: max(0, S - p)]
            if rnd() < 0.8:                                      # usually after the image, sometimes on top of it
                row[p: p + len(blk)] = torch.tensor(blk, dtype=row.dtype)
        for _s in range(ri(0, 2) if rnd() < 0.5 else 0):         # stray sentinels
            row[ri(0, S)] = list(t.values())[ri(0, 6)]
        rows.append(row)
    return rows


def recover_map(ids, emb_out, tok_emb, pooled, frames):
    """Which source produced each row of the reference's inputs_embeds (exact float equality; the candidates are bit-exact)."""
    S = ids.shape[0]
    m = torch.full((S,), -2, dtype=torch.int32)
    for s in range(S):
        row = emb_out[s]
        if torch.equal(row, tok_emb[ids[s]]):
            m[s] = -1
            continue
        hit = (pooled == row).all(-1).nonzero()
        if len(hit):
            m[s] = int(hit[0])
            continue
        hit = (frames == row).all(-1).nonzero()
        assert len(hit), ("unexplained row", s)
        m[s] = 256 + int(hit[0])
    return m


@torch.no_grad()
def main():
    spec = dataclasses.replace(syn.TINY, name="tiny-fuzz", vit_layers=1, num_hidden_layers=1, mm_vision_select_layer=-1)
    sd = syn.make_state_dict(spec, 0)
    with tempfile.TemporaryDirectory() as tmp:
        ref = G.build_reference(spec, sd, tmp)
        tk = syn.sentinel_ids(spec)
        tok = O.SentinelIds(tk["im_patch_token"], tk["im_start_token"], tk["im_end_token"], tk["vi_frame_token"], tk["vi_start_token"], tk["vi_end_token"])
        px = syn.make_pixels(1, T, 0)
        feats = O.encode_images(sd, px, -1, num_layers=1)[0]                 # [T,257,H]; bit-exact with the reference (make_golden.py)
        pooled, frames = feats[:, 1:].mean(0), feats[:, 0]
        tok_emb = sd["model.embed_tokens.weight"]
        grabbed, orig = {}, transformers.LlamaModel.forward

        def spy(self, *a, **k):
            grabbed["e"] = k["inputs_embeds"].clone()
            return orig(self, *a, **k)

        rows = make_rows(spec, N_CASES, T)
        results, kinds = [], {}
        transformers.LlamaModel.forward = spy
        try:
            for i, row in enumerate(rows):
                try:
                    ref(row[None], images=px, use_cache=False)
                    if (row == tok.im_patch_token).sum() == 0:
                        res = ("plain", None)
                        assert torch.equal(grabbed["e"][0], tok_emb[row])
                    else:
                        res = ("map", recover_map(row, grabbed["e"][0], tok_emb, pooled, frames))
                except ValueError as e:
                    res = ("ValueError", str(e))
                except IndexError as e:
                    res = ("IndexError", None)
                results.append(res)
                kinds[res[0]] = kinds.get(res[0], 0) + 1
                # the oracle must do the same thing
                try:
                    if (row == tok.im_patch_token).sum() == 0:
                        mine = ("plain", None)
                    else:
                        emb = O.splice_one(row, tok_emb[row], feats, tok)
                        mine = ("map", recover_map(row, emb, tok_emb, pooled, frames))
                except ValueError as e:
                    mine = ("ValueError", str(e))
                except IndexError:
                    mine = ("IndexError", None)
                assert mine[0] == res[0], (i, mine[0], res[0])
                if res[0] == "map":
                    assert torch.equal(mine[1], res[1]), i
                elif res[0] == "ValueError":
                    assert mine[1] == res[1], (i, mine[1], res[1])
        finally:
            transformers.LlamaModel.forward = orig
    print("reference outcomes:", kinds)
    # int16 holds every id and map entry of the tiny vocabulary and keeps the fixture under 1 MB
    assert max(int(r.abs().max()) for r in rows) < 2 ** 15 and all(k != "map" or int(v.abs().max()) < 2 ** 15 for k, v in results)
    rows = [r.to(torch.int16) for r in rows]
    results = [(k, v.to(torch.int16) if k == "map" else v) for k, v in results]
    torch.save(dict(T=T, rows=rows, results=results), os.path.join(os.path.dirname(HERE), "tests", "golden", "ref_splice_fuzz.pt"))
    print("oracle == reference on", N_CASES, "fuzzed rows; wrote tests/golden/ref_splice_fuzz.pt")


if __name__ == "__main__":
    main()
