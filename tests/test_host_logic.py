"""CPU: the C-ABI library loads, exports every declared symbol, and its HOST logic (the exact integer
splice plan) agrees with the oracle / the reference's golden cases.  No compute call needs a GPU here."""
import ctypes as C
import os
import re

import pytest
import torch

import helpers as Hh
from oracle import valley_oracle as O
from valley_b200 import _lib, synthetic as syn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    hdr = open(os.path.join(ROOT, "include", "valley_b200.h")).read()
    declared = set(re.findall(r"\b(vly_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    for name in sorted(declared):
        assert hasattr(lib, name), f"libvalley_b200.so does not export {name}"
    assert declared <= set(_lib.SIGNATURES), declared - set(_lib.SIGNATURES)
    assert b"sm_100a" in lib.vly_version()


def test_no_cpu_fallback_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from valley_b200.model import ValleyConfig, ValleyLlamaForCausalLM
    with pytest.raises(Exception) as ei:
        ValleyLlamaForCausalLM(ValleyConfig.from_spec(syn.TINY), 0)
    assert "no CUDA device" in str(ei.value) or "CUDA" in str(ei.value)


def plan(ids, T, tokens):
    lib = _lib.load()
    ids = ids.to(torch.int64).contiguous()
    B, S = ids.shape
    smap, iidx = torch.empty(B, S, dtype=torch.int32), torch.empty(B, dtype=torch.int32)
    code = lib.vly_build_splice_map(C.cast(ids.data_ptr(), C.POINTER(C.c_int64)), B, S, T, C.byref(tokens),
                                    C.cast(smap.data_ptr(), C.POINTER(C.c_int32)), C.cast(iidx.data_ptr(), C.POINTER(C.c_int32)))
    return code, smap, iidx


def vly_tokens(spec, **over):
    t = dict(syn.sentinel_ids(spec))
    t.update(over)
    return _lib.VlyTokens(t["im_patch_token"], t["im_start_token"], t["im_end_token"], t["vi_frame_token"], t["vi_start_token"], t["vi_end_token"])


def oracle_map(ids_row, T, tok, H=8):
    """Run the oracle's splice on marker embeddings to recover the source map it implies."""
    S = ids_row.shape[0]
    emb = torch.full((S, H), -1.0)
    feat = torch.zeros(T, 257, H)
    feat[:, 1:, :] = torch.arange(256, dtype=torch.float32)[None, :, None]        # mean over T keeps j
    feat[:, 0, :] = (256 + torch.arange(T, dtype=torch.float32))[:, None]
    out = O.splice_one(ids_row, emb, feat, tok)
    return out[:, 0].round().to(torch.int32)


@pytest.mark.parametrize("T", [1, 3, 8])
def test_splice_plan_equals_oracle_on_golden_cases(T):
    spec = syn.TINY
    tok, t = Hh.oracle_tok(spec), syn.sentinel_ids(spec)
    base = syn.make_prompt_ids(spec, 1, T, 0)[0]
    mid = [t["im_start_token"]] + [t["im_patch_token"]] * 256 + [t["im_end_token"]]
    cases = {
        "plain_video": base,
        "video_fallback_count": torch.where(torch.arange(base.numel()) == int((base == t["vi_frame_token"]).nonzero()[0]), torch.tensor(5), base),
        "two_images": torch.cat([base, torch.tensor(mid), torch.tensor([9, 10])]),
        "image_only": torch.cat([torch.tensor([1, 11, 12]), torch.tensor(mid), torch.tensor([13, 14, 15])]),
        "vi_end_misplaced": torch.where(torch.arange(base.numel()) == int((base == t["vi_end_token"]).nonzero()[0]), torch.tensor(6), base),
    }
    for name, row in cases.items():
        code, smap, iidx = plan(row[None], T, vly_tokens(spec))
        assert code == 0, (name, _lib.load().vly_last_error())
        assert iidx[0] == 0
        assert torch.equal(smap[0], oracle_map(row, T, tok)), name


def test_splice_plan_mixed_batch_and_unset_video_tokens():
    spec = syn.TINY
    T = 3
    base = syn.make_prompt_ids(spec, 1, T, 0)[0]
    plain = torch.randint(3, spec.vocab_size - 8, base.shape, generator=torch.Generator().manual_seed(5))
    code, smap, iidx = plan(torch.stack([plain, base, plain, base]), T, vly_tokens(spec))
    assert code == 0 and iidx.tolist() == [-1, 0, -1, 1]            # cur_image_idx advances only for multimodal rows
    assert (smap[0] == -1).all() and (smap[2] == -1).all() and torch.equal(smap[1], smap[3])
    # vi_* ids never set on vision_tower.config -> AttributeError in the reference -> image-only result
    code, smap2, _ = plan(base[None], T, vly_tokens(spec, vi_frame_token=-1, vi_start_token=-1, vi_end_token=-1))
    assert code == 0 and smap2.max() == 255 and (smap2 >= 0).sum() == 256


def test_splice_plan_errors_match_reference_messages():
    spec = syn.TINY
    t = syn.sentinel_ids(spec)
    base = syn.make_prompt_ids(spec, 1, 3, 0)[0]
    lib = _lib.load()
    unbalanced = base.clone()
    unbalanced[(unbalanced == t["im_end_token"]).nonzero()[0]] = 7
    code, _, _ = plan(unbalanced[None], 3, vly_tokens(spec))
    assert code == _lib.VLY_ERR_IM_COUNT and lib.vly_last_error() == b"The number of im_start_token and im_end_token should be the same"
    with pytest.raises(ValueError):
        _lib.check(code)
    cut = torch.cat([unbalanced, torch.tensor([t["im_end_token"]])])
    code, _, _ = plan(cut[None], 3, vly_tokens(spec))
    assert code == _lib.VLY_ERR_IM_CUT and lib.vly_last_error() == b"Seems that the image is cut."
    short = base[: int((base == t["im_start_token"]).nonzero()[0]) + 100].clone()
    short[-1] = t["im_end_token"]                                   # counts balanced, block runs past the row
    code, _, _ = plan(short[None], 3, vly_tokens(spec))
    assert code == _lib.VLY_ERR_INDEX
    with pytest.raises(IndexError):
        _lib.check(code)
    g = torch.load(os.path.join(os.path.dirname(__file__), "golden", "ref_tiny.pt"))
    for case, d in g["errors"].items():                              # the reference's own failing inputs
        code, _, _ = plan(d["ids"], 3, vly_tokens(spec))
        assert code < 0 and lib.vly_last_error().decode() == d["message"], case


def test_empty_and_degenerate_inputs():
    spec = syn.TINY
    code, smap, iidx = plan(torch.zeros(0, 5, dtype=torch.int64), 3, vly_tokens(spec))
    assert code == 0
    code, smap, iidx = plan(torch.full((2, 4), 5, dtype=torch.int64), 0, vly_tokens(spec))
    assert code == 0 and (smap == -1).all() and iidx.tolist() == [-1, -1]


@pytest.mark.parametrize("h,w", [(360, 640), (640, 360), (256, 340), (300, 256), (200, 150), (224, 224), (720, 1280), (255, 257),
                                 (481, 853), (1080, 1920), (257, 255), (2160, 3840), (258, 258)])
def test_preprocess_plan_and_tables_match_oracle(h, w):
    """Host side of vly_preprocess_frames (no GPU): resized size, crop origin and Pillow's fixed-point tables, exact."""
    import numpy as np
    from oracle import preprocess_oracle as P
    from valley_b200 import video
    nh, nw, cy, cx = video.preprocess_plan(h, w)
    assert (nh, nw) == P.resize_sizes(h, w)
    assert (cy, cx) == P.crop_origin(nh, nw)
    for n_in, n_out in ((h, nh), (w, nw)):
        k, xmin, cnt, kk = video.resample_coeffs(n_in, n_out)
        ok, oxmin, ocnt, okk = P.bilinear_coeffs(n_in, n_out)
        assert k == ok and np.array_equal(xmin, oxmin) and np.array_equal(cnt, ocnt) and np.array_equal(kk, okk)


def test_frame_index_selection_matches_oracle():
    import numpy as np
    from oracle import preprocess_oracle as P
    from valley_b200 import video
    for n in (1, 7, 8, 9, 100, 1234):
        assert np.array_equal(video.fixed_frame_indices(n), P.fixed_frame_indices(n))
        assert np.array_equal(video.fixed_frame_indices(n), np.linspace(0, n - 1, 8).astype(np.int_))
    for n, fps in ((300, 29.97), (50, 24.0), (1000, 59.94)):
        assert np.array_equal(video.fps_frame_indices(n, fps), P.fps_frame_indices(n, fps))
    with pytest.raises(ValueError):
        video.preprocess_plan(0, 10)


def _write_checkpoint(tmp, spec, sd, fmt):
    """HF save_pretrained layout: config.json (+ a local CLIP config dir) and two weight shards with an index."""
    import json
    import os
    vt = os.path.join(tmp, "clip")
    os.makedirs(vt, exist_ok=True)
    json.dump(dict(hidden_size=spec.vit_hidden, intermediate_size=spec.vit_mlp, num_hidden_layers=spec.vit_layers,
                   num_attention_heads=spec.vit_heads, image_size=spec.vit_image, patch_size=spec.vit_patch, layer_norm_eps=spec.vit_eps),
              open(os.path.join(vt, "config.json"), "w"))
    json.dump(dict(architectures=["ValleyLlamaForCausalLM"], model_type="valley", hidden_size=spec.hidden_size,
                   num_hidden_layers=spec.num_hidden_layers, num_attention_heads=spec.num_attention_heads,
                   intermediate_size=spec.intermediate_size, vocab_size=spec.vocab_size, rms_norm_eps=spec.rms_norm_eps,
                   max_position_embeddings=spec.max_position_embeddings, mm_vision_tower=vt, mm_vision_select_layer=spec.mm_vision_select_layer,
                   use_mm_proj=True, mm_hidden_size=spec.vit_hidden, mm_use_im_start_end=True, torch_dtype="float16"),
              open(os.path.join(tmp, "config.json"), "w"))
    names = list(sd)
    halves = [names[: len(names) // 2], names[len(names) // 2:]]
    wm = {}
    for i, part in enumerate(halves):
        if fmt == "safetensors":
            from safetensors.torch import save_file
            fn = f"model-{i + 1:05d}-of-00002.safetensors"
            save_file({k: sd[k].contiguous() for k in part}, os.path.join(tmp, fn))
        else:
            fn = f"pytorch_model-{i + 1:05d}-of-00002.bin"
            torch.save({k: sd[k] for k in part}, os.path.join(tmp, fn))
        wm.update({k: fn for k in part})
    idx = "model.safetensors.index.json" if fmt == "safetensors" else "pytorch_model.bin.index.json"
    json.dump(dict(metadata={}, weight_map=wm), open(os.path.join(tmp, idx), "w"))


@pytest.mark.parametrize("fmt", ["safetensors", "bin"])
def test_checkpoint_directory_reader(tmp_path, fmt):
    """from_pretrained's host side: config.json (+ CLIP geometry from a local tower dir) and sharded weights, streamed by name."""
    from valley_b200 import checkpoint
    from valley_b200.model import ValleyConfig
    spec = syn.TINY
    sd = {k: v.half() for k, v in syn.make_state_dict(spec, 0).items()}
    _write_checkpoint(str(tmp_path), spec, sd, fmt)
    cfg = ValleyConfig(**checkpoint.read_config(str(tmp_path)))
    assert (cfg.hidden_size, cfg.num_hidden_layers, cfg.vit_layers, cfg.vit_heads, cfg.vocab_size) == (512, 2, 3, 16, 1032)
    assert cfg.patch_pooling_method == "mean" and cfg.mm_vision_select_layer == -2
    got = dict(checkpoint.iter_checkpoint(str(tmp_path)))
    assert set(got) == set(sd) and all(torch.equal(got[k], sd[k]) for k in sd)
    assert len(checkpoint.weight_files(str(tmp_path))) == 2
    with pytest.raises(FileNotFoundError):
        checkpoint.weight_files(str(tmp_path / "clip"))


def test_lora_adapter_is_merged_into_the_streamed_weights(tmp_path):
    """run_valley.py:26-37 (merge_and_unload): W + (B @ A) * lora_alpha / r on the adapted projections, everything else untouched."""
    import json
    import os
    from safetensors.torch import save_file
    from valley_b200 import checkpoint
    spec = syn.TINY
    sd = syn.make_state_dict(spec, 0)
    base = tmp_path / "base"
    base.mkdir()
    _write_checkpoint(str(base), spec, sd, "safetensors")
    lora = tmp_path / "valley-lora"
    lora.mkdir()
    g = torch.Generator().manual_seed(9)
    r, alpha, H, I = 16, 32, spec.hidden_size, spec.intermediate_size
    targets = {"model.layers.0.self_attn.q_proj": (H, H), "model.layers.1.mlp.down_proj": (H, I), "model.layers.1.mlp.up_proj": (I, H)}
    ad = {}
    for mod, (o, i) in targets.items():
        ad[f"base_model.model.{mod}.lora_A.weight"] = torch.randn(r, i, generator=g) * 0.05
        ad[f"base_model.model.{mod}.lora_B.weight"] = torch.randn(o, r, generator=g) * 0.05
    save_file(ad, str(lora / "adapter_model.safetensors"))
    json.dump(dict(r=r, lora_alpha=alpha, base_model_name_or_path=str(base), target_modules=list(targets), peft_type="LORA"),
              open(lora / "adapter_config.json", "w"))
    assert checkpoint.is_lora_dir(str(lora)) and not checkpoint.is_lora_dir(str(base))
    assert checkpoint.resolve_lora_base(str(lora)) == str(base)
    merged = dict(checkpoint.iter_checkpoint_merged(str(base), str(lora)))
    assert set(merged) == set(sd)
    for name, w in sd.items():
        mod = name[: -len(".weight")] if name.endswith(".weight") else None
        if mod in targets:
            want = w.double() + (ad[f"base_model.model.{mod}.lora_B.weight"].double() @ ad[f"base_model.model.{mod}.lora_A.weight"].double()) * (alpha / r)
            assert torch.allclose(merged[name].double(), want, rtol=1e-5, atol=1e-6) and not torch.equal(merged[name], w)
        else:
            assert torch.equal(merged[name], w), name
    # an adapter for a weight the base does not have is an error, not a silent no-op
    ad["base_model.model.model.layers.7.self_attn.q_proj.lora_A.weight"] = torch.zeros(r, H)
    ad["base_model.model.model.layers.7.self_attn.q_proj.lora_B.weight"] = torch.zeros(H, r)
    save_file(ad, str(lora / "adapter_model.safetensors"))
    with pytest.raises(KeyError):
        list(checkpoint.iter_checkpoint_merged(str(base), str(lora)))


def test_ctypes_structs_match_the_c_header(tmp_path):
    """The ctypes mirrors in valley_b200/_lib.py must have the layout gcc gives the structs of include/valley_b200.h
    (a silent mismatch would scramble every config field / sampling parameter)."""
    import ctypes as C
    import os
    import shutil
    import subprocess
    from valley_b200 import _lib
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    structs = {"vly_config": _lib.VlyConfig, "vly_tokens": _lib.VlyTokens, "vly_sampling": _lib.VlySampling}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "valley_b200.h"', "int main(void) {"]
    for cname, ct in structs.items():
        lines.append(f'  printf("{cname} size %zu\\n", sizeof({cname}));')
        for fname, _ in ct._fields_:
            lines.append(f'  printf("{cname} {fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "abi_probe.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "abi_probe"
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split("\n")
    got = {tuple(l.split()[:2]): int(l.split()[2]) for l in out if l}
    for cname, ct in structs.items():
        assert got[(cname, "size")] == C.sizeof(ct), cname
        for fname, _ in ct._fields_:
            assert got[(cname, fname)] == getattr(ct, fname).offset, (cname, fname)
    # enum values used across the boundary
    assert (_lib.VLY_F32, _lib.VLY_BF16, _lib.VLY_F16) == (0, 1, 2)
    assert _lib.POOLING == {"mean": 0, "max": 1, "temporal_importance": 2, "temporal_transformer": 3}


def test_prompt_helpers_and_config_flags():
    """Pure string / config logic of the reference surface (no GPU): valley_model.py:381-422, :40-52; model_worker.py:338-368."""
    from valley_b200 import serving
    from valley_b200.model import ValleyConfig, ValleyLlamaForCausalLM
    # pooling variant selection: the later flag wins (valley_model.py:40-52 sets the attribute in that order)
    assert ValleyConfig().patch_pooling_method == "mean"
    assert ValleyConfig(use_patch_importance_pooling=True).patch_pooling_method == "temporal_importance"
    assert ValleyConfig(use_patch_importance_pooling=True, use_delta_transformer=True).patch_pooling_method == "temporal_transformer"
    with pytest.raises(ValueError):
        ValleyConfig(patch_pooling_method="median")
    assert ValleyConfig(some_hf_key=3).some_hf_key == 3                      # unknown HF config keys are kept, not rejected
    # <video> expansion (model_worker.py:338-341)
    p = serving.expand_video_prompt("a <video> b", 3, True)
    assert p == "a <im_start>" + "<im_patch>" * 256 + "<im_end><vi_start>" + "<vi_frame>" * 3 + "<vi_end> b"
    assert serving.expand_video_prompt("a <video> b", 3, False) == "a " + "<im_patch>" * 256 + " b"
    # left truncation (model_worker.py:367-368)
    ids = list(range(3000))
    assert serving.truncate_source(ids, 2048, 256) == ids[-(2048 - 256 - 8):]
    assert serving.truncate_source(ids[:100], 2048, 256) == ids[:100]
    # process_response (valley_model.py:405-422) needs no model state
    pr = ValleyLlamaForCausalLM.process_response
    assert pr(None, ["### Assistant: hello there ### Human: x"]) == ["hello there"]
    assert pr(None, ["Valley: Response: ok"]) == ["ok"]
    assert pr(None, ["   plain"]) == ["plain"]


def test_splice_plan_and_oracle_match_the_reference_on_fuzzed_rows():
    """400 random rows with well-formed / corrupted / truncated / misplaced <im_*> and <vi_*> blocks, each one pushed through the
    LIVE reference by oracle/make_golden_splice_fuzz.py: the C host plan and the oracle must do exactly what the reference did --
    same source map, or the same exception (type and message)."""
    g = torch.load(os.path.join(os.path.dirname(__file__), "golden", "ref_splice_fuzz.pt"))
    spec, T = syn.TINY, g["T"]
    tok, lib = Hh.oracle_tok(spec), _lib.load()
    seen = {}
    for i, (row, (kind, val)) in enumerate(zip(g["rows"], g["results"])):
        row = row.long()                                             # stored as int16 to keep the fixture small
        if kind == "map":
            val = val.int()
        seen[kind] = seen.get(kind, 0) + 1
        code, smap, iidx = plan(row[None], T, vly_tokens(spec))
        if kind == "plain":
            assert code == 0 and int(iidx[0]) == -1 and bool((smap == -1).all()), i
        elif kind == "map":
            assert code == 0 and int(iidx[0]) == 0, (i, lib.vly_last_error())
            assert torch.equal(smap[0], val), i
            assert torch.equal(oracle_map(row, T, tok), val), i
        elif kind == "ValueError":
            assert code in (_lib.VLY_ERR_IM_COUNT, _lib.VLY_ERR_IM_CUT) and lib.vly_last_error().decode() == val, (i, code, val)
            with pytest.raises(ValueError) as ei:
                oracle_map(row, T, tok)
            assert str(ei.value) == val, i
        else:
            assert kind == "IndexError" and code == _lib.VLY_ERR_INDEX, (i, code)
            with pytest.raises(IndexError):
                oracle_map(row, T, tok)
    assert seen["map"] >= 40 and seen["ValueError"] >= 100 and seen["IndexError"] >= 10 and seen["plain"] >= 50


def test_load_video_directory_of_images_branch_equals_the_reference(tmp_path):
    """load_video's directory branch (data_util.py:282-302: rglob, linspace selection, PIL open, optional square resize,
    CLIPImageProcessor) -- host code, no GPU.  The fixture (oracle/make_golden_imgdir.py, written from the LIVE reference) holds
    the SHA-256 of every frame the reference produced, keyed by file name: the directory order is whatever the file system
    returns, so the check is per selected file."""
    import hashlib
    import importlib.util
    import numpy as np
    from valley_b200 import video
    here = os.path.dirname(__file__)
    g = torch.load(os.path.join(here, "golden", "ref_imgdir.pt"))
    spec = importlib.util.spec_from_file_location("make_golden_imgdir_images", os.path.join(os.path.dirname(here), "oracle", "make_golden_imgdir.py"))
    src = open(spec.origin).read()
    ns = {}
    # only the image generator of the script (its module-level imports need /root/reference): the function is self-contained
    start, end = src.index("def make_images"), src.index("def sha(")
    from PIL import Image
    exec(src[start:end], {"np": np, "Image": Image, "os": os, "SIZES": g["sizes"]}, ns)
    for method, sizes, seed0 in (("centercrop", g["sizes"], 500), ("resize", g["same"], 700)):
        d = tmp_path / method
        d.mkdir()
        names = ns["make_images"](str(d), sizes, seed0)
        for n_fixed in sorted({3, len(names)}):
            picked = video.select_image_dir_frames(str(d), "fixed", n_fixed)
            assert len(picked) == n_fixed and {p.name for p in picked} <= set(names)
            out = video.load_image_dir(str(d), None, "fixed", n_fixed, method)
            assert out.shape == (n_fixed, 3, 224, 224) and out.dtype == torch.float32
            for k, p in enumerate(picked):
                want = g["frames"][(method, p.name)]
                assert torch.equal(out[k].flatten()[::997], want["sample"]), (method, p.name)
                assert hashlib.sha256(out[k].contiguous().numpy().tobytes()).hexdigest() == want["sha256"], (method, p.name)
    with pytest.raises(ValueError, match="Input folder is not support this frame mode"):
        video.load_image_dir(str(tmp_path / "centercrop"), None, "fps")
    with pytest.raises(ValueError, match='Frame mode is only support "fps" or "fixed"'):
        video.load_image_dir(str(tmp_path / "centercrop"), None, "other")


def test_keywords_stopping_criteria_matches_the_reference_semantics():
    """valley/util/data_util.py:40-56: the FIRST call only records the prompt length (the first generated token is never tested
    alone), later calls decode row 0 of output_ids[:, start_len:] and stop on any keyword.  Pure host logic."""
    from valley_b200.model import KeywordsStoppingCriteria

    class Tok:
        def batch_decode(self, ids, skip_special_tokens=True):
            return ["".join(chr(int(t)) for t in row) for row in ids]

    prompt = torch.tensor([[ord(c) for c in "ab"]])
    crit = KeywordsStoppingCriteria(["###"], Tok(), prompt)
    grow = lambda s: torch.tensor([[ord(c) for c in "ab" + s]])
    assert crit(grow("###")) is False                 # first call: start_len recorded, nothing tested (the reference's quirk)
    assert crit.start_len == 2
    assert crit(grow("x#")) is False
    assert crit(grow("x##")) is False
    assert crit(grow("x###")) is True
    assert crit(grow("###y"), scores=None) is True
    two = KeywordsStoppingCriteria(["STOP", "\n\n"], Tok(), prompt)
    two(grow(""))
    assert two(grow("abc\n\n")) is True and two(grow("abc\n")) is False
