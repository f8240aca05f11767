"""Generate golden vectors by running the UNMODIFIED reference (/root/reference)
on CPU in fp32.  Run once in the build container:

    python tests/golden/gen_golden.py

Outputs (committed, small):
  tests/golden/dit_c1.pt       — config C1 (SURVEY §8d): hidden 256, 2 heads x128, inner 512,
                                 1 layer, text_dim 64, b=2, latent t=4,h=w=16 (N=384).
                                 state_dict (bf16-representable fp32 stored as bf16), inputs,
                                 per-stage reference outputs (patch-embed tokens, block output,
                                 final output).
  tests/golden/dit_index.pt    — integer-coded index maps: patchify order, unpatchify scatter,
                                 the three RoPE tables (incl. the pooled, W-shifted pose table).
  tests/golden/sampler.pt      — sigma schedule make_flow_timesteps(0,50,shift 5), CFG+Euler step.
  tests/golden/vae_small.pt    — WanVAE_ decode of a [1,16,3,8,8] latent (dim=16 narrow variant
                                 of the same architecture), state_dict + output.
  tests/golden/mixin_surface.json — the reference's DiffusionTransformer built with its mixin targets
                                 pointed at scail_b200.dit: mixin classes, hook origins, parameter shapes.
The GPU box never runs this (no /root/reference there); tests read the .pt files.
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_harness as H  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def bf16_sd(model):
    return {k: v.detach().to(torch.bfloat16).clone() for k, v in model.state_dict().items()}


def c1_inputs(seed=0, b=2, t=4, h=16, w=16, text_dim=64, L=32):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g).to(torch.bfloat16).float()
    ctx = r(b, L, text_dim)
    ctx[0, 1:] = 0  # uncond: empty prompt, only EOS row survives the UMT5 mask (SURVEY §8d)
    ctx[1, 20:] = 0
    return dict(
        x=r(b, t, 16, h, w), ref_concat=r(1, 1, 16, h, w), concat_smpl_render=r(1, t, 16, h // 2, w // 2),
        concat_images=torch.zeros(1, t, 16, h, w), context=ctx, image_clip_features=r(1, 257, 1280),
        timesteps=torch.tensor([500.0, 500.0]),
    )


@torch.no_grad()
def gen_dit():
    model = H.build_reference_dit(seed=1234, hidden=256, heads=2, inner=512, layers=1, text_dim=64)
    inp = c1_inputs()
    cap = {}
    pe = model.mixins["patch_embed"]
    ad = model.mixins["adaln_layer"]
    orig_we, orig_lf = pe.word_embedding_forward, ad.layer_forward

    def we(*a, **k):
        o = orig_we(*a, **k)
        cap["tokens"] = o.clone()
        return o

    def lf(hs, mask, *a, **k):
        o = orig_lf(hs, mask, *a, **k)
        cap.setdefault("block_out", []).append(o.clone())
        for key in ("emb", "final_layer_emb", "encoder_outputs", "image_clip_features"):
            cap[key] = k[key].clone()
        return o

    model.hooks["word_embedding_forward"] = we
    model.hooks["layer_forward"] = lf
    out = model(inp["x"], timesteps=inp["timesteps"], context=inp["context"], y=None,
                concat_images=inp["concat_images"], ref_concat=inp["ref_concat"],
                concat_smpl_render=inp["concat_smpl_render"], image_clip_features=inp["image_clip_features"])
    assert "tokens" in cap and "block_out" in cap, "capture hooks were not called"
    torch.save({"cfg": dict(hidden=256, heads=2, inner=512, layers=1, text_dim=64, max_frames=21, max_h=150, max_w=150),
                "state_dict": bf16_sd(model), "inputs": inp, "tokens": cap["tokens"],
                "block_out": cap["block_out"][0], "adaln_emb": cap["emb"], "time_emb": cap["final_layer_emb"],
                "text_ctx": cap["encoder_outputs"], "clip_ctx": cap["image_clip_features"], "out": out},
               os.path.join(OUT, "dit_c1.pt"))
    print("dit_c1: out", tuple(out.shape), float(out.abs().mean()))

    # ---- integer-coded index maps -------------------------------------------------
    import dit_video_crossattn_sc_xc as ref
    from einops import rearrange

    b, t, h, w = 1, 3, 8, 12
    # patchify: feed a conv whose weight copies input element (c=0, p, q) id into 4 output channels
    def ids(tt, hh, ww, base):
        return (base + torch.arange(tt * hh * ww, dtype=torch.float32)).reshape(1, tt, 1, hh, ww)

    img_ids, ref_ids, pose_ids = ids(t, h, w, 0), ids(1, h, w, 100000), ids(t, h // 2, w // 2, 200000)
    pe2 = ref.ImagePatchEmbeddingMixin(1, 4, (1, 2, 2))
    for conv in (pe2.proj, pe2.proj_pose):
        conv.weight.zero_(); conv.bias.zero_()
        for o in range(4):
            conv.weight[o, 0, 0, o // 2, o % 2] = 1.0
    tok_ids = pe2.word_embedding_forward(None, images=img_ids, ref_concat=ref_ids, concat_smpl_render=pose_ids)
    # unpatchify: token n, feature f -> value n*64+f
    n_ref, n_seq, n_pose = h * w // 4, t * h * w // 4, t * (h // 2) * (w // 2) // 4
    N = n_ref + n_seq + n_pose
    code = (torch.arange(N)[:, None] * 64 + torch.arange(64)[None]).float()[None]
    unp = ref.unpatchify(code, c=16, patch_size=(1, 2, 2), w=w // 2, h=h // 2, ref_length=n_ref,
                         seq_length=n_seq, rope_T=t, rope_H=h // 2, rope_W=w // 2)
    # rope tables through the reference mixin, applied to all-ones / unit vectors
    rp = ref.Rotary3DPositionEmbeddingMixin(150, 150, 21, 256, 128, interleaved_rope=True)
    kw = dict(rope_T=t, rope_H=h // 2, rope_W=w // 2, rope_H_shift=0, rope_W_shift=0, global_rope_H=0,
              global_rope_W=120, ref_length=n_ref, seq_length=n_seq, pose_length=n_pose)
    ones = torch.ones(1, 1, N, 128)
    # t*cos + rotate_half(t)*sin with t = ones: even idx -> cos - sin, odd idx -> cos + sin
    rot = rp.attention_fn(ones, ones, ones, None, old_impl=lambda q, k, v, m, **kk: (q, k), **kw)
    q_rot = rot[0]
    cos = 0.5 * (q_rot[..., 0::2] + q_rot[..., 1::2])  # both halves of a pair share the angle
    sin = 0.5 * (q_rot[..., 1::2] - q_rot[..., 0::2])
    torch.save({"geom": dict(t=t, h=h, w=w), "tok_ids": tok_ids.to(torch.int64), "unpatchify": unp.to(torch.int64),
                "rope_cos_pairs": cos[0, 0], "rope_sin_pairs": sin[0, 0]}, os.path.join(OUT, "dit_index.pt"))
    print("dit_index: tok_ids", tuple(tok_ids.shape), "unp", tuple(unp.shape))

    # ---- sampler bits ----------------------------------------------------------------
    from sgm.modules.diffusionmodules.sampling import make_flow_timesteps
    from sgm.modules.diffusionmodules.guiders import VanillaCFG

    sig = make_flow_timesteps(0, 50, verbose=False, shift_scale=5, mode="normal")
    g = torch.Generator().manual_seed(3)
    x = torch.randn(1, 4, 16, 8, 8, generator=g)
    v = torch.randn(2, 4, 16, 8, 8, generator=g)
    guided = VanillaCFG(scale=4)(v, sig[3])
    x_next = x + (sig[4] - sig[3]) * guided
    torch.save({"sigmas": sig, "x": x, "v": v, "x_next": x_next, "i": 3}, os.path.join(OUT, "sampler.pt"))


@torch.no_grad()
def gen_vae():
    res = {}
    for tag, dim, shape in (("narrow", 16, (1, 16, 3, 8, 8)),):
        vae = H.build_reference_vae(seed=7, dim=dim)
        g = torch.Generator().manual_seed(11)
        z = torch.randn(*shape, generator=g).to(torch.bfloat16).float()
        scale = [torch.tensor(H.VAE_MEAN), 1.0 / torch.tensor(H.VAE_STD)]
        out = vae.decode(z, scale).float().clamp_(-1, 1)
        sd = {k: v.to(torch.bfloat16) for k, v in vae.state_dict().items()
              if k.startswith("decoder.") or k.startswith("conv2.")}
        res[tag] = {"dim": dim, "z": z, "out": out, "state_dict": sd}
        # encode path (SURVEY §8f rank 2): video [1,3,9,32,32] -> mu [1,16,3,4,4]
        video = torch.randn(1, 3, 9, 32, 32, generator=g).clamp(-1, 1).to(torch.bfloat16).float()
        mu = vae.encode(video, scale).float()
        esd = {k: v.to(torch.bfloat16) for k, v in vae.state_dict().items()
               if k.startswith("encoder.") or k.startswith("conv1.")}
        torch.save({"dim": dim, "video": video, "mu": mu, "state_dict": esd}, os.path.join(OUT, "vae_encode_small.pt"))
        print("vae encode", tag, tuple(mu.shape), float(mu.abs().mean()))
        print("vae", tag, tuple(out.shape), float(out.abs().mean()))
    torch.save(res["narrow"], os.path.join(OUT, "vae_small.pt"))
    return res


def gen_mixin_surface():
    """What the reference's own DiffusionTransformer makes of scail_b200.dit when the YAML `target:` strings point at it:
    the module and class of every mixin it instantiated, the mixin each SAT hook was collected from
    (BaseModel.collect_hooks_), and the stock model's parameter shapes (which the plugged-in model must reproduce)."""
    import importlib
    import json
    H.setup()
    import dit_video_crossattn_sc_xc as ref
    import scail_b200.dit as ours
    importlib.reload(ours)  # real SAT BaseMixins now that SAT is importable
    cfg = dict(hidden=256, heads=2, inner=512, layers=1, text_dim=64)
    stock = ref.DiffusionTransformer(**H.dit_config(**cfg))
    mine = ref.DiffusionTransformer(**H.dit_config(mixin_module="scail_b200.dit", **cfg))
    shapes = {k: list(v.shape) for k, v in stock.state_dict().items()}
    assert {k: list(v.shape) for k, v in mine.state_dict().items()} == shapes
    surface = {"config": cfg, "param_shapes": shapes,
               "mixins": {k: [type(m).__module__, type(m).__name__] for k, m in mine.mixins.items()},
               "hook_origins": dict(mine.hook_origins)}
    with open(os.path.join(OUT, "mixin_surface.json"), "w") as f:
        json.dump(surface, f, indent=1, sort_keys=True)
        f.write("\n")
    print("mixin surface:", surface["hook_origins"])


if __name__ == "__main__":
    which = sys.argv[1:] or ["dit", "vae", "mixins"]
    if "dit" in which:
        gen_dit()
    if "vae" in which:
        gen_vae()
    if "mixins" in which:
        gen_mixin_surface()
