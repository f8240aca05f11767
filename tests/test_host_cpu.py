"""CPU tests of the host side: the C-ABI library loads and exports every declared symbol, the product path
refuses to run without CUDA (no CPU fallback), RoPE tables are bit-identical to the oracle, parameter names match
the reference's, and the mixins present the surface the reference's own DiffusionTransformer accepted through the
YAML `target:` plug-in mechanism (recorded in tests/golden/mixin_surface.json)."""
import os
import re
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_cabi_exports_every_declared_symbol():
    from scail_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "scail_b200.h")).read()
    declared = set(re.findall(r"^(?:int|const char\*)\s+(scail_\w+)\s*\(", hdr, flags=re.M))
    assert len(declared) >= 18
    h = _lib.lib()
    for name in declared:
        assert hasattr(h, name), name
    assert declared - {"scail_last_error"} == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert h.scail_version() == 100


def test_no_cpu_fallback():
    from scail_b200 import ops
    from scail_b200.dit import DiffusionTransformer
    from scail_b200.wan_vae import WanVAE
    with pytest.raises(RuntimeError):
        ops.gemm(torch.zeros(8, 8, dtype=torch.bfloat16), torch.zeros(8, 8, dtype=torch.bfloat16))
    m = DiffusionTransformer(hidden_size=256, num_attention_heads=2, inner_hidden_size=512, num_layers=1, text_dim=64,
                             time_embed_dim=256)
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 2, 16, 8, 8), timesteps=torch.zeros(1), context=torch.zeros(1, 4, 64),
          ref_concat=torch.zeros(1, 1, 16, 8, 8), concat_smpl_render=torch.zeros(1, 2, 16, 4, 4),
          image_clip_features=torch.zeros(1, 257, 1280))
    v = WanVAE(dim=16, device="cpu")
    with pytest.raises(RuntimeError):
        v.decode([torch.zeros(16, 1, 4, 4)])
    if not torch.cuda.is_available():  # without a device the library itself reports the failure
        from scail_b200 import _lib
        assert _lib.lib().scail_device_sm_count(0) < 0
        assert b"CUDA" in _lib.lib().scail_last_error()


def test_product_does_not_import_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "scail_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f
                assert "import baseline" not in src and "from baseline" not in src, f  # the library-path arm is bench-only


def test_rope_tables_bit_identical_to_oracle():
    from oracle import dit_oracle as O
    from scail_b200 import rope
    for (T, H, W) in [(3, 4, 6), (4, 8, 8), (21, 32, 32)]:
        c, s = rope.build_tables_cpu(128, T, H, W)
        c2, s2 = O.rope_tables(128, T, H, W, 21, 150, 150)
        assert torch.equal(c, c2) and torch.equal(s, s2)
    c, s = rope.build_tables_cpu(128, 2, 4, 4, 2, 4)  # SP-style shifts (dit_video_crossattn_sc_xc.py:1578-1585)
    c2, s2 = O.rope_tables(128, 2, 4, 4, 21, 150, 150, h_shift=2, w_shift=4)
    assert torch.equal(c, c2) and torch.equal(s, s2)


def test_state_dict_names_match_reference_golden():
    from scail_b200.dit import DiffusionTransformer
    from scail_b200.wan_vae import WanVAE
    g = torch.load(os.path.join(GOLD, "dit_c1.pt"))
    cfg = g["cfg"]
    m = DiffusionTransformer(hidden_size=cfg["hidden"], num_attention_heads=cfg["heads"], inner_hidden_size=cfg["inner"],
                             num_layers=cfg["layers"], text_dim=cfg["text_dim"], time_embed_dim=cfg["hidden"])
    ours = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    ref = {k: tuple(v.shape) for k, v in g["state_dict"].items()}
    assert ours == ref
    gv = torch.load(os.path.join(GOLD, "vae_small.pt"))
    v = WanVAE(dim=gv["dim"], device="cpu")
    ours = {k: tuple(t.shape) for k, t in v.model.state_dict().items()}
    ge = torch.load(os.path.join(GOLD, "vae_encode_small.pt"))
    ref = {k: tuple(t.shape) for k, t in gv["state_dict"].items()}
    ref.update({k: tuple(t.shape) for k, t in ge["state_dict"].items()})
    assert ours == ref  # decoder.* + conv2.* (decode) and encoder.* + conv1.* (encode): the whole Wan2.1_VAE.pth layout


def test_sampler_schedule_matches_golden():
    from scail_b200 import sampler
    s = torch.load(os.path.join(GOLD, "sampler.pt"))
    assert torch.equal(sampler.make_flow_timesteps(50, 5.0), s["sigmas"])


def test_bench_flop_model():
    sys.path.insert(0, ROOT)
    import bench
    assert bench.seq_len() == 27904
    assert abs(bench.block_flops(27904) / 1e12 - 33.144) < 0.01          # BASELINE.md table
    assert abs(bench.forward_flops(27904) / 1e12 - 1325.8) < 0.1


def test_mixins_plug_into_reference_model():
    """Golden tests/golden/mixin_surface.json records the reference's DiffusionTransformer built with its YAML target
    strings pointed at scail_b200.dit: instantiate_from_config resolved them to this module's mixin classes,
    BaseModel.collect_hooks_ took the DiT hooks from those mixins, and the model had exactly the stock reference's
    parameter names and shapes.  The mixins and model here must still present that surface."""
    import json
    import scail_b200.dit as ours
    g = json.load(open(os.path.join(GOLD, "mixin_surface.json")))
    c = g["config"]
    m = ours.DiffusionTransformer(hidden_size=c["hidden"], num_attention_heads=c["heads"], inner_hidden_size=c["inner"],
                                  num_layers=c["layers"], text_dim=c["text_dim"], time_embed_dim=c["hidden"])
    assert {k: list(v.shape) for k, v in m.state_dict().items()} == g["param_shapes"]
    plugged = {k for k, (module, _) in g["mixins"].items() if module == ours.__name__}
    assert {"adaln_layer", "patch_embed", "pos_embed", "final_layer"} <= plugged
    for k in plugged:
        assert type(m.mixins[k]) is getattr(ours, g["mixins"][k][1]), k
    for hook in ("word_embedding_forward", "layer_forward", "final_forward", "position_embedding_forward",
                 "attention_forward", "cross_attention_forward"):
        assert g["hook_origins"][hook] in plugged, hook
    for hook, origin in g["hook_origins"].items():
        if origin in plugged:
            assert callable(getattr(m.mixins[origin], hook, None)), (hook, origin)


def test_bench_dump_outputs_within_budget_and_repeatable(tmp_path, monkeypatch):
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 4096)
    small, big = torch.randn(2, 3, 5), torch.randn(1, 21, 16, 8, 8)
    for d in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(str(d), {"small": small, "big": big})
    a, b = np.load(tmp_path / "a" / "small.npy"), np.load(tmp_path / "a" / "big.npy")
    assert a.dtype == np.float32 and np.array_equal(a, small.numpy())
    assert b.dtype == np.float32 and b.nbytes + a.nbytes <= 4096 and np.isin(b, big.numpy()).all()
    assert np.array_equal(b, np.load(tmp_path / "b" / "big.npy"))


def test_bench_reference_arm_json_contract():
    """`bench.py --impl reference` (the CPU arm: oracle port on the host cores, bounded sample) prints one JSON line with
    the contract's keys.  Uses a reduced sample so the CPU suite stays short."""
    import json
    import subprocess
    code = ("import sys, json; sys.argv=['bench.py','--impl','reference','--steps','1','--warmup','0'];"
            "import bench; bench.CPU_ARM_BUDGET_S=0.0; bench.main()")  # budget 0 -> the reduced 9x32x32 sample
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["unit"] == "steps/s" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["e2e"] == {"value": d["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0 and d["config"]["seq_len"] == 27904


def test_sample_long_matches_reference_golden():
    """RFSamplerLong (sampling.py:986-1085) host logic vs the golden produced by the UNMODIFIED reference sampler driving a
    deterministic stand-in network (tests/golden/gen_sampler_long.py): tile scheduling, triangular blend, CFG (incl. the uncond
    padding rule of guiders.py:52-53), Euler update, flow schedule."""
    import sys
    from scail_b200 import sampler
    gdir = os.path.join(os.path.dirname(__file__), "golden")
    sys.path.insert(0, gdir)
    from fake_network import fake_network
    g = torch.load(os.path.join(gdir, "sampler_long.pt"))

    def denoise(x_tile, sigma, c_k, u_k):  # VanillaCFG.prepare_inputs + __call__ around the stand-in network
        ctx = sampler.prepare_context(c_k, u_k)
        both = dict(crossattn=ctx, concat_smpl_render=c_k["concat_smpl_render"])
        v = fake_network(torch.cat([x_tile] * 2), torch.cat([sigma.view(1) * 1000.0] * 2), both)
        vu, vc = v.chunk(2)
        return vu + g["scale"] * (vc - vu)

    out = sampler.sample_long(None, g["x"].clone(), g["cond"], g["uc"], g["tile_indices"], num_steps=g["num_steps"],
                              shift_scale=g["shift_scale"], scale=g["scale"], denoise=denoise)
    assert out.shape == g["out"].shape
    assert torch.allclose(out, g["out"], rtol=0, atol=2e-6), float((out - g["out"]).abs().max())
    assert sampler.make_tile_indices(13, 5, 4) == g["tile_indices"]


def test_checkpoint_layout_roundtrip_and_error_behaviour(tmp_path):
    """SAT checkpoint layout (sat/training/model_io.py:36-48, 233-356): latest -> <iter>/mp_rank_00_model_states.pt ->
    sd['module'] with the engine prefix; missing keys raise unless force_inference, unexpected keys only warn."""
    import pytest
    from scail_b200 import checkpoint as C
    from scail_b200.dit import DiffusionTransformer
    cfg = dict(hidden_size=256, num_attention_heads=2, inner_hidden_size=512, num_layers=1, text_dim=64, time_embed_dim=256)
    torch.manual_seed(0)
    a = DiffusionTransformer(**cfg)
    C.save_checkpoint(a, str(tmp_path), 1000)
    assert open(tmp_path / "latest").read() == "1000" and (tmp_path / "1000" / "mp_rank_00_model_states.pt").is_file()
    torch.manual_seed(1)
    b = DiffusionTransformer(**cfg)
    assert C.load_checkpoint(b, str(tmp_path)) == 1000 and not b.training
    for (k, va), (_, vb) in zip(a.state_dict().items(), b.state_dict().items()):
        assert torch.equal(va, vb), k
    # a checkpoint that lacks a parameter: inference refuses unless forced (model_io.py:303-307)
    sd = torch.load(tmp_path / "1000" / "mp_rank_00_model_states.pt")
    del sd["module"][C.DIT_PREFIX + "mixins.final_layer.linear.bias"]
    sd["module"][C.DIT_PREFIX + "not_a_parameter"] = torch.zeros(1)
    sd["module"]["conditioner.something"] = torch.zeros(1)  # other engine sub-modules are filtered out by the prefix
    torch.save(sd, tmp_path / "1000" / "mp_rank_00_model_states.pt")
    with pytest.warns(UserWarning, match="unexpected_keys"), pytest.raises(ValueError, match="Missing keys for inference"):
        C.load_checkpoint(b, str(tmp_path))
    with pytest.warns(UserWarning):
        assert C.load_checkpoint(b, str(tmp_path), force_inference=True) == 1000
    (tmp_path / "latest").write_text("garbage")
    with pytest.raises(ValueError, match="Invalid metadata"):
        C.load_checkpoint(b, str(tmp_path))
    (tmp_path / "latest").write_text("release")
    assert C.get_checkpoint_name(str(tmp_path), *C.get_checkpoint_iteration(str(tmp_path))).endswith("release/mp_rank_00_model_states.pt")
