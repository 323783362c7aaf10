"""CPU tests: the oracle against the golden vectors produced by code run from the original Diffuman4D repository
(tests/golden/gen_golden.py), and the oracle's own invariants (the reference's runtime checks, SURVEY.md section 4)."""
import os

import pytest
import torch

from diffuman4d_b200.config import SchedulerConfig, UNetConfig
from oracle import unet_oracle as O
from oracle.pipeline_oracle import (DDIMOracle, build_windows, denoise_window_oracle, sliding_iterative_denoise_oracle)

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_pose_encoder_matches_reference_golden():
    g = torch.load(os.path.join(GOLD, "pose_encoder.pt"))
    pe = O.PoseEncoder(out_channels=32)
    pe.load_state_dict(g["state_dict"])
    with torch.no_grad():
        y = pe(g["x"])
    torch.testing.assert_close(y, g["y"], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("tag,attn2", [("no_attn2", False), ("attn2", True)])
def test_multiview_block_matches_reference_golden(tag, attn2):
    g = torch.load(os.path.join(GOLD, "mv_block.pt"))[tag]
    blk = O.MultiviewTransformerBlock(64, 2, attn2)
    blk.load_state_dict(g["state_dict"])
    with torch.no_grad():
        y3 = blk(g["x"], num_frames=3)
        y1 = blk(g["x"], num_frames=1)
    torch.testing.assert_close(y3, g["y_3d"], rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(y1, g["y_2d"], rtol=1e-5, atol=1e-5)
    assert (y3 - y1).abs().max() > 1e-3  # the 3-D reshape really changes the result


def test_plucker_fixture_range():
    g = torch.load(os.path.join(GOLD, "plucker.pt"))
    assert g["plucker"].shape[1] == 6 and g["plucker"].abs().max() <= 3.0


def test_oracle_unet_shapes_and_determinism():
    cfg = UNetConfig.tiny()
    m = O.build_oracle(cfg, seed=1)
    F = 4
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2 * F, 11, 16, 16, generator=g)
    t = torch.randint(0, 1000, (2 * F,), generator=g)
    sk = torch.rand(2 * F, 3, 128, 128, generator=g) * 2 - 1
    with torch.no_grad():
        y = m(x, t, sk, ["spatial", "spatial"], F)
        y2 = O.build_oracle(cfg, seed=1)(x, t, sk, ["spatial", "spatial"], F)
        yt = m(x, t, sk, ["temporal", "temporal"], F)
    assert y.shape == (2 * F, 4, 16, 16)
    torch.testing.assert_close(y, y2)
    assert (y - yt).abs().max() > 1e-4  # frame-index embedding is live (zero-init branch re-randomised)
    with pytest.raises(ValueError):
        m(x, t, sk, ["spatial"], F)  # UNET:524-525


def test_oracle_3d_attention_mixes_frames():
    cfg = UNetConfig.tiny(enable_pose_encoder=False, in_channels=11)
    m = O.build_oracle(cfg, seed=2)
    F = 2
    g = torch.Generator().manual_seed(0)
    x = torch.randn(F, 11, 8, 8, generator=g)
    t = torch.tensor([10, 500])
    with torch.no_grad():
        y = m(x, t, None, ["spatial"], F)
        x2 = x.clone()
        x2[1] += 1.0
        y2 = m(x2, t, None, ["spatial"], F)
    assert (y[0] - y2[0]).abs().max() > 1e-5  # frame 0's output depends on frame 1's input


def test_ddim_tables_and_step():
    s = DDIMOracle(SchedulerConfig())
    ts = s.set_timesteps(18)
    assert ts.tolist() == [55 * i + 1 for i in range(17, -1, -1)]
    x = torch.randn(1, 4, 8, 8)
    e = torch.randn(1, 4, 8, 8)
    a_t, a_p = s.alphas_cumprod[936], s.alphas_cumprod[881]
    x0 = (x - (1 - a_t).sqrt() * e) / a_t.sqrt()
    torch.testing.assert_close(s.step(e, 936, x), a_p.sqrt() * x0 + (1 - a_p).sqrt() * e)
    # last step uses final_alpha_cumprod (= alphas_cumprod[0], set_alpha_to_one False)
    a_t = s.alphas_cumprod[1]
    x0 = (x - (1 - a_t).sqrt() * e) / a_t.sqrt()
    a_f = s.alphas_cumprod[0]
    torch.testing.assert_close(s.step(e, 1, x), a_f.sqrt() * x0 + (1 - a_f).sqrt() * e)
    sv = DDIMOracle(SchedulerConfig(prediction_type="v_prediction"))
    sv.set_timesteps(18)
    out = sv.step(e, 936, x)
    a_t, a_p = sv.alphas_cumprod[936], sv.alphas_cumprod[881]
    x0 = a_t.sqrt() * x - (1 - a_t).sqrt() * e
    ee = a_t.sqrt() * e + (1 - a_t).sqrt() * x
    torch.testing.assert_close(out, a_p.sqrt() * x0 + (1 - a_p).sqrt() * ee)


def test_window_schedule_worked_example():
    """SURVEY.md section 3.2: 48 cams, inputs {1,13,25,37}, window 12, stride 2 -> 22 windows with wrap-around."""
    mask = torch.ones(48)
    mask[[1, 13, 25, 37]] = 0
    tgt, inp = torch.where(mask != 0)[0], torch.where(mask == 0)[0]
    tw, iw = build_windows(tgt, inp, "spatial", 12, 2)
    assert len(tw) == 22
    assert tw[0].tolist() == [0, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12]
    assert tw[21].tolist()[:2] == [46, 47] and tw[21].tolist()[2] == 0
    assert all(torch.equal(i, inp) for i in iw)
    # temporal: T=16 frames of the cond cam then 16 of the target cam
    mask = torch.cat([torch.zeros(16), torch.ones(16)])
    tgt, inp = torch.where(mask != 0)[0], torch.where(mask == 0)[0]
    tw, iw = build_windows(tgt, inp, "temporal", 12, 2)
    assert len(tw) == 8 and tw[0].tolist() == list(range(16, 28)) and iw[0].tolist() == list(range(0, 12))


@pytest.mark.parametrize("tag", ["pose_tem_linear", "attn2_convproj_nopose", "two_3d_levels"])
def test_oracle_unet_matches_reference_unet_golden(tag):
    """The oracle UNet against the reference's own ``UNetMultiviewConditionModel`` constructor + forward, block classes,
    ``TransformerMultiviewModel``, ``MultiviewTransformerBlock`` and ``PoseEncoder`` run on stubs of the upstream LEAF
    classes only (tests/golden/gen_golden.py::gen_unet).  Pins the wiring: embeddings, pose-encoder add, block order, skip
    bookkeeping, which levels are 3-D, proj order, output head -- and the diffusers-layout key/shape spec of the product."""
    from diffuman4d_b200.config import UNetConfig
    from diffuman4d_b200.weights import random_state_dict, state_dict_spec
    from oracle.unet_oracle import OracleUNet
    c = torch.load(os.path.join(GOLD, "unet_ref.pt"))["cases"][tag]
    cfg = UNetConfig(**c["cfg"])
    spec = {k: tuple(v) for k, v in state_dict_spec(cfg).items()}
    assert spec == c["ref_state_dict_shapes"]          # product weight-key contract == reference module tree
    m = OracleUNet(cfg)
    m.load_state_dict(random_state_dict(cfg, seed=c["seed"], dtype=torch.float32), strict=True)
    m.eval()
    for r in c["runs"].values():
        sk = None if r["skeletons"] is None else r["skeletons"].float()   # stored as float16, exactly
        with torch.no_grad():
            y = m(r["sample"], r["timestep"], sk, r["domains"], r["num_frames"])
        torch.testing.assert_close(y, r["out"], rtol=2e-4, atol=2e-5)


def test_oracle_unet_num_frames_error_matches_reference():
    from diffuman4d_b200.config import UNetConfig
    from oracle.unet_oracle import OracleUNet
    g = torch.load(os.path.join(GOLD, "unet_ref.pt"))
    cfg = UNetConfig(**g["cases"]["two_3d_levels"]["cfg"])
    m = OracleUNet(cfg)
    x = torch.zeros(4, cfg.in_channels, 8, 8)
    with pytest.raises(ValueError) as e:
        m(x, torch.zeros(4, dtype=torch.int64), torch.zeros(4, 3, 64, 64), ["spatial"], 3)
    assert str(e.value) == g["num_frames_error"]


def _fake_unet(cin):
    import sys
    sys.path.insert(0, GOLD)
    from fake_unet import make_fake_unet
    return make_fake_unet(cin)


@pytest.mark.parametrize("tag", ["call_pose_cfg", "call_nopose_nocfg", "call_pose_cfg_vpred"])
def test_window_step_matches_reference_pipeline_golden(tag):
    """The oracle's window step against the reference's own ``Diffuman4DPipeline.__call__`` (PIPE:345-425) run on stubs of
    the upstream surface (tests/golden/gen_golden.py::gen_pipeline): assembly, CFG negatives, cond aliasing, per-frame steps."""
    c = torch.load(os.path.join(GOLD, "pipeline_ref.pt"))["cases"][tag]
    i = c["in"]
    s = DDIMOracle(SchedulerConfig(prediction_type=c["prediction_type"]))
    s.set_timesteps(c["n_steps_table"])
    assert torch.equal(s.timesteps, c["timesteps_table"])
    cin = 4 + 6 + (0 if c["pose"] else 4) + 1
    lat, ti = denoise_window_oracle(
        _fake_unet(cin), s, latents=i["latents"].clone(), pixel_latents=i["pixel_latents"], plucker=i["plucker"],
        skeletons=i["skeletons"].float(), cond_mask=i["cond_mask"], timestep_indices=i["timestep_indices"], domain="spatial",
        guidance_scale=c["guidance"], num_inference_steps=2, enable_pose_encoder=c["pose"])
    torch.testing.assert_close(lat, c["out_latents"], rtol=1e-5, atol=1e-6)
    assert torch.equal(ti, c["out_timestep_indices"])


@pytest.mark.parametrize("tag", ["slide_spatial", "slide_temporal_bidir"])
def test_sliding_loop_matches_reference_pipeline_golden(tag):
    """Oracle AND product window schedule / sliding loop against the reference's ``sliding_iterative_denoise``
    (PIPE:439-559) run on the same stubs: visited windows, per-window timestep indices, final grid, bookkeeping."""
    from diffuman4d_b200.pipeline import build_windows as product_build_windows
    c = torch.load(os.path.join(GOLD, "pipeline_ref.pt"))["cases"][tag]
    i = c["in"]
    mask = i["cond_mask_latents"]
    tgt, inp = torch.where(mask[:, 0, 0, 0] != 0)[0], torch.where(mask[:, 0, 0, 0] == 0)[0]
    for bw in (build_windows, product_build_windows):
        tw, iw = bw(tgt, inp, c["domain"], c["window_size"], c["sliding_stride"], 0, c["bidirectional"])
        per_round = [torch.cat([a, b]) for a, b in zip(iw, tw)]
        assert len(c["window_frames"]) == len(per_round)  # one alternation per call (PIPE:503-518)
        for got, ref in zip(per_round, c["window_frames"]):
            assert torch.equal(got, ref)
    s = DDIMOracle(SchedulerConfig())
    out = sliding_iterative_denoise_oracle(
        _fake_unet(11), s, pixel_latents=i["pixel_latents"], plucker=i["plucker"], skeletons=i["skeletons"].float(),
        cond_mask=mask, latents=i["latents"], domain=c["domain"], timestep_indices=i["timestep_indices"], window_size=c["window_size"],
        sliding_stride=c["sliding_stride"], bidirectional=c["bidirectional"], num_denoising_steps=1,
        alternation_rounds=c["alternation_rounds"], guidance_scale=2.0, enable_pose_encoder=True)
    torch.testing.assert_close(out["latents"], c["out_latents"], rtol=1e-5, atol=1e-6)
    assert torch.equal(out["timestep_indices"], c["out_timestep_indices"])
    assert torch.equal(out["fully_denoised"], c["fully_denoised"])


def test_sliding_argument_errors_match_reference_messages():
    """PIPE:464,481,486: same exception type and text as the reference raised in the generator run."""
    errs = torch.load(os.path.join(GOLD, "pipeline_ref.pt"))["errors"]
    n, h, w = 8, 8, 8
    mask = torch.ones(n, 1, h, w)
    mask[:2] = 0
    base = dict(pixel_latents=torch.zeros(n, 4, h, w), plucker=torch.zeros(n, 6, h, w), skeletons=None, cond_mask=mask,
                latents=torch.zeros(n, 4, h, w), domain="spatial", window_size=3, num_denoising_steps=1, alternation_rounds=1)
    cases = {"stride": dict(sliding_stride=2, timestep_indices=torch.zeros(n, dtype=torch.int64)),
             "unequal_targets": dict(sliding_stride=1, timestep_indices=torch.tensor([0, 0, 1, 1, 1, 1, 1, 2])),
             "nonzero_inputs": dict(sliding_stride=1, timestep_indices=torch.tensor([1, 0, 0, 0, 0, 0, 0, 0]))}
    for tag, kw in cases.items():
        assert errs[tag] is not None
        with pytest.raises(ValueError) as e:
            sliding_iterative_denoise_oracle(_stub_unet, DDIMOracle(SchedulerConfig()), **{**base, **kw})
        assert str(e.value) == errs[tag]


def _stub_unet(x, t, sk, domains, nf):
    return 0.1 * x[:, :4] + 0.01 * t.float()[:, None, None, None] / 1000


def test_sliding_loop_invariants_and_aliasing():
    g = torch.Generator().manual_seed(3)
    n, h, w = 16, 8, 8
    mask = torch.ones(n, 1, h, w)
    mask[[1, 5, 9, 13]] = 0
    pix = torch.randn(n, 4, h, w, generator=g)
    lat = torch.randn(n, 4, h, w, generator=g)
    args = dict(pixel_latents=pix, plucker=torch.randn(n, 6, h, w, generator=g), skeletons=None, cond_mask=mask,
                latents=lat, domain="spatial", timestep_indices=torch.zeros(n, dtype=torch.long), window_size=4,
                sliding_stride=2, alternation_rounds=3, guidance_scale=2.0, enable_pose_encoder=True)
    s = DDIMOracle(SchedulerConfig())
    out = sliding_iterative_denoise_oracle(_stub_unet, s, **args)
    tgt = mask[:, 0, 0, 0] != 0
    assert (out["timestep_indices"][tgt] == 2).all() and (out["timestep_indices"][~tgt] == 0).all()
    # cond frames come back as the image latents (reference aliasing quirk, PIPE:375-379)
    torch.testing.assert_close(out["latents"][~tgt], pix[~tgt])
    assert not out["fully_denoised"].any()
    with pytest.raises(ValueError):
        sliding_iterative_denoise_oracle(_stub_unet, s, **{**args, "window_size": 3})  # 3*1 % 2 != 0
    bad = torch.zeros(n, dtype=torch.long)
    bad[0] = 1
    with pytest.raises(ValueError):
        sliding_iterative_denoise_oracle(_stub_unet, s, **{**args, "timestep_indices": bad})


def test_denoise_window_oracle_cfg_and_cond_handling():
    g = torch.Generator().manual_seed(4)
    F, h, w = 6, 8, 8
    mask = torch.ones(F, 1, h, w)
    mask[:2] = 0
    s = DDIMOracle(SchedulerConfig())
    s.set_timesteps(18)
    seen = {}

    def unet(x, t, sk, domains, nf):
        seen["x"], seen["t"], seen["domains"], seen["nf"] = x.clone(), t.clone(), domains, nf
        return torch.zeros(x.shape[0], 4, h, w)

    lat = torch.randn(F, 4, h, w, generator=g)
    pix = torch.randn(F, 4, h, w, generator=g)
    plk = torch.randn(F, 6, h, w, generator=g)
    ti = torch.tensor([0, 0, 3, 3, 2, 2])
    new, ti2 = denoise_window_oracle(unet, s, latents=lat.clone(), pixel_latents=pix, plucker=plk, skeletons=None,
                                     cond_mask=mask, timestep_indices=ti, domain="temporal", guidance_scale=2.0)
    x = seen["x"]
    assert x.shape == (2 * F, 11, h, w) and seen["domains"] == ["temporal", "temporal"] and seen["nf"] == F
    assert (x[:2, :4] == 1).all()                       # negative half: cond frames are "white"
    torch.testing.assert_close(x[F:F + 2, :4], pix[:2])  # positive half: cond frames are the image latents
    assert (x[:F, 4:10] == 0).all() and torch.equal(x[F:, 4:10], plk)
    assert seen["t"][:2].tolist() == [0, 0] and seen["t"][2].item() == s.timesteps[3].item()
    assert ti2.tolist() == [0, 0, 4, 4, 3, 3]
    torch.testing.assert_close(new[:2], pix[:2])
