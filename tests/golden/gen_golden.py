"""Generate golden fixtures by RUNNING code from a checkout of the original Diffuman4D repository (zju3dv/Diffuman4D).
The outputs are committed, so the tests never need that checkout.

Pinned here:
  pose_encoder.pt   -- the reference ``PoseEncoder`` (src/diffusers/models/unets/pose_encoder.py), imported
                       directly by file path (it only needs torch/numpy/einops).
  mv_block.pt       -- the reference ``MultiviewTransformerBlock.forward`` (src/diffusers/models/attention.py:22-153)
                       running ITS OWN code on top of a stub of the un-installed upstream base class
                       ``diffusers.models.attention.BasicTransformerBlock`` (the stub = our restatement of
                       upstream 0.33.1; the 3-D token reshape and residual wiring are the reference's).
  plucker.pt        -- ``calc_plucker_embeds`` from src/data/utils/ray_utils.py on a small camera ring (realistic
                       value ranges for the bench's synthetic Plucker channels).

  pipeline_ref.pt   -- the reference ``Diffuman4DPipeline.__call__`` (PIPE:345-425) and ``sliding_iterative_denoise``
                       (PIPE:439-559) running THEIR OWN code (input assembly, CFG negatives, cond-frame aliasing,
                       per-frame scheduler steps, window schedule, invariants) on stubs of the un-installed upstream
                       surface: ``DiffusionPipeline`` plumbing, a per-frame-deep-copyable scheduler backed by our DDIM
                       restatement, an identity "VAE", and ``tests/golden/fake_unet.py`` as ``pipeline.unet``.

  unet_ref.pt       -- the reference ``UNetMultiviewConditionModel`` (UNET:149-598: constructor AND forward) with the
                       reference's own block classes (BLK: get_*_block, CrossAttnDown/Up/MidBlockMultiview),
                       ``TransformerMultiviewModel`` (TRF), ``MultiviewTransformerBlock`` (ATT) and ``PoseEncoder``,
                       running on stubs of the upstream LEAF classes only (ResnetBlock2D, Down/Upsample2D,
                       Down/UpBlock2D, Transformer2DModel base, BasicTransformerBlock, Attention, Timesteps,
                       TimestepEmbedding = the oracle's restatements behind the upstream constructor signatures).
                       Weights come from ``diffuman4d_b200.weights.random_state_dict`` loaded with strict=True, which
                       also pins the product's diffusers-layout key/shape spec against the reference module tree.

Every fixture stays under 1 MB: the pixel-resolution skeletons are drawn as float16-representable values and stored as
float16 (exact; the tests upcast them to float32), and pipeline_ref.pt keeps only the latent-resolution inputs the tests
feed to the oracle, not the pixel-resolution images and masks the reference encoded them from.

Run:  python tests/golden/gen_golden.py <Diffuman4D checkout>      (from the repo root)
"""
import importlib.util
import os
import sys
import types

import torch
import torch.nn as nn

REF = None  # the Diffuman4D checkout, set from the command line
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))


def load_by_path(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def gen_pose_encoder():
    pe_mod = load_by_path("ref_pose_encoder", f"{REF}/src/diffusers/models/unets/pose_encoder.py")
    torch.manual_seed(11)
    pe = pe_mod.PoseEncoder(out_channels=32)
    with torch.no_grad():  # un-zero the zero-init projection so the output is informative
        pe.final_proj.weight.normal_(0, 0.1)
        pe.final_proj.bias.normal_(0, 0.1)
        for m in pe.conv_layers:
            if isinstance(m, nn.Conv2d):
                m.bias.normal_(0, 0.1)
    x = torch.rand(2, 3, 32, 40) * 2 - 1
    with torch.no_grad():
        y = pe(x)
    torch.save({"state_dict": pe.state_dict(), "x": x, "y": y}, f"{HERE}/pose_encoder.pt")
    print("pose_encoder", tuple(y.shape), float(y.abs().mean()))


def gen_mv_block():
    from oracle import unet_oracle as O

    class StubAttention(O.Attention):
        def forward(self, x, encoder_hidden_states=None, attention_mask=None, **kw):
            assert encoder_hidden_states is None and attention_mask is None
            return super().forward(x)

    class StubBasicTransformerBlock(nn.Module):
        """minimal upstream BasicTransformerBlock (layer_norm, geglu) for the reference subclass"""

        def __init__(self, dim, heads, attn2):
            super().__init__()
            self.norm_type = "layer_norm"
            self.pos_embed = None
            self.only_cross_attention = False
            self._chunk_size = None
            self._chunk_dim = 0
            self.norm1 = nn.LayerNorm(dim, eps=1e-5)
            self.attn1 = StubAttention(dim, heads)
            self.norm2 = nn.LayerNorm(dim, eps=1e-5) if attn2 else None
            self.attn2 = StubAttention(dim, heads) if attn2 else None
            self.norm3 = nn.LayerNorm(dim, eps=1e-5)
            self.ff = O.FeedForward(dim)

    # stub the import surface of src/diffusers/models/attention.py:1-10
    d = types.ModuleType("diffusers")
    du = types.ModuleType("diffusers.utils")
    dut = types.ModuleType("diffusers.utils.torch_utils")
    dm = types.ModuleType("diffusers.models")
    dma = types.ModuleType("diffusers.models.attention")
    import logging as _logging
    du.logging = types.SimpleNamespace(get_logger=_logging.getLogger)
    dut.maybe_allow_in_graph = lambda c: c
    dma._chunked_feed_forward = None
    dma.BasicTransformerBlock = StubBasicTransformerBlock
    for name, mod in [("diffusers", d), ("diffusers.utils", du), ("diffusers.utils.torch_utils", dut),
                      ("diffusers.models", dm), ("diffusers.models.attention", dma)]:
        sys.modules[name] = mod
    ref_att = load_by_path("ref_attention", f"{REF}/src/diffusers/models/attention.py")

    out = {}
    for tag, attn2 in (("no_attn2", False), ("attn2", True)):
        torch.manual_seed(5 if attn2 else 4)
        blk = ref_att.MultiviewTransformerBlock(64, 2, attn2)
        with torch.no_grad():
            for p in blk.parameters():
                p.normal_(0, 0.15)
        x = torch.randn(6, 16, 64)  # (b t) hw c with b=2, t=3
        with torch.no_grad():
            y3 = blk(x, num_frames=3)
            y1 = blk(x, num_frames=1)
        out[tag] = {"state_dict": blk.state_dict(), "x": x, "y_3d": y3, "y_2d": y1}
        print("mv_block", tag, float(y3.abs().mean()), float((y3 - y1).abs().mean()))
    torch.save(out, f"{HERE}/mv_block.pt")


def gen_plucker():
    ray = load_by_path("ref_ray_utils", f"{REF}/src/data/utils/ray_utils.py")
    import math
    n, h, w = 6, 16, 16
    Ks, c2ws = [], []
    for i in range(n):
        a = 2 * math.pi * i / n
        eye = torch.tensor([2.5 * math.cos(a), 0.3, 2.5 * math.sin(a)])
        fwd = -eye / eye.norm()
        up = torch.tensor([0.0, 1.0, 0.0])
        right = torch.linalg.cross(fwd, up)
        right = right / right.norm()
        up2 = torch.linalg.cross(right, fwd)
        c2w = torch.eye(4)
        c2w[:3, 0], c2w[:3, 1], c2w[:3, 2], c2w[:3, 3] = right, -up2, fwd, eye
        c2ws.append(c2w)
        K = torch.tensor([[1.2 * w, 0, w / 2], [0, 1.2 * w, h / 2], [0, 0, 1.0]])
        Ks.append(K)
    Ks, c2ws = torch.stack(Ks), torch.stack(c2ws)
    try:
        pl = ray.calc_plucker_embeds(h, w, Ks, c2ws)
    except TypeError:
        import inspect
        print("calc_plucker_embeds signature:", inspect.signature(ray.calc_plucker_embeds))
        raise
    rel = ray.calc_relative_poses(c2ws)                      # what the dataset feeds the embedding (DATA:162-165)
    pl_rel = ray.calc_plucker_embeds(h, w, Ks, rel)
    torch.save({"K": Ks, "c2w": c2ws, "plucker": pl, "rel_poses": rel, "plucker_rel": pl_rel}, f"{HERE}/plucker.pt")
    print("plucker", tuple(pl.shape), float(pl.min()), float(pl.max()))


def gen_unet():
    """Run the reference UNet (its own wiring) on upstream-leaf stubs; see the module docstring."""
    import dataclasses
    import functools
    import inspect

    from diffuman4d_b200.config import UNetConfig
    from diffuman4d_b200.weights import random_state_dict
    from oracle import unet_oracle as O

    NS = types.SimpleNamespace

    def register_to_config(init):  # upstream: binds the constructor arguments into self.config before the body runs
        @functools.wraps(init)
        def wrapper(self, *args, **kwargs):
            ba = inspect.signature(init).bind(self, *args, **kwargs)
            ba.apply_defaults()
            object.__setattr__(self, "config", NS(**{k: v for k, v in ba.arguments.items() if k != "self"}))
            init(self, *args, **kwargs)
        return wrapper

    class ModelMixin(nn.Module):
        @property
        def dtype(self):
            return next(self.parameters()).dtype

        @property
        def device(self):
            return next(self.parameters()).device

    class _Empty:
        pass

    @dataclasses.dataclass
    class BaseOutput:
        pass

    class StubAttention(O.Attention):
        def forward(self, x, encoder_hidden_states=None, attention_mask=None, **kw):
            assert encoder_hidden_states is None and attention_mask is None
            return super().forward(x)

    class BasicTransformerBlock(nn.Module):  # upstream constructor signature (R-6), layer_norm / geglu only
        def __init__(self, dim, num_attention_heads, attention_head_dim, dropout=0.0, cross_attention_dim=None,
                     activation_fn="geglu", num_embeds_ada_norm=None, attention_bias=False, only_cross_attention=False,
                     double_self_attention=False, upcast_attention=False, norm_elementwise_affine=True,
                     norm_type="layer_norm", norm_eps=1e-5, final_dropout=False, attention_type="default", **kw):
            super().__init__()
            assert dim == num_attention_heads * attention_head_dim and activation_fn == "geglu" and dropout == 0.0
            assert norm_type == "layer_norm" and not attention_bias and not only_cross_attention
            self.norm_type, self.pos_embed, self.only_cross_attention = norm_type, None, only_cross_attention
            self._chunk_size, self._chunk_dim = None, 0
            self.norm1 = nn.LayerNorm(dim, eps=norm_eps)
            self.attn1 = StubAttention(dim, num_attention_heads)
            if cross_attention_dim is not None or double_self_attention:
                assert cross_attention_dim in (None, dim)  # encoder_hidden_states is never passed => width-C context
                self.norm2 = nn.LayerNorm(dim, eps=norm_eps)
                self.attn2 = StubAttention(dim, num_attention_heads)
            else:
                self.norm2, self.attn2 = None, None
            self.norm3 = nn.LayerNorm(dim, eps=norm_eps)
            self.ff = O.FeedForward(dim)

    class Transformer2DModel(ModelMixin):  # upstream base: continuous-input path only (R-5)
        def __init__(self, num_attention_heads=16, attention_head_dim=88, in_channels=None, out_channels=None, num_layers=1,
                     dropout=0.0, norm_num_groups=32, cross_attention_dim=None, attention_bias=False, sample_size=None,
                     num_vector_embeds=None, patch_size=None, activation_fn="geglu", num_embeds_ada_norm=None,
                     use_linear_projection=False, only_cross_attention=False, double_self_attention=False,
                     upcast_attention=False, norm_type="layer_norm", norm_elementwise_affine=True, norm_eps=1e-5,
                     attention_type="default", caption_channels=None, interpolation_scale=None,
                     use_additional_conditions=None):
            super().__init__()
            loc = dict(locals())
            self.config = NS(**{k: v for k, v in loc.items() if k not in ("self", "__class__", "loc")})
            self.use_linear_projection = use_linear_projection
            self.num_attention_heads, self.attention_head_dim = num_attention_heads, attention_head_dim
            self.inner_dim = num_attention_heads * attention_head_dim
            self.in_channels = in_channels
            self.out_channels = in_channels if out_channels is None else out_channels
            self.gradient_checkpointing = False
            self.is_input_continuous, self.is_input_vectorized, self.is_input_patches = True, False, False
            self._init_continuous_input(norm_type=norm_type)

        def _operate_on_continuous_inputs(self, hidden_states):
            batch, _, height, width = hidden_states.shape
            hidden_states = self.norm(hidden_states)
            if not self.use_linear_projection:
                hidden_states = self.proj_in(hidden_states)
                inner_dim = hidden_states.shape[1]
                hidden_states = hidden_states.permute(0, 2, 3, 1).reshape(batch, height * width, inner_dim)
            else:
                inner_dim = hidden_states.shape[1]
                hidden_states = hidden_states.permute(0, 2, 3, 1).reshape(batch, height * width, inner_dim)
                hidden_states = self.proj_in(hidden_states)
            return hidden_states, inner_dim

        def _get_output_for_continuous_inputs(self, hidden_states, residual, batch_size, height, width, inner_dim):
            if not self.use_linear_projection:
                hidden_states = hidden_states.reshape(batch_size, height, width, inner_dim).permute(0, 3, 1, 2).contiguous()
                hidden_states = self.proj_out(hidden_states)
            else:
                hidden_states = self.proj_out(hidden_states)
                hidden_states = hidden_states.reshape(batch_size, height, width, inner_dim).permute(0, 3, 1, 2).contiguous()
            return hidden_states + residual

    class ResnetBlock2D(O.ResnetBlock2D):
        def __init__(self, *, in_channels, out_channels=None, temb_channels=512, eps=1e-6, groups=32, groups_out=None,
                     dropout=0.0, time_embedding_norm="default", non_linearity="swish", output_scale_factor=1.0,
                     pre_norm=True, **kw):
            assert time_embedding_norm == "default" and output_scale_factor == 1.0 and dropout == 0.0 and pre_norm
            assert groups_out in (None, groups) and non_linearity in ("silu", "swish") and not kw
            super().__init__(in_channels, out_channels or in_channels, temb_channels, groups, eps)

        def forward(self, x, temb, *a, **k):
            return super().forward(x, temb)

    class Downsample2D(O.Downsample2D):
        def __init__(self, channels, use_conv=False, out_channels=None, padding=1, name="conv", **kw):
            assert use_conv and padding == 1 and name == "op" and out_channels in (None, channels)
            super().__init__(channels)

        def forward(self, x, *a, **k):
            return super().forward(x)

    class Upsample2D(O.Upsample2D):
        def __init__(self, channels, use_conv=False, use_conv_transpose=False, out_channels=None, name="conv", **kw):
            assert use_conv and not use_conv_transpose and out_channels in (None, channels)
            super().__init__(channels)

        def forward(self, x, output_size=None, *a, **k):
            assert output_size is None  # upsample_size is always None on this path (R-3)
            return super().forward(x)

    class DownBlock2D(nn.Module):  # upstream unet_2d_blocks.DownBlock2D (R-4)
        def __init__(self, in_channels, out_channels, temb_channels, dropout=0.0, num_layers=1, resnet_eps=1e-6,
                     resnet_time_scale_shift="default", resnet_act_fn="swish", resnet_groups=32, resnet_pre_norm=True,
                     output_scale_factor=1.0, add_downsample=True, downsample_padding=1):
            super().__init__()
            self.resnets = nn.ModuleList([
                ResnetBlock2D(in_channels=in_channels if i == 0 else out_channels, out_channels=out_channels,
                              temb_channels=temb_channels, eps=resnet_eps, groups=resnet_groups, dropout=dropout,
                              time_embedding_norm=resnet_time_scale_shift, non_linearity=resnet_act_fn,
                              output_scale_factor=output_scale_factor, pre_norm=resnet_pre_norm) for i in range(num_layers)])
            self.downsamplers = nn.ModuleList([Downsample2D(out_channels, use_conv=True, out_channels=out_channels,
                                                            padding=downsample_padding, name="op")]) if add_downsample else None
            self.gradient_checkpointing = False

        def forward(self, hidden_states, temb=None, *a, **k):
            output_states = ()
            for resnet in self.resnets:
                hidden_states = resnet(hidden_states, temb)
                output_states = output_states + (hidden_states,)
            if self.downsamplers is not None:
                for d in self.downsamplers:
                    hidden_states = d(hidden_states)
                output_states = output_states + (hidden_states,)
            return hidden_states, output_states

    class UpBlock2D(nn.Module):  # upstream unet_2d_blocks.UpBlock2D (R-4)
        def __init__(self, in_channels, prev_output_channel, out_channels, temb_channels, resolution_idx=None, dropout=0.0,
                     num_layers=1, resnet_eps=1e-6, resnet_time_scale_shift="default", resnet_act_fn="swish",
                     resnet_groups=32, resnet_pre_norm=True, output_scale_factor=1.0, add_upsample=True):
            super().__init__()
            resnets = []
            for i in range(num_layers):
                res_skip_channels = in_channels if (i == num_layers - 1) else out_channels
                resnet_in_channels = prev_output_channel if i == 0 else out_channels
                resnets.append(ResnetBlock2D(in_channels=resnet_in_channels + res_skip_channels, out_channels=out_channels,
                                             temb_channels=temb_channels, eps=resnet_eps, groups=resnet_groups, dropout=dropout,
                                             time_embedding_norm=resnet_time_scale_shift, non_linearity=resnet_act_fn,
                                             output_scale_factor=output_scale_factor, pre_norm=resnet_pre_norm))
            self.resnets = nn.ModuleList(resnets)
            self.upsamplers = nn.ModuleList([Upsample2D(out_channels, use_conv=True, out_channels=out_channels)]) if add_upsample else None
            self.gradient_checkpointing = False
            self.resolution_idx = resolution_idx

        def forward(self, hidden_states, res_hidden_states_tuple, temb=None, upsample_size=None, *a, **k):
            for resnet in self.resnets:
                res_hidden_states = res_hidden_states_tuple[-1]
                res_hidden_states_tuple = res_hidden_states_tuple[:-1]
                hidden_states = torch.cat([hidden_states, res_hidden_states], dim=1)
                hidden_states = resnet(hidden_states, temb)
            if self.upsamplers is not None:
                for u in self.upsamplers:
                    hidden_states = u(hidden_states, upsample_size)
            return hidden_states

    class TimestepEmbedding(O.TimestepEmbedding):
        def __init__(self, in_channels, time_embed_dim, act_fn="silu", out_dim=None, post_act_fn=None, cond_proj_dim=None):
            assert act_fn == "silu" and out_dim is None and post_act_fn is None and cond_proj_dim is None
            super().__init__(in_channels, time_embed_dim)

        def forward(self, sample, condition=None):
            assert condition is None
            return super().forward(sample)

    class Timesteps(nn.Module):
        def __init__(self, num_channels, flip_sin_to_cos, downscale_freq_shift, scale=1):
            super().__init__()
            self.num_channels, self.flip, self.shift = num_channels, flip_sin_to_cos, downscale_freq_shift

        def forward(self, timesteps):
            return O.timestep_embedding(timesteps, self.num_channels, self.flip, self.shift)

    def get_activation(name):
        assert name in ("silu", "swish")
        return nn.SiLU()

    import logging as _logging
    log_ns = NS(get_logger=_logging.getLogger)
    mods = {
        "diffusers": {}, "diffusers.configuration_utils": {"ConfigMixin": _Empty, "register_to_config": register_to_config},
        "diffusers.loaders": {"PeftAdapterMixin": type("PeftAdapterMixin", (), {}),
                              "UNet2DConditionLoadersMixin": type("UNet2DConditionLoadersMixin", (), {})},
        "diffusers.loaders.single_file_model": {"FromOriginalModelMixin": type("FromOriginalModelMixin", (), {})},
        "diffusers.utils": {"BaseOutput": BaseOutput, "logging": log_ns, "deprecate": lambda *a, **k: None,
                            "is_torch_version": lambda *a, **k: True},
        "diffusers.utils.torch_utils": {"apply_freeu": None, "maybe_allow_in_graph": lambda c: c},
        "diffusers.models": {}, "diffusers.models.activations": {"get_activation": get_activation},
        "diffusers.models.embeddings": {"TimestepEmbedding": TimestepEmbedding, "Timesteps": Timesteps},
        "diffusers.models.modeling_utils": {"ModelMixin": ModelMixin},
        "diffusers.models.attention_processor": {"Attention": StubAttention, "AttnAddedKVProcessor": object,
                                                 "AttnAddedKVProcessor2_0": object},
        "diffusers.models.normalization": {"AdaGroupNorm": object},
        "diffusers.models.resnet": {"Downsample2D": Downsample2D, "ResnetBlock2D": ResnetBlock2D, "Upsample2D": Upsample2D},
        "diffusers.models.unets": {}, "diffusers.models.unets.unet_2d_blocks": {"DownBlock2D": DownBlock2D, "UpBlock2D": UpBlock2D},
        "diffusers.models.transformers": {}, "diffusers.models.transformers.transformer_2d": {"Transformer2DModel": Transformer2DModel},
        "diffusers.models.modeling_outputs": {"Transformer2DModelOutput": type("Transformer2DModelOutput", (), {"__init__": lambda self, sample=None: setattr(self, "sample", sample)})},
        "diffusers.models.attention": {"BasicTransformerBlock": BasicTransformerBlock, "_chunked_feed_forward": None},
        "refmodels": {}, "refmodels.unets": {}, "refmodels.transformers": {},
    }
    for name, attrs in mods.items():
        m = types.ModuleType(name)
        m.__path__ = []
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m

    def load_ref(modname, relpath):  # the reference's own files, loaded as the package `refmodels` (= src/diffusers/models)
        spec = importlib.util.spec_from_file_location(modname, f"{REF}/src/diffusers/models/{relpath}")
        mod = importlib.util.module_from_spec(spec)
        mod.__package__ = modname.rsplit(".", 1)[0]
        sys.modules[modname] = mod
        spec.loader.exec_module(mod)
        return mod

    load_ref("refmodels.attention", "attention.py")
    load_ref("refmodels.transformers.transformer_multiview", "transformers/transformer_multiview.py")
    load_ref("refmodels.unets.pose_encoder", "unets/pose_encoder.py")
    load_ref("refmodels.unets.unet_multiview_blocks", "unets/unet_multiview_blocks.py")
    ref_unet_mod = load_ref("refmodels.unets.unet_multiview_condition", "unets/unet_multiview_condition.py")

    out = {"cases": {}}
    micro = dict(block_out_channels=(32, 64, 64, 64), attention_head_dim=(1, 2, 2, 2), norm_num_groups=16)
    variants = {
        "pose_tem_linear": UNetConfig(**micro),                                             # the shipped layout in miniature
        "attn2_convproj_nopose": UNetConfig(**micro, in_channels=15, cross_attention_dim=(32, 64, 64, 64),
                                            use_linear_projection=False, enable_tem_embeds=False, enable_pose_encoder=False),
        "two_3d_levels": UNetConfig(**micro, num_3d_attn_blocks=2),
    }
    g = torch.Generator().manual_seed(77)
    for tag, cfg in variants.items():
        model = ref_unet_mod.UNetMultiviewConditionModel(
            in_channels=cfg.in_channels, out_channels=cfg.out_channels, block_out_channels=cfg.block_out_channels,
            layers_per_block=cfg.layers_per_block, attention_head_dim=cfg.attention_head_dim,
            cross_attention_dim=cfg.cross_attention_dim, use_linear_projection=cfg.use_linear_projection,
            norm_num_groups=cfg.norm_num_groups, norm_eps=cfg.norm_eps, flip_sin_to_cos=cfg.flip_sin_to_cos,
            freq_shift=cfg.freq_shift, num_3d_attn_blocks=cfg.num_3d_attn_blocks, enable_tem_embeds=cfg.enable_tem_embeds,
            enable_pose_encoder=cfg.enable_pose_encoder)
        ref_keys = {k: tuple(v.shape) for k, v in model.state_dict().items()}
        sd = random_state_dict(cfg, seed=5, dtype=torch.float32)
        missing = model.load_state_dict(sd, strict=True)  # product key/shape spec == reference module tree
        model.eval()
        F_, h, w = 3, 8, 8
        runs = {}
        for dom_tag, domains in (("spatial_cfg", ["spatial", "spatial"]), ("temporal", ["temporal"])):
            nf = F_ if dom_tag == "spatial_cfg" else 4
            B = nf * len(domains)
            x = torch.randn(B, cfg.in_channels, h, w, generator=g)
            t = torch.randint(0, 1000, (B,), generator=g)
            sk = (torch.rand(B, 3, 8 * h, 8 * w, generator=g) * 2 - 1).half().float() if cfg.enable_pose_encoder else None
            with torch.no_grad():
                y = model(x, t, skeletons=sk, domains=domains, num_frames=nf, return_dict=False)[0]
            runs[dom_tag] = {"sample": x, "timestep": t, "skeletons": None if sk is None else sk.half(), "domains": domains,
                             "num_frames": nf, "out": y}
            print("unet", tag, dom_tag, tuple(y.shape), float(y.abs().mean()))
        out["cases"][tag] = {"cfg": cfg.to_dict(), "seed": 5, "ref_state_dict_shapes": ref_keys, "runs": runs}
    # the reference's own argument check (UNET:524-525)
    try:
        model(x, t, skeletons=sk, domains=["spatial"], num_frames=3, return_dict=False)
        out["num_frames_error"] = None
    except ValueError as e:
        out["num_frames_error"] = str(e)
    print("unet error ->", out["num_frames_error"])
    torch.save(out, f"{HERE}/unet_ref.pt")


_RANDN_CALLS = [0]


def _counter_randn(shape, generator=None, device=None, dtype=None):
    """stand-in for diffusers.utils.torch_utils.randn_tensor: the k-th call draws from Generator(9000 + k), so the tests can
    reproduce the initial noise of every task (only sliding_iterative_denoise with latents=None reaches it, PIPE:175)."""
    g = torch.Generator().manual_seed(9000 + _RANDN_CALLS[0])
    _RANDN_CALLS[0] += 1
    return torch.randn(tuple(shape), generator=g).to(dtype=dtype)


def _load_ref_pipeline():
    """The reference pipeline module on stubs of the upstream plumbing -> (module, make_pipe)."""
    import contextlib

    from diffuman4d_b200.config import SchedulerConfig
    from oracle.pipeline_oracle import DDIMOracle

    sys.path.insert(0, HERE)
    from fake_unet import make_fake_unet

    # ---- stub the import surface of PIPE:14-34
    class _Mixin:
        pass

    class StubDiffusionPipeline:
        def __init__(self):
            pass

        def register_modules(self, **kw):
            for k, v in kw.items():
                setattr(self, k, v)

        @property
        def _execution_device(self):
            return torch.device("cpu")

        device = torch.device("cpu")  # DiffusionPipeline.device (read by SAMP:177)

        @contextlib.contextmanager
        def progress_bar(self, total=None):
            yield types.SimpleNamespace(update=lambda *a, **k: None)

        def maybe_free_model_hooks(self):
            pass

    class StubImageProcessor:
        def __init__(self, vae_scale_factor=8):
            self.vae_scale_factor = vae_scale_factor

        def postprocess(self, images, output_type="pt", do_denormalize=None):
            return images

    import logging as _logging
    mods = {
        "diffusers": {},
        "diffusers.image_processor": {"VaeImageProcessor": StubImageProcessor},
        "diffusers.loaders": {"FromSingleFileMixin": type("FromSingleFileMixin", (_Mixin,), {}),
                              "IPAdapterMixin": type("IPAdapterMixin", (_Mixin,), {}),
                              "StableDiffusionLoraLoaderMixin": type("StableDiffusionLoraLoaderMixin", (_Mixin,), {}),
                              "TextualInversionLoaderMixin": type("TextualInversionLoaderMixin", (_Mixin,), {})},
        "diffusers.models": {"AutoencoderKL": object},
        "diffusers.schedulers": {"KarrasDiffusionSchedulers": object},
        "diffusers.utils": {"logging": types.SimpleNamespace(get_logger=_logging.getLogger),
                            "replace_example_docstring": lambda doc: (lambda f: f)},
        "diffusers.utils.torch_utils": {"randn_tensor": _counter_randn},
        "diffusers.pipelines": {},
        "diffusers.pipelines.pipeline_utils": {"DiffusionPipeline": StubDiffusionPipeline,
                                               "StableDiffusionMixin": type("StableDiffusionMixin", (_Mixin,), {})},
        # the reference package layout (relative import PIPE:33)
        "refsrc": {}, "refsrc.pipelines": {}, "refsrc.pipelines.diffuman4d": {}, "refsrc.models": {},
        "refsrc.models.unets": {},
        "refsrc.models.unets.unet_multiview_condition": {"UNetMultiviewConditionModel": object},
    }
    for name, attrs in mods.items():
        m = types.ModuleType(name)
        m.__path__ = []
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m
    name = "refsrc.pipelines.diffuman4d.pipeline_diffuman4d"
    spec = importlib.util.spec_from_file_location(name, f"{REF}/src/diffusers/pipelines/diffuman4d/pipeline_diffuman4d.py")
    pipe_mod = importlib.util.module_from_spec(spec)
    pipe_mod.__package__ = "refsrc.pipelines.diffuman4d"
    sys.modules[name] = pipe_mod
    spec.loader.exec_module(pipe_mod)
    pipe_mod.decode_vae = lambda vae, latents, generator=None, batch_size=8: latents  # identity "VAE"

    class RefScheduler(DDIMOracle):
        """the upstream scheduler surface the reference touches (PIPE:265-271,376,420)"""

        def set_timesteps(self, n, device=None):
            super().set_timesteps(n)

        def scale_model_input(self, x, t):
            return x

        def step(self, noise, t, latent, return_dict=False):
            return (super().step(noise, int(t), latent),)

    class FakeVAE:
        dtype = torch.float32
        device = torch.device("cpu")
        config = types.SimpleNamespace(block_out_channels=[1, 1, 1, 1], scaling_factor=1.0)

        def encode(self, x):  # 8x average pooling, 3 -> 4 channels (only sliding_iterative_denoise encodes)
            z = torch.nn.functional.avg_pool2d(x, 8)
            z = torch.cat([z, z.mean(dim=1, keepdim=True)], dim=1)
            return types.SimpleNamespace(latent_dist=types.SimpleNamespace(sample=lambda: z))

    class UNetAdapter:
        def __init__(self, in_channels, pose):
            self.fn = make_fake_unet(in_channels)
            self.config = types.SimpleNamespace(time_cond_proj_dim=None, enable_pose_encoder=pose)

        def __call__(self, x, timestep=None, skeletons=None, domains=None, num_frames=1, return_dict=False):
            return (self.fn(x, timestep, skeletons, domains, num_frames),)

    def make_pipe(pose, prediction_type="epsilon"):
        cin = 4 + 6 + (0 if pose else 4) + 1
        sc = SchedulerConfig(prediction_type=prediction_type)
        return pipe_mod.Diffuman4DPipeline(FakeVAE(), UNetAdapter(cin, pose), RefScheduler(sc)), cin

    return pipe_mod, make_pipe


def gen_pipeline():
    """Run the reference pipeline class on stubs; see the module docstring."""
    pipe_mod, make_pipe = _load_ref_pipeline()
    out = {"cases": {}}
    h = w = 8
    g = torch.Generator().manual_seed(2024)
    rn = lambda *s: torch.randn(*s, generator=g)

    # ---- (A)/(B): one window through __call__ (2 inference steps, staggered timestep indices)
    for tag, pose, guidance, pred in (("call_pose_cfg", True, 2.0, "epsilon"), ("call_nopose_nocfg", False, 1.0, "epsilon"),
                                      ("call_pose_cfg_vpred", True, 3.5, "v_prediction")):
        pipe, cin = make_pipe(pose, pred)
        F_ = 5
        mask = torch.ones(F_, 1, h, w)
        mask[:2] = 0
        inp = {"latents": rn(F_, 4, h, w), "pixel_latents": rn(F_, 4, h, w), "plucker": rn(F_, 6, h, w).clamp(-1, 1),
               "skeletons": ((torch.rand(F_, 3, 8 * h, 8 * w, generator=g) * 2 - 1) if pose
                             else rn(F_, 4, h, w)).half().float(),
               "cond_mask": mask, "timestep_indices": torch.tensor([0, 0, 1, 2, 3])}
        schedulers, timesteps = pipe.parepare_schedulers(6, F_)
        ti = inp["timestep_indices"].clone()
        res = pipe(pixel_values_latents=inp["pixel_latents"].clone(), plucker_embeds_latents=inp["plucker"].clone(),
                   skeletons_latents=inp["skeletons"].clone(), cond_masks_latents=inp["cond_mask"].clone(),
                   latents=inp["latents"].clone(), domains=["spatial"], num_inference_steps=2, schedulers=schedulers,
                   timesteps=timesteps, timestep_indices=ti, guidance_scale=guidance, output_type="latent")
        out["cases"][tag] = {"pose": pose, "guidance": guidance, "prediction_type": pred, "n_steps_table": 6,
                             "in": {**inp, "skeletons": inp["skeletons"].half()},
                             "timesteps_table": timesteps.clone(), "out_latents": res, "out_timestep_indices": ti}
        print("pipeline", tag, float(res.abs().mean()), ti.tolist())

    # ---- (C)/(D): sliding_iterative_denoise, spatial and temporal, recording every window the reference visits
    for tag, domain, n_in, n_tg, ws, stride, bidir, rounds in (("slide_spatial", "spatial", 2, 6, 3, 1, False, 2),
                                                               ("slide_temporal_bidir", "temporal", 4, 4, 2, 2, True, 1)):
        pipe, cin = make_pipe(True)
        windows = []
        orig_call = pipe_mod.Diffuman4DPipeline.__call__

        class Recording(pipe_mod.Diffuman4DPipeline):
            def __call__(self, **kw):
                # frame ids are tagged into plucker[:, 0, 0, 0] below, so the visited window can be read back here
                windows.append({"timestep_indices": kw["timestep_indices"].clone(),
                                "frames": (kw["plucker_embeds_latents"][:, 0, 0, 0] * 100).round().long()})
                return orig_call(self, **kw)

        pipe.__class__ = Recording
        n = n_in + n_tg
        mask = torch.ones(n, 1, 8 * h, 8 * w)
        mask[:n_in] = 0
        pixel = torch.rand(n, 3, 8 * h, 8 * w, generator=g) * 2 - 1
        inp = {"pixel_values": pixel, "plucker": rn(n, 6, h, w).clamp(-1, 1),
               "skeletons": (torch.rand(n, 3, 8 * h, 8 * w, generator=g) * 2 - 1).half().float(), "cond_masks": mask,
               "latents": rn(n, 4, h, w), "timestep_indices": torch.zeros(n, dtype=torch.int64)}
        inp["plucker"][:, 0, 0, 0] = torch.arange(n, dtype=torch.float32) / 100
        res = pipe.sliding_iterative_denoise(
            pixel_values=inp["pixel_values"].clone(), plucker_embeds=inp["plucker"].clone(), skeletons=inp["skeletons"].clone(),
            cond_masks=inp["cond_masks"].clone(), latents=inp["latents"].clone(), domain=domain,
            timestep_indices=inp["timestep_indices"].clone(), window_size=ws, sliding_stride=stride, sliding_shift=0,
            bidirectional=bidir, num_denoising_steps=1, alternation_rounds=rounds, guidance_scale=2.0, tqdm=lambda it, total=None: it)
        z = torch.nn.functional.avg_pool2d(pixel, 8)
        inp["pixel_latents"] = torch.cat([z, z.mean(dim=1, keepdim=True)], dim=1)  # what the fake VAE encoded
        inp["cond_mask_latents"] = torch.nn.functional.interpolate(mask, size=(h, w), mode="nearest")
        stored = {k: v for k, v in inp.items() if k not in ("pixel_values", "cond_masks")}
        stored["skeletons"] = inp["skeletons"].half()
        out["cases"][tag] = {"domain": domain, "window_size": ws, "sliding_stride": stride, "bidirectional": bidir,
                             "alternation_rounds": rounds, "in": stored, "out_latents": res["latents"],
                             "out_timestep_indices": res["timestep_indices"], "fully_denoised": res["fully_denoised"],
                             "window_timestep_indices": [w_["timestep_indices"] for w_ in windows],
                             "window_frames": [w_["frames"] for w_ in windows], "n_input": n_in}
        print("pipeline", tag, float(res["latents"].abs().mean()), res["timestep_indices"].tolist(), len(windows), "windows")

    # ---- the reference's argument checks (PIPE:464,481,486,547)
    errs = {}
    pipe, _ = make_pipe(True)
    n = 8
    mask = torch.ones(n, 1, 8 * h, 8 * w)
    mask[:2] = 0
    base = dict(pixel_values=torch.zeros(n, 3, 8 * h, 8 * w), plucker_embeds=torch.zeros(n, 6, h, w),
                skeletons=torch.zeros(n, 3, 8 * h, 8 * w), cond_masks=mask, latents=torch.zeros(n, 4, h, w), domain="spatial",
                window_size=3, num_denoising_steps=1, alternation_rounds=1, tqdm=lambda it, total=None: it)
    for tag, kw in (("stride", dict(sliding_stride=2, timestep_indices=torch.zeros(n, dtype=torch.int64))),
                    ("unequal_targets", dict(sliding_stride=1, timestep_indices=torch.tensor([0, 0, 1, 1, 1, 1, 1, 2]))),
                    ("nonzero_inputs", dict(sliding_stride=1, timestep_indices=torch.tensor([1, 0, 0, 0, 0, 0, 0, 0])))):
        try:
            pipe.sliding_iterative_denoise(**{**base, **kw})
            errs[tag] = None
        except ValueError as e:
            errs[tag] = str(e)
        print("pipeline error", tag, "->", errs[tag])
    out["errors"] = errs
    torch.save(out, f"{HERE}/pipeline_ref.pt")


def gen_sampler():
    """Drive the reference's ``SlidingIterativeSampler`` (src/samplers/sliding_iterative_sampler.py) -- its task lists,
    sample loading, grid bookkeeping -- with the reference pipeline-on-stubs above and the synthetic dataset."""
    pipe_mod, make_pipe = _load_ref_pipeline()
    sys.path.insert(0, HERE)
    from synthetic_dataset import SyntheticSpaTemDataset
    import logging as _logging

    saved = []

    class RankedLogger:
        def __init__(self, *a, **k):
            self._l = _logging.getLogger("ref")

        def __getattr__(self, name):
            return getattr(self._l, name)

    mods = {"src": {}, "src.data": {}, "src.data.spatem_dataset": {"SpaTemDataset": object},
            "src.diffusers": {}, "src.diffusers.pipelines": {}, "src.diffusers.pipelines.diffuman4d": {},
            "src.diffusers.pipelines.diffuman4d.pipeline_diffuman4d": {"Diffuman4DPipeline": pipe_mod.Diffuman4DPipeline},
            "src.samplers": {}, "src.samplers.utils": {},
            "src.samplers.utils.sampling_utils": {
                "save_sampling_results": lambda sample, output_dir=None: saved.append(
                    {"alt": sample["alt"], "domain": sample["domain"], "domain_label": sample["domain_label"],
                     "labels": list(sample["labels"]), "timestep_indices": sample["timestep_indices"].clone(),
                     "fully_denoised": sample["fully_denoised"].clone()}),
                "check_sampling_results": lambda *a, **k: True},
            "src.utils": {"RankedLogger": RankedLogger}}
    for name, attrs in mods.items():
        m = types.ModuleType(name)
        m.__path__ = []
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m
    samp_mod = load_by_path("src.samplers.sliding_iterative_sampler", f"{REF}/src/samplers/sliding_iterative_sampler.py")

    out = {"cases": {}}
    for tag, kw in (("v6_t4_stride1", dict(spa_label_range=[0, 6, 1], tem_label_range=[0, 4, 1], input_spa_labels=[1, 4],
                                           window_size=2, sliding_stride=1, bidirectional=True, alternation_rounds=3)),
                    ("v5_t2_stride2_unidir", dict(spa_labels=[0, 2, 3, 5, 7], tem_labels=[3, 9], input_spa_labels=[2],
                                                   window_size=2, sliding_stride=2, bidirectional=False, alternation_rounds=2))):
        saved.clear()
        _RANDN_CALLS[0] = 0
        n_cams = 8
        pipe, _ = make_pipe(True)
        sampler = samp_mod.SlidingIterativeSampler(dataset=SyntheticSpaTemDataset(n_cams), pipelines=[pipe], output_dir=None,
                                                   num_denoising_steps=1, guidance_scale=2.0, sliding_shift=0, **kw)
        sampler.execute_tasks()
        grid = {(s, t): sampler.latents[s][t].clone() for s in sampler.spa_labels for t in sampler.tem_labels}
        ti = {(s, t): int(sampler.timestep_indices[s][t]) for s in sampler.spa_labels for t in sampler.tem_labels}
        out["cases"][tag] = {"kwargs": kw, "n_cams": n_cams, "all_tasks": sampler.all_tasks, "grid_latents": grid,
                             "grid_timestep_indices": ti, "saved": list(saved)}
        print("sampler", tag, len(saved), "tasks", sorted(set(ti.values())),
              float(torch.stack(list(grid.values())).abs().mean()))
    # the constructor's argument checks (SAMP:72-90)
    errs = {}
    for tag, kw in (("window_gt_targets", dict(spa_label_range=[0, 4, 1], input_spa_labels=[1], window_size=4)),
                    ("targets_mod_stride", dict(spa_label_range=[0, 6, 1], input_spa_labels=[1], window_size=2, sliding_stride=2)),
                    ("tems_mod_stride", dict(spa_label_range=[0, 6, 1], input_spa_labels=[1, 4], tem_label_range=[0, 3, 1],
                                             window_size=2, sliding_stride=2)),
                    ("window_gt_tems", dict(spa_label_range=[0, 6, 1], input_spa_labels=[1, 4], tem_label_range=[0, 1, 1],
                                            window_size=2, alternation_rounds=2)),
                    ("no_spa", dict(spa_label_range=None, spa_labels=None))):
        try:
            samp_mod.SlidingIterativeSampler(dataset=None, pipelines=[], **{"tem_label_range": [0, 4, 1], **kw})
            errs[tag] = None
        except ValueError as e:
            errs[tag] = str(e)
        print("sampler error", tag, "->", errs[tag])
    out["errors"] = errs
    torch.save(out, f"{HERE}/sampler_ref.pt")


if __name__ == "__main__":
    if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "src", "diffusers")):
        raise SystemExit("usage: python tests/golden/gen_golden.py <Diffuman4D checkout>")
    REF = os.path.abspath(sys.argv[1])
    gen_sampler()
    gen_unet()
    gen_pipeline()
    gen_pose_encoder()
    gen_mv_block()
    try:
        gen_plucker()
    except Exception as e:  # value-range fixture only; not a parity gate
        print("plucker fixture skipped:", repr(e))
