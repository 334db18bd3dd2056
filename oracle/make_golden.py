"""Generate tests/golden/*.npz from the REAL reference modules.

TEST INFRASTRUCTURE.  Run in the build container only (needs /root/reference):

    python -m oracle.make_golden

The reference ships no golden vectors (SURVEY.md §4), so these fixtures are
outputs of the reference's own ``DiffusionTransformer`` / ``OobleckEncoder`` /
``OobleckDecoder`` / ``AudioAutoencoder`` / ``RotaryEmbedding`` / ``SnakeBeta``
classes on seeded inputs.  Weights are NOT stored: they are re-derived from the
seed by ``oracle.dit_oracle.make_dit_weights`` / ``oracle.oobleck_oracle
.make_oobleck_weights`` (torch CPU generator, same torch build on the GPU box)
and a checksum of them is stored to detect RNG drift.
"""
import json
import os

import numpy as np
import torch

from . import dit_oracle as do
from . import oobleck_oracle as oo
from . import ref_shims

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

DIT_SMALL = dict(io_channels=64, embed_dim=256, depth=2, num_heads=4, cond_token_dim=128,
                 global_cond_dim=256, project_cond_tokens=False,
                 transformer_type="continuous_transformer")
DEC_SMALL = dict(out_channels=2, channels=32, c_mults=[1, 2, 4], strides=[2, 4, 8], latent_dim=8,
                 use_snake=True, final_tanh=False)
ENC_SMALL = dict(in_channels=2, channels=32, c_mults=[1, 2, 4], strides=[2, 4, 8], latent_dim=16,
                 use_snake=True)


def weights_checksum(sd):
    return float(sum(v.double().abs().sum() for v in sd.values()))


def _np(t):
    return t.detach().cpu().numpy()


def gen_dit(ref, gtype, path, patch_size=1, qk_norm=False):
    cfg = dict(DIT_SMALL, global_cond_type=gtype)
    seed = 11 if gtype == "prepend" else 12
    if patch_size > 1:
        cfg["patch_size"] = patch_size
        seed = 13
    if qk_norm:
        cfg["attn_kwargs"] = {"qk_norm": True}
        seed = 14
    sd = do.make_dit_weights(cfg, seed=seed)
    m = ref.dit.DiffusionTransformer(**cfg).eval()
    m.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(100 + seed)
    B, L, M = 2, 200, 10
    x = torch.randn(B, 64, L, generator=g)
    t = torch.rand(B, generator=g)
    c = torch.randn(B, M, 128, generator=g)
    ge = torch.randn(B, 256, generator=g)
    neg = torch.randn(B, M, 128, generator=g)
    out = {"cfg": json.dumps(cfg), "seed": seed, "wsum": weights_checksum(sd),
           "x": _np(x), "t": _np(t), "cross": _np(c), "glob": _np(ge), "neg": _np(neg)}
    with torch.no_grad():
        out["y_nocfg"] = _np(m(x, t, cross_attn_cond=c, global_embed=ge, cfg_scale=1.0))
        out["y_cfg7"] = _np(m(x, t, cross_attn_cond=c, global_embed=ge, cfg_scale=7.0))
        out["y_cfg4_phi"] = _np(m(x, t, cross_attn_cond=c, global_embed=ge, cfg_scale=4.0, scale_phi=0.7))
        out["y_neg3"] = _np(m(x, t, cross_attn_cond=c, global_embed=ge, negative_cross_attn_cond=neg, cfg_scale=3.0))
        y, info = m(x, t, cross_attn_cond=c, global_embed=ge, cfg_scale=1.0, return_info=True)
        out["hidden_last"] = _np(info["hidden_states"][-1])
    np.savez_compressed(path, **out)


def gen_dit_concat_prepend(ref, path):
    """input_concat_cond (16 extra channels, half the latent length: exercises the nearest-neighbour resize) and
    prepend_cond (3 tokens of width 96) through the real DiffusionTransformer (models/dit.py:157-173,185-195,281-311)."""
    cfg = dict(DIT_SMALL, input_concat_dim=16, prepend_cond_dim=96)
    seed = 15
    sd = do.make_dit_weights(cfg, seed=seed)
    m = ref.dit.DiffusionTransformer(**cfg).eval()
    m.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(100 + seed)
    B, L, M = 2, 200, 10
    x = torch.randn(B, 64, L, generator=g)
    t = torch.rand(B, generator=g)
    c = torch.randn(B, M, 128, generator=g)
    ge = torch.randn(B, 256, generator=g)
    ic = torch.randn(B, 16, L // 2, generator=g)
    pc = torch.randn(B, 3, 96, generator=g)
    out = {"cfg": json.dumps(cfg), "seed": seed, "wsum": weights_checksum(sd),
           "x": _np(x), "t": _np(t), "cross": _np(c), "glob": _np(ge), "concat": _np(ic), "prepend": _np(pc)}
    kw = dict(cross_attn_cond=c, global_embed=ge, input_concat_cond=ic, prepend_cond=pc,
              prepend_cond_mask=torch.ones(B, 3, dtype=torch.bool))
    with torch.no_grad():
        out["y_nocfg"] = _np(m(x, t, cfg_scale=1.0, **kw))
        out["y_cfg5"] = _np(m(x, t, cfg_scale=5.0, **kw))
        out["y_cfg3_phi"] = _np(m(x, t, cfg_scale=3.0, scale_phi=0.5, **kw))
        out["y_concat_only"] = _np(m(x, t, cross_attn_cond=c, global_embed=ge, input_concat_cond=ic, cfg_scale=4.0))
    np.savez_compressed(path, **out)


def gen_rope(ref, path):
    rot = ref.transformer.RotaryEmbedding(32)
    freqs, _ = rot.forward_from_seq_len(1025)
    g = torch.Generator().manual_seed(5)
    q = torch.randn(1, 2, 1025, 64, generator=g)
    q_rot = ref.transformer.apply_rotary_pos_emb(q, freqs)
    # one-hot index probe: rows of the identity through rotate_half show the pairing
    eye = torch.eye(32)
    pairing = ref.transformer.rotate_half(eye)
    np.savez_compressed(path, inv_freq=_np(rot.inv_freq), freqs=_np(freqs), q=_np(q[:, :, ::41]),
                        q_rot=_np(q_rot[:, :, ::41]), pos=np.arange(1025)[::41], pairing=_np(pairing))


def gen_snake(ref, path):
    g = torch.Generator().manual_seed(6)
    sn = ref.blocks.SnakeBeta(24)
    with torch.no_grad():
        sn.alpha.copy_(torch.randn(24, generator=g) * 0.5)
        sn.beta.copy_(torch.randn(24, generator=g) * 0.5)
    x = torch.randn(3, 24, 301, generator=g) * 3.0
    with torch.no_grad():
        y = sn(x)
    np.savez_compressed(path, alpha=_np(sn.alpha), beta=_np(sn.beta), x=_np(x), y=_np(y))


def gen_oobleck(ref, path):
    dsd = oo.make_oobleck_weights(oo.decoder_param_shapes(DEC_SMALL), seed=21,
                                  transposed=oo.decoder_transposed_prefixes(DEC_SMALL))
    esd = oo.make_oobleck_weights(oo.encoder_param_shapes(ENC_SMALL), seed=22)
    dec = ref.autoencoders.OobleckDecoder(**DEC_SMALL).eval()
    enc = ref.autoencoders.OobleckEncoder(**ENC_SMALL).eval()
    dec.load_state_dict(dsd, strict=True)
    enc.load_state_dict(esd, strict=True)
    g = torch.Generator().manual_seed(23)
    z = torch.randn(2, 8, 40, generator=g)
    a = torch.randn(2, 2, 64 * 37, generator=g) * 0.5
    with torch.no_grad():
        audio = dec(z)
        h = enc(a)
    # AudioAutoencoder wrapper incl. chunked reconstruct with Bartlett cross-fade
    bott = ref.bottleneck.VAEBottleneck()
    ae = ref.autoencoders.AudioAutoencoder(enc, dec, latent_dim=8, downsampling_ratio=64, sample_rate=16000,
                                           io_channels=2, bottleneck=bott).eval()
    torch.manual_seed(77)
    with torch.no_grad():
        rec = ae.reconstruct_audio(a.clone(), chunked=True, chunk_size=7, overlap=1, max_batch_size=3)
    torch.manual_seed(78)
    with torch.no_grad():
        dec_chunked = ae.decode_audio(z.clone(), chunked=True, chunk_size=16, overlap=4, max_batch_size=2)
    np.savez_compressed(path, dec_cfg=json.dumps(DEC_SMALL), enc_cfg=json.dumps(ENC_SMALL),
                        dec_seed=21, enc_seed=22, dec_wsum=weights_checksum(dsd), enc_wsum=weights_checksum(esd),
                        z=_np(z), audio=_np(audio), a=_np(a), h=_np(h), rec=_np(rec), rec_seed=77,
                        dec_chunked=_np(dec_chunked))


# BASELINE.json configs[0]: Oobleck VAE reconstruct, 1 s mono 16 kHz white noise, the full SA-Open / SA-2.0 VAE
# (autoencoders/stable_audio_2_0_vae.json with audio_channels / in_channels / out_channels / io_channels = 1,
# sample_rate 16000; SURVEY.md Appendix B), reconstruct_audio(chunked=True, chunk_size=7, overlap=1,
# max_batch_size=20) as reconstruct_audios.py calls it for 1 s frames.
MONO_ENC = dict(in_channels=1, channels=128, c_mults=[1, 2, 4, 8, 16], strides=[2, 4, 4, 8, 8], latent_dim=128,
                use_snake=True)
MONO_DEC = dict(out_channels=1, channels=128, c_mults=[1, 2, 4, 8, 16], strides=[2, 4, 4, 8, 8], latent_dim=64,
                use_snake=True, final_tanh=False)


class seeded_randn_like:
    """Replaces torch.randn_like (the VAE draw, reference models/bottleneck.py:50) by draws from a seeded CPU
    generator, so that the reference run here and the native run on the GPU box see the same noise."""

    def __init__(self, seed):
        self.gen = torch.Generator().manual_seed(seed)

    def __call__(self, t, **kw):
        return torch.randn(t.shape, generator=self.gen, dtype=torch.float32).to(device=t.device, dtype=t.dtype)

    def __enter__(self):
        self.prev = torch.randn_like
        torch.randn_like = self
        return self

    def __exit__(self, *exc):
        torch.randn_like = self.prev


class cpu_stream_randn_like:
    """Replaces torch.randn_like by draws from the DEFAULT CPU generator (moved to the tensor's device): after
    torch.manual_seed(s) a CUDA run sees the numbers the CPU reference drew when gen_oobleck made its golden."""

    def __call__(self, t, **kw):
        return torch.randn(t.shape, dtype=torch.float32).to(device=t.device, dtype=t.dtype)

    def __enter__(self):
        self.prev = torch.randn_like
        torch.randn_like = self
        return self

    def __exit__(self, *exc):
        torch.randn_like = self.prev


def gen_config1(ref, path):
    esd = oo.make_oobleck_weights(oo.encoder_param_shapes(MONO_ENC), seed=31)
    dsd = oo.make_oobleck_weights(oo.decoder_param_shapes(MONO_DEC), seed=32,
                                  transposed=oo.decoder_transposed_prefixes(MONO_DEC))
    cfg = {"model_type": "autoencoder", "sample_size": 65536, "sample_rate": 16000, "audio_channels": 1,
           "model": {"encoder": {"type": "oobleck", "config": MONO_ENC}, "decoder": {"type": "oobleck", "config": MONO_DEC},
                     "bottleneck": {"type": "vae"}, "latent_dim": 64, "downsampling_ratio": 2048, "io_channels": 1}}
    # = create_autoencoder_from_config(cfg) (autoencoders.py:737-787); built directly because the factory's lazy
    # relative imports need the reference registered in sys.modules, which ref_shims deliberately avoids
    enc = ref.autoencoders.OobleckEncoder(**MONO_ENC)
    dec = ref.autoencoders.OobleckDecoder(**MONO_DEC)
    ae = ref.autoencoders.AudioAutoencoder(enc, dec, latent_dim=64, downsampling_ratio=2048, sample_rate=16000,
                                           io_channels=1, bottleneck=ref.bottleneck.VAEBottleneck()).eval()
    ae.encoder.load_state_dict(esd, strict=True)
    ae.decoder.load_state_dict(dsd, strict=True)
    g = torch.Generator().manual_seed(33)
    audio = 0.5 * torch.randn(1, 1, 16000, generator=g).clamp(-1, 1)      # SURVEY.md 8(d) config 1
    with torch.no_grad(), seeded_randn_like(34):
        rec = ae.reconstruct_audio(audio.clone(), chunked=True, chunk_size=7, overlap=1, max_batch_size=20)
    np.savez_compressed(path, model_cfg=json.dumps(cfg), enc_seed=31, dec_seed=32, noise_seed=34,
                        enc_wsum=weights_checksum(esd), dec_wsum=weights_checksum(dsd), audio=_np(audio), rec=_np(rec))


# ------------------------------------------------------------------------------------------------------------------
# Reference outputs for tests/test_oracle_vs_reference.py and the chunking test of tests/test_host_logic.py.
# ------------------------------------------------------------------------------------------------------------------
def keys_and_shapes(sd):
    """A state dict's key -> shape map as one JSON string (what a strict load of it checks)."""
    return json.dumps({k: list(v.shape) for k, v in sorted(sd.items())})


def seeded_state_dict(sd, seed):
    """Seeded values for every tensor of `sd` (fan-in scaled), so that a module's weights need not be stored."""
    g = torch.Generator().manual_seed(seed)
    return {k: torch.randn(v.shape, generator=g) / (v.shape[-1] ** 0.5 if v.dim() > 1 else 1.0)
            for k, v in sorted(sd.items())}


def sample_index(shape, n=512, seed=0):
    """A fixed seeded sample of n flat indices of a tensor of `shape` (what a golden keeps of a large output)."""
    numel = int(np.prod(shape))
    return torch.randperm(numel, generator=torch.Generator().manual_seed(seed))[:min(n, numel)].sort().values


class FakeT5Tokenizer:
    """Stands for AutoTokenizer.from_pretrained('t5-base') (no model files offline): whitespace 'tokens', padded."""

    def __call__(self, texts, truncation=True, max_length=128, padding="max_length", return_tensors="pt"):
        ids = torch.zeros(len(texts), max_length, dtype=torch.long)
        mask = torch.zeros(len(texts), max_length, dtype=torch.long)
        for i, t in enumerate(texts):
            toks = [(sum(map(ord, w)) % 1000) + 1 for w in t.split()][:max_length]
            ids[i, :len(toks)] = torch.tensor(toks)
            mask[i, :len(toks)] = 1
        return {"input_ids": ids, "attention_mask": mask}


class FakeT5Encoder(torch.nn.Module):
    """Stands for T5EncoderModel.from_pretrained('t5-base'): a seeded embedding table."""

    def __init__(self, dim=768):
        super().__init__()
        g = torch.Generator().manual_seed(3)
        self.emb = torch.nn.Parameter(torch.randn(1001, dim, generator=g))

    def forward(self, input_ids=None, attention_mask=None):
        return {"last_hidden_state": self.emb[input_ids]}


def txt2audio_cfg_with_t5(cfg):
    """stable_audio_2_0.json conditions on CLAP text features (laion_clap + a checkpoint file: an absent third-party
    model); its prompt branch is swapped for the T5 one, the DiT / VAE / number-conditioner parts stay as shipped."""
    cfg = json.loads(json.dumps(cfg))
    for c in cfg["model"]["conditioning"]["configs"]:
        if c["type"] == "clap_text":
            c["type"], c["config"] = "t5", {"t5_model_name": "t5-base", "max_length": 128}
    return cfg


def txt2audio_small(cfg):
    """The same model cut to 2 DiT blocks and a 2-stage VAE, small enough to build with real tensors."""
    small = json.loads(json.dumps(cfg))
    small["model"]["diffusion"]["config"]["depth"] = 2
    for half in ("encoder", "decoder"):
        c = small["model"]["pretransform"]["config"][half]["config"]
        c["c_mults"], c["strides"], c["channels"] = [1, 2], [2, 4], 32
    small["model"]["pretransform"]["config"]["downsampling_ratio"] = 8
    return small


TXT2AUDIO_META = [{"prompt": "warm analog pad with slow attack", "seconds_start": 0, "seconds_total": 30},
                  {"prompt": "drum loop 120 bpm", "seconds_start": 5, "seconds_total": 47}]
TXT2AUDIO_PROMPT_ROWS = 8           # >= the most words of a TXT2AUDIO_META prompt


def toy_denoiser():
    """Linear v-prediction stand-in of the sampler tests (seeded)."""
    torch.manual_seed(0)
    w = torch.randn(4, 4) * 0.3
    return w, lambda x, t, **kw: torch.einsum("ij,bjl->bil", w, x) * (1 + t[:, None, None])


INPAINT_MASK_ARGS = dict(cropfrom=10.0, pastefrom=20.0, pasteto=90.0, maskstart=25.0, maskend=80.0, softnessL=12.0,
                         softnessR=7.0, marination=0.2)


def dit_case(gtype, seed):
    """Config, weights and seeded inputs of one tiny DiffusionTransformer case of gen_dit_cases."""
    cfg = dict(io_channels=64, embed_dim=128, depth=3, num_heads=2, cond_token_dim=64, global_cond_dim=128,
               project_cond_tokens=bool(seed), transformer_type="continuous_transformer", global_cond_type=gtype)
    g = torch.Generator().manual_seed(seed)
    x, t = torch.randn(3, 64, 33, generator=g), torch.rand(3, generator=g)
    c, ge = torch.randn(3, 7, 64, generator=g), torch.randn(3, 128, generator=g)
    return cfg, do.make_dit_weights(cfg, seed=seed), (x, t, c, ge)


DIT_CASE_GUIDANCE = {"cfg1": dict(cfg_scale=1.0), "cfg5": dict(cfg_scale=5.0), "cfg5_phi": dict(cfg_scale=5.0, scale_phi=0.5)}


def gen_dit_cases(ref, path):
    """DiffusionTransformer outputs at three guidance settings for prepend / adaLN global conditioning, 2 seeds
    (a sample_index() sample of each output; the inputs are re-derived from the seed, their checksum is kept)."""
    out = {}
    for gtype in ("prepend", "adaLN"):
        for seed in (0, 1):
            cfg, sd, (x, t, c, ge) = dit_case(gtype, seed)
            m = ref.dit.DiffusionTransformer(**cfg).eval()
            m.load_state_dict(sd, strict=True)
            p = f"{gtype}_{seed}_"
            out.update({p + "wsum": weights_checksum(sd), p + "xsum": float(sum(v.double().abs().sum() for v in (x, c, ge)))})
            with torch.no_grad():
                for name, kw in DIT_CASE_GUIDANCE.items():
                    y = m(x, t, cross_attn_cond=c, global_embed=ge, **kw)
                    out[p + name] = _np(y.flatten()[sample_index(y.shape)])
    np.savez_compressed(path, **out)


def gen_module_keys(ref, path):
    """State-dict keys and shapes of the reference's DiT (both global-conditioning layouts), Oobleck decoder and
    encoder, and of the autoencoder built by its factory from the shipped SA-2.0 VAE config (stored alongside)."""
    out = {}
    for gtype in ("prepend", "adaLN"):
        cfg = dict(io_channels=64, embed_dim=128, depth=2, num_heads=2, cond_token_dim=64, global_cond_dim=128,
                   project_cond_tokens=False, transformer_type="continuous_transformer", global_cond_type=gtype)
        out[f"dit_{gtype}_cfg"] = json.dumps(cfg)
        out[f"dit_{gtype}_keys"] = keys_and_shapes(ref.dit.DiffusionTransformer(**cfg).state_dict())
    dcfg = dict(out_channels=2, channels=32, c_mults=[1, 2, 4], strides=[2, 4, 8], latent_dim=8, use_snake=True,
                final_tanh=False)
    ecfg = dict(in_channels=2, channels=32, c_mults=[1, 2, 4], strides=[2, 4, 8], latent_dim=16, use_snake=True)
    out["decoder_cfg"], out["encoder_cfg"] = json.dumps(dcfg), json.dumps(ecfg)
    out["decoder_keys"] = keys_and_shapes(ref.autoencoders.OobleckDecoder(**dcfg).state_dict())
    out["encoder_keys"] = keys_and_shapes(ref.autoencoders.OobleckEncoder(**ecfg).state_dict())
    cfg_path = os.path.join(ref_shims.REFERENCE_ROOT, "stable_audio_tools/configs/model_configs/autoencoders",
                            "stable_audio_2_0_vae.json")
    vae_cfg = json.load(open(cfg_path))
    with ref_shims.reference_modules(ref):
        vae = ref.factory.create_model_from_config(json.loads(json.dumps(vae_cfg)))
    out["vae_cfg"], out["vae_keys"] = json.dumps(vae_cfg), keys_and_shapes(vae.state_dict())
    out["vae_downsampling_ratio"] = vae.downsampling_ratio
    np.savez_compressed(path, **out)


def gen_sampler_cases(ref, path):
    """The reference's sample_k (driving the restated k-diffusion samplers) on a toy denoiser: plain sampling with
    injected SDE noise, and init-audio / inpainting sampling with every random draw from one seeded stream."""
    import functools
    K = __import__("k_diffusion")
    w, toy = toy_denoiser()
    noise = torch.randn(2, 4, 16)
    seq = torch.stack([torch.randn(2, 4, 16) for _ in range(8)])
    out = {"w": _np(w), "noise": _np(noise), "sde_noise": _np(seq)}
    for st in ("dpmpp-2m-sde", "dpmpp-3m-sde"):
        # the reference sample_k has no noise_sampler argument: bind it into the sampler it calls
        fn_name = "sample_dpmpp_2m_sde" if "2m" in st else "sample_dpmpp_3m_sde"
        orig = getattr(K.sampling, fn_name)
        it = iter(seq)
        setattr(K.sampling, fn_name, functools.partial(orig, noise_sampler=lambda s, sn: next(it)))
        try:
            out[f"{st}_plain"] = _np(ref.sampling.sample_k(toy, noise.clone(), steps=8, sampler_type=st, sigma_min=0.3,
                                                           sigma_max=50, device="cpu"))
        finally:
            setattr(K.sampling, fn_name, orig)
    L = 48
    out["mask"] = _np(ref.generation.build_mask(L, INPAINT_MASK_ARGS))
    w, toy = toy_denoiser()
    inp_noise, init = torch.randn(2, 4, L), torch.randn(2, 4, L)
    out.update(inpaint_noise=_np(inp_noise), inpaint_init=_np(init))
    mask = torch.from_numpy(out["mask"])
    for st in ("dpmpp-2m-sde", "dpmpp-3m-sde"):
        for name, m in (("inpaint", mask), ("variation", None)):
            with seeded_randn_like(5):
                out[f"{st}_{name}"] = _np(ref.sampling.sample_k(toy, inp_noise.clone(), init.clone(), m, steps=7,
                                                                sampler_type=st, sigma_min=0.3, sigma_max=20,
                                                                device="cpu"))
    np.savez_compressed(path, **out)


def gen_number_conditioner(ref, path):
    with ref_shims.reference_modules(ref):
        import importlib
        cond = importlib.import_module("stable_audio_tools.models.conditioners")
    a = cond.NumberConditioner(64, min_val=0, max_val=512)
    a.load_state_dict(seeded_state_dict(a.state_dict(), 41))
    x, m = a([0.0, 12.5, 600.0])
    np.savez_compressed(path, keys=keys_and_shapes(a.state_dict()), x=_np(x), mask=_np(m))


class fake_t5:
    """with fake_t5(): transformers' T5 tokenizer / encoder loaders return FakeT5Tokenizer / FakeT5Encoder."""

    def __enter__(self):
        import transformers
        from unittest import mock
        self.patches = [mock.patch.object(transformers.AutoTokenizer, "from_pretrained",
                                          classmethod(lambda cls, *a, **k: FakeT5Tokenizer())),
                        mock.patch.object(transformers.T5EncoderModel, "from_pretrained",
                                          classmethod(lambda cls, *a, **k: FakeT5Encoder()))]
        for p in self.patches:
            p.start()
        return self

    def __exit__(self, *exc):
        for p in self.patches:
            p.stop()


def gen_txt2audio(ref, path):
    """The shipped text-to-audio configs through the reference's factory (T5 replaced by the fakes above): full-size
    state-dict keys / shapes and wrapper attributes, and for the 2-block cut (conditioner weights from
    seeded_state_dict(.., 42)) the conditioner's outputs for TXT2AUDIO_META and get_conditioning_inputs of those.
    With the T5 prompt branch both configs give the same model, so everything but the configs is stored once.  Of the
    prompt embedding only the first TXT2AUDIO_PROMPT_ROWS token rows are kept (the rest is padding, exactly zero), of
    cross_attn_cond only the rows after the 128 prompt tokens (the prompt rows equal the prompt embedding)."""
    out, shared = {}, None
    with fake_t5():
        for name in ("stable_audio_open_1_0", "stable_audio_2_0"):
            cfg = json.load(open(os.path.join(ref_shims.REFERENCE_ROOT, "stable_audio_tools/configs/model_configs",
                                              "txt2audio", name + ".json")))
            out[name + "/cfg"] = json.dumps(cfg)
            cfg = txt2audio_cfg_with_t5(cfg)
            with torch.device("meta"), ref_shims.reference_modules(ref):
                full = ref.factory.create_model_from_config(json.loads(json.dumps(cfg)))
            mine = {"keys": keys_and_shapes(full.state_dict()),
                    "attrs": json.dumps({k: getattr(full, k) for k in ("min_input_length", "io_channels",
                                                                       "cross_attn_cond_ids", "global_cond_ids")})}
            torch.manual_seed(0)
            with ref_shims.reference_modules(ref):
                small = ref.factory.create_model_from_config(txt2audio_small(cfg)).eval()
            mine["small_keys"] = keys_and_shapes(small.state_dict())
            small.conditioner.load_state_dict(seeded_state_dict(small.conditioner.state_dict(), 42))
            with torch.no_grad():
                ct = small.conditioner(TXT2AUDIO_META)
            for k, (t, m) in ct.items():
                mine[f"ct/{k}"], mine[f"ct_mask/{k}"] = _np(t.float()), _np(m.float())
            prompt = mine["ct/prompt"]
            assert prompt.shape == (2, 128, 768) and not prompt[:, TXT2AUDIO_PROMPT_ROWS:].any()
            mine["ct/prompt"] = prompt[:, :TXT2AUDIO_PROMPT_ROWS]
            ci = small.get_conditioning_inputs(ct)
            assert torch.equal(ci["cross_attn_cond"][:, :128], ct["prompt"][0])
            mine["ci/cross_attn_cond_tail"] = _np(ci["cross_attn_cond"][:, 128:].float())
            for k in ("cross_attn_mask", "global_cond"):
                mine[f"ci/{k}"] = _np(ci[k].float())
            if shared is None:
                shared = mine
            assert set(mine) == set(shared) and all(np.array_equal(mine[k], shared[k]) for k in mine), name
    np.savez_compressed(path, **out, **shared)


class FakeEncoder(torch.nn.Module):
    """Average-pool 'encoder' (ratio 4, 2 -> 3 channels) so the chunking logic runs on the CPU."""

    def forward(self, x):
        p = torch.nn.functional.avg_pool1d(x, 4)
        return torch.cat([p, p[:, :1] * 0.5 - 3.0], dim=1)


class FakeDecoder(torch.nn.Module):
    def forward(self, z):
        return torch.repeat_interleave(z[:, :2] + z[:, 2:3] * 0.25, 4, dim=-1)


def gen_chunked_fakes(ref, path):
    """The reference AudioAutoencoder's chunked encode / decode / reconstruct around the linear fakes above."""
    ae = ref.autoencoders.AudioAutoencoder(FakeEncoder(), FakeDecoder(), latent_dim=3, downsampling_ratio=4,
                                           sample_rate=16000, io_channels=2, bottleneck=None)
    torch.manual_seed(0)
    a = torch.randn(2, 2, 4 * 37)
    z = torch.randn(2, 3, 41)
    np.savez_compressed(
        path, a=_np(a), z=_np(z),
        enc=_np(ae.encode_audio(a.clone(), chunked=True, chunk_size=8, overlap=2, max_batch_size=3)),
        dec=_np(ae.decode_audio(z.clone(), chunked=True, chunk_size=8, overlap=2, max_batch_size=2)),
        rec=_np(ae.reconstruct_audio(a.clone(), chunked=True, chunk_size=8, overlap=2, max_batch_size=4)))


def gen_reference_cases(ref):
    gen_dit_cases(ref, os.path.join(GOLDEN_DIR, "dit_cases_tiny.npz"))
    gen_module_keys(ref, os.path.join(GOLDEN_DIR, "module_keys.npz"))
    gen_sampler_cases(ref, os.path.join(GOLDEN_DIR, "sampler_cases.npz"))
    gen_number_conditioner(ref, os.path.join(GOLDEN_DIR, "number_conditioner.npz"))
    gen_txt2audio(ref, os.path.join(GOLDEN_DIR, "txt2audio_configs.npz"))
    gen_chunked_fakes(ref, os.path.join(GOLDEN_DIR, "chunked_fake_autoencoder.npz"))


def main():
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    ref = ref_shims.import_reference()
    gen_reference_cases(ref)
    gen_dit(ref, "prepend", os.path.join(GOLDEN_DIR, "dit_prepend_small.npz"))
    gen_dit(ref, "adaLN", os.path.join(GOLDEN_DIR, "dit_adaln_small.npz"))
    gen_dit(ref, "prepend", os.path.join(GOLDEN_DIR, "dit_patch2_small.npz"), patch_size=2)
    gen_dit(ref, "prepend", os.path.join(GOLDEN_DIR, "dit_qknorm_small.npz"), qk_norm=True)
    gen_dit_concat_prepend(ref, os.path.join(GOLDEN_DIR, "dit_concat_prepend_small.npz"))
    gen_rope(ref, os.path.join(GOLDEN_DIR, "rope_1025.npz"))
    gen_snake(ref, os.path.join(GOLDEN_DIR, "snake_beta.npz"))
    gen_oobleck(ref, os.path.join(GOLDEN_DIR, "oobleck_small.npz"))
    gen_config1(ref, os.path.join(GOLDEN_DIR, "config1_mono16k.npz"))
    for f in sorted(os.listdir(GOLDEN_DIR)):
        print(f, os.path.getsize(os.path.join(GOLDEN_DIR, f)))


if __name__ == "__main__":
    main()
