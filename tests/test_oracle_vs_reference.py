"""CPU: the oracle restatements and the drop-in modules against outputs, state-dict keys and shipped configs of the
REAL reference modules, stored as golden data (tests/golden, made by oracle/make_golden.py:gen_reference_cases):
fresh DiT cases beyond tests/test_oracle_golden.py, state-dict key parity, the reference's factory on its shipped
configs, its sampler front end and its number conditioner."""
import json

import numpy as np
import pytest
import torch

from helpers import load_golden, max_abs, rel_l2
from oracle import dit_oracle as do
from oracle import make_golden as mg


def _keys_and_shapes(golden_json):
    return {k: tuple(v) for k, v in json.loads(str(golden_json)).items()}


def _state_keys(sd):
    return {k: tuple(v.shape) for k, v in sd.items()}


@pytest.mark.parametrize("gtype", ["prepend", "adaLN"])
@pytest.mark.parametrize("seed", [0, 1])
def test_dit_oracle_vs_live_reference(gtype, seed):
    g = load_golden("dit_cases_tiny.npz")
    p = f"{gtype}_{seed}_"
    cfg, sd, (x, t, c, ge) = mg.dit_case(gtype, seed)
    assert abs(mg.weights_checksum(sd) - float(g[p + "wsum"])) <= 1e-9 * float(g[p + "wsum"])
    xsum = float(sum(v.double().abs().sum() for v in (x, c, ge)))
    assert abs(xsum - float(g[p + "xsum"])) <= 1e-9 * xsum, "seeded inputs drifted from the golden run"
    with torch.no_grad():
        for name, kw in mg.DIT_CASE_GUIDANCE.items():
            y = do.dit_forward(sd, cfg, x, t, c, ge, **kw)
            assert max_abs(y.flatten()[mg.sample_index(y.shape)], torch.from_numpy(g[p + name])) <= 1e-5, name


def test_dropin_state_dict_keys_match_reference():
    from stable_audio_tools.models.autoencoders import OobleckDecoder, OobleckEncoder
    from stable_audio_tools.models.dit import DiffusionTransformer
    g = load_golden("module_keys.npz")
    for gtype in ("prepend", "adaLN"):
        cfg = json.loads(str(g[f"dit_{gtype}_cfg"]))
        theirs = _keys_and_shapes(g[f"dit_{gtype}_keys"])
        assert _state_keys(DiffusionTransformer(**cfg).state_dict()) == theirs
        assert set(do.dit_param_shapes(cfg)) == set(theirs)
    dcfg, ecfg = json.loads(str(g["decoder_cfg"])), json.loads(str(g["encoder_cfg"]))
    assert _state_keys(OobleckDecoder(**dcfg).state_dict()) == _keys_and_shapes(g["decoder_keys"])
    assert _state_keys(OobleckEncoder(**ecfg).state_dict()) == _keys_and_shapes(g["encoder_keys"])


def test_reference_json_configs_build_with_the_dropin_factory():
    """The reference's shipped autoencoder config (stable_audio_2_0_vae.json) builds through the drop-in
    create_model_from_config with the reference's state-dict keys."""
    from stable_audio_tools import create_model_from_config
    g = load_golden("module_keys.npz")
    mine = create_model_from_config(json.loads(str(g["vae_cfg"])))
    assert set(mine.state_dict()) == set(_keys_and_shapes(g["vae_keys"]))
    assert mine.downsampling_ratio == int(g["vae_downsampling_ratio"]) == 2048


def test_sampler_wiring_vs_reference_sample_k():
    """The reference's own sample_k (driving the restated k-diffusion samplers) and the drop-in sample_k produce the
    same trajectory for the same toy denoiser and injected noise."""
    from stable_audio_tools.inference import sampling as mine
    g = load_golden("sampler_cases.npz")
    w, toy = mg.toy_denoiser()
    assert torch.equal(w, torch.from_numpy(g["w"]))
    noise, seq = torch.from_numpy(g["noise"]), torch.from_numpy(g["sde_noise"])
    for st in ("dpmpp-2m-sde", "dpmpp-3m-sde"):
        it = iter(seq)
        b = mine.sample_k(toy, noise.clone(), steps=8, sampler_type=st, sigma_min=0.3, sigma_max=50, device="cpu",
                          noise_sampler=lambda s, sn: next(it))
        assert rel_l2(b, torch.from_numpy(g[f"{st}_plain"])) < 1e-5


def test_number_conditioner_and_multiconditioner_match_reference():
    """The 'next' row conditioners (SURVEY 8f): same state-dict keys and outputs as the reference's."""
    from stable_audio_tools.models import conditioners as mine
    g = load_golden("number_conditioner.npz")
    b = mine.NumberConditioner(64, min_val=0, max_val=512)
    assert _state_keys(b.state_dict()) == _keys_and_shapes(g["keys"])
    b.load_state_dict(mg.seeded_state_dict(b.state_dict(), 41))
    xb, mb = b([0.0, 12.5, 600.0])
    assert torch.equal(xb, torch.from_numpy(g["x"])) and torch.equal(mb, torch.from_numpy(g["mask"]))
    assert xb.shape == (3, 1, 64)
    mc = mine.MultiConditioner({"seconds_start": b, "seconds_total": mine.NumberConditioner(64, 0, 512)})
    out = mc([{"seconds_start": 0, "seconds_total": [30]}, {"seconds_start": 1, "seconds_total": 47}])
    assert out["seconds_total"][0].shape == (2, 1, 64)


def test_oracle_sample_k_inpainting_and_mask_vs_live_reference():
    """oracle.sampler_oracle.sample_k / build_mask (used by the GPU init-audio test as the checker) against the
    reference's own sample_k (inference/sampling.py:144-228) and build_mask (generation.py:270-292): same toy
    denoiser, every random draw (SDE noise and the inpainting callback's re-noising) from one seeded stream via a
    patched torch.randn_like."""
    from oracle import sampler_oracle as so
    from oracle.make_golden import seeded_randn_like
    g = load_golden("sampler_cases.npz")
    L = 48
    mask = so.build_mask(L, mg.INPAINT_MASK_ARGS)
    assert torch.equal(mask, torch.from_numpy(g["mask"]))
    w, toy = mg.toy_denoiser()
    noise, init = torch.from_numpy(g["inpaint_noise"]), torch.from_numpy(g["inpaint_init"])
    for st in ("dpmpp-2m-sde", "dpmpp-3m-sde"):
        for name, m in (("inpaint", mask), ("variation", None)):
            with seeded_randn_like(5):
                b = so.sample_k(toy, noise.clone(), init.clone(), m, steps=7, sampler_type=st, sigma_min=0.3, sigma_max=20)
            assert rel_l2(b, torch.from_numpy(g[f"{st}_{name}"])) < 1e-6


@pytest.fixture
def fake_t5(monkeypatch):
    import transformers
    monkeypatch.setattr(transformers.AutoTokenizer, "from_pretrained",
                        classmethod(lambda cls, *a, **k: mg.FakeT5Tokenizer()))
    monkeypatch.setattr(transformers.T5EncoderModel, "from_pretrained",
                        classmethod(lambda cls, *a, **k: mg.FakeT5Encoder()))


@pytest.mark.parametrize("cfg_name", ["stable_audio_open_1_0.json", "stable_audio_2_0.json"])
def test_shipped_txt2audio_configs_build_and_load_reference_state_dict(fake_t5, cfg_name):
    """SURVEY 8(f)2 / 8(b): create_model_from_config on the reference's SHIPPED text-to-audio configs (T5 stubbed: no
    HF files offline; SA-2.0's CLAP prompt branch swapped for the T5 one).  (1) at full size on the meta device: same
    state-dict keys and shapes as the reference's own factory; (2) with depth cut to 2 and real tensors: a state dict
    with the reference's keys loads strictly, and with the same (seeded) conditioner weights the conditioner (stub T5 +
    NumberConditioners through MultiConditioner) and get_conditioning_inputs give the reference's tensors."""
    from stable_audio_tools import create_model_from_config
    g = load_golden("txt2audio_configs.npz")
    cfg = mg.txt2audio_cfg_with_t5(json.loads(str(g[cfg_name[:-len(".json")] + "/cfg"])))
    with torch.device("meta"):
        mine = create_model_from_config(json.loads(json.dumps(cfg)))
    theirs = _keys_and_shapes(g["keys"])
    assert _state_keys(mine.state_dict()) == theirs, sorted(set(theirs) ^ set(mine.state_dict()))[:10]
    attrs = json.loads(str(g["attrs"]))
    assert mine.min_input_length == attrs["min_input_length"] and mine.io_channels == attrs["io_channels"] == 64
    assert mine.cross_attn_cond_ids == attrs["cross_attn_cond_ids"] and mine.global_cond_ids == attrs["global_cond_ids"]
    mine = create_model_from_config(mg.txt2audio_small(cfg)).eval()
    sd = mine.state_dict()
    assert _state_keys(sd) == _keys_and_shapes(g["small_keys"])
    sd.update({"conditioner." + k: v for k, v in mg.seeded_state_dict(mine.conditioner.state_dict(), 42).items()})
    mine.load_state_dict(sd, strict=True)
    with torch.no_grad():
        ct_m = mine.conditioner(mg.TXT2AUDIO_META)
    assert set(ct_m) == {"prompt", "seconds_start", "seconds_total"}
    prompt = np.zeros((2, 128, 768), np.float32)
    prompt[:, :mg.TXT2AUDIO_PROMPT_ROWS] = g["ct/prompt"]
    ct_t = {k: (torch.from_numpy(prompt if k == "prompt" else g["ct/" + k]), torch.from_numpy(g["ct_mask/" + k]))
            for k in ct_m}
    for k in ct_t:
        assert ct_m[k][0].shape == ct_t[k][0].shape and max_abs(ct_m[k][0].float(), ct_t[k][0]) <= 1e-5
        assert torch.equal(ct_m[k][1].to(torch.float32), ct_t[k][1])
    assert ct_m["prompt"][0].shape == (2, 128, 768) and float(ct_m["prompt"][0][0, 6:].abs().max()) == 0.0   # padding = zeros
    ci_m = mine.get_conditioning_inputs(ct_m)
    assert ci_m["cross_attn_cond"].shape == (2, 130, 768) and ci_m["global_cond"].shape == (2, 1536)
    assert max_abs(ci_m["cross_attn_cond"][:, :128].float(), ct_t["prompt"][0]) <= 1e-5
    assert max_abs(ci_m["cross_attn_cond"][:, 128:].float(), torch.from_numpy(g["ci/cross_attn_cond_tail"])) <= 1e-5
    for k in ("cross_attn_mask", "global_cond"):
        assert max_abs(ci_m[k].float(), torch.from_numpy(g["ci/" + k])) <= 1e-5
