"""CPU: host-side logic of the drop-in package (no kernels): sampler arithmetic, sigma schedule,
conditioning routing, chunk / cross-fade orchestration, rank sharding, gloo world_size-2 path."""
import math
import os
import subprocess
import sys

import pytest
import torch

from helpers import load_golden, rel_l2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sigma_schedule_and_vdenoiser_scalings():
    from stable_audio_tools.inference.sampling import VDenoiser, get_sigmas_polyexponential
    s = get_sigmas_polyexponential(100, 0.3, 500.0, 1.0)
    assert s.shape == (101,) and s[-1] == 0
    assert abs(float(s[0]) - 500.0) < 1e-3 and abs(float(s[99]) - 0.3) < 1e-6
    assert bool((s[:-1][1:] < s[:-1][:-1]).all())
    # log-linear for rho = 1
    r = torch.log(s[:100])
    assert float((r[1:] - r[:-1]).std()) < 1e-5
    seen = {}

    def inner(x, t, **kw):
        seen["x"], seen["t"] = x, t
        return torch.zeros_like(x)

    d = VDenoiser(inner)
    x = torch.randn(2, 3, 5)
    sig = torch.tensor([2.0, 0.5])
    out = d(x, sig)
    c_in = 1 / (sig ** 2 + 1).sqrt()
    assert torch.allclose(seen["x"], x * c_in[:, None, None])
    assert torch.allclose(seen["t"], sig.atan() * 2 / math.pi)
    assert torch.allclose(out, x / (sig ** 2 + 1)[:, None, None])


@pytest.mark.parametrize("name", ["dpmpp-2m-sde", "dpmpp-3m-sde"])
def test_dropin_samplers_match_oracle_samplers(name):
    """Host-scalar implementation (no device syncs in the loop) == tensor-arithmetic restatement."""
    from oracle import sampler_oracle as so
    from stable_audio_tools.inference import sampling as mine
    torch.manual_seed(0)
    w = torch.randn(4, 4) * 0.2

    def toy(x, t, **kw):
        return torch.einsum("ij,bjl->bil", w, x) * (1 + t[:, None, None])

    seq = [torch.randn(2, 4, 16) for _ in range(12)]

    def ns():
        it = iter(seq)
        return lambda a, b: next(it)

    sig = mine.get_sigmas_polyexponential(12, 0.3, 80.0)
    x0 = torch.randn(2, 4, 16) * sig[0]
    fn_m = mine.SAMPLERS[name]
    fn_o = so.sample_dpmpp_2m_sde if "2m" in name else so.sample_dpmpp_3m_sde
    a = fn_m(mine.VDenoiser(toy), x0.clone(), sig, noise_sampler=ns())
    b = fn_o(so.VDenoiser(toy), x0.clone(), sig, noise_sampler=ns())
    assert rel_l2(a, b) < 1e-5


def test_sample_k_initialisation_modes():
    from stable_audio_tools.inference.sampling import sample_k
    calls = []

    def toy(x, t, **kw):
        calls.append(kw)
        return torch.zeros_like(x)

    noise = torch.ones(1, 2, 8)
    out = sample_k(toy, noise, steps=3, sampler_type="dpmpp-3m-sde", sigma_min=0.5, sigma_max=10, device="cpu",
                   noise_sampler=lambda a, b: torch.zeros(1, 2, 8), cfg_scale=3.0, cross_attn_cond=None)
    assert len(calls) == 3 and calls[0]["cfg_scale"] == 3.0
    assert torch.isfinite(out).all()
    with pytest.raises(NotImplementedError):
        sample_k(toy, noise, steps=3, sampler_type="no-such-sampler", device="cpu")


def test_get_conditioning_inputs_routing():
    from stable_audio_tools.models.diffusion import ConditionedDiffusionModelWrapper
    w = ConditionedDiffusionModelWrapper(torch.nn.Identity(), None, io_channels=64, sample_rate=44100, min_input_length=2048,
                                         cross_attn_cond_ids=["prompt", "seconds_start", "seconds_total"],
                                         global_cond_ids=["seconds_start", "seconds_total"])
    B = 2
    cond = {"prompt": (torch.randn(B, 128, 768), torch.ones(B, 128)),
            "seconds_start": (torch.randn(B, 1, 768), torch.ones(B, 1)),
            "seconds_total": (torch.randn(B, 1, 768), torch.ones(B, 1))}
    out = w.get_conditioning_inputs(cond)
    assert out["cross_attn_cond"].shape == (B, 130, 768) and out["cross_attn_mask"].shape == (B, 130)
    assert out["global_cond"].shape == (B, 1536)
    assert torch.equal(out["cross_attn_cond"][:, 128], cond["seconds_start"][0][:, 0])
    neg = w.get_conditioning_inputs(cond, negative=True)
    assert set(neg) == {"negative_cross_attn_cond", "negative_cross_attn_mask", "negative_global_cond",
                        "negative_input_concat_cond"}


def test_chunked_encode_decode_reconstruct_match_reference_or_closed_form():
    """With linear, position-wise fake encoder/decoder the Bartlett cross-fade weights sum to one on
    the overlaps, so chunked == unchunked away from the padded tail; the reference AudioAutoencoder driven
    with the same fakes (tests/golden/chunked_fake_autoencoder.npz) gave the same tensors bit for bit."""
    from oracle.make_golden import FakeDecoder, FakeEncoder
    from stable_audio_tools.models.autoencoders import AudioAutoencoder
    ae = AudioAutoencoder(FakeEncoder(), FakeDecoder(), latent_dim=3, downsampling_ratio=4, sample_rate=16000,
                          io_channels=2, bottleneck=None)
    g = load_golden("chunked_fake_autoencoder.npz")
    a, z = torch.from_numpy(g["a"]), torch.from_numpy(g["z"])
    enc_c = ae.encode_audio(a.clone(), chunked=True, chunk_size=8, overlap=2, max_batch_size=3)
    dec_c = ae.decode_audio(z.clone(), chunked=True, chunk_size=8, overlap=2, max_batch_size=2)
    rec_c = ae.reconstruct_audio(a.clone(), chunked=True, chunk_size=8, overlap=2, max_batch_size=4)
    assert enc_c.shape == (2, 3, 37) and dec_c.shape == (2, 2, 41 * 4) and rec_c.shape == a.shape
    assert rel_l2(enc_c, ae.encode_audio(a, chunked=False)) < 1e-5
    assert rel_l2(dec_c, ae.decode_audio(z, chunked=False)) < 1e-5
    assert torch.equal(enc_c, torch.from_numpy(g["enc"]))
    assert torch.equal(dec_c, torch.from_numpy(g["dec"]))
    assert torch.equal(rec_c, torch.from_numpy(g["rec"]))


def test_vae_bottleneck_sampling_follows_the_torch_rng():
    from oracle import oobleck_oracle as oo
    from stable_audio_tools.models.bottleneck import VAEBottleneck
    h = torch.randn(2, 8, 5)
    torch.manual_seed(3)
    z = VAEBottleneck().encode(h)
    torch.manual_seed(3)
    noise = torch.randn(2, 4, 5)
    assert torch.allclose(z, oo.vae_encode(h, noise))


def test_rank_sharding_is_a_partition():
    from stable_audio_tools.utils.torch_common import shard_for_rank
    items = list(range(64))
    for world in (1, 2, 4, 8, 5):
        shards = [shard_for_rank(items, r, world) for r in range(world)]
        assert sorted(sum(shards, [])) == items
        assert shards[0] == items[0::world]


def test_gloo_world_size_2_conditioning_broadcast_and_sharding(tmp_path):
    """The N>1 host path of bench.py / generate: rank 0 owns the conditioning, one broadcast, then
    items[rank::world] - run with 2 gloo processes on CPU."""
    script = tmp_path / "w.py"
    script.write_text(f"""
import os, sys, torch, torch.distributed as td
sys.path.insert(0, {os.path.join(ROOT, 'friendly-stable-audio-tools_b200')!r})
from stable_audio_tools.utils.torch_common import shard_for_rank, get_rank, get_world_size
td.init_process_group('gloo')
r, w = get_rank(), get_world_size()
g = torch.Generator().manual_seed(7)
cond = torch.randn(8, 5, 3, generator=g) if r == 0 else torch.zeros(8, 5, 3)
td.broadcast(cond, 0)
mine = cond[r::w]
want = torch.randn(8, 5, 3, generator=torch.Generator().manual_seed(7))[r::w]
assert torch.equal(mine, want)
assert shard_for_rank(list(range(8))) == list(range(8))[r::w]
t = torch.tensor([float(r + 1)])
td.all_reduce(t, op=td.ReduceOp.MAX)
assert t.item() == w
td.destroy_process_group()
import sys
sys.stdout.write('rank %d ok' % r + chr(10))   # one write per rank: the two ranks share the pipe
sys.stdout.flush()
""")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    import socket
    with socket.socket() as sk:                     # a port that is free right now (no fixed port to collide on)
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)],
                       capture_output=True, text=True, timeout=240, env=env)
    assert p.returncode == 0, p.stdout + p.stderr
    assert "rank 0 ok" in p.stdout and "rank 1 ok" in p.stdout


def test_every_sampler_type_solves_the_gaussian_toy_problem():
    """All sampler_type values of the reference's sample_k (inference/sampling.py:211-228) exist and solve a
    problem with a closed-form answer: data ~ N(0, s^2), optimal denoiser D(x, sigma) = x s^2 / (s^2 + sigma^2);
    the probability-flow ODE gives x(sigma) = x(sigma_max) sqrt((s^2 + sigma^2) / (s^2 + sigma_max^2)), and the
    stochastic samplers must end with standard deviation s."""
    import math
    from stable_audio_tools.inference import sampling as S
    s0, smin, smax = 0.7, 0.03, 80.0

    def model_fn(xin, t, **kw):      # the v-objective network whose VDenoiser wrapping equals D
        sigma = torch.tan(t * math.pi / 2).view(-1, *([1] * (xin.ndim - 1)))
        x = xin * (sigma ** 2 + 1).sqrt()
        den = x * s0 ** 2 / (s0 ** 2 + sigma ** 2)
        return (den - x / (sigma ** 2 + 1)) / (-sigma / (sigma ** 2 + 1).sqrt())

    assert set(S.SAMPLERS) == {"k-heun", "k-lms", "k-dpmpp-2s-ancestral", "k-dpm-2", "k-dpm-fast", "k-dpm-adaptive",
                               "dpmpp-2m-sde", "dpmpp-3m-sde"}
    torch.manual_seed(0)
    noise = torch.randn(4, 8, 2048, dtype=torch.float64)
    tol = {"k-heun": 5e-3, "k-lms": 2e-3, "k-dpm-2": 1e-3, "k-dpm-fast": 5e-4, "k-dpm-adaptive": 5e-2}
    for name in S.SAMPLERS:
        torch.manual_seed(1)
        out = S.sample_k(model_fn, noise, steps=60, sampler_type=name, sigma_min=smin, sigma_max=smax, device="cpu")
        assert out.shape == noise.shape and torch.isfinite(out).all()
        if name in tol:
            end = smin if name in ("k-dpm-fast", "k-dpm-adaptive") else 0.0    # those two stop at sigma_min
            ref = noise * smax * math.sqrt(s0 ** 2 + end ** 2) / math.sqrt(s0 ** 2 + smax ** 2)
            assert float((out - ref).norm() / ref.norm()) < tol[name], name
        else:
            assert abs(float(out.std()) - s0) < 0.02, name


def test_rectified_flow_euler_sampler():
    """sample_rf / sample_discrete_euler: a constant velocity field integrates exactly, a variation starts from
    the (1 - sigma_max, sigma_max) mix, and the model is called once per step with t on the uniform grid."""
    from stable_audio_tools.inference.sampling import sample_rf
    seen = []

    def model_fn(x, t, scale=1.0, **kw):
        seen.append(float(t[0]))
        return torch.full_like(x, 2.0) * scale

    noise = torch.randn(2, 4, 16)
    out = sample_rf(model_fn, noise, steps=8, sigma_max=1, device="cpu", scale=0.5)
    assert torch.allclose(out, noise - 1.0, atol=1e-6)              # x(0) = x(1) - 1 * v with v = 1
    assert len(seen) == 8 and abs(seen[0] - 1.0) < 1e-6 and abs(seen[-1] - 0.125) < 1e-6
    init = torch.ones(2, 4, 16)
    out = sample_rf(model_fn, noise, init_data=init, steps=4, sigma_max=0.25, device="cpu", scale=0.0)
    assert torch.allclose(out, init * 0.75 + noise * 0.25, atol=1e-6)


def test_unsupported_dit_inputs_fail_loudly_on_the_host():
    """Options outside the built path raise before anything touches the GPU (no silent fallback)."""
    from stable_audio_tools.models.dit import DiffusionTransformer
    base = dict(io_channels=64, embed_dim=256, depth=1, num_heads=4, cond_token_dim=128, global_cond_dim=256,
                project_cond_tokens=False)
    with pytest.raises(NotImplementedError):
        DiffusionTransformer(**base, transformer_type="x-transformers")
    with pytest.raises(NotImplementedError):                             # prepend tokens need the "prepend" layout
        DiffusionTransformer(**base, transformer_type="continuous_transformer", prepend_cond_dim=8,
                             global_cond_type="adaLN")
    mc = DiffusionTransformer(**base, transformer_type="continuous_transformer", input_concat_dim=8, prepend_cond_dim=32)
    assert mc.preprocess_conv.weight.shape == (72, 72, 1) and mc.transformer.project_in.weight.shape == (256, 72)
    assert mc.to_prepend_embed[0].weight.shape == (256, 32) and mc.postprocess_conv.weight.shape == (64, 64, 1)
    with pytest.raises(ValueError):                                      # concat input missing
        mc(torch.randn(1, 64, 32), torch.rand(1))
    m = DiffusionTransformer(**base, transformer_type="continuous_transformer", patch_size=2,
                             attn_kwargs={"qk_norm": True})
    assert m.patch_size == 2 and m.qk_norm and m.transformer.layers[0].self_attn.qk_norm
    assert m.transformer.project_in.weight.shape == (256, 128)          # io_channels * patch_size
    x, t = torch.randn(1, 64, 32), torch.rand(1)
    with pytest.raises(Exception) as ei:                                 # CPU tensors: no CPU path exists
        m(x, t, cross_attn_cond=torch.randn(1, 4, 128), global_embed=torch.randn(1, 256))
    assert "CUDA" in str(ei.value) or "cuda" in str(ei.value)


def test_stream_decode_needs_cuda_latents():
    from stable_audio_tools.utils.audio_utils import float_to_int16_audio, stream_decode_int16
    with pytest.raises(RuntimeError):
        next(stream_decode_int16(lambda z: z, torch.zeros(1, 2, 8)))
    pcm = float_to_int16_audio(torch.tensor([[0.5, -2.0, 1.0]]))
    assert pcm.dtype == torch.int16 and pcm.tolist() == [[8191, -32767, 16383]]    # peak 2 > 1 -> normalised
    assert float_to_int16_audio(torch.tensor([[0.5, -0.25]]), maximize=True).tolist() == [[32767, -16383]]


def test_loading_through_a_parent_module_marks_the_native_weights_stale():
    """nn.Module.load_state_dict on a parent recurses through _load_from_state_dict and never calls the child's
    load_state_dict; the native copy must still be refreshed (a post hook on the child sets the flag)."""
    from stable_audio_tools.models.autoencoders import OobleckDecoder
    from stable_audio_tools.models.diffusion import DiTWrapper
    w = DiTWrapper(io_channels=64, embed_dim=256, depth=1, num_heads=4, cond_token_dim=128, global_cond_dim=256,
                   project_cond_tokens=False, transformer_type="continuous_transformer")
    w.model.__dict__["_weights_dirty"] = False             # as after a first forward
    w.load_state_dict(w.state_dict())                       # through the PARENT
    assert w.model.__dict__["_weights_dirty"] is True
    holder = torch.nn.ModuleDict({"dec": OobleckDecoder(out_channels=2, channels=32, c_mults=[1, 2], strides=[2, 4],
                                                        latent_dim=8, use_snake=True, final_tanh=False)})
    holder["dec"].__dict__["_dirty"] = False
    holder.load_state_dict(holder.state_dict())
    assert holder["dec"].__dict__["_dirty"] is True


def test_adaptive_solver_reports_every_iteration_with_the_pre_update_estimate():
    """k-diffusion's dpm_adaptive calls the callback once per iteration (accepted or not) with a running index and
    denoised = x_old - sigma(s_old) * eps(x_old, s_old)."""
    from stable_audio_tools.inference.sampling import VDenoiser, sample_dpm_adaptive
    seen = []

    def model_fn(x, t, **kw):
        return 0.3 * x

    x0 = torch.randn(1, 2, 8)
    den = VDenoiser(model_fn)

    def cb(a):
        seen.append((a["i"], a["x"].clone(), a["denoised"].clone(), float(a["sigma"])))

    sample_dpm_adaptive(den, x0.clone() * 5.0, 0.3, 5.0, callback=cb, rtol=0.01, atol=0.01)
    assert [s[0] for s in seen] == list(range(len(seen))) and len(seen) >= 2
    first = seen[0]
    expect = den(x0 * 5.0, torch.tensor([5.0]))              # the estimate at the initial state / sigma_max
    assert torch.allclose(first[2], expect, atol=1e-5)


_SHARDED_WORKER = r'''
import os, sys, torch, torch.distributed as td
sys.path.insert(0, {pkg!r})
from stable_audio_tools.inference.distributed import generate_sharded


class StubConditioner(torch.nn.Module):          # stands for T5 + number embedders: text length / seconds -> tensors
    calls = 0

    def set_device(self, device):
        pass

    def forward(self, meta):
        StubConditioner.calls += 1
        g = torch.Generator().manual_seed(11)
        table = torch.randn(64, 6, 8, generator=g)
        p = torch.stack([table[len(m["prompt"]) % 64] for m in meta])
        s = torch.tensor([[float(m["seconds_total"])] for m in meta]).view(-1, 1, 1).expand(-1, 1, 8).contiguous() / 50.0
        return {{"prompt": (p, torch.ones(len(meta), 6, dtype=torch.bool)), "seconds_total": (s, torch.ones(len(meta), 1))}}


class StubDenoiser(torch.nn.Module):             # a per-row ELEMENTWISE function of (x, t, cond): CPU matmuls pick
    def __init__(self):                           # shape-dependent summation orders, which is not what is tested here
        super().__init__()
        self.w = torch.nn.Parameter(torch.linspace(-0.3, 0.3, 4).view(1, 4, 1))

    def forward(self, x, t, cross_attn_cond=None, global_cond=None, cfg_scale=1.0, **kw):
        c = (cross_attn_cond[:, 0, 0] + cross_attn_cond[:, 3, 5] + global_cond[:, 2]).view(-1, 1, 1)
        return torch.tanh(x.roll(1, dims=1) * self.w) * (0.5 + t.view(-1, 1, 1)) + 0.1 * c * cfg_scale


class Model(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.model, self.conditioner, self.pretransform = StubDenoiser(), StubConditioner(), None
        self.io_channels, self.sample_rate, self.diffusion_objective, self.min_input_length = 4, 16000, "v", 1

    def get_conditioning_inputs(self, ct, negative=False):
        cross = torch.cat([ct["prompt"][0], ct["seconds_total"][0]], dim=1)
        return {{"cross_attn_cond": cross, "cross_attn_mask": None, "global_cond": ct["seconds_total"][0].squeeze(1)}}


meta = [{{"prompt": "x" * (3 + 5 * i), "seconds_total": 10 + i}} for i in range(7)]      # 7 prompts: ragged shards
kw = dict(steps=5, cfg_scale=3.0, sample_size=24, batch_size=2, seed=77, device="cpu", sigma_min=0.3, sigma_max=20.0)
single = dict(generate_sharded(Model(), meta, rank=0, world_size=1, **kw))               # the 1-rank answer, locally
td.init_process_group("gloo")
r, w = td.get_rank(), td.get_world_size()
StubConditioner.calls = 0
mine = generate_sharded(Model(), meta, **kw)
assert [i for i, _ in mine] == list(range(7))[r::w]
assert StubConditioner.calls == (1 if r == 0 else 0)                # the conditioner ran on rank 0 only
for i, y in mine:
    assert y.shape == (4, 24) and torch.equal(y, single[i]), (r, i)   # per-prompt result independent of the world size
td.destroy_process_group()
sys.stdout.write("rank %d ok" % r + chr(10))
sys.stdout.flush()
'''


def test_generate_sharded_gloo_world_2_equals_single_rank(tmp_path):
    """inference/distributed.generate_sharded (the product form of the reference's generate.py:78-151): rank 0 runs the
    conditioner once, ONE broadcast of its output, items[rank::world] sharding, per-prompt seeding - every prompt's
    result with 2 ranks equals the 1-rank result bit for bit (SURVEY.md 7.1b distributed test)."""
    import socket
    script = tmp_path / "sharded.py"
    script.write_text(_SHARDED_WORKER.format(pkg=os.path.join(ROOT, "friendly-stable-audio-tools_b200")))
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)],
                       capture_output=True, text=True, timeout=300, env=dict(os.environ, MASTER_ADDR="127.0.0.1"))
    assert p.returncode == 0, p.stdout + p.stderr
    assert "rank 0 ok" in p.stdout and "rank 1 ok" in p.stdout
