#!/usr/bin/env python
"""Generate golden vectors by running the REAL reference (TEST INFRASTRUCTURE).

Runs only in the build container (needs ``/root/reference``); the fixtures it
writes to ``tests/golden/*.npz`` are committed and travel to the GPU box.

    python oracle/make_golden.py            # regenerate everything

Each fixture stores: the constructor kwargs (json), the state-dict spec
(names + shapes, json) and (seed, gain) for ``oracle.synth.synth_state_dict``,
a checksum of the synthesised weights, the seeded inputs' (shape, seed) and the
reference outputs.  Weights themselves are regenerated, not stored.
"""

import json
import os
import sys
import types
import warnings

import numpy as np

warnings.filterwarnings("ignore")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def import_reference(ref_root="/root/reference"):
    """Import parallel_wavegan read-only with the two environmental shims of
    SURVEY.md 8(c): scipy.signal.kaiser alias, stub modules for absent deps."""
    import scipy.signal
    import scipy.signal.windows

    scipy.signal.kaiser = scipy.signal.windows.kaiser
    for name in ["h5py", "librosa", "librosa.filters", "soundfile", "kaldiio", "tensorboardX", "matplotlib", "matplotlib.pyplot"]:
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["librosa"].filters = sys.modules["librosa.filters"]

    def _mel(sr, n_fft, n_mels=128, fmin=0.0, fmax=None, **kw):
        from oracle.ref_ops import slaney_mel_filterbank

        return slaney_mel_filterbank(sr, n_fft, n_mels, fmin, fmax)

    sys.modules["librosa.filters"].mel = _mel
    if ref_root not in sys.path:
        sys.path.insert(0, ref_root)
    import parallel_wavegan  # noqa: F401

    return parallel_wavegan


import torch  # noqa: E402

from oracle import synth  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def spec_of(module):
    return [(k, list(v.shape)) for k, v in module.state_dict().items()]


def load_synth(module, seed, gain, keep=()):
    spec = [(k, s) for k, s in spec_of(module) if not any(k.endswith(x) for x in keep)]
    sd = synth.synth_state_dict(spec, seed, gain)
    missing = module.load_state_dict(sd, strict=False)
    assert not missing.unexpected_keys, missing
    return spec, sd


def save(name, meta, **arrays):
    os.makedirs(GOLD, exist_ok=True)
    arrays = {k: (v.detach().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)) for k, v in arrays.items()}
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), meta=json.dumps(meta), **arrays)
    sizes = {k: v.shape for k, v in arrays.items()}
    print(f"[golden] {name}: {sizes}")


def gen_hifigan(name, kwargs, B, T, seed, gain):
    from parallel_wavegan.models import HiFiGANGenerator

    torch.manual_seed(0)
    m = HiFiGANGenerator(**kwargs).eval()
    spec, sd = load_synth(m, seed, gain)
    c = synth.randn((B, kwargs.get("in_channels", 80), T), seed + 1)
    with torch.no_grad():
        y = m(c)
        y_inf = m.inference(c[0].t())
    meta = dict(kind="hifigan_generator", kwargs=kwargs, spec=spec, seed=seed, gain=gain, checksum=synth.checksum(sd), c_shape=list(c.shape), c_seed=seed + 1)
    print("   out std %.3f absmax %.3f" % (y.std(), y.abs().max()))
    save(name, meta, y=y, y_inf=y_inf)


def gen_melgan(name, kwargs, B, T, seed, gain, pqmf_subbands=None):
    from parallel_wavegan.layers import PQMF
    from parallel_wavegan.models import MelGANGenerator

    torch.manual_seed(0)
    m = MelGANGenerator(**kwargs).eval()
    spec, sd = load_synth(m, seed, gain)
    c = synth.randn((B, kwargs.get("in_channels", 80), T), seed + 1)
    arrays = {}
    with torch.no_grad():
        y = m(c)
        arrays["y"] = y
        if pqmf_subbands:
            pq = PQMF(pqmf_subbands)
            arrays["y_pqmf"] = pq.synthesis(y)
            m.pqmf = pq
            arrays["y_inf"] = m.inference(c[0].t())
    meta = dict(kind="melgan_generator", kwargs=kwargs, spec=spec, seed=seed, gain=gain, checksum=synth.checksum(sd), c_shape=list(c.shape), c_seed=seed + 1, pqmf_subbands=pqmf_subbands)
    print("   out std %.3f absmax %.3f" % (y.std(), y.abs().max()))
    save(name, meta, **arrays)


def gen_pwg(name, kwargs, B, frames, seed, gain):
    from parallel_wavegan.models import ParallelWaveGANGenerator

    torch.manual_seed(0)
    kw = json.loads(json.dumps(kwargs))  # the ctor mutates upsample_params
    m = ParallelWaveGANGenerator(**kw).eval()
    spec, sd = load_synth(m, seed, gain)
    ctx = kwargs.get("aux_context_window", 2)
    hop = int(np.prod(kwargs.get("upsample_params", {"upsample_scales": [4, 4, 4, 4]})["upsample_scales"]))
    c = synth.randn((B, kwargs.get("aux_channels", 80), frames + 2 * ctx), seed + 1)
    z = synth.randn((B, 1, frames * hop), seed + 2)
    with torch.no_grad():
        y = m(z, c)
        c_up = m.upsample_net(c)
        x0 = m.first_conv(z)
        x1, s1 = m.conv_layers[0](x0, c_up)
        # inference(): replicate-pad the conditioning by ctx (parallel_wavegan.py:229-261)
        y_inf = m.inference(c=c[0, :, ctx : c.shape[-1] - ctx].t(), x=z[0].t())
    meta = dict(kind="pwg_generator", kwargs=kwargs, spec=spec, seed=seed, gain=gain, checksum=synth.checksum(sd), c_shape=list(c.shape), c_seed=seed + 1, z_shape=list(z.shape), z_seed=seed + 2)
    print("   out std %.3f absmax %.3f" % (y.std(), y.abs().max()))
    save(name, meta, y=y, c_up=c_up[:, :, :512], x1=x1[:, :, :256], s1=s1[:, :, :256], y_inf=y_inf)


def gen_style_melgan(name, kwargs, B, T, seed, gain):
    from parallel_wavegan.models import StyleMelGANGenerator

    torch.manual_seed(0)
    m = StyleMelGANGenerator(**kwargs).eval()
    spec, sd = load_synth(m, seed, gain)
    c = synth.randn((B, kwargs.get("aux_channels", 80), T), seed + 1)
    z = synth.randn((B, kwargs.get("in_channels", 128), 1), seed + 2)
    with torch.no_grad():
        y = m(c, z)
        x0 = m.noise_upsample(z)
        x1, c1 = m.blocks[0](x0, c)
    meta = dict(kind="style_melgan_generator", kwargs=kwargs, spec=spec, seed=seed, gain=gain, checksum=synth.checksum(sd),
                c_shape=list(c.shape), c_seed=seed + 1, z_shape=list(z.shape), z_seed=seed + 2)
    print("   out std %.3f absmax %.3f" % (y.std(), y.abs().max()))
    save(name, meta, y=y, x0=x0, x1=x1, c1=c1)


def gen_pqmf():
    from parallel_wavegan.layers import PQMF

    for n in (2, 3, 4, 8):
        pq = PQMF(n)
        x = synth.randn((2, 1, 32 * n * 3), 100 + n)
        with torch.no_grad():
            a = pq.analysis(x)
            s = pq.synthesis(a)
        meta = dict(kind="pqmf", subbands=n, x_shape=list(x.shape), x_seed=100 + n)
        save(f"pqmf_{n}", meta, analysis_filter=pq.analysis_filter, synthesis_filter=pq.synthesis_filter, analysis=a, synthesis=s)


def gen_conv_cases():
    """ATen conv semantics the kernels must reproduce (index arithmetic cases)."""
    import torch.nn.functional as F

    cases = []
    arrays = {}
    i = 0
    for (cin, cout, k, s, d, g, pad, T) in [
        (4, 6, 3, 1, 1, 1, 1, 37),
        (8, 8, 7, 1, 3, 1, 9, 50),
        (8, 16, 41, 4, 1, 4, 20, 257),
        (16, 16, 5, 3, 1, 1, 2, 100),
        (1, 16, 15, 1, 1, 1, 7, 64),
        (12, 1, 3, 1, 2, 1, 2, 45),
    ]:
        x = synth.randn((2, cin, T), 200 + i)
        w = synth.randn((cout, cin // g, k), 300 + i, 0.3)
        b = synth.randn((cout,), 400 + i, 0.1)
        y = F.conv1d(x, w, b, stride=s, padding=pad, dilation=d, groups=g)
        cases.append(dict(op="conv1d", cin=cin, cout=cout, k=k, stride=s, dilation=d, groups=g, padding=pad, T=T, idx=i))
        arrays[f"y{i}"] = y
        i += 1
    for (cin, cout, s, T) in [(8, 4, 8, 11), (6, 6, 5, 9), (4, 8, 3, 13), (8, 4, 2, 17)]:
        x = synth.randn((2, cin, T), 200 + i)
        w = synth.randn((cin, cout, 2 * s), 300 + i, 0.3)
        b = synth.randn((cout,), 400 + i, 0.1)
        y = F.conv_transpose1d(x, w, b, stride=s, padding=s // 2 + s % 2, output_padding=s % 2)
        cases.append(dict(op="conv_transpose1d", cin=cin, cout=cout, k=2 * s, stride=s, T=T, idx=i))
        arrays[f"y{i}"] = y
        i += 1
    save("conv_cases", dict(kind="conv_cases", cases=cases), **arrays)


def summarize(outs):
    """Compact fingerprint of a (nested) list of feature maps: shape, float64 sum / L2, head+tail."""
    arrays, shapes = {}, []
    flat = []
    for i, o in enumerate(outs):
        if isinstance(o, (list, tuple)):
            for j, t in enumerate(o):
                flat.append((f"o{i}_{j}", t))
        else:
            flat.append((f"o{i}", o))
    for name, t in flat:
        t = t.detach()
        v = t.reshape(-1).double()
        arrays[name + "_stat"] = np.array([float(v.sum()), float(v.norm())])
        arrays[name + "_head"] = t.reshape(-1)[:96].clone()
        arrays[name + "_tail"] = t.reshape(-1)[-96:].clone()
        shapes.append((name, list(t.shape)))
    return arrays, shapes


def gen_discriminator(name, cls_name, kwargs, B, T, seed, gain, train_mode=False, np_seed=None, keep=()):
    import parallel_wavegan.models as M

    torch.manual_seed(0)
    m = getattr(M, cls_name)(**json.loads(json.dumps(kwargs)))
    m.train(train_mode)
    spec, sd = load_synth(m, seed, gain, keep=keep)
    x = synth.randn((B, 1, T), seed + 1, 0.5)
    if np_seed is not None:  # StyleMelGANDiscriminator draws its window positions with np.random.randint (style_melgan.py:330)
        np.random.seed(np_seed)
    with torch.no_grad():
        outs = m(x)
    if isinstance(outs, torch.Tensor):
        outs = [outs]
    arrays, shapes = summarize(outs)
    final = [o[-1] if isinstance(o, (list, tuple)) else o for o in outs]
    for i, f in enumerate(final):
        arrays[f"final{i}"] = f
    if train_mode:  # spectral-norm power iteration mutates weight_u / weight_v
        for k, v in m.state_dict().items():
            if k.endswith("weight_u"):
                arrays["u__" + k.replace(".", "__")] = v
    meta = dict(kind="discriminator", cls=cls_name, kwargs=kwargs, spec=spec, seed=seed, gain=gain, checksum=synth.checksum(sd),
                x_shape=list(x.shape), x_seed=seed + 1, x_scale=0.5, shapes=shapes, train_mode=train_mode, np_seed=np_seed)
    save(name, meta, **arrays)


def gen_losses():
    from parallel_wavegan.losses import (DiscriminatorAdversarialLoss, FeatureMatchLoss, GeneratorAdversarialLoss,
                                         MelSpectrogram, MelSpectrogramLoss, MultiResolutionSTFTLoss)
    from parallel_wavegan.losses.stft_loss import stft

    x = synth.randn((3, 8192), 501, 0.3)
    y = synth.randn((3, 8192), 502, 0.3)
    y = 0.7 * y + 0.3 * x
    arrays = {}
    mr = MultiResolutionSTFTLoss()
    sc, mag = mr(x, y)
    arrays["mr_default"] = torch.stack([sc, mag])
    sc, mag = mr(x.view(1, 3, -1), y.view(1, 3, -1))
    arrays["mr_3d"] = torch.stack([sc, mag])
    mr2 = MultiResolutionSTFTLoss([64, 128, 256], [16, 32, 64], [64, 128, 256])  # test/test_parallel_wavegan.py sizes
    sc, mag = mr2(x[:, :2048], y[:, :2048])
    arrays["mr_small"] = torch.stack([sc, mag])
    arrays["stft_mag"] = stft(x[:1, :4096], 1024, 120, 600, torch.hann_window(600))[:, :8]
    for tag, kw in (("v1", dict(fs=22050, fft_size=1024, hop_size=256, win_length=None, window="hann", num_mels=80, fmin=0, fmax=11025, log_base=None)),
                    ("default", dict())):
        ms = MelSpectrogram(**kw)
        arrays[f"mel_{tag}"] = ms(x[:2])
        arrays[f"melmat_{tag}"] = ms.melmat
        arrays[f"mel_loss_{tag}"] = MelSpectrogramLoss(**kw)(x.unsqueeze(1), y.unsqueeze(1)).reshape(1)
    # GAN losses on synthetic discriminator outputs (lists of lists, last = logits)
    g = torch.Generator().manual_seed(77)
    outs_hat = [[torch.randn(2, 4, 50, generator=g), torch.randn(2, 8, 25, generator=g), torch.randn(2, 1, 25, generator=g)] for _ in range(3)]
    outs = [[torch.randn(2, 4, 50, generator=g), torch.randn(2, 8, 25, generator=g), torch.randn(2, 1, 25, generator=g)] for _ in range(3)]
    for lt in ("mse", "hinge"):
        arrays[f"gen_adv_{lt}"] = GeneratorAdversarialLoss(loss_type=lt)(outs_hat).reshape(1)
        r, f = DiscriminatorAdversarialLoss(loss_type=lt)(outs_hat, outs)
        arrays[f"dis_adv_{lt}"] = torch.stack([r, f])
    arrays["feat_match"] = FeatureMatchLoss()(outs_hat, outs).reshape(1)
    arrays["feat_match_noavg"] = FeatureMatchLoss(False, False, True)(outs_hat, outs).reshape(1)
    save("losses", dict(kind="losses"), **arrays)


def gen_checkpoint():
    """The training checkpoint the reference writes (bin/train.py:112-146): a HiFi-GAN generator after one RAdam step
    on seeded gradients, the default multi-scale multi-period discriminator and a fresh Adam for it.  Stored: the
    layouts (state-dict names + shapes, optimizer groups, optimizer state keys), the seeds, checksums of every tensor
    group and the first parameter's optimizer state.  The tensors themselves are rebuilt from the seeds by the test."""
    import parallel_wavegan.models as M
    from parallel_wavegan.optimizers import RAdam

    kwargs = dict(in_channels=80, out_channels=1, channels=64, kernel_size=7, upsample_scales=[8, 8, 2, 2],
                  upsample_kernel_sizes=[16, 16, 4, 4], resblock_kernel_sizes=[3, 7, 11],
                  resblock_dilations=[[1, 3, 5], [1, 3, 5], [1, 3, 5]])
    torch.manual_seed(0)
    g, d = M.HiFiGANGenerator(**kwargs), M.HiFiGANMultiScaleMultiPeriodDiscriminator()
    g_spec, _ = load_synth(g, 11, 1.0)
    d_spec, _ = load_synth(d, 12, 1.0)
    opt_g = RAdam(g.parameters(), lr=1e-3)
    for i, p in enumerate(g.parameters()):
        p.grad = synth.randn(p.shape, 5000 + i, 0.01)
    opt_g.step()
    sd_g, sd_d = opt_g.state_dict(), torch.optim.Adam(d.parameters()).state_dict()
    state = [sd_g["state"][i] for i in range(len(sd_g["state"]))]
    meta = dict(kind="checkpoint", g_kwargs=kwargs, g_spec=g_spec, g_seed=11, d_spec=d_spec, d_seed=12, gain=1.0,
                grad_seed=5000, grad_scale=0.01, g_param_groups=sd_g["param_groups"], d_param_groups=sd_d["param_groups"],
                state_keys=list(state[0].keys()), step=state[0]["step"],
                g_checksum=synth.checksum(g.state_dict()), d_checksum=synth.checksum(d.state_dict()),
                exp_avg_checksum=synth.checksum({i: s["exp_avg"] for i, s in enumerate(state)}),
                exp_avg_sq_checksum=synth.checksum({i: s["exp_avg_sq"] for i, s in enumerate(state)}))
    save("checkpoint_ref", meta, exp_avg_p0=state[0]["exp_avg"], exp_avg_sq_p0=state[0]["exp_avg_sq"])


def main():
    import_reference()
    if "style_disc" in sys.argv[1:]:  # regenerate only the fixture added in round 2
        gen_discriminator("style_melgan_disc", "StyleMelGANDiscriminator", {}, B=2, T=6000, seed=65, gain=1.4, np_seed=21, keep=("_filter",))
        return
    if "checkpoint" in sys.argv[1:]:  # regenerate only the checkpoint-interchange fixture
        gen_checkpoint()
        return
    gen_checkpoint()
    gen_losses()
    gen_discriminator("style_melgan_disc", "StyleMelGANDiscriminator", {}, B=2, T=6000, seed=65, gain=1.4, np_seed=21, keep=("_filter",))
    gen_discriminator("hifigan_msmpd_v1", "HiFiGANMultiScaleMultiPeriodDiscriminator", {}, B=2, T=8192, seed=61, gain=1.4)
    gen_discriminator("hifigan_msmpd_v1_train", "HiFiGANMultiScaleMultiPeriodDiscriminator", {}, B=1, T=4099, seed=62, gain=1.4, train_mode=True)
    gen_discriminator("melgan_msd", "MelGANMultiScaleDiscriminator", dict(downsample_scales=[4, 4, 4], max_downsample_channels=512), B=2, T=16200, seed=63, gain=1.4)
    gen_discriminator("pwg_disc", "ParallelWaveGANDiscriminator", {}, B=2, T=5000, seed=64, gain=1.4)
    gen_conv_cases()
    gen_pqmf()
    # reference unit-test shapes (test/test_hifigan.py:35-53)
    small_hifi = dict(in_channels=80, out_channels=1, channels=32, kernel_size=7, upsample_scales=[8, 8, 2, 2], upsample_kernel_sizes=[16, 16, 4, 4], resblock_kernel_sizes=[3, 7, 11], resblock_dilations=[[1, 3, 5], [1, 3, 5], [1, 3, 5]], use_additional_convs=True, bias=True, nonlinear_activation="LeakyReLU", nonlinear_activation_params={"negative_slope": 0.1}, use_weight_norm=True, use_causal_conv=False)
    gen_hifigan("hifigan_small", small_hifi, B=2, T=16, seed=11, gain=1.15)
    v1 = dict(small_hifi, channels=512)
    gen_hifigan("hifigan_v1", v1, B=1, T=12, seed=12, gain=1.15)
    no_add = dict(small_hifi, use_additional_convs=False, bias=False, resblock_kernel_sizes=[3, 5], resblock_dilations=[[1, 3], [1, 2]], upsample_scales=[5, 3, 2], upsample_kernel_sizes=[10, 6, 4], channels=64)
    gen_hifigan("hifigan_odd", no_add, B=2, T=9, seed=13, gain=1.3)
    # multi-band MelGAN v2 (egs/csmsc/voc1/conf/multi_band_melgan.v2.yaml:35-45)
    mb = dict(in_channels=80, out_channels=4, kernel_size=7, channels=384, upsample_scales=[5, 5, 3], stack_kernel_size=3, stacks=4, use_weight_norm=True, use_causal_conv=False)
    gen_melgan("mb_melgan_v2", mb, B=2, T=12, seed=21, gain=0.8, pqmf_subbands=4)
    mel_small = dict(in_channels=80, out_channels=1, kernel_size=7, channels=32, upsample_scales=[4, 4], stack_kernel_size=3, stacks=2, use_weight_norm=True, use_final_nonlinear_activation=False)
    gen_melgan("melgan_small", mel_small, B=2, T=20, seed=22, gain=1.2)
    # causal variants (test/test_hifigan.py:198-226, test/test_melgan.py causal cases)
    gen_hifigan("hifigan_causal", dict(small_hifi, use_causal_conv=True), B=2, T=16, seed=14, gain=1.15)
    gen_melgan("melgan_causal", dict(mel_small, use_causal_conv=True, use_final_nonlinear_activation=True), B=2, T=20, seed=23, gain=1.2)
    # StyleMelGAN v1 (egs/csmsc/voc1/conf/style_melgan.v1.yaml:31-50; test/test_style_melgan.py:24-42): the noise
    # path fixes the length, T = prod(noise_upsample_scales) = 88 frames for one noise frame
    style = dict(in_channels=128, aux_channels=80, channels=64, out_channels=1, kernel_size=9, dilation=2, bias=True,
                 noise_upsample_scales=[11, 2, 2, 2], noise_upsample_activation="LeakyReLU",
                 noise_upsample_activation_params={"negative_slope": 0.2}, upsample_scales=[2, 2, 2, 2, 2, 2, 2, 2, 1],
                 upsample_mode="nearest", gated_function="softmax", use_weight_norm=True)
    gen_style_melgan("style_melgan_v1", style, B=2, T=88, seed=41, gain=1.0)
    style_small = dict(style, in_channels=16, channels=32, aux_channels=10, noise_upsample_scales=[3, 2], upsample_scales=[2, 3, 1],
                       gated_function="sigmoid", kernel_size=5, dilation=3)
    gen_style_melgan("style_melgan_small", style_small, B=2, T=6, seed=42, gain=1.0)
    # PWG v1 (egs/ljspeech/voc1/conf/parallel_wavegan.v1.yaml:28-46)
    pwg = dict(in_channels=1, out_channels=1, kernel_size=3, layers=30, stacks=3, residual_channels=64, gate_channels=128, skip_channels=64, aux_channels=80, aux_context_window=2, dropout=0.0, use_weight_norm=True, use_causal_conv=False, upsample_conditional_features=True, upsample_net="ConvInUpsampleNetwork", upsample_params={"upsample_scales": [4, 4, 4, 4]})
    gen_pwg("pwg_v1", pwg, B=1, frames=10, seed=31, gain=1.0)
    # test/test_parallel_wavegan.py:31-52 shapes
    pwg_small = dict(pwg, layers=6, stacks=3, residual_channels=8, gate_channels=16, skip_channels=8, aux_channels=10, aux_context_window=0, upsample_params={"upsample_scales": [4, 4]})
    gen_pwg("pwg_small", pwg_small, B=2, frames=16, seed=32, gain=1.0)
    for extra in sys.argv[1:]:
        pass


if __name__ == "__main__":
    main()
