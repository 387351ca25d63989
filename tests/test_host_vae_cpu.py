"""Host-side logic of the causal-VAE drop-in (`opensora/models/hunyuan_vae/*`: NDHWC plumbing, weight packing incl. the
narrow first / last layers, causal padding, first-frame up-sampling, down-sampling strides, mid-block attention, the
tiled / blended modes) on the CPU through the stand-in of the binding, against the goldens produced by EXECUTING the
reference classes (tests/golden/vae_blocks.npz, vae_tiled.npz)."""
import os

import numpy as np
import pytest
import torch

from tests.util import rel_l2

HERE = os.path.dirname(os.path.abspath(__file__))


def _golden(name):
    return {k: torch.from_numpy(v) for k, v in np.load(os.path.join(HERE, "golden", name)).items()}


def _model(G, **kw):
    from opensora.registry import MODELS, build_module

    m = build_module(dict(type="hunyuan_vae", block_out_channels=(16, 32, 32, 32), layers_per_block=1, norm_num_groups=4,
                          latent_channels=4, **kw), MODELS, device_map="cpu")
    m.encoder.load_state_dict({k[4:]: v for k, v in G.items() if k.startswith("enc.")})
    m.decoder.load_state_dict({k[4:]: v for k, v in G.items() if k.startswith("dec.")})
    return m


def test_encoder_decoder_against_reference_goldens(fake_osb):
    from oracle import vae_oracle as V

    G = _golden("vae_blocks.npz")
    m = _model(G).to(torch.bfloat16)
    down, up = V.stage_plan(4, 4, 8)
    Wb = {k: v.to(torch.bfloat16) for k, v in G.items()}
    ze_bf = V.encoder({k[4:]: v for k, v in Wb.items() if k.startswith("enc.")}, Wb["enc_x"], groups=4, strides=down)
    yd_bf = V.decoder({k[4:]: v for k, v in Wb.items() if k.startswith("dec.")}, Wb["enc_y"][:, :4], groups=4, factors=up)
    fe, fd = rel_l2(ze_bf, G["enc_y"]), rel_l2(yd_bf, G["dec_y"])
    with torch.no_grad():
        z = m._to_ncdhw(m.encoder(m._to_ndhwc(G["enc_x"].to(torch.bfloat16), cpad=8)))
        y = m._to_ncdhw(m.decoder(m._to_ndhwc(G["enc_y"][:, :4].to(torch.bfloat16))))
    assert z.shape == G["enc_y"].shape and rel_l2(z, G["enc_y"]) < max(1.5 * fe, 1e-2)
    assert y.shape == G["dec_y"].shape and rel_l2(y, G["dec_y"]) < max(1.5 * fd, 1e-2)
    convs = [c for c in fake_osb.calls if c[0] == "conv3d"]
    assert any(c[1][3] for c in convs), "the 3-channel input layer uses the narrow (kw x channels folded) packing"
    assert {c[1][2] for c in convs} >= {(1, 1, 1), (1, 2, 2), (2, 2, 2)}, "down-samplers run as strided convolutions"


@pytest.mark.parametrize("tag,sp,tp", [("none", False, False), ("spatial", True, False), ("temporal", False, True), ("both", True, True)])
def test_tiled_modes_against_reference_goldens(fake_osb, tag, sp, tp):
    from oracle import vae_oracle as V

    G, GT = _golden("vae_blocks.npz"), _golden("vae_tiled.npz")
    m = _model(G, sample_size=32, sample_tsize=8, use_spatial_tiling=sp, use_temporal_tiling=tp)
    with torch.no_grad():
        m.quant_conv.weight.copy_(GT["quant_w"]); m.quant_conv.bias.copy_(GT["quant_b"])
        m.post_quant_conv.weight.copy_(GT["post_w"]); m.post_quant_conv.bias.copy_(GT["post_b"])
    m = m.to(torch.bfloat16)
    with torch.no_grad():
        z = m.encode(GT["x"], sample_posterior=False)
        y = m.decode(GT[f"z_{tag}"])
    down, up = V.stage_plan(4, 4, 8)
    bf = lambda d, pfx: {k[len(pfx):]: v.to(torch.bfloat16) for k, v in d.items() if k.startswith(pfx)}  # noqa: E731
    We, Wd = bf(G, "enc."), bf(G, "dec.")
    qw, qb, pw, pb = (GT[k].to(torch.bfloat16) for k in ("quant_w", "quant_b", "post_w", "post_b"))
    encode, decode = V.tiled_autoencoder(lambda x: V.causal_conv3d(V.encoder(We, x, groups=4, strides=down), qw, qb),
                                         lambda t: V.decoder(Wd, V.causal_conv3d(t, pw, pb), groups=4, factors=up),
                                         sample_size=32, sample_tsize=8, spatial=sp, temporal=tp)
    zf = rel_l2(0.476986 * encode(GT["x"].to(torch.bfloat16))[:, :4], GT[f"z_{tag}"])
    yf = rel_l2(decode((GT[f"z_{tag}"] / 0.476986).to(torch.bfloat16)), GT[f"y_{tag}"])
    assert z.shape == GT[f"z_{tag}"].shape and y.shape == GT[f"y_{tag}"].shape
    assert rel_l2(z, GT[f"z_{tag}"]) < max(1.5 * zf, 1e-2) and rel_l2(y, GT[f"y_{tag}"]) < max(1.5 * yf, 1e-2)


def test_causal_conv_is_causal_and_latent_size_api(fake_osb):
    from opensora.models.hunyuan_vae.unet_causal_3d_blocks import CausalConv3d
    from opensora.registry import MODELS, build_module

    torch.manual_seed(0)
    c = CausalConv3d(64, 64, 3).to(torch.bfloat16)
    x = torch.randn(1, 5, 6, 7, 64).to(torch.bfloat16)
    y0 = c(x)
    x2 = x.clone()
    x2[:, -1] += 1.0
    y1 = c(x2)
    assert torch.equal(y0[:, :-1], y1[:, :-1]) and not torch.equal(y0[:, -1], y1[:, -1])
    m = build_module(dict(type="hunyuan_vae", block_out_channels=(16, 32, 32, 32), layers_per_block=1, norm_num_groups=4,
                          latent_channels=4), MODELS, device_map="cpu").to(torch.bfloat16)
    v = torch.rand(1, 3, 9, 32, 32) * 2 - 1
    with torch.no_grad():
        z = m.encode(v, sample_posterior=False)
        rec, _, z2 = m(v, sample_posterior=False)
    assert list(z.shape) == [1, 4] + m.get_latent_size([9, 32, 32]) and rec.shape == v.shape and torch.equal(z, z2)


def test_posterior_distribution_matches_the_reference_class():
    """`DiagonalGaussianDistribution` (sample with a seeded generator, kl with and without a second distribution, nll, mode,
    the deterministic switch, token-shaped parameters) against what the reference's own class computed on the same
    parameters (tests/golden/ref_classes.npz, tests/golden/make_golden_ref_classes.py)."""
    from opensora.models.hunyuan_vae.vae import DiagonalGaussianDistribution as Ours

    G = np.load(os.path.join(HERE, "golden", "ref_classes.npz"))
    for i, shape in enumerate(((2, 8, 3, 4, 5), (2, 8, 6, 7), (2, 9, 8))):
        R = {k[len(f"post{i}."):]: torch.from_numpy(G[k]) for k in G.files if k.startswith(f"post{i}.")}
        par, par2 = R["par"], R["par2"]
        assert par.shape == shape
        a, a2 = Ours(par), Ours(par2)
        assert torch.equal(a.mode(), R["mode"]) and torch.equal(a.std, R["std"]) and torch.equal(a.logvar, R["logvar"])
        sa = a.sample(torch.Generator().manual_seed(11))
        assert torch.equal(sa, R["sample"]) and sa.shape == a.mean.shape
        torch.testing.assert_close(a.kl(), R["kl"], rtol=1e-6, atol=1e-6)
        torch.testing.assert_close(a.kl(a2), R["kl2"], rtol=1e-6, atol=1e-6)
        if par.ndim >= 4:
            dims = list(range(1, par.ndim))
            torch.testing.assert_close(a.nll(sa, dims), R["nll"], rtol=1e-6, atol=1e-5)
        d = Ours(par, deterministic=True)
        assert torch.equal(d.sample(), d.mean) and float(d.kl()) == 0.0 and float(d.nll(sa)) == 0.0
    with pytest.raises(NotImplementedError):
        Ours(torch.zeros(4, 4))


def _tp_worker(rank, world, port, ret):
    import sys

    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from tests import fake_osb200

        sys.modules["osb200"] = fake_osb200
        fake_osb200.ACC_DTYPE = torch.float64   # whole vs sharded convolutions: no summation-order noise (see the stand-in)
        import opensora.models.hunyuan_vae.unet_causal_3d_blocks as U
        from opensora.acceleration.communications import gather_forward_split_backward_var_len

        torch.manual_seed(11)   # the same model on every rank (quant / post_quant convolutions are not in the golden file)
        G = _golden("vae_blocks.npz")
        m = _model(G, sample_size=32, sample_tsize=8).to(torch.bfloat16)
        real_stats, real_combine = fake_osb200.group_stats, U._combine_group_stats

        def whole_video_stats(x, groups, eps=1e-6):
            """Statistics of the gathered frames through the SAME routine the un-sharded decode uses: isolates the halo /
            padding / up-sampling logic (bit-level comparison) from the rounding of the combined statistics."""
            g = U._TemporalShard.group
            if g is None:
                return real_stats(x, groups, eps)
            lens = [torch.zeros(1, dtype=torch.long) for _ in range(world)]
            dist.all_gather(lens, torch.tensor([x.shape[1]]), group=g)
            return real_stats(gather_forward_split_backward_var_len(x, 1, g, [int(v) for v in lens]), groups, eps)

        torch.manual_seed(3)
        out = {}
        # 7 latent frames: 4 + 3 (world 2) / 3 + 2 + 2 (world 3) -> every rank >= the 2-frame halo; 3 frames: too few to
        # shard, decoded replicated
        for name, z in (("z7", torch.randn(1, 4, 7, 8, 8)), ("z3", torch.randn(1, 4, 3, 8, 8))):
            with torch.no_grad():
                m.enable_temporal_parallel(None)
                fake_osb200.reset()
                whole = m.decode(z)
                whole_frames = sum(c[1][0][1] for c in fake_osb200.calls if c[0] == "vae_prep")
                m.enable_temporal_parallel(dist.group.WORLD)
                fake_osb200.reset()
                sharded = m.decode(z)
                shard_frames = sum(c[1][0][1] for c in fake_osb200.calls if c[0] == "vae_prep")
                fake_osb200.group_stats, U._combine_group_stats = whole_video_stats, (lambda s, *a: s)
                try:
                    exact = m.decode(z)
                finally:
                    fake_osb200.group_stats, U._combine_group_stats = real_stats, real_combine
                tiled_sharded = tiled = whole
                if world == 2 and name == "z7":
                    m.enable_spatial_tiling(True)      # 8x8 latent > the 4x4 tile: every spatial tile is frame-sharded too
                    tiled_sharded = m.decode(z)
                    m.enable_temporal_parallel(None)
                    tiled = m.decode(z)
                    m.enable_spatial_tiling(False)
            out[name] = dict(shapes=(tuple(whole.shape), tuple(sharded.shape), tuple(exact.shape)), rel=rel_l2(sharded, whole),
                             rel_exact_stats=rel_l2(exact, whole), bit_identical=bool(torch.equal(exact, whole)),
                             rel_tiled=rel_l2(tiled_sharded, tiled), frames=(whole_frames, shard_frames))
        # the encoder: 25 pixel frames -> 7 latent frames, sharded 13 + 12 (world 2) / 9 + 8 + 8 (world 3) pixel frames; two
        # temporally strided stages whose halo depth depends on the parity of a rank's first frame.  8 frames (not 4k + 1)
        # and 9 frames (3 latent frames: too short) are encoded replicated.
        for name, v in (("x25", torch.rand(1, 3, 25, 32, 32) * 2 - 1), ("x8", torch.rand(1, 3, 8, 32, 32) * 2 - 1),
                        ("x9", torch.rand(1, 3, 9, 32, 32) * 2 - 1)):
            with torch.no_grad():
                m.enable_temporal_parallel(None)
                fake_osb200.reset()
                whole = m.encode(v, sample_posterior=False)
                whole_frames = sum(c[1][0][1] for c in fake_osb200.calls if c[0] == "vae_prep")
                m.enable_temporal_parallel(dist.group.WORLD)
                fake_osb200.reset()
                sharded = m.encode(v, sample_posterior=False)
                shard_frames = sum(c[1][0][1] for c in fake_osb200.calls if c[0] == "vae_prep")
                fake_osb200.group_stats, U._combine_group_stats = whole_video_stats, (lambda s, *a: s)
                try:
                    exact = m.encode(v, sample_posterior=False)
                finally:
                    fake_osb200.group_stats, U._combine_group_stats = real_stats, real_combine
                m.enable_temporal_parallel(None)
            out[name] = dict(shapes=(tuple(whole.shape), tuple(sharded.shape), tuple(exact.shape)), rel=rel_l2(sharded, whole),
                             rel_exact_stats=rel_l2(exact, whole), bit_identical=bool(torch.equal(exact, whole)), rel_tiled=0.0,
                             frames=(whole_frames, shard_frames))
        ret[rank] = out
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(900)
@pytest.mark.parametrize("world", [2, 3])
def test_frame_sharded_decode_matches_the_whole_decode(world):
    """SURVEY.md 8e "VAE T-shard with halo": the decoder's up path and the encoder's down path sharded by frames over `world`
    gloo ranks (causal halo from the left neighbour - two frames, or one where a x2 upsample / the parity of a strided stage
    makes one enough -, GroupNorm statistics combined over the ranks, first-frame rules on rank 0 only) against the same model
    working on the whole tensor on one rank.
      * with the statistics taken from the gathered frames by the un-sharded routine, every convolution sees the same bf16
        inputs as in the whole run: the outputs must be BIT-IDENTICAL (the halo / padding / stride logic is exact; the
        stand-in accumulates in fp64 here so that the CPU kernels' summation order cannot flip a bf16 rounding);
      * with the real combination (per-rank mean / variance + counts) the statistics differ in the last fp32 bits, which
        flips bf16 roundings through ~25 normalised layers: same size as the model's own bf16 noise, bounded here."""
    import torch.multiprocessing as mp

    port = 29500 + (os.getpid() + 11 * world) % 2000
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_tp_worker, args=(world, port, ret), nprocs=world, join=True)
    for r in range(world):
        print(r, dict(ret[r]))
        for name, o in ret[r].items():
            assert o["shapes"][0] == o["shapes"][1] == o["shapes"][2], (r, name, o)
            assert o["bit_identical"], (r, name, o)
            assert o["rel"] < 1.5e-2 and o["rel_tiled"] < 1.5e-2, (r, name, o)
        for name in ("z7", "x25"):
            whole_frames, shard_frames = ret[r][name]["frames"]
            assert shard_frames < 0.85 * whole_frames, (r, name, whole_frames, shard_frames)   # worked on a share of the frames
        for name in ("z3", "x8", "x9"):                                                        # not shardable: replicated
            assert ret[r][name]["frames"][0] == ret[r][name]["frames"][1], (r, name)


def test_frame_partition_and_stat_combination():
    from opensora.models.hunyuan_vae.unet_causal_3d_blocks import frame_partition

    assert frame_partition(17, 8) == [3, 2, 2, 2, 2, 2, 2, 2] and frame_partition(8, 2) == [4, 4] and sum(frame_partition(33, 4)) == 33
    # the identity _combine_group_stats uses, against a direct computation
    torch.manual_seed(0)
    parts = [torch.randn(n) * s + o for n, s, o in ((50, 1.0, 3.0), (20, 0.2, -1.0), (130, 2.0, 0.5))]
    n = torch.tensor([float(p.numel()) for p in parts]).double()
    m = torch.stack([p.double().mean() for p in parts])
    v = torch.stack([p.double().var(unbiased=False) for p in parts])
    gm = (n * m).sum() / n.sum()
    gv = (n * (v + (m - gm) ** 2)).sum() / n.sum()
    whole = torch.cat(parts).double()
    assert abs(gm - whole.mean()) < 1e-12 and abs(gv - whole.var(unbiased=False)) < 1e-12
