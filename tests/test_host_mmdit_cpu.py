"""Host-side logic of the MMDiT drop-in (`opensora/models/mmdit/{layers,model}.py`: processors, both QKV layouts, both RoPE
layouts, modulation plumbing, the conditioning residual) on the CPU, through the stand-in of the binding, against the
oracle that tests/test_oracle_cpu.py pins to the executed reference source."""
import os

import pytest
import torch

from tests.test_mmdit_gpu import CFG, _ids
from tests.util import rel_l2

HERE = os.path.dirname(os.path.abspath(__file__))


def _rand_model(fused, liger=False):
    from opensora.registry import MODELS, build_module

    torch.manual_seed(7)
    m = build_module(dict(type="flux", fused_qkv=fused, use_liger_rope=liger, **CFG), MODELS, device_map="cpu",
                     torch_dtype=torch.float32)
    g = torch.Generator().manual_seed(11)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if n.endswith("scale"):
                p.copy_(1 + 0.2 * torch.randn(p.shape, generator=g))
            elif p.dim() == 1 or "cond_in" in n:
                p.copy_(0.05 * torch.randn(p.shape, generator=g))
    return m.to(torch.bfloat16)


@pytest.mark.parametrize("fused,liger", [(True, False), (False, False), (False, True)])
def test_mmdit_model_host_logic(fake_osb, fused, liger):
    from oracle import mmdit_oracle as M

    m = _rand_model(fused, liger)
    B, Lt, (T, H, W) = 2, 24, (2, 4, 6)
    g = torch.Generator().manual_seed(3)
    rb = lambda *s: torch.randn(*s, generator=g).to(torch.bfloat16)  # noqa: E731
    txt_ids, img_ids = _ids(B, Lt, T, H, W)
    inp = dict(img=rb(B, T * H * W, 64), img_ids=img_ids, txt=rb(B, Lt, 128), txt_ids=txt_ids,
               timesteps=torch.tensor([0.3, 0.8]), y_vec=rb(B, 96), cond=rb(B, T * H * W, 68), guidance=torch.tensor([4.0, 7.5]))
    with torch.no_grad():
        out = m(**inp)
    cfg = dict(CFG, fused_qkv=fused, use_liger_rope=liger)
    W32 = {k: v.float() for k, v in m.state_dict().items()}
    finp = {k: (v.float() if v.is_floating_point() else v) for k, v in inp.items()}
    ref = M.model_forward(W32, cfg, finp["img"], finp["img_ids"], finp["txt"], finp["txt_ids"], finp["timesteps"],
                          finp["y_vec"], cond=finp["cond"], guidance=finp["guidance"])
    Wb = dict(m.state_dict())
    noise = M.model_forward(Wb, cfg, inp["img"], inp["img_ids"], inp["txt"], inp["txt_ids"], inp["timesteps"].to(torch.bfloat16),
                            inp["y_vec"], cond=inp["cond"], guidance=inp["guidance"].to(torch.bfloat16))
    r, rn = rel_l2(out, ref), rel_l2(noise, ref)
    assert out.shape == ref.shape
    assert r < 2e-2 and r < max(1.5 * rn, 5e-3), (r, rn)
    # one attention call per block over the joint txt|img sequence, with the second norm-weight pair for the img part
    attn = [c for c in fake_osb.calls if c[0] == "attn_short"]
    assert len(attn) == CFG["depth"] + CFG["depth_single_blocks"]
    assert all(c[1][1] == Lt + T * H * W for c in attn)


def test_processor_hook_is_the_plugin_point(fake_osb):
    from opensora.models.mmdit.layers import DoubleStreamBlockProcessor

    m = _rand_model(True)
    seen = []

    class Spy(DoubleStreamBlockProcessor):
        def __call__(self, attn, img, txt, vec, pe):
            seen.append(tuple(img.shape))
            return super().__call__(attn, img, txt, vec, pe)

    for b in m.double_blocks:
        assert isinstance(b.get_processor(), DoubleStreamBlockProcessor)
        b.set_processor(Spy())
    txt_ids, img_ids = _ids(1, 8, 1, 4, 4)
    bf = torch.bfloat16
    with torch.no_grad():
        out = m(img=torch.randn(1, 16, 64).to(bf), img_ids=img_ids, txt=torch.randn(1, 8, 128).to(bf), txt_ids=txt_ids,
                timesteps=torch.tensor([0.5]), y_vec=torch.randn(1, 96).to(bf), cond=torch.randn(1, 16, 68).to(bf),
                guidance=torch.tensor([4.0]))
    assert len(seen) == CFG["depth"] and out.shape == (1, 16, 64) and torch.isfinite(out.float()).all()


def _strip_to_reference_attributes(block, ref_attrs):
    """Deletes every public attribute, submodule and parameter the reference's class of the same module does not have
    (`ref_attrs`: '<module path>:<name>' of the reference's objects), so the block offers exactly the reference's attributes."""
    allowed = {}
    for a in ref_attrs:
        path, name = str(a).split(":")
        allowed.setdefault(path, set()).add(name)
    for path, m in list(block.named_modules()):
        assert path in allowed, f"module {path!r} has no counterpart in the reference's block"
        have = {k for k in vars(m) if not k.startswith("_")} | set(m._modules) | set(m._parameters) | set(m._buffers)
        for name in have - allowed[path]:
            delattr(m, name)
    assert set(allowed) == {p for p, _ in block.named_modules()}


@pytest.mark.parametrize("fused", [True, False])
def test_processors_run_on_the_reference_own_blocks(fake_osb, fused):
    """INTEGRATION.md 2: the processors are installed with `set_processor` on block objects that have only the reference's
    attributes and parameters (this package's blocks stripped to the attribute lists recorded from the REFERENCE's own
    `opensora/models/mmdit/layers.py` classes) and must reproduce what the reference's blocks compute with their stock
    processors (tests/golden/ref_classes.npz, tests/golden/make_golden_ref_classes.py: the same seeded weights and inputs,
    drawn here in the reference's parameter order)."""
    import numpy as np

    from opensora.models.mmdit.layers import (DoubleStreamBlock, DoubleStreamBlockProcessor, EmbedND, SingleStreamBlock,
                                              SingleStreamBlockProcessor)

    G = np.load(os.path.join(HERE, "golden", "ref_classes.npz"))
    tag = "mmdit_" + ("fused" if fused else "split")
    torch.manual_seed(5)
    C, H, B, Lt, Li = 256, 2, 2, 24, 48
    dbl = DoubleStreamBlock(C, H, mlp_ratio=4.0, qkv_bias=True, fused_qkv=fused).eval()
    sgl = SingleStreamBlock(C, H, mlp_ratio=4.0, fused_qkv=fused).eval()
    with torch.no_grad():
        for blk, kind in ((dbl, "double"), (sgl, "single")):
            params = dict(blk.named_parameters())
            assert sorted(params) == sorted(str(n) for n in G[f"{tag}.{kind}_params"])
            for n in G[f"{tag}.{kind}_params"]:
                p = params[str(n)]
                p.copy_(torch.randn_like(p) * (0.2 if n.endswith("scale") else 0.05) + (1.0 if n.endswith("scale") else 0.0))
            _strip_to_reference_attributes(blk, G[f"{tag}.{kind}_attrs"])
    ids = torch.zeros(B, Lt + Li, 3)
    ids[:, Lt:, 0] = torch.arange(Li) // 16
    ids[:, Lt:, 1] = (torch.arange(Li) // 4) % 4
    ids[:, Lt:, 2] = torch.arange(Li) % 4
    pe = EmbedND(dim=C // H, theta=10000, axes_dim=[16, 56, 56])(ids)
    bf = torch.bfloat16
    img, txt, vec = torch.randn(B, Li, C).to(bf), torch.randn(B, Lt, C).to(bf), torch.randn(B, C).to(bf)
    head = torch.cat([t.float().flatten()[:8] for t in (img, txt, vec)])
    assert torch.equal(head, torch.from_numpy(G[f"{tag}.inputs_head"])), "seeded draws differ from the golden run's"
    with torch.no_grad():
        dbl_b, sgl_b = dbl.to(bf), sgl.to(bf)
        dbl_b.set_processor(DoubleStreamBlockProcessor())
        sgl_b.set_processor(SingleStreamBlockProcessor())
        out_i, out_t = dbl_b(img, txt, vec, pe)
        out_x = sgl_b(torch.cat((txt, img), 1), vec, pe)
        # cached packed weights follow the parameters (a second call after an in-place update must see the new values)
        if not fused:
            sgl_b.q_proj.weight.mul_(1.0)
            sgl_b(torch.cat((txt, img), 1), vec, pe)
    rn = float(G[f"{tag}.bf16_rel_l2"])   # the reference's own bf16 path against its fp32 output
    shapes = ((B, Li, C), (B, Lt, C), (B, Lt + Li, C))
    for got, key, shape in zip((out_i, out_t, out_x), ("out_img", "out_txt", "out_single"), shapes):
        ref = torch.from_numpy(G[f"{tag}.{key}"])   # the reference's fp32 output at every 7th element
        r = rel_l2(got.float().flatten()[::7], ref)
        assert got.shape == shape and r < max(2.0 * rn, 6e-3), (key, r, rn)
    names = [c[0] for c in fake_osb.calls]
    assert names.count("attn_short") == (2 if fused else 3) and "ln_modulate" in names


def test_per_step_constants_are_hoisted(fake_osb):
    """SURVEY.md 8f-2: ONE grouped GEMM projects `vec` through every block's modulation layer (the reference launches
    2*depth + depth_single tiny ones), and `pe` is computed once for id tensors that do not change between steps."""
    m = _rand_model(True)
    C, nd, ns = CFG["hidden_size"], CFG["depth"], CFG["depth_single_blocks"]
    txt_ids, img_ids = _ids(1, 8, 1, 4, 4)
    bf = torch.bfloat16
    inp = dict(img=torch.randn(1, 16, 64).to(bf), img_ids=img_ids, txt=torch.randn(1, 8, 128).to(bf), txt_ids=txt_ids,
               timesteps=torch.tensor([0.5]), y_vec=torch.randn(1, 96).to(bf), cond=torch.randn(1, 16, 68).to(bf),
               guidance=torch.tensor([4.0]))
    calls = []
    orig = m.pe_embedder.forward
    m.pe_embedder.forward = lambda ids: (calls.append(1), orig(ids))[1]
    with torch.no_grad():
        fake_osb.reset()
        a = m(**inp)
        mod_width = (2 * nd * 6 + ns * 3) * C
        grouped = [c for c in fake_osb.calls if c[0] == "gemm" and c[1][1] == mod_width]
        single = [c for c in fake_osb.calls if c[0] == "gemm" and c[1][1] in (6 * C, 3 * C) and c[1][0] == 1]
        assert len(grouped) == 1 and not single, (len(grouped), len(single))
        b = m(**dict(inp, timesteps=torch.tensor([0.4])))      # next step: same id tensors
        assert len(calls) == 1, "pe must be cached across steps"
        m(**dict(inp, img_ids=img_ids.clone()))                # other id tensors: recomputed
        assert len(calls) == 2
    assert a.shape == b.shape == (1, 16, 64)


def _mmdit_sp_worker(rank, world, port, ret):
    import os
    import sys

    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from tests import fake_osb200

        sys.modules["osb200"] = fake_osb200
        fake_osb200.ACC_DTYPE = torch.float64   # row-local GEMMs on a row subset: no M-dependent summation-order noise
        res = []
        for fused, liger, (B, Lt, T, H, W) in ((True, False, (2, 24, 2, 4, 6)), (False, True, (1, 8, 1, 4, 6)), (True, False, (1, 40, 1, 2, 4))):
            m = _rand_model(fused, liger)
            g = torch.Generator().manual_seed(3)
            rb = lambda *s: torch.randn(*s, generator=g).to(torch.bfloat16)  # noqa: E731
            txt_ids, img_ids = _ids(B, Lt, T, H, W)
            inp = dict(img=rb(B, T * H * W, 64), img_ids=img_ids, txt=rb(B, Lt, 128), txt_ids=txt_ids, timesteps=torch.rand(B, generator=g),
                       y_vec=rb(B, 96), cond=rb(B, T * H * W, 68), guidance=torch.full((B,), 4.0))
            with torch.no_grad():
                single = m(**inp)
                m.enable_sequence_parallel(dist.group.WORLD)
                splits = m._sp_splits(Lt, T * H * W)
                sharded = m(**inp)
                m.enable_sequence_parallel(None)
            res.append((bool(torch.equal(single, sharded)), splits is not None, tuple(sharded.shape)))
        ret[rank] = res
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_mmdit_ulysses_sequence_parallel_world2():
    """The MMDiT drop-in with the joint txt|img sequence split over two gloo ranks (Ulysses all-to-all around every
    attention, var-len exit gather) reproduces the single-rank output BIT FOR BIT (the stand-in accumulates in fp64 here) - including the layout where one rank
    holds all the text and the other image tokens only, both QKV and RoPE layouts - and falls back to the unsharded path
    when a rank would get no image tokens (the reference's rule, distributed.py:615-617)."""
    import os

    import torch.multiprocessing as mp

    port = 29500 + (os.getpid() + 11) % 2000
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_mmdit_sp_worker, args=(2, port, ret), nprocs=2, join=True)
    for rank in (0, 1):
        r = ret.get(rank)
        assert r is not None and all(ok for ok, _, _ in r), r
        assert [used for _, used, _ in r] == [True, True, False], r   # case 3: 40 text + 8 image tokens -> rank 0 has no image token
