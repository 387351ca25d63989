"""Generates tests/golden/ref_classes.npz by EXECUTING the reference's own classes (loaded by path through
oracle/ref_loader.py from a checkout of the reference; it is not needed to run the tests):

    python tests/golden/make_golden_ref_classes.py

* `mmdit_<fused|split>.*`: the reference's DoubleStreamBlock / SingleStreamBlock (models/mmdit/layers.py) with seeded
  weights and inputs - the draw order and seeds of tests/test_host_mmdit_cpu.py, which regenerates them - run with their
  stock processors in fp32 (outputs stored at every 7th element) and in bf16 (stored as its rel-L2 error only).  Also the
  parameter names in creation order and every module's public attribute names, so the test can build this package's
  blocks with exactly the reference's parameters and attributes.
* `post<i>.*`: the reference's DiagonalGaussianDistribution (models/hunyuan_vae/vae.py) on three parameter shapes."""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import ref_loader  # noqa: E402
from tests.util import rel_l2  # noqa: E402

SAMPLE_STRIDE = 7  # prime: the sample covers every token and every channel of the [B, L, 256] outputs


def public_attributes(module):
    """'<module path>:<attribute>' for every public attribute, submodule, parameter and buffer of every module."""
    out = []
    for path, m in module.named_modules():
        names = {k for k in vars(m) if not k.startswith("_")} | set(m._modules) | set(m._parameters) | set(m._buffers)
        out += [f"{path}:{n}" for n in sorted(names)]
    return np.array(out)


def mmdit_blocks(out):
    R, _, _ = ref_loader.load_mmdit()
    bf = torch.bfloat16
    for fused in (True, False):
        tag = "mmdit_" + ("fused" if fused else "split")
        torch.manual_seed(5)
        C, H, B, Lt, Li = 256, 2, 2, 24, 48
        dbl = R.DoubleStreamBlock(C, H, mlp_ratio=4.0, qkv_bias=True, fused_qkv=fused).eval()
        sgl = R.SingleStreamBlock(C, H, mlp_ratio=4.0, fused_qkv=fused).eval()
        with torch.no_grad():
            for blk in (dbl, sgl):
                for n, p in blk.named_parameters():
                    p.copy_(torch.randn_like(p) * (0.2 if n.endswith("scale") else 0.05) + (1.0 if n.endswith("scale") else 0.0))
        ids = torch.zeros(B, Lt + Li, 3)
        ids[:, Lt:, 0] = torch.arange(Li) // 16
        ids[:, Lt:, 1] = (torch.arange(Li) // 4) % 4
        ids[:, Lt:, 2] = torch.arange(Li) % 4
        pe = R.EmbedND(dim=C // H, theta=10000, axes_dim=[16, 56, 56])(ids)
        img, txt, vec = torch.randn(B, Li, C).to(bf), torch.randn(B, Lt, C).to(bf), torch.randn(B, C).to(bf)
        with torch.no_grad():
            ref_i, ref_t = dbl(img.float(), txt.float(), vec.float(), pe)
            ref_x = sgl(torch.cat((txt, img), 1).float(), vec.float(), pe)
            noise_i, _ = dbl.to(bf)(img, txt, vec, pe)
        out[f"{tag}.double_params"] = np.array([n for n, _ in dbl.named_parameters()])
        out[f"{tag}.single_params"] = np.array([n for n, _ in sgl.named_parameters()])
        out[f"{tag}.double_attrs"] = public_attributes(dbl)
        out[f"{tag}.single_attrs"] = public_attributes(sgl)
        out[f"{tag}.inputs_head"] = torch.cat([t.float().flatten()[:8] for t in (img, txt, vec)]).numpy()
        for k, v in (("out_img", ref_i), ("out_txt", ref_t), ("out_single", ref_x)):
            out[f"{tag}.{k}"] = v.flatten()[::SAMPLE_STRIDE].numpy()
        out[f"{tag}.bf16_rel_l2"] = np.array(rel_l2(noise_i.float(), ref_i))


def posterior(out):
    _, Rvae = ref_loader.load_hunyuan_vae()
    g = torch.Generator().manual_seed(5)
    for i, shape in enumerate(((2, 8, 3, 4, 5), (2, 8, 6, 7), (2, 9, 8))):
        par = torch.randn(*shape, generator=g) * 3.0
        par2 = torch.randn(*shape, generator=g)
        b, b2 = Rvae.DiagonalGaussianDistribution(par), Rvae.DiagonalGaussianDistribution(par2)
        sb = b.sample(torch.Generator().manual_seed(11))
        res = dict(par=par, par2=par2, mode=b.mode(), std=b.std, logvar=b.logvar, sample=sb, kl=b.kl(), kl2=b.kl(b2))
        if par.ndim >= 4:
            res["nll"] = b.nll(sb, list(range(1, par.ndim)))
        out.update({f"post{i}.{k}": v.numpy() for k, v in res.items()})


def main():
    assert ref_loader.available(), "needs a checkout of the reference (oracle/ref_loader.py)"
    out = {}
    mmdit_blocks(out)
    posterior(out)
    path = os.path.join(HERE, "ref_classes.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
