"""Generates tests/golden/*.npz by running the UNMODIFIED reference (/root/reference) on seeded weights/inputs.
TEST INFRASTRUCTURE. Runs only in the build container (the reference tree is not on the GPU box); the produced
fixtures are committed. At generation time the oracle restatement is also checked against the reference, so a
fixture is never written from a disagreeing pair.

    python oracle/make_golden.py            # writes tests/golden/

Stubs needed to import the reference here (SURVEY.md §8c / Appendix D): `webdataset` (not installed; only
create_dataloader uses it), torchvision.models.vgg16 -> weights=None (no network), LPIPS.load_from_pretrained -> no-op
(vgg.pth unreachable, and its fallback NameErrors on the missing `import os`), single-rank gloo group for GradNorm.
"""
import os
import sys
import types

sys.dont_write_bytecode = True
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("VQB_REFERENCE", "/root/reference")
sys.path.insert(0, REF)
sys.path.insert(1, REPO)
sys.modules["webdataset"] = types.ModuleType("webdataset")
os.environ["WANDB_MODE"] = "disabled"

import numpy as np
import torch
import torch.distributed as dist
import torchvision.models as M

_vgg16 = M.vgg16
M.vgg16 = lambda pretrained=False, **kw: _vgg16(weights=None)
import utils as ref_utils  # noqa: E402  (the reference's utils.py)

ref_utils.LPIPS.load_from_pretrained = lambda self, name="vgg_lpips": None
import ae as ref_ae  # noqa: E402
import vae_trainer as ref_vt  # noqa: E402

from oracle import loss_oracle as LO  # noqa: E402
from oracle import lpips_oracle as LP  # noqa: E402
from oracle import seeded  # noqa: E402
from oracle import step_oracle as SO  # noqa: E402
from oracle import vae_oracle as VO  # noqa: E402

torch.set_grad_enabled(True)
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
OUT = os.path.join(REPO, "tests", "golden")
os.makedirs(OUT, exist_ok=True)
os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT="29533", RANK="0", WORLD_SIZE="1")
dist.init_process_group("gloo")


def close(a, b, tol, what):
    a, b = torch.as_tensor(a).detach().double(), torch.as_tensor(b).detach().double()
    diff = (a - b).norm().item()
    # mathematically-zero gradients (a conv bias in front of a 1-channel-per-group GroupNorm) are pure rounding noise
    floor = 1e-6 * (b.numel() ** 0.5)
    assert diff <= tol * b.norm().item() + floor, \
        f"oracle disagrees with reference on {what}: |a-b|={diff:.3e} |b|={b.norm().item():.3e}"
    return diff


def save(name, **arrs):
    np.savez_compressed(os.path.join(OUT, name + ".npz"),
                        **{k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in arrs.items()})
    print("wrote", name, {k: tuple(np.asarray(v.detach() if torch.is_tensor(v) else v).shape) for k, v in arrs.items()})


def vae_case(name, cfg: VO.VAEConfig, N, R, with_attn=False):
    ref = ref_ae.VAE(resolution=cfg.resolution, in_channels=cfg.in_channels, ch=cfg.ch, out_ch=cfg.out_ch,
                     ch_mult=list(cfg.ch_mult), num_res_blocks=cfg.num_res_blocks, z_channels=cfg.z_channels,
                     use_attn=False, decoder_also_perform_hr=cfg.decoder_also_perform_hr, use_wavelet=False)
    if with_attn:  # the reference cannot construct use_attn=True at HEAD (ae.py:233-235); AttnBlock itself works
        c = cfg.ch * cfg.ch_mult[-1]
        ref.encoder.mid.attn_1 = ref_ae.AttnBlock(c)
        ref.decoder.mid.attn_1 = ref_ae.AttnBlock(cfg.ch * cfg.dec_ch_mult[-1])
    sd = seeded.fill_state_dict(ref.state_dict(), name)
    # residual branches must matter in a parity test: conv2 is ~0 at the reference's init (ae.py:120)
    ref.load_state_dict(sd)
    x = seeded.tensor(name + "/x", (N, cfg.in_channels, R, R), 1.0, "uniform")
    dec, z = ref(x)
    loss = dec.pow(2).mean() + z.pow(2).mean()
    loss.backward()
    grads = {k: p.grad.detach().clone() for k, p in ref.named_parameters()}
    # oracle
    osd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    odec, oz = VO.vae_forward(osd, x, cfg)
    oloss = odec.pow(2).mean() + oz.pow(2).mean()
    oloss.backward()
    close(oz, z, 1e-5, name + " z")
    close(odec, dec, 1e-5, name + " dec")
    for k in grads:
        close(osd[k].grad, grads[k], 1e-4, name + " grad " + k)
    keys = sorted(grads)
    gn = np.array([grads[k].norm().item() for k in keys], dtype=np.float64)
    pick = [k for k in keys if k in ("encoder.conv_in.weight", "decoder.conv_out.weight",
                                     "encoder.down.0.downsample.conv.weight", "decoder.up.1.upsample.conv.weight",
                                     "encoder.mid.block_1.norm1.weight", "decoder.mid.attn_1.qkv.weight")]
    save(name, z=z, dec=dec, loss=loss, grad_keys=np.array(keys), grad_norms=gn,
         **{"grad::" + k: grads[k] for k in pick})


def lpips_case():
    name = "lpips_small"
    torch.manual_seed(0)
    ref = ref_utils.LPIPS().eval()
    sd = seeded.fill_state_dict(ref.state_dict(), "lpips")
    ref.load_state_dict(sd)
    a = seeded.tensor(name + "/a", (2, 3, 32, 32), 1.0, "uniform").requires_grad_(True)
    b = seeded.tensor(name + "/b", (2, 3, 32, 32), 1.0, "uniform")
    val = ref(a, b)
    val.mean().backward()
    a2 = a.detach().clone().requires_grad_(True)
    oval = LP.lpips_forward(sd, a2, b)
    oval.mean().backward()
    close(oval, val, 1e-5, "lpips value")
    close(a2.grad, a.grad, 1e-4, "lpips input grad")
    save(name, val=val, grad_a=a.grad)


def patchd_case():
    name = "patchd_small"
    torch.manual_seed(0)
    ref = ref_utils.PatchDiscriminator()
    sd = seeded.fill_state_dict(ref.state_dict(), "patchd")
    ref.load_state_dict(sd)
    x = seeded.tensor(name + "/x", (2, 3, 32, 32), 1.0, "uniform").requires_grad_(True)
    y = ref(x)
    (y * seeded.tensor(name + "/gy", y.shape)).sum().backward()
    grads = {k: p.grad.detach().clone() for k, p in ref.named_parameters()}
    osd = {k: v.clone().requires_grad_(torch.is_floating_point(v) and "scaling" not in k) for k, v in sd.items()}
    x2 = x.detach().clone().requires_grad_(True)
    oy = LP.patchd_forward(osd, x2)
    (oy * seeded.tensor(name + "/gy", y.shape)).sum().backward()
    close(oy, y, 1e-5, "patchd logits")
    close(x2.grad, x.grad, 1e-4, "patchd input grad")
    for k in grads:
        close(osd[k].grad, grads[k], 1e-4, "patchd grad " + k)
    keys = sorted(grads)
    save(name, logits=y, grad_x=x.grad, grad_keys=np.array(keys),
         grad_norms=np.array([grads[k].norm().item() for k in keys]),
         **{"grad::" + k: grads[k] for k in ("binary_classifier1.0.weight", "binary_classifier5.0.weight",
                                              "slice1.0.0.weight")})


def losses_case():
    name = "losses"
    r = seeded.tensor(name + "/real", (4, 16))
    f = seeded.tensor(name + "/fake", (4, 16))
    out = {}
    for dt in ("hinge", "bce"):
        l, ar, af, acc = ref_vt.gan_disc_loss(r, f, dt)
        ol, oar, oaf, oacc = LO.gan_disc_loss(r, f, dt)
        close(ol, l, 1e-6, "gan_disc_loss " + dt)
        assert abs(ar - oar) < 1e-6 and abs(af - oaf) < 1e-6 and abs(acc - oacc) < 1e-9
        out[dt] = np.array([l.item(), ar, af, acc])
    x = seeded.tensor(name + "/x", (2, 3, 32, 32), 1.0, "uniform")
    xr = seeded.tensor(name + "/xr", (2, 3, 32, 32), 1.0, "uniform")
    z = seeded.tensor(name + "/z", (2, 4, 8, 8))
    vl, st = ref_vt.vae_loss_function(x, xr, z)
    ovl, ost = LO.vae_loss_function(x, xr, z)
    close(ovl, vl, 1e-6, "vae_loss_function")
    for k in st:
        assert abs(st[k] - ost[k]) < 1e-5, k
    heat = ref_vt.blurriness_heatmap(x)
    close(LO.blurriness_heatmap(x), heat, 1e-5, "blurriness_heatmap")
    # low-pass branch of the recon loss (do_pool=False) works in the reference; the pooled branch crashes (fact 4)
    vl2, st2 = ref_vt.vae_loss_function(x, xr, z, do_pool=False, do_recon=True)
    ovl2, ost2 = LO.vae_loss_function(x, xr, z, do_pool=False, do_recon=True)
    close(ovl2, vl2, 1e-6, "vae_loss lowpass")
    assert abs(st2["recon_loss"] - ost2["recon_loss"]) < 1e-6
    # GradNorm backward
    g_in = seeded.tensor(name + "/gn_x", (2, 3, 8, 8)).requires_grad_(True)
    gy = seeded.tensor(name + "/gn_gy", (2, 3, 8, 8))
    (ref_vt.gradnorm(g_in, 0.5) * gy).sum().backward()
    g2 = g_in.detach().clone().requires_grad_(True)
    (LO.gradnorm(g2, 0.5) * gy).sum().backward()
    close(g2.grad, g_in.grad, 1e-6, "gradnorm backward")
    # wavelet
    wv = ref_utils.wavelet_transform_multi_channel(x)
    close(LP.wavelet_transform_multi_channel(x), wv, 1e-6, "wavelet")
    save(name, hinge=out["hinge"], bce=out["bce"], vae_loss=vl, kl_loss=st["kl_loss"], abs_z=st["average_of_abs_z"],
         std_abs_z=st["std_of_abs_z"], heat=heat, lowpass_recon=st2["recon_loss"], gradnorm_grad=g_in.grad, wavelet=wv)


def step_case():
    """Restates vae_trainer.py:530-708 around the reference's own modules/functions (train_ddp itself cannot run)."""
    name = "step_small"
    cfg = VO.VAEConfig(resolution=32, ch=32, ch_mult=(1, 2), num_res_blocks=1, z_channels=4)
    torch.manual_seed(0)
    vae = ref_ae.VAE(resolution=32, in_channels=3, ch=32, out_ch=3, ch_mult=[1, 2], num_res_blocks=1, z_channels=4,
                     use_attn=False, decoder_also_perform_hr=False, use_wavelet=False)
    vsd = seeded.fill_state_dict(vae.state_dict(), name + "/vae")
    vae.load_state_dict(vsd)
    lp = ref_utils.LPIPS().eval()
    lsd = seeded.fill_state_dict(lp.state_dict(), "lpips")
    lp.load_state_dict(lsd)
    disc = ref_utils.PatchDiscriminator()
    dsd = seeded.fill_state_dict(disc.state_dict(), "patchd")
    disc.load_state_dict(dsd)
    real = seeded.tensor(name + "/real", (2, 3, 32, 32), 1.0, "uniform")
    res = {}
    for gan in (False, True):
        vae.zero_grad()
        z = vae.encoder(real)
        z = z.clamp(-8.0, 8.0)
        z_s = vae.reg(z)
        recon = vae.decoder(z_s)
        percep = lp(ref_vt.gradnorm(recon), real).mean()
        vl, _ = ref_vt.vae_loss_function(real, ref_vt.gradnorm(recon, weight=0.001), z)
        if gan:
            g = -disc(ref_vt.gradnorm(recon, weight=1.0)).mean()
            loss = percep + g + vl
        else:
            loss = percep + vl
        loss.backward()
        grads = {k: p.grad.detach().clone() for k, p in vae.named_parameters()}
        osd = {k: v.clone().requires_grad_(True) for k, v in vsd.items()}
        o = SO.generator_step(osd, lsd, dsd, real, cfg, do_clamp=True, do_ganloss=gan, disc_type="hinge")
        close(o["loss"], loss, 1e-5, f"step loss gan={gan}")
        for k in grads:
            close(osd[k].grad, grads[k], 2e-4, f"step grad {k} gan={gan}")
        keys = sorted(grads)
        tag = "gan" if gan else "nogan"
        res[tag + "_loss"] = loss.detach()
        res[tag + "_percep"] = percep.detach()
        res[tag + "_grad_norms"] = np.array([grads[k].norm().item() for k in keys])
        res[tag + "_grad_conv_in"] = grads["encoder.conv_in.weight"]
        res["grad_keys"] = np.array(keys)
        res["recon"] = recon.detach()
    # discriminator step (hinge + LeCam)
    disc.zero_grad()
    rp, fp = disc(real), disc(res["recon"])
    dl, ar, af, acc = ref_vt.gan_disc_loss(rp, fp, "hinge")
    lec = (rp - 0.05).pow(2).mean() + (fp - 0.1).pow(2).mean()
    (dl.mean() + 0.1 * lec).backward()
    dgr = {k: p.grad.detach().clone() for k, p in disc.named_parameters()}
    osd = {k: v.clone().requires_grad_(torch.is_floating_point(v) and "scaling" not in k) for k, v in dsd.items()}
    o = SO.discriminator_step(osd, real, res["recon"], "hinge", True, (0.1, 0.05))
    close(o["d_loss"], dl.mean() + 0.1 * lec, 1e-5, "d step loss")
    for k in dgr:
        close(osd[k].grad, dgr[k], 2e-4, "d step grad " + k)
    dkeys = sorted(dgr)
    res["d_loss"] = (dl.mean() + 0.1 * lec).detach()
    res["d_grad_keys"] = np.array(dkeys)
    res["d_grad_norms"] = np.array([dgr[k].norm().item() for k in dkeys])
    save(name, **res)


def ckpt_case(name="ref_ckpt_step_small"):
    """A checkpoint exactly as the reference writes it (vae_trainer.py:436-438,903-906): torch.save of the state_dict of
    the DDP-wrapped reference VAE (keys prefixed `module.`), here for the step_small model so that the loaded drop-in must
    reproduce that fixture's reconstruction."""
    from torch.nn.parallel import DistributedDataParallel as DDP

    vae = ref_ae.VAE(resolution=32, in_channels=3, ch=32, out_ch=3, ch_mult=[1, 2], num_res_blocks=1, z_channels=4,
                     use_attn=False, decoder_also_perform_hr=False, use_wavelet=False)
    vae.load_state_dict(seeded.fill_state_dict(vae.state_dict(), "step_small/vae"))
    ddp = DDP(vae)
    path = os.path.join(OUT, name + ".pt")
    torch.save({k: v.half() if False else v for k, v in ddp.state_dict().items()}, path)
    print("wrote", path, os.path.getsize(path), "bytes,", len(ddp.state_dict()), "tensors")


def init_case(name="ref_init_seed123"):
    """The reference's initial weights after torch.manual_seed(123) (vae_trainer.py:374-378) for a VAE with two res
    blocks per level and the HR decoder level: parameter creation order and init calls decide every value. 2.3M floats
    do not fit a fixture, so each tensor is stored as shape + SHA-256 of its float32 bytes (bit-exact either way)."""
    import hashlib
    import json

    torch.manual_seed(123)
    m = ref_ae.VAE(64, 3, 32, 3, [1, 2], 2, 4, False, True, False)
    table = [{"key": k, "shape": list(v.shape), "dtype": str(v.dtype).replace("torch.", ""),
              "sha256": hashlib.sha256(v.detach().contiguous().numpy().tobytes()).hexdigest()}
             for k, v in m.state_dict().items()]
    path = os.path.join(OUT, name + ".json")
    with open(path, "w") as f:
        f.write("[\n" + ",\n".join(json.dumps(e) for e in table) + "\n]\n")
    print("wrote", path, len(table), "tensors")


def _sub(tag, grads, res, keys, budget=60_000):
    """Full gradient tensors are too large for a fixture at ch=128: store every s-th element of the flattened tensor
    (s = smallest stride keeping <= budget elements; s == 1 keeps it whole) as `<tag>grad::<key>` and s as
    `<tag>stride::<key>`; the exact norm of every tensor is in `<tag>grad_norms`."""
    for k in keys:
        g = grads[k].detach().flatten()
        s = max(1, -(-g.numel() // budget))
        res[f"{tag}grad::{k}"] = g[::s].clone()
        res[f"{tag}stride::{k}"] = np.int64(s)


FLUX_PICK = ("encoder.conv_in.weight", "encoder.down.0.block.0.conv1.weight", "encoder.down.0.downsample.conv.weight",
             "encoder.down.1.block.0.nin_shortcut.weight", "encoder.down.3.block.1.conv2.weight",
             "encoder.mid.block_1.norm1.weight", "encoder.conv_out.weight", "decoder.conv_in.weight",
             "decoder.mid.block_2.conv1.weight", "decoder.up.1.upsample.conv.weight",
             "decoder.up.0.block.0.nin_shortcut.weight", "decoder.up.0.block.2.conv2.weight",
             "decoder.up.0.block.1.norm2.bias", "decoder.norm_out.weight", "decoder.conv_out.weight")


def flux_step_case(name="step_flux", R=256):
    """BASELINE.json configs[1]/[2] at B=1: ch=128, mult 1,2,4,4, z=16, 256x256 — the generator step without and with
    the PatchDiscriminator term, then the discriminator step (hinge + LeCam), driven through the reference's own
    modules exactly like step_case (vae_trainer.py:530-708)."""
    import time

    cfg = VO.VAEConfig(resolution=R, ch=128, ch_mult=(1, 2, 4, 4), num_res_blocks=2, z_channels=16)
    torch.manual_seed(0)
    vae = ref_ae.VAE(resolution=R, in_channels=3, ch=128, out_ch=3, ch_mult=[1, 2, 4, 4], num_res_blocks=2,
                     z_channels=16, use_attn=False, decoder_also_perform_hr=False, use_wavelet=False)
    vsd = seeded.fill_state_dict(vae.state_dict(), name + "/vae")
    vae.load_state_dict(vsd)
    lp = ref_utils.LPIPS().eval()
    lsd = seeded.fill_state_dict(lp.state_dict(), "lpips")
    lp.load_state_dict(lsd)
    disc = ref_utils.PatchDiscriminator()
    dsd = seeded.fill_state_dict(disc.state_dict(), "patchd")
    disc.load_state_dict(dsd)
    real = seeded.tensor(name + "/real", (1, 3, R, R), 1.0, "uniform")
    res = {}
    for gan in (False, True):
        t0 = time.time()
        vae.zero_grad()
        z = vae.encoder(real)
        z = z.clamp(-8.0, 8.0)
        z_s = vae.reg(z)
        recon = vae.decoder(z_s)
        percep = lp(ref_vt.gradnorm(recon), real).mean()
        vl, _ = ref_vt.vae_loss_function(real, ref_vt.gradnorm(recon, weight=0.001), z)
        if gan:
            g = -disc(ref_vt.gradnorm(recon, weight=1.0)).mean()
            loss = percep + g + vl
        else:
            loss = percep + vl
        loss.backward()
        print(f"  reference step gan={gan}: {time.time() - t0:.1f} s, loss {loss.item():.6f}", flush=True)
        grads = {k: p.grad.detach().clone() for k, p in vae.named_parameters()}
        osd = {k: v.clone().requires_grad_(True) for k, v in vsd.items()}
        o = SO.generator_step(osd, lsd, dsd, real, cfg, do_clamp=True, do_ganloss=gan, disc_type="hinge")
        close(o["loss"], loss, 1e-5, f"flux step loss gan={gan}")
        for k in grads:
            close(osd[k].grad, grads[k], 5e-4, f"flux step grad {k} gan={gan}")
        keys = sorted(grads)
        tag = "gan_" if gan else "nogan_"
        res[tag + "loss"] = loss.detach()
        res[tag + "percep"] = percep.detach()
        res[tag + "grad_norms"] = np.array([grads[k].norm().item() for k in keys])
        _sub(tag, grads, res, FLUX_PICK)
        res["grad_keys"] = np.array(keys)
        res["recon"] = recon.detach()
        res["z"] = z.detach()
    disc.zero_grad()
    rp, fp = disc(real), disc(res["recon"])
    dl, ar, af, acc = ref_vt.gan_disc_loss(rp, fp, "hinge")
    lec = (rp - 0.05).pow(2).mean() + (fp - 0.1).pow(2).mean()
    (dl.mean() + 0.1 * lec).backward()
    dgr = {k: p.grad.detach().clone() for k, p in disc.named_parameters()}
    osd = {k: v.clone().requires_grad_(torch.is_floating_point(v) and "scaling" not in k) for k, v in dsd.items()}
    o = SO.discriminator_step(osd, real, res["recon"], "hinge", True, (0.1, 0.05))
    close(o["d_loss"], dl.mean() + 0.1 * lec, 1e-5, "flux d step loss")
    for k in dgr:
        close(osd[k].grad, dgr[k], 5e-4, "flux d step grad " + k)
    dkeys = sorted(dgr)
    res["d_loss"] = (dl.mean() + 0.1 * lec).detach()
    res["d_logits_real"] = rp.detach()
    res["d_logits_fake"] = fp.detach()
    res["d_grad_keys"] = np.array(dkeys)
    res["d_grad_norms"] = np.array([dgr[k].norm().item() for k in dkeys])
    _sub("d_", dgr, res, ("slice1.0.0.weight", "slice3.0.10.weight", "binary_classifier1.0.weight",
                          "binary_classifier3.0.weight", "binary_classifier5.0.weight"))
    res["recon"] = res["recon"].half()  # 3x256x256 image: fp16 storage keeps 3+ digits more than the test tolerance
    save(name, **res)


def flux_hr_case(name="vae_flux_hr", R=256):
    """BASELINE.json configs[4] topology at B=1: ch=128 encoder at 256^2, decoder with the extra x2 "HR" level
    (ae.py:381) -> 512^2 output."""
    import time

    cfg = VO.VAEConfig(resolution=R, ch=128, ch_mult=(1, 2, 4, 4), num_res_blocks=2, z_channels=16,
                       decoder_also_perform_hr=True)
    ref = ref_ae.VAE(resolution=R, in_channels=3, ch=128, out_ch=3, ch_mult=[1, 2, 4, 4], num_res_blocks=2,
                     z_channels=16, use_attn=False, decoder_also_perform_hr=True, use_wavelet=False)
    sd = seeded.fill_state_dict(ref.state_dict(), name)
    ref.load_state_dict(sd)
    x = seeded.tensor(name + "/x", (1, 3, R, R), 1.0, "uniform")
    t0 = time.time()
    dec, z = ref(x)
    loss = dec.pow(2).mean() + z.pow(2).mean()
    loss.backward()
    print(f"  reference HR fwd+bwd: {time.time() - t0:.1f} s, out {tuple(dec.shape)}", flush=True)
    grads = {k: p.grad.detach().clone() for k, p in ref.named_parameters()}
    osd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    odec, oz = VO.vae_forward(osd, x, cfg)
    (odec.pow(2).mean() + oz.pow(2).mean()).backward()
    close(oz, z, 1e-5, name + " z")
    close(odec, dec, 1e-5, name + " dec")
    for k in grads:
        close(osd[k].grad, grads[k], 5e-4, name + " grad " + k)
    keys = sorted(grads)
    res = {"z": z.detach(), "dec": dec.detach().half(), "loss": loss.detach(), "grad_keys": np.array(keys),
           "grad_norms": np.array([grads[k].norm().item() for k in keys], dtype=np.float64)}
    _sub("", grads, res, ("encoder.conv_in.weight", "decoder.conv_out.weight", "decoder.up.4.block.0.conv1.weight",
                          "decoder.up.4.upsample.conv.weight", "decoder.up.0.block.2.conv2.weight",
                          "decoder.up.3.block.1.norm1.weight"))
    save(name, **res)


if __name__ == "__main__":
    only = sys.argv[1:]
    if only:  # e.g. `python oracle/make_golden.py flux_step flux_hr` (the ch=128 cases take minutes of CPU time)
        for c in only:
            {"flux_step": flux_step_case, "flux_hr": flux_hr_case, "ckpt": ckpt_case, "init": init_case}[c]()
        dist.destroy_process_group()
        sys.exit(0)
    vae_case("vae_small", VO.VAEConfig(resolution=32, ch=32, ch_mult=(1, 2), num_res_blocks=2, z_channels=4), 2, 32)
    vae_case("vae_attn", VO.VAEConfig(resolution=32, ch=32, ch_mult=(1, 2), num_res_blocks=1, z_channels=4,
                                      use_attn=True), 2, 32, with_attn=True)
    vae_case("vae_hr", VO.VAEConfig(resolution=32, ch=32, ch_mult=(1, 2), num_res_blocks=1, z_channels=4,
                                    decoder_also_perform_hr=True), 1, 32)
    lpips_case()
    patchd_case()
    losses_case()
    step_case()
    flux_step_case()
    flux_hr_case()
    ckpt_case()
    init_case()
    dist.destroy_process_group()
    print("all golden fixtures written to", OUT)
