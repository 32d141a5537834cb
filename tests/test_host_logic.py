"""CPU: host-side logic above the C ABI — convolution geometry (views/taps/tap maps of plans.py) checked by emulating
the kernel's documented semantics in PyTorch, drop-in surface (class names, state_dict keys, init parity with the
reference's stored weight digests), split-K heuristics, CLI flags."""
import os
import random

import pytest
import torch
import torch.nn.functional as F

import plans
from oracle import lpips_oracle as LP
from oracle import vae_oracle as VO


def emulate_conv_gemm(g: plans.ConvGeom, a: torch.Tensor, wp: torch.Tensor, Cout: int):
    """include/vqb200.h semantics of vqb_conv_gemm: out[n,h,w,co] = sum_t sum_c view_t[n,h+dh,w+dw,c] * wp[co][t][c],
    reads outside a view are zero. a: flat fp32 buffer of the A tensor; wp [Cout][T][C]."""
    out = torch.zeros(g.N, g.Ho, g.Wo, Cout)
    flat = a.reshape(-1)
    for t_i, (v, dw, dh) in enumerate(g.taps):
        vw = g.views[v]
        for n in range(g.N):
            for h in range(g.Ho):
                hh = h + dh
                if not (0 <= hh < vw.Hv) or n >= vw.Nv:
                    continue
                for w in range(g.Wo):
                    ww = w + dw
                    if not (0 <= ww < vw.Wv):
                        continue
                    off = vw.offset + n * vw.sn + hh * vw.sh + ww * vw.sw
                    out[n, h, w] += wp[:, t_i, :] @ flat[off:off + g.C]
    return out


def pack(w, tapmap, transpose):
    Cout, Cin = w.shape[:2]
    wt = w.reshape(Cout, Cin, -1)[:, :, tapmap]
    return wt.permute(1, 2, 0).contiguous() if transpose else wt.permute(0, 2, 1).contiguous()


def test_geom_s1_matches_conv2d():
    torch.manual_seed(0)
    x, w = torch.randn(2, 5, 6, 8), torch.randn(4, 8, 3, 3)
    g = plans.geom_s1(2, 5, 6, 8, 3)
    out = emulate_conv_gemm(g, x, pack(w, g.tapmap, False), 4)
    ref = F.conv2d(x.permute(0, 3, 1, 2), w, padding=1).permute(0, 2, 3, 1)
    assert torch.allclose(out, ref, atol=1e-4)


def test_geom_s1_dgrad_matches_conv_transpose():
    torch.manual_seed(1)
    dy, w = torch.randn(1, 5, 4, 8), torch.randn(8, 3, 3, 3)  # w: [Cout=8, Cin=3]
    g = plans.geom_s1_dgrad(1, 5, 4, 8, 3)
    out = emulate_conv_gemm(g, dy, pack(w, g.tapmap, True), 3)
    ref = F.conv_transpose2d(dy.permute(0, 3, 1, 2), w, padding=1).permute(0, 2, 3, 1)
    assert torch.allclose(out, ref, atol=1e-4)


def test_geom_s2_matches_padded_stride2_conv():
    """Downsample (ae.py:150-154): F.pad(x,(0,1,0,1)) then conv3x3 stride 2 — the pad is the view's zero fill."""
    torch.manual_seed(2)
    x, w = torch.randn(2, 6, 8, 8), torch.randn(5, 8, 3, 3)
    g = plans.geom_s2(2, 6, 8, 8)
    out = emulate_conv_gemm(g, x, pack(w, g.tapmap, False), 5)
    ref = F.conv2d(F.pad(x.permute(0, 3, 1, 2), (0, 1, 0, 1)), w, stride=2).permute(0, 2, 3, 1)
    assert out.shape == ref.shape and torch.allclose(out, ref, atol=1e-4)


def test_geom_s2_dgrad_classes_cover_the_transposed_conv():
    torch.manual_seed(3)
    N, H, W, C, Co = 1, 6, 4, 8, 8
    dy, w = torch.randn(N, H // 2, W // 2, Co), torch.randn(Co, C, 3, 3)
    dx = torch.zeros(N, H, W, C)
    for ph, pw, g in plans.geom_s2_dgrad_classes(N, H, W, Co):
        dx[:, ph::2, pw::2, :] = emulate_conv_gemm(g, dy, pack(w, g.tapmap, True), C)
    x = torch.zeros(N, C, H, W, requires_grad=True)
    y = F.conv2d(F.pad(x, (0, 1, 0, 1)), w, stride=2)
    (ref,) = torch.autograd.grad(y, x, dy.permute(0, 3, 1, 2))
    assert torch.allclose(dx, ref.permute(0, 2, 3, 1), atol=1e-4)


@pytest.mark.parametrize("k", [2, 4])
def test_geom_patch_matches_strided_conv(k):
    torch.manual_seed(4)
    x, w = torch.randn(2, 8, 8, 8), torch.randn(3, 8, k, k)
    g = plans.geom_patch(2, 8, 8, 8, k)
    out = emulate_conv_gemm(g, x, pack(w, g.tapmap, False), 3)
    ref = F.conv2d(x.permute(0, 3, 1, 2), w, stride=k).permute(0, 2, 3, 1)
    assert torch.allclose(out, ref, atol=1e-4)


def test_cpad_and_desc_fields():
    assert [plans.cpad(c) for c in (1, 3, 8, 9, 16, 128)] == [8, 8, 8, 16, 16, 128]
    g = plans.geom_s2(2, 8, 8, 16)
    d = plans.conv_desc(g, 32, plans.nhwc_strides(4, 4, 32), flags=3)
    assert (d.C, d.Cout, d.N, d.H, d.W, d.nviews, d.ntaps, d.flags) == (16, 32, 2, 4, 4, 4, 9, 3)
    assert d.views[3].offset == (8 + 1) * 16 and d.views[3].sw == 32 and d.views[3].sh == 2 * 8 * 16
    wd = plans.wgrad_desc(g, 32, 4)
    assert wd.dy_view.Wv == 4 and wd.ksplit == 4 and wd.ntaps == 9


def test_ksplit_heuristic_bounds():
    import ops

    for (N, H, W, C, Co) in [(8, 256, 256, 128, 128), (8, 64, 64, 512, 512), (1, 4, 4, 64, 64), (2, 32, 32, 16, 512)]:
        g = plans.geom_s1(N, H, W, C, 3)
        ks = ops.choose_ksplit(g, Co)
        assert 1 <= ks <= 512


def test_dropin_surface_names_and_keys():
    import ae
    import utils
    import vae_trainer as vt

    for name in ("swish", "StandardizedC2d", "FP32GroupNorm", "AttnBlock", "ResnetBlock", "Downsample", "Upsample",
                 "Encoder", "Decoder", "DiagonalGaussian", "VAE", "AutoEncoder"):
        assert hasattr(ae, name), name
    for name in ("LPIPS", "ScalingLayer", "NetLinLayer", "vgg16", "normalize_tensor", "spatial_average",
                 "PatchDiscriminator", "prepare_filter", "wavelet_transform_multi_channel"):
        assert hasattr(utils, name), name
    for name in ("GradNormFunction", "gradnorm", "avg_scalar_over_nodes", "gan_disc_loss", "create_dataloader",
                 "blurriness_heatmap", "vae_loss_function", "cleanup", "train_ddp"):
        assert hasattr(vt, name), name
    cfg = VO.VAEConfig(resolution=64, ch=32, ch_mult=(1, 2, 4), num_res_blocks=2, z_channels=8, use_attn=True)
    m = ae.VAE(64, 3, 32, 3, [1, 2, 4], 2, 8, True, False, False)
    sd = m.state_dict()
    sh = VO.state_dict_shapes(cfg)
    assert set(sd) == set(sh) and all(tuple(sd[k].shape) == tuple(sh[k]) for k in sh)
    hr = ae.VAE(64, 3, 32, 3, [1, 2], 1, 4, False, True, False)
    assert len(hr.decoder.up) == 3 and hr.decoder.ffactor == 4  # ch_mult + [4] (ae.py:381)
    import warnings

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        assert set(utils.LPIPS().state_dict()) == set(LP.lpips_state_dict_shapes())
        assert set(utils.PatchDiscriminator().state_dict()) == set(LP.patchd_state_dict_shapes())
        assert all(not p.requires_grad for p in utils.LPIPS().parameters())


def test_cli_flags_match_reference():
    import vae_trainer as vt

    names = {p.name: p for p in vt.train_ddp.params}
    expected = {"dataset_url": "synthetic", "test_dataset_url": "synthetic", "num_epochs": 2, "batch_size": 8,
                "do_ganloss": False, "learning_rate_vae": 1e-5, "learning_rate_disc": 2e-4, "vae_resolution": 256,
                "vae_in_channels": 3, "vae_ch": 256, "vae_ch_mult": "1,2,4,4", "vae_num_res_blocks": 2,
                "vae_z_channels": 16, "run_name": "run", "max_steps": 1000, "evaluate_every_n_steps": 250,
                "load_path": None, "do_clamp": False, "clamp_th": 8.0, "max_spatial_dim": 256, "do_attn": False,
                "decoder_also_perform_hr": False, "project_name": "vae_sweep_attn_lr_width", "crop_invariance": False,
                "flip_invariance": False, "do_compile": False, "use_wavelet": False,
                "augment_before_perceptual_loss": False, "downscale_factor": 16, "use_lecam": False,
                "disc_type": "bce"}
    extensions = {"use_vq", "vq_codebook_size", "vq_beta"}  # BASELINE config 4; not in the reference
    assert set(names) - extensions == set(expected) and extensions <= set(names)
    for k, v in expected.items():
        assert names[k].default == v, k
    assert names["do_ganloss"].is_flag and names["do_clamp"].is_flag


def test_seeded_init_matches_reference_bit_for_bit():
    """torch.manual_seed(s); VAE(...) must produce the reference's initial weights (same parameter creation order and
    init calls). tests/golden/ref_init_seed123.json holds shape and SHA-256 of every tensor the unmodified reference
    created (oracle/make_golden.py init)."""
    import hashlib
    import json

    import ae

    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_init_seed123.json")) as f:
        ref = json.load(f)
    torch.manual_seed(123)
    mine = ae.VAE(64, 3, 32, 3, [1, 2], 2, 4, False, True, False).state_dict()
    assert list(mine) == [e["key"] for e in ref]
    for e in ref:
        v = mine[e["key"]]
        assert list(v.shape) == e["shape"] and str(v.dtype) == "torch." + e["dtype"], e["key"]
        assert hashlib.sha256(v.contiguous().numpy().tobytes()).hexdigest() == e["sha256"], e["key"]


def test_geom_upsample_fold_matches_nearest_upsample_conv():
    """Folded 2x2 phase convs == conv3x3(nearest_x2(x)) (SURVEY.md Appendix A) incl. the dgrad geometry."""
    torch.manual_seed(5)
    N, h, w, C, Co = 1, 4, 5, 8, 8
    x, wt = torch.randn(N, h, w, C), torch.randn(Co, C, 3, 3)
    ref = F.conv2d(F.interpolate(x.permute(0, 3, 1, 2), scale_factor=2.0, mode="nearest"), wt, padding=1)
    out = torch.zeros(N, 2 * h, 2 * w, Co)

    def fold(mask_list, transpose):
        wf = torch.stack([sum(wt.reshape(Co, C, 9)[:, :, t] for t in range(9) if (m >> t) & 1) for m in mask_list], 2)
        return wf.permute(1, 2, 0).contiguous() if transpose else wf.permute(0, 2, 1).contiguous()  # [R][slot][K]

    for ph in range(2):
        for pw in range(2):
            g = plans.geom_up_fwd(N, h, w, C, ph, pw)
            out[:, ph::2, pw::2, :] = emulate_conv_gemm(g, x, fold(g.tapmask, False), Co)
    assert torch.allclose(out, ref.permute(0, 2, 3, 1), atol=1e-4)
    dy = torch.randn(N, 2 * h, 2 * w, Co)
    xr = x.permute(0, 3, 1, 2).clone().requires_grad_(True)
    y = F.conv2d(F.interpolate(xr, scale_factor=2.0, mode="nearest"), wt, padding=1)
    (gref,) = torch.autograd.grad(y, xr, dy.permute(0, 3, 1, 2))
    gd = plans.geom_up_dgrad(N, h, w, Co)
    gx = emulate_conv_gemm(gd, dy, fold(gd.tapmask, True), C)
    assert torch.allclose(gx, gref.permute(0, 2, 3, 1), atol=1e-4)


def test_ksplit_fills_one_wave_of_148_ctas():
    """Split-K is sized so that (tiles x splits) fills ONE wave of 148 persistent CTAs (measured faster than >= 2 waves,
    DESIGN.md 3.2) for the weight-gradient shapes of the FLUX config at B=32."""
    import ops

    for (N, H, W, C, Co, tiles) in [(32, 32, 32, 512, 512, 36), (32, 256, 256, 128, 128, 6), (32, 64, 64, 512, 512, 36),
                                    (32, 128, 128, 256, 256, 9), (32, 128, 128, 128, 256, 6)]:
        ks = ops.choose_ksplit(plans.geom_s1(N, H, W, C, 3), Co)
        assert tiles * ks <= 148 and tiles * ks >= 0.9 * 148, (N, H, W, C, Co, ks)


def test_geom_fat3_matches_conv2d():
    """Fat-pixel first-layer conv: 3 taps of one 64-element K run over the zero-framed 8-channel image (+ slack), weights
    [Cout][kh][kw*8 + c] zero beyond column 24, == conv3x3 p1 over the 3 real channels; same for the data-gradient form."""
    torch.manual_seed(11)
    N, H, W, Co = 2, 5, 6, 4
    x = torch.randn(N, 3, H, W)
    wt = torch.randn(Co, 3, 3, 3)
    framed = torch.zeros(N * (H + 2) * (W + 2) * 8 + 64)
    fv = framed[:N * (H + 2) * (W + 2) * 8].view(N, H + 2, W + 2, 8)
    fv[:, 1:H + 1, 1:W + 1, :3] = x.permute(0, 2, 3, 1)
    g = plans.geom_fat3(N, H, W)
    assert g.C == plans.FAT_K == 64 and len(g.taps) == 3
    w9 = torch.zeros(Co, 9, 8)
    w9[:, :, :3] = wt.reshape(Co, 3, 9).permute(0, 2, 1)  # [Cout][tap = kh*3+kw][c]
    w64 = torch.zeros(Co, 3, 64)
    w64[:, :, :24] = w9.view(Co, 3, 24)  # what ops._fat_weights builds from the ordinary [Cout][9][8] packing
    out = emulate_conv_gemm(g, framed, w64, Co)
    ref = F.conv2d(x, wt, padding=1).permute(0, 2, 3, 1)
    assert torch.allclose(out, ref, atol=1e-4)


def test_dx_colsum_side_channel_only_matches_the_very_tensor():
    """ops._take_dx_colsum hands the bias gradient produced by the GroupNorm backward pass to the conv backward only for
    the same, unmodified dx tensor; anything else falls back to vqb_colsum."""
    import ops

    dx, cs = torch.randn(2, 3, 3, 8), torch.randn(8)
    ops._dx_colsum_slot[0] = (dx, dx._version, cs)
    assert ops._take_dx_colsum(torch.randn(2, 3, 3, 8), 8) is None           # another tensor
    assert ops._take_dx_colsum(dx, 16) is None                              # channel count mismatch
    assert ops._take_dx_colsum(dx, 8) is cs and ops._dx_colsum_slot[0] is None  # hit consumes the slot
    ops._dx_colsum_slot[0] = (dx, dx._version, cs)
    dx.add_(1.0)                                                             # accumulated into in place
    assert ops._take_dx_colsum(dx, 8) is None
    ops._dx_colsum_slot[0] = None


def test_reference_written_checkpoint_loads_strict_incl_orig_mod_keys():
    """§8(f2) / vae_trainer.py:505-513,903-906: a checkpoint exactly as the reference writes it (state_dict of the
    DDP-wrapped VAE, `module.` keys; tests/golden/ref_ckpt_step_small.pt was saved from the unmodified reference by
    oracle/make_golden.py) loads strict into the drop-in, also when a torch.compile'd encoder/decoder left `_orig_mod.`
    infixes in the keys; a save from the drop-in has the identical key set and tensors."""
    import io

    import ae
    import vae_trainer as vt
    from helpers import seeded_sd

    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_ckpt_step_small.pt")
    ref_sd = torch.load(path, map_location="cpu")
    cfg = VO.VAEConfig(resolution=32, ch=32, ch_mult=(1, 2), num_res_blocks=1, z_channels=4)
    want = seeded_sd(VO.state_dict_shapes(cfg), "step_small/vae")
    for variant in ("plain", "orig_mod"):
        vae = vt.FlatAllReduceDDP(ae.VAE(32, 3, 32, 3, [1, 2], 1, 4, False, False, False))
        sd = ref_sd
        if variant == "orig_mod":
            sd = {k.replace("module.encoder.", "module.encoder._orig_mod.").replace("module.decoder.",
                  "module.decoder._orig_mod."): v for k, v in ref_sd.items()}
        status = vt.load_vae_checkpoint(vae, sd)
        assert not status.missing_keys and not status.unexpected_keys
        for k, v in vae.module.state_dict().items():
            assert torch.equal(v, want[k]), k
        buf = io.BytesIO()
        torch.save(vae.state_dict(), buf)  # what train_ddp writes (:903-906)
        buf.seek(0)
        back = torch.load(buf, map_location="cpu")
        assert list(back.keys()) == list(ref_sd.keys())
        assert all(torch.equal(back[k], ref_sd[k]) for k in back)


def test_image_grid_layout():
    import vae_trainer as vt

    imgs = torch.arange(8, dtype=torch.float32).view(8, 1, 1, 1).expand(8, 3, 4, 4).contiguous()
    g = vt.make_image_grid(imgs, 4)
    assert g.shape == (3, 16, 16)
    for i in range(2):
        for j in range(4):
            assert torch.all(g[:, i * 4:(i + 1) * 4, j * 4:(j + 1) * 4] == i * 4 + j)
    assert torch.all(g[:, 8:] == 0)  # the reference allocates 4D x 4D and fills the top half (:872-893)


def test_lpips_without_offline_opt_in_refuses_random_weights(tmp_path, monkeypatch):
    """ADVICE r1 (medium): missing vgg.pth must be an error unless VQB_OFFLINE=1 was set explicitly."""
    import utils

    lp = utils.LPIPS()  # constructed offline (conftest sets VQB_OFFLINE=1)
    monkeypatch.chdir(tmp_path)
    monkeypatch.setenv("VQB_OFFLINE", "0")
    with pytest.raises(RuntimeError, match="vgg.pth"):
        lp.load_from_pretrained()
    monkeypatch.setenv("VQB_OFFLINE", "1")
    lp.load_from_pretrained()  # explicit opt-in: keeps the random lin layers


def test_latent_augment_flip_crop_matches_reference_restatement():
    """§8 a11 (vae_trainer.py:567-621): flips with channel negation + matched latent/image crops, including the python
    `random` draw order, against the line-by-line restatement in oracle/loss_oracle.py, over many seeds and both
    decoder scales."""
    import vae_trainer as vt
    from oracle import loss_oracle as LO

    torch.manual_seed(0)
    fired = set()
    for seed in range(40):
        for hr in (False, True):
            for flip, crop in ((True, True), (True, False), (False, True), (False, False)):
                z = torch.randn(2, 16, 32, 32)
                img = torch.randn(2, 3, 1024 if hr else 512, 1024 if hr else 512)
                random.seed(seed)
                a_z, a_img = vt.latent_augment(z, z.clone(), img, flip, crop, 16, hr)
                after_a = random.random()
                random.seed(seed)
                b_z, b_img = LO.latent_augment(z, z.clone(), img, flip, crop, 16, hr)
                after_b = random.random()
                assert a_z.shape == b_z.shape and a_img.shape == b_img.shape
                assert torch.equal(a_z, b_z) and torch.equal(a_img, b_img) and after_a == after_b
                fired.add((a_z.shape != z.shape, not torch.equal(a_z[..., :1, :1], z[..., :1, :1])))
                if a_z.shape != z.shape:  # crop: image crop is the latent crop scaled by the decoder factor
                    f = 32 if hr else 16
                    assert a_img.shape[-2] == a_z.shape[-2] * f and a_img.shape[-1] == a_z.shape[-1] * f
                    assert a_z.shape[-1] >= 12 and a_z.shape[-2] >= 12
    assert (True, True) in fired or (True, False) in fired  # crops did fire
    # negated channel blocks: horizontal flip touches [-4:-2], vertical flip [-2:]
    z = torch.randn(1, 16, 8, 8)
    random.seed(3)  # find a seed state where only the first flip fires
    for s in range(200):
        random.seed(s)
        r1, r2 = random.random(), random.random()
        if r1 < 0.5 <= r2:
            random.seed(s)
            zz, _ = vt.latent_augment(z, z.clone(), torch.zeros(1, 3, 128, 128), True, False)
            assert torch.equal(zz[:, :12], torch.flip(z, [-1])[:, :12])
            assert torch.equal(zz[:, 12:14], -torch.flip(z, [-1])[:, 12:14])
            assert torch.equal(zz[:, 14:], torch.flip(z, [-1])[:, 14:])
            break
    else:
        raise AssertionError("no seed found")


def test_product_blurriness_heatmap_and_recon_branches_vs_reference_golden():
    """§8 a17/a18: the PRODUCT functions (vae_trainer.blurriness_heatmap, vae_loss_function low-pass and pooled
    branches) against the reference golden (losses.npz) / the oracle."""
    import numpy as np

    import vae_trainer as vt
    from helpers import golden, rel_l2
    from oracle import loss_oracle as LO
    from oracle import seeded

    g = golden("losses")
    x = seeded.tensor("losses/x", (2, 3, 32, 32), 1.0, "uniform")
    xr = seeded.tensor("losses/xr", (2, 3, 32, 32), 1.0, "uniform")
    z = seeded.tensor("losses/z", (2, 4, 8, 8))
    assert rel_l2(vt.blurriness_heatmap(x), g["heat"]) < 1e-5
    vl, st = vt.vae_loss_function(x, xr, z)
    assert abs(float(vl) - float(g["vae_loss"])) < 1e-6 and abs(float(st["kl_loss"]) - float(g["kl_loss"])) < 1e-6
    assert abs(float(st["average_of_abs_z"]) - float(g["abs_z"])) < 1e-6
    assert abs(float(st["std_of_abs_z"]) - float(g["std_abs_z"])) < 1e-5
    _, st2 = vt.vae_loss_function(x, xr, z, do_pool=False, do_recon=True)
    assert abs(float(st2["recon_loss"]) - float(g["lowpass_recon"])) < 1e-6
    # pooled branch (crashes in the reference with UnboundLocalError, fact 4): pinned by the oracle's reading of :181-187
    _, st3 = vt.vae_loss_function(x, xr, z, do_pool=True, do_recon=True)
    _, ost3 = LO.vae_loss_function(x, xr, z, do_pool=True, do_recon=True)
    assert abs(float(st3["recon_loss"]) - float(ost3["recon_loss"])) < 1e-6


def test_flat_params_slots_collect_and_zero_grad_on_cpu():
    """flat.FlatParams host logic (pure storage; the kernels are CUDA-only): parameters become views of one buffer with
    1024-element slots, gradient slots are handed out once per accumulation window, `collect()` copies gradients produced
    elsewhere into their slots and reports which parameters are active, `zero_grad()` re-arms the slots."""
    import flat
    import ops

    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(7, 5), torch.nn.Tanh(), torch.nn.Linear(5, 3))
    before = [p.detach().clone() for p in net.parameters()]
    st = flat.FlatParams(net.parameters())
    assert st.total % flat.CHUNK == 0 and st.total == 4 * flat.CHUNK  # 35, 5, 15, 3 elements -> one chunk each
    for p, b, o in zip(st.plist, before, st.offsets):
        assert torch.equal(p.detach(), b) and p.data_ptr() == st.params.data_ptr() + 4 * o and o % flat.CHUNK == 0
    # the slot of a parameter is handed out once; a second request inside the same window gets a temporary
    w = st.plist[0]
    g1 = ops.grad_out(w)
    assert g1.data_ptr() == st.grads.data_ptr() + 4 * st.offsets[0] and g1.shape == w.shape
    g2 = ops.grad_out(w)
    assert g2.data_ptr() != g1.data_ptr() and g2.shape == w.shape
    # autograd produces ordinary gradients -> collect() moves them into the slots and flags activity
    x = torch.randn(4, 7)
    net(x).sum().backward()
    st.plist[3].grad = None  # pretend the last bias got no gradient
    ref = [None if p.grad is None else p.grad.detach().clone() for p in st.plist]
    active = st.collect()
    assert active == (True, True, True, False)
    for i, (p, r) in enumerate(zip(st.plist, ref)):
        if r is None:
            assert p.grad is None
        else:
            assert p.grad.data_ptr() == st.grads.data_ptr() + 4 * st.offsets[i] and torch.equal(p.grad, r)
    assert st.collect() == active  # idempotent, nothing left to copy
    st.zero_grad()
    assert all(p.grad is None for p in st.plist)
    assert ops.grad_out(w).data_ptr() == st.grads.data_ptr() + 4 * st.offsets[0]  # re-armed
    # pad elements of every slot stay zero in the parameter buffer
    for p, o in zip(st.plist, st.offsets):
        assert torch.all(st.params[o + p.numel():o + flat.CHUNK] == 0)


def test_flat_adamw_refuses_cpu_and_keeps_scheduler_semantics():
    """FlatAdamW is a torch.optim.Optimizer (LambdaLR works on its param_groups, per-parameter state views exist); its
    step() must fail loudly without CUDA — there is no CPU optimizer fallback."""
    import flat

    net = torch.nn.Linear(4, 4)
    opt = flat.FlatAdamW([{"params": [net.weight], "lr": 1e-3}, {"params": [net.bias], "lr": 1e-2}], weight_decay=1e-3)
    sch = torch.optim.lr_scheduler.LambdaLR(opt, lambda s: 0.5)
    sch.step()
    assert abs(opt.param_groups[0]["lr"] - 5e-4) < 1e-12 and abs(opt.param_groups[1]["lr"] - 5e-3) < 1e-12
    assert set(opt.state[net.weight]) == {"exp_avg", "exp_avg_sq"} and opt.state[net.weight]["exp_avg"].shape == (4, 4)
    net(torch.randn(2, 4)).sum().backward()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        opt.step()


def test_bench_config_table_matches_baseline_json():
    """bench.py's --config table covers BASELINE.json configs[1..4] with BASELINE.md's FLOP accounting."""
    import importlib.util
    import json

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(root, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    base = json.load(open(os.path.join(root, "BASELINE.json")))
    assert len(base["configs"]) == 5
    assert {c["idx"] for c in b.CONFIGS.values()} == {1, 2, 3, 4}
    assert b.CONFIGS["lpips"]["tflop"] == 2.780 and b.CONFIGS["gan"]["tflop"] == 3.107 and b.CONFIGS["hr512"]["tflop"] == 9.98
    assert b.CONFIGS["hr512"]["res"] == 512 and b.CONFIGS["hr512"]["hr"] and b.CONFIGS["vq"]["vq"]


def test_trainer_only_graphs_steps_without_host_random_branches():
    """The CUDA-graph replay is only allowed when nothing the host decides per step can change the captured work: no
    flip / crop invariance, no perceptual-loss augmentation, and LPIPS in eval mode (train mode draws fresh dropout seeds
    on the host for every call — a replayed graph would freeze the mask)."""
    import vae_trainer as vt

    kw = dict(vae_resolution=32, vae_ch=32, vae_ch_mult="1,2", vae_num_res_blocks=1, vae_z_channels=4, max_steps=10)
    assert vt.Trainer("cpu", cuda_graph=True, lpips_eval=True, **kw)._graph_wanted
    assert not vt.Trainer("cpu", cuda_graph=True, lpips_eval=False, **kw)._graph_wanted
    assert not vt.Trainer("cpu", cuda_graph=True, lpips_eval=True, flip_invariance=True, **kw)._graph_wanted
    assert not vt.Trainer("cpu", cuda_graph=True, lpips_eval=True, crop_invariance=True, **kw)._graph_wanted
    assert not vt.Trainer("cpu", cuda_graph=False, lpips_eval=True, **kw)._graph_wanted
    tr = vt.Trainer("cpu", cuda_graph=True, lpips_eval=False, **kw)
    assert tr.lpips.training and tr.graph_launches_per_step is None
    # the two optimizer groups of vae_trainer.py:455-465 (conv_in at 1e-4, the rest at lr / ch) and D's single group
    g = tr.optimizer_G.param_groups
    assert len(g) == 2 and g[0]["initial_lr"] == 1e-5 / 32 and g[1]["initial_lr"] == 1e-4  # (lr itself is in warm-up)
    assert len(g[1]["params"]) == 4  # encoder/decoder conv_in weight + bias
    assert len(tr.optimizer_D.param_groups) == 1
