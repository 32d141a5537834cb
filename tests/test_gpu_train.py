"""GPU (-m gpu): the optimizer side of the step and multi-step / multi-rank behaviour of the Trainer.

  * vqb_adamw_flat vs torch.optim.AdamW (the optimizer of vae_trainer.py:455-475) over several steps, incl. two lr groups,
    a cosine schedule and parameters without a gradient;
  * regression for the stale-operand bug of round 1 (fused optimizers do not bump Tensor._version): after every
    optimizer step the cached bf16 GEMM operands equal a fresh packing of the updated master weights, for torch's own
    fused AdamW too, and the loss moves;
  * N=2 NCCL: gradients of two ranks on half-batches, averaged by FlatAllReduceDDP, equal the single-rank gradients on
    the full batch (skipped on a 1-GPU box).
"""
import os
import sys

import numpy as np
import pytest
import torch

from helpers import cosine, rel_l2

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _mk_params(seed, shapes):
    g = torch.Generator().manual_seed(seed)
    return [torch.nn.Parameter((torch.randn(s, generator=g) * 0.1).cuda()) for s in shapes]


def test_flat_adamw_matches_torch_adamw():
    import flat

    shapes = [(64, 32, 3, 3), (64,), (3, 7), (1025,), (128, 64, 1, 1), (5,)]
    ours, ref = _mk_params(0, shapes), _mk_params(0, shapes)
    groups = lambda ps: [{"params": ps[:4], "lr": 1e-3}, {"params": ps[4:], "lr": 1e-2}]
    o1 = flat.FlatAdamW(groups(ours), weight_decay=1e-3, betas=(0.9, 0.95))
    o2 = torch.optim.AdamW(groups(ref), weight_decay=1e-3, betas=(0.9, 0.95), foreach=False, fused=False)
    sch = lambda o: torch.optim.lr_scheduler.LambdaLR(o, lambda s: 0.5 * (1 + np.cos(np.pi * s / 20)))
    s1, s2 = sch(o1), sch(o2)
    gen = torch.Generator(device="cuda").manual_seed(1)
    for step in range(12):
        o1.zero_grad()
        o2.zero_grad()
        for i, (a, b) in enumerate(zip(ours, ref)):
            if i == 3 and step < 2:
                continue  # a parameter without gradient is skipped by both (its step count then lags in torch: same group
                # step here, so only compare it after it has been active)
            gr = torch.randn(a.shape, device="cuda", generator=gen) * (0.01 if i != 1 else 10.0)
            a.grad = gr.clone()
            b.grad = gr.clone()
        o1.step()
        o2.step()
        s1.step()
        s2.step()
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(zip(ours, ref)):
        if i == 3:
            continue
        e = rel_l2(a, b)
        print(f"adamw param {i} {tuple(a.shape)}: rel {e:.2e}")
        assert e < 2e-6, (i, e)
    # gradients were adopted into the flat buffer and parameters are views of the flat parameter buffer
    st = o1.store
    assert all(p.data_ptr() == st.params.data_ptr() + 4 * o for p, o in zip(st.plist, st.offsets))
    assert all(p.grad.data_ptr() == st.grads.data_ptr() + 4 * o for p, o in zip(st.plist, st.offsets))


def _fresh_pack_matches(module):
    """Every cached bf16 operand of every conv of `module` equals a fresh packing of the current fp32 weight."""
    import ae
    import ops

    n = 0
    for m in module.modules():
        if not isinstance(m, ae.StandardizedC2d):
            continue
        for key, ent in m._packed._store.items():
            Cout, Cin, T, nslots, transpose, Kpad, fold, sg, ld_g, ld_r = ent.spec
            if sg != nslots:
                fresh = ops._new_pack_entry(m.weight, ent.tm.tolist(), bool(transpose), Kpad, bool(fold), fat=True)
            else:
                fresh = ops._new_pack_entry(m.weight, ent.tm.tolist(), bool(transpose), Kpad, bool(fold))
            ops._run_pack([fresh])
            assert torch.equal(fresh.out, ent.out), (key, tuple(ent.out.shape))
            n += 1
    return n


@pytest.mark.parametrize("optimizer", ["flat", "torch_fused"])
def test_packed_weights_follow_optimizer_steps(optimizer):
    """ADVICE r1 (high): fused AdamW updates parameters without bumping `_version`; the packed-operand caches must be
    refreshed anyway (global optimizer post-step hook -> one vqb_pack_weights_multi launch)."""
    import ae
    import vae_trainer as vt

    torch.manual_seed(0)
    vae = ae.VAE(32, 3, 32, 3, [1, 2], 1, 4, False, False, False).cuda()
    with torch.no_grad():
        for blk in [m for m in vae.modules() if isinstance(m, ae.ResnetBlock)]:
            blk.conv2.weight.normal_(0, 0.05)  # the reference's near-zero conv2 init would hide the residual branch
    if optimizer == "flat":
        import flat

        opt = flat.FlatAdamW([{"params": list(vae.parameters()), "lr": 3e-3}], weight_decay=1e-3, betas=(0.9, 0.95))
    else:
        opt = torch.optim.AdamW(vae.parameters(), lr=3e-3, weight_decay=1e-3, betas=(0.9, 0.95), fused=True)
    x = (torch.rand(2, 3, 32, 32, device="cuda") * 2 - 1)
    losses = []
    for it in range(4):
        opt.zero_grad(set_to_none=True)
        dec, z = vae(x)
        loss = (dec - x).pow(2).mean() + 0.1 * z.pow(2).mean()
        loss.backward()
        opt.step()
        losses.append(loss.item())
        n = _fresh_pack_matches(vae)
        assert n > 20
    print(f"\n{optimizer}: losses {losses}")
    assert losses[-1] < losses[0] * 0.98, "the model does not learn: forward keeps using stale packed weights"


def test_trainer_two_steps_learns_and_repacks():
    import vae_trainer as vt

    tr = vt.Trainer("cuda:0", vae_resolution=32, vae_ch=32, vae_ch_mult="1,2", vae_num_res_blocks=1, vae_z_channels=4,
                    do_clamp=True, do_ganloss=True, disc_type="hinge", use_lecam=True, max_steps=100,
                    learning_rate_vae=3e-2, lpips_eval=True)
    x = torch.rand(2, 3, 256, 256) * 2 - 1
    w0 = tr.vae.module.decoder.conv_out.weight.detach().clone()
    d0 = tr.discriminator.module.binary_classifier1[0].weight.detach().clone()
    outs = [tr.step(x) for _ in range(3)]
    torch.cuda.synchronize()
    assert not torch.equal(w0, tr.vae.module.decoder.conv_out.weight.detach())
    assert not torch.equal(d0, tr.discriminator.module.binary_classifier1[0].weight.detach())
    assert _fresh_pack_matches(tr.vae.module) > 20 and _fresh_pack_matches(tr.discriminator.module) > 10
    assert all(torch.isfinite(o["overall_vae_loss"]) for o in outs)


# ----------------------------------------------------------------------------------------------------------------------
def _nccl_worker(rank, world, port, q):
    sys.path.insert(0, os.path.join(ROOT, "vqgan-training_b200"))
    sys.path.insert(1, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank), VQB_OFFLINE="1")
    import torch.distributed as dist

    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(f"cuda:{rank}"))
    import random

    import vae_trainer as vt

    tr = vt.Trainer(f"cuda:{rank}", vae_resolution=64, vae_ch=64, vae_ch_mult="1,2", vae_num_res_blocks=1,
                    vae_z_channels=4, do_clamp=True, do_ganloss=False, max_steps=100, lpips_eval=True)
    g = torch.Generator().manual_seed(5)
    full = torch.rand(4, 3, 256, 256, generator=g) * 2 - 1
    half = full[rank * 2:(rank + 1) * 2].contiguous()
    random.seed(1)  # same flip decision on both ranks
    # run the loss/backward/all-reduce part of the step; the optimizer still collects the gradients into the flat
    # buffer but does not update the weights
    tr.optimizer_G.launch = lambda *a, **k: None
    tr.step(half)
    torch.cuda.synchronize()
    st = tr.optimizer_G.store
    q.put((rank, st.grads.float().cpu().numpy()))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_nccl_gradients_equal_single_rank_full_batch():
    """SURVEY §8(e): DP ranks on half-batches + all-reduce(AVG) == one rank on the concatenated batch (rel 1e-3).
    GradNorm's rank-averaged norm differs from the full-batch norm by construction (mean of two half-batch norms vs
    the norm of the whole), so the comparison uses weight-gradient DIRECTION per tensor group and a common scale."""
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29700 + os.getpid() % 200
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=600) for _ in procs], key=lambda t_: t_[0])
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    g0, g1 = res[0][1], res[1][1]
    assert np.array_equal(g0, g1), "ranks disagree after the all-reduce"

    # single rank, full batch (no process group): same seeds
    import random

    import vae_trainer as vt

    tr = vt.Trainer("cuda:0", vae_resolution=64, vae_ch=64, vae_ch_mult="1,2", vae_num_res_blocks=1, vae_z_channels=4,
                    do_clamp=True, do_ganloss=False, max_steps=100, lpips_eval=True)
    g = torch.Generator().manual_seed(5)
    full = torch.rand(4, 3, 256, 256, generator=g) * 2 - 1
    random.seed(1)
    tr.optimizer_G.launch = lambda *a, **k: None
    tr.step(full)
    torch.cuda.synchronize()
    ref = tr.optimizer_G.store.grads.float().cpu().numpy()
    # decoder gradients flow through GradNorm: rank-mean of half-batch norms vs full-batch norm -> one common factor
    st = tr.optimizer_G.store
    names = [n for n, _ in tr.vae.named_parameters()]
    # same ordering as the optimizer groups: "not conv_in" first, then conv_in
    order = [n for n in names if "conv_in" not in n] + [n for n in names if "conv_in" in n]
    dec = np.zeros(ref.shape, dtype=bool)
    for n, p, o in zip(order, st.plist, st.offsets):
        if n.startswith("module.decoder."):
            dec[o:o + p.numel()] = True
    scale = float(np.dot(g0[dec], ref[dec]) / np.dot(ref[dec], ref[dec]))
    e_dec = np.linalg.norm(g0[dec] - scale * ref[dec]) / np.linalg.norm(scale * ref[dec])
    c_all = float(np.dot(g0, ref) / (np.linalg.norm(g0) * np.linalg.norm(ref)))
    print(f"\nN=2 vs N=1 full batch: decoder-grad rel err {e_dec:.3e} at common GradNorm scale {scale:.4f}; "
          f"cosine over all {ref.size} gradient elements {c_all:.6f}")
    # measured 4.5e-3: the two sides run different per-rank batch sizes (2 vs 4 samples per tile stream), so the fused
    # GroupNorm statistics sum in a different order and bf16 rounding turns that into ~0.5 % noise; exact logic errors
    # (a missed slot, a wrong average) show up as O(1)
    assert e_dec < 1.5e-2 and c_all > 0.999


def test_lpips_train_mode_dropout_matches_reference_arithmetic_with_same_mask():
    """VERDICT r1 missing #4: the reference trains with LPIPS's Dropout(0.5) live (utils.py:79-89, vae_trainer.py:477).
    The fused tail's counter-based mask is materialised (vqb_lpips_dropout_mask) and fed to the reference arithmetic
    (oracle restatement, fp32 CPU) as an explicit keep mask: value and input gradient must agree like in eval mode; the
    mask must be ~Bernoulli(1/2); eval mode must ignore it; two calls draw different masks."""
    import ops
    import utils
    from helpers import seeded_sd
    from oracle import lpips_oracle as LP
    from oracle import seeded

    sd = seeded_sd(LP.lpips_state_dict_shapes(), "lpips")
    m = utils.LPIPS()
    m.load_state_dict(sd, strict=True)
    m = m.cuda().train()
    a = seeded.tensor("lpips_small/a", (2, 3, 64, 64), 1.0, "uniform").cuda().requires_grad_(True)
    b = seeded.tensor("lpips_small/b", (2, 3, 64, 64), 1.0, "uniform").cuda()
    m.dropout_seeds = [11, 22, 33, 44, 55]
    val = m(a, b)
    val.mean().backward()
    chns, hw = [64, 128, 256, 512, 512], [64, 32, 16, 8, 4]
    masks = []
    for s, c, r in zip(m.dropout_seeds, chns, hw):
        mk = ops.lpips_dropout_mask(s, 2, r * r, c, "cuda")
        frac = mk.float().mean().item()
        assert abs(frac - 0.5) < 0.02, frac
        masks.append(mk.view(2, r, r, c).permute(0, 3, 1, 2).float().cpu())
    a2 = a.detach().cpu().clone().requires_grad_(True)
    ref = LP.lpips_forward(sd, a2, b.cpu(), keep_masks=masks)
    ref.mean().backward()
    e = rel_l2(val, ref)
    c = cosine(a.grad, a2.grad)
    r = a.grad.norm().item() / a2.grad.norm().item()
    print(f"\nlpips train-mode dropout: value rel {e:.3e}  grad cos {c:.5f}  norm ratio {r:.4f}")
    assert e < 2e-2 and c > 0.99 and abs(r - 1) < 0.06
    # eval mode ignores the seeds; unseeded train-mode calls draw fresh masks
    m.eval()
    v_eval = m(a.detach(), b)
    assert rel_l2(v_eval, LP.lpips_forward(sd, a.detach().cpu(), b.cpu())) < 2e-2
    m.train()
    m.dropout_seeds = None
    v1, s1 = m(a.detach(), b), m.last_dropout_seeds
    v2, s2 = m(a.detach(), b), m.last_dropout_seeds
    assert s1 != s2 and not torch.equal(v1, v2)


def test_loaded_reference_checkpoint_reproduces_golden_and_flip_equivariant_eval():
    """§8(f2): the reference-written checkpoint, loaded through load_vae_checkpoint, reproduces the reference's
    reconstruction (step_small golden); Trainer.evaluate() (vae_trainer.py:811-893) with flip_invariance decodes the
    (-1,-2)-flipped latent with its last four channels negated and flips the image back — checked against the same
    recipe restated over the fp32 CPU oracle."""
    import vae_trainer as vt
    from helpers import golden, seeded_sd
    from oracle import seeded
    from oracle import vae_oracle as VO

    g = golden("step_small")
    cfg = VO.VAEConfig(resolution=32, ch=32, ch_mult=(1, 2), num_res_blocks=1, z_channels=4)
    path = os.path.join(ROOT, "tests", "golden", "ref_ckpt_step_small.pt")
    for flip in (False, True):
        tr = vt.Trainer("cuda:0", vae_resolution=32, vae_ch=32, vae_ch_mult="1,2", vae_num_res_blocks=1,
                        vae_z_channels=4, do_clamp=True, flip_invariance=flip, max_steps=10, lpips_eval=True)
        vt.load_vae_checkpoint(tr.vae, path)
        real = seeded.tensor("step_small/real", (2, 3, 32, 32), 1.0, "uniform")
        z = tr.vae.module.encoder(real.cuda()).clamp(-8, 8)
        recon = tr.vae.module.decoder(tr.vae.module.reg(z))
        e = rel_l2(recon, g["recon"])
        print(f"\nloaded checkpoint (flip={flip}): recon rel_l2 vs reference golden {e:.3e}")
        assert e < 2e-2
        # evaluation path on 256^2 inputs (the encoder always sees the 256^2 area resize)
        big = seeded.tensor("eval/x", (3, 3, 256, 256), 1.0, "uniform")
        ev = tr.evaluate([(big,)])
        sd = seeded_sd(VO.state_dict_shapes(cfg), "step_small/vae")
        zo = VO.reg(VO.encoder_forward(sd, big, cfg).clamp(-8, 8))
        if flip:
            zo = torch.flip(zo, [-1, -2]).clone()
            zo[:, -4:] = -zo[:, -4:]
        ro = (VO.decoder_forward(sd, zo, cfg) * 0.5 + 0.5).clamp(0, 1)
        if flip:
            ro = torch.flip(ro, [-1, -2])
        e2 = rel_l2(ev["raw_reconstructed"], ro)
        print(f"  evaluate(): reconstruction rel_l2 vs oracle recipe {e2:.3e}; grid {tuple(ev['test_images'].shape)}")
        assert e2 < 2e-2 and ev["test_images"].shape == (3, 1024, 1024)
        assert rel_l2(ev["test_images"][:, :256, :256], (big[0] * 0.5 + 0.5).clamp(0, 1)) < 1e-6


def test_wavelet_front_end_kernel_vs_reference_golden():
    """§8(f3) / utils.py:229-247: the fused wavelet + layout kernel against the reference's output (losses.npz `wavelet`,
    produced by the unmodified reference) — bf16 storage rounding only — and through Encoder(use_wavelet=True)."""
    import ae
    import ops
    import utils
    from helpers import golden
    from oracle import seeded

    g = golden("losses")
    x = seeded.tensor("losses/x", (2, 3, 32, 32), 1.0, "uniform").cuda()
    y = ops.wavelet_to_nhwc(x, utils.filters_expanded)
    assert y.shape == (2, 16, 16, 16) and torch.all(y[..., 12:] == 0)
    got = y[..., :12].permute(0, 3, 1, 2).float()
    e = rel_l2(got, g["wavelet"])
    print(f"\nwavelet kernel vs reference: rel_l2 {e:.3e}")
    assert e < 4e-3  # bf16 rounding of the stored result (2^-9 relative per element)
    ref_bf16 = torch.from_numpy(g["wavelet"]).cuda().to(torch.bfloat16).float()
    assert (got - ref_bf16).abs().max().item() <= 2 * ref_bf16.abs().max().item() * 2 ** -8
    # through the encoder: fused front-end == ATen front-end + layout kernel
    torch.manual_seed(0)
    enc = ae.Encoder(resolution=64, in_channels=3, ch=32, ch_mult=[1, 2], num_res_blocks=1, z_channels=4, use_attn=False,
                     use_wavelet=True).cuda()
    xi = torch.rand(2, 3, 64, 64, device="cuda") * 2 - 1
    z_fused = enc(xi)
    z_aten = enc(xi.clone().requires_grad_(True))  # requires_grad input takes the ATen wavelet path
    assert rel_l2(z_fused, z_aten) < 1e-2


@pytest.mark.parametrize("shape", [(2, 32, 32, 128, 128), (2, 16, 16, 256, 512), (1, 64, 64, 128, 256), (3, 16, 32, 512, 256)])
def test_fused_groupnorm_backward_statistics_in_dgrad_epilogue(shape):
    """The data-gradient launch of the conv that consumes swish(GroupNorm(x)) accumulates (sum du, sum du*xhat) in its
    epilogue (vqb_conv_gemm_gnbwd) and the GroupNorm backward skips its reduction pass. Checked (a) against the unfused
    path (same kernels otherwise) and (b) against fp32 PyTorch autograd of the same block on the same bf16-rounded
    inputs, for dx, dgamma, dbeta and the conv's weight gradient; the fused path must actually have been taken."""
    import ae
    import native
    import ops
    import torch.nn.functional as F

    N, H, W, Cin, Cout = shape
    fuse_default = ops._GN_BWD_FUSE
    torch.manual_seed(0)
    norm = ae.FP32GroupNorm(32, Cin, eps=1e-6, affine=True).cuda()
    conv = ae.StandardizedC2d(Cin, Cout, kernel_size=3, stride=1, padding=1).cuda()
    with torch.no_grad():
        norm.weight.normal_(1.0, 0.2)
        norm.bias.normal_(0.0, 0.2)
    x0 = (torch.randn(N, H, W, Cin, device="cuda") * 1.5 + 0.3).to(torch.bfloat16)
    gy = torch.randn(N, H, W, Cout, device="cuda").to(torch.bfloat16)
    res = {}
    for fuse in (False, True, False):  # the first pass also warms the one-time weight packing launches
        ops._GN_BWD_FUSE = fuse
        for p_ in list(norm.parameters()) + list(conv.parameters()):
            p_.grad = None
        x = x0.clone().requires_grad_(True)
        a = ae.Act(x, Cin)
        h, skip = norm.forward_with_skip(a, silu=True)
        l0 = ops.gnbwd_fused_launches
        y = conv.forward_act(h)
        (y.t.float() * gy.float()).sum().backward()
        res[fuse] = (x.grad.float().clone(), norm.weight.grad.clone(), norm.bias.grad.clone(), conv.weight.grad.clone())
        res[("launches", fuse)] = ops.gnbwd_fused_launches - l0
    ops._GN_BWD_FUSE = fuse_default
    assert res[("launches", True)] == 1 and res[("launches", False)] == 0, "the fused path was not taken"
    # fp32 reference
    xr = x0.float().permute(0, 3, 1, 2).contiguous().requires_grad_(True)
    gw, gb = norm.weight.detach().clone().requires_grad_(True), norm.bias.detach().clone().requires_grad_(True)
    cw = conv.weight.detach().to(torch.bfloat16).float().requires_grad_(True)
    hh = F.group_norm(xr, 32, gw, gb, 1e-6)
    hh = (hh * torch.sigmoid(hh)).to(torch.bfloat16).float()  # the stored activation is bf16
    yy = F.conv2d(hh, cw, conv.bias.detach(), padding=1)
    (yy * gy.float().permute(0, 3, 1, 2)).sum().backward()
    ref = (xr.grad.permute(0, 2, 3, 1), gw.grad, gb.grad, cw.grad)
    names = ("dx", "dgamma", "dbeta", "dW")
    for i, nm in enumerate(names):
        e_fu = rel_l2(res[True][i], res[False][i])
        e_f, e_u = rel_l2(res[True][i], ref[i]), rel_l2(res[False][i], ref[i])
        print(f"  {shape} {nm}: fused vs unfused {e_fu:.2e}; vs fp32 torch: fused {e_f:.2e} unfused {e_u:.2e}")
        assert e_fu < 5e-3 and e_f < max(1.3 * e_u, 1e-2), nm


@pytest.mark.parametrize("gan", [False, True])
def test_cuda_graph_step_matches_eager_step(gan):
    """The whole step (fwd, bwd, both optimizers, weight re-pack) replayed as ONE CUDA graph must train like the eager
    step: same host-side random stream, same losses / weights up to bf16 noise over 8 steps (3 eager warm-up steps, the
    capture, then replays), with learning-rate schedule and bias corrections still advancing (device-resident record)."""
    import random

    import vae_trainer as vt

    def run(graph):
        tr = vt.Trainer("cuda:0", vae_resolution=64, vae_ch=32, vae_ch_mult="1,2", vae_num_res_blocks=1, vae_z_channels=4,
                        do_clamp=True, do_ganloss=gan, disc_type="hinge", use_lecam=gan, max_steps=50,
                        learning_rate_vae=2e-2, lpips_eval=True, cuda_graph=graph)
        random.seed(123)
        g = torch.Generator().manual_seed(9)
        batches = [(torch.rand(2, 3, 256, 256, generator=g) * 2 - 1).pin_memory() for _ in range(3)]
        losses = []
        for i in range(8):
            o = tr.step(batches[i % 3])
            losses.append(float(o["overall_vae_loss"]))
        torch.cuda.synchronize()
        w = tr.vae.module.decoder.conv_out.weight.detach().float().clone()
        return tr, losses, w, random.random()

    tr_e, le, we, re_ = run(False)
    tr_g, lg, wg, rg = run(True)
    assert tr_e.graph_launches_per_step is None and tr_g.graph_launches_per_step > 100
    print(f"\ngan={gan}: eager losses {['%.4f' % v for v in le]}\n          graph losses {['%.4f' % v for v in lg]}  "
          f"({tr_g.graph_launches_per_step} native launches per replay)")
    assert re_ == rg, "graph mode must consume the host random stream exactly like the eager step"
    for a, b in zip(le, lg):
        assert abs(a - b) <= 2e-2 * max(abs(a), 0.05), (le, lg)
    assert le[-1] != le[3] and lg[-1] != lg[3]
    assert rel_l2(wg, we) < 2e-2
    assert tr_g.optimizer_G.param_groups[0]["step"] == 8 and tr_e.optimizer_G.param_groups[0]["step"] == 8


def test_multi_pack_kernel_matches_single_tensor_pack_kernels():
    """vqb_pack_weights_multi (tile-based, one launch for every cached operand) against the per-tensor reference kernels
    vqb_pack_weights / vqb_pack_weights_fold and a torch restatement of the fat-pixel layout: bit-exact."""
    import ops
    import plans

    torch.manual_seed(0)
    cases = [(128, 128, 3, list(range(9)), False, 128, False), (256, 128, 3, list(range(8, -1, -1)), True, 256, False),
             (3, 128, 3, list(range(9)), False, 128, False), (128, 3, 3, list(range(9)), True, 128, False),
             (64, 32, 4, list(range(16)), False, 32, False), (512, 512, 1, [0], True, 512, False),
             (256, 256, 3, [0b000011011, 0b000110110, 0b011011000, 0b110110000], False, 256, True),
             (130, 70, 3, list(range(9)), False, 72, False)]
    ents, refs, keep = [], [], []
    for (Cout, Cin, k, tapmap, transpose, Kpad, fold) in cases:
        w = torch.randn(Cout, Cin, k, k, device="cuda")
        keep.append(w)  # entries hold weak references to their weights
        ents.append(ops._new_pack_entry(w, tapmap, transpose, Kpad, fold))
        refs.append(ops.pack_weights(w, tapmap, transpose, Kpad, fold))
    wf = torch.randn(64, 3, 3, 3, device="cuda")
    fat = ops._new_pack_entry(wf, list(range(9)), False, 8, False, fat=True)
    ops._run_pack(ents + [fat])  # ONE launch for all jobs
    torch.cuda.synchronize()
    for e, r, c in zip(ents, refs, cases):
        assert torch.equal(e.out, r), c
    plain = ops.pack_weights(wf, list(range(9)), False, 8)  # [64][9][8]
    want = torch.zeros(64, 3, plans.FAT_K, device="cuda", dtype=torch.bfloat16)
    want[:, :, :24] = plain.view(64, 3, 24)
    assert torch.equal(fat.out, want)


@pytest.mark.parametrize("ratio", [5.0, 20.0])
def test_fused_groupnorm_statistics_with_large_mean(ratio):
    """ADVICE r1 (low): the conv epilogue accumulates per-channel sum / sum-of-squares in fp32 atomics and the variance is
    E[x^2] - mean^2. With |mean| / std = `ratio` inside a group the cancellation costs ~ratio^2 * 1e-7 relative on the
    variance: measured here, and required to stay below the bf16 resolution of the normalised output (4e-3) up to a
    mean/std of 20 (the residual stream of this network stays below ~5)."""
    import ae
    import torch.nn.functional as F

    torch.manual_seed(0)
    C = 128
    conv = ae.StandardizedC2d(C, C, kernel_size=1, stride=1, padding=0).cuda()
    norm = ae.FP32GroupNorm(32, C, eps=1e-6, affine=True).cuda()
    with torch.no_grad():
        conv.weight.copy_(torch.eye(C).view(C, C, 1, 1) + 0.01 * torch.randn(C, C, 1, 1))
        conv.bias.fill_(ratio)  # every channel of a group shifted by `ratio` standard deviations
    x = torch.randn(4, 64, 64, C, device="cuda").to(torch.bfloat16)
    with torch.no_grad():
        h = conv.forward_act(ae.Act(x, C), want_stats=True)
        assert h.stats is not None, "the fused statistics path was not taken"
        y = norm(h, silu=False).t.float()
        ref = F.group_norm(h.t.float().permute(0, 3, 1, 2), 32, norm.weight, norm.bias, 1e-6).permute(0, 2, 3, 1)
    e = rel_l2(y, ref)
    print(f"\nfused GroupNorm statistics at |mean|/std = {ratio}: output rel-L2 vs fp32 group_norm {e:.2e}")
    assert e < 4e-3
