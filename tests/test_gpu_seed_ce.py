"""GPU suite (-m gpu): the sparse seed cross-entropy (csrc/seed.cuh seed_ce_forward_kernel / seed_ce_backward_kernel,
through SeedCrossEntropyFunction and FusedTcamLosses) against torch's cross-entropy in float64 on the label map the
same seeds paint (oracle/seeding.py seed_labels_from_sel).

The bar is torch's own float32 cross-entropy on that map, which is what SelfLearningTcams computes on a label map:
the loss and the gradient must be within twice its error of float64, plus 4 roundings of the reference.  Pointwise the
gradient also has a floor of four roundings of g/count: softmax - 1 cancels on a confident pixel, as it does in torch.
"""
import numpy as np
import pytest

from tcam_wsol_video_b200 import synth

pytestmark = pytest.mark.gpu

IGNORE = -255
U = 2.0 ** -24
LAMBDA_CE, LAMBDA_CRF = 0.75, 2e-9
G_CE, G_FUSED = 0.625, 1.25        # grad_outputs other than 1 (dyadic: the reference's scaling is exact)


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


def _distinct(rng, hw, n):
    return rng.choice(hw, size=min(n, hw), replace=False)


def _hand_sel(placement, b, h, w, ksz, kmax, seed):
    """sel [B,2,kmax] int32 with the seeds placed on purpose; unused slots are trailing -1 (as the seeder leaves them)."""
    rng = np.random.default_rng(seed)
    hw = h * w
    sel = np.full((b, 2, kmax), -1, np.int64)

    def put(i, side, pix):
        pix = list(dict.fromkeys(int(p) for p in pix))[:kmax]    # distinct within a side, order kept
        sel[i, side, :len(pix)] = pix

    for i in range(b):
        nf = kmax if i == 0 else int(rng.integers(0, kmax + 1))
        nb = kmax if i == 0 else int(rng.integers(0, kmax + 1))
        if placement == "corners":          # every corner and border, then random pixels
            ym, xm = h // 2, w // 2
            put(i, 0, [0, w - 1, (h - 1) * w, hw - 1] + list(_distinct(rng, hw, kmax)))
            put(i, 1, [xm, (h - 1) * w + xm, ym * w, ym * w + w - 1] + list(_distinct(rng, hw, nb)))
        elif placement == "overlap":        # one side's seeds packed into a small box: windows overlap
            y0, x0 = int(rng.integers(0, max(1, h - 2 * ksz))), int(rng.integers(0, max(1, w - 2 * ksz)))
            ys, xs = rng.integers(0, 2 * ksz, nf + 1), rng.integers(0, 2 * ksz, nf + 1)
            put(i, 0, [min(h - 1, y0 + y) * w + min(w - 1, x0 + x) for y, x in zip(ys, xs)])
            put(i, 1, _distinct(rng, hw, nb))
        elif placement == "conflict":       # each bg seed next to a fg seed: windows claimed by both sides
            fg = _distinct(rng, hw, nf)
            put(i, 0, fg)
            put(i, 1, [min(h - 1, p // w + int(rng.integers(0, ksz))) * w + min(w - 1, p % w + int(rng.integers(0, ksz)))
                       for p in fg])
        elif placement == "bg_only":
            put(i, 1, _distinct(rng, hw, nb))
        elif placement == "empty_batch":
            pass
        else:                               # random; "empty_sample" leaves sample 1 without any seed
            if placement == "empty_sample" and i == 1:
                continue
            put(i, 0, _distinct(rng, hw, nf))
            put(i, 1, _distinct(rng, hw, nb))
    return sel.astype(np.int32)


def _seeder_sel(torch, b, h, w, ksz, k, seed):
    """SparseSeeds from TCAMSeeder(rng_parity=False): fused kernel for k <= 32, select + labels kernels above."""
    from tcam_wsol_video_b200.tcam_seeding import TCAMSeeder
    g = torch.Generator().manual_seed(seed)
    low = torch.rand((b, 1, 7, 7), generator=g)
    cam = torch.nn.functional.interpolate(low, size=(h, w), mode="bilinear", align_corners=False).cuda()
    seeder = TCAMSeeder(seed_tech="seed_weighted", min_=k, max_=k, max_p=0.6, min_p=0.1, fg_erode_k=11,
                        fg_erode_iter=0, ksz=ksz, support_background=True, multi_label_flag=False,
                        seg_ignore_idx=IGNORE, cuda_id=0, roi_method="roi_all", p_min_area_roi=0.05, use_roi=True,
                        rng_parity=False)
    torch.manual_seed(seed)
    return seeder(cam, None, sparse=True)


def _logits(torch, kind, labels, k, seed):
    """[B,K,H,W] float32 CUDA logits of the given kind; `labels` [B,H,W] (CPU long) place the confident margins."""
    b, h, w = labels.shape
    g = torch.Generator().manual_seed(seed)
    z = torch.randn((b, k, h, w), generator=g, dtype=torch.float64)
    lab = labels != IGNORE
    at = lab.unsqueeze(1) & (torch.arange(k).view(1, k, 1, 1) == labels.clamp(min=0).unsqueeze(1))
    if kind.startswith("scale"):                        # scale3, scale30, scale80
        z = z * float(kind[5:])
    elif kind.startswith("confident"):                  # confident3+8: 3*randn, the label class wins by 8
        scale, margin = (float(v) for v in kind[9:].split("+"))
        z = z * scale
        zmax = z.max(dim=1, keepdim=True).values
        z = torch.where(at, zmax + margin, z)
    elif kind in ("minus1e30", "minusinf"):             # a non-label class at -1e30 / -inf on every labelled pixel
        other = lab.unsqueeze(1) & (torch.arange(k).view(1, k, 1, 1) == ((labels.clamp(min=0) + 1) % k).unsqueeze(1))
        z = torch.where(other, -1e30 if kind == "minus1e30" else float("-inf"), z)
    elif kind == "tied":
        z = z[:, :1].expand(b, k, h, w)
    elif kind == "denormal":
        z[:, k - 1] = 1e-41
    return z.float().contiguous().cuda()


def _reference(torch, z, labels, go):
    """(float64 loss, float64 gradient) and (torch float32 loss, gradient): F.cross_entropy(ignore_index) on the map."""
    import torch.nn.functional as F
    z64 = z.detach().double().cpu().requires_grad_(True)
    l64 = F.cross_entropy(z64, labels, ignore_index=IGNORE)
    l64.backward(torch.tensor(go, dtype=torch.float64))
    z32 = z.detach().clone().requires_grad_(True)
    l32 = F.cross_entropy(z32, labels.cuda(), ignore_index=IGNORE)
    l32.backward(torch.tensor(go, device="cuda"))
    return (l64.item(), z64.grad.numpy()), (l32.item(), z32.grad.double().cpu().numpy())


def _check_loss(got, ref64, t32, what):
    if np.isnan(ref64):
        assert np.isnan(got) and np.isnan(t32), what
        return
    assert abs(got - ref64) <= 2 * abs(t32 - ref64) + 4 * U * abs(ref64), (what, got, ref64, t32)


def _check_grad(got, ref64, t32, coef, what):
    """Normwise: 2x torch's error + 4 roundings; pointwise: the same with a floor of 4 roundings of |coef| (the size of
    the operands of p - 1)."""
    err, terr = np.abs(got - ref64), np.abs(t32 - ref64)
    norm = np.abs(ref64).max()
    assert err.max() <= 2 * terr.max() + 4 * U * norm, (what, err.max(), terr.max(), norm)
    bad = err > 2 * terr + 4 * U * np.abs(ref64) + 4 * U * abs(coef)
    assert not bad.any(), (what, int(bad.sum()), float(err[bad].max()), float(terr[bad].max()), coef)


# (id, B, K, H, W, ksz, kmax, placement, logits)
CASES = [
    ("readme", 5, 2, 224, 224, 3, 1, "random", "randn"),
    ("corners-even", 5, 2, 224, 224, 4, 3, "corners", "scale3"),
    ("corners-ksz2", 5, 3, 37, 53, 2, 32, "corners", "randn"),
    ("overlap", 1, 4, 37, 53, 5, 40, "overlap", "randn"),
    ("conflict-k10", 5, 10, 37, 53, 3, 3, "conflict", "scale30"),
    ("conflict-k21", 5, 21, 37, 53, 4, 32, "conflict", "scale80"),
    ("b300", 300, 2, 37, 53, 3, 3, "random", "randn"),
    ("b300-k10", 300, 10, 37, 53, 1, 1, "random", "scale3"),
    ("row", 5, 2, 1, 97, 3, 3, "random", "randn"),
    ("column", 5, 3, 83, 1, 4, 3, "corners", "randn"),
    ("ksz7-4x5", 1, 2, 4, 5, 7, 3, "bg_only", "randn"),   # every window covers the frame
    ("bg-only", 5, 3, 37, 53, 3, 3, "bg_only", "randn"),
    ("empty-sample", 5, 2, 37, 53, 3, 32, "empty_sample", "randn"),
    ("empty-batch", 5, 4, 37, 53, 3, 3, "empty_batch", "randn"),
    ("confident3+8", 5, 2, 37, 53, 5, 32, "random", "confident3+8"),
    ("confident20+10", 5, 2, 37, 53, 5, 32, "random", "confident20+10"),
    ("confident50+12", 5, 2, 37, 53, 5, 32, "random", "confident50+12"),
    ("confident-k10", 5, 10, 37, 53, 3, 32, "random", "confident20+10"),
    ("minus1e30", 5, 3, 37, 53, 3, 3, "random", "minus1e30"),
    ("minusinf", 5, 2, 37, 53, 3, 3, "conflict", "minusinf"),
    ("tied", 5, 4, 37, 53, 3, 3, "random", "tied"),
    ("denormal", 5, 3, 37, 53, 2, 3, "random", "denormal"),
    ("seeder-fused", 5, 2, 224, 224, 3, 3, "seeder", "randn"),
    ("seeder-fused-b300", 300, 2, 37, 53, 5, 1, "seeder", "confident3+8"),
    ("seeder-two-kernel", 5, 3, 37, 53, 2, 40, "seeder", "randn"),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_seed_cross_entropy_against_float64(torch_cuda, case):
    """Per case: the painted map and the count exactly; loss and gradient (SeedCrossEntropyFunction and
    FusedTcamLosses) against float64 within twice torch's float32 error; a gradient of exactly 0 off the labelled
    pixels, and on the fused path bit for bit the CRF-only backward there; the fused total is fl(crf + fl(lambda*ce));
    two identical calls are bit-identical."""
    torch = torch_cuda
    from oracle import seeding as oseed
    from tcam_wsol_video_b200 import ops
    from tcam_wsol_video_b200.dense_crf_loss import SeedCrossEntropyFunction
    from tcam_wsol_video_b200.losses import ConRanFieldTcams, FusedTcamLosses, SelfLearningTcams
    from tcam_wsol_video_b200.tcam_seeding import SparseSeeds
    name, b, k, h, w, ksz, kmax, placement, kind = case
    seed = sum(map(ord, name))
    if placement == "seeder":
        seeds = _seeder_sel(torch, b, h, w, ksz, kmax, seed)
        assert seeds.kmax == kmax
    else:
        seeds = SparseSeeds(torch.from_numpy(_hand_sel(placement, b, h, w, ksz, kmax, seed)).cuda(), ksz, IGNORE, h, w)
    labels = oseed.seed_labels_from_sel(seeds.sel.cpu(), ksz, h, w, IGNORE)
    assert torch.equal(seeds.dense().cpu(), labels), name
    labelled = labels != IGNORE
    n = int(labelled.sum())
    assert (n == 0) == (placement == "empty_batch"), name
    z = _logits(torch, kind, labels, k, seed)
    off = ~labelled.unsqueeze(1).expand(b, k, h, w).numpy()

    # SeedCrossEntropyFunction (what SelfLearningTcams runs on SparseSeeds), grad_output G_CE
    (ref_l, ref_g), (t32_l, t32_g) = _reference(torch, z, labels, G_CE)
    runs = []
    for _ in range(2):
        zz = z.clone().requires_grad_(True)
        loss = SeedCrossEntropyFunction.apply(zz, seeds.sel, ksz)
        count = loss.grad_fn.count.item()
        loss.backward(torch.full_like(loss, G_CE))
        runs.append((loss.item(), count, zz.grad.cpu().numpy()))
    assert runs[0][0] == runs[1][0] or np.isnan(runs[0][0]), name
    assert np.array_equal(runs[0][2], runs[1][2]), name
    got_l, count, got_g = runs[0]
    assert count == n, (name, count, n)
    _check_loss(got_l, ref_l, t32_l, name)
    assert (got_g[off] == 0).all(), name
    if n == 0:
        assert (got_g == 0).all() and (t32_g == 0).all(), name
    else:
        _check_grad(got_g, ref_g, t32_g, G_CE / n, name)

    # FusedTcamLosses: CRF + LAMBDA_CE * CE as one node, the CE gradient added in place; grad_output G_FUSED
    raw = torch.from_numpy(synth.make_images(b, h, w, "natural", seed=seed).astype(np.uint8)).cuda()
    sl = SelfLearningTcams(cuda_id=0, lambda_=LAMBDA_CE)
    crf = ConRanFieldTcams(cuda_id=0, lambda_=LAMBDA_CRF, sigma_rgb=15., sigma_xy=100., scale_factor=1.0,
                           fuse_softmax=True)
    fused = FusedTcamLosses(sl, crf)
    ces = []
    for _ in range(2):
        zz = z.clone().requires_grad_(True)
        total = fused(epoch=0, fcams=zz, raw_img=raw, seeds=seeds)
        crf_l, ce_l = np.float32(fused.last_crf.item()), np.float32(fused.last_ce.item())
        assert np.float32(total.item()) == np.float32(crf_l + np.float32(np.float32(LAMBDA_CE) * ce_l)) or n == 0, name
        ces.append(ce_l)
        node = total.grad_fn
        total.backward(torch.full_like(total, G_FUSED))
        # the CRF-only backward from the same AS (bit-exact given AS)
        crf_only = ops.crf_backward_logits(node.AS, node.logits, torch.full((1,), G_FUSED, device="cuda"),
                                           float(node.N), node.crf_weight).cpu().numpy()
        fg = zz.grad.cpu().numpy()
        assert np.array_equal(fg[off], crf_only[off]), name
    assert ces[0] == ces[1] or np.isnan(ces[0]), name
    _check_loss(float(ces[0]), ref_l, t32_l, name + " fused")
    if n:
        scale = LAMBDA_CE * G_FUSED / G_CE
        ce_part = fg.astype(np.float64) - crf_only.astype(np.float64)
        # the in-place add rounds once more at the size of the sum
        slack = U * np.abs(fg.astype(np.float64))
        err = np.abs(ce_part - ref_g * scale)
        terr = np.abs(t32_g - ref_g) * scale
        assert err.max() <= 2 * terr.max() + 4 * U * np.abs(ref_g * scale).max() + slack.max(), name
        bad = err > 2 * terr + 4 * U * np.abs(ref_g * scale) + 4 * U * LAMBDA_CE * G_FUSED / n + slack
        assert not bad.any(), (name, int(bad.sum()))


def test_fused_losses_in_a_cuda_graph(torch_cuda):
    """FusedTcamLosses captured on a fresh stream with SparseSeeds from rng_parity=False, replayed 3x on new logits and
    new seeds: every replay's cross-entropy and count equal an eager call's bit for bit, its gradient equals the
    CRF-only backward of the replay's AS plus the eager cross-entropy backward, bit for bit (the final-fold ticket is
    back at zero after every replay).  Then an eager call with another B on the same stream (scratch cached per B)."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    from tcam_wsol_video_b200.losses import ConRanFieldTcams, FusedTcamLosses, SelfLearningTcams
    from tcam_wsol_video_b200.tcam_seeding import SparseSeeds
    b, k, h, w, ksz, kmax = 6, 3, 48, 56, 3, 4
    sl = SelfLearningTcams(cuda_id=0, lambda_=LAMBDA_CE)
    crf = ConRanFieldTcams(cuda_id=0, lambda_=LAMBDA_CRF, sigma_rgb=15., sigma_xy=100., scale_factor=1.0,
                           fuse_softmax=True)
    fused = FusedTcamLosses(sl, crf)
    raw = torch.from_numpy(synth.make_images(b, h, w, "natural", seed=4).astype(np.uint8)).cuda()
    logits = torch.zeros((b, k, h, w), device="cuda", requires_grad=True)
    sel = torch.full((b, 2, kmax), -1, dtype=torch.int32, device="cuda")
    seeds = SparseSeeds(sel, ksz, IGNORE, h, w)

    def load(seed):
        s = _seeder_sel(torch, b, h, w, ksz, kmax, seed)
        sel.copy_(s.sel)
        with torch.no_grad():
            logits.copy_(torch.randn((b, k, h, w), generator=torch.Generator().manual_seed(seed)) * 3)

    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        load(1)
        graph = torch.cuda.CUDAGraph()
        logits.grad = None
        with torch.cuda.graph(graph, stream=stream):
            total = fused(epoch=0, fcams=logits, raw_img=raw, seeds=seeds)
            total.backward()
        node_as, crf_w, n_frames = total.grad_fn.AS, total.grad_fn.crf_weight, total.grad_fn.N
        g_ce, g_crf = fused.last_ce, fused.last_crf
        for seed in (2, 3, 4):
            load(seed)
            logits.grad.zero_()
            graph.replay()
            stream.synchronize()
            got_grad = logits.grad.clone()
            z = logits.detach().clone()
            eager_loss, eager_count, _ = ops.seed_ce_forward(z, sel, ksz)
            assert g_ce.item() == eager_loss.item() and np.isfinite(eager_loss.item()), seed
            assert np.float32(total.item()) == np.float32(np.float32(g_crf.item()) +
                                                          np.float32(np.float32(LAMBDA_CE) * np.float32(g_ce.item())))
            one = torch.ones(1, device="cuda")
            want = ops.crf_backward_logits(node_as, z, one, float(n_frames), crf_w)
            ops.seed_ce_backward_(want, z, sel, ksz, eager_count, one, LAMBDA_CE)
            assert torch.equal(got_grad, want), seed
            # and an eager FusedTcamLosses call on the same inputs gives the same cross-entropy
            zz = z.clone().requires_grad_(True)
            fused(epoch=0, fcams=zz, raw_img=raw, seeds=seeds)
            assert fused.last_ce.item() == eager_loss.item(), seed
            fused.last_ce, fused.last_crf = g_ce, g_crf
        # another B on the same stream
        b2 = 3
        s2 = _seeder_sel(torch, b2, h, w, ksz, kmax, 9)
        z2 = torch.randn((b2, k, h, w), generator=torch.Generator().manual_seed(9)).cuda()
        labels = s2.dense().cpu()
        got = ops.seed_ce_forward(z2, s2.sel, ksz)[0].item()
        (ref_l, _), (t32_l, _) = _reference(torch, z2, labels, 1.0)
        _check_loss(got, ref_l, t32_l, "B=3 after the graph")
    torch.cuda.synchronize()
