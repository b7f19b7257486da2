"""Deterministic mode of head training (trainer.deterministic): the fixed-order variants of every reduction of the training
step, the trainer, fit_head and train_model with the mode on, and its refusals. The config plumbing and the ABI refusals
need no GPU."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

DEV = "cuda"
ROOT = Path(__file__).resolve().parent.parent
gpu = pytest.mark.gpu
BF16, F32 = torch.bfloat16, torch.float32


# ----------------------------------------------------------------------------------------------- config (CPU)
def _entry_data(tmp_path, n_per_sample=4):
    import pandas as pd
    from cryovit_b200.host import hdf

    rng = np.random.default_rng(4)
    rows = []
    for s in ("A", "B"):
        for i in range(n_per_sample):
            feats = (0.1 * rng.standard_normal((384, 4, 3, 3))).astype(np.float16)
            feats[0] = 2.0 * np.sign(rng.standard_normal((4, 3, 3)))
            lab = (np.repeat(np.repeat(feats[0].astype(np.float32), 16, axis=1), 16, axis=2) > 0).astype(np.int8)
            lab[0, :8] = -1
            hdf.write_tomogram(tmp_path / "data" / "tomograms" / s / f"{s}{i}.hdf",
                               {"data": rng.integers(0, 256, (4, 48, 48), dtype=np.uint8), "labels/mito": lab, "dino_features": feats})
            rows.append((s, f"{s}{i}.hdf", i % 2))
    (tmp_path / "data" / "csv").mkdir(parents=True, exist_ok=True)
    pd.DataFrame(rows, columns=["sample", "tomo_name", "split_id"]).to_csv(tmp_path / "data" / "csv" / "splits.csv", index=False)
    return ["model=cryovit", "+experiments=multi_mito", "datamodule.sample=[A,B]", "datamodule.split_id=0", "+model.in_channels=384",
            f"paths.data_dir={tmp_path / 'data'}"]


@pytest.mark.parametrize("override, want", [(None, False), ("+trainer.deterministic=false", False),
                                            ("+trainer.deterministic=true", True), ("+trainer.deterministic=warn", "warn")])
def test_run_trainer_passes_trainer_deterministic_to_fit_head(tmp_path, monkeypatch, override, want):
    from cryovit.config import compose
    from cryovit_b200.host import train_model

    got = {}

    def fake_fit_head(*args, **kw):
        got.update(kw)
        return {}

    monkeypatch.setattr(train_model, "fit_head", fake_fit_head)
    common = _entry_data(tmp_path)
    cfg = compose("train_model", common + [f"paths.exp_dir={tmp_path / 'exp'}"] + ([override] if override else []))
    train_model.run_trainer(cfg)
    assert got["deterministic"] == want and type(got["deterministic"]) is type(want)


def test_run_trainer_refuses_an_unknown_deterministic_value(tmp_path, monkeypatch):
    from cryovit.config import compose
    from cryovit_b200.host import train_model

    monkeypatch.setattr(train_model, "fit_head", lambda *a, **k: pytest.fail("fit_head reached"))
    cfg = compose("train_model", _entry_data(tmp_path) + [f"paths.exp_dir={tmp_path / 'exp'}", "+trainer.deterministic=sometimes"])
    with pytest.raises(ValueError, match="trainer.deterministic"):
        train_model.run_trainer(cfg)


def test_fit_head_refuses_an_unknown_deterministic_value():
    from cryovit_b200.host.fit import fit_head

    with pytest.raises(ValueError, match="deterministic"):
        fit_head([], in_channels=384, deterministic="yes")


# ----------------------------------------------------------------------------------------------- ABI refusals (CPU)
def test_det_entry_points_refuse_missing_or_small_scratch():
    """Every *_det entry point returns CVIT_ERR_INVALID for a null scratch or one element short of *_det_partials, before any
    CUDA call (the pointers are never dereferenced)."""
    from cryovit_b200 import _lib, build

    build.build()
    lib = _lib.load()
    f = 1 << 20  # 16-byte aligned, never dereferenced
    cases = {
        # name: (args before scratch, partials args)
        "cvit_groupnorm_ndhwc_bf16_det": ((f, f, f, f, f, 4096, 128, 16, 1e-3), (4096, 128, 16)),
        "cvit_seg_stats_det": ((f, f, 1 << 20, 0.5, f), (1 << 20,)),
        "cvit_colsum_bf16_det": ((f, f, 1 << 16, 64), (1 << 16, 64)),
        "cvit_gelu_bwd_colsum_bf16_det": ((f, f, f, f, 1 << 16, 64), (1 << 16, 64)),
        "cvit_gelu_bwd_colsum_unshuffle_bf16_det": ((f, f, f, f, 4, 64, 64, 32), (4, 64, 64, 32)),
        "cvit_groupnorm_bwd_gelu_ndhwc_bf16_det": ((f, f, f, f, f, f, f, 4096, 128, 16, 1e-3, f, f, 0), (4096, 128, 16)),
        "cvit_wgrad_tc8_ndhwc_det": ((f, f, f, 4, 64, 64, 1), (4, 64, 64)),
        "cvit_wgrad_tcn_ndhwc_det": ((f, f, f, 4, 64, 64, 32, 16, 2), (4, 64, 64, 32, 16)),
        "cvit_wgrad_mn_ndhwc_det": ((f, f, f, 4, 32, 32, 1024, 192, 8, 27, 1), (4, 32, 32, 1024, 192, 27)),
        "cvit_wgrad_splitk_det": ((f, f, f, f, 1024, 1536, 4096, 4096, 4096, 1), (1024, 1536, 4096, 1)),
    }
    for name, (pre, part) in cases.items():
        need = getattr(lib, name + "_partials")(*part)
        assert need > 0, name
        fn = getattr(lib, name)
        assert fn(*pre, None, need, None) == -1, name
        assert "scratch" in lib.cvit_last_error().decode(), name
        assert fn(*pre, f, need - 1, None) == -1, name
        assert "scratch" in lib.cvit_last_error().decode(), name
    assert lib.cvit_colsum_bf16_det_partials(0, 64) == 0


# ----------------------------------------------------------------------------------------------- per kernel (GPU)
def _mixed(shape, seed, dtype=BF16):
    """Seeded values of both signs over six decades, so that the summation order shows in the bits."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    mag = torch.exp(torch.empty(shape, device=DEV).uniform_(-7.0, 7.0, generator=g))
    sign = torch.where(torch.rand(shape, device=DEV, generator=g) < 0.5, -1.0, 1.0)
    return (sign * mag * 0.01).to(dtype)


def _rel(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


class _Scratch:
    def __init__(self):
        self.bufs = {}

    def __call__(self, n, dtype=F32):
        b = self.bufs.get(dtype)
        if b is None or b.numel() < n:
            b = self.bufs[dtype] = torch.empty(max(n, 1), device=DEV, dtype=dtype)
        return b


def _check(run, ref64, tol=1e-4):
    """run(det) -> output tensor (fresh each call). Two deterministic launches are bit-identical; they agree with the float64
    reference and with the atomic twin (det=None) within fp32 accumulation error."""
    det = _Scratch()
    a = run(det).clone()
    det.bufs = {k: torch.full_like(v, float("nan")) for k, v in det.bufs.items()}  # no reliance on the scratch's old contents
    b = run(det).clone()
    twin = run(None).clone()
    torch.cuda.synchronize()
    assert torch.equal(a, b)
    assert _rel(a, ref64) <= tol, _rel(a, ref64)
    assert _rel(a, twin) <= tol, _rel(a, twin)
    return a


# the production step (fp16 1536 x 128 x 32 x 32 features, 128 x 512 x 512 labels): (D, H, W, C, G) of the four GroupNorms
GN_SHAPES = [(128, 32, 32, 1024, 128), (128, 64, 64, 128, 16), (128, 128, 128, 32, 8), (128, 256, 256, 32, 8)]


@gpu
@pytest.mark.parametrize("shape", GN_SHAPES)
def test_groupnorm_stats_det(cuda_lib, shape):
    from cryovit_b200 import ops

    D, H, W, C, G = shape
    x = _mixed((D, H, W, C), 1)
    gamma, beta = torch.rand(C, device=DEV) + 0.5, torch.rand(C, device=DEV) - 0.5

    def run(det):
        out, stats = torch.empty_like(x), torch.empty(2 * G, device=DEV)
        ops.groupnorm_ndhwc(x, out, gamma, beta, stats, G, 1e-3, det=det)
        return stats

    xg = x.double().view(-1, G, C // G)
    ref = torch.cat([xg.sum(dim=(0, 2)), (xg * xg).sum(dim=(0, 2))])
    _check(run, ref)


@gpu
def test_seg_stats_det(cuda_lib):
    from cryovit_b200 import ops

    n = 128 * 512 * 512
    g = torch.Generator(device=DEV).manual_seed(2)
    probs = torch.rand(n, device=DEV, generator=g)
    lab = (torch.rand(n, device=DEV, generator=g) < 0.4).float()
    lab[: n // 10] = -1

    def run(det):
        return ops.seg_stats(probs, lab, det=det)

    m = lab > -1
    p, y = probs.double()[m], lab.double()[m]
    hge, hgt = (p >= 0.5).double(), (p > 0.5).double()
    ref = torch.stack([p.sum(), y.sum(), (p * y).sum(), (y * hge).sum(), hge.sum(), (y * hgt).sum(), ((1 - y) * hgt).sum(),
                       (y * (1 - hgt)).sum()])
    got = _check(run, ref, tol=1e-9)
    assert torch.equal(got[[1, 3, 4, 5, 6, 7]], ref[[1, 3, 4, 5, 6, 7]])


@gpu
@pytest.mark.parametrize("shape", [(128, 512, 512, 8), (128, 256, 256, 16), (128, 128, 128, 32), (128, 32, 32, 192)])
def test_colsum_det(cuda_lib, shape):
    from cryovit_b200 import train_ops as T

    x = _mixed(shape, 3)

    def run(det):
        out = torch.zeros(shape[-1], device=DEV)
        T.colsum(x, out, det=det)
        return out

    _check(run, x.double().reshape(-1, shape[-1]).sum(0))


def _gelu_grad64(z):
    z = z.double()
    return 0.5 * (1 + torch.erf(z / 2 ** 0.5)) + z * torch.exp(-0.5 * z * z) / (2 * torch.pi) ** 0.5


@gpu
@pytest.mark.parametrize("shape", [(128, 32, 32, 192), (128, 64, 64, 64), (128, 256, 256, 16)])
def test_gelu_bwd_colsum_det(cuda_lib, shape):
    from cryovit_b200 import train_ops as T

    da, z = _mixed(shape, 4), _mixed(shape, 5)

    def run(det):
        dz, db = torch.empty_like(da), torch.zeros(shape[-1], device=DEV)
        T.gelu_bwd(da, z, dz, db, det=det)
        return db

    dz_stored = (da.double() * _gelu_grad64(z)).to(BF16)  # the sums are over the stored bf16 gradient
    _check(run, dz_stored.double().reshape(-1, shape[-1]).sum(0))


@gpu
def test_gelu_bwd_unshuffle_det(cuda_lib):
    from cryovit_b200 import train_ops as T

    shape = (128, 512, 512, 8)
    da, z = _mixed(shape, 6), _mixed(shape, 7)

    def run(det):
        dzun, db = torch.empty(128, 256, 256, 32, device=DEV, dtype=BF16), torch.zeros(8, device=DEV)
        T.gelu_bwd_unshuffle(da, z, dzun, db, det=det)
        return torch.cat([db, dzun.float().flatten()[:4096]])

    dz_stored = (da.double() * _gelu_grad64(z)).to(BF16).double()
    ref_un = dz_stored.view(128, 256, 2, 256, 2, 8).permute(0, 1, 3, 2, 4, 5).reshape(-1)[:4096]
    _check(run, torch.cat([dz_stored.reshape(-1, 8).sum(0), ref_un]))


@gpu
@pytest.mark.parametrize("case", ["gelu_unshuffle", "gelu_proj", "plain"])
def test_groupnorm_bwd_det(cuda_lib, case):
    from cryovit_b200 import train_ops as T

    if case == "gelu_unshuffle":   # block 1's GroupNorm over block 0's transposed-convolution output
        D, H, W, C, G = 128, 64, 64, 128, 16
    else:                          # block 0's GroupNorm over the projection
        D, H, W, C, G = 128, 32, 32, 1024, 128
    x, dy, z = _mixed((D, H, W, C), 8), _mixed((D, H, W, C), 9), _mixed((D, H, W, C), 10)
    gamma = torch.rand(C, device=DEV) + 0.5
    xg = x.double().view(-1, G, C // G)
    stats = torch.cat([xg.sum(dim=(0, 2)), (xg * xg).sum(dim=(0, 2))]).float()

    def run(det):
        dgam, dbet, db = torch.empty(C, device=DEV), torch.empty(C, device=DEV), torch.zeros(C, device=DEV)
        if case == "plain":
            dx = torch.empty_like(x)
            T.groupnorm_bwd(x, dy, dx, gamma, stats, dgam, dbet, G, 1e-3, det=det)
            return torch.cat([dgam, dbet])
        dz = torch.empty((D, H // 2, W // 2, 4 * C) if case == "gelu_unshuffle" else (D, H, W, C), device=DEV, dtype=BF16)
        T.groupnorm_bwd_gelu(x, dy, dz, gamma, stats, dgam, dbet, G, 1e-3, z, db, case == "gelu_unshuffle", det=det)
        return torch.cat([dgam, dbet, db])

    n = x.numel() // G
    mean = stats[:G].double() / n
    rstd = 1.0 / torch.sqrt((stats[G:].double() / n - mean * mean).clamp_min(0) + 1e-3)
    xhat = ((xg - mean[None, :, None]) * rstd[None, :, None]).reshape(-1, C)
    dyf = dy.double().reshape(-1, C)
    ref = [(dyf * xhat).sum(0), dyf.sum(0)]
    if case != "plain":
        # db: the column sums of the stored d(z) (the trainer's kernel output), checked against the twin and run to run here;
        # its float64 value follows from dgamma / dbeta, which are checked against float64 above
        det = _Scratch()
        got = run(det)
        twin = run(None)
        assert torch.equal(got, run(det))
        assert _rel(got[2 * C:], twin[2 * C:]) <= 1e-4
        assert _rel(got[:2 * C], torch.cat(ref)) <= 1e-4 and _rel(got[:2 * C], twin[:2 * C]) <= 1e-4
        return
    _check(run, torch.cat(ref))


def _wgrad64(x, dz, dil):
    """float64 dW[27, Cout, Cin] of the 3x3x3 depth-dilated "same" convolution (tap = (kd*3+kh)*3+kw)."""
    xi = x.double().permute(3, 0, 1, 2)[None]
    gi = dz.double().permute(3, 0, 1, 2)[None]
    w = torch.nn.grad.conv3d_weight(xi, (gi.shape[1], xi.shape[1], 3, 3, 3), gi, padding=(dil, 1, 1), dilation=(dil, 1, 1))
    return w.permute(2, 3, 4, 0, 1).reshape(27, gi.shape[1], xi.shape[1])


# (D, H, W, Cin, Cout, dil): the production layers of each kernel; the float64 reference runs on the first 16 planes
WGRAD_SHAPES = [(128, 512, 512, 8, 8, 1), (128, 256, 256, 32, 16, 2), (128, 256, 256, 16, 16, 1), (128, 128, 128, 32, 32, 8),
                (128, 32, 32, 1024, 192, 32), (128, 32, 32, 192, 192, 24), (128, 64, 64, 128, 64, 16), (128, 64, 64, 64, 64, 12)]


@gpu
@pytest.mark.parametrize("shape", WGRAD_SHAPES)
def test_conv_weight_gradient_det(cuda_lib, shape):
    """wgrad_tc8 (8 -> 8), wgrad_tcn (16 / 32 channels), wgrad_mn (>= 64 channels) at the step's shapes: bit-identical runs,
    the atomic twin at the full depth, float64 on the first 16 planes (the same kernels, a shorter reduction)."""
    from cryovit_b200 import train_ops as T

    D, H, W, Cin, Cout, dil = shape
    x, dz = _mixed((D, H, W, Cin), 11), _mixed((D, H, W, Cout), 12)
    run = lambda det, x=x, dz=dz: T.conv_weight_gradient(x, dz, dil, {}, det=det).contiguous()
    det = _Scratch()
    a = run(det).clone()
    b = run(det).clone()
    twin = run(None)
    assert torch.equal(a, b)
    assert _rel(a, twin) <= 1e-4, _rel(a, twin)
    xs, dzs = x[:16].contiguous(), dz[:16].contiguous()
    got = T.conv_weight_gradient(xs, dzs, dil, {}, det=det)
    assert _rel(got, _wgrad64(xs, dzs, dil)) <= 1e-4


@gpu
def test_rows_weight_gradients_det(cuda_lib):
    """The 1x1x1 / transposed-convolution weight gradients: wgrad_mn in rows mode (block 0's transposed convolution) and the
    split-K GEMM of the projection on the channels-first fp16 path."""
    from cryovit_b200 import train_ops as T

    R = 128 * 32 * 32
    x, dz = _mixed((R, 192), 13), _mixed((R, 512), 14)
    run = lambda det: T.rows_weight_gradient(x, dz, det=det).contiguous()
    _check(run, dz.double().t() @ x.double())
    feats_t, dzp = _mixed((1536, R), 15), _mixed((R, 1024), 16)  # features as they lie (C, vox), bf16
    dzt = torch.empty(1024, R, device=DEV, dtype=BF16)
    T.to_cfirst_padded(dzp.view(1, 1, R, 1024), dzt, 0, 0, 0)
    koff = torch.zeros(1, dtype=torch.int32, device=DEV)

    def run_sk(det):
        out = torch.zeros(1, 1024, 1536, device=DEV)
        T.wgrad_splitk(dzt, feats_t, out, koff, R, det=det)
        return out

    _check(run_sk, dzp.double().t() @ feats_t.double().t())


# ----------------------------------------------------------------------------------------------- the step (GPU)
def _crop(seed, C=1536, D=128, h=32, w=32):
    g = torch.Generator().manual_seed(seed)
    feats = torch.randn(C, D, h, w, generator=g).half()
    lab = (torch.rand(D, 16 * h, 16 * w, generator=g) < 0.3).float()
    lab[:, :64, :] = -1  # an ignored region
    return feats.to(DEV), lab.to(DEV)


def _five_steps(env_graph="1", deterministic=True, seed=3):
    """Five steps of a fresh trainer at the production crop: eager, eager, capture, replay, replay (CVIT_TRAIN_GRAPH=1)."""
    from cryovit_b200.train import CryoVITHeadTrainerB200

    old = os.environ.get("CVIT_TRAIN_GRAPH")
    os.environ["CVIT_TRAIN_GRAPH"] = env_graph
    try:
        tr = CryoVITHeadTrainerB200(1536, seed=seed, deterministic=deterministic)
        losses = []
        for k in range(5):
            f, l = _crop(100 + k)
            losses.append(tr.train_step(f, l).clone())
        torch.cuda.synchronize()
        return tr, torch.stack(losses)
    finally:
        if old is None:
            os.environ.pop("CVIT_TRAIN_GRAPH", None)
        else:
            os.environ["CVIT_TRAIN_GRAPH"] = old


@gpu
def test_deterministic_step_is_bit_reproducible(cuda_lib):
    prev = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
    torch.use_deterministic_algorithms(True)
    try:
        runs = [_five_steps("1"), _five_steps("1"), _five_steps("0")]
    finally:
        torch.use_deterministic_algorithms(prev[0], warn_only=prev[1])
    (a, la), (b, lb), (c, lc) = runs
    assert a._graphs and any("graph" in e for e in a._graphs.values())  # steps 3-5 ran as a capture and replays
    for t in ("flat_p", "flat_m", "flat_v", "flat_g"):
        assert torch.equal(getattr(a, t), getattr(b, t)), t
        assert torch.equal(getattr(a, t), getattr(c, t)), t
    assert torch.equal(la, lb) and torch.equal(la, lc)
    assert torch.isfinite(la).all()


@gpu
def test_deterministic_step_computes_the_default_gradients(cuda_lib):
    """One step's gradient bucket, per parameter: deterministic against default within the larger of twice the default path's
    own run-to-run difference and 1e-4 (relative L2)."""
    from cryovit_b200.head import state_dict_keys
    from cryovit_b200.train import CryoVITHeadTrainerB200

    f, l = _crop(7)

    def grads(deterministic):
        tr = CryoVITHeadTrainerB200(1536, seed=3, deterministic=deterministic)
        tr.forward_backward(f, l)
        torch.cuda.synchronize()
        return {k: v.clone() for k, v in tr.g.items()}

    d0, d1, det = grads(False), grads(False), grads(True)
    worst = 0.0
    for k in state_dict_keys():
        noise = _rel(d1[k], d0[k])
        r = _rel(det[k], d0[k])
        worst = max(worst, r)
        assert r <= max(2 * noise, 1e-4), (k, r, noise)
    print(f"\n[deterministic] worst relative L2 gradient difference from the default path: {worst:.2e}")


# ----------------------------------------------------------------------------------------------- fit_head and train_model
def _toy_split(root: Path, n_train: int, n_val: int, seed: int = 4):
    from cryovit.datasets import TomoDataset
    from cryovit_b200.host import hdf

    rng = np.random.default_rng(seed)
    recs = []
    for i in range(n_train + n_val):
        feats = (0.1 * rng.standard_normal((384, 4, 3, 3))).astype(np.float16)
        feats[0] = 2.0 * np.sign(rng.standard_normal((4, 3, 3)))
        lab = (np.repeat(np.repeat(feats[0].astype(np.float32), 16, axis=1), 16, axis=2) > 0).astype(np.int8)
        lab[0, :8] = -1
        hdf.write_tomogram(root / "S" / f"t{i}.hdf", {"data": np.zeros((4, 48, 48), np.uint8), "labels/mito": lab, "dino_features": feats})
        recs.append({"sample": "S", "tomo_name": f"t{i}.hdf"})
    mk = lambda r, train: TomoDataset(r, "dino_features", "mito", "split_id", root, train=train)
    return mk(recs[:n_train], True), mk(recs[n_train:], False)


def _fit(tmp_path, tag, deterministic, validate=True):
    import pandas as pd
    from cryovit_b200.host.fit import fit_head
    from cryovit_b200.host.metrics import DiceLoss, DiceMetric, F1Metric
    from cryovit_b200.host.validate import Validator
    from oracle import head as ohead

    train, val = _toy_split(tmp_path / "data", 4, 2)
    v = Validator(val, 384, {"dice_loss": DiceLoss()}, {"dice_metric": DiceMetric(0.5), "f1_metric": F1Metric()}, 1, 1.0) if validate else None
    sd = fit_head(train, in_channels=384, max_epochs=3, lr=2e-3, swa_epoch_start=1, exp_dir=tmp_path / tag,
                  state_dict=ohead.random_state_dict(384, seed=5), validator=v, deterministic=deterministic)
    csv = tmp_path / tag / "validation.csv"
    return sd, (pd.read_csv(csv).drop(columns=["seconds"]) if csv.exists() else None)


@gpu
def test_fit_head_deterministic_runs_are_identical(cuda_lib, tmp_path):
    prev = torch.are_deterministic_algorithms_enabled()
    a, va = _fit(tmp_path, "a", True)
    assert torch.are_deterministic_algorithms_enabled() == prev  # restored on exit
    b, vb = _fit(tmp_path, "b", True)
    c, vc = _fit(tmp_path, "c", True, validate=False)
    assert all(torch.equal(a[k], b[k]) for k in a)
    assert va.equals(vb) and len(va) == 3
    assert vc is None and all(torch.equal(a[k], c[k]) for k in a)  # validation changes nothing in the training run
    wa, wb = (torch.load(tmp_path / t / "weights.pt") for t in ("a", "b"))
    assert all(torch.equal(wa[k], wb[k]) for k in wa)


@gpu
def test_fit_head_default_mode_control(cuda_lib, tmp_path):
    """The same two runs in the default mode: the atomics' run-to-run difference, printed (expected non-zero), not asserted."""
    a, _ = _fit(tmp_path, "a", False)
    b, _ = _fit(tmp_path, "b", False)
    diff = max(float((a[k] - b[k]).abs().max()) for k in a)
    print(f"\n[control] default mode, two fit_head runs: max |weight difference| = {diff:.3e}")


@gpu
def test_train_model_deterministic_twice_gives_equal_weights(cuda_lib, tmp_path):
    common = _entry_data(tmp_path)
    env = dict(os.environ, PYTHONPATH=str(ROOT) + os.pathsep + os.environ.get("PYTHONPATH", ""))
    weights = []
    for tag in ("one", "two"):
        r = subprocess.run([sys.executable, "-m", "cryovit.training.train_model", *common, f"paths.exp_dir={tmp_path / tag}",
                            "trainer.max_epochs=3", "+trainer.deterministic=true"], cwd=str(ROOT), env=env, capture_output=True,
                           text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        weights.append(torch.load(next((tmp_path / tag).rglob("weights.pt"))))
    assert weights[0].keys() == weights[1].keys()
    assert all(torch.equal(weights[0][k], weights[1][k]) for k in weights[0])


# ----------------------------------------------------------------------------------------------- refusals (GPU)
@gpu
@pytest.mark.parametrize("switch", ["CVIT_TRAIN_FUSE_DGRAD_GELU=1", "CVIT_WGRAD_TC8=0", "CVIT_WGRAD_TCN=0"])
def test_deterministic_trainer_refuses_atomic_switches(cuda_lib, monkeypatch, switch):
    from cryovit_b200._lib import CryovitB200Error
    from cryovit_b200.train import CryoVITHeadTrainerB200

    k, v = switch.split("=")
    monkeypatch.setenv(k, v)
    with pytest.raises(CryovitB200Error, match=k):
        CryoVITHeadTrainerB200(384, deterministic=True)
    CryoVITHeadTrainerB200(384)  # the default mode keeps the switch
