"""Image-quality metrics ``KPlanesModel.get_image_metrics_and_images`` reports (NS/models/kplanes.py:290-295, 454-515).

PSNR and SSIM are restated in torch with torchmetrics' defaults (the reference instantiates
``PeakSignalNoiseRatio(data_range=1.0)`` and ``structural_similarity_index_measure``): evaluation tooling, computed
once per eval image, not part of the hot path.  LPIPS (pretrained AlexNet) and the RetinaNet-based ``DynMetric`` need
downloaded weights; they are used through the reference's own objects when those import, and their keys are simply
absent otherwise -- never an exception in the middle of a training run.
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn.functional as F


def psnr(target: torch.Tensor, preds: torch.Tensor, data_range: float = 1.0) -> torch.Tensor:
    """10 log10(data_range^2 / mse) over the whole tensor (torchmetrics PeakSignalNoiseRatio, base 10, dim None)."""
    mse = torch.mean((preds - target) ** 2)
    return 10.0 * torch.log10(torch.as_tensor(data_range**2, device=mse.device, dtype=mse.dtype) / mse)


def ssim(preds: torch.Tensor, target: torch.Tensor, kernel_size: int = 11, sigma: float = 1.5, k1: float = 0.01,
         k2: float = 0.03, data_range: Optional[float] = None) -> torch.Tensor:
    """torchmetrics.functional.structural_similarity_index_measure defaults: [B,C,H,W] inputs, gaussian 11x11 window with
    sigma 1.5, reflect padding cropped from the result, data_range = max(range(preds), range(target)), mean over batch."""
    full = ssim_map(preds, target, kernel_size, sigma, k1, k2, data_range)
    return full.reshape(full.shape[0], -1).mean(-1).mean()


def ssim_map(preds: torch.Tensor, target: torch.Tensor, kernel_size: int = 11, sigma: float = 1.5, k1: float = 0.01,
             k2: float = 0.03, data_range: Optional[float] = None) -> torch.Tensor:
    """The SSIM map ``ssim`` averages: [B,C,H-10,W-10] for the default window, entry (y, x) = the window centred on
    pixel (y+5, x+5)."""
    if data_range is None:
        data_range = float(max(preds.max() - preds.min(), target.max() - target.min()))
    c1, c2 = (k1 * data_range) ** 2, (k2 * data_range) ** 2
    channels = preds.shape[1]
    dist = torch.arange((1 - kernel_size) / 2, (1 + kernel_size) / 2, 1, dtype=preds.dtype, device=preds.device)
    gauss = torch.exp(-((dist / sigma) ** 2) / 2)
    gauss = (gauss / gauss.sum())[None]
    kernel = (gauss.t() @ gauss).expand(channels, 1, kernel_size, kernel_size)
    pad = (kernel_size - 1) // 2
    preds = F.pad(preds, (pad, pad, pad, pad), mode="reflect")
    target = F.pad(target, (pad, pad, pad, pad), mode="reflect")
    stack = torch.cat((preds, target, preds * preds, target * target, preds * target))
    out = F.conv2d(stack, kernel, groups=channels)
    b = preds.shape[0]
    mu_p, mu_t, pp, tt, pt = (out[i * b:(i + 1) * b] for i in range(5))
    sig_p, sig_t, sig_pt = pp - mu_p**2, tt - mu_t**2, pt - mu_p * mu_t
    full = ((2 * mu_p * mu_t + c1) * (2 * sig_pt + c2)) / ((mu_p**2 + mu_t**2 + c1) * (sig_p + sig_t + c2))
    return full[..., pad:-pad, pad:-pad]


def region_psnr_ssim(pred: torch.Tensor, target: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
    """Per-image PSNR and SSIM of a region and of its complement: pred, target [B,H,W,3] with H, W >= 11, mask [B,H,W]
    (non-zero: the dynamic region) -> [B,4] = (psnr_dynamic, ssim_dynamic, psnr_static, ssim_static) in pred's dtype,
    on pred's device.  The torch statement of ``ops.image_metrics_masked``:

    - PSNR of a region R: 10 log10(1 / mse_R), mse_R the mean squared error over R's pixels and their 3 channels;
    - SSIM of R: the mean of ``ssim_map`` (C1 / C2 from the whole image's data range) over the windows whose centre
      pixel lies in R, all 3 channels;
    - NaN for a region without a pixel, and for the SSIM of a region without a window centre (one that only touches the
      5-pixel border)."""
    if pred.dim() != 4 or pred.shape[-1] != 3 or target.shape != pred.shape or mask.shape != pred.shape[:3]:
        raise ValueError(f"region_psnr_ssim: pred, target [B,H,W,3] and mask [B,H,W] (got {tuple(pred.shape)}, "
                         f"{tuple(target.shape)}, {tuple(mask.shape)})")
    b, h, w = mask.shape
    if h < 11 or w < 11:
        raise ValueError(f"region_psnr_ssim: {h}x{w} images are smaller than the 11x11 SSIM window")
    out = torch.empty((b, 4), dtype=pred.dtype, device=pred.device)
    for k in range(b):
        p4, t4 = torch.moveaxis(pred[k], -1, 0)[None], torch.moveaxis(target[k], -1, 0)[None]
        sq = (pred[k] - target[k]) ** 2
        full = ssim_map(t4, p4)[0]  # the model's argument order, as get_image_metrics_and_images calls ssim
        dyn = mask[k] != 0
        for r, sel in enumerate((dyn, ~dyn)):
            out[k, 2 * r] = 10.0 * torch.log10(1.0 / sq[sel].mean())
            out[k, 2 * r + 1] = full[:, sel[5:h - 5, 5:w - 5]].mean()
    return out


DELTA_THRESHOLDS = (1.25, 1.5625, 1.953125)  # 1.25 ** k, k = 1, 2, 3: exact in binary


def depth_metrics(pred: torch.Tensor, gt: torch.Tensor, directions_norm: Optional[torch.Tensor] = None,
                  mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Per-image depth error of rendered depth against ground truth: pred, gt, directions_norm [B,H,W] or [B,H,W,1], mask
    [B,H,W] (non-zero: the dynamic region) -> float64 [B,R,8] on pred's device, row = (n_valid, abs_rel, sq_rel, rmse,
    rmse_log, delta1, delta2, delta3); R = 1 (whole image) without a mask, 3 (whole, dynamic, static) with one.  The torch
    statement of ``ops.depth_metrics``:

    - ground truth g = gt * directions_norm in the inputs' dtype (z-depth to distance along the unit ray, as
      ``depth_loss`` does for ``is_euclidean_depth=False``), or gt without ``directions_norm``;
    - a pixel is valid where g is finite and > 0 (sky / background: 0 or inf);
    - in float64, p = max(pred, 1e-6), e = p - g over a region's valid pixels: abs_rel = mean |e| / g, sq_rel =
      mean e^2 / g, rmse = sqrt(mean e^2), rmse_log = sqrt(mean (log p - log g)^2), delta_k = the share of
      max(p / g, g / p) < 1.25^k;
    - n_valid = 0 and NaN for the other seven in a region without a valid pixel."""
    pred, gt = (t.squeeze(-1) if t.dim() == 4 and t.shape[-1] == 1 else t for t in (pred, gt))
    if directions_norm is not None and directions_norm.dim() == 4 and directions_norm.shape[-1] == 1:
        directions_norm = directions_norm.squeeze(-1)
    if (pred.dim() != 3 or gt.shape != pred.shape or (directions_norm is not None and directions_norm.shape != pred.shape)
            or (mask is not None and mask.shape != pred.shape)):
        raise ValueError(f"depth_metrics: pred, gt, directions_norm and mask must be [B,H,W] (got {tuple(pred.shape)}, "
                         f"{tuple(gt.shape)}, {None if directions_norm is None else tuple(directions_norm.shape)}, "
                         f"{None if mask is None else tuple(mask.shape)})")
    g = gt if directions_norm is None else gt * directions_norm
    valid = torch.isfinite(g) & (g > 0)
    p, g = pred.double().clamp_min(1e-6), g.double()
    regions = [torch.ones_like(valid)] if mask is None else [torch.ones_like(valid), mask != 0, mask == 0]
    out = torch.full((pred.shape[0], len(regions), 8), float("nan"), dtype=torch.float64, device=pred.device)
    for b in range(pred.shape[0]):
        for r, region in enumerate(regions):
            sel = valid[b] & region[b]
            pp, gg = p[b][sel], g[b][sel]
            out[b, r, 0] = pp.numel()
            if pp.numel() == 0:
                continue
            # means as sum / n, correctly rounded: on CUDA, .mean() and "/ n" with a Python n multiply by 1 / n
            n = torch.tensor(float(pp.numel()), dtype=torch.float64, device=pp.device)
            e = pp - gg
            ratio = torch.maximum(pp / gg, gg / pp)
            out[b, r, 1] = (e.abs() / gg).sum() / n
            out[b, r, 2] = (e * e / gg).sum() / n
            out[b, r, 3] = ((e * e).sum() / n).sqrt()
            out[b, r, 4] = (((pp.log() - gg.log()) ** 2).sum() / n).sqrt()
            for k, t in enumerate(DELTA_THRESHOLDS):
                out[b, r, 5 + k] = (ratio < t).sum(dtype=torch.float64) / n
    return out


def optional_lpips(device):
    """torchmetrics' LearnedPerceptualImagePatchSimilarity if importable AND its weights are available, else None."""
    try:
        from torchmetrics.image.lpip import LearnedPerceptualImagePatchSimilarity

        return LearnedPerceptualImagePatchSimilarity(normalize=True).to(device)
    except Exception:
        return None


def optional_dynmetric(device):
    """The reference's RetinaNet-based dynamic-region metric (NS/utils/dynmetric.py) if nerfstudio is importable."""
    try:
        from nerfstudio.utils.dynmetric import DynMetric

        return DynMetric(device=device)
    except Exception:
        return None
