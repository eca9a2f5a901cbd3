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
