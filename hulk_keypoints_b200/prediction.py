"""Prediction -- host-side mirror of reference src/prediction.py:8-66.

`predict` keeps the reference's contract (3-D input gains a batch axis, the model's forward output is
returned on the model's device).  Deliberate, documented deviation (SURVEY.md §0.2): constructing a
Prediction puts the model in eval() mode -- the reference scripts never call .eval(), so as written
they normalise each image with its own batch statistics; the B200 inference path folds the running
statistics instead ("BN folded at inference").  Pass bn_mode="as_written" to keep train-mode BN.

Additive API: `decode(heatmap)` runs the argmax of reference prediction.py:46 on the GPU for EVERY batch
element (the reference's `plot` decodes element 0 only, on the host); `peaks(heatmap)` returns every thresholded local maximum of
each channel, the top N per map.
"""
from __future__ import annotations

import numpy as np
import torch

from . import ops


class Prediction:
    def __init__(self, model, num_keypoints, img_height, img_width, use_cuda, bn_mode: str = "eval"):
        self.model = model
        self.num_keypoints = num_keypoints
        self.img_height = img_height
        self.img_width = img_width
        self.use_cuda = use_cuda
        if bn_mode not in ("eval", "as_written"):
            raise ValueError("bn_mode must be 'eval' or 'as_written'")
        if bn_mode == "eval":
            self.model.eval()

    def predict(self, imgs):
        # imgs: torch.Tensor (3, H, W) or (B, 3, H, W)
        if imgs.dim() == 3:
            imgs = imgs.unsqueeze(0)
        elif imgs.dim() != 4:
            raise ValueError(f"expected a 3-D or 4-D image tensor, got {tuple(imgs.shape)}")
        return self.model.forward(imgs)

    def decode(self, heatmap):
        """(B,K,H,W) heatmap (CUDA tensor or numpy) -> (B,K,2) int64 numpy array of (y, x) peaks."""
        if isinstance(heatmap, np.ndarray):
            heatmap = torch.from_numpy(np.ascontiguousarray(heatmap, dtype=np.float32)).cuda()
        heat = heatmap.detach().float().contiguous()
        return ops.argmax_decode(heat).cpu().numpy().astype(np.int64)

    def peaks(self, heatmap, max_peaks: int = 16, threshold: float = 0.5, min_distance: int = 8):
        """Additive API: every instance per channel of a (B,K,H,W) heatmap (CUDA tensor or numpy) -> numpy (yx int64 (B,K,N,2) as
        (y, x), score float32 (B,K,N), count int64 (B,K)): local maxima >= threshold, at most one per (2r+1)^2 window (r =
        min_distance), the top N = max_peaks per map by score; unused slots (-1, -1) / -inf.  See ops.peak_decode."""
        ops.check_peak_args(max_peaks, threshold, min_distance)
        if isinstance(heatmap, np.ndarray):
            heatmap = torch.from_numpy(np.ascontiguousarray(heatmap, dtype=np.float32)).cuda()
        yx, score, count = ops.peak_decode(heatmap.detach().float().contiguous(), max_peaks, threshold, min_distance)
        return yx.cpu().numpy().astype(np.int64), score.cpu().numpy(), count.cpu().numpy().astype(np.int64)

    # ---- kept callable for API parity; host-side helpers of the reference (prediction.py:26-38) ----
    def softmax(self, x):
        e_x = np.exp(x - np.max(x))
        return e_x / e_x.sum()

    def expectation(self, d):
        """Soft-argmax of one (H, W) map, as written in reference prediction.py:31-38: the map is flattened in the order of
        `d.T.ravel()` while the index arrays assume row-major order (x = i % W, y = i // W), so for H != W rows and columns mix;
        kept as is for result parity (the reference computes it in `plot` and discards it).  Truncated to int.
        A CUDA tensor goes through the hk_soft_argmax reduction kernel (one pass over the map); a numpy array takes the
        reference's own host formula (this method is a host-side helper there)."""
        if isinstance(d, torch.Tensor) and d.is_cuda:
            if d.dim() != 2:
                raise ValueError("expectation takes one (H, W) map; use expectation_batch for (B,K,H,W)")
            exp_xy, exp_int = ops.soft_argmax(d.detach().float().contiguous())
            if bool(torch.isnan(exp_xy).any()):
                raise ValueError("cannot convert float NaN to integer")   # what int(np.dot(...)) raises in the reference
            return [int(v) for v in exp_int.tolist()]
        d = np.asarray(d)
        width, height = d.T.shape
        p = self.softmax(d.T.ravel())
        flat = np.arange(width * height)
        return [int(np.dot(p, flat % width)), int(np.dot(p, flat // width))]

    def expectation_batch(self, heatmap):
        """Additive API: soft-argmax of every map of a (B,K,H,W) CUDA heatmap in one launch pair -> (exp_xy fp64 (B,K,2) = (E[x'], E[y'])
        with the reference's index convention, exp_int int32 (B,K,2) = its int() truncation), both on the GPU."""
        return ops.soft_argmax(heatmap.detach().float().contiguous())

    def plot(self, img, heatmap, image_id=0, cls=None, classes=None):
        """Overlay visualisation (reference prediction.py:40-66): host-side cv2 drawing, out of the hot
        path.  Peaks come from `decode` (GPU) instead of a host argmax."""
        import cv2

        print("Running inferences on image: %d" % image_id)
        heatmap = np.asarray(heatmap)
        peaks = self.decode(heatmap[:1])[0]
        overlays = []
        for i in range(self.num_keypoints):
            h = heatmap[0][i]
            pred_y, pred_x = int(peaks[i][0]), int(peaks[i][1])
            vis = cv2.normalize(h, None, 0, 255, cv2.NORM_MINMAX).astype(np.uint8)
            vis = cv2.applyColorMap(vis, cv2.COLORMAP_JET)
            overlay = cv2.addWeighted(img, 0.65, vis, 0.35, 0)
            overlay = cv2.circle(overlay, (pred_x, pred_y), 4, (0, 0, 0), -1)
            overlays.append(overlay)
        half = self.num_keypoints // 2
        left = cv2.vconcat(overlays[:half]) if half else None
        right = cv2.vconcat(overlays[half:])
        result = cv2.hconcat((left, right)) if left is not None else right
        if cls is not None:
            cv2.putText(result, classes[cls], (10, 55), cv2.FONT_HERSHEY_SIMPLEX, 0.7, (255, 255, 255), 2)
        cv2.imwrite('preds/out%04d.png' % image_id, result)
