"""TEST INFRASTRUCTURE: the reference's caller-side sequence around the hot path, restated so that it can run
against the drop-in module without the reference installed.

Each step cites the reference lines it follows; nothing here is imported by the product package.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn as nn


class CallerModel:
    """What `bin_model` does with netG on the inference path, and nothing else:
    __init__      bin_model.py:38-42   netG = define_G(opt).to(device); netG = DataParallel(netG)   (non-dist)
    load          base_model.py:89-103 strict load_state_dict after prefix stripping
    test_set_input bin_model.py:258-267 B1..B11 = testData[k].to(device)                             (nframes == 6)
    test_forward  bin_model.py:379-380 self.Ft_p = self.netG(B1, B3, B5, B7, B9, B11)
    """

    def __init__(self, net: nn.Module, device, device_ids: Optional[Sequence[int]] = None):
        self.device = torch.device(device)
        self.netG = nn.DataParallel(net.to(self.device), device_ids=device_ids)     # bin_model.py:38,42
        self.netG.eval()                                                            # bin_model.py:295 (test())
        self.Ft_p = None

    def load_state_dict_like_load_network(self, sd):                                # base_model.py:89-103
        net = self.netG.module if isinstance(self.netG, nn.DataParallel) else self.netG
        clean = {}
        for k, v in sd.items():
            k = k[len("InterpNet."):] if k.startswith("InterpNet.") else k
            clean[k] = v
        net.load_state_dict(clean, strict=True)

    def test_set_input(self, testData):                                             # bin_model.py:258-267
        B1, B3, B5, B7, B9, B11, _ = testData
        self.B = [t.to(self.device) for t in (B1, B3, B5, B7, B9, B11)]

    def test_forward(self):                                                         # bin_model.py:379-380
        self.Ft_p = self.netG(*self.B)


def pad_like_test_py(frames_chw: Sequence[torch.Tensor]) -> Tuple[List[torch.Tensor], Tuple[int, int, int, int]]:
    """test.py:338-371: per-image (3,H,W) tensors -> replicate-padded (1,3,Hp,Wp); returns (padded, (l, r, t, b))."""
    intWidth, intHeight = frames_chw[0].size(2), frames_chw[0].size(1)
    if intWidth != ((intWidth >> 7) << 7):
        intWidth_pad = (((intWidth >> 7) + 1) << 7)
        pl = int((intWidth_pad - intWidth) / 2)
        pr = intWidth_pad - intWidth - pl
    else:
        pl = pr = 32
    if intHeight != ((intHeight >> 7) << 7):
        intHeight_pad = (((intHeight >> 7) + 1) << 7)
        pt = int((intHeight_pad - intHeight) / 2)
        pb = intHeight_pad - intHeight - pt
    else:
        pt = pb = 32
    pader = torch.nn.ReplicationPad2d([pl, pr, pt, pb])
    return [pader(torch.unsqueeze(u, 0)) for u in frames_chw], (pl, pr, pt, pb)


def tensor2img(t: torch.Tensor) -> np.ndarray:
    """utils/util.py:113-137 for one 3-D image, out_type uint8, min_max (0, 1): HWC BGR."""
    t = t.squeeze().float().cpu().clamp_(0, 1)
    img = np.transpose(t.numpy()[[2, 1, 0], :, :], (1, 2, 0))
    return (img * 255.0).round().astype(np.uint8)


def run_test_py_window(model: CallerModel, frames_chw: Sequence[torch.Tensor]):
    """One iteration of the test.py loop body (test.py:334-402) without the file IO: returns the three cropped
    uint8 HWC BGR images test.py writes (Ft_p[13], [8], [12]) and the raw 14-tuple."""
    H, W = frames_chw[0].size(1), frames_chw[0].size(2)
    dev = model.device
    testData = [f.to(dev) for f in frames_chw]                                       # test.py:334-336
    testData, (pl, pr, pt, pb) = pad_like_test_py(testData)                          # test.py:348-371
    testData.append(torch.unsqueeze(torch.tensor(0), 0))                             # test.py:372
    prev = torch.is_grad_enabled()
    torch.set_grad_enabled(False)                                                    # test.py:368
    try:
        model.test_set_input(testData)                                               # test.py:378
        model.test_forward()                                                         # test.py:379
    finally:
        torch.set_grad_enabled(prev)
    crop = lambda t: tensor2img(t.squeeze(0))[pt:pt + H, pl:pl + W, :]               # test.py:394-398
    return [crop(model.Ft_p[k]) for k in (13, 8, 12)], model.Ft_p, (pl, pr, pt, pb)
