"""Raw-tile input: the reference's input pipeline fused into the patch-embedding and decoder kernels (SURVEY.md 8(f) rank 2).

The reference standardises every band on the host in float64, converts to fp32, (EnMAP) clips, (Houston) zero-pads 48 -> 50
bands, and per training step crops one image_size window out of the 64x64 tile for the whole batch
(src/data_enmap.py:241-249,303-304,454-457,517-522; src/data_houston2018.py:257-274,442-445; pretrain.py:99-107) -- so a
fp32 cube per sample crosses PCIe and HBM.  Here the tiles stay in their sensor dtype (int16) on the device and
`model(RawTiles(...))` makes the kernels read pixels through that pipeline on the fly (csrc/pixel_source.cuh): same values, bit for
bit, no fp32 cube in memory.
"""
import ctypes as C

import torch

from . import _lib

_DT = {torch.int16: _lib.RAW_I16, torch.uint16: _lib.RAW_U16, torch.float32: _lib.RAW_F32}


class RawTiles:
    """tiles [B, raw_bands, tile_h, tile_w] (CUDA; int16 / uint16 / float32) + per-band means / stds (the `.means` / `.stds` of the
    reference's StandardizeEnMAP / StandardizeHouston2018) + the crop window.  Quacks like the [B, bands, H, W] cube where the
    modules only need its shape / device."""

    def __init__(self, tiles, means, stds, *, image_size, crop=(0, 0), pad_bands=0, clip=None, windows=(1, 1), stride=None,
                 window_range=None):
        """windows=(rows, cols): that grid of image_size windows per tile, taken as consecutive samples (tile-major, row-major).
        stride=(sy, sx) (or one int): window step in pixels, 1 <= stride <= image_size, default image_size (no overlap); with an
        explicit stride a last window row / column that would cross the tile border is snapped flush with it.
        window_range=(first, count): only global windows [first, first + count) (global index = tile * rows * cols + window),
        so a scene's windows can run in chunks; default all of them."""
        if not tiles.is_cuda:
            raise RuntimeError("maskedsst_b200: RawTiles needs CUDA tiles (there is no CPU path)")
        if tiles.dtype not in _DT or tiles.dim() != 4:
            raise RuntimeError(f"maskedsst_b200: tiles must be a 4-D int16 / uint16 / float32 tensor, got {tiles.dtype} {tuple(tiles.shape)}")
        self.tiles = tiles if tiles.is_contiguous() else tiles.contiguous()
        nb = tiles.shape[1]
        self.means = torch.as_tensor(means, dtype=torch.float64).reshape(-1).to(tiles.device)
        self.stds = torch.as_tensor(stds, dtype=torch.float64).reshape(-1).to(tiles.device)
        if self.means.numel() != nb or self.stds.numel() != nb:
            raise RuntimeError(f"maskedsst_b200: need one mean / std per raw band ({nb}), got {self.means.numel()} / {self.stds.numel()}")
        self.image_size, self.pad_bands, self.clip = int(image_size), int(pad_bands), clip
        self.windows = (int(windows[0]), int(windows[1]))   # (rows, cols) of image_size windows per tile taken as consecutive samples
        if self.windows[0] < 1 or self.windows[1] < 1:
            raise RuntimeError(f"maskedsst_b200: windows {self.windows} must be >= 1")
        self.snap = stride is not None   # explicit stride: the last window row / column may be snapped to the tile border
        sy, sx = (self.image_size, self.image_size) if stride is None else ((stride, stride) if isinstance(stride, int) else stride)
        self.stride = (int(sy), int(sx))
        if not all(1 <= v <= self.image_size for v in self.stride):
            raise RuntimeError(f"maskedsst_b200: stride {self.stride} must be in [1, image_size={self.image_size}]")
        self.crop = (0, 0)
        self.set_crop(*crop)
        self.set_window_range(*(window_range if window_range is not None else (0, self.num_windows)))

    @property
    def num_windows(self):
        """Windows over all tiles (the samples when no window_range is set)."""
        return self.tiles.shape[0] * self.windows[0] * self.windows[1]

    def set_crop(self, y0, x0):
        """Window origin inside the tile, shared by the batch (pretrain.py:99-107 draws it with randint(0, 64 - image_size))."""
        y0, x0 = int(y0), int(x0)
        th, tw = self.tiles.shape[2:]
        s, (wy, wx), (sy, sx) = self.image_size, self.windows, self.stride
        if self.snap:   # only the last row / column may need the snap: ceil((extent - s) / stride) + 1 windows at most
            ok = (0 <= y0 and y0 + s <= th and (wy - 1) * sy < th - y0 - s + sy and
                  0 <= x0 and x0 + s <= tw and (wx - 1) * sx < tw - x0 - s + sx)
        else:
            ok = 0 <= y0 and y0 + wy * s <= th and 0 <= x0 and x0 + wx * s <= tw
        if not ok:
            raise RuntimeError(f"maskedsst_b200: crop ({y0},{x0}) + {self.windows} x {s} (stride {self.stride}) outside the {th}x{tw} tile")
        self.crop = (y0, x0)
        return self

    def set_window_range(self, first, count):
        """Read global windows [first, first + count) only (one chunk of a scene)."""
        first, count = int(first), int(count)
        if not (0 <= first and 1 <= count and first + count <= self.num_windows):
            raise RuntimeError(f"maskedsst_b200: window range ({first}, {count}) outside [0, {self.num_windows})")
        self.window_range = (first, count)
        return self

    @property
    def shape(self):
        return torch.Size((self.window_range[1], self.tiles.shape[1] + self.pad_bands, self.image_size, self.image_size))

    @property
    def device(self):
        return self.tiles.device

    def c_struct(self):
        lo, hi = self.clip if self.clip is not None else (0.0, 0.0)
        _, nb, th, tw = self.tiles.shape
        return _lib.RawInput(self.tiles.data_ptr(), _DT[self.tiles.dtype], nb, th, tw, self.crop[0], self.crop[1],
                             self.means.data_ptr(), self.stds.data_ptr(), int(self.clip is not None), float(lo), float(hi),
                             self.windows[0], self.windows[1], self.stride[0], self.stride[1], self.window_range[0])

    def materialize(self):
        """The fp32 cube the reference would have built (unfused equivalent, torch ops; for callers that need the tensor)."""
        (y0, x0), s, (wy, wx), (sy, sx) = self.crop, self.image_size, self.windows, self.stride
        th, tw = self.tiles.shape[2:]
        dev = self.tiles.device
        g = torch.arange(self.window_range[0], self.window_range[0] + self.window_range[1], device=dev)
        t, w = g // (wy * wx), g % (wy * wx)
        oy = y0 + torch.clamp_max((w // wx) * sy, th - y0 - s)   # the origin rule of csrc/pixel_source.cuh (window_origin)
        ox = x0 + torch.clamp_max((w % wx) * sx, tw - x0 - s)
        r = torch.arange(s, device=dev)
        band = torch.arange(self.tiles.shape[1], device=dev)
        win = self.tiles[t[:, None, None, None], band[None, :, None, None], (oy[:, None] + r)[:, None, :, None],
                         (ox[:, None] + r)[:, None, None, :]]   # [n, raw_bands, s, s]
        win = win.to(torch.int32).to(torch.float64) if win.dtype != torch.float32 else win.to(torch.float64)
        x = ((win - self.means[None, :, None, None]) / self.stds[None, :, None, None]).to(torch.float32)
        if self.clip is not None:
            x = torch.clip(x, min=self.clip[0], max=self.clip[1])
        if self.pad_bands:
            x = torch.nn.functional.pad(x, (0, 0, 0, 0, 0, self.pad_bands), "constant", 0)
        return x.contiguous()


def raw_ptr(struct):
    return C.pointer(struct)
