"""Input side of the drop-in: `load_images` with the reference's signature and results (mapanything/utils/image.py:134-332),
resize / crop / normalise on the GPU.

The reference decodes every file with Pillow, resizes it with PIL.Image.resize (LANCZOS when shrinking, BICUBIC when
enlarging; cropping.py:188-275), centre-crops (cropping.py:385-467) and normalises with torchvision (image.py:291-296),
all on the host.  Here baseline JPEG files are decoded on the GPU (csrc/jpeg.cu, bit for bit Pillow's libjpeg-turbo
decode; only the compressed stream is uploaded) and every other file with Pillow, whose RGB bytes are uploaded; then
two integer kernels (csrc/image.cu) reproduce Pillow's 8-bit resampling bit for bit, fused with the crop and the
normalisation: the returned views hold `img` as a CUDA fp32 (1, 3, H, W) tensor that `MapAnything.infer` consumes without
another host->device copy.  There is no host fallback for the resize.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib, ops
from ._lib import check
from .inference import IMAGE_NORMALIZATION_DICT

try:  # same optional dependency as the reference (image.py:24-32)
    from pillow_heif import register_heif_opener

    register_heif_opener()
    heif_support_enabled = True
except ImportError:
    heif_support_enabled = False

MA_FILTER_LANCZOS, MA_FILTER_BICUBIC = 1, 3

# Fixed aspect-ratio -> (W, H) tables of the released model (image.py:40-65)
RESOLUTION_MAPPINGS = {
    518: {
        1.000: (518, 518), 1.321: (518, 392), 1.542: (518, 336), 1.762: (518, 294), 2.056: (518, 252), 3.083: (518, 168),
        0.757: (392, 518), 0.649: (336, 518), 0.567: (294, 518), 0.486: (252, 518),
    },
    512: {
        1.000: (512, 512), 1.333: (512, 384), 1.524: (512, 336), 1.778: (512, 288), 2.000: (512, 256), 3.200: (512, 160),
        0.750: (384, 512), 0.656: (336, 512), 0.562: (288, 512), 0.500: (256, 512),
    },
}
ASPECT_RATIO_KEYS = {k: sorted(v.keys()) for k, v in RESOLUTION_MAPPINGS.items()}


def find_closest_aspect_ratio(aspect_ratio: float, resolution_set: int) -> Tuple[int, int]:
    """(target_width, target_height) of the table entry whose aspect-ratio key is closest (image.py:74-90)."""
    closest_key = min(ASPECT_RATIO_KEYS[resolution_set], key=lambda x: abs(x - aspect_ratio))
    return RESOLUTION_MAPPINGS[resolution_set][closest_key]


# ------------------------------------------------------------------------------------------------ device resampler
class _AxisTables:
    """Pillow's resampling windows of one axis (in_size -> out_size): host bounds for planning, device copies for the kernels."""

    __slots__ = ("bounds", "d_bounds", "d_coeffs", "d_packed", "out_size")

    def __init__(self, in_size: int, out_size: int, filt: int, device: torch.device):
        lib = _lib.load()
        ks = C.c_int(0)
        check(lib.ma_resample_coeffs(in_size, out_size, filt, C.byref(ks), None, None), "ma_resample_coeffs")
        self.bounds = np.empty((out_size, 2), np.int32)
        coeffs = np.empty((ks.value, out_size), np.int32)
        check(lib.ma_resample_coeffs(in_size, out_size, filt, C.byref(ks), self.bounds.ctypes.data, coeffs.ctypes.data),
              "ma_resample_coeffs")
        packed = np.empty((3, (ks.value + 3) // 4, out_size), np.uint32)   # byte-split coefficients for the dp4a kernel
        check(lib.ma_resample_pack_coeffs(coeffs.ctypes.data, ks.value, out_size, packed.ctypes.data), "ma_resample_pack_coeffs")
        self.d_bounds = torch.from_numpy(self.bounds).to(device)
        self.d_coeffs = torch.from_numpy(coeffs).to(device)
        self.d_packed = torch.from_numpy(packed.view(np.int32)).to(device)
        self.out_size = out_size


_TABLES: Dict[tuple, _AxisTables] = {}


def _tables(in_size: int, out_size: int, filt: int, device: torch.device) -> _AxisTables:
    key = (in_size, out_size, filt, str(device))
    t = _TABLES.get(key)
    if t is None:
        if len(_TABLES) > 64:
            _TABLES.clear()
        t = _TABLES[key] = _AxisTables(in_size, out_size, filt, device)
    return t


def resize_plan(W1: int, H1: int, target: Tuple[int, int]) -> Tuple[int, int, int, int, int]:
    """(resized W, resized H, filter, crop left, crop top) the reference applies to a W1 x H1 image for target (W, H):
    scale so that the resized image contains the crop (cropping.py:236-247), centred crop (cropping.py:440-446)."""
    out_res = np.array(target)
    in_res = np.array((W1, H1))
    scale_final = max(out_res / in_res) + 1e-8
    rw, rh = (int(v) for v in np.floor(in_res * scale_final).astype(int))
    filt = MA_FILTER_LANCZOS if scale_final < 1 else MA_FILTER_BICUBIC
    return rw, rh, filt, (rw - target[0]) // 2, (rh - target[1]) // 2


def resize_crop_normalize(img_u8: torch.Tensor, target: Tuple[int, int], norm_type: Optional[str] = "dinov2",
                          return_u8: bool = False, crop_offset: Optional[Tuple[int, int]] = None):
    """img_u8: CUDA uint8 (H, W, 3) or a batch (n, H, W, 3) of same-size frames, packed RGB -> fp32 (n, 3, th, tw)
    normalised images (n = 1 for a single frame) and / or the uint8 (n, th, tw, 3) images when return_u8, bit-exact with
    PIL resize + crop + torchvision ToTensor/Normalize.  One launch of each of the two kernels for the whole batch.
    crop_offset = (left, top) in the resized image; default: the centred crop of the image-only path."""
    single = img_u8.dim() == 3
    if single:
        img_u8 = img_u8[None]
    if not img_u8.is_cuda or img_u8.dtype != torch.uint8 or img_u8.dim() != 4 or img_u8.shape[3] != 3 or img_u8.stride(3) != 1 \
            or img_u8.stride(2) != 3:
        raise ValueError("resize_crop_normalize expects CUDA uint8 (H, W, 3) / (n, H, W, 3) tensors with packed RGB pixels")
    n, H1, W1, _ = img_u8.shape
    tw, th = int(target[0]), int(target[1])
    rw, rh, filt, left, top = resize_plan(W1, H1, (tw, th))
    if crop_offset is not None:
        left, top = int(crop_offset[0]), int(crop_offset[1])
    if left < 0 or top < 0 or left + tw > rw or top + th > rh:
        raise ValueError(f"crop box ({left}, {top}, {left + tw}, {top + th}) leaves the resized image {rw}x{rh}")
    dev = img_u8.device
    th_, tv_ = _tables(W1, rw, filt, dev), _tables(H1, rh, filt, dev)
    y0 = int(tv_.bounds[top, 0])
    y1 = int(tv_.bounds[top + th - 1, 0] + tv_.bounds[top + th - 1, 1])
    sx0 = int(th_.bounds[left, 0])
    sx1 = int(th_.bounds[left + tw - 1, 0] + th_.bounds[left + tw - 1, 1])
    lib = _lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    tmp = torch.empty(n, y1 - y0, tw, 3, device=dev, dtype=torch.uint8)
    check(lib.ma_resample_h_u8rgb(img_u8.data_ptr(), img_u8.stride(1), img_u8.stride(0), n, y0, y1 - y0, sx0, sx1,
                                  th_.d_bounds.data_ptr(), th_.d_coeffs.data_ptr(), th_.d_packed.data_ptr(),
                                  th_.d_coeffs.shape[0], rw, left, tw,
                                  tmp.data_ptr(), stream),
          "ma_resample_h_u8rgb")
    out = out8 = None
    m3 = s3 = None
    if norm_type is not None:
        if norm_type not in IMAGE_NORMALIZATION_DICT:
            raise ValueError(
                f"Unknown image normalization type: {norm_type}. Available options: {list(IMAGE_NORMALIZATION_DICT.keys())}"
            )
        mean, std = IMAGE_NORMALIZATION_DICT[norm_type]
        m3, s3 = (C.c_float * 3)(*mean), (C.c_float * 3)(*std)
        out = torch.empty(n, 3, th, tw, device=dev, dtype=torch.float32)
    if return_u8 or out is None:
        out8 = torch.empty(n, th, tw, 3, device=dev, dtype=torch.uint8)
    check(lib.ma_resample_v_norm_u8rgb(tmp.data_ptr(), n, y1 - y0, tw, y0, tv_.d_bounds.data_ptr(), tv_.d_coeffs.data_ptr(),
                                       tv_.d_coeffs.shape[0], rh, top, th, m3, s3, None if out is None else out.data_ptr(),
                                       None if out8 is None else out8.data_ptr(), stream), "ma_resample_v_norm_u8rgb")
    ops._count(2)
    if single and out8 is not None:
        out8 = out8[0]
    if out is None:
        return out8
    return (out, out8) if return_u8 else out


class _Uploader:
    """Host -> device copies of decoded frames through two reusable pinned staging buffers."""

    def __init__(self, device: torch.device):
        self.device = device
        self.bufs: List[Optional[torch.Tensor]] = [None, None]
        self.events: List[Optional[torch.cuda.Event]] = [None, None]
        self.i = 0

    def upload(self, arr: np.ndarray, dst: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Copies `arr` into `dst` (a contiguous CUDA uint8 tensor of the same size) or into a new device tensor."""
        arr = np.ascontiguousarray(arr)
        n = arr.size
        j = self.i
        self.i ^= 1
        if self.events[j] is not None:
            self.events[j].synchronize()  # the previous copy out of this staging buffer has completed
        if self.bufs[j] is None or self.bufs[j].numel() < n:
            self.bufs[j] = torch.empty(max(n, 1 << 20), dtype=torch.uint8, pin_memory=True)
        self.bufs[j][:n].numpy()[...] = arr.reshape(-1)
        if dst is None:
            dst = torch.empty(arr.shape, dtype=torch.uint8, device=self.device)
        dst.view(-1).copy_(self.bufs[j][:n], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self.events[j] = ev
        return dst


def jpeg_parse(data: bytes, with_blob: bool = True):
    """ma_jpeg_parse: (JpegInfo, uint8 blob or None), or None when the file is not a baseline frame the GPU decodes."""
    lib = _lib.load()
    info = _lib.JpegInfo()
    buf = np.frombuffer(data, np.uint8)
    if not with_blob:
        return (info, None) if lib.ma_jpeg_parse(buf.ctypes.data, buf.size, C.byref(info), None, 0) == _lib.MA_OK else None
    # one pass over the file: a blob of this capacity takes the unstuffed data directly (the tables after it are about a
    # tenth of it; a file with more, e.g. a restart marker every few bytes, is parsed again into a blob of the exact size)
    blob = np.empty(buf.size + buf.size // 2 + (1 << 16), np.uint8)
    info.blob_bytes = 0
    if lib.ma_jpeg_parse(buf.ctypes.data, buf.size, C.byref(info), blob.ctypes.data, blob.size) != _lib.MA_OK:
        if info.blob_bytes <= blob.size:
            return None
        blob = np.empty(info.blob_bytes, np.uint8)
        check(lib.ma_jpeg_parse(buf.ctypes.data, buf.size, C.byref(info), blob.ctypes.data, blob.size), "ma_jpeg_parse")
    return info, blob[:info.blob_bytes]


class _JpegBatch:
    """Frames waiting for one ma_jpeg_decode call: their blobs, infos, output slots and EXIF orientations.  The batch is
    decoded when its device workspace would pass `budget` bytes (coefficients + sample planes: ~130 B per pixel of a
    4:4:4 frame), so the memory it takes stays bounded like the slabs'."""

    def __init__(self, up: "_Uploader", budget: int = 1 << 30):
        self.up, self.budget = up, budget
        self.items: list = []   # (blob, info, out tensor, orientation, payload)
        self.ws_bytes = 0

    @staticmethod
    def _ws(info) -> int:
        return 128 * info.nblocks + info.plane_bytes + 32 * info.nsubseq

    def add(self, blob, info, out: torch.Tensor, orientation: int, payload) -> list:
        """Queues a frame; decodes the pending ones first when it would pass the budget (returns flush()'s list)."""
        failed = self.flush() if self.items and self.ws_bytes + self._ws(info) > self.budget else []
        self.items.append((blob, info, out, orientation, payload))
        self.ws_bytes += self._ws(info)
        return failed

    def flush(self) -> list:
        """Decodes the pending frames; returns the payloads of frames the decoder reported (to be decoded by Pillow)."""
        if not self.items:
            return []
        items, self.items, self.ws_bytes = self.items, [], 0
        n = len(items)
        offs = np.cumsum([0] + [b.size for b, *_ in items])
        cat = np.empty(int(offs[-1]), np.uint8)
        for (b, *_), o in zip(items, offs):
            cat[o:o + b.size] = b
        d_blobs = self.up.upload(cat)
        infos = (_lib.JpegInfo * n)(*[it[1] for it in items])
        offsets = (C.c_int64 * n)(*[int(o) for o in offs[:-1]])
        outs = (C.c_void_p * n)(*[it[2].data_ptr() for it in items])
        orient = (C.c_int32 * n)(*[it[3] for it in items])
        lib = _lib.load()
        ws_bytes = C.c_int64(0)
        check(lib.ma_jpeg_workspace(infos, n, C.byref(ws_bytes)), "ma_jpeg_workspace")
        ws = torch.empty(ws_bytes.value, dtype=torch.uint8, device=self.up.device)
        status = torch.empty(n, dtype=torch.int32, device=self.up.device)
        check(lib.ma_jpeg_decode(d_blobs.data_ptr(), offsets, infos, n, outs, orient, ws.data_ptr(), ws_bytes.value,
                                 status.data_ptr(), torch.cuda.current_stream().cuda_stream), "ma_jpeg_decode")
        ops._count(30)
        st = status.cpu().numpy()
        ops.JPEG_ROUTES["gpu"] += int((st == 0).sum())
        return [it[4] for it, s in zip(items, st) if s != 0]


def _open_for_gpu(path: str):
    """(blob, info, orientation) when the file goes to the GPU decoder: Pillow's header-only open reports a JPEG in mode
    RGB or L, and ma_jpeg_parse accepts it (baseline sequential Huffman, 8-bit, grayscale or YCbCr 4:4:4 / 4:2:2 /
    4:2:0 / 4:4:0).  The EXIF orientation is read through Pillow (getexif, with its XMP fallback) like exif_transpose."""
    import PIL.Image

    try:
        with PIL.Image.open(path) as im:
            if im.format != "JPEG" or im.mode not in ("RGB", "L"):
                return None
            orientation = im.getexif().get(0x0112, 1)
    except Exception:  # noqa: BLE001  (Pillow's own route reports the error)
        return None
    with open(path, "rb") as fh:
        data = fh.read()
    parsed = jpeg_parse(data)
    if parsed is None:
        return None
    info, blob = parsed
    return blob, info, orientation if orientation in (2, 3, 4, 5, 6, 7, 8) else 1


_RESIZE_MODES = ["fixed_mapping", "longest_side", "square", "fixed_size"]


def _check_resize_args(resize_mode, size) -> None:
    """Argument checks shared by load_images and preprocess_inputs; messages as in the reference (image.py:165-188, :371-394)."""
    if resize_mode not in _RESIZE_MODES:
        raise ValueError(f"Resize_mode must be one of {_RESIZE_MODES}, got '{resize_mode}'")
    needs_int, needs_pair = resize_mode in ("longest_side", "square"), resize_mode == "fixed_size"
    if (needs_int or needs_pair) and size is None:
        raise ValueError(f"Size parameter is required for resize_mode='{resize_mode}'")
    if needs_int and not isinstance(size, int):
        raise ValueError(f"Size must be an int for resize_mode='{resize_mode}', got {type(size)}")
    if needs_pair:
        if not isinstance(size, (tuple, list)) or len(size) != 2:
            raise ValueError(f"Size must be a tuple/list of (width, height) for resize_mode='fixed_size', got {size}")
        if not all(isinstance(x, int) for x in size):
            raise ValueError(f"Size values must be integers for resize_mode='fixed_size', got {size}")


def _target_size(aspect_ratios: Sequence[float], resize_mode: str, size, patch_size: int, resolution_set: int, verbose: bool):
    """One (W, H) for all images from their average aspect ratio (image.py:240-289)."""
    average_aspect_ratio = sum(aspect_ratios) / len(aspect_ratios)
    if verbose:
        print(f"Calculated average aspect ratio: {average_aspect_ratio:.3f} from {len(aspect_ratios)} images")
    if resize_mode == "fixed_mapping":
        return tuple(find_closest_aspect_ratio(average_aspect_ratio, resolution_set))
    if resize_mode == "square":
        side = round((size // patch_size)) * patch_size
        return (side, side)
    if resize_mode == "longest_side":
        if average_aspect_ratio >= 1:  # width is the longest side
            return (size, round((size // patch_size) / average_aspect_ratio) * patch_size)
        return (round((size // patch_size) * average_aspect_ratio) * patch_size, size)
    return ((size[0] // patch_size) * patch_size, (size[1] // patch_size) * patch_size)  # fixed_size


def load_images(
    folder_or_list,
    resize_mode="fixed_mapping",
    size=None,
    norm_type="dinov2",
    patch_size=14,
    verbose=False,
    bayer_format=False,
    resolution_set=518,
    stride=1,
    device=None,
):
    """Same contract as the reference `load_images` (image.py:134-332): a list of view dicts with `img` (1, 3, H, W) fp32,
    `true_shape`, `idx`, `instance`, `data_norm_type`; every image is brought to ONE target size chosen from the average
    aspect ratio.  `img` lives on `device` (default: the current CUDA device)."""
    _check_resize_args(resize_mode, size)

    if isinstance(folder_or_list, str):
        if verbose:
            print(f"Loading images from {folder_or_list}")
        root, folder_content = folder_or_list, sorted(os.listdir(folder_or_list))
    elif isinstance(folder_or_list, list):
        if verbose:
            print(f"Loading a list of {len(folder_or_list)} images")
        root, folder_content = "", folder_or_list
    else:
        raise ValueError(f"Bad {folder_or_list=} ({type(folder_or_list)})")

    if norm_type not in IMAGE_NORMALIZATION_DICT:
        raise ValueError(
            f"Unknown image normalization type: {norm_type}. Available options: {list(IMAGE_NORMALIZATION_DICT.keys())}"
        )
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if dev.type != "cuda":
        raise RuntimeError("mapanything_b200.load_images resizes on the GPU: pass a CUDA device")

    import PIL.Image
    from PIL.ImageOps import exif_transpose

    exts = [".jpg", ".jpeg", ".png"] + ([".heic", ".heif"] if heif_support_enabled else [])
    exts = tuple(exts)
    # first pass: decode baseline JPEGs on the GPU and every other file on the host (Pillow, like the reference), start
    # the uploads, collect aspect ratios
    up = _Uploader(dev)
    jpegs = _JpegBatch(up)
    loaded, aspect_ratios = [], []
    slabs: Dict[Tuple[int, int], List[list]] = {}   # (W, H) -> [[device tensor (cap, H, W, 3), frames used], ...]
    slab_bytes = 256 << 20                          # frames per slab = what fits 256 MB (at least 1, at most 64)

    def slot(W1: int, H1: int, path: str) -> torch.Tensor:
        # frames of one size are uploaded side by side, so the resize runs as one batched launch per slab
        lst = slabs.setdefault((W1, H1), [])
        if not lst or lst[-1][1] == lst[-1][0].shape[0]:
            cap = max(1, min(64, slab_bytes // (H1 * W1 * 3)))
            lst.append([torch.empty(cap, H1, W1, 3, dtype=torch.uint8, device=dev), 0])
        slab = lst[-1]
        loaded.append([path, (W1, H1), len(lst) - 1, slab[1], W1, H1])
        slab[1] += 1
        aspect_ratios.append(W1 / H1)
        return slab[0][slab[1] - 1]

    def pillow_decode(path: str):
        if bayer_format:
            import cv2

            color_bayer = cv2.imread(os.path.join(root, path), cv2.IMREAD_UNCHANGED)
            img = PIL.Image.fromarray(cv2.cvtColor(color_bayer, cv2.COLOR_BAYER_RG2BGR))
            return exif_transpose(img).convert("RGB")
        return exif_transpose(PIL.Image.open(os.path.join(root, path))).convert("RGB")

    def redo_with_pillow(entries: list) -> None:
        # frames the GPU decoder reported: Pillow decodes them into the same slot, or the file is skipped like any
        # other file Pillow cannot read
        for entry in entries:
            path, key, si, fi = entry[:4]
            try:
                up.upload(np.asarray(pillow_decode(path)), slabs[key][si][0][fi])
                ops.JPEG_ROUTES["pillow"] += 1
            except Exception as e:  # noqa: BLE001
                if verbose:
                    print(f"Warning: Could not load {path}: {e}")
                k = next(i for i, x in enumerate(loaded) if x is entry)
                del loaded[k], aspect_ratios[k]

    with torch.cuda.device(dev):
        for i, path in enumerate(folder_content):
            if i % stride != 0 or not path.lower().endswith(exts):
                continue
            gpu = None if bayer_format else _open_for_gpu(os.path.join(root, path))
            if gpu is not None:
                blob, info, orientation = gpu
                W1, H1 = (info.height, info.width) if orientation >= 5 else (info.width, info.height)
                out = slot(W1, H1, path)
                redo_with_pillow(jpegs.add(blob, info, out, orientation, loaded[-1]))
                continue
            try:
                img = pillow_decode(path)
                W1, H1 = img.size
                up.upload(np.asarray(img), slot(W1, H1, path))
                ops.JPEG_ROUTES["pillow"] += 1
            except Exception as e:  # noqa: BLE001  (the reference skips unreadable files the same way)
                if verbose:
                    print(f"Warning: Could not load {path}: {e}")
                continue
        redo_with_pillow(jpegs.flush())
        if not loaded:
            raise ValueError("No valid images found")
        target_size = _target_size(aspect_ratios, resize_mode, size, patch_size, resolution_set, verbose)
        if verbose:
            print(f"Using target resolution {target_size[0]}x{target_size[1]} (W x H) for all images")
        # second pass: resize + crop + normalise on the device, ONE pair of launches per slab of same-size frames
        resized = {key: [resize_crop_normalize(t[:used], target_size, norm_type) for t, used in lst] for key, lst in slabs.items()}
        tensors = [resized[key][si][fi:fi + 1] for _, key, si, fi, _, _ in loaded]
        del slabs
        imgs = []
        for (path, _, _, _, W1, H1), t in zip(loaded, tensors):
            H2, W2 = t.shape[2], t.shape[3]
            if verbose:
                print(f" - Adding {path} with resolution {W1}x{H1} --> {W2}x{H2}")
            imgs.append(dict(img=t, true_shape=np.int32([[H2, W2]]), idx=len(imgs), instance=str(len(imgs)),
                             data_norm_type=[norm_type]))
    if verbose:
        print(f" (Found {len(imgs)} images)")
    return imgs


# ------------------------------------------------------------------------------------------------ preprocess_inputs
def _nearest_indices(src: int, dst: int) -> np.ndarray:
    """Source offsets of cv2.resize(INTER_NEAREST) for one axis (OpenCV resizeNN), the resize the reference applies to
    depth maps (cropping.py:248-255)."""
    inv = 1.0 / (float(dst) / float(src))
    return np.minimum(np.floor(np.arange(dst) * inv).astype(np.int64), src - 1).astype(np.int32)


def _camera_matrix_of_crop(K: np.ndarray, input_resolution, output_resolution, scaling=1, offset_factor=0.5) -> np.ndarray:
    """Intrinsics after scaling by `scaling` and removing `offset_factor` of the margins (cropping.py:278-318); the same
    numpy operations in the same order and dtype as the reference, because the crop box is rounded from its result."""
    margins = np.asarray(input_resolution) * scaling - output_resolution
    assert np.all(margins >= 0.0)
    offset = offset_factor * margins
    out = K.copy()
    out[0, 2] += 0.5   # OpenCV -> COLMAP pixel-centre convention
    out[1, 2] += 0.5
    out[:2, :] *= scaling
    out[:2, 2] -= offset
    out[0, 2] -= 0.5   # and back
    out[1, 2] -= 0.5
    return out


def _image_to_device_u8(img, view_idx: int, dev: torch.device, up: _Uploader) -> torch.Tensor:
    """The image forms preprocess_inputs accepts (image.py:493-521) as a CUDA uint8 (H, W, 3) tensor.  Tensors are converted
    as the reference does, (img * 255).clamp(0, 255).byte() when img.max() <= 1 else img.clamp(0, 255).byte(), evaluated in
    the tensor's own dtype: host tensors with that expression before the upload, CUDA fp32 tensors with ma_f32_to_u8 (the same
    fp32 multiply, clamp and truncation), CUDA uint8 tensors as they are unless they hold only 0s and 1s, and every other
    CUDA dtype with the expression on the device (a fp16 image rounds img * 255 to fp16 and a fp64 image keeps fp64, so an
    fp32 kernel would give other bytes)."""
    import PIL.Image

    if isinstance(img, torch.Tensor):
        if img.ndim != 3 or img.shape[2] != 3:
            raise ValueError(f"Expected tensor shape (H, W, 3) for img in view {view_idx}, got {img.shape}")
        if not img.is_cuda:
            if img.max() <= 1.0:
                return up.upload((img * 255).clamp(0, 255).byte().numpy())
            return up.upload(img.clamp(0, 255).byte().numpy())
        img = img.to(dev)
        in_unit_range = bool(img.max() <= 1.0)
        if img.dtype == torch.uint8:
            return (img * 255 if in_unit_range else img).contiguous()
        if img.dtype != torch.float32:
            return ((img * 255).clamp(0, 255) if in_unit_range else img.clamp(0, 255)).byte().contiguous()
        x = img.contiguous()
        out = torch.empty(x.shape, device=dev, dtype=torch.uint8)
        check(_lib.load().ma_f32_to_u8(x.data_ptr(), x.numel(), 255.0 if in_unit_range else 1.0, out.data_ptr(),
                                       torch.cuda.current_stream().cuda_stream), "ma_f32_to_u8")
        ops._count()
        return out
    if isinstance(img, np.ndarray):
        if img.ndim != 3 or img.shape[2] != 3:
            raise ValueError(f"Expected array shape (H, W, 3) for img in view {view_idx}, got {img.shape}")
        if img.dtype != np.uint8:
            img = (img * 255).clip(0, 255).astype(np.uint8)
        return up.upload(img)
    if isinstance(img, PIL.Image.Image):
        return up.upload(np.asarray(img))
    raise ValueError(f"Unsupported image type in view {view_idx}: {type(img)}")


def _image_hw(img, view_idx: int) -> Tuple[int, int]:
    import PIL.Image

    if isinstance(img, torch.Tensor):
        if img.ndim == 3 and img.shape[2] == 3:
            return img.shape[0], img.shape[1]
        raise ValueError(f"Expected tensor shape (H, W, 3) for img in view {view_idx}, got {img.shape}")
    if isinstance(img, PIL.Image.Image):
        return img.size[1], img.size[0]
    if isinstance(img, np.ndarray):
        if img.ndim == 3 and img.shape[2] == 3:
            return img.shape[0], img.shape[1]
        raise ValueError(f"Expected array shape (H, W, 3) for img in view {view_idx}, got {img.shape}")
    raise ValueError(f"Unsupported image type in view {view_idx}: {type(img)}")


def _to_host_array(data, expected_shape, name: str, view_idx: int) -> np.ndarray:
    if isinstance(data, torch.Tensor):
        data = data.cpu().numpy()
    if not isinstance(data, np.ndarray):
        raise ValueError(f"Expected tensor or array for {name} in view {view_idx}, got {type(data)}")
    if expected_shape is not None and data.shape != expected_shape:
        raise ValueError(f"Expected shape {expected_shape} for {name} in view {view_idx}, got {data.shape}")
    return data


def _resize_crop_depth(depth, H1: int, W1: int, rw: int, rh: int, left: int, top: int, tw: int, th: int, dev) -> torch.Tensor:
    """depth (H1, W1) float -> CUDA fp32 (1, th, tw): nearest resize to (rh, rw) and crop, one gather kernel."""
    if isinstance(depth, torch.Tensor):
        d = depth.to(dev, torch.float32).contiguous()
    else:
        d = torch.from_numpy(np.ascontiguousarray(depth, dtype=np.float32)).to(dev)
    yi = torch.from_numpy(_nearest_indices(H1, rh)[top:top + th].copy()).to(dev)
    xi = torch.from_numpy(_nearest_indices(W1, rw)[left:left + tw].copy()).to(dev)
    out = torch.empty(1, th, tw, device=dev, dtype=torch.float32)
    check(_lib.load().ma_gather_rows_cols_f32(d.data_ptr(), d.stride(0), yi.data_ptr(), xi.data_ptr(), th, tw, out.data_ptr(),
                                              torch.cuda.current_stream().cuda_stream), "ma_gather_rows_cols_f32")
    ops._count()
    return out


def preprocess_inputs(
    input_views,
    resize_mode="fixed_mapping",
    size=None,
    norm_type="dinov2",
    patch_size=14,
    resolution_set=518,
    verbose=False,
    device=None,
):
    """Same contract as the reference `preprocess_inputs` (image.py:335-675): brings the images AND the optional
    multi-modal inputs of every view (intrinsics or ray directions, depth_z, camera poses) to one target resolution.
    Images are resampled like load_images; depth with nearest neighbour; intrinsics follow the scale and a
    principal-point preserving crop (cropping.py:278-318, :362-381).  `img` and `depth_z` are returned on `device`."""
    _check_resize_args(resize_mode, size)
    if not input_views:
        raise ValueError("input_views cannot be empty")

    aspect_ratios = []
    for view_idx, view in enumerate(input_views):
        if "img" not in view:
            if verbose:
                print(f"Warning: View {view_idx} has no 'img' key, skipping for aspect ratio calculation")
            continue
        H, W = _image_hw(view["img"], view_idx)
        aspect_ratios.append(W / H)
    if not aspect_ratios:
        raise ValueError("No valid images found in input_views")
    target_size = _target_size(aspect_ratios, resize_mode, size, patch_size, resolution_set, verbose)
    tw, th = target_size
    if verbose:
        print(f"Using target resolution {target_size[0]}x{target_size[1]} (W x H) for all views")
    if norm_type not in IMAGE_NORMALIZATION_DICT:
        raise ValueError(
            f"Unknown image normalization type: {norm_type}. Available options: {list(IMAGE_NORMALIZATION_DICT.keys())}"
        )
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if dev.type != "cuda":
        raise RuntimeError("mapanything_b200.preprocess_inputs resizes on the GPU: pass a CUDA device")

    up = _Uploader(dev)
    processed_views = []
    with torch.cuda.device(dev):
        for view_idx, view in enumerate(input_views):
            if "img" not in view:
                raise ValueError(f"View {view_idx} missing required 'img' key")
            d_img = _image_to_device_u8(view["img"], view_idx, dev, up)
            H1, W1 = d_img.shape[0], d_img.shape[1]

            depthmap = None
            if "depth_z" in view:
                depthmap = view["depth_z"]
                if depthmap.ndim != 2:
                    raise ValueError(f"Expected shape (H, W) for depth_z in view {view_idx}, got {depthmap.shape}")
                assert tuple(depthmap.shape[:2]) == (H1, W1)
            has_intrinsics, has_ray_directions = "intrinsics" in view, "ray_directions" in view
            if has_intrinsics and has_ray_directions:
                raise ValueError(
                    f"View {view_idx} cannot have both 'intrinsics' and 'ray_directions'. "
                    "Please provide only one as they are redundant (ray_directions can be used to recover intrinsics)."
                )
            intrinsics = None
            if has_intrinsics:
                intrinsics = _to_host_array(view["intrinsics"], (3, 3), "intrinsics", view_idx)
            if has_ray_directions:
                rays = view["ray_directions"]
                if rays.ndim != 3 or rays.shape[2] != 3:
                    raise ValueError(f"Expected shape (H, W, 3) for ray_directions in view {view_idx}, got {rays.shape}")
                from .inference import intrinsics_from_rays

                rays_t = rays if isinstance(rays, torch.Tensor) else torch.from_numpy(rays)
                intrinsics = intrinsics_from_rays(rays_t.to(dev, torch.float32)[None])[0].cpu().numpy()

            # rescale so that the image contains the crop, then crop (cropping.py:236-275, :425-458)
            rw, rh, _, left, top = resize_plan(W1, H1, target_size)
            if intrinsics is not None:
                in_res, res = np.array((W1, H1)), np.array((rw, rh))
                scale_final = max(np.array(target_size) / in_res) + 1e-8
                intrinsics = _camera_matrix_of_crop(intrinsics, in_res, res, scaling=scale_final)
                new_intrinsics = _camera_matrix_of_crop(intrinsics, (rw, rh), target_size, offset_factor=0.5)
                left, top = (int(v) for v in np.int32(np.round(intrinsics[:2, 2] - new_intrinsics[:2, 2])))
                intrinsics = intrinsics.copy()
                intrinsics[0, 2] -= left
                intrinsics[1, 2] -= top

            processed_view = {
                "img": resize_crop_normalize(d_img, target_size, norm_type, crop_offset=(left, top)),
                "data_norm_type": [norm_type],
            }
            if depthmap is not None:
                processed_view["depth_z"] = _resize_crop_depth(depthmap, H1, W1, rw, rh, left, top, tw, th, dev)
            if intrinsics is not None:
                processed_view["intrinsics"] = torch.from_numpy(intrinsics)[None]

            if "camera_poses" in view:
                camera_poses = view["camera_poses"]
                if isinstance(camera_poses, tuple):
                    def batched(c):
                        if isinstance(c, torch.Tensor):
                            return c[None]
                        return torch.from_numpy(c)[None] if isinstance(c, np.ndarray) else torch.tensor(c)[None]

                    quats, trans = camera_poses
                    processed_view["camera_poses"] = (batched(quats), batched(trans))
                elif isinstance(camera_poses, torch.Tensor):
                    processed_view["camera_poses"] = camera_poses[None]
                elif isinstance(camera_poses, np.ndarray):
                    processed_view["camera_poses"] = torch.from_numpy(camera_poses)[None]
                else:
                    raise ValueError(
                        f"Unsupported camera_poses format: {type(camera_poses)}. Expected tuple (quats, trans) or matrix (tensor/array)."
                    )
            for key, value in view.items():
                if key not in ["img", "depth_z", "intrinsics", "ray_directions", "camera_poses"]:
                    processed_view[key] = value
            processed_views.append(processed_view)
            if verbose:
                print(f"Processed view {view_idx} with keys: {list(processed_view.keys())}")
    if verbose:
        print(f"Successfully processed {len(processed_views)} views")
    return processed_views
