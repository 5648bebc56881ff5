"""
Host-side mirror of PyLC's utils/tools.py for the tiled-segmentation path: same function names,
argument meaning, return types and error behaviour (print + exit(1) / assert), with every
per-pixel body replaced by an sm_100a kernel call through the C ABI (pylc_b200.ops).

    get_image / adjust_to_tile   host (OpenCV decode + INTER_AREA fit), reference tools.py:77-206
    class_encode                 pylc_class_encode,            reference tools.py:412-449
    colourize                    pylc_colourise_u8,            reference tools.py:322-358
    reconstruct                  pylc_stitch_probs +
                                 pylc_resample_encode_confusion, reference tools.py:209-319
    coshuffle / collate / load_files / mk_path / confirm_write_file   host, unchanged semantics

There is no CPU path for the kernels: without a CUDA device these functions raise PylcError.
"""
import collections
import itertools
import os
from concurrent.futures import ThreadPoolExecutor
from math import ceil

import cv2
import numpy as np
import torch

from .. import ops
from .._lib import PylcError
from ..config import defaults


def _device():
    if not torch.cuda.is_available():
        raise PylcError("pylc_b200 needs a CUDA device (B200); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def decode_threads():
    """Host threads used to decode image files ahead of the GPU (`PYLC_DECODE_THREADS`; 0 or 1 = decode in the
    calling thread, as the reference does).  OpenCV's decoders release the GIL, so files decode in parallel."""
    env = os.environ.get("PYLC_DECODE_THREADS")
    if env is not None:
        return max(0, int(env))
    return min(8, os.cpu_count() or 1)


def ordered_prefetch(fn, items, workers=None, depth=None):
    """Generator over fn(item) for every item IN ORDER, with up to `depth` results computed ahead on `workers`
    host threads -- the file loop of Extractor.extract / test.py (reference extract.py:132-150, test.py:52-61)
    decodes file k+1.. while file k is on the GPU.  An exception (or the reference's exit(1)) raised by fn
    surfaces in the caller at that item's position; workers <= 1 degenerates to a plain sequential loop."""
    items = list(items)
    workers = decode_threads() if workers is None else int(workers)
    if workers <= 1 or len(items) <= 1:
        for it in items:
            yield fn(it)
        return
    depth = max(1, int(depth) if depth else workers + 2)
    todo = iter(items)
    with ThreadPoolExecutor(max_workers=workers, thread_name_prefix="pylc-decode") as pool:
        ahead = collections.deque(pool.submit(fn, it) for it in itertools.islice(todo, depth))
        try:
            while ahead:
                res = ahead.popleft().result()
                for it in itertools.islice(todo, 1):
                    ahead.append(pool.submit(fn, it))
                yield res
        finally:
            for fut in ahead:
                fut.cancel()


def rgb2hex(color):
    """[R, G, B] -> '#rrggbb' (reference tools.py:24-39)."""
    return "#{:02x}{:02x}{:02x}".format(int(color[0]), int(color[1]), int(color[2]))


def grayscale(img):
    """[H,W,3] -> channel mean [H,W]; other channel counts are reported and left alone (reference tools.py:59-74)."""
    if img.shape[2] == 3:
        return np.mean(img, axis=2)
    print("Grayscaling skipped: Image is already single-channel." if img.shape[2] == 1
          else "Grayscaling stopped: Image channel is invalid.")


def map_palette(img_array, key):
    """Re-map class indices through `key` (new value per old index), reference tools.py:388-409."""
    index = np.digitize(img_array.numpy().ravel(), range(len(key)), right=True)
    return torch.tensor(np.asarray(key)[index].reshape(img_array.shape))


def add_noise(img, w, h):
    """Gaussian noise (variance 10) added to every channel, min-max normalised back to u8 (reference tools.py:496-533)."""
    gaussian = np.random.normal(0, 10 ** 0.5, (w, h))
    if img.ndim == 2:
        noisy = img + gaussian
    else:
        noisy = np.zeros(img.shape, np.float32)
        for k in range(3):
            noisy[:, :, k] = img[:, :, k] + gaussian
    cv2.normalize(noisy, noisy, 0, 255, cv2.NORM_MINMAX, dtype=-1)
    return noisy.astype(np.uint8)


def is_grayscale(img):
    """True when all three channels are identical (reference tools.py:27-43)."""
    if img.ndim < 3 or img.shape[2] == 1:
        return True
    return bool(np.array_equal(img[:, :, 0], img[:, :, 1]) and np.array_equal(img[:, :, 1], img[:, :, 2]))


def get_image(img_path, ch=3, scale=None, tile_size=None, interpolate=cv2.INTER_AREA):
    """Decode an image to u8 [H,W] (ch=1) or RGB [H,W,3] (ch=3), optionally rescaled
    (reference tools.py:77-148).  Returns (img, w, h, w_resized, h_resized).
    Unlike the reference a colour image given with ch=1 is not prompted about: it is decoded with
    IMREAD_GRAYSCALE exactly as the reference does after the prompt."""
    assert ch == 3 or ch == 1, 'Invalid number of input channels:\t{}.'.format(ch)
    assert os.path.exists(img_path), 'Image path {} does not exist.'.format(img_path)
    if not tile_size:
        tile_size = defaults.tile_size
    if ch == 3:
        img = cv2.imread(img_path, cv2.IMREAD_COLOR)
        if is_grayscale(img):
            print('\nInput image is grayscale but process expects colour (RGB).\n\tApplication stopped.')
            exit(1)
        img = cv2.cvtColor(img, cv2.COLOR_BGR2RGB)
    else:
        img = cv2.imread(img_path, cv2.IMREAD_GRAYSCALE)
    height, width = img.shape[:2]
    height_resized, width_resized = height, width
    if scale:
        min_dim = min(height, width)
        if min_dim < tile_size:
            scale = tile_size / min_dim
        dim = (int(scale * width), int(scale * height))
        img = cv2.resize(img, dim, interpolation=interpolate)
        height_resized, width_resized = img.shape[:2]
    return img, width, height, width_resized, height_resized


def fit_dims(w, h, tile_size):
    """Target size of adjust_to_tile (reference tools.py:178-192)."""
    aspect = w / h
    w_fit = (w // tile_size) * tile_size
    h_fit = (ceil(w_fit / aspect) // tile_size) * tile_size
    return w_fit, h_fit


def adjust_to_tile(img, tile_size, stride, ch, interpolate=cv2.INTER_AREA):
    """Resize an image to a whole number of tiles (reference tools.py:151-206).  Stays on the host:
    the same OpenCV call gives the same bytes.  Returns (img, w_fitted, h_fitted, offset)."""
    h, w = img.shape[:2]
    assert tile_size % stride == 0 and stride <= tile_size, "Tile size must be multiple of stride."
    w_fit, h_fit = fit_dims(w, h, tile_size)
    img_resized = cv2.resize(img, (w_fit, h_fit), interpolation=interpolate)
    h_resized = img_resized.shape[0]
    h_crop = h_resized - int(h_resized / tile_size) * tile_size
    img_cropped = img_resized[h_crop:h_resized]
    return img_cropped, img_cropped.shape[1], img_cropped.shape[0], h_crop


def class_encode(img_array, palette):
    """RGB mask [N,3,H,W] u8 -> class indices [N,H,W] u8 (reference tools.py:412-449): unmatched
    colours become class 1, later palette duplicates win.  CUDA tensors stay on the device; CPU
    tensors / arrays are uploaded and the result is returned on the CPU like the reference's."""
    assert img_array.shape[1] == 3, "Input data must be 3 channel (RGB)"
    on_host = not (torch.is_tensor(img_array) and img_array.is_cuda)
    t = torch.as_tensor(img_array)
    if t.dtype != torch.uint8:
        t = t.to(torch.uint8)
    if on_host:
        t = t.contiguous().pin_memory().to(_device(), non_blocking=True)
    try:
        out = ops.class_encode_nchw(t, palette)
    except PylcError as inst:
        print(inst)
        print('Mask cannot be encoded by selected palette. Please check schema settings.')
        exit(1)
    return out.cpu() if on_host else out


def colourize_lut(n_classes, palette):
    """Final colour of each label under the reference's sequential in-place passes
    (tools.py:352-356): label i takes palette[i]; a grey palette colour [k,k,k] with i < k < C is
    re-mapped by pass k.  For both shipped schemas this is the palette itself."""
    lut = []
    for i in range(n_classes):
        cur = [int(v) for v in palette[i]]
        for j in range(i + 1, n_classes):
            if cur == [j, j, j]:
                cur = [int(v) for v in palette[j]]
        lut.append(cur)
    return lut


def colourize(img, n_classes, palette=None):
    """Label map [n,h,w] -> RGB [n,h,w,3] (reference tools.py:322-358).  Returns the reference's
    dtype (int64 ndarray) for host input, a u8 CUDA tensor for CUDA input."""
    palette = palette if palette is not None else defaults.palette_rgb
    lut = colourize_lut(n_classes, palette)
    on_host = not (torch.is_tensor(img) and img.is_cuda)
    t = torch.as_tensor(np.ascontiguousarray(img) if on_host else img)
    if on_host:
        if t.numel() and (int(t.min()) < 0 or int(t.max()) >= n_classes):
            raise PylcError("colourize: label outside [0, n_classes)")
        t = t.to(torch.uint8).pin_memory().to(_device(), non_blocking=True)
    elif t.dtype != torch.uint8:
        t = t.to(torch.uint8)
    rgb = ops.colourise_u8(t, lut)
    return rgb.cpu().numpy().astype(np.int64) if on_host else rgb


def stitch_geometry(meta):
    """(nr, nc, T, S, h, w, w_full, h_full) for reconstruct, from meta.extract (tools.py:224-236)."""
    ex = meta.extract
    T, S = meta.tile_size, meta.stride
    w, h = ex['w_fitted'], ex['h_fitted']
    nc = w // S - 1 if S < T else w // S
    nr = h // S - 1 if S < T else h // S
    return nr, nc, T, S, h, w, ex['w_scaled'], ex['h_scaled']


def reconstruct_device(logits, meta, want_rgb=True, want_labels=True):
    """Device half of reconstruct: fused stitch + softmax + argmax (+ colourise) at fitted
    resolution, then nearest-neighbour resample to (w_scaled, h_scaled).  Returns a dict of CUDA
    tensors: labels [h,w] u8, pred_full [h_full,w_full] u8, pred_rgb [h_full,w_full,3] u8."""
    nr, nc, T, S, h, w, w_full, h_full = stitch_geometry(meta)
    if meta.extract.get('offset', 0):
        raise PylcError("non-zero crop offset is outside the reference's contract (always 0)")
    if isinstance(logits, (list, tuple)):
        logits = [t if t.is_cuda else t.to(_device(), non_blocking=True) for t in logits]
        if len(logits) == 1:
            logits = logits[0]
    elif not logits.is_cuda:
        logits = logits.to(_device(), non_blocking=True)
    lut = colourize_lut(meta.n_classes, meta.palette_rgb)
    labels, _, _ = ops.stitch_argmax_colour(logits, nr, nc, T, S)
    res = ops.resample_encode_confusion(labels, w_full, h_full, lut_rgb=lut, n_classes=meta.n_classes,
                                        want_pred=want_labels, want_rgb=want_rgb)
    res["labels"] = labels
    return res


def reconstruct(logits, meta):
    """Tile logits (list of [b,C,T,T] f32 batches) -> full-sized RGB mask, np.float32
    [h_scaled, w_scaled, 3] (reference tools.py:209-319), with the reference's band semantics
    (SURVEY.md A.3).  Logits never leave the device; only the RGB mask is copied back."""
    res = reconstruct_device(logits, meta, want_rgb=True, want_labels=False)
    return res["pred_rgb"].cpu().numpy().astype(np.float32)


def coshuffle(img_array, mask_array, permutation=None):
    """Shuffle images and masks with one permutation (reference tools.py:361-385).  `permutation`
    (extension) injects the index order for reproducible parity tests."""
    idx_arr = np.arange(len(img_array)) if permutation is None else np.asarray(permutation)
    if permutation is None:
        np.random.shuffle(idx_arr)
    if torch.is_tensor(img_array):
        idx = torch.as_tensor(idx_arr, device=img_array.device)
        return img_array[idx], mask_array[idx.to(mask_array.device)]
    return img_array[idx_arr], mask_array[idx_arr]


def load_files(path, exts):
    """File path(s) with the given extension(s) (reference tools.py:597-626)."""
    if not os.path.exists(path):
        print('File not found:\n\t{} .'.format(path))
        exit(1)
    files = []
    if os.path.isfile(path):
        ext = os.path.splitext(os.path.basename(path))[1]
        assert ext in exts, "File {} of type {} is invalid.".format(path, ext)
        files.append(path)
    elif os.path.isdir(path):
        files.extend(sorted(os.path.join(path, f) for f in os.listdir(path) if any(ext in f for ext in exts)))
    return files


def collate(img_dir, mask_dir=None):
    """Match image / mask files by base name (reference tools.py:629-680)."""
    img_files = load_files(img_dir, ['.tif', '.tiff', '.jpg', '.jpeg'])
    if not mask_dir:
        return img_files
    img_paths = {os.path.splitext(os.path.basename(f))[0]: f for f in img_files}
    mask_files = load_files(mask_dir, ['.png'])
    mask_paths = {os.path.splitext(os.path.basename(f))[0]: f for f in mask_files}
    files = []
    for name, img_path in img_paths.items():
        if name not in mask_paths:
            print('\nMask not found for image {}.'.format(name))
            exit(1)
        files.append({'img': img_path, 'mask': mask_paths.pop(name)})
    if mask_paths:
        print('\nImage not found for mask(s):\n\t{}.'.format("\n\t".join(mask_paths.values())))
        exit(1)
    return files


def get_fname(path):
    if os.path.isfile(path):
        return os.path.splitext(os.path.basename(path))[0]
    return path


def mk_path(path, check=True):
    """Create a directory if missing (reference tools.py:697-723)."""
    if os.path.exists(path):
        return path
    if check or input("\nRequested directory does not exist:\n\t{}"
                      "\n\nCreate?  (Enter 'Y' or 'y' for yes): ".format(path)) in ['Y', 'y']:
        os.makedirs(path, exist_ok=True)
        print('\nDirectory created:\n\t{}.'.format(path))
        return path
    print('Application stopped.')
    exit(0)


def confirm_write_file(file_path):
    """Ask before overwriting (reference tools.py:726-743)."""
    return True if not os.path.exists(file_path) or \
        input("\nFile {} exists.\n\tOverwrite?  (Enter 'Y' or 'y' for yes): ".format(file_path)) in ['Y', 'y'] \
        else False


# ---- augmentation warps (reference tools.py:452-594) ---------------------------------------------------
# Host OpenCV calls, kept call for call: the same library on the same arguments gives the same bytes as the
# reference (random_state drives both the corner jitter and the brightness shift).  Outside the accelerated
# path (SURVEY.md 8f-3): a tile is 256 KB and the reference applies at most four warps per tile.

def channel_shift(img, random_state):
    """Random brightness: + int(U(10, 20)), clipped to u8 (reference tools.py:528-553)."""
    shift_val = int(random_state.uniform(10, 20))
    return np.uint8(np.clip(np.int16(img) + shift_val, 0, 255))


def perspective_shift(img, mask, random_state):
    """Random perspective jitter of four fixed control points, reflect-101 border, 30-px crop and resize
    back to the tile size; masks use nearest-neighbour throughout (reference tools.py:556-594)."""
    w = mask.shape[0]
    h = mask.shape[1]
    alpha = 0.06 * w
    pts1 = np.float32([[56, 65], [368, 52], [28, 387], [389, 390]])
    pts2 = pts1 + random_state.uniform(-alpha, alpha, size=pts1.shape).astype(np.float32)
    m_trans = cv2.getPerspectiveTransform(pts1, pts2)
    img = cv2.warpPerspective(img, m_trans, (w, h), flags=cv2.INTER_AREA, borderMode=cv2.BORDER_REFLECT_101)
    mask = cv2.warpPerspective(mask, m_trans, (w, h), flags=cv2.INTER_NEAREST, borderMode=cv2.BORDER_REFLECT_101)
    img = img[30:w - 30, 30:h - 30]
    img = cv2.resize(img.astype('float32'), (w, h), interpolation=cv2.INTER_AREA)
    mask = mask[30:w - 30, 30:h - 30]
    mask = cv2.resize(mask.astype('float32'), (w, h), interpolation=cv2.INTER_NEAREST)
    return img, mask


def augment_params(random_state, w):
    """The random draws of perspective_shift + channel_shift in the reference's order (tools.py:577-580, 550) without
    touching pixels: (INVERSE perspective matrix 3x3 f64 = cv2.invert(cv2.getPerspectiveTransform(pts1, pts2)), which is
    what cv2.warpPerspective applies; brightness shift int) -- the job record of pylc_augment_tiles_u8."""
    pts1 = np.float32([[56, 65], [368, 52], [28, 387], [389, 390]])
    pts2 = pts1 + random_state.uniform(-0.06 * w, 0.06 * w, size=pts1.shape).astype(np.float32)
    m_inv = cv2.invert(cv2.getPerspectiveTransform(pts1, pts2))[1]
    return m_inv, int(random_state.uniform(10, 20))


def augment_transform(img, mask, random_state=None):
    """img [1,ch,T,T], mask [1,T,T] -> (img [ch,T,T] or [T,T], mask [T,T]), perspective shift then brightness
    shift (reference tools.py:452-492)."""
    assert img.shape[2:] == mask.shape[1:], \
        "Image dimensions {} must match mask shape {}.".format(img.shape, mask.shape[:2])
    if random_state is None:
        random_state = np.random.RandomState(None)
    nch = img.shape[1]
    img = np.squeeze(np.moveaxis(img, 1, -1), axis=0)
    mask = np.squeeze(mask, axis=0)
    img, mask = perspective_shift(img, mask, random_state)
    img = channel_shift(img, random_state)
    if nch == 3:
        img = np.moveaxis(img, -1, 0)
    return img, mask
