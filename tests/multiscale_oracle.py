"""CPU oracle of multi-scale inference (pylc_multiscale_combine).

Two statements of the same quantity.  (a) is the definition in float64: every member's probability plane is
sampled onto the output grid with cv2.resize(INTER_NEAREST), the members are averaged, the label is the first
argmax and the confidence round(255 * mean[label]).  (b) restates the kernel's f32 operation order -- the sum in
scale order, times f32(1/K), first argmax, rint(x * 255) clipped to 255 -- and must match the kernel bit for
bit.  Both sample with OpenCV itself, independently of the package's index maps."""
import cv2
import numpy as np


def sample_nearest(plane, w_full, h_full):
    """cv2.resize(plane, (w_full, h_full), INTER_NEAREST) of a [C, h, w] map, class by class (an exact copy of
    source values, so the dtype is kept)."""
    return np.stack([cv2.resize(np.ascontiguousarray(p), (w_full, h_full), interpolation=cv2.INTER_NEAREST) for p in plane])


def combine_f64(probs, w_full, h_full):
    """(a) (mean [C, H, W] f64, labels [H, W] u8, confidence [H, W] u8)."""
    mean = sum(sample_nearest(np.asarray(p, dtype=np.float64), w_full, h_full) for p in probs) / len(probs)
    labels = np.argmax(mean, axis=0)
    p = np.take_along_axis(mean, labels[None], axis=0)[0]
    return mean, labels.astype(np.uint8), np.minimum(255, np.rint(p * 255.0)).astype(np.uint8)


def combine_f32(probs, w_full, h_full):
    """(b) (mean [C, H, W] f32, labels [H, W] u8, confidence [H, W] u8) in the kernel's f32 operation order."""
    s = sample_nearest(np.asarray(probs[0], dtype=np.float32), w_full, h_full)
    for p in probs[1:]:
        s = s + sample_nearest(np.asarray(p, dtype=np.float32), w_full, h_full)
    mean = s * np.float32(1.0 / len(probs))
    labels = np.argmax(mean, axis=0)
    p = np.take_along_axis(mean, labels[None], axis=0)[0]
    q = np.minimum(np.float32(255), np.rint(p * np.float32(255)))
    return mean, labels.astype(np.uint8), q.astype(np.uint8)
