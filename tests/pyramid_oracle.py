"""numpy restatement of the box-filtered pyramid levels (csrc/pyramid.cu, vqae_b200.pyramid): per channel,
the exact int64 sum S of each f x f block, then (S + f^2 / 2) // f^2 -- the box mean rounded half up."""
import numpy as np


def reduce(img: np.ndarray, f: int) -> np.ndarray:
    """uint8 [H, W, C] (or [H, W]) with f dividing H and W -> uint8 [H/f, W/f, C]."""
    h, w = img.shape[:2]
    assert h % f == 0 and w % f == 0, (img.shape, f)
    s = img.astype(np.int64).reshape(h // f, f, w // f, f, *img.shape[2:]).sum(axis=(1, 3))
    return ((s + f * f // 2) // (f * f)).astype(np.uint8)


def pyramid(canvas: np.ndarray, factors) -> dict:
    """{f: reduce(canvas, f)}; with f dividing the patch size this is the level of a whole canvas."""
    return {int(f): reduce(canvas, int(f)) for f in factors}


def gather_patches(canvas: np.ndarray, h: int, w: int, r0: int, c0: int, rc: int, first: int, n: int) -> np.ndarray:
    """Patches first .. first + n - 1 of the addressing (r0 + q // rc, c0 + q % rc) as [n, h, w, 3]."""
    out = []
    for q in range(first, first + n):
        r, c = r0 + q // rc, c0 + q % rc
        out.append(canvas[r * h:(r + 1) * h, c * w:(c + 1) * w])
    return np.stack(out)
