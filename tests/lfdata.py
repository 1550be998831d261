"""Deterministic synthetic light fields (no file access): a procedural textured base image — a sum of sinusoids
with LCG-drawn frequencies/phases plus LCG-placed constant rectangles for edges — cropped at integer disparities
(1 px per view), as SURVEY.md section 8(d) prescribes. Noise comes from the oracle's mt19937ar restatement."""
import numpy as np


def _lcg(seed):
    state = seed & 0xFFFFFFFF
    while True:
        state = (1664525 * state + 1013904223) & 0xFFFFFFFF
        yield state / 4294967296.0


def base_image(H, W, C=3, seed=12345):
    g = _lcg(seed)
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float64)
    img = np.zeros((C, H, W), np.float64)
    for c in range(C):
        acc = np.zeros((H, W), np.float64)
        for _ in range(24):
            fx, fy = (next(g) - 0.5) * 0.9, (next(g) - 0.5) * 0.9
            ph, amp = next(g) * 6.283185307179586, 0.3 + next(g)
            acc += amp * np.sin(fx * xx + fy * yy + ph)
        img[c] = acc
    for _ in range(max(8, (H * W) // 2000)):
        y0, x0 = int(next(g) * H), int(next(g) * W)
        hh, ww = 4 + int(next(g) * 24), 4 + int(next(g) * 24)
        val = [(next(g) - 0.5) * 6 for _ in range(C)]
        for c in range(C):
            img[c, y0:y0 + hh, x0:x0 + ww] += val[c]
    img -= img.min()
    img *= 255.0 / img.max()
    return img.astype(np.float32)


def synth_lf(aw, ah, H, W, C=3, disparity=1, seed=12345):
    """[ah*aw, C, H, W] float32 in [0, 255], row-major SAI order, integer disparity per view."""
    cs, ct = ah // 2, aw // 2
    pad_y, pad_x = disparity * ah, disparity * aw
    base = base_image(H + 2 * pad_y, W + 2 * pad_x, C, seed)
    out = np.empty((ah * aw, C, H, W), np.float32)
    for s in range(ah):
        for t in range(aw):
            oy, ox = pad_y + disparity * (s - cs), pad_x + disparity * (t - ct)
            out[s * aw + t] = base[:, oy:oy + H, ox:ox + W]
    return out


def plan_levels(plan):
    """Windows of a static plan (lfbm5d_step_plan rows) grouped by level: [[rows of level 0], [level 1], ...] in schedule order."""
    levels = [[] for _ in range(int(plan[:, 4].max()) + 1)] if len(plan) else []
    for w in plan:
        levels[int(w[4])].append(w)
    return levels


def window_sais(w, prm, mask=None):
    """Global indices of the SAIs of plan window w; with a mask only the non-empty ones."""
    import lfbm5d_b200 as L
    asw = 2 * int(prm.an) + 1
    out = []
    for s in range(int(w[2]), int(w[2]) + asw):
        for t in range(int(w[3]), int(w[3]) + asw):
            st = s * int(prm.awidth) + t if int(prm.ang_major) == L.ROWMAJOR else s + t * int(prm.aheight)
            if mask is None or mask[st]:
                out.append(st)
    return out
