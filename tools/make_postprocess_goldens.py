"""Golden vectors for mug_diffusion_b200/postprocess.py from the UNMODIFIED reference (mug/data/utils.py), run in this container:
    python tools/make_postprocess_goldens.py        -> tests/golden/postprocess.json, tests/golden/postprocess_seeds.json
Synthetic charts (seeded): notes on a 1/4 or 1/8 grid of a known bpm/offset with jitter, chords, long notes and deliberate mini-jacks."""
import importlib.util
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def chart(seed, bpm, offset, n, div=4, jitter=3.0, ln_ratio=0.15, jack_ratio=0.08):
    rng = np.random.default_rng(seed)
    step = 60000 / bpm / div
    slots = np.sort(rng.choice(n * 3, n, replace=False))
    lines = []
    prev = None
    for k in slots:
        t = int(offset + step * k + rng.normal(0, jitter))
        cols = rng.choice(4, rng.choice([1, 1, 1, 2, 3]), replace=False)
        for c in cols:
            x = int((c + 0.5) * 128)
            if rng.random() < ln_ratio:
                lines.append((t, f"{x},192,{t},128,0,{t + int(step * rng.integers(2, 9))}:0:0:0:0:"))
            else:
                lines.append((t, f"{x},192,{t},1,0,0:0:0:0:"))
        if prev is not None and rng.random() < jack_ratio:
            c = prev
            tj = t + int(rng.integers(30, 85))
            lines.append((tj, f"{int((c + 0.5) * 128)},192,{tj},1,0,0:0:0:0:"))
        prev = int(cols[0])
    lines.sort(key=lambda p: p[0])
    return [l for _, l in lines]


CASES = [dict(seed=1, bpm=187.3, offset=412, n=260), dict(seed=2, bpm=240.0, offset=1033, n=400, div=8, jitter=2.0),
         dict(seed=3, bpm=152.5, offset=95, n=120, jitter=4.0, ln_ratio=0.3), dict(seed=4, bpm=299.0, offset=2500, n=300, jack_ratio=0.2),
         dict(seed=5, bpm=175.0, offset=0, n=40, jitter=0.0, ln_ratio=0.0)]
SEEDS = [11, 12, 13]


def seed_case(seed):
    """a denser-jack chart whose bpm, offset and grid follow from the seed"""
    return dict(seed=seed, bpm=150 + 13.7 * seed % 140, offset=300 + seed, n=150, div=4 if seed % 2 else 8, jack_ratio=0.15)


def main():
    spec = importlib.util.spec_from_file_location("ref_utils", "/root/reference/mug/data/utils.py")
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    out = []
    for c in CASES:
        lines = chart(**c)
        dejack = ref.remove_intractable_mania_mini_jacks(lines, verbose=False)
        grid, bpm, off = ref.gridify(dejack, verbose=False)
        dejack2 = ref.remove_intractable_mania_mini_jacks(grid, verbose=False, jack_interval=60)
        out.append(dict(case=c, n_in=len(lines), dejack=dejack, grid=grid, bpm=float(bpm), offset=float(off), dejack_after_grid=dejack2))
        print(c, len(lines), "->", len(dejack), "->", len(dejack2), "bpm", bpm, "offset", off)
    json.dump(out, open(os.path.join(ROOT, "tests", "golden", "postprocess.json"), "w"))
    out = []
    for seed in SEEDS:
        c = seed_case(seed)
        dejack = ref.remove_intractable_mania_mini_jacks(chart(**c), verbose=False)
        grid, bpm, off = ref.gridify(dejack, verbose=False)
        out.append(dict(case=c, dejack=dejack, grid=grid, bpm=float(bpm), offset=float(off)))
    json.dump(out, open(os.path.join(ROOT, "tests", "golden", "postprocess_seeds.json"), "w"))


if __name__ == "__main__":
    sys.exit(main())
