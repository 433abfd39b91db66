"""BASELINE.json configs[0] on the GPU: the UNMODIFIED reference run on a B200 in eager fp32 (TF32 off, cuDNN autotuner off)
on the bike clip of cfg1_bike.npz, as shipped and with `get_similarity` evaluated in float64 (tests/ref_runner.py,
exact_similarity=True).  Needs the reference tree (baseline/_ref, or CUTIE_REFERENCE_ROOT) and a GPU:
    python tests/golden/make_golden_bike_gpu.py [out.npz]
Writes (default tests/golden/cfg1_bike_gpu_ref.npz), for the first propagated frame -- the one the bike tests assert --
the segment() logits of both runs at a fixed, seeded sample of the decoder-stride grid of cfg1_bike.npz's `logits_s4`
(every 4th pixel, offset 2), and the float64-similarity run's output masks of frames 0 and 1 at full resolution.
A sample, not the whole grid: the full logits of one frame are ~5 MB."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests.ref_runner import run_reference_clip             # noqa: E402
from tests.test_gpu_zz_cfg1_bike import _inputs              # noqa: E402

GOLDEN = os.path.dirname(os.path.abspath(__file__))
SAMPLE = 6144                      # of the 120 x 216 decoder-stride positions


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(GOLDEN, 'cfg1_bike_gpu_ref.npz')
    g = np.load(os.path.join(GOLDEN, 'cfg1_bike.npz'))
    frames, mask, objects = _inputs(g)
    runs = {name: run_reference_clip(frames, mask, objects, device='cuda', max_internal_size=480, snapshot=False,
                                     exact_similarity=(name == 'exact')) for name in ('plain', 'exact')}
    lg = {name: r['logits'][1][0, :, 2::4, 2::4] for name, r in runs.items()}        # [1+K, 120, 216]
    C, hs, ws = lg['exact'].shape
    idx = np.sort(np.random.default_rng(0).choice(hs * ws, SAMPLE, replace=False)).astype(np.int32)
    pick = lambda t: t.reshape(C, -1)[:, torch.from_numpy(idx).long()].numpy().astype(np.float32)
    np.savez_compressed(out, s4_index=idx, s4_shape=np.array([hs, ws]),
                        logits_shape=np.array(runs['exact']['logits'][1].shape),
                        plain_logits_f1=pick(lg['plain']), exact_logits_f1=pick(lg['exact']),
                        exact_masks=np.stack([m.numpy().astype(np.uint8) for m in runs['exact']['masks'][:2]], 0),
                        device=np.array(torch.cuda.get_device_name(0)), torch_version=np.array(torch.__version__))
    print('wrote', out, {k: tuple(v.shape) for k, v in np.load(out).items()})


if __name__ == '__main__':
    main()
