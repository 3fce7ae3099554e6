"""Generates the committed golden fixtures under tests/golden/ (run where the reference sources are present).

  consistency_*.npz : seeded flow pairs (+ frame) and the {0,255} masks written by the REFERENCE's own
                      consistencyChecker binary (oracle/_ref/consistencyChecker, compiled unmodified from the
                      reference's consistencyChecker/ by oracle/Makefile), 3- and 4-argument mode.
  clip_64x96.npz    : fp64 PyTorch-oracle outputs of a 3-frame synthetic clip (net + recurrence);
                      the torch restatement is "parity unpinned" (Torch7 cannot run here), see DESIGN.md.
Inputs are regenerated from seeds by fav_b200.synth at test time; only outputs are stored.
"""
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "fast-artistic-videos_b200"))
import torch  # noqa: E402

from fav_b200 import synth  # noqa: E402
from oracle import net_oracle, pyoracle  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

CONSISTENCY_CASES = [  # (H, W, frame idx, fw-noise sigma, seed)
    (64, 96, 2, 0.0, 1), (100, 76, 3, 0.6, 2), (97, 75, 2, 0.6, 3), (256, 256, 2, 0.6, 4), (240, 320, 4, 0.3, 5),
    (72, 88, 5, 0.5, 11)]


def consistency_inputs(H, W, idx, sigma, seed):
    rng = np.random.default_rng(seed)
    bw = synth.make_backward_flow(H, W, idx)
    fw = synth.make_forward_flow(H, W, idx)
    if sigma > 0:
        fw = (fw + rng.normal(0, sigma, size=fw.shape)).astype(np.float32)
    fr = synth.make_frame(H, W, idx)
    fr[:, :, : W // 2] = 0.5  # flat half: the structure term matters there
    fr[:, H // 3: H // 2, :] = np.linspace(0, 1, W, dtype=np.float32)[None, None, :]
    img255 = np.clip(np.rint(fr * 255.0), 0, 255).astype(np.float32)
    return bw, fw, fr, img255


def write_consistency(case):
    """consistency_{H}x{W}.npz of one CONSISTENCY_CASES entry: the reference binary's masks, bit-packed."""
    assert os.path.exists(pyoracle.REF_CHECKER), "build oracle/_ref first (make -C oracle ref)"
    H, W, idx, sigma, seed = case
    bw, fw, fr, _ = consistency_inputs(H, W, idx, sigma, seed)
    d = tempfile.mkdtemp()
    synth.write_flo(d + "/bw.flo", bw); synth.write_flo(d + "/fw.flo", fw); synth.write_ppm(d + "/f.ppm", fr)
    pyoracle.run_ref_checker(d + "/bw.flo", d + "/fw.flo", d + "/r3.pgm")
    pyoracle.run_ref_checker(d + "/bw.flo", d + "/fw.flo", d + "/r4.pgm", d + "/f.ppm")
    r3, r4 = synth.read_pgm(d + "/r3.pgm"), synth.read_pgm(d + "/r4.pgm")
    assert set(np.unique(r3)) <= {0, 255} and set(np.unique(r4)) <= {0, 255}
    np.savez_compressed(os.path.join(HERE, f"consistency_{H}x{W}.npz"), ref3=np.packbits(r3 == 255),
                        ref4=np.packbits(r4 == 255), shape=np.array([H, W]),
                        params=np.array([idx, sigma, seed], np.float64))
    print(H, W, "zeros", (r3 == 0).sum(), (r4 == 0).sum())


def main():
    for case in CONSISTENCY_CASES:
        write_consistency(case)
    H, W = 64, 96
    outs = net_oracle.run_clip(net_oracle.NetOracle(style="candy", dtype=torch.float64), H, W, 3)
    np.savez_compressed(os.path.join(HERE, "clip_64x96.npz"), outs=np.stack(outs).astype(np.float32))
    print("clip", np.stack(outs).shape)


if __name__ == "__main__":
    main()
