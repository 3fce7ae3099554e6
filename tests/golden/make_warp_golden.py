"""Golden vectors of the REFERENCE's own CUDA warp kernel (run on a GPU: `python tests/golden/make_warp_golden.py OUTDIR`).

oracle/_ref/libref_warp.so = stnbdhw/BilinearSamplerBDHW.cu:48-109 compiled for sm_100a (oracle/Makefile refwarp), built
only where the reference sources are present.  Writes to OUTDIR (default: this directory)
  warp_ref.npz        outputs on the seeded inputs of WARP_CASES, in full: pins oracle/fav_oracle.c:orc_warp_bdhw on the
                      CPU (tests/test_oracle.py) and the product's warp on the GPU (tests/test_gpu_refwarp.py);
  warp_ref_shapes.npz outputs at the BASELINE.json shapes of SHAPES (real and stress flows), the reference-order temporal
                      prior composition and a batched / resized call: each as the SHA-256 of the full array (a bit-exact
                      pin that fits in a few bytes at 4K) plus a seeded sample of its values (tells how far a mismatch is).
Inputs are regenerated from seeds at test time; only outputs are stored."""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "fast-artistic-videos_b200"))

from fav_b200 import synth  # noqa: E402

WARP_CASES = [  # (name, C, Hin, Win, Hout, Wout, flow kind)
    ("real_64x96", 3, 64, 96, 64, 96, "real"), ("stress_64x96", 3, 64, 96, 64, 96, "stress"),
    ("real_97x75", 3, 97, 75, 97, 75, "real"), ("stress_33x129", 1, 33, 129, 33, 129, "stress"),
    ("resize_40x56_to_52x44", 5, 40, 56, 52, 44, "rand"), ("sentinel_32x48", 1, 32, 48, 32, 48, "sentinel")]

# the five BASELINE.json config shapes (256^2 tiny, 720p, 1080p, 2048^2 VR face, 4K) + ragged small ones
SHAPES = [(256, 256), (720, 1280), (1080, 1920), (2048, 2048), (2160, 3840), (97, 75), (33, 129)]
PRIOR_SHAPE = (360, 640)
N_SAMPLE = 2048


def warp_inputs(case):
    name, C, Hin, Win, Ho, Wo, kind = case
    rng = np.random.default_rng(sum(map(ord, name)))
    if C == 3:
        img = synth.make_frame(Hin, Win, 1) * 1.2 - 0.1
    else:
        img = rng.uniform(-0.2, 1.2, size=(C, Hin, Win)).astype(np.float32)
    if kind == "real":
        flow = synth.checker_to_lua(synth.make_backward_flow(Ho, Wo, 2))
    elif kind == "stress":
        flow = synth.stress_flow(Ho, Wo)
    elif kind == "sentinel":  # vr_helper.lua:10 maps: 99999 outside the strip, a real offset inside
        flow = np.full((2, Ho, Wo), 99999.0, np.float32)
        flow[:, :, Wo // 3: Wo // 2] = rng.uniform(-5, 5, size=(2, Ho, Wo // 2 - Wo // 3)).astype(np.float32)
    else:
        flow = rng.uniform(-9, 9, size=(2, Ho, Wo)).astype(np.float32)
    return np.ascontiguousarray(img, np.float32), np.ascontiguousarray(flow, np.float32)


def shape_inputs(H, W):
    """Frame and the two flows ('real', 'stress'; Lua (dy,dx) layout) warped at each of SHAPES."""
    img = np.ascontiguousarray(synth.make_frame(H, W, 1) * 1.2 - 0.1, np.float32)
    return img, {"real": synth.checker_to_lua(synth.make_backward_flow(H, W, 2)), "stress": synth.stress_flow(H, W)}


def prior_inputs():
    """content, previous stylized frame, flow (dy,dx), certainty at PRIOR_SHAPE."""
    from oracle import net_oracle

    H, W = PRIOR_SHAPE
    return (synth.make_frame(H, W, 2), synth.make_frame(H, W, 1) * 1.2 - 0.1,
            synth.checker_to_lua(synth.make_backward_flow(H, W, 2)), net_oracle.make_cert(H, W, 2))


def batch_inputs():
    """2 x 5 channels warped to a 13x36 grid, and the all-99999 sentinel flow (vr_helper.lua:10) over a 20x28 image."""
    rng = np.random.default_rng(0)
    img = rng.uniform(size=(2, 5, 20, 28)).astype(np.float32)
    grid = rng.uniform(-6, 6, size=(2, 2, 13, 36)).astype(np.float32)
    return img, grid, np.full((1, 2, 20, 28), 99999.0, np.float32)


def digest(a) -> str:
    """SHA-256 of a float32 array's values (-0.0 counted as 0.0, as torch.equal does)."""
    return hashlib.sha256((np.ascontiguousarray(a, np.float32) + np.float32(0)).tobytes()).hexdigest()


def sample(a) -> np.ndarray:
    """N_SAMPLE values of a at indices seeded by its size."""
    flat = np.ascontiguousarray(a, np.float32).reshape(-1)
    return flat[np.sort(np.random.default_rng(flat.size).integers(0, flat.size, N_SAMPLE))]


def main(outdir):
    import torch

    from oracle import refwarp

    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    out = {}
    for case in WARP_CASES:
        img, flow = warp_inputs(case)
        out[case[0]] = refwarp.warp(T(img)[None], T(flow)[None])[0].cpu().numpy()
    shapes = {}

    def put(key, a):
        shapes[key + "_sha256"], shapes[key + "_sample"] = np.array(digest(a)), sample(a)

    for H, W in SHAPES:
        img, flows = shape_inputs(H, W)
        for kind, flow in flows.items():
            put(f"{H}x{W}_{kind}", refwarp.warp(T(img)[None], T(flow)[None])[0].cpu().numpy())
    # the temporal prior composed from the reference kernel's warp with torch ops in the reference's order
    _, p, flow, cert = prior_inputs()
    warped = refwarp.warp(T(p)[None], T(flow)[None])[0]
    mean = torch.tensor([103.939, 116.779, 123.68], device="cuda").view(3, 1, 1)
    pre = warped[[2, 1, 0]] * 255.0 - mean                 # preprocess.lua:57-62: index, mul(255), add(-1, mean)
    put("prior", (torch.zeros_like(pre) + pre * T(cert)).cpu().numpy())  # core.lua:167 fill(vgg-mean = 0) + cmul
    img, grid, sentinel = batch_inputs()
    shapes["batch"] = refwarp.warp(T(img), T(grid)).cpu().numpy()
    shapes["sentinel"] = refwarp.warp(T(img[:1]), T(sentinel)).cpu().numpy()
    torch.cuda.synchronize()
    os.makedirs(outdir, exist_ok=True)
    np.savez_compressed(os.path.join(outdir, "warp_ref.npz"), **out)
    np.savez_compressed(os.path.join(outdir, "warp_ref_shapes.npz"), **shapes)
    print("wrote", outdir, {k: v.shape for k, v in out.items()}, sorted(shapes))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.dirname(os.path.abspath(__file__)))
