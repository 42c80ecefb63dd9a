"""Build-container script: the real-image parity set (SURVEY.md §8d: frames of
VisionPilot/software_defined_vehicle/OpenADKit/Test/traffic-driving.mp4).

Decodes 8 frames of the reference's own 1920x1080 test video, commits them as lossless stills
(tests/golden/real/frame_XX.png at 640x320 = Pillow-bicubic resize of the decoded frame, the caller-side resize of
Models/visualizations/SceneSeg/image_visualization.py:108-109; one full-resolution frame for the fused resize), and the
outputs of the UNMODIFIED reference modules (oracle/ref_import.py) on them with the synthetic checkpoints
(no real weights are reachable offline): class maps / masks and a stride-8 logits sample (margins are recomputed from the oracle at test time).

Usage: python scripts/make_real_golden.py     (needs /root/reference)
"""
import hashlib
import os
import sys

import cv2
import numpy as np
import torch
from PIL import Image

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import net, ref_import, synth  # noqa: E402

VIDEO = os.path.join(ref_import.REFERENCE_ROOT, "VisionPilot/software_defined_vehicle/OpenADKit/Test/traffic-driving.mp4")
OUT = os.path.join(synth.GOLDEN_DIR, "real")
FRAMES = (0, 4, 8, 12, 16, 20, 24, 28)      # 8 of the first 32 frames
FULL_RES = 12                                # this one is also kept at 1920x1080


def main():
    assert os.path.exists(VIDEO), VIDEO
    os.makedirs(OUT, exist_ok=True)
    cap = cv2.VideoCapture(VIDEO)
    frames = {}
    for i in range(max(FRAMES) + 1):
        ok, bgr = cap.read()
        assert ok
        if i in FRAMES:
            frames[i] = np.ascontiguousarray(bgr[:, :, ::-1])           # RGB, as PIL callers see it
    smalls = {}
    for i, rgb in frames.items():
        assert rgb.shape == (1080, 1920, 3)
        small = np.asarray(Image.fromarray(rgb).resize((640, 320)))      # Pillow default: BICUBIC with antialias
        smalls[i] = small
        Image.fromarray(small).save(os.path.join(OUT, f"frame_{i:02d}.png"), optimize=True)
    Image.fromarray(frames[FULL_RES]).save(os.path.join(OUT, f"frame_{FULL_RES:02d}_1080p.png"), optimize=True)
    torch.set_num_threads(8)            # tests/test_oracle_real_images.py evaluates the oracle with the same count
    for m in net.MODELS:
        ref = ref_import.build_network(m, synth.synth_state_dict(m))
        rec = {"threads": np.int64(torch.get_num_threads())}     # the count the goldens were computed with
        for i, small in smalls.items():
            with torch.no_grad():
                o = ref(net.to_tensor_normalize(small))
            post = np.asarray(net.postprocess(m, o))
            o = o[0].numpy()
            rec[f"sample_{i}"] = o[:, ::8, ::8].astype(np.float32)
            rec[f"std_{i}"] = np.float64(o.std())
            rec[f"small_sha_{i}"] = np.frombuffer(hashlib.sha256(small.tobytes()).digest(), dtype=np.uint8)
            if m == "scene_seg":
                rec[f"post_{i}"] = post.astype(np.uint8)
            elif m == "domain_seg":
                rec[f"post_{i}"] = post.astype(np.uint8)[..., 0]
            elif m == "ego_lanes":
                rec[f"post_{i}"] = net.ego_lanes_masks(o)[1].astype(np.uint8)
            print(m, i, "std", o.std(), flush=True)
        path = os.path.join(OUT, f"{m}_real.npz")
        np.savez_compressed(path, **rec)
        print("wrote", path, os.path.getsize(path) // 1024, "KiB")
    print("stills:", sum(os.path.getsize(os.path.join(OUT, f)) for f in os.listdir(OUT) if f.endswith(".png")) // 1024, "KiB")


if __name__ == "__main__":
    main()
