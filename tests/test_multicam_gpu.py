"""Config 5 (BASELINE.json configs[4], SURVEY.md §8e) on real GPUs through the C-ABI (include/vp_b200_multicam.h):
every rank runs EgoLanes on its own camera frame and the device lateral post-process on its own lane
masks; ONE ncclAllGather (issued from C++, communicator created in C++ from a 128-byte id) exchanges the fused
feature maps + PathFinder measurements; every rank fuses the measurements with the reference's
Estimator::update rule on the GPU.  Needs >= 2 GPUs (skipped on a single-GPU machine).  No torch.distributed
here: the id travels through a file."""
import os
import time

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _worker(rank, world, vpw, out_dir):
    import ctypes as C
    from autoware_vision_pilot_b200 import _lib as L
    from autoware_vision_pilot_b200 import engine as E
    from autoware_vision_pilot_b200 import lateral, multicam
    from oracle import lateral as olat
    from oracle import synth
    torch.cuda.set_device(rank)
    id_path = os.path.join(out_dir, "nccl_id.bin")
    if rank == 0:
        with open(id_path + ".tmp", "wb") as f:
            f.write(multicam.make_unique_id())
        os.replace(id_path + ".tmp", id_path)
    t0 = time.time()
    while not os.path.exists(id_path):
        assert time.time() - t0 < 120, "rank 0 never published the NCCL id"
        time.sleep(0.05)
    uid = open(id_path, "rb").read()

    stream = torch.cuda.Stream()
    eng = E.Engine([E.EGO_LANES], [vpw], gpu_id=rank, resize_mode=E.RESIZE_PIL_BICUBIC, stream=stream.cuda_stream)
    mc = multicam.MultiCamera(uid, rank, world, rank, stream=stream.cuda_stream)
    lat = lateral.LateralPostProcess(device=f"cuda:{rank}")
    frame = synth.synth_frame(multicam.frame_seed(rank, 0))
    eng.infer(frame)
    local_feat = eng.read_tap("0/fused")                               # fp32 [1456,10,20], exact 16-bit values
    # lane masks of THIS camera: synthetic lanes (the synthetic checkpoint's masks are noise); rank 1 sees no
    # right lane -> its measurement has NaN slots, the "no measurement" branch of Estimator::update
    masks = torch.from_numpy(olat.synth_lane_masks(15 + rank, drop_right=(rank == 1))).float().cuda()
    results = []
    with torch.cuda.stream(stream):
        for it in range(2):
            lat.update_device(masks.data_ptr(), 80, 160, stream=stream.cuda_stream, autosteer_steering_rad=0.01 * rank)
            mc.step_engine(eng, 0, lat._out.data_ptr(), predict=(it == 1))
            mc.sync()
            feats, meas, state = mc.read()
            results.append({"feats": feats.copy(), "meas": meas.copy(), "state": state.copy(), "lat": lat.result()})
    us = mc.time_allgather(200)
    torch.save({"local_feat": local_feat, "results": results, "allgather_us": us}, os.path.join(out_dir, f"r{rank}.pt"))
    mc.close()
    eng.close()


def test_multicamera_allgather_and_fusion(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    from autoware_vision_pilot_b200 import weights as W
    from oracle import post, synth
    world = min(torch.cuda.device_count(), 8)
    vpw = W.write_vpw(synth.synth_state_dict("ego_lanes"), str(tmp_path / "ego.vpw"))
    mp.spawn(_worker, args=(world, vpw, str(tmp_path)), nprocs=world, join=True)
    outs = [torch.load(tmp_path / f"r{r}.pt", weights_only=False) for r in range(world)]

    def nan_eq(a, b):
        return np.array_equal(np.nan_to_num(a, nan=-7.0), np.nan_to_num(b, nan=-7.0))

    # which cameras see a valid lane pair (PathFinder runs, main.cpp:565): the CPU restatement of the lateral chain
    from oracle import lateral as olat
    exp_ran = []
    for r in range(world):
        f, t = olat.LaneFilter(), olat.LaneTracker()
        row = []
        for it in range(2):
            o = f.update(olat.synth_lane_masks(15 + r, drop_right=(r == 1)))
            row.append(bool(t.update(o.left, o.right).bev_valid))
        exp_ran.append(row)
    assert sum(row[0] for row in exp_ran) >= 2                        # the fusion really fuses several cameras
    exp_state = post.initial_state()
    for it in range(2):
        # what every camera contributed: its device PathFinder measurement, checked against the restatement of
        # path_finder.cpp:97-157 on that camera's own fitted curves
        exp_meas = np.stack([o["results"][it]["lat"]["pf_meas"] for o in outs])
        for r, o in enumerate(outs):
            lr = o["results"][it]["lat"]
            m = lr["pf_meas"]
            assert np.isnan(m[0, 0]) and np.isnan(m[3, 0]) and np.isnan(m[13, 0])
            assert np.allclose(m[:, 1], post.pathfinder_measurement([0, 0, 0], [0, 0, 0], 0.0, 4.0)[:, 1], rtol=1e-15)
            assert bool(lr["pf_ran"]) == exp_ran[r][it], f"rank {r} frame {it}: PathFinder ran {lr['pf_ran']}"
            if lr["pf_ran"]:
                # the device measurement == path_finder.cpp:97-157 restated on this camera's own fitted curves
                # (lane-width slot: the camera's Estimator mean before the update = 4.0 on the first frame)
                assert m[9, 0] == 0.01 * r and m[10, 0] == 0.01 * r
                if it == 0:
                    ref = post.pathfinder_measurement(lr["pf_left_coeff"], lr["pf_right_coeff"], 0.01 * r, 4.0)
                    assert nan_eq(np.isnan(ref[:, 0]), np.isnan(m[:, 0]))
                    assert np.allclose(np.nan_to_num(m[:, 0]), np.nan_to_num(ref[:, 0]), rtol=1e-12, atol=1e-12)
            else:
                assert np.isnan(m[:, 0]).all()                          # camera without valid lanes: "no measurement"
        if it == 1:
            exp_state[:, 1] += 0.25                                     # Estimator::predict, proc_SD 0.5
        for m in exp_meas:
            exp_state = post.estimator_update(exp_state, m)
        for r, o in enumerate(outs):
            res = o["results"][it]
            # all-gather == stack of the per-rank payloads, bit-exact
            got = res["feats"].view(np.float16).astype(np.float32).transpose(0, 3, 1, 2)
            for k in range(world):
                assert np.array_equal(got[k], outs[k]["local_feat"]), (r, k)
            assert nan_eq(res["meas"], exp_meas)
            # fused state == fp64 restatement of estimator.cpp:24-74 applied in rank order
            assert np.allclose(res["state"], exp_state, rtol=1e-13, atol=0), (r, it)
    for o in outs[1:]:
        assert np.array_equal(o["results"][1]["state"], outs[0]["results"][1]["state"])   # every rank holds the same state
    us = max(o["allgather_us"] for o in outs)
    print(f"config5 ok: world {world}, ncclAllGather of 582624 B/rank = {us:.1f} us (max over ranks)")


def test_engines_on_two_devices_from_other_threads(tmp_path):
    """ADVICE r1: every C-ABI entry point runs under a device guard — engines on two GPUs in ONE process, each driven from
    a thread whose current device is the OTHER GPU, give the single-engine results."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import threading
    from autoware_vision_pilot_b200 import engine as E
    from autoware_vision_pilot_b200 import weights as W
    from oracle import synth
    vpw = W.write_vpw(synth.synth_state_dict("ego_lanes"), str(tmp_path / "ego.vpw"))
    frames = [synth.synth_frame(0), synth.synth_frame(1)]
    ref = []
    for f in frames:
        e = E.Engine([E.EGO_LANES], [vpw], gpu_id=0, resize_mode=E.RESIZE_PIL_BICUBIC)
        e.infer(f)
        ref.append(e.raw(0).copy())
        e.close()
    engs = [E.Engine([E.EGO_LANES], [vpw], gpu_id=g, resize_mode=E.RESIZE_PIL_BICUBIC) for g in (0, 1)]
    out = [None, None]

    def work(i):
        torch.cuda.set_device(1 - i)                      # the "wrong" device is current in this thread
        for _ in range(3):
            engs[i].infer(frames[i])
        out[i] = engs[i].raw(0).copy()
        assert torch.cuda.current_device() == 1 - i       # the guard restored the caller's device

    ts = [threading.Thread(target=work, args=(i,)) for i in (0, 1)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert np.array_equal(out[0], ref[0]) and np.array_equal(out[1], ref[1])
