"""Pin oracle/net.py against the UNMODIFIED reference modules (skipped where the reference sources are not
present, see oracle/ref_import.py), its EfficientNet-B0 encoder against torchvision (the module the reference's
backbone.py:9 builds, so that part runs everywhere), and the weight sharing of the synthetic checkpoints."""
import numpy as np
import pytest
import torch

from oracle import net, ref_import, resize, synth

needs_reference = pytest.mark.skipif(not ref_import.available(), reason="reference sources not present")


@needs_reference
@pytest.mark.parametrize("model", net.MODELS)
def test_state_dict_spec_matches_reference(model):
    sd = synth.synth_state_dict(model)
    ref = ref_import.build_network(model, sd)            # strict load: names + shapes
    assert list(ref.state_dict().keys()) == [n for n, _, _ in synth.state_dict_spec(model)]


@needs_reference
@pytest.mark.parametrize("model", ["scene_seg", "ego_lanes"])
def test_forward_equals_reference(model):
    sd = synth.synth_state_dict(model)
    ref = ref_import.build_network(model, sd)
    x = net.to_tensor_normalize(resize.pil_bicubic_resize(synth.synth_frame(2), 640, 320))
    with torch.no_grad():
        a = ref(x)
    b = net.forward(model, sd, x)
    assert a.shape == b.shape
    assert (a - b).abs().max().item() <= 1e-5 * max(1.0, a.abs().max().item())


@pytest.mark.parametrize("model", net.MODELS)
def test_encoder_spec_matches_torchvision(model):
    """Every encoder tensor of the synthetic state_dict: name (after the model's prefix), order and shape of
    torchvision's efficientnet_b0().features."""
    import torchvision
    enc = net.PREFIX[model]["enc"]
    spec = [(n[len(enc):], tuple(shape)) for n, shape, _ in synth.state_dict_spec(model) if n.startswith(enc)]
    ref = torchvision.models.efficientnet_b0(weights=None).features.state_dict()
    assert spec == [(k, tuple(v.shape)) for k, v in ref.items()]


@pytest.mark.parametrize("model", ["scene_seg", "ego_lanes"])
def test_encoder_forward_equals_torchvision(model):
    """The oracle's encoder taps (backbone.py:11-22: features 0, 2, 3, 4, 8) == torchvision's efficientnet_b0().features
    with the synthetic weights, full tensors, on a seeded frame."""
    import torchvision
    enc = net.PREFIX[model]["enc"]
    sd = synth.synth_state_dict(model)
    ref = torchvision.models.efficientnet_b0(weights=None).features.eval()
    ref.load_state_dict({k[len(enc):]: v for k, v in sd.items() if k.startswith(enc)}, strict=True)
    x = net.to_tensor_normalize(resize.pil_bicubic_resize(synth.synth_frame(2), 640, 320))
    want = []
    with torch.no_grad():
        h = x
        for i, layer in enumerate(ref):
            h = layer(h)
            if i in (0, 2, 3, 4, 8):
                want.append(h)
    taps = {}
    net.forward(model, sd, x, taps=taps)
    for i, a in enumerate(want):
        b = taps[f"f{i}"]
        assert a.shape == b.shape
        assert (a - b).abs().max().item() <= 1e-5 * max(1.0, a.abs().max().item()), f"f{i}"


def test_shared_parts_are_byte_identical():
    ss = synth.synth_state_dict("scene_seg")
    dsg = synth.synth_state_dict("domain_seg")
    s3d = synth.synth_state_dict("scene_3d")
    for part in ("enc", "ctx", "neck"):
        p0, p1 = net.PREFIX["scene_seg"][part], net.PREFIX["domain_seg"][part]
        for k, v in ss.items():
            if k.startswith(p0):
                assert torch.equal(v, dsg[p1 + k[len(p0):]])
    p0, p1 = net.PREFIX["scene_seg"]["enc"], net.PREFIX["scene_3d"]["enc"]
    n = 0
    for k, v in ss.items():
        if k.startswith(p0):
            assert torch.equal(v, s3d[p1 + k[len(p0):]])
            n += 1
    assert n == 358
    # and the unshared variant really differs
    s3d_ns = synth.synth_state_dict("scene_3d", share=False)
    assert not torch.equal(s3d_ns[p1 + "0.0.weight"], ss[p0 + "0.0.weight"])


@needs_reference
def test_infer_helper_postprocess_matches_oracle(tmp_path):
    """Boundary #1: the reference's SceneSegNetworkInfer end to end vs oracle pre/post."""
    from PIL import Image
    sd = synth.synth_state_dict("scene_seg")
    ck = tmp_path / "ss.pth"
    torch.save(sd, ck)
    infer = ref_import.infer_class("scene_seg")(checkpoint_path=str(ck))
    small = resize.pil_bicubic_resize(synth.synth_frame(4), 640, 320)
    got = infer.inference(Image.fromarray(small))
    exp = net.postprocess("scene_seg", net.forward("scene_seg", sd, net.to_tensor_normalize(small)))
    assert got.dtype == np.int64 and got.shape == (320, 640)
    assert np.array_equal(got, exp)
