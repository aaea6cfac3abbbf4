"""Device JPEG loader (SURVEY 8f-3) against PIL -- the decoder the reference calls at compute_feats.py:28 -- bit for
bit, through the C-ABI (dsmil_jpeg_parse_batch + dsmil_jpeg_decode_batch), and through embed_bag."""
import io
import os

import numpy as np
import pytest
import torch
from PIL import Image

import jpeg_cases as jc

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


def _to_tensor(rgb):                                    # VF.to_tensor of a uint8 HWC image
    return torch.from_numpy(rgb).permute(2, 0, 1).contiguous().float().div(255)


def _check(files):
    from dsmil_wsi_b200 import jpeg
    u8, f32, status = jpeg.decode_files(files, DEV)
    assert status == [0] * len(files)
    u8, f32 = u8.cpu().numpy(), f32.cpu()
    for i, data in enumerate(files):
        want = jc.pil_rgb(data)
        assert np.array_equal(u8[i], want), f"file {i}: {np.abs(u8[i].astype(int) - want.astype(int)).max()}"
        assert torch.equal(f32[i], _to_tensor(want)), f"file {i} (float form)"


@pytest.mark.parametrize("hw", [(224, 224), (256, 256), (223, 217), (17, 33), (8, 8), (1, 1), (5, 3), (100, 2), (64, 250)])
@pytest.mark.parametrize("subsampling", [0, 1, 2])
def test_decode_matches_pil_bit_for_bit(hw, subsampling):
    h, w = hw
    files = []
    for img in (jc.noise(h, w, 1), jc.histology_like(h, w, 2)):
        for q in (30, 70, 95, 100):
            for extra in ({}, {"restart_marker_blocks": 5}):
                files.append(jc.encode(img, quality=q, subsampling=subsampling, **extra))
    _check(files)


def test_reference_patch_batch_128x224_q70():
    _check(jc.patch_files(128))


def test_channels_last_float_output_holds_the_same_values():
    from dsmil_wsi_b200 import jpeg
    files = jc.patch_files(5, 64, 48)
    pb = jpeg.parse_batch(files)
    dec = jpeg.JpegBatchDecoder(DEV)
    a = torch.empty(5, 3, 64, 48, device=DEV)
    b = torch.empty(5, 3, 64, 48, device=DEV, memory_format=torch.channels_last)
    dec.decode(pb, out_f32=a)
    dec.decode(pb, out_f32=b)
    torch.cuda.synchronize()
    assert b.is_contiguous(memory_format=torch.channels_last) and torch.equal(a, b)
    assert torch.equal(a[0].cpu(), _to_tensor(jc.pil_rgb(files[0])))


def test_mixed_tables_grey_and_optimised_in_one_batch():
    img = jc.histology_like(96, 80, 3)
    b = io.BytesIO()
    Image.fromarray(img).convert("L").save(b, format="JPEG", quality=70)
    files = [jc.encode(img, quality=70), jc.encode(img, quality=70, optimize=True), b.getvalue(),
             jc.encode(img, quality=40, subsampling=0), jc.encode(img, quality=90, subsampling=1, restart_marker_rows=1)]
    _check(files)


def test_batch_with_a_progressive_file_is_refused_not_misdecoded():
    from dsmil_wsi_b200 import jpeg
    img = jc.histology_like(32, 32, 0)
    files = [jc.encode(img, quality=70), jc.encode(img, quality=70, progressive=True)]
    with pytest.raises(ValueError, match="not decodable on the device"):
        jpeg.decode_files(files, DEV)
    # the kernels themselves skip a flagged record: status -2, the other file still decodes
    pb = jpeg.parse_batch(files)
    assert pb.statuses.tolist() == [0, -2]
    dec = jpeg.JpegBatchDecoder(DEV)
    u8 = torch.zeros(2, 32, 32, 3, dtype=torch.uint8, device=DEV)
    status = dec.decode(pb, out_u8=u8)
    torch.cuda.synchronize()
    assert status.cpu().tolist() == [0, -2]
    assert np.array_equal(u8[0].cpu().numpy(), jc.pil_rgb(files[0])) and int(u8[1].sum()) == 0


def test_damaged_entropy_data_does_not_hang_or_write_out_of_bounds():
    from dsmil_wsi_b200 import jpeg
    good = jc.encode(jc.noise(64, 64, 5), quality=90)
    rng = np.random.default_rng(0)
    files = [good]
    for k in range(6):
        b = bytearray(good)
        lo = len(b) // 2
        for pos in rng.integers(lo, len(b) - 2, size=20):
            b[pos] = int(rng.integers(0, 255))
        files.append(bytes(b[: len(b) - 2 - 50 * k]))
    pb = jpeg.parse_batch(files)
    assert pb.statuses.tolist()[0] == 0
    dec = jpeg.JpegBatchDecoder(DEV)
    guard = torch.full((len(files) + 1, 64, 64, 3), 7, dtype=torch.uint8, device=DEV)
    status = dec.decode(pb, out_u8=guard[:len(files)])
    torch.cuda.synchronize()
    st = status.cpu().tolist()
    assert st[0] == 0 and all(s in (0, -1) for s in st)
    assert np.array_equal(guard[0].cpu().numpy(), jc.pil_rgb(good))
    assert bool((guard[len(files)] == 7).all())


def test_abi_rejects_bad_arguments():
    from dsmil_wsi_b200 import _lib
    lib = _lib.load()
    assert lib.dsmil_jpeg_workspace_bytes(-1, 8, 8, 10) < 0
    assert lib.dsmil_jpeg_workspace_bytes(4, 0, 8, 10) < 0
    need = lib.dsmil_jpeg_workspace_bytes(4, 224, 224, 1000)
    assert need >= 4 * 3 * 224 * 224 * 3
    buf = torch.zeros(4096, dtype=torch.uint8, device=DEV)
    rc = lib.dsmil_jpeg_decode_batch(buf.data_ptr(), 100, buf.data_ptr(), 1, 8, 8, buf.data_ptr(), None, 0, buf.data_ptr(),
                                     buf.data_ptr(), 16, None)
    assert rc == -2                                     # DSMIL_ERR_WORKSPACE


def _write_bag(tmp_path, n, seed=0, **kw):
    bag = tmp_path / "class0" / "bag0"
    bag.mkdir(parents=True)
    for i, data in enumerate(jc.patch_files(n, seed=seed, **kw)):
        (bag / f"{i}_{i}.jpeg").write_bytes(data)
    return str(bag)


def test_embed_bag_device_route_equals_host_route(tmp_path, monkeypatch):
    """The loop of compute_feats.py:58-82 from patch FILES: decoding on the device gives the backbone the same
    tensor as PIL on the host, so features and scores agree."""
    import torchvision.models as models
    import dsmil as mil
    from dsmil_wsi_b200 import embed
    bag = _write_bag(tmp_path, 150)                     # 128 + a ragged batch of 22
    torch.manual_seed(0)
    resnet = models.resnet18(weights=None, norm_layer=torch.nn.InstanceNorm2d)
    resnet.fc = torch.nn.Identity()
    ic = mil.IClassifier(resnet, 512, 2).to(DEV).eval()
    paths = embed.list_patches(bag)
    monkeypatch.setenv("DSMIL_B200_JPEG", "gpu")
    f_dev, c_dev = embed.embed_bag(paths, ic, batch_size=128, num_workers=4)
    monkeypatch.setenv("DSMIL_B200_JPEG", "host")
    f_host, c_host = embed.embed_bag(paths, ic, batch_size=128, num_workers=4)
    assert f_dev.shape == (150, 512) and c_dev.shape == (150, 2)
    assert torch.allclose(f_dev, f_host, rtol=0, atol=1e-5), float((f_dev - f_host).abs().max())
    assert torch.allclose(c_dev, c_host, rtol=0, atol=1e-5)


def test_embed_bag_auto_route_falls_to_pil_for_a_progressive_patch(tmp_path, monkeypatch):
    import dsmil as mil
    from dsmil_wsi_b200 import embed
    bag = _write_bag(tmp_path, 6, h=64, w=64)
    prog = jc.encode(jc.histology_like(64, 64, 99), quality=70, progressive=True)
    with open(os.path.join(bag, "9_9.jpeg"), "wb") as f:
        f.write(prog)

    class Tiny(torch.nn.Module):
        def forward(self, x):
            return x.mean(dim=(2, 3)).repeat(1, 4)      # [B, 12] "features" that expose the decoded pixels
    ic = mil.IClassifier(Tiny(), 12, 2).to(DEV).eval()
    paths = sorted(embed.list_patches(bag))
    monkeypatch.setenv("DSMIL_B200_JPEG", "auto")
    f_auto, _ = embed.embed_bag(paths, ic, batch_size=4, num_workers=2)      # batch 0 on the device, batch 1 through PIL
    monkeypatch.setenv("DSMIL_B200_JPEG", "host")
    f_host, _ = embed.embed_bag(paths, ic, batch_size=4, num_workers=2)
    assert torch.equal(f_auto, f_host)
    monkeypatch.setenv("DSMIL_B200_JPEG", "gpu")
    with pytest.raises(RuntimeError, match="not decodable on the device"):
        embed.embed_bag(paths, ic, batch_size=4, num_workers=2)


def test_embed_bag_graph_replay_equals_eager_launches(tmp_path, monkeypatch):
    """Full batches go through one CUDA-graph replay of the embedder, the ragged tail eagerly: same features."""
    import torchvision.models as models
    import dsmil as mil
    from dsmil_wsi_b200 import embed
    bag = _write_bag(tmp_path, 70, h=64, w=64)          # 4 full batches of 16 + 6
    torch.manual_seed(0)
    resnet = models.resnet18(weights=None, norm_layer=torch.nn.InstanceNorm2d)
    resnet.fc = torch.nn.Identity()
    ic = mil.IClassifier(resnet, 512, 2).to(DEV).eval()
    paths = embed.list_patches(bag)
    monkeypatch.setenv("DSMIL_B200_EMBED_GRAPH", "1")
    f_g, c_g = embed.embed_bag(paths, ic, batch_size=16, num_workers=2)
    assert embed._GRAPHS.get(ic) is not None and embed._GRAPHS[ic][1] is not None, "the embedder was not captured"
    f_g2, _ = embed.embed_bag(paths, ic, batch_size=16, num_workers=2)          # cached graph, second bag
    monkeypatch.setenv("DSMIL_B200_EMBED_GRAPH", "0")
    f_e, c_e = embed.embed_bag(paths, ic, batch_size=16, num_workers=2)
    assert f_g.shape == (70, 512)
    assert torch.equal(f_g, f_g2)
    assert torch.allclose(f_g, f_e, rtol=0, atol=1e-5) and torch.allclose(c_g, c_e, rtol=0, atol=1e-5)
    # new parameter tensors (e.g. a checkpoint loaded by re-assignment) invalidate the capture
    ic.fc.weight = torch.nn.Parameter(ic.fc.weight.detach().clone() * 2.0)
    monkeypatch.setenv("DSMIL_B200_EMBED_GRAPH", "1")
    _, c_new = embed.embed_bag(paths, ic, batch_size=16, num_workers=2)
    monkeypatch.setenv("DSMIL_B200_EMBED_GRAPH", "0")
    _, c_new_e = embed.embed_bag(paths, ic, batch_size=16, num_workers=2)
    assert torch.allclose(c_new, c_new_e, rtol=0, atol=1e-5) and not torch.allclose(c_new, c_g)


def test_staging_buffers_come_from_the_staging_stream(tmp_path, monkeypatch):
    """The staging thread writes the slot buffers on its own stream while the embedder runs on the compute stream.
    Taken from the compute stream's pool, a slot could get a block the embedder has freed while its queued kernels
    still use it, and the next batch's decode would race with them (rows of the second batch came out wrong)."""
    import dsmil as mil
    from dsmil_wsi_b200 import embed

    class Tiny(torch.nn.Module):
        def forward(self, x):
            return x.mean(dim=(2, 3)).repeat(1, 4)
    ic = mil.IClassifier(Tiny(), 12, 2).to(DEV).eval()
    paths = embed.list_patches(_write_bag(tmp_path, 10, h=64, w=48))       # 3 batches of 4: both slots
    for route in ("gpu", "host"):
        monkeypatch.setenv("DSMIL_B200_JPEG", route)
        embed.embed_bag(paths, ic, batch_size=4, num_workers=2)
    st = next(s for s in embed._STAGING.values() if (s.batch, s.H, s.W) == (4, 64, 48))
    torch.cuda.synchronize()
    segments = torch.cuda.memory_snapshot()
    for t in st.dev_f32 + st.dev_u8:
        seg = next(g for g in segments if g["address"] <= t.data_ptr() < g["address"] + g["total_size"])
        assert seg["stream"] == st.stream.cuda_stream
