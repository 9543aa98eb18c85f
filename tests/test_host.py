"""CPU-only host-logic tests of the drop-in module (no kernels run)."""
import os

import numpy as np
import pytest
import torch

from climsr_b200.models import ESRGANGenerator


def test_state_dict_matches_reference_golden(golden_dir):
    z = np.load(os.path.join(golden_dir, "gen_tiny_refinit.npz"))
    torch.manual_seed(0)
    net = ESRGANGenerator(in_channels=2, out_channels=1, nf=64, nb=1, gc=16)
    sd = net.state_dict()
    ref_names = [k[3:] for k in z.files if k.startswith("sd/")]
    assert list(sd.keys()) == ref_names
    # same creation order + same seed -> bit-identical default init as the reference ctor (esrgan.py:72-87)
    for k in ref_names:
        assert np.array_equal(sd[k].numpy(), z["sd/" + k]), k


def test_ctor_signature_and_kwargs():
    net = ESRGANGenerator(in_channels=3, out_channels=1, nf=64, nb=2, gc=16, scaling_factor=4, scale_factor=4, foo="bar")
    assert net.scale_factor == 4
    assert sum(p.numel() for p in net.parameters()) > 0
    with pytest.raises(ValueError):
        ESRGANGenerator(in_channels=3, out_channels=3)      # SRCNN tail only ever worked with 1 (esrgan.py:87,100)
    with pytest.raises(ValueError):
        ESRGANGenerator(in_channels=3, out_channels=1, scaling_factor=2)


def test_param_counts_match_survey():
    count = lambda m: sum(p.numel() for p in m.parameters())  # noqa: E731
    assert count(ESRGANGenerator(3, 1, 64, 11, 16)) == 4_278_530
    assert count(ESRGANGenerator(4, 1, 64, 11, 16)) == 4_279_106
    assert count(ESRGANGenerator(4, 1, 64, 23, 32)) == 16_715_906


def test_forward_validates_shapes():
    net = ESRGANGenerator(2, 1, 64, 1, 16).eval()
    with torch.no_grad():
        with pytest.raises(ValueError):
            net(torch.rand(1, 3, 8, 8), torch.rand(1, 1, 32, 32), torch.rand(1, 1, 32, 32))
        with pytest.raises(ValueError):
            net(torch.rand(1, 2, 8, 8), torch.rand(1, 1, 16, 16), torch.rand(1, 1, 32, 32))


def test_load_state_dict_from_oracle_names():
    from oracle import synth
    sd = synth.make_state_dict(4, 1, 64, 2, 16, seed=3)
    net = ESRGANGenerator(4, 1, 64, 2, 16)
    missing, unexpected = net.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    # Lightning checkpoints prefix the generator with "generator." and are loaded with strict=False (inference.py:125)
    pref = {"generator." + k: v for k, v in sd.items()}
    holder = torch.nn.Module()
    holder.generator = ESRGANGenerator(4, 1, 64, 2, 16)
    r = holder.load_state_dict(pref, strict=False)
    assert not r.missing_keys and not r.unexpected_keys


def test_scaler_and_data_wrappers_refuse_cpu_and_validate_shapes():
    """Error conventions of the drop-in boundary (SURVEY 8b): no CPU fallback - CPU tensors raise CsrError before any
    kernel is touched; shape mistakes raise ValueError like the reference's numpy / torch shape checks."""
    from climsr_b200 import CsrError
    from climsr_b200.data import aug_code, make_lr_batch, random_aug_codes
    from climsr_b200.normalization import MinMaxScaler
    sc = MinMaxScaler(feature_range=(-1.0, 1.0))
    assert (sc.a, sc.b, sc.eps, sc.nan_substitution) == (-1.0, 1.0, 1e-8, 0.0)          # normalization.py:26-35 defaults
    assert MinMaxScaler().feature_range == (0.0, 1.0)
    x = torch.zeros((2, 8, 8))
    with pytest.raises(CsrError):
        sc.normalize(x, [0.0, 0.0], [1.0, 1.0])
    with pytest.raises(CsrError):
        sc.denormalize(torch.zeros((2, 1, 8, 8)), [0.0, 0.0], [1.0, 1.0])
    with pytest.raises(CsrError):
        make_lr_batch(torch.zeros((1, 1, 8, 8)), torch.zeros((1, 1, 8, 8)), torch.zeros((1, 1, 8, 8)))
    # augmentation codes: bit0 vertical flip, bit1 horizontal flip, bits 2-3 rot90 factor (climate_dataset.py:152-170)
    assert [aug_code(False, False, 0), aug_code(True, False, 0), aug_code(False, True, 0), aug_code(True, True, 3)] == [0, 1, 2, 15]
    codes = random_aug_codes(256, torch.Generator().manual_seed(0))
    assert codes.dtype == torch.int32 and int(codes.min()) >= 0 and int(codes.max()) <= 15
    assert set(random_aug_codes(64, torch.Generator().manual_seed(1), v_flip=False, h_flip=False, random_90_rotation=False).tolist()) == {0}
    # with every transform enabled all three draws occur about half of the time
    assert 0.3 < float((codes & 1).float().mean()) < 0.7 and 0.3 < float(((codes >> 1) & 1).float().mean()) < 0.7


def test_gradient_bucketer_layout_is_reverse_parameter_order():
    """Buckets follow the order gradients become final in backward (last layers first), capped by bucket_mb."""
    from climsr_b200.parallel import GradientBucketer
    net = ESRGANGenerator(in_channels=4, out_channels=1, nf=64, nb=1, gc=16)
    b = GradientBucketer(net.parameters(), bucket_mb=0.25, comm_dtype=torch.bfloat16)
    flat = [p for bucket in b.buckets for p in bucket]
    params = [p for p in net.parameters() if p.requires_grad]
    assert len(flat) == len(params) and all(a is c for a, c in zip(flat, reversed(params)))
    assert sum(b.bucket_bytes()) == 2 * sum(p.numel() for p in params)
    assert all(nbytes <= 0.25 * (1 << 20) or len(bucket) == 1 for nbytes, bucket in zip(b.bucket_bytes(), b.buckets))


def test_derived_device_state_is_never_copied_or_pickled():
    """ADVICE r1: copy.deepcopy / torch.save of the module must not duplicate raw CsrPlan* handles or packed blobs."""
    import copy
    import io
    from climsr_b200.models import ESRGANGenerator
    net = ESRGANGenerator(4, 1, 64, 2, 16)
    net._plans[(1, 2, 3)] = (0, None)          # a null handle: csr_plan_destroy(NULL) is a no-op
    net._packed_key = ("x",)
    twin = copy.deepcopy(net)
    assert twin._plans == {} and twin._packed_key is None and twin._ordered_cache is None
    assert all(torch.equal(a, b) for a, b in zip(net.state_dict().values(), twin.state_dict().values()))
    assert all(a.data_ptr() != b.data_ptr() for a, b in zip(net.parameters(), twin.parameters()))
    buf = io.BytesIO()
    torch.save(net, buf)
    buf.seek(0)
    back = torch.load(buf, weights_only=False)
    assert back._plans == {} and back._packed is None and back.nb == 2
    net._plans.clear()


def test_optimizer_steps_bump_the_shared_weight_epoch():
    """Fused optimizers do not bump parameter version counters; a process-wide optimizer post-step hook bumps the epoch that is
    part of the pack-cache key (climsr_b200/models/_common.py)."""
    from climsr_b200.models import ESRGANGenerator
    from climsr_b200.models import _common as E
    net = ESRGANGenerator(4, 1, 64, 1, 16)
    for p in net.parameters():
        p.grad = torch.zeros_like(p)
    for opt in (torch.optim.AdamW(net.parameters(), lr=1e-3), torch.optim.SGD(net.parameters(), lr=1e-3)):
        e0 = E._WEIGHT_EPOCH[0]
        opt.step()
        assert E._WEIGHT_EPOCH[0] == e0 + 1
    assert net._dirty is False
    net.mark_weights_dirty()
    assert net._dirty is True


@pytest.mark.parametrize("kind", ["rcan", "discriminator"])
def test_rcan_and_discriminator_derived_state_is_never_copied_or_pickled(kind):
    """copy.deepcopy / torch.save of RCAN and Discriminator leave their weight packs and captured graphs behind."""
    import copy
    import io
    from climsr_b200.models.discriminator import Discriminator
    from climsr_b200.models.rcan import RCAN
    net = RCAN(n_resgroups=1, n_resblocks=1) if kind == "rcan" else Discriminator()
    conv = next(m for m in net.modules() if isinstance(m, torch.nn.Conv2d))
    net._layer_pack(conv, force=True)          # a CPU scratch: sized and allocated, nothing packed
    assert net._pack_cache._entries
    if kind == "discriminator":
        net._slots = {("key",): [object()]}
        net._calls = {("key",): 3}
    buf = io.BytesIO()
    torch.save(net, buf)
    buf.seek(0)
    for twin in (copy.deepcopy(net), torch.load(buf, weights_only=False)):
        assert not any(k in twin.__dict__ for k in ("_pack_cache", "_slots", "_calls"))
        assert list(twin.state_dict()) == list(net.state_dict())
        assert all(torch.equal(a, b) for a, b in zip(net.state_dict().values(), twin.state_dict().values()))
        assert all(a.data_ptr() != b.data_ptr() for a, b in zip(net.parameters(), twin.parameters()))


def test_weights_key_follows_optimizer_steps_and_in_place_updates():
    from climsr_b200.models._common import weights_key
    conv = torch.nn.Conv2d(4, 8, 3)
    params = list(conv.parameters())
    key = weights_key(params, conv.weight.device)
    assert weights_key(params, conv.weight.device) == key
    for p in params:
        p.grad = torch.ones_like(p)
    torch.optim.AdamW(params, lr=1e-3, fused=False).step()
    stepped = weights_key(params, conv.weight.device)
    assert stepped != key
    with torch.no_grad():
        conv.bias.add_(1.0)
    assert weights_key(params, conv.weight.device) != stepped


def test_layer_pack_cache_keys_and_forced_packs():
    """A hit reuses the scratch as prepacked; a forced call (the conv packs) leaves no key, so the next call packs again; an
    optimizer step invalidates every entry; the scratch is allocated once per layer and device."""
    from climsr_b200.models._common import LayerPackCache
    conv = torch.nn.Conv2d(64, 64, 3, padding=1)
    cache = LayerPackCache()
    scratch, pre, new = cache.get(conv)
    assert (pre, new) == (False, True) and scratch.dtype == torch.uint8 and scratch.numel() > 0
    assert cache.get(conv) == (scratch, True, False)
    assert cache.get(conv, force=True) == (scratch, False, False)
    assert cache.get(conv) == (scratch, False, False)
    assert cache.get(conv) == (scratch, True, False)
    conv.weight.grad = torch.zeros_like(conv.weight)
    torch.optim.SGD([conv.weight], lr=0.0).step()
    assert cache.get(conv) == (scratch, False, False)
    transposed, pre, new = cache.get(conv, transposed=True)
    assert transposed is not scratch and (pre, new) == (False, True)
