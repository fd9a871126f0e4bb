"""mdn_instance_mask_union_table (the union that reads its (pointer, count) table from device memory, so a CUDA graph can
replay it on new instance masks) against mdn_instance_mask_union, under the SIMT emulator; loss_utils.InstanceMaskTable's
checks; and the new entry point's argument errors in the real library (no GPU needed)."""
import ctypes as C

import pytest
import torch

from emu_harness import emulated
from mdn_sfm_b200 import loss_utils, synthetic


def _instances(counts, H, W, seed, odd_offset=()):
    """A list of {"instances": obj} with counts[b] random masks of sample b; samples in `odd_offset` live at an odd byte
    address (a slice of a larger buffer), which forces the kernels' one-byte path."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for b, n in enumerate(counts):
        m = torch.rand(n, H, W, generator=g) > 0.8
        if b in odd_offset:
            buf = torch.zeros(n * H * W + 1, dtype=torch.bool)
            buf[1:] = m.reshape(-1)
            m = buf[1:].view(n, H, W)
            assert m.data_ptr() % 2 == 1 or n == 0
        out.append({"instances": synthetic.SyntheticInstances(m)})
    return out


def _unions(inst, batch, lib):
    """(old host-table union, new device-table union) of the same batch: (B, H, W) uint8 each."""
    H, W = loss_utils._pred_masks(inst)[0].shape[-2:]
    table = loss_utils.InstanceMaskTable(batch, H, W, "cpu").load(inst)
    B, H, W = table.batch, table.height, table.width
    new = torch.full((B, H, W), 7, dtype=torch.uint8)
    lib.call("mdn_instance_mask_union_table", table.ptrs.data_ptr(), table.counts.data_ptr(), new.data_ptr(), B, H * W, 0)
    masks = [m.view(torch.uint8) for m in loss_utils._pred_masks(inst)]
    if not isinstance(inst, list):
        masks = masks * batch
    old = torch.full((B, H, W), 9, dtype=torch.uint8)
    counts = (C.c_int32 * B)(*[m.shape[0] for m in masks])
    lib.call("mdn_instance_mask_union", (C.c_void_p * B)(*[m.data_ptr() for m in masks]), counts, old.data_ptr(), B, H * W, 0)
    ref = torch.stack([(m.sum(0) != 0) if m.shape[0] else torch.zeros(H, W, dtype=torch.bool) for m in masks]).to(torch.uint8)
    return old, new, ref


@pytest.mark.parametrize("H,W", [(16, 24), (15, 22), (15, 21)], ids=["hw%4==0", "hw%2==0", "hw-odd"])
def test_table_union_equals_the_host_table_union(H, W):
    """Four-, two- and one-byte paths (chosen from hw and pointer alignment), counts with zeros, one sample at an odd
    byte address."""
    inst = _instances([3, 0, 1, 5, 0, 2], H, W, seed=H * W, odd_offset=(3,))
    with emulated() as lib:
        old, new, ref = _unions(inst, 6, lib)
    assert torch.equal(old, new)
    assert torch.equal(new, ref)


def test_table_union_at_kitti_size_and_beyond_one_chunk():
    """375 x 1242 (two bytes per thread, four pixel pairs in flight) and a batch of 40: more samples than the host-table
    entry point passes per launch, in one launch."""
    inst = _instances([2, 0], 375, 1242, seed=1)
    with emulated() as lib:
        old, new, ref = _unions(inst, 2, lib)
        assert torch.equal(old, new) and torch.equal(new, ref)
        counts = [(b * 7) % 4 for b in range(40)]
        inst = _instances(counts, 9, 20, seed=2, odd_offset=(5, 17))
        old, new, ref = _unions(inst, 40, lib)
    assert torch.equal(old, new) and torch.equal(new, ref)


def test_bare_instances_and_the_resized_levels():
    """A bare Instances fills every sample of the table with its masks: the same bytes as the eager broadcast of the
    (1, H, W) union; instance_masks_u8 with a table equals it with the list / bare form at every pyramid level."""
    sizes = [(32, 48), (16, 24), (8, 12)]
    inst = _instances([3, 0, 2], 64, 96, seed=5)
    bare = inst[0]["instances"]
    with emulated() as lib:
        old, new, ref = _unions(bare, 4, lib)
        assert torch.equal(old, new) and torch.equal(new, ref)
        eager_list = loss_utils.instance_masks_u8(inst, sizes, "cpu", lib, batch=3)
        eager_bare = loss_utils.instance_masks_u8(bare, sizes, "cpu", lib, batch=4)
        t_list = loss_utils.InstanceMaskTable(3, 64, 96, "cpu").load(inst)
        t_bare = loss_utils.InstanceMaskTable(4, 64, 96, "cpu").load(bare)
        got_list = loss_utils.instance_masks_u8(t_list, sizes, "cpu", lib, batch=3)
        got_bare = loss_utils.instance_masks_u8(t_bare, sizes, "cpu", lib, batch=4)
    for a, b in zip(eager_list + eager_bare, got_list + got_bare):
        assert a.shape == b.shape and torch.equal(a, b)


def test_table_load_checks_each_mask():
    """load() accepts what the eager path hands the kernel unchanged (bool / uint8, contiguous, (N, H, W) of the table's
    size, on the table's device) and refuses the rest; a reload points the table at the new batch."""
    m = lambda *s, **kw: torch.zeros(*s, **kw).bool()
    one = lambda t: [{"instances": synthetic.SyntheticInstances(t)}]
    with emulated():
        t = loss_utils.InstanceMaskTable(1, 8, 12, "cpu")
        with pytest.raises(TypeError, match="bool or uint8"):
            t.load(one(torch.zeros(1, 8, 12)))
        with pytest.raises(ValueError, match="contiguous"):
            t.load(one(m(1, 12, 8).transpose(1, 2)))
        with pytest.raises(ValueError, match=r"\(N, 8, 12\)"):
            t.load(one(m(1, 8, 13)))
        with pytest.raises(ValueError, match=r"\(N, 8, 12\)"):
            t.load(one(m(8, 12)))
        with pytest.raises(ValueError, match="holds 2 samples"):
            t.load(one(m(1, 8, 12)) * 2)
        a, b = m(2, 8, 12), torch.zeros(0, 8, 12, dtype=torch.uint8)
        t.load(one(a))
        assert int(t.ptrs[0]) == a.data_ptr() and int(t.counts[0]) == 2
        t.load(one(b))
        assert int(t.counts[0]) == 0 and t.masks[0] is not None and t.masks[0].shape[0] == 0
        with pytest.raises(ValueError, match="instance table on meta"):
            loss_utils.InstanceMaskTable(1, 8, 12, "meta").load(one(m(1, 8, 12)))


def test_error_codes_of_the_table_union():
    """Argument checks of mdn_instance_mask_union_table return status codes before any launch."""
    from mdn_sfm_b200 import _cabi, build
    lib = _cabi.Library(build.build())
    for args in ((None, 16, 16), (16, None, 16), (16, 16, None)):
        with pytest.raises(RuntimeError, match=r"\(-2\).*NULL"):
            lib.call("mdn_instance_mask_union_table", *args, 1, 16, None)
    for batch, hw in ((0, 16), (-1, 16), (65536, 16), (1, 0), (1, -5)):
        with pytest.raises(RuntimeError, match=r"\(-1\).*out of range"):
            lib.call("mdn_instance_mask_union_table", 16, 16, 16, batch, hw, None)
