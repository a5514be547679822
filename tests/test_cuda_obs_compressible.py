"""GPU: engine-owned observation blocks in compressible device memory (mfb_alloc_device).  The allocator's blocks are
zeroed and readable like any device memory, and observe() / observe_groups() into them give the same bits as
observe(out=...) into ordinary torch tensors."""
import ctypes
import gc

import numpy as np
import pytest

from scenarios import c4_positions, generate_map_positions

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def alloc(nbytes):
    from mfmarl_b200.lib import check, load_library
    lib = load_library()
    ptr, comp = ctypes.c_void_p(), ctypes.c_int()
    check(lib.mfb_alloc_device(nbytes, 0, ctypes.byref(ptr), ctypes.byref(comp)))
    return lib, ptr, comp.value


def test_allocator_grants_compression_on_b200():
    lib, ptr, comp = alloc(64 << 20)
    try:
        if "B200" in torch.cuda.get_device_name(0):
            assert comp == 1
    finally:
        assert lib.mfb_free_device(ptr) == 0
    assert lib.mfb_free_device(None) == 0
    assert lib.mfb_free_device(ctypes.c_void_p(ptr.value + 16)) != 0      # not a block of the allocator


def test_fresh_block_reads_zero():
    from mfmarl_b200.battle import _DeviceBlock
    from mfmarl_b200.lib import load_library
    lib, dev = load_library(), torch.device("cuda:0")
    shape = (3, 1000, 1183)                    # 14.2 MB: not a multiple of the allocation granularity
    t = _DeviceBlock(lib, shape, torch.float32, dev).tensor()
    assert t.shape == shape and t.dtype == torch.float32 and t.is_cuda
    assert not t.view(torch.int32).any()
    t.fill_(3.0)
    torch.cuda.synchronize()
    del t
    gc.collect()
    t = _DeviceBlock(lib, shape, torch.float32, dev).tensor()
    assert not t.view(torch.int32).any()
    b = _DeviceBlock(lib, (5, 13, 13, 8), torch.bfloat16, dev).tensor()
    assert b.dtype == torch.bfloat16 and b.shape == (5, 13, 13, 8) and not b.view(torch.int16).any()


def make(E, map_size, cap, pos, **kw):
    from mfmarl_b200 import BatchedGridWorld
    env = BatchedGridWorld(E, map_size=map_size, capacity=cap, rng="philox", seed=3, auto_reset=True, **kw)
    env.reset()
    env.add_agents(0, pos[0])
    env.add_agents(1, pos[1])
    return env


CASES = {
    "c3_shape": dict(E=32, map_size=40, cap=64, pos=lambda: generate_map_positions(40), kw=dict(max_steps=25)),
    "c4_record": dict(E=2, map_size=80, cap=512, pos=c4_positions, kw=dict(max_steps=30, obs_record=True)),
    "concurrent": dict(E=16, map_size=40, cap=64, pos=lambda: generate_map_positions(40),
                       kw=dict(max_steps=20, concurrent_step_envs=16)),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_engine_blocks_equal_caller_tensors(case):
    c = CASES[case]
    env = make(c["E"], c["map_size"], c["cap"], c["pos"](), **c["kw"])
    E, cap = env.n_envs, env.capacity
    gen = torch.Generator(device="cuda:0")
    gen.manual_seed(11)
    view, feat = env.observe()
    if "B200" in torch.cuda.get_device_name(0):
        assert env.obs_compressed is True
    ref_view, ref_feat = torch.zeros_like(view), torch.zeros_like(feat)
    for s in range(60):
        num = torch.from_numpy(env.get_num()).cuda()
        v, f = env.observe()
        assert v.data_ptr() == view.data_ptr() and f.data_ptr() == feat.data_ptr()      # reused, engine-owned
        env.observe(out=(ref_view, ref_feat))
        # every row, stale ones included: both blocks received exactly the same writes since they were zero
        assert torch.equal(v.view(torch.int32), ref_view.view(torch.int32)), "view differs at step %d" % s
        assert torch.equal(f.view(torch.int32), ref_feat.view(torch.int32)), "feature differs at step %d" % s
        live = torch.arange(cap, device=num.device) < num[..., None]                  # [E, 2, cap]
        for dtype in (torch.float32, torch.bfloat16):
            groups = env.observe_groups(dtype=dtype)
            for g in range(2):
                vg, fg = groups[g]
                want = ref_view[:, g].to(dtype)
                if dtype == torch.bfloat16:
                    want = torch.cat([want, torch.zeros_like(want[..., :1])], dim=-1)
                m = live[:, g]
                bits = torch.int16 if dtype == torch.bfloat16 else torch.int32
                assert torch.equal(vg[m].view(bits), want[m].view(bits)), "observe_groups %s g%d step %d" % (dtype, g, s)
                assert torch.equal(fg[m].view(torch.int32), ref_feat[:, g][m].view(torch.int32))
        actions = torch.randint(0, 21, (E, 2, cap), generator=gen, device="cuda:0", dtype=torch.int32)
        env.step(actions)
    assert env.get("episode").min() > 0, "the run never crossed an auto-reset"


def test_view_outlives_engine():
    env = make(4, 40, 64, generate_map_positions(40))
    view, feat = env.observe()
    want_v, want_f = view.cpu(), feat.cpu()
    del env
    gc.collect()
    torch.cuda.synchronize()
    assert torch.equal(view.cpu().view(torch.int32), want_v.view(torch.int32))
    assert torch.equal(feat.cpu().view(torch.int32), want_f.view(torch.int32))
    assert float(view.sum()) == float(want_v.sum())


def test_copy_to_pinned_host():
    env = make(64, 40, 64, generate_map_positions(40))
    gen = torch.Generator(device="cuda:0")
    gen.manual_seed(5)
    for _ in range(5):
        env.observe()
        env.step(torch.randint(0, 21, (64, 2, env.capacity), generator=gen, device="cuda:0", dtype=torch.int32))
    view, _ = env.observe()
    host = torch.empty(view.shape, dtype=view.dtype).pin_memory()
    host.copy_(view, non_blocking=True)
    torch.cuda.synchronize()
    assert torch.equal(host.cuda().view(torch.int32), view.view(torch.int32))
    assert np.count_nonzero(host.numpy()) > 0
