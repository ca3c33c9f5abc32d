"""VRAM tiering: a region's bytes are bit-identical before/after any migration, its device
address never changes, budgets are enforced, and the LRU policy keeps the working set home."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

R = 32 << 20


def _ndev():
    import torch
    return torch.cuda.device_count()


def _want_digest(seed):
    import oracle
    return oracle.digest(oracle.pattern(seed, R))


def test_host_tier_round_trip_single_gpu():
    import oracle
    from tensor_fusion_b200 import vram as V
    with V.VSpace(home=0, va_bytes=32 * R, region_bytes=R, home_budget=8 * R, host_budget=16 * R) as vs:
        assert vs.n_regions == 32 and vs.region_bytes == R
        for r in range(8):
            vs.populate(r, V.HOME)
            vs.fill_pattern(r, 1000 + r)
        for r in range(8, 12):
            vs.populate(r, V.HOST)
            vs.write(r, 0, oracle.pattern(1000 + r, R))
        with pytest.raises(V.TfwError) as e:
            vs.populate(12, V.HOME)                      # home budget is 8 regions
        assert e.value.status == 4
        assert vs.digest(3) == _want_digest(1003)         # device pattern kernel == oracle restatement
        assert np.array_equal(vs.read(5, R - 4096, 4096), oracle.pattern(1005, R)[-4096:])
        # evict 4 HOME regions to host and bring the 4 HOST regions home, one batch each
        res = vs.migrate([0, 1, 2, 3], [V.HOST] * 4)
        assert res["bytes"] == 4 * R and vs.residency(2)[0] == V.HOST
        with pytest.raises(V.TfwError):
            vs.digest(2)                                  # cold region: not mapped until prefetched
        res = vs.migrate([8, 9, 10, 11], [V.HOME] * 4)
        assert res["bytes"] == 4 * R
        for r in range(8, 12):
            assert vs.residency(r) == (V.HOME, 0) and vs.digest(r) == _want_digest(1000 + r)
        assert np.array_equal(vs.read(1, 0, R), oracle.pattern(1001, R))       # still intact in host DRAM
        vs.migrate([4, 5, 6, 7], [V.HOST] * 4)
        vs.migrate([0, 1, 2, 3], [V.HOME] * 4)
        for r in range(4):
            assert vs.digest(r) == _want_digest(1000 + r)
        st = vs.stats()
        assert st["regions_home"] == 8 and st["regions_host"] == 4
        assert st["evict_bytes_host"] == 8 * R and st["prefetch_bytes_host"] == 8 * R
        with pytest.raises(V.TfwError):
            vs.migrate([0, 0], [V.HOST, V.HOST])           # duplicate region in one batch


def test_client_pointer_survives_migration():
    """A kernel of the worker writes through the vGPU address before and after the region moved."""
    import oracle
    from tensor_fusion_b200 import vram as V
    from tensor_fusion_b200.worker import Worker
    with V.VSpace(home=0, va_bytes=4 * R, region_bytes=R, home_budget=2 * R, host_budget=2 * R) as vs, Worker() as w:
        vs.populate(1, V.HOME)
        ptr = vs.base + 1 * R
        src = w.dev_alloc(R)
        w.dev_write(src, oracle.pattern(7, R))
        w.move_batch([(ptr + 13, src + 5, R - 64, 0)])            # misaligned copy into the region
        w.flush()
        vs.migrate([1], [V.HOST])
        vs.migrate([1], [V.HOME])                                   # new physical memory, same address
        want = np.zeros(R, dtype=np.uint8)
        want[13:13 + R - 64] = oracle.pattern(7, R)[5:5 + R - 64]
        assert np.array_equal(w.dev_read(ptr, R), want)
        w.move_batch([(ptr, 0, 4096, 0xCD)])
        assert np.all(w.dev_read(ptr, 4096) == 0xCD)
        w.dev_free(src)


def test_lru_policy_sweeps_and_zipf_single_gpu():
    """C4 access pattern in miniature: 3 sequential sweeps then Zipf(1.1), seed 42; every region
    keeps its bytes while the policy shuffles it between HBM and host DRAM."""
    import oracle
    from tensor_fusion_b200 import vram as V
    n, budget = 24, 8
    with V.VSpace(home=0, va_bytes=n * R, region_bytes=R, home_budget=budget * R, host_budget=n * R) as vs:
        for r in range(n):
            vs.populate(r, V.HOME if r < budget else V.HOST)
            if r < budget:
                vs.fill_pattern(r, 50 + r)
            else:
                vs.write(r, 0, oracle.pattern(50 + r, R))
        seq = [r for _ in range(3) for r in range(n)]
        rng = np.random.default_rng(42)
        seq += [int(min(n - 1, z - 1)) for z in rng.zipf(1.1, 200)]
        for r in seq:
            vs.access(r)
            assert vs.residency(r)[0] == V.HOME
        vs.quiesce()                                      # evictions run in the background: let them land
        st = vs.stats()
        # the policy keeps one region of the budget free (or being freed) so that the next miss finds room at once
        assert budget - 1 <= st["regions_home"] <= budget and st["regions_host"] == n - st["regions_home"]
        assert 0 <= st["policy_evictions"] - st["policy_prefetches"] <= 1 and st["policy_prefetches"] >= 3 * n - budget
        assert st["policy_hits"] > 50                     # Zipf head stays resident
        for r in range(n):
            if vs.residency(r)[0] == V.HOME:
                assert vs.digest(r) == _want_digest(50 + r)
            else:
                assert oracle.digest(vs.read(r, 0, R)) == _want_digest(50 + r)


def test_fixed_frames_are_never_remapped_and_keep_every_byte():
    """TFW_VS_FIXED_FRAMES: frame f backs every region r with r % frames == f through aliased mappings made once; a region
    coming home evicts its frame's occupant, no VMM call after create.  Sweeps (where direct-mapped == LRU), then a Zipf
    pattern full of conflict misses: every region keeps its bytes, wherever it lives."""
    import oracle
    from tensor_fusion_b200 import vram as V
    n, budget = 24, 8
    peers = list(range(1, _ndev()))[:3]
    with pytest.raises(V.TfwError):                       # a VA cannot name its frame and the region's peer backing
        V.VSpace(home=0, va_bytes=n * R, region_bytes=R, home_budget=budget * R, host_budget=n * R, flags=V.FIXED_FRAMES | V.PEER_IN_PLACE)
    for ahead in (0, 2):
        with V.VSpace(home=0, va_bytes=n * R, region_bytes=R, home_budget=budget * R, peer_budget=n * R if peers else 0,
                      host_budget=0 if peers else n * R, peers=peers, prefetch_ahead=ahead, flags=V.FIXED_FRAMES) as vs:
            for r in range(n):
                vs.access(r)
                vs.fill_pattern(r, 9000 + r)
            want = [_want_digest(9000 + r) for r in range(n)]
            vmm0 = vs.stats()["vmm_ns"]
            got, _ = vs.sweep(5, 3 * n)
            assert got == [want[(5 + i) % n] for i in range(3 * n)]
            rng = np.random.default_rng(7)
            for r in [int(min(n - 1, z - 1)) for z in rng.zipf(1.1, 150)] + [3, 11, 19, 3, 11, 19]:   # 3, 11, 19 share frame 3
                vs.access(r)
                assert vs.residency(r)[0] == V.HOME and vs.digest(r) == want[r]
            vs.quiesce()
            st = vs.stats()
            assert st["remaps"] == 0 and (peers or st["vmm_ns"] == vmm0), st   # no region VA was touched since the space was set up
            assert st["regions_home"] <= budget and st["regions_home"] + st["regions_peer"] + st["regions_host"] == n
            home = [r for r in range(n) if vs.residency(r)[0] == V.HOME]
            assert len({r % budget for r in home}) == len(home)            # one region per frame
            for r in range(n):                                              # cold regions answer through their backing's alias
                if vs.residency(r)[0] == V.HOST:
                    assert oracle.digest(vs.read(r, 0, R)) == want[r]
                else:
                    assert vs.digest(r) == want[r]
            # the explicit interface goes through the frames too: 19 lives in frame 3, 3 wants to come home
            assert vs.residency(19)[0] == V.HOME and vs.residency(3)[0] != V.HOME
            with pytest.raises(V.TfwError):
                vs.migrate([3], [V.HOME])
            vs.migrate([19, 3], [V.PEER if peers else V.HOST, V.HOME], [0, -1] if peers else None)
            assert vs.residency(3)[0] == V.HOME and vs.digest(3) == want[3]
            assert vs.residency(19)[0] != V.HOME
            assert (vs.digest(19) if peers else oracle.digest(vs.read(19, 0, R))) == want[19]


@pytest.mark.parametrize("ahead", [0, 2])
def test_pipelined_sweep_keeps_every_byte(ahead):
    """The policy path as one native loop (tfw_vspace_sweep): access + a digest kernel per region on a bound client
    stream, migrations asynchronous -- prefetch of region k+1.. and eviction of the LRU region run while the client
    reads region k.  Three laps over 24 regions with 8 resident: every digest equals the oracle's, every lap."""
    from tensor_fusion_b200 import vram as V
    n, budget = 24, 8
    peers = list(range(1, _ndev()))[:3]
    with V.VSpace(home=0, va_bytes=n * R, region_bytes=R, home_budget=budget * R, peer_budget=n * R if peers else 0,
                  host_budget=0 if peers else n * R, peers=peers, prefetch_ahead=ahead) as vs:
        for r in range(n):
            vs.access(r)                                  # first touch: zero-filled HOME backing, colder regions leave
            vs.fill_pattern(r, 7000 + r)
        want = [_want_digest(7000 + r) for r in range(n)]
        got, secs = vs.sweep(5, 3 * n)                    # starts in the middle, wraps around the address space
        assert got == [want[(5 + i) % n] for i in range(3 * n)]
        st = vs.stats()
        assert st["regions_home"] + st["regions_peer"] + st["regions_host"] == n and budget - 1 - ahead <= st["regions_home"] <= budget
        moved = st["prefetch_bytes_peer"] + st["prefetch_bytes_host"]
        assert moved >= (3 * n - budget) * R              # a sequential sweep over 3x the budget misses every time
        if ahead:
            # how many early prefetches find room depends on how fast evictions finish against the reading kernel
            # (NVLink: nearly all of them, PCIe with these small regions: about one access in five)
            assert st["policy_prefetch_ahead"] > 0 and st["policy_hits_inflight"] + st["policy_hits"] >= st["policy_prefetch_ahead"] - ahead
        # and the explicit, synchronous interface still works on the same space afterwards
        vs.migrate([0, 1], [V.PEER if peers else V.HOST] * 2, [0, 0] if peers else None)
        vs.migrate([0, 1], [V.HOME] * 2)
        assert vs.digest(0) == want[0] and vs.digest(1) == want[1]


@pytest.mark.parametrize("flags", [0, 1])
def test_peer_tier_round_trip(flags):
    """Needs >= 2 GPUs: evict to peer HBM over NVLink (mover kernel / copy engine), read it
    back THROUGH the same vGPU address, prefetch, stripe a batch over all peers."""
    if _ndev() < 2:
        pytest.skip("needs at least 2 GPUs")
    from tensor_fusion_b200 import vram as V
    peers = list(range(1, _ndev()))
    n = 16
    with V.VSpace(home=0, va_bytes=n * R, region_bytes=R, home_budget=n * R, peer_budget=n * R, host_budget=2 * R,
                  peers=peers, flags=flags) as vs:
        for r in range(n):
            vs.populate(r, V.HOME)
            vs.fill_pattern(r, 900 + r)
        slots = [r % len(peers) for r in range(n)]
        res = vs.migrate(list(range(n)), [V.PEER] * n, slots)          # one batch, striped over the peers
        assert res["bytes"] == n * R and res["launches"] == (0 if flags == 1 else n)   # one pull kernel per region, on the GPU that receives it
        for r in range(n):
            assert vs.residency(r) == (V.PEER, peers[slots[r]])
            assert vs.digest(r) == _want_digest(900 + r)                 # home GPU reads peer HBM through the VA
        vs.fill_pattern(3, 4242)                                          # and writes it
        vs.migrate([3, 5], [V.HOST, V.PEER], [-1, (slots[5] + 1) % len(peers)])   # peer->host, peer->other peer (or no-op)
        vs.migrate(list(range(n)), [V.HOME] * n)
        for r in range(n):
            assert vs.residency(r) == (V.HOME, 0)
            assert vs.digest(r) == _want_digest(4242 if r == 3 else 900 + r)
        st = vs.stats()
        assert st["evict_bytes_peer"] >= n * R and st["prefetch_bytes_peer"] >= (n - 1) * R


def test_policy_prefers_peer_hbm_over_host():
    if _ndev() < 2:
        pytest.skip("needs at least 2 GPUs")
    from tensor_fusion_b200 import vram as V
    peers = list(range(1, _ndev()))
    n, budget = 12, 4
    with V.VSpace(home=0, va_bytes=n * R, region_bytes=R, home_budget=budget * R, peer_budget=3 * R, host_budget=n * R,
                  peers=peers) as vs:
        for r in range(budget):
            vs.populate(r, V.HOME)
            vs.fill_pattern(r, r)
        for r in range(budget, n):
            vs.populate(r, V.HOST)
        for r in list(range(n)) * 2:
            vs.access(r)
        vs.quiesce()
        st = vs.stats()
        assert 1 <= st["regions_peer"] <= 3 * len(peers)                  # victims go to peer HBM while it has room
        assert st["regions_peer"] + st["regions_host"] == n - st["regions_home"] and budget - 1 <= st["regions_home"] <= budget
        assert st["evict_bytes_peer"] >= 3 * len(peers) * R               # the peers were filled before host was used
        for r in range(budget):
            t, _ = vs.residency(r)
            if t != V.HOST:
                assert vs.digest(r) == _want_digest(r)


def test_worker_buffers_live_in_the_tiered_space():
    """north_star (c) under the worker: client buffers are allocated in a tiered vGPU address space
    whose HBM budget (8 x 16 MiB) is far smaller than what the trace keeps alive; cold regions go to host
    DRAM and come back on touch, and every client-visible byte still equals the oracle's replay."""
    import oracle
    from tensor_fusion_b200 import trace, wire
    from tensor_fusion_b200.worker import Worker
    Rr = 4 << 20
    tiering = dict(va_bytes=1024 * Rr, region_bytes=Rr, home_budget=8 * Rr, host_budget=640 * Rr)
    raw = trace.gen_c1(seed=4242, ncalls=700, max_buffer_bytes=40 << 20, error_permille=5)
    rep = oracle.Replay(raw)
    with Worker(tiering=tiering, chunk_bytes=8 << 20) as w:
        n, resp = w.run(raw)
        assert n == raw.nbytes
        assert resp == rep.responses()
        assert w.stats()["vram_peak_bytes"] > 2 * 8 * Rr                 # far more live bytes than the 32 MiB HBM budget
        for h in rep.live_handles():
            assert np.array_equal(w.read(h), rep.buffer(h)), f"buffer {h}"
    # one buffer bigger than the whole HBM budget streams through in pieces
    Rr = 16 << 20
    tiering = dict(va_bytes=64 * Rr, region_bytes=Rr, home_budget=8 * Rr, host_budget=32 * Rr)
    big = 12 * Rr + 12345
    rng = np.random.default_rng(8)
    data = rng.integers(0, 256, big, dtype=np.uint8)
    b = wire.Builder().malloc(1, big).h2d(1, 0, data.tobytes()).memset(1, 5, 1000, 0x77).d2h(1, big - 5000, 5000).sync()
    rep = oracle.Replay(bytes(b))
    with Worker(tiering=tiering, chunk_bytes=8 << 20) as w:
        _, resp = w.run(bytes(b))
        assert resp == rep.responses()
        assert np.array_equal(w.read(1), rep.buffer(1))


def test_freeze_to_host_and_resume():
    """FreezeWorker / "freeze to mem": every resident region of the vGPU goes to host DRAM (its HBM is
    released), submissions are refused while frozen, and after resume the buffers read back bit-identical."""
    import oracle
    from tensor_fusion_b200 import _native as N
    from tensor_fusion_b200 import trace, wire
    from tensor_fusion_b200.worker import Worker
    Rr = 8 << 20
    tiering = dict(va_bytes=128 * Rr, region_bytes=Rr, home_budget=16 * Rr, host_budget=64 * Rr)
    raw = trace.gen_c1(seed=606, ncalls=300, max_buffer_bytes=12 << 20, error_permille=0)
    rep = oracle.Replay(raw)
    with Worker(tiering=tiering) as w:
        _, resp = w.run(raw)
        assert resp == rep.responses()
        moved = w.freeze()
        assert moved > 0 and moved % Rr == 0
        assert w.freeze() == 0                                   # idempotent
        with pytest.raises(N.TfwError) as e:
            w.submit(bytes(wire.Builder().sync()))
        assert e.value.status == N.TFW_ERR_NOT_SUPPORTED
        w.resume()
        for h in rep.live_handles():
            assert np.array_equal(w.read(h), rep.buffer(h))
        _, resp2 = w.run(bytes(wire.Builder().sync()))
        assert len(resp2) == 64
