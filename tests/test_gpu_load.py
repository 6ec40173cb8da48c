"""GPU parity tests: everything goes through the C ABI (ctypes) and is compared bit for bit with the oracle."""
import json
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

from kukeon_b200 import gpupool, modelhub
from oracle import oracle
from tests import helpers
from tools import synth

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MB = 1 << 20


def assert_pool_matches(m, device, shards, recs, mode=0, flags=0, n_parts=1, part=0):
    exp, plan = oracle.expected_pool(shards, recs, mode, flags, n_parts, part)
    got = m.read(device, 0, len(exp))
    for p in plan:
        a, b = p["pool_offset"], p["pool_offset"] + p["nbytes"]
        if not np.array_equal(got[a:b], exp[a:b]):
            bad = np.flatnonzero(got[a:b] != exp[a:b])
            raise AssertionError(f"{p['name']} ({p['dtype']} {p['shape']}): {bad.size} bytes differ, first at +{bad[0]}")
    return exp, plan


def load_and_check(pool, path, **kw):
    shards, recs = oracle.index_path(path)
    m = pool.load(path, **kw)
    try:
        assert m.tensors() == recs
        exp, plan = assert_pool_matches(m, pool.devices[0], shards, recs, flags=kw.get("flags", 0))
        for p in plan[:4]:
            assert m.checksum(pool.devices[0], p["pool_offset"], p["nbytes"]) == oracle.checksum(exp[p["pool_offset"]:p["pool_offset"] + p["nbytes"]])
        return m.stats()
    finally:
        m.release()


def test_mixed_safetensors_every_op(pool, tmp_path):
    p = str(tmp_path / "m.safetensors")
    helpers.mixed_safetensors(p)
    st = load_and_check(pool, p)
    assert st["n_loads"] == 1 and st["file_bytes"] == sum(r["nbytes"] for r in oracle.index_path(p)[1])


def test_unpadded_header_exercises_the_misaligned_path(pool, tmp_path):
    # an unpadded header shifts every tensor off 16-byte alignment relative to its neighbours' sizes
    for pad in (False, True):
        p = str(tmp_path / f"m{int(pad)}.safetensors")
        tensors = [("a", "BF16", [7]), ("b", "BF16", [33, 77]), ("c", "F32", [129, 65]), ("d", "F16", [7, 1001]), ("e", "U8", [3]),
                   ("f", "BF16", [4099]), ("g", "F32", [5]), ("h", "F16", [2, 3]), ("i", "U8", [1021]), ("j", "BF16", [64, 512])]
        synth.write_safetensors(p, tensors, 5, pad_header=pad)
        load_and_check(pool, p)


def test_golden_files(pool):
    load_and_check(pool, os.path.join(G, "st_mixed.safetensors"))
    load_and_check(pool, os.path.join(G, "sharded"))
    load_and_check(pool, os.path.join(G, "q4k.gguf"))


def test_golden_q4k_values_vs_gguf_py_fixture(pool):
    p = os.path.join(G, "q4k.gguf")
    outs = np.load(p + ".bf16.npz")
    m = pool.load(p)
    try:
        for name in outs.files:
            pl = m.placements(name)[0]
            got = m.read(0, pl.pool_offset, pl.nbytes).view(np.uint16)
            assert pl.dtype == "BF16" and np.array_equal(got, outs[name]), name
    finally:
        m.release()


# ---- Q4_K_M mixes (Q4_K + Q6_K + Q8_0): value parity of the two most common companions of Q4_K, kept at the front of the suite ----
def test_q4_k_m_style_mixed_quants_q6k_q8_0(pool, tmp_path):
    """Real Q4_K_M GGUFs mix Q4_K with Q6_K (and Q8_0 appears in other presets): bit-exact vs the oracle and vs the
    committed gguf-py fixture."""
    from tests.test_plan import q4km_tensors
    p = str(tmp_path / "q4km.gguf")
    synth.write_gguf(p, q4km_tensors(hidden=512, ffn=1536, layers=2, vocab=1024), 9)
    load_and_check(pool, p)
    g = os.path.join(G, "q4km_mix.gguf")
    load_and_check(pool, g)
    outs = np.load(g + ".bf16.npz")
    m = pool.load(g)
    try:
        for name in outs.files:
            pl = m.placements(name)[0]
            assert np.array_equal(m.read(0, pl.pool_offset, pl.nbytes).view(np.uint16), outs[name]), name
    finally:
        m.release()


def test_gguf_alignment_8_puts_quant_blocks_off_16_byte_boundaries(pool, tmp_path):
    """general.alignment = 8: block-quantised tensors start 8 bytes off a 16-byte boundary, so the kernel's byte-assembled
    shared-memory reads (not the vector ones) feed the dequantisers."""
    from tests.test_plan import q4km_tensors
    p = str(tmp_path / "a8.gguf")
    tensors = [("pad.weight", "F32", [2])] + q4km_tensors(hidden=256, ffn=512, layers=1, vocab=256) + [("tail.weight", "F16", [3])]
    synth.write_gguf(p, tensors, 21, alignment=8)
    recs = gpupool.index(p)
    assert any(r["dtype"] == "Q4_K" and r["file_offset"] % 16 == 8 for r in recs)
    assert any(r["dtype"] == "Q6_K" and r["file_offset"] % 16 == 8 for r in recs)
    load_and_check(pool, p)


def test_q4_k_m_mix_through_the_eight_destination_ladder(native, tmp_path):
    import subprocess
    import sys
    from tests.test_plan import q4km_tensors
    g2 = str(tmp_path / "q4km.gguf")
    synth.write_gguf(g2, q4km_tensors(), 9)
    env = dict(os.environ, KUKEON_GPULOAD_TEST_NDST="8")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", _NDST_CHILD, root, f"{g2}:0"], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-3000:]


def test_q4_k_m_mix_virtual_rank_broadcast(pool, tmp_path):
    from tests.test_plan import q4km_tensors
    g = str(tmp_path / "q4km.gguf")
    synth.write_gguf(g, q4km_tensors(), 9)
    shards, recs = oracle.index_path(g)
    ms = _virtual_ranks(pool, g, gpupool.MODE_BROADCAST, 4, 0)
    try:
        for m in ms:
            m.load_part()
        for m in ms:
            assert_pool_matches(m, 0, shards, recs, flags=0)
    finally:
        for m in ms:
            m.release()


def test_llama_multishard_small_chunks(native, tmp_path):
    d = str(tmp_path / "llama")
    synth.make_llama(d, dict(hidden=256, ffn=704, layers=3, kv_dim=64, vocab=3000), max_shard_bytes=3_000_000)
    with gpupool.Pool([0], n_staging_buffers=4, staging_buffer_bytes=1 * MB, n_reader_threads=2) as pl:
        st = load_and_check(pl, d)
        assert st["parts"][0]["chunks"] >= 4
        load_and_check(pl, d, mode=gpupool.MODE_BROADCAST)  # one device: degenerates to a single load


def test_mixtral_style_gguf_q4k(pool, tmp_path):
    p = str(tmp_path / "mix.gguf")
    synth.write_gguf(p, synth.mixtral_gguf_tensors(hidden=256, ffn=768, layers=2, experts=2, vocab=512, kv_dim=256), 7)
    load_and_check(pool, p)


def test_q4k_many_blocks_vs_c_oracle(pool, tmp_path, coracle):
    p = str(tmp_path / "big.gguf")
    synth.write_gguf(p, [("w", "Q4_K", [2048, 4096]), ("n", "F32", [4096])], 11)  # 32768 blocks, 16 MiB of bf16
    shards, recs = oracle.index_path(p)
    m = pool.load(p)
    try:
        r = [x for x in recs if x["name"] == "w"][0]
        raw = np.fromfile(p, np.uint8, count=r["nbytes"], offset=r["file_offset"])
        want = coracle.q4k_to_bf16(raw).reshape(-1)
        pl = m.placements("w")[0]
        got = m.read(0, pl.pool_offset, pl.nbytes).view(np.uint16)
        assert np.array_equal(got, want)
        assert m.checksum(0, pl.pool_offset, pl.nbytes) == coracle.checksum(want)
    finally:
        m.release()


def test_gpt2_conv1d_transpose(pool, tmp_path):
    p = str(tmp_path / "gpt2.safetensors")
    synth.make_gpt2(p, n_layer=2, d=96, vocab=301, n_pos=40)
    load_and_check(pool, p, flags=gpupool.LOAD_GPT2_CONV1D_T)
    load_and_check(pool, p, flags=gpupool.LOAD_GPT2_CONV1D_T | gpupool.LOAD_KEEP_F32)
    for dt in ("F16", "BF16"):
        q = str(tmp_path / f"gpt2_{dt}.safetensors")
        synth.write_safetensors(q, synth.gpt2_tensors(n_layer=1, d=40, vocab=50, n_pos=8, dtype=dt), 3)
        load_and_check(pool, q, flags=gpupool.LOAD_GPT2_CONV1D_T)
    for dt, d in (("F32", 41), ("F16", 43), ("BF16", 37)):  # rows that are not 16-byte multiples: direct-global path
        q = str(tmp_path / f"gpt2_{dt}_{d}.safetensors")
        synth.write_safetensors(q, synth.gpt2_tensors(n_layer=2, d=d, vocab=50, n_pos=8, dtype=dt), 3)
        load_and_check(pool, q, flags=gpupool.LOAD_GPT2_CONV1D_T)


def test_special_values_nan_inf_subnormal(pool, tmp_path):
    v = np.load(os.path.join(G, "cast_vectors.npz"))
    f32 = np.concatenate([v["f32_in"], np.array([0x7FC00000, 0xFFC00000, 0x7F800001, 0xFFFFFFFF, 0x7F800000, 0xFF800000], np.uint32)])
    f16 = np.arange(0, 1 << 16, dtype=np.uint16)  # every half, NaNs included
    bf = np.arange(0, 1 << 16, dtype=np.uint16)   # every bf16 pattern must pass through verbatim
    hdr, data, off = {}, b"", 0
    for name, dt, arr in (("f32", "F32", f32), ("f16", "F16", f16), ("bf16", "BF16", bf)):
        raw = arr.tobytes()
        hdr[name] = {"dtype": dt, "shape": [len(arr)], "data_offsets": [off, off + len(raw)]}
        data += raw
        off += len(raw)
    p = str(tmp_path / "special.safetensors")
    helpers.write_raw_safetensors(p, hdr, data)
    m = pool.load(p)
    try:
        g = lambda n: m.read(0, m.placements(n)[0].pool_offset, m.placements(n)[0].nbytes).view(np.uint16)
        assert np.array_equal(g("f32"), oracle.f32_bits_to_bf16(f32))
        assert np.array_equal(g("f16"), oracle.f16_bits_to_bf16(f16))
        assert np.array_equal(g("bf16"), bf)
    finally:
        m.release()
    # Q4_K with non-finite / zero / subnormal super-block scales
    blocks = np.frombuffer(np.random.default_rng(1).bytes(144 * 64), np.uint8).reshape(64, 144).copy()
    specials = [0x7C00, 0xFC00, 0x7E00, 0x0000, 0x8000, 0x0001, 0x7BFF, 0x03FF]
    for i, s in enumerate(specials):
        blocks[i, 0:2] = np.array([s], "<u2").view(np.uint8)
        blocks[8 + i, 2:4] = np.array([s], "<u2").view(np.uint8)
    q = str(tmp_path / "special.gguf")
    import struct
    head = struct.pack("<IIQQ", 0x46554747, 3, 1, 0) + struct.pack("<Q", 1) + b"w" + struct.pack("<I", 2) + struct.pack("<2Q", 256, 64) + struct.pack("<IQ", 12, 0)
    head += b"\0" * ((-len(head)) % 32)
    open(q, "wb").write(head + blocks.tobytes())
    m = pool.load(q)
    try:
        pl = m.placements("w")[0]
        got = m.read(0, pl.pool_offset, pl.nbytes).view(np.uint16).reshape(64, 256)
        assert np.array_equal(got, oracle.dequant_q4k_bf16(blocks))
    finally:
        m.release()


def test_eight_concurrent_sessions_share_one_load(pool, tmp_path):
    d = str(tmp_path / "llama")
    synth.make_llama(d, dict(hidden=128, ffn=352, layers=2, kv_dim=32, vocab=1000), max_shard_bytes=10_000_000)
    out, errs = [None] * 8, []

    def session(i):
        try:
            out[i] = pool.load(d)
        except Exception as e:  # noqa: BLE001
            errs.append(e)

    th = [threading.Thread(target=session, args=(i,)) for i in range(8)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errs
    assert len({m.handle for m in out}) == 1, "all sessions must get the same resident model"
    info = out[0].info()
    assert info["refcount"] == 8 and info["loaded"] and out[0].stats()["n_loads"] == 1
    hooks = modelhub.CellHooks(out[0])
    hooks.start_cell("cell-a"); hooks.start_cell("cell-a"); hooks.start_cell("cell-b")
    assert out[0].info()["refcount"] == 10 and hooks.active == 2
    hooks.stop_cell("cell-a"); hooks.stop_cell("cell-a"); hooks.stop_cell("cell-b")
    assert out[0].info()["refcount"] == 8
    with pytest.raises(gpupool.ErrBusy):
        pool.close()
    for m in out[:-1]:
        m.release()
    assert out[-1].info()["refcount"] == 1
    shards, recs = oracle.index_path(d)
    assert_pool_matches(out[-1], 0, shards, recs)  # still resident and intact
    out[-1].release()
    m2 = pool.load(d)  # a fresh load after the last release
    assert m2.stats()["n_loads"] == 1
    m2.release()


_CHILD = r'''
import sys, json, numpy as np
from cuda.bindings import runtime as cudart
hpath, off, n, want_uuid = sys.argv[1], int(sys.argv[2]), int(sys.argv[3]), sys.argv[4]
h = cudart.cudaIpcMemHandle_t(); h.reserved = open(hpath, "rb").read()
# the agent finds the GPU by the UUID the daemon exported (KUKEON_GPUPOOL_DEVICE_UUID), not by the daemon's ordinal
err, cnt = cudart.cudaGetDeviceCount(); assert err == 0, err
dev = None
for i in range(cnt):
    err, pr = cudart.cudaGetDeviceProperties(i); assert err == 0, err
    b = bytes(pr.uuid.bytes)
    u = "GPU-%s-%s-%s-%s-%s" % (b[0:4].hex(), b[4:6].hex(), b[6:8].hex(), b[8:10].hex(), b[10:16].hex())
    if u == want_uuid: dev = i
assert dev is not None, ("no device with uuid", want_uuid)
err, = cudart.cudaSetDevice(dev); assert err == 0, err
err, ptr = cudart.cudaIpcOpenMemHandle(h, cudart.cudaIpcMemLazyEnablePeerAccess); assert err == 0, err
buf = np.empty(n, np.uint8)
err, = cudart.cudaMemcpy(buf.ctypes.data, ptr + off, n, cudart.cudaMemcpyKind.cudaMemcpyDeviceToHost); assert err == 0, err
sys.stdout.write(buf.tobytes().hex())
cudart.cudaIpcCloseMemHandle(ptr)
'''


def test_mount_exports_manifest_and_ipc_handle_to_another_process(pool, tmp_path):
    p = str(tmp_path / "m.safetensors")
    helpers.mixed_safetensors(p)
    shards, recs = oracle.index_path(p)
    m = pool.load(p)
    try:
        spec = modelhub.Mount(m, 0, str(tmp_path / "cell" / "container"))
        man = json.load(open(os.path.join(spec.host_dir, "manifest.json")))
        want, total = oracle.plan_pool(recs)
        assert man["kind"] == "PoolManifest" and man["poolBytes"] == total and man["device"] == 0
        for w, g in zip(want, man["tensors"]):
            assert (g["name"], g["dtype"], g["shape"], g["offset"], g["nbytes"]) == (w["name"], w["dtype"], w["shape"], w["pool_offset"], w["nbytes"])
        assert spec.mounts == [{"destination": "/run/kukeon/gpupool", "type": "bind", "source": spec.host_dir, "options": ["rbind", "ro"]}]
        assert any(e.startswith("KUKEON_GPUPOOL_MANIFEST=") for e in spec.env)
        ident = gpupool.device_identity(0)
        env = dict(e.split("=", 1) for e in spec.env)
        assert env["KUKEON_GPUPOOL_DEVICE_UUID"] == ident["uuid"] == man["deviceUUID"] and ident["uuid"].startswith("GPU-") and len(ident["uuid"]) == 40
        assert env["KUKEON_GPUPOOL_PCI_BUS_ID"] == ident["pci_bus_id"] == man["pciBusId"]
        if os.path.exists(os.path.join(modelhub.NVIDIA_PROC_GPUS, ident["pci_bus_id"], "information")):  # device node from the driver's table, not from the ordinal
            minor = modelhub.device_minor(ident["pci_bus_id"])
            wd = modelhub.Mount(m, 0, str(tmp_path / "cell" / "container2"), with_devices=True)
            assert f"/dev/nvidia{minor}" in [d["path"] for d in wd.devices] and "/dev/nvidiactl" in [d["path"] for d in wd.devices]
        else:  # a container can mask the driver's table (the directory present, this GPU's entry absent): no node is guessed then
            with pytest.raises(FileNotFoundError):
                modelhub.Mount(m, 0, str(tmp_path / "cell" / "container2"), with_devices=True)
        assert os.path.getsize(os.path.join(spec.host_dir, "ipc.handle")) == 64
        t = want[7]  # h.bf16.big
        r = subprocess.run([sys.executable, "-c", _CHILD, os.path.join(spec.host_dir, "ipc.handle"), str(t["pool_offset"]), "4096", ident["uuid"]],
                           capture_output=True, text=True, timeout=120)
        assert r.returncode == 0, r.stderr[-2000:]
        exp, _ = oracle.expected_pool(shards, recs)
        assert bytes.fromhex(r.stdout) == exp[t["pool_offset"]:t["pool_offset"] + 4096].tobytes()
    finally:
        m.release()


def test_resident_convert_equals_streaming_load(native, tmp_path):
    d = str(tmp_path / "llama")
    synth.make_llama(d, dict(hidden=256, ffn=704, layers=3, kv_dim=64, vocab=3000), max_shard_bytes=3_000_000)
    shards, recs = oracle.index_path(d)
    with gpupool.Pool([0], n_staging_buffers=2, staging_buffer_bytes=1 * MB, n_reader_threads=1) as pl:
        m = pl.load(d, flags=gpupool.LOAD_DEFER)
        try:
            assert not m.info()["loaded"]
            m.stage_resident()
            tot, per = m.convert_resident()
            assert tot > 0 and len(per) == len(shards), "one launch per shard"
            assert_pool_matches(m, 0, shards, recs)
            m.unstage_resident()
            with pytest.raises(gpupool.ErrState):
                m.convert_resident()
            m.load_part()
            assert m.info()["loaded"]
            assert_pool_matches(m, 0, shards, recs)
        finally:
            m.release()


def test_zero_copy_staging_matches(native, tmp_path):
    p = str(tmp_path / "m.safetensors")
    helpers.mixed_safetensors(p)
    with gpupool.Pool([0], n_staging_buffers=2, staging_buffer_bytes=2 * MB, n_reader_threads=1, flags=gpupool.CFG_ZEROCOPY) as pl:
        load_and_check(pl, p)
        load_and_check(pl, os.path.join(G, "q4k.gguf"))


def test_medium_checkpoint_checksum_of_checksums(native, tmp_path, coracle):
    """~1 GB bf16 llama slice: size-independent property — the pool's device-side checksum per tensor equals the
    oracle checksum of the file bytes (passthrough), and a checksum over the per-tensor checksums agrees."""
    shm = "/dev/shm" if os.path.isdir("/dev/shm") else str(tmp_path)
    d = os.path.join(shm, f"kk_medium_{os.getpid()}")
    try:
        synth.make_llama(d, dict(hidden=2048, ffn=5632, layers=6, kv_dim=512, vocab=32000), max_shard_bytes=300_000_000)
        shards, recs = oracle.index_path(d)
        with gpupool.Pool([0]) as pl:
            m = pl.load(d)
            try:
                sums_gpu, sums_cpu = [], []
                for r in recs:
                    p = m.placements(r["name"])[0]
                    sums_gpu.append(m.checksum(0, p.pool_offset, p.nbytes))
                    raw = np.fromfile(shards[r["shard"]], np.uint8, count=r["nbytes"], offset=r["file_offset"])
                    sums_cpu.append(coracle.checksum(raw))
                assert sums_gpu == sums_cpu
                assert oracle.checksum(np.array(sums_gpu, np.uint64)) == oracle.checksum(np.array(sums_cpu, np.uint64))
                st = m.stats()
                assert st["file_bytes"] == sum(r["nbytes"] for r in recs) and st["load_gbps"] > 0
            finally:
                m.release()
    finally:
        import shutil
        shutil.rmtree(d, ignore_errors=True)


@pytest.mark.skipif(not os.path.isdir("/dev/shm"), reason="the mapped read path is the default for shards on tmpfs only")
def test_tmpfs_shards_take_the_mapped_streaming_read_path_bit_exact(pool, coracle):
    """Shards on tmpfs are read through a mapping with streaming stores and per-range MADV_DONTNEED (kk_loader.cpp read_chunk), everything else with
    pread: both must produce the same pool.  An unpadded header puts every range off page and 32-byte boundaries; tensors of 3 B .. 9 MB mix the
    long (> 256 KiB, mapped) and short (pread) ranges in one chunk."""
    d = f"/dev/shm/kk_mapped_{os.getpid()}"
    os.makedirs(d, exist_ok=True)
    try:
        p = os.path.join(d, "m.safetensors")
        tensors = [("a", "BF16", [7]), ("b", "BF16", [1537, 3001]), ("c", "F32", [1025, 513]), ("d", "U8", [3]), ("e", "F16", [999, 1001]),
                   ("f", "BF16", [300_001]), ("g", "F32", [5]), ("h", "BF16", [2048, 1024]), ("i", "U8", [1021])]
        synth.write_safetensors(p, tensors, 11, pad_header=False)
        st = load_and_check(pool, p)
        assert st["n_loads"] == 1
        shards, recs = oracle.index_path(p)
        m = pool.load(p)
        try:
            sums = [m.checksum(pool.devices[0], pl.pool_offset, pl.nbytes) for pl in (m.placements(r["name"])[0] for r in recs)]
        finally:
            m.release()
        code = ("import sys, json; sys.path.insert(0, %r)\n"
                "from kukeon_b200 import gpupool\n"
                "with gpupool.Pool([0]) as pl:\n"
                "    m = pl.load(%r)\n"
                "    print(json.dumps([m.checksum(0, q.pool_offset, q.nbytes) for q in (m.placements(t['name'])[0] for t in m.tensors())]))\n"
                "    m.release()\n") % (os.path.dirname(G[:-len('/golden')]), p)
        for mode in ("pread", "mapped"):
            out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, KUKEON_GPULOAD_READ=mode), capture_output=True, text=True, timeout=300)
            assert out.returncode == 0, out.stderr[-2000:]
            assert json.loads(out.stdout.strip().splitlines()[-1]) == sums, mode
    finally:
        import shutil
        shutil.rmtree(d, ignore_errors=True)


def _shm_free() -> int:
    try:
        st = os.statvfs("/dev/shm")
        return st.f_bavail * st.f_frsize
    except OSError:
        return 0


@pytest.mark.skipif(_shm_free() < 40 << 30, reason="needs ~20 GB of /dev/shm for the full-size checkpoint")
def test_full_size_llama3_8b_round_trip_properties(native, coracle):
    """BASELINE config 2 at its full size (291 tensors, 16,060,522,496 B): index == oracle, every tensor's
    device-side checksum == oracle checksum of the file bytes (bf16 passthrough is the identity), a checksum
    of checksums ties it together, and a second load (idempotence) leaves the pool bit-identical."""
    import shutil
    d = f"/dev/shm/kk_full8b_{os.getpid()}"
    try:
        synth.make_llama(d, synth.LLAMA3_8B)
        shards, recs = oracle.index_path(d)
        assert len(recs) == 291 and len(shards) == 4 and sum(r["nbytes"] for r in recs) == 16_060_522_496
        assert gpupool.index(d) == recs
        with gpupool.Pool([0]) as pl:
            m = pl.load(d)
            try:
                assert m.info()["pool_bytes"] == 16_060_522_496  # every slot already 256-aligned: no padding
                gpu_sums = [m.checksum(0, p.pool_offset, p.nbytes) for p in (m.placements(r["name"])[0] for r in recs)]
                cpu_sums = []
                for r in recs:
                    mm = np.memmap(shards[r["shard"]], np.uint8, "r", offset=r["file_offset"], shape=(r["nbytes"],))
                    cpu_sums.append(coracle.checksum(mm))
                    del mm
                assert gpu_sums == cpu_sums
                whole = m.checksum(0, 0, 16_060_522_496)
                m.load_part()  # idempotence: loading again must not change a byte
                assert m.checksum(0, 0, 16_060_522_496) == whole
                assert oracle.checksum(np.array(gpu_sums, np.uint64)) == oracle.checksum(np.array(cpu_sums, np.uint64))
            finally:
                m.release()
    finally:
        shutil.rmtree(d, ignore_errors=True)


@pytest.mark.skipif(_shm_free() < 40 << 30, reason="needs /dev/shm for the checkpoint")
def test_large_q4k_linearity_and_checksum(native, coracle):
    """Mixtral-shaped GGUF (2 layers, ~1.7 GB of Q4_K blocks -> ~6 GB bf16): device checksum of every dequantised
    tensor == checksum of the C oracle's output for it."""
    import shutil
    p = f"/dev/shm/kk_q4k_{os.getpid()}.gguf"
    try:
        synth.write_gguf(p, synth.mixtral_gguf_tensors(layers=2), 8007)
        shards, recs = oracle.index_path(p)
        with gpupool.Pool([0]) as pl:
            m = pl.load(p)
            try:
                checked = 0
                for r in recs:
                    if r["dtype"] != "Q4_K" or r["nbytes"] > 600 << 20:
                        continue
                    raw = np.fromfile(p, np.uint8, count=r["nbytes"], offset=r["file_offset"])
                    want = coracle.checksum(coracle.q4k_to_bf16(raw))
                    q = m.placements(r["name"])[0]
                    assert m.checksum(0, q.pool_offset, q.nbytes) == want, r["name"]
                    checked += 1
                assert checked >= 10
            finally:
                m.release()
    finally:
        if os.path.exists(p):
            os.remove(p)


_NDST_CHILD = r'''
import os, sys
sys.path.insert(0, sys.argv[1])
import numpy as np
from kukeon_b200 import gpupool
from oracle import oracle
paths = sys.argv[2:]
with gpupool.Pool([0], n_staging_buffers=2, staging_buffer_bytes=1 << 20, n_reader_threads=1) as pl:
    for spec in paths:
        path, flags = spec.rsplit(":", 1)
        flags = int(flags)
        shards, recs = oracle.index_path(path)
        m = pl.load(path, flags=flags)
        try:
            exp, plan = oracle.expected_pool(shards, recs, 0, flags)
            got = m.read(0, 0, len(exp))
            for p in plan:
                a, b = p["pool_offset"], p["pool_offset"] + p["nbytes"]
                assert np.array_equal(got[a:b], exp[a:b]), f"n_dst={os.environ['KUKEON_GPULOAD_TEST_NDST']}: {p['name']} differs"
            m.stage_resident(); m.convert_resident()
            got = m.read(0, 0, len(exp))
            for p in plan:
                a, b = p["pool_offset"], p["pool_offset"] + p["nbytes"]
                assert np.array_equal(got[a:b], exp[a:b]), f"resident n_dst={os.environ['KUKEON_GPULOAD_TEST_NDST']}: {p['name']} differs"
        finally:
            m.release()
print("ok")
'''


@pytest.mark.parametrize("ndst", [3, 8])
def test_multi_destination_store_paths_on_one_gpu(native, tmp_path, ndst):
    """The fused fan-out stores every output vector to n_dst pools.  KUKEON_GPULOAD_TEST_NDST aliases the extra
    destinations onto the local pool so every op's n-destination path (incl. 8 = a full HGX box) runs on one GPU."""
    d = str(tmp_path / "llama")
    synth.make_llama(d, dict(hidden=256, ffn=704, layers=2, kv_dim=64, vocab=3000), max_shard_bytes=3_000_000)
    mixed = str(tmp_path / "m.safetensors")
    helpers.mixed_safetensors(mixed, pad_header=False)
    g = str(tmp_path / "mix.gguf")
    synth.write_gguf(g, synth.mixtral_gguf_tensors(hidden=256, ffn=768, layers=1, experts=2, vocab=512, kv_dim=256), 7)
    f = str(tmp_path / "gpt2.safetensors")
    synth.make_gpt2(f, n_layer=2, d=96, vocab=301, n_pos=40)
    f2 = str(tmp_path / "gpt2_odd.safetensors")
    synth.write_safetensors(f2, synth.gpt2_tensors(n_layer=1, d=40, vocab=50, n_pos=8, dtype="F16"), 3)
    f3 = str(tmp_path / "gpt2_d41.safetensors")  # rows of 41/123/164 elements: not 16-byte multiples -> direct-global transpose path
    synth.write_safetensors(f3, synth.gpt2_tensors(n_layer=2, d=41, vocab=50, n_pos=8), 4)
    env = dict(os.environ, KUKEON_GPULOAD_TEST_NDST=str(ndst))
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", _NDST_CHILD, root, f"{d}:0", f"{mixed}:0", f"{g}:0", f"{f}:1", f"{f}:3", f"{f2}:1", f"{f3}:1", f"{f3}:3"],
                       capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-3000:]


def test_raw_fanout_degenerates_on_one_gpu(pool, tmp_path):
    """KK_FANOUT_RAW = gather the file bytes into a raw image, then convert locally.  On one GPU there is nobody to
    gather from, but both stages (H2D into the image, convert from the image) still run and must match the oracle."""
    g = str(tmp_path / "mix.gguf")
    synth.write_gguf(g, synth.mixtral_gguf_tensors(hidden=256, ffn=768, layers=2, experts=2, vocab=512, kv_dim=256), 7)
    load_and_check(pool, g, mode=gpupool.MODE_BROADCAST, fanout=gpupool.FANOUT_RAW)
    p = str(tmp_path / "m.safetensors")
    helpers.mixed_safetensors(p)
    load_and_check(pool, p, mode=gpupool.MODE_BROADCAST, fanout=gpupool.FANOUT_RAW)
    with pytest.raises(gpupool.ErrInvalid):
        pool.load(p, mode=gpupool.MODE_SINGLE, fanout=gpupool.FANOUT_RAW)
    # deferred flavour (what bench.py drives): stage 1, then kk_convert_local
    shards, recs = oracle.index_path(g)
    m = pool.load(g, mode=gpupool.MODE_BROADCAST, fanout=gpupool.FANOUT_RAW, flags=gpupool.LOAD_DEFER)
    try:
        m.load_part()
        m.convert_local()
        assert_pool_matches(m, 0, shards, recs)
        m.stage_resident()
        tot, per = m.convert_resident()  # no peers: nothing to fan out
        assert per == [] and m.convert_local() > 0
        assert_pool_matches(m, 0, shards, recs)
    finally:
        m.release()


def _virtual_ranks(pool, path, mode, n, flags=0):
    """N ranks hosted by ONE process on ONE GPU: rank i = model (part i of n); pools attached to each other by raw
    device pointer (KK_BUF_POOL_PTR).  Runs the real multi-rank kernels (fused fan-out, row-split exchange)."""
    ms = [pool.load(path, mode=mode, fanout=gpupool.FANOUT_P2P, flags=flags | gpupool.LOAD_DEFER, part_index=i, part_count=n) for i in range(n)]
    assert len({m.handle for m in ms}) == n
    ptrs = [m.pool_ptr(0)[0] for m in ms]
    need_peers = mode == gpupool.MODE_BROADCAST or (flags & gpupool.LOAD_SCATTER_EXCHANGE)
    if need_peers:
        for i, m in enumerate(ms):
            for j in range(n):
                if j != i:
                    m.peer_attach_local_pointer(j, ptrs[j])
    return ms


@pytest.mark.parametrize("n", [2, 4, 8])
def test_virtual_ranks_broadcast_on_one_gpu(pool, tmp_path, n):
    d = str(tmp_path / "llama")
    synth.make_llama(d, dict(hidden=256, ffn=704, layers=2, kv_dim=64, vocab=3000), max_shard_bytes=3_000_000)
    g = str(tmp_path / "q4k.gguf")  # Q4_K + F32 here; the Q4_K_M mix (Q6_K, Q8_0) runs the same way in test_q4_k_m_mix_virtual_rank_broadcast
    synth.write_gguf(g, synth.mixtral_gguf_tensors(hidden=256, ffn=768, layers=2, experts=2, vocab=512, kv_dim=256), 9)
    f = str(tmp_path / "gpt2.safetensors")
    synth.make_gpt2(f, n_layer=2, d=96, vocab=301, n_pos=40)
    for path, flags in ((d, 0), (g, 0), (f, gpupool.LOAD_GPT2_CONV1D_T)):
        shards, recs = oracle.index_path(path)
        ms = _virtual_ranks(pool, path, gpupool.MODE_BROADCAST, n, flags)
        try:
            for m in ms:
                m.load_part()  # rank i converts its 1/n and stores it into all n pools
            for m in ms:
                assert_pool_matches(m, 0, shards, recs, flags=flags)
            for m in ms:       # and again from the resident image (what bench.py times)
                m.stage_resident()
            for m in ms:
                m.convert_resident()
            for m in ms:
                assert_pool_matches(m, 0, shards, recs, flags=flags)
        finally:
            for m in ms:
                m.release()


@pytest.mark.parametrize("n", [2, 4, 8])
def test_virtual_ranks_scatter_exchange_on_one_gpu(pool, tmp_path, n):
    """KK_LOAD_SCATTER_EXCHANGE: rank i ingests whole rows of the row-parallel tensors and the KK_OP_ROWSPLIT tiles deal
    every row's column slices to the n pools; every rank's pool must equal its oracle slice pool."""
    d = str(tmp_path / "llama")
    synth.make_llama(d, dict(hidden=512, ffn=1408, layers=2, kv_dim=128, vocab=2048), max_shard_bytes=6_000_000)
    shards, recs = oracle.index_path(d)
    for flags in (gpupool.LOAD_SCATTER_EXCHANGE, 0):
        ms = _virtual_ranks(pool, d, gpupool.MODE_SCATTER, n, flags)
        try:
            for m in ms:
                m.load_part()
            for i, m in enumerate(ms):
                assert_pool_matches(m, 0, shards, recs, mode=gpupool.MODE_SCATTER, n_parts=n, part=i)
            if flags:
                for m in ms:
                    m.stage_resident()
                for m in ms:
                    m.convert_resident()
                for i, m in enumerate(ms):
                    assert_pool_matches(m, 0, shards, recs, mode=gpupool.MODE_SCATTER, n_parts=n, part=i)
                st = ms[0].stats()
                assert st["local_src_bytes"] < st["file_bytes"] / n * 1.1 + (1 << 20)
        finally:
            for m in ms:
                m.release()
    # without the peers attached an exchange load must refuse, not silently drop the slices of other ranks
    m = pool.load(d, mode=gpupool.MODE_SCATTER, flags=gpupool.LOAD_SCATTER_EXCHANGE | gpupool.LOAD_DEFER, part_index=0, part_count=n)
    try:
        with pytest.raises(gpupool.ErrState, match="not reachable"):
            m.load_part()
    finally:
        m.release()


def test_concurrent_loads_of_different_checkpoints_share_the_staging_ring_safely(pool, tmp_path):
    """Several cells starting at once with DIFFERENT models: the loads share one device's pinned ring and must not
    trample each other's slots (they serialise on the device's pipeline lock)."""
    paths = []
    for i in range(4):
        d = str(tmp_path / f"llama{i}")
        synth.make_llama(d, dict(hidden=256, ffn=704, layers=2, kv_dim=64, vocab=1500 + 100 * i), seed=100 + i, max_shard_bytes=3_000_000)
        paths.append(d)
    g = str(tmp_path / "mix.gguf")
    synth.write_gguf(g, synth.mixtral_gguf_tensors(hidden=256, ffn=768, layers=1, experts=2, vocab=512, kv_dim=256), 7)
    paths.append(g)
    out, errs = [None] * len(paths), []

    def session(i):
        try:
            out[i] = pool.load(paths[i])
        except Exception as e:  # noqa: BLE001
            errs.append(e)

    th = [threading.Thread(target=session, args=(i,)) for i in range(len(paths))]
    [t.start() for t in th]
    [t.join() for t in th]
    try:
        assert not errs, errs
        assert len({m.handle for m in out}) == len(paths)
        for p, m in zip(paths, out):
            shards, recs = oracle.index_path(p)
            assert_pool_matches(m, 0, shards, recs)
    finally:
        for m in out:
            if m is not None:
                m.release()
