"""f3 (SURVEY.md §8(f)): the `models:` manifest schema and the in-process `kuke model` verbs — table-driven in the style of the
reference's validateVolumes tests (internal/controller/create_container_test.go) and `kuke image` tests (cmd/kuke/image/*_test.go)."""
import io
import json
import os

import pytest
import yaml

from kukeon_b200 import cli, gpupool, schema
from kukeon_b200.schema import Err, SchemaError, validate_models
from tools import synth

TD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "testdata")


@pytest.fixture()
def models_dir(native, tmp_path):
    synth.make_llama(str(tmp_path / "llama"), dict(hidden=64, ffn=176, layers=1, kv_dim=16, vocab=100), max_shard_bytes=10_000_000)
    synth.make_gpt2(str(tmp_path / "gpt2.safetensors"), n_layer=1, d=32, vocab=50, n_pos=8)
    return str(tmp_path)


def test_validate_models_accepts_and_normalises(models_dir):
    specs = schema.validate_models([
        {"name": " llama ", "source": f" {models_dir}/llama ", "mode": "Broadcast", "devices": [1, 0]},
        {"name": "gpt2", "source": f"{models_dir}/gpt2.safetensors", "target": "/weights", "options": {"gpt2Conv1dTranspose": True, "keepF32": False, "f8ToBf16": True}},
    ])
    assert [(s.name, s.mode, s.devices, s.target) for s in specs] == [("llama", gpupool.MODE_BROADCAST, [1, 0], schema.DEFAULT_TARGET), ("gpt2", gpupool.MODE_SINGLE, [], "/weights")]
    assert specs[0].source == f"{models_dir}/llama"
    assert specs[1].flags == gpupool.LOAD_GPT2_CONV1D_T | gpupool.LOAD_F8_TO_BF16
    assert schema.validate_models(None) == [] and schema.validate_models([]) == []


@pytest.mark.parametrize("entry,sentinel,detail", [
    ({"source": "/x"}, Err.ModelNameRequired, "model[0]"),
    ({"name": "a"}, Err.ModelSourceRequired, "model[0]"),
    ({"name": "a", "source": "   "}, Err.ModelSourceRequired, "model[0]"),
    ({"name": "a", "source": "llama"}, Err.ModelSourceNotAbsolute, 'model[0] source "llama"'),
    ({"name": "a", "source": "meta-llama/Llama-3-8B"}, Err.ModelRegistryNotSupported, 'model[0] source "meta-llama/Llama-3-8B"'),
    ({"name": "a", "source": "hf://meta-llama/Llama-3-8B"}, Err.ModelRegistryNotSupported, "hf://"),
    ({"name": "a", "source": "/no/such/checkpoint"}, Err.ModelSourceNotFound, 'model[0] source "/no/such/checkpoint"'),
    ({"name": "a", "source": "/", "target": "weights"}, Err.ModelTargetNotAbsolute, 'model[0] target "weights"'),
    ({"name": "a", "source": "/", "mode": "replicate"}, Err.ModelModeUnknown, 'model[0] mode "replicate"'),
    ({"name": "a", "source": "/", "devices": [0, 0]}, Err.ModelDevicesInvalid, "model[0] devices"),
    ({"name": "a", "source": "/", "devices": [-1]}, Err.ModelDevicesInvalid, "model[0] devices"),
    ({"name": "a", "source": "/", "devices": [True]}, Err.ModelDevicesInvalid, "model[0] devices"),
    ({"name": "a", "source": "/", "devices": list(range(9))}, Err.ModelDevicesInvalid, "model[0] devices"),
    ({"name": "a", "source": "/", "options": {"fp4": True}}, Err.ModelOptionUnknown, 'model[0] option "fp4"'),
])
def test_validate_models_rejections_carry_sentinel_index_and_value(entry, sentinel, detail):
    with pytest.raises(schema.SchemaError) as ei:
        schema.validate_models([entry])
    assert ei.value.sentinel == sentinel and str(ei.value).startswith(sentinel + " (") and detail in str(ei.value)


def test_duplicate_names_and_index_of_the_offender():
    with pytest.raises(schema.SchemaError) as ei:
        schema.validate_models([{"name": "a", "source": "/"}, {"name": "b", "source": "/"}, {"name": "a", "source": "/"}])
    assert ei.value.sentinel == Err.ModelNameDuplicate and 'model[2] name "a"' in str(ei.value)


def load_manifest(models_dir):
    text = open(os.path.join(TD, "cell_with_models.yaml")).read().replace("__MODELS__", models_dir)
    return text, yaml.safe_load(text)


@pytest.mark.parametrize("bad", ["../escape", "a/b", "..", ".", ".hidden", "nul\0byte", "sp ace", "semi;colon"])
def test_model_names_that_could_leave_the_cell_directory_are_refused(bad):
    """models[].name becomes <cell dir>/gpupool/<name> on the host and a mount target in the container (ADVICE r1: path traversal): one path
    component of [A-Za-z0-9._-], refused at validation time — before anything is loaded or a refcount is taken."""
    with pytest.raises(SchemaError) as ei:
        validate_models([{"name": bad, "source": "/x"}], stat=lambda p: None)
    assert ei.value.sentinel == Err.ModelNameInvalid and "model[0]" in str(ei.value)


def test_cell_manifest_models_per_container(models_dir):
    _, doc = load_manifest(models_dir)
    got = schema.models_of_cell(doc)
    assert list(got) == ["work"] and [s.name for s in got["work"]] == ["llama", "gpt2"]
    assert got["work"][0].mode == gpupool.MODE_BROADCAST and got["work"][0].devices == [0, 1]
    assert got["work"][1].flags == gpupool.LOAD_GPT2_CONV1D_T
    doc["spec"]["containers"][1]["models"][1]["source"] = "gpt2.safetensors"
    with pytest.raises(schema.SchemaError) as ei:
        schema.models_of_cell(doc)
    assert ei.value.sentinel == Err.ModelSourceNotAbsolute and 'container "work": model[1] source "gpt2.safetensors"' in str(ei.value)
    with pytest.raises(ValueError, match="expected kind Cell"):
        schema.models_of_cell({"kind": "Realm"})


def run(argv):
    out = io.StringIO()
    rc = cli.main(argv, out)
    return rc, out.getvalue()


def test_model_pull_table_json_yaml(models_dir):
    rc, text = run(["model", "pull", f"{models_dir}/llama"])
    lines = text.splitlines()
    assert rc == 0 and lines[0].split() == ["NAME", "DTYPE", "SHAPE", "SHARD", "SIZE"]
    assert any(l.split()[:3] == ["model.embed_tokens.weight", "BF16", "100x64"] for l in lines)
    assert lines[-1].startswith("12 tensors, 1 shard(s), ")
    rc, text = run(["model", "pull", f"{models_dir}/llama", "-o", "json"])
    doc = json.loads(text)
    assert rc == 0 and doc["tensors"] == gpupool.index(f"{models_dir}/llama") and len(doc["shards"]) == 1
    rc, text = run(["model", "pull", f"{models_dir}/gpt2.safetensors", "-o", "yaml"])
    assert rc == 0 and yaml.safe_load(text)["tensors"][0]["dtype"] == "F32"
    with pytest.raises(SystemExit, match="invalid output format: xml"):
        run(["model", "pull", f"{models_dir}/llama", "-o", "xml"])


def test_model_plan_summarises_bytes_per_gpu(models_dir):
    rc, text = run(["model", "plan", f"{models_dir}/llama", "--mode", "broadcast", "--gpus", "4", "-o", "json"])
    doc = json.loads(text)
    assert rc == 0 and doc["gpus"] == 4 and len(doc["ingestBytesPerGpu"]) == 4
    assert sum(doc["ingestBytesPerGpu"]) == doc["fileBytes"] and len(set(doc["poolBytesPerGpu"])) == 1
    rc, text = run(["model", "plan", f"{models_dir}/llama", "--mode", "scatter", "--gpus", "2", "-o", "json"])
    sc = json.loads(text)
    assert rc == 0 and max(sc["poolBytesPerGpu"]) < doc["poolBytesPerGpu"][0]
    rc, text = run(["model", "plan", f"{models_dir}/gpt2.safetensors", "--option", "gpt2Conv1dTranspose"])
    assert rc == 0 and text.splitlines()[0].split() == ["GPU", "INGESTS", "POOL"]
    rc, text = run(["model", "plan", f"{models_dir}/llama", "--mode", "broadcast", "--gpus", "2", "--full", "-o", "json"])
    assert rc == 0 and "parts" in json.loads(text)


def test_model_validate_and_errors(models_dir, tmp_path, capsys):
    text, _ = load_manifest(models_dir)
    mf = tmp_path / "cell.yaml"
    mf.write_text(text)
    rc, out = run(["model", "validate", str(mf)])
    assert rc == 0 and out.splitlines()[-1] == "2 model(s) valid" and "model llama: 12 tensors" in out
    mf.write_text(text.replace("mode: broadcast", "mode: everywhere"))
    rc, _ = run(["model", "validate", str(mf)])
    assert rc == 1 and Err.ModelModeUnknown in capsys.readouterr().err
    rc, _ = run(["model", "pull", str(tmp_path / "missing.gguf")])
    assert rc == 1 and "KK_ENOENT" in capsys.readouterr().err
    rc, _ = run(["model", "ls"])
    assert rc == 2 and "kukeond" in capsys.readouterr().err


def test_format_size_matches_the_reference_helper():
    assert [cli.format_size(n) for n in (-1, 0, 1023, 1024, 1536, 16060522496)] == ["-", "0 B", "1023 B", "1.0 KiB", "1.5 KiB", "15.0 GiB"]


class _StubModel:
    """Mount only needs export(device) -> (64-byte handle, manifest dict)."""

    def __init__(self, tag):
        self.tag = tag

    def export(self, device):
        return bytes([self.tag]) * 64, {"apiVersion": "kukeon.gpupool/v1", "device": device, "deviceUUID": f"GPU-0000000{device}-aaaa-bbbb-cccc-dddddddddddd",
                                        "pciBusId": f"0000:{0x1b + device:02x}:00.0", "tensors": [{"name": f"w{self.tag}"}]}


class _StubVmmModel:
    """A VMM pool as Mount sees it: export_fd(device) -> (fd, mapped bytes) and manifest(device); the fd is that of a plain file."""

    def __init__(self, path):
        self.path = path

    def export_fd(self, device):
        return os.open(self.path, os.O_RDONLY), os.path.getsize(self.path)

    def manifest(self, device):
        return {"apiVersion": "kukeon.gpupool/v1", "device": device, "deviceUUID": "GPU-00000000-aaaa-bbbb-cccc-dddddddddddd", "pciBusId": "0000:1b:00.0",
                "tensors": []}


def test_vmm_mount_serves_the_pool_fd_from_a_directory_deeper_than_sun_path(tmp_path):
    """The staged pool.sock lives in the cell's metadata directory, whatever its depth: a socket path longer than sockaddr_un allows is still
    bound by Mount and reached by receive_pool_fd."""
    from kukeon_b200 import modelhub
    pool_file = tmp_path / "pool.bin"
    pool_file.write_bytes(bytes(range(256)) * 16)
    cdir = str(tmp_path / ("realm-" + "r" * 40) / ("cell-" + "c" * 40) / "container")
    spec = modelhub.Mount(_StubVmmModel(str(pool_file)), 0, cdir)
    try:
        sock = os.path.join(spec.host_dir, "pool.sock")
        assert len(sock) > 108 and os.path.exists(sock)
        assert "KUKEON_GPUPOOL_FD_SOCKET=/run/kukeon/gpupool/pool.sock" in spec.env
        fd, size = modelhub.receive_pool_fd(sock)
        try:
            assert size == 4096 and os.pread(fd, 4096, 0) == pool_file.read_bytes()
        finally:
            os.close(fd)
    finally:
        modelhub.unmount(spec)
    assert not os.path.exists(sock)


def test_mount_single_and_named_models(tmp_path):
    from kukeon_b200 import modelhub
    cdir = str(tmp_path / "cell" / "work")
    one = modelhub.Mount(_StubModel(1), 0, cdir)
    assert one.mounts == [{"destination": "/run/kukeon/gpupool", "type": "bind", "source": f"{cdir}/gpupool", "options": ["rbind", "ro"]}]
    # the container is told WHICH GPU by UUID / PCI bus id — never by the daemon's CUDA ordinal, which means nothing in another process
    assert one.env == ["KUKEON_GPUPOOL_MANIFEST=/run/kukeon/gpupool/manifest.json", "KUKEON_GPUPOOL_IPC_HANDLE=/run/kukeon/gpupool/ipc.handle",
                       "KUKEON_GPUPOOL_DEVICE_UUID=GPU-00000000-aaaa-bbbb-cccc-dddddddddddd", "KUKEON_GPUPOOL_PCI_BUS_ID=0000:1b:00.0"]
    assert open(f"{cdir}/gpupool/ipc.handle", "rb").read() == b"\x01" * 64
    a = modelhub.Mount(_StubModel(2), 0, cdir, name="llama-3.8b")
    b = modelhub.Mount(_StubModel(3), 1, cdir, name="gpt2", target="/weights/")
    assert a.mounts[0]["destination"] == "/run/kukeon/gpupool/llama-3.8b" and a.mounts[0]["source"] == f"{cdir}/gpupool/llama-3.8b"
    assert a.env[0] == "KUKEON_GPUPOOL_MANIFEST_LLAMA_3_8B=/run/kukeon/gpupool/llama-3.8b/manifest.json" and a.env[2] == "KUKEON_GPUPOOL_DEVICE_UUID_LLAMA_3_8B=GPU-00000000-aaaa-bbbb-cccc-dddddddddddd"
    assert b.mounts[0]["destination"] == "/weights/gpt2" and b.env[1] == "KUKEON_GPUPOOL_IPC_HANDLE_GPT2=/weights/gpt2/ipc.handle"
    assert json.load(open(f"{cdir}/gpupool/gpt2/manifest.json"))["tensors"][0]["name"] == "w3"
    assert oct(os.stat(f"{cdir}/gpupool/gpt2/ipc.handle").st_mode & 0o777) == "0o640"
    merged = modelhub.merge_mounts([a, b])
    assert len(merged.mounts) == 2 and len(merged.env) == 8
    with pytest.raises(ValueError, match="same container path"):
        modelhub.merge_mounts([a, a])
    for bad in ("..", "a/b"):
        with pytest.raises(ValueError, match="directory name"):
            modelhub.Mount(_StubModel(4), 0, cdir, name=bad)


def test_merge_mounts_deduplicates_device_nodes(tmp_path):
    import stat as st_mod
    from types import SimpleNamespace

    from kukeon_b200 import modelhub

    def fake_stat(p):
        table = {"/dev/nvidiactl": (195, 255), "/dev/nvidia-uvm": (510, 0), "/dev/nvidia0": (195, 0), "/dev/nvidia1": (195, 1)}
        if p not in table:
            raise FileNotFoundError(p)
        return SimpleNamespace(st_mode=st_mod.S_IFCHR | 0o666, st_rdev=os.makedev(*table[p]))

    # the driver's own table: CUDA ordinal 0 sits at bus 1b = /dev/nvidia1, ordinal 1 at bus 1c = /dev/nvidia0 (ordinals follow CUDA_DEVICE_ORDER,
    # minors follow PCI enumeration — ADVICE r1: treating the ordinal as the minor exposes the wrong node)
    proc = tmp_path / "proc"
    for bus, minor in (("0000:1b:00.0", 1), ("0000:1c:00.0", 0)):
        os.makedirs(proc / bus)
        (proc / bus / "information").write_text(f"Model: \t\t NVIDIA B200\nIRQ:   \t\t 16\nGPU UUID: \t GPU-x\nBus Location: \t {bus}\nDevice Minor: \t {minor}\n")
    minor_of = lambda bus: modelhub.device_minor(bus, proc_root=str(proc))  # noqa: E731
    assert minor_of("0000:1B:00.0") == 1
    with pytest.raises(OSError):
        minor_of("0000:ff:00.0")
    cdir = str(tmp_path / "c")
    a = modelhub.Mount(_StubModel(1), 0, cdir, with_devices=True, stat=fake_stat, name="a", minor_of=minor_of)
    b = modelhub.Mount(_StubModel(2), 0, cdir, with_devices=True, stat=fake_stat, name="b", minor_of=minor_of)
    c = modelhub.Mount(_StubModel(3), 1, cdir, with_devices=True, stat=fake_stat, name="c", minor_of=minor_of)
    assert [d["path"] for d in a.devices][-1] == "/dev/nvidia1" and [d["path"] for d in c.devices][-1] == "/dev/nvidia0"
    merged = modelhub.merge_mounts([a, b, c])
    assert [d["path"] for d in merged.devices] == ["/dev/nvidiactl", "/dev/nvidia-uvm", "/dev/nvidia1", "/dev/nvidia0"]
    assert len(merged.device_cgroup) == 4 and all(r["allow"] and r["access"] == "rw" for r in merged.device_cgroup)
