"""Host-side mirror of the Go API the north_star adds to kukeon's `internal/modelhub`:
`Pull`, `Load`, `Mount` plus the per-Cell acquire/release hooks.

None of these exist in the reference (SURVEY.md §8(a2-a6)); the shapes below follow the seams they would
sit next to so that the Go shim in INTEGRATION.md is a line-for-line transliteration:

* `Pull`   — local-path resolution + tensor index (nearest analogue: ctr image pull, internal/ctr/image.go:91).
* `Load`   — one call into the C ABI per checkpoint; N concurrent callers share one load
             (runner.StartCell call site, internal/controller/runner/start.go:785-790).
* `Mount`  — stages `<cell metadata dir>/gpupool/{manifest.json,ipc.handle}` atomically
             (internal/metadata/metadata.go:105-140) and returns the OCI bind mount
             (`bindVolumeMount`, internal/ctr/spec.go:526-543) and `KUKEON_GPUPOOL_*` env entries
             (`kukeonDefaultEnv`, internal/ctr/spec.go:464-482) a `ctr.BuildOption` would add.

All data movement happens in libkukeon_gpuload.so; this file never touches tensor bytes.

Trust model of a mounted pool (the unit of isolation in kukeon is the cell; N cells share ONE HBM copy of a model):

* cudaMalloc pools are exported as a cudaIpcMemHandle (`ipc.handle`).  Whoever opens it gets a READ-WRITE mapping — the `ro` bind mount
  protects only the files.  Use this only when every cell that mounts the model belongs to one trust domain.  `Mount` checksums the pool
  on the device before handing it to a further cell and refuses when it no longer matches the checksum recorded at the first mount
  (tamper DETECTION; pools are whole 2 MiB multiples so a handle never exposes a neighbouring allocation).
* VMM pools (`Pool(..., flags=CFG_VMM_POOLS)`) are exported as a POSIX file descriptor, passed over the Unix socket `pool.sock` staged next
  to the manifest (SCM_RIGHTS; the socket is reachable through the same read-only bind mount).  The consumer maps it with
  `gpupool.ImportedPool(fd, ...)` = `kk_import_fd(..., KK_IMPORT_READONLY)`: a store through that mapping faults in the consumer.
  This is the mode for cells that do not trust each other (tamper PREVENTION for consumers using the library's importer; a consumer
  that calls the driver itself can still ask for a writable mapping of an fd it was given, so hand the fd only to cells that are allowed
  to read the weights, and keep a private copy per trust domain when that is not enough).
"""
from __future__ import annotations

import json
import os
import socket
import struct
import tempfile
import threading
from dataclasses import dataclass, field
from typing import Dict, List, Optional

from . import gpupool
from .gpupool import FANOUT_NONE, FANOUT_P2P, MODE_BROADCAST, MODE_SCATTER, MODE_SINGLE  # noqa: F401

CONTAINER_GPUPOOL_DIR = "/run/kukeon/gpupool"  # bind-mount target inside the agent container
ENV_MANIFEST = "KUKEON_GPUPOOL_MANIFEST"
ENV_IPC_HANDLE = "KUKEON_GPUPOOL_IPC_HANDLE"
ENV_DEVICE_UUID = "KUKEON_GPUPOOL_DEVICE_UUID"  # "GPU-xxxxxxxx-...": what cudaGetDeviceProperties().uuid / nvidia-smi -L print inside the container too
ENV_PCI_BUS_ID = "KUKEON_GPUPOOL_PCI_BUS_ID"
ENV_FD_SOCKET = "KUKEON_GPUPOOL_FD_SOCKET"      # VMM pools: Unix socket that hands out the pool's file descriptor (SCM_RIGHTS) + its mapped size


@dataclass
class ModelRef:
    """Result of Pull: where the checkpoint lives and what is in it."""
    path: str
    shards: List[str]
    tensors: List[dict]

    @property
    def file_bytes(self) -> int:
        return sum(t["nbytes"] for t in self.tensors)


def Pull(path: str) -> ModelRef:
    """Resolve a local checkpoint (directory with model.safetensors.index.json / model.safetensors /
    *.gguf, or a single file) and index it.  No network: "pull" is local-path only (SURVEY.md §8(a2))."""
    return ModelRef(path=os.path.realpath(path), shards=gpupool.index_shards(path), tensors=gpupool.index(path))


def Load(pool: gpupool.Pool, ref: ModelRef | str, mode: int = MODE_SINGLE, fanout: int = FANOUT_P2P, flags: int = 0,
         part_index: int = 0, part_count: int = 0) -> gpupool.Model:
    """Make the checkpoint resident in the pool(s).  Returns a refcounted Model; a second Load of the same
    checkpoint returns the same resident copy with its count bumped."""
    path = ref.path if isinstance(ref, ModelRef) else ref
    return pool.load(path, mode=mode, fanout=fanout, flags=flags, part_index=part_index, part_count=part_count)


@dataclass
class MountSpec:
    """What a `ctr.WithGPUWeights(...)` BuildOption would append to the container's OCI spec."""
    mounts: List[dict] = field(default_factory=list)
    env: List[str] = field(default_factory=list)
    host_dir: str = ""
    devices: List[dict] = field(default_factory=list)        # OCI linux.devices
    device_cgroup: List[dict] = field(default_factory=list)  # OCI linux.resources.devices allow rules


NVIDIA_PROC_GPUS = "/proc/driver/nvidia/gpus"


def device_minor(pci_bus_id: str, proc_root: str = NVIDIA_PROC_GPUS) -> int:
    """Minor number of the /dev/nvidia<N> node of the GPU at `pci_bus_id` ("dddd:bb:dd.f"), from the driver's own table
    (`<proc_root>/<bus id>/information`, line "Device Minor: N").  A CUDA ordinal is NOT that number: ordinals follow CUDA_DEVICE_ORDER
    (fastest first by default) and CUDA_VISIBLE_DEVICES, minors follow PCI enumeration (ADVICE r1)."""
    path = os.path.join(proc_root, pci_bus_id.lower(), "information")
    with open(path) as f:
        for line in f:
            k, _, v = line.partition(":")
            if k.strip() == "Device Minor":
                return int(v.strip())
    raise LookupError(f"{path}: no 'Device Minor' line")


def device_nodes(minors, stat=os.stat) -> tuple:
    """"next" row f2 (SURVEY.md §8(f)): the NVIDIA character devices an agent container needs to map an exported pool
    — /dev/nvidiactl, /dev/nvidia-uvm, /dev/nvidia-uvm-tools and /dev/nvidia<minor> for each exported GPU — as
    OCI `linux.devices` entries plus the matching device-cgroup allow rules (the reference's spec builder emits
    neither today: internal/ctr/spec.go:218-380).  `minors` are device-node minor numbers (device_minor()), not CUDA ordinals.
    Nodes that do not exist on the host are skipped."""
    import stat as st_mod
    paths = ["/dev/nvidiactl", "/dev/nvidia-uvm", "/dev/nvidia-uvm-tools"] + [f"/dev/nvidia{d}" for d in sorted(set(minors))]
    devs, rules = [], []
    for p in paths:
        try:
            s = stat(p)
        except OSError:
            continue
        if not st_mod.S_ISCHR(s.st_mode):
            continue
        major, minor = os.major(s.st_rdev), os.minor(s.st_rdev)
        devs.append({"path": p, "type": "c", "major": major, "minor": minor, "fileMode": 0o666, "uid": 0, "gid": 0})
        rules.append({"allow": True, "type": "c", "major": major, "minor": minor, "access": "rw"})
    return devs, rules


def _atomic_write(path: str, data: bytes, mode: int = 0o644) -> None:
    d = os.path.dirname(path)
    fd, tmp = tempfile.mkstemp(prefix=".meta-", suffix=".tmp", dir=d)
    try:
        os.fchmod(fd, mode)
        os.write(fd, data)
        os.fsync(fd)
    finally:
        os.close(fd)
    os.rename(tmp, path)
    try:
        dfd = os.open(d, os.O_RDONLY)
        os.fsync(dfd)
        os.close(dfd)
    except OSError:
        pass


def _env_suffix(name: str) -> str:
    """`llama-3.8b` -> `_LLAMA_3_8B` (POSIX environment names: upper-case letters, digits, underscore)."""
    return "_" + "".join(c.upper() if c.isalnum() else "_" for c in name)


def Mount(model: gpupool.Model, device: int, container_dir: str, with_devices: bool = False, stat=os.stat, name: str = "",
          target: str = CONTAINER_GPUPOOL_DIR, identity=None, minor_of=None, verify: bool = True) -> MountSpec:
    """Export `device`'s pool for one agent container: write the manifest + IPC handle under
    `<container_dir>/gpupool/` and describe the read-only bind mount and env that expose them.

    `name` (the `models[].name` of the manifest schema, kukeon_b200/schema.py) gives the model its own sub-directory and
    env names — `<container_dir>/gpupool/<name>/`, `<target>/<name>/`, `KUKEON_GPUPOOL_MANIFEST_<NAME>` — so that one container can
    attach several models; without it the single-model layout above is used."""
    if name and (name in (".", "..") or "/" in name or "\0" in name):
        raise ValueError(f"model name {name!r} cannot be used as a directory name")
    vmm = _is_vmm(model, device)
    handle, manifest = (b"", model.manifest(device)) if vmm else model.export(device)
    if verify and not vmm:
        verify_pool(model, device, int(manifest.get("poolBytes", 0)))  # an IPC handle maps read-write in every cell that opened it: detect a pool some earlier cell has written to
    host_dir = os.path.join(container_dir, "gpupool", name) if name else os.path.join(container_dir, "gpupool")
    dest = f"{target.rstrip('/')}/{name}" if name else target
    sfx = _env_suffix(name) if name else ""
    os.makedirs(host_dir, mode=0o750, exist_ok=True)
    _atomic_write(os.path.join(host_dir, "manifest.json"), json.dumps(manifest, separators=(",", ":")).encode())
    extra_env = []
    if vmm:
        srv = PoolFdServer(model, device, os.path.join(host_dir, "pool.sock"))
        srv.start()
        _FD_SERVERS[os.path.join(host_dir, "pool.sock")] = srv
        extra_env.append(f"{ENV_FD_SOCKET}{sfx}={dest}/pool.sock")
    else:
        _atomic_write(os.path.join(host_dir, "ipc.handle"), handle, 0o640)
    # What the container is told about the GPU: its UUID and PCI bus id (stable everywhere), never the daemon's ordinal — a container that sees
    # only /dev/nvidia3 enumerates that GPU as ordinal 0, so cudaSetDevice(<host ordinal>) would fail there.  The agent picks the CUDA device
    # whose UUID matches (or, with a single exposed node, device 0).
    ident = identity(device) if identity else {"uuid": manifest.get("deviceUUID", ""), "pci_bus_id": manifest.get("pciBusId", "")}
    devs, rules = [], []
    if with_devices:
        minor = minor_of(ident["pci_bus_id"]) if minor_of else device_minor(ident["pci_bus_id"])
        devs, rules = device_nodes([minor], stat)
    return MountSpec(
        mounts=[{"destination": dest, "type": "bind", "source": host_dir, "options": ["rbind", "ro"]}],
        env=[f"{ENV_MANIFEST}{sfx}={dest}/manifest.json"] + ([] if vmm else [f"{ENV_IPC_HANDLE}{sfx}={dest}/ipc.handle"]) +
            [f"{ENV_DEVICE_UUID}{sfx}={ident['uuid']}", f"{ENV_PCI_BUS_ID}{sfx}={ident['pci_bus_id']}"] + extra_env,
        host_dir=host_dir, devices=devs, device_cgroup=rules,
    )


def _is_vmm(model, device: int) -> bool:
    """True when `device`'s pool can (only) be exported as a file descriptor.  Stub models of the CPU tests have no export_fd."""
    fn = getattr(model, "export_fd", None)
    if fn is None:
        return False
    try:
        fd, _ = fn(device)
    except gpupool.ErrUnsupported:
        return False
    os.close(fd)
    return True


_POOL_SUMS: Dict[tuple, int] = {}


def verify_pool(model, device: int, pool_bytes: int) -> None:
    """Tamper detection for IPC-exported pools: the device-side checksum of the whole pool is recorded at the first Mount and must still match
    at every later one (kk_checksum streams the pool at HBM read rate: milliseconds for 16 GB).  Raises RuntimeError when it does not —
    the daemon should then reload the model instead of handing corrupted weights to one more cell."""
    csum = getattr(model, "checksum", None)
    if csum is None:
        return  # CPU-tier stub
    n = pool_bytes // 8 * 8
    if n == 0:
        return
    key = (id(getattr(model, "_pool", None)), int(model._h.value or 0), device)
    got = csum(device, 0, n)
    want = _POOL_SUMS.setdefault(key, got)
    if got != want:
        raise RuntimeError(f"pool of device {device} changed since it was first mounted (checksum {got:#x} != {want:#x}): some cell wrote to the shared weights")


def forget_pool(model) -> None:
    """Drop the recorded checksums of a model that is being released (its handle value may be reused)."""
    h = int(model._h.value or 0)
    for k in [k for k in _POOL_SUMS if k[1] == h]:
        del _POOL_SUMS[k]


_SUN_PATH_MAX = 107  # sockaddr_un.sun_path: 108 bytes including the terminating NUL


def _at_unix_path(op, path: str):
    """`op(address)` — a socket's bind or connect — for the Unix socket at `path`.  A cell's metadata directory can be deeper than sun_path
    allows; a longer path is reached as /proc/self/fd/<directory fd>/<name>, which the kernel resolves to the same file."""
    if len(os.fsencode(path)) <= _SUN_PATH_MAX:
        return op(path)
    dfd = os.open(os.path.dirname(path) or ".", os.O_PATH | os.O_DIRECTORY)
    try:
        return op(f"/proc/self/fd/{dfd}/{os.path.basename(path)}")
    finally:
        os.close(dfd)


class PoolFdServer(threading.Thread):
    """Hands the file descriptor of a VMM pool to whoever connects to `path` (a Unix socket staged in the directory that is bind-mounted
    read-only into the agent container — like a docker.sock, the socket stays connectable through the mount).  One message per connection:
    8 bytes little-endian mapped size, with the fd attached as SCM_RIGHTS ancillary data.  In kukeond this is a goroutine next to the attachable
    sockets (internal/ctr/attachable.go:100-185 binds Unix sockets into containers the same way)."""

    def __init__(self, model, device: int, path: str):
        super().__init__(daemon=True)
        self.model, self.device, self.path = model, device, path
        self._stop = threading.Event()
        try:
            os.unlink(path)
        except FileNotFoundError:
            pass
        self.sock = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
        _at_unix_path(self.sock.bind, path)
        os.chmod(path, 0o660)
        self.sock.listen(16)
        self.sock.settimeout(0.2)
        self.served = 0

    def run(self) -> None:
        while not self._stop.is_set():
            try:
                conn, _ = self.sock.accept()
            except socket.timeout:
                continue
            except OSError:
                break
            with conn:
                try:
                    fd, size = self.model.export_fd(self.device)
                    try:
                        socket.send_fds(conn, [struct.pack("<Q", size)], [fd])
                        self.served += 1
                    finally:
                        os.close(fd)
                except Exception:  # noqa: BLE001 - a failing client must not take the server down
                    pass

    def stop(self) -> None:
        self._stop.set()
        try:
            self.sock.close()
        finally:
            try:
                os.unlink(self.path)
            except FileNotFoundError:
                pass


_FD_SERVERS: Dict[str, PoolFdServer] = {}


def unmount(spec: MountSpec) -> None:
    """Stop the fd server of a VMM mount (KillCell / DeleteCell path); the staged directory is removed with the cell's metadata."""
    srv = _FD_SERVERS.pop(os.path.join(spec.host_dir, "pool.sock"), None)
    if srv is not None:
        srv.stop()


def receive_pool_fd(sock_path: str) -> tuple:
    """Agent side: connect to the staged socket, returns (fd, mapped_bytes).  The caller maps it with gpupool.ImportedPool and closes the fd."""
    with socket.socket(socket.AF_UNIX, socket.SOCK_STREAM) as c:
        _at_unix_path(c.connect, sock_path)
        msg, fds, _, _ = socket.recv_fds(c, 8, 1)
        if len(msg) != 8 or len(fds) != 1:
            raise OSError("pool fd server sent no descriptor")
        return fds[0], struct.unpack("<Q", msg)[0]


def merge_mounts(specs: List[MountSpec]) -> MountSpec:
    """What the container's BuildOptions add up to when several models are mounted: all mounts and env entries, device nodes and
    cgroup rules de-duplicated (two models on the same GPU need /dev/nvidia0 once)."""
    out = MountSpec()
    for s in specs:
        out.mounts += s.mounts
        out.env += s.env
        for d in s.devices:
            if d not in out.devices:
                out.devices.append(d)
        for r in s.device_cgroup:
            if r not in out.device_cgroup:
                out.device_cgroup.append(r)
    dests = [m["destination"] for m in out.mounts]
    if len(set(dests)) != len(dests):
        raise ValueError(f"two models would be mounted at the same container path: {sorted(d for d in dests if dests.count(d) > 1)[0]}")
    return out


class CellHooks:
    """Per-Cell reference counting ("N concurrent agent Sessions" == N Cells, SURVEY.md §8(a5)).
    acquire() in StartCell; release() from KillCell / StopCell / DeleteCell — idempotent per cell because
    those teardown paths overlap in the reference (markCellFailed calls KillCell, runner/start.go:192-242)."""

    def __init__(self, model: gpupool.Model):
        self.model = model
        self._cells: Dict[str, bool] = {}

    def start_cell(self, cell_id: str) -> None:
        if self._cells.get(cell_id):
            return
        self.model.acquire()
        self._cells[cell_id] = True

    def stop_cell(self, cell_id: str) -> None:
        if self._cells.pop(cell_id, None):
            self.model.release()

    @property
    def active(self) -> int:
        return len(self._cells)
