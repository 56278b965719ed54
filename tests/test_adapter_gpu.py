"""-m gpu: the voxblox-side adapter (include/voxblox_b200/gpu_integrators.h), compiled against the
reference's own headers and run next to the reference's CPU integrators (oracle/adapter_test.cc).
The binary is built by oracle/Makefile where the reference's sources exist and travels with the
repository tree; it runs against this tree's engine library."""
import os
import shutil
import struct
import subprocess

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "oracle", "_ref", "adapter_test")
ENGINE = "libvoxblox_b200.so"


def _engine_by_name(path):
    """Rewrites, in place, a DT_NEEDED entry that names the engine by a path (binaries linked with the engine's
    file path record the directory they were built in) to the bare library name, so that the loader searches
    for it.  The shorter name is written over the old one in .dynstr; no offset changes."""
    with open(path, "r+b") as f:
        elf = bytearray(f.read())
        assert elf[:5] == b"\x7fELF\x02", "adapter_test is not a 64-bit ELF file"
        shoff, = struct.unpack_from("<Q", elf, 0x28)
        shentsize, shnum = struct.unpack_from("<HH", elf, 0x3A)
        sections = [struct.unpack_from("<IIQQQQIIQQ", elf, shoff + k * shentsize) for k in range(shnum)]
        for _, sh_type, _, _, off, size, link, _, _, entsize in sections:
            if sh_type != 6:  # SHT_DYNAMIC
                continue
            strtab = sections[link][4]
            for e in range(off, off + size, entsize):
                tag, val = struct.unpack_from("<qQ", elf, e)
                if tag != 1:  # DT_NEEDED
                    continue
                start = strtab + val
                name = bytes(elf[start:elf.index(b"\0", start)])
                if b"/" in name and os.path.basename(name) == ENGINE.encode():
                    elf[start:start + len(name)] = ENGINE.encode() + b"\0" * (len(name) - len(ENGINE))
        f.seek(0)
        f.write(elf)


@pytest.mark.skipif(not os.path.exists(EXE), reason="oracle/_ref/adapter_test not built (the reference's sources are absent)")
def test_drop_in_adapter_against_reference_classes(tmp_path):
    exe = str(tmp_path / "adapter_test")
    shutil.copy2(EXE, exe)
    _engine_by_name(exe)
    env = dict(os.environ, LD_LIBRARY_PATH=os.pathsep.join(
        [os.path.join(ROOT, "voxblox_b200")] + [p for p in os.environ.get("LD_LIBRARY_PATH", "").split(os.pathsep) if p]))
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300, env=env)
    print(out.stdout, out.stderr)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "ADAPTER TEST OK" in out.stdout
