"""Makes the reference's test programs in oracle/_ref/ load the libdeflate_b200.so of the tree they sit in.

Programs linked by an older recipe name the library by the absolute path of the tree they were built in
(DT_NEEDED ".../libdeflate_b200/libdeflate_b200.so"), so they stop loading once that tree is moved or
deleted.  Their RUNPATH, $ORIGIN/../../libdeflate_b200, already finds the library by its bare name, and that
name is the tail of the stored path string.  So the DT_NEEDED entry is pointed at that tail.  Only the
entry's 8-byte string offset changes; the string table and the code are left as they are.
"""
import glob
import os
import struct
import tempfile

LIBNAME = b"libdeflate_b200.so"
PT_LOAD, PT_DYNAMIC = 1, 2
DT_NULL, DT_NEEDED, DT_STRTAB = 0, 1, 5


def _vaddr_to_offset(img, phdrs, addr):
    for p_type, p_offset, p_vaddr, p_filesz in phdrs:
        if p_type == PT_LOAD and p_vaddr <= addr < p_vaddr + p_filesz:
            return addr - p_vaddr + p_offset
    raise ValueError("address 0x%x is in no PT_LOAD segment" % addr)


def relocate_needed(path):
    """Rewrites an absolute DT_NEEDED naming libdeflate_b200.so to the bare name; returns True if it did."""
    img = bytearray(open(path, "rb").read())
    if img[:4] != b"\x7fELF" or img[4] != 2 or img[5] != 1:
        raise ValueError("%s: not a little-endian ELF64 file" % path)
    phoff, = struct.unpack_from("<Q", img, 0x20)
    phentsize, phnum = struct.unpack_from("<HH", img, 0x36)
    phdrs = []
    for i in range(phnum):
        o = phoff + i * phentsize
        p_type, = struct.unpack_from("<I", img, o)
        p_offset, p_vaddr = struct.unpack_from("<QQ", img, o + 8)
        p_filesz, = struct.unpack_from("<Q", img, o + 32)
        phdrs.append((p_type, p_offset, p_vaddr, p_filesz))
    dyn = [p for p in phdrs if p[0] == PT_DYNAMIC]
    if not dyn:
        return False
    entries = []
    for o in range(dyn[0][1], dyn[0][1] + dyn[0][3], 16):
        tag, val = struct.unpack_from("<qQ", img, o)
        if tag == DT_NULL:
            break
        entries.append((o, tag, val))
    strtab = _vaddr_to_offset(img, phdrs, next(v for _, t, v in entries if t == DT_STRTAB))
    changed = False
    for o, tag, val in entries:
        if tag != DT_NEEDED:
            continue
        s = strtab + val
        name = bytes(img[s:img.index(b"\0", s)])
        if name != LIBNAME and name.endswith(b"/" + LIBNAME):
            struct.pack_into("<Q", img, o + 8, val + len(name) - len(LIBNAME))
            changed = True
    if changed:
        fd, tmp = tempfile.mkstemp(dir=os.path.dirname(path))
        with os.fdopen(fd, "wb") as f:
            f.write(img)
        os.chmod(tmp, os.stat(path).st_mode & 0o7777)
        os.replace(tmp, path)
    return changed


def relocate_all(ref_dir):
    progs = [p for p in glob.glob(os.path.join(ref_dir, "test_*")) + [os.path.join(ref_dir, "benchmark")] if os.path.isfile(p)]
    return [p for p in progs if relocate_needed(p)]


if __name__ == "__main__":
    import sys
    for p in relocate_all(sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")):
        print("oracle/_ref: DT_NEEDED now names libdeflate_b200.so in", os.path.basename(p))
