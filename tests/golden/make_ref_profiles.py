"""Copy the reference's ICC profiles (libvips/colour/profiles) into tests/golden/profiles for
tests/test_icc.py.  Run where the reference tree exists:

    python tests/golden/make_ref_profiles.py /path/to/libvips-source

cmyk.icm is 939 KiB, 717 KiB of which are characterisation data under three text tags that no
transform reads.  Its copy keeps the tags a relative-colorimetric transform and its white and
black points use (header, desc, cprt, wtpt, bkpt, clrt, A2B0/1/2, B2A1), byte for byte: lcms2 and
the project's evaluator give the same results for it as for the whole profile.
"""
import os
import struct
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CMYK_DROPPED = {b"targ", b"DevD", b"CIED", b"gamt", b"B2A0", b"B2A2"}


def drop_tags(data, drop):
    """the profile without the tags in `drop`; shared tag data stays shared, the profile ID is cleared"""
    n = struct.unpack(">I", data[128:132])[0]
    tags = [struct.unpack(">4sII", data[132 + 12 * i:144 + 12 * i]) for i in range(n)]
    keep = [t for t in tags if t[0] not in drop]
    body, pos, where = b"", 128 + 4 + 12 * len(keep), {}
    for off, size in sorted({(o, s) for _, o, s in keep}):
        pad = -pos % 4
        body += b"\0" * pad
        pos += pad
        where[(off, size)] = pos
        body += data[off:off + size]
        pos += size
    table = struct.pack(">I", len(keep)) + b"".join(struct.pack(">4sII", sig, where[(o, s)], s) for sig, o, s in keep)
    out = bytearray(data[:128] + table + body + b"\0" * (-pos % 4))
    out[0:4] = struct.pack(">I", len(out))
    out[84:100] = bytes(16)
    return bytes(out)


def main(src):
    dst = os.path.join(HERE, "profiles")
    os.makedirs(dst, exist_ok=True)
    for name in ("sRGB.icm", "p3.icm", "sGrey.icm", "cmyk.icm"):
        with open(os.path.join(src, "libvips", "colour", "profiles", name), "rb") as f:
            data = f.read()
        if name == "cmyk.icm":
            data = drop_tags(data, CMYK_DROPPED)
        with open(os.path.join(dst, name), "wb") as f:
            f.write(data)
        print("wrote %s: %d bytes" % (os.path.join(dst, name), len(data)))


if __name__ == "__main__":
    main(sys.argv[1])
