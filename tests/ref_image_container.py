"""Plain-Python reference of the image container (DESIGN.md section 7), built on `struct` alone.

    pack(y_bytes, z_bytes, ids_keep, fields) -> bytes
    parse(data) -> dict of the header fields, "ids_keep", "z", "y"    (ValueError for a container that is not well formed)
    model_tag(tables, scale_table) -> int                            (FNV-1a 32 over the scale table and both CDF table sets)
    canonical_ids_restore(ids_keep, L) -> list                       (what the decoder rebuilds from ids_keep)

`fields`: img_size, patch_size, mode (accuracy mode, `(flags >> 3) & 7`), y_lanes, z_lanes, tag; K = len(ids_keep).
"""
import struct

MAGIC = 0x45414D54          # b"TMAE"
VERSION = 1
HEADER = 28


def id_bits(L):
    return max(1, (L - 1).bit_length())


def _pack_ids(ids, w):
    acc, nbits, out = 0, 0, []
    for v in ids:
        acc |= int(v) << nbits
        nbits += w
        while nbits >= 32:
            out.append(acc & 0xFFFFFFFF)
            acc >>= 32
            nbits -= 32
    if nbits:
        out.append(acc)
    return struct.pack(f"<{len(out)}I", *out)


def _unpack_ids(words_bytes, K, w):
    n = len(words_bytes) // 4
    acc = 0
    for i, v in enumerate(struct.unpack(f"<{n}I", words_bytes)):
        acc |= v << (32 * i)
    return [(acc >> (j * w)) & ((1 << w) - 1) for j in range(K)]


def pack(y_bytes, z_bytes, ids_keep, fields):
    L = (fields["img_size"] // fields["patch_size"]) ** 2
    K = len(ids_keep)
    head = struct.pack("<7I", MAGIC, VERSION | fields["mode"] << 8 | fields["y_lanes"] << 16 | fields["z_lanes"] << 24,
                       fields["img_size"] | fields["patch_size"] << 16, K, fields["tag"], len(z_bytes), len(y_bytes))
    return head + _pack_ids(ids_keep, id_bits(L)) + bytes(z_bytes) + bytes(y_bytes)


def parse(data):
    data = bytes(data)
    if len(data) < HEADER or len(data) % 4:
        raise ValueError("header: a container is a multiple of 4 bytes, at least 28")
    magic, w1, w2, w3, tag, z_len, y_len = struct.unpack_from("<7I", data)
    if magic != MAGIC or w1 & 0xFF != VERSION or w2 >> 24 or w3 >> 16:
        raise ValueError("header: magic, version or reserved bits")
    f = {"mode": (w1 >> 8) & 0xFF, "y_lanes": (w1 >> 16) & 0xFF, "z_lanes": w1 >> 24, "img_size": w2 & 0xFFFF,
         "patch_size": (w2 >> 16) & 0xFF, "K": w3, "tag": tag}
    if f["patch_size"] == 0:
        raise ValueError("header: patch_size 0")
    L = (f["img_size"] // f["patch_size"]) ** 2
    w = id_bits(L)
    ids_len = 4 * ((f["K"] * w + 31) // 32)
    if z_len % 4 or y_len % 4 or HEADER + ids_len + z_len + y_len != len(data):
        raise ValueError("header: section lengths")
    f["ids_keep"] = _unpack_ids(data[HEADER: HEADER + ids_len], f["K"], w)
    if any(v >= L for v in f["ids_keep"]) or len(set(f["ids_keep"])) != f["K"]:
        raise ValueError("patch ids")
    z0 = HEADER + ids_len
    f["z"], f["y"] = data[z0: z0 + z_len], data[z0 + z_len:]
    return f


def _fnv1a(x, data):
    for b in data:
        x = ((x ^ b) * 16777619) & 0xFFFFFFFF
    return x


def model_tag(tables, scale_table):
    """tables: MCM.entropy_tables() (compressai's buffer names); scale_table: the scale table as floats."""
    x = _fnv1a(2166136261, struct.pack(f"<{len(scale_table)}f", *[float(v) for v in scale_table]))
    for prefix in ("gaussian_conditional.", "entropy_bottleneck."):
        cdf, ln, off = (tables[prefix + k].tolist() for k in ("_quantized_cdf", "_cdf_length", "_offset"))
        for t in range(len(ln)):
            row = [ln[t], off[t]] + cdf[t][: ln[t]]
            x = _fnv1a(x, struct.pack(f"<{len(row)}i", *row))
    return x


def canonical_ids_restore(ids_keep, L):
    K = len(ids_keep)
    out = [None] * L
    for j, p in enumerate(ids_keep):
        out[p] = j
    rest = iter(range(K, L))
    return [v if v is not None else next(rest) for v in out]
