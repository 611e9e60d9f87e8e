"""Plain-Python reference of the picture container (DESIGN.md section 7, "The picture container"), built on `struct` and the
image-container reference (tests/ref_image_container.py).

    pack(tiles, height, width) -> bytes          tiles: the T image containers of the picture in raster order
    parse(data, height=None, width=None, img_size=None) -> {"H", "W", "T", "tiles"}
                                                 ValueError("picture header ...") for every condition the GPU parse refuses
                                                 with TMAE_PIC_HEADER (H / W / T are checked when the call's are given)
    tile_count(height, width, img_size) -> int   rows * cols of tiling.tile_grid
"""
import struct

from tests import ref_image_container as I

MAGIC = 0x50414D54          # b"TMAP"
VERSION = 1


def tile_count(height, width, img_size):
    return (-(-height // img_size)) * (-(-width // img_size))


def pack(tiles, height, width):
    tiles = [bytes(t) for t in tiles]
    head = struct.pack(f"<4I{len(tiles)}I", MAGIC, VERSION, height | width << 16, len(tiles), *[len(t) for t in tiles])
    return head + b"".join(tiles)


def parse(data, height=None, width=None, img_size=None):
    data = bytes(data)
    if len(data) < 16 or len(data) % 4:
        raise ValueError("picture header: a picture is a multiple of 4 bytes, at least 16")
    magic, version, hw, T = struct.unpack_from("<4I", data)
    H, W = hw & 0xFFFF, hw >> 16
    if magic != MAGIC or version != VERSION:
        raise ValueError("picture header: magic, version or reserved bits")
    if (height is not None and H != height) or (width is not None and W != width):
        raise ValueError("picture header: height / width")
    if img_size is not None and T != tile_count(H, W, img_size):
        raise ValueError("picture header: tile count")
    if len(data) < 4 * (4 + T):
        raise ValueError("picture header: length table")
    lens = struct.unpack_from(f"<{T}I", data, 16)
    if any(n % 4 for n in lens) or 4 * (4 + T) + sum(lens) != len(data):
        raise ValueError("picture header: tile lengths")
    tiles, off = [], 4 * (4 + T)
    for n in lens:
        tiles.append(data[off: off + n])
        off += n
    return {"H": H, "W": W, "T": T, "tiles": tiles}


def parse_all(data, height=None, width=None, img_size=None):
    """parse, then every tile through the image-container reference."""
    f = parse(data, height, width, img_size)
    f["tile_fields"] = [I.parse(t) for t in f["tiles"]]
    return f
