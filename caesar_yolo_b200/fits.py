"""Minimal FITS primary-HDU access for the hot path (astropy.io.fits / fitsio are not dependencies of this build).
Replaces utils.get_fits_header / read_fits / read_fits_crop of the reference (caesar_yolo/utils.py:150-164,
193-246, 340-418): the pixel payload is handed to the GPU in its raw big-endian byte order (BITPIX -32) and decoded
there (byte swap + non-finite -> 0 fused into the first load of the preprocessing kernels)."""
import os

import numpy as np

_BITPIX_DTYPE = {8: ">u1", 16: ">i2", 32: ">i4", 64: ">i8", -32: ">f4", -64: ">f8"}


def _value(s):
    s = s.strip()
    if not s:
        return None
    if s[0] == "'":
        end = s.find("'", 1)
        while end != -1 and end + 1 < len(s) and s[end + 1] == "'":
            end = s.find("'", end + 2)
        return s[1:end].replace("''", "'").rstrip()
    s = s.split("/")[0].strip()
    if s in ("T", "F"):
        return s == "T"
    for conv in (int, lambda v: float(v.replace("D", "E"))):
        try:
            return conv(s)
        except ValueError:
            pass
    return s


class FitsImage(object):
    """Header + memory-mapped payload of the primary HDU.  For NAXIS=4 cubes the plane [0,0] is used
    (utils.py:378-380)."""

    def __init__(self, path):
        self.path = path
        self.header = {}
        off = 0
        with open(path, "rb") as f:
            done = False
            while not done:
                block = f.read(2880)
                if len(block) < 2880:
                    raise IOError("truncated FITS header in %s" % path)
                off += 2880
                for i in range(36):
                    card = block[i * 80:(i + 1) * 80].decode("ascii", "replace")
                    key = card[:8].strip()
                    if key == "END":
                        done = True
                        break
                    if card[8:10] == "= ":
                        self.header[key] = _value(card[10:])
        h = self.header
        naxis = h.get("NAXIS", 0)
        if naxis not in (2, 4):   # read_fits / read_fits_crop accept 2-D images and 4-D cubes only (utils.py:207-216,378-386)
            raise ValueError("Invalid/unsupported number of channels found in file %s (nchan=%s)" % (path, naxis))
        self.nx, self.ny = int(h["NAXIS1"]), int(h["NAXIS2"])
        self.bitpix = int(h["BITPIX"])
        self.offset = off
        self.bscale, self.bzero = h.get("BSCALE", 1), h.get("BZERO", 0)
        self.raw = np.memmap(path, dtype=np.dtype(_BITPIX_DTYPE[self.bitpix]), mode="r", offset=off,
                             shape=(self.ny, self.nx))

    @property
    def is_raw_f32(self):
        """True when rows can be shipped to the GPU byte-for-byte (big-endian float32, no scaling)."""
        return self.bitpix == -32 and self.bscale == 1 and self.bzero == 0

    def rows(self, y0, y1):
        """Rows [y0,y1) as a C-contiguous array: raw big-endian float32 when is_raw_f32, else native float32."""
        a = self.raw[y0:y1]
        if self.is_raw_f32:
            return np.ascontiguousarray(a)
        out = a.astype(np.float32)
        if self.bscale != 1 or self.bzero != 0:
            out = out * np.float32(self.bscale) + np.float32(self.bzero)
        return out


def pixel_scale_matrix(h):
    """2x2 matrix (degrees per pixel) from intermediate world coordinates to pixel offsets of a FITS header dict: the CD
    matrix when any CDi_j card is present, else CDELTi times the PCi_j matrix (identity when absent), else CDELTi with
    the CROTA2 rotation (Calabretta & Greisen 2002, eq. 189).  None without CDELT1/2 or CD cards."""
    if any(("CD%d_%d" % (i, j)) in h for i in (1, 2) for j in (1, 2)):
        return np.array([[float(h.get("CD%d_%d" % (i, j), 0.0)) for j in (1, 2)] for i in (1, 2)])
    if "CDELT1" not in h or "CDELT2" not in h:
        return None
    c1, c2 = float(h["CDELT1"]), float(h["CDELT2"])
    if any(("PC%d_%d" % (i, j)) in h for i in (1, 2) for j in (1, 2)):
        pc = np.array([[float(h.get("PC%d_%d" % (i, j), 1.0 if i == j else 0.0)) for j in (1, 2)] for i in (1, 2)])
        return np.array([[c1], [c2]]) * pc
    rho = np.radians(float(h.get("CROTA2", 0.0)))
    return np.array([[c1 * np.cos(rho), -c2 * np.sin(rho)], [c1 * np.sin(rho), c2 * np.cos(rho)]])


def beam_area_pix(h):
    """Solid angle of the Gaussian restoring beam in pixels, pi * BMAJ * BMIN / (4 ln 2) / |det(pixel scale matrix)|
    (BMAJ / BMIN: FWHM in degrees); None when the cards are missing or degenerate.  The flux density of a source is
    its pixel sum divided by this (Jy for a Jy/beam image)."""
    m = pixel_scale_matrix(h)
    if m is None or "BMAJ" not in h or "BMIN" not in h:
        return None
    det = abs(float(np.linalg.det(m)))
    area = np.pi * float(h["BMAJ"]) * float(h["BMIN"]) / (4.0 * np.log(2.0))
    if not (det > 0 and area > 0 and np.isfinite(det) and np.isfinite(area)):
        return None
    return area / det


def celestial_projection(h):
    """'SIN' or 'TAN' when CTYPE1/2 are RA---SIN / DEC--SIN or RA---TAN / DEC--TAN, else None."""
    t1, t2 = str(h.get("CTYPE1", "")).strip().upper(), str(h.get("CTYPE2", "")).strip().upper()
    for proj in ("SIN", "TAN"):
        if t1 == "RA---" + proj and t2 == "DEC--" + proj:
            return proj
    return None


def pixel_to_world(h, x, y):
    """(ra, dec) in degrees of 0-based pixel coordinates x (column), y (row) for the SIN and TAN projections (Calabretta
    & Greisen 2002, sections 2-3 and 5.1: zenithal projections with the reference point at the native pole; SIN without
    the PV obliqueness terms).  The native longitude of the celestial pole is the LONPOLE card, by default 180 deg, or 0
    when CRVAL2 = 90 (C&G sect. 2.4).  FITS pixels are 1-based: p = x + 1.  Points outside the projection's domain give
    NaN.  None when the header has no SIN / TAN celestial WCS."""
    proj = celestial_projection(h)
    m = pixel_scale_matrix(h)
    if proj is None or m is None or any(k not in h for k in ("CRVAL1", "CRVAL2", "CRPIX1", "CRPIX2")):
        return None
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    d1 = x + 1.0 - float(h["CRPIX1"])
    d2 = y + 1.0 - float(h["CRPIX2"])
    xi = np.radians(m[0, 0] * d1 + m[0, 1] * d2)          # intermediate world coordinates (projection plane)
    eta = np.radians(m[1, 0] * d1 + m[1, 1] * d2)
    r = np.hypot(xi, eta)
    phi = np.arctan2(xi, -eta)                              # native longitude
    with np.errstate(invalid="ignore"):
        theta = np.arctan2(1.0, r) if proj == "TAN" else np.arccos(r)   # native latitude
    a0, d0 = np.radians(float(h["CRVAL1"])), np.radians(float(h["CRVAL2"]))
    # default LONPOLE (C&G 2002 eq. 8 with theta_0 = 90 deg): 0 for a reference point at the north pole, else 180
    phi_p = np.radians(float(h.get("LONPOLE", 0.0 if float(h["CRVAL2"]) >= 90.0 else 180.0)))
    dphi = phi - phi_p
    st, ct = np.sin(theta), np.cos(theta)
    ra = a0 + np.arctan2(-ct * np.sin(dphi), st * np.cos(d0) - ct * np.sin(d0) * np.cos(dphi))
    dec = np.arcsin(np.clip(st * np.sin(d0) + ct * np.cos(d0) * np.cos(dphi), -1.0, 1.0))
    return np.degrees(ra) % 360.0, np.degrees(dec)


def write_fits(data, path):
    """Minimal primary-HDU writer (utils.write_fits, caesar_yolo/utils.py:126-134: `fits.PrimaryHDU(data)` with no
    header): 2-D float32 / float64 array -> big-endian payload padded to 2880-byte blocks."""
    a = np.asarray(data)
    if a.ndim != 2 or a.dtype.kind != 'f':
        raise ValueError("write_fits: 2-D floating-point array expected")
    bitpix = -32 if a.dtype.itemsize == 4 else -64

    def card(key, val, comment=""):
        v = ("%20s" % val) if not isinstance(val, str) else val
        c = "%-8s= %s" % (key, v)
        if comment:
            c += " / " + comment
        return ("%-80s" % c)[:80]
    cards = [card("SIMPLE", "T", "conforms to FITS standard"), card("BITPIX", bitpix, "array data type"),
             card("NAXIS", 2, "number of array dimensions"), card("NAXIS1", a.shape[1]), card("NAXIS2", a.shape[0]),
             card("EXTEND", "T"), "%-80s" % "END"]
    hdr = "".join(cards)
    hdr += " " * (-len(hdr) % 2880)
    payload = np.ascontiguousarray(a, dtype='>f4' if bitpix == -32 else '>f8').tobytes()
    with open(path, "wb") as f:
        f.write(hdr.encode("ascii"))
        f.write(payload)
        f.write(b"\0" * (-len(payload) % 2880))


def format_card(key, value, comment=""):
    """One 80-character header card.  Logicals and numbers are right-justified to column 30 (fixed format; a float
    whose shortest round-trip form is longer than 20 characters extends past it, which the free format allows); floats
    always carry a '.' and an uppercase 'E' exponent; strings are quoted from column 11, embedded quotes doubled, and
    padded to at least 8 characters."""
    if isinstance(value, (bool, np.bool_)):
        v = "%20s" % ("T" if value else "F")
    elif isinstance(value, (int, np.integer)):
        v = "%20d" % value
    elif isinstance(value, (float, np.floating)):
        if not np.isfinite(value):
            raise ValueError("%s: a FITS header value must be finite" % key)
        s = repr(float(value))
        mant, _, exp = s.partition("e")
        if "." not in mant:
            mant += ".0"
        v = "%20s" % (mant + ("E" + exp if exp else ""))
    else:
        v = "'%-8s'" % str(value).replace("'", "''")
    c = "%-8s= %s" % (key, v)
    if comment:
        c += " / " + comment
    if len(c) > 80:
        raise ValueError("%s: card longer than 80 characters" % key)
    return "%-80s" % c


# cards of the image header that a map keeps: the celestial WCS of axes 1 and 2, the unit and the beam
_WCS_AXIS_KEYS = ("CTYPE", "CRVAL", "CDELT", "CUNIT")
_WCS_KEYS = ("CD1_1", "CD1_2", "CD2_1", "CD2_2", "PC1_1", "PC1_2", "PC2_1", "PC2_2", "CROTA2", "LONPOLE", "LATPOLE",
             "RADESYS", "EQUINOX", "BUNIT", "BMAJ", "BMIN", "BPA")


def map_header(h, nx, ny, x0=0, y0=0, bkgmask=False, bkgest='mean', bunit=True):
    """Header (bytes, a multiple of 2880) of a 2-D BITPIX -32 map of nx x ny pixels whose pixel (0, 0) is pixel (x0, y0)
    of the image with header dict h: the WCS cards of axes 1 and 2, BUNIT and the beam are copied, and CRPIX1/2 are
    shifted by (x0, y0), so every map pixel has the sky position of the image pixel under it.  bkgmask: the catalog
    boxes were masked out of the node boxes (card BKGMASK = T; no card otherwise).  bkgest: the centre of the node
    clipping; 'median' writes BKGEST = 'MEDIAN', the mean writes no card.  bunit=False leaves BUNIT out, for a map
    without the image's unit (the S/N map)."""
    cards = [format_card("SIMPLE", True, "conforms to FITS standard"), format_card("BITPIX", -32, "array data type"),
             format_card("NAXIS", 2, "number of array dimensions"), format_card("NAXIS1", int(nx)),
             format_card("NAXIS2", int(ny))]
    for a, off in ((1, x0), (2, y0)):
        for k in _WCS_AXIS_KEYS:
            if "%s%d" % (k, a) in h:
                cards.append(format_card("%s%d" % (k, a), h["%s%d" % (k, a)]))
        if "CRPIX%d" % a in h:
            cards.append(format_card("CRPIX%d" % a, h["CRPIX%d" % a] - off))
    cards += [format_card(k, h[k]) for k in _WCS_KEYS if k in h and (bunit or k != "BUNIT")]
    if bkgmask:
        cards.append(format_card("BKGMASK", True, "catalog boxes masked out of the node boxes"))
    if bkgest == 'median':
        cards.append(format_card("BKGEST", "MEDIAN", "node bkg: sigma-clipped median"))
    cards.append("%-80s" % "END")
    txt = "".join(cards)
    return (txt + " " * (-len(txt) % 2880)).encode("ascii")


def write_map_rows(path, header, rows, row_begin, nx, ny, rank=0, world=1, piece_bytes=1 << 26):
    """Writes one FITS map in parallel by rows.  rows: this rank's map rows [row_begin, row_begin + len(rows)) as a
    device tensor [n, nx] of 4-byte words already in FITS byte order; header: map_header bytes.  Rank 0 writes the
    header and sizes the file (payload padded to 2880 bytes with zeros); after a barrier, every rank writes its rows
    with pwrite through pinned staging in pieces of ~piece_bytes; a second barrier ends the call.  No rank holds more
    than its own rows."""
    import torch
    if world > 1:
        import torch.distributed as dist
    if rank == 0:
        payload = nx * ny * 4
        with open(path, "wb") as f:
            f.write(header)
            f.truncate(len(header) + payload + (-payload % 2880))
    if world > 1:
        dist.barrier()
    n = int(rows.shape[0]) if rows is not None else 0
    if n:
        step = max(1, piece_bytes // (nx * 4))
        pin = torch.empty((min(step, n), nx), dtype=torch.int32, pin_memory=rows.is_cuda)
        fd = os.open(path, os.O_WRONLY)
        try:
            for r in range(0, n, step):
                k = min(step, n - r)
                pin[:k].copy_(rows[r:r + k])
                buf = memoryview(pin[:k].numpy()).cast("B")
                off = len(header) + (row_begin + r) * nx * 4
                done = 0
                while done < len(buf):
                    done += os.pwrite(fd, buf[done:], off + done)
        finally:
            os.close(fd)
    if world > 1:
        dist.barrier()


def read_raster(path):
    """`matplotlib.pyplot.imread` restated over PIL (matplotlib is not a dependency of this build) for the PNG / JPG
    branch of SFinder.run (caesar_yolo/inference.py:511-520).  PNG: float32 in [0, 1] — 8-bit samples / 255, 16-bit
    grey / 65535, palette and grey+alpha images expanded to RGBA first (matplotlib.image._pil_png_to_float_array);
    anything else (JPG): the uint8 array PIL decodes (matplotlib.image.pil_to_array)."""
    from PIL import Image
    with Image.open(path) as im:
        im.load()
        if im.format == 'PNG':
            mode = im.mode
            if mode == '1':
                return np.asarray(im.convert('L'), dtype=np.float32) / np.float32(255)   # bool -> 0 / 1
            if mode == 'L':
                return np.divide(np.asarray(im), 2 ** 8 - 1, dtype=np.float32)
            if mode.startswith('I;16') or mode == 'I':
                a = np.asarray(im)
                return np.divide(a, 2 ** 16 - 1, dtype=np.float32)
            if mode == 'RGB':
                return np.divide(np.asarray(im), 2 ** 8 - 1, dtype=np.float32)
            return np.divide(np.asarray(im.convert('RGBA')), 2 ** 8 - 1, dtype=np.float32)   # P, LA, RGBA, ...
        if im.mode in ('RGBA', 'RGBX', 'RGB', 'L'):
            return np.asarray(im).copy()
        return np.asarray(im.convert('RGBA')).copy()
