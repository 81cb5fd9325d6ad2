"""Plain restatement of the baseline JPEG file libjpeg-turbo writes (Pillow: quality=q, subsampling=0|2, optimize=False,
restart_marker_rows=1), integer step by integer step: the definition of K6's files in include/hmrm.h, in numpy.
Run as a script: compares this model with Pillow byte for byte over sizes, qualities, both chroma modes and several
restart intervals, and prints the largest number of entropy-coded bytes any 8x8 block took."""
import io, sys
import numpy as np
from PIL import Image

LUMA = [16,11,10,16,24,40,51,61,12,12,14,19,26,58,60,55,14,13,16,24,40,57,69,56,14,17,22,29,51,87,80,62,
        18,22,37,56,68,109,103,77,24,35,55,64,81,104,113,92,49,64,78,87,103,121,120,101,72,92,95,98,112,100,103,99]
CHROMA = [17,18,24,47,99,99,99,99,18,21,26,66,99,99,99,99,24,26,56,99,99,99,99,99,47,66,99,99,99,99,99,99] + [99]*32
ZZ = [0,1,8,16,9,2,3,10,17,24,32,25,18,11,4,5,12,19,26,33,40,48,41,34,27,20,13,6,7,14,21,28,
      35,42,49,56,57,50,43,36,29,22,15,23,30,37,44,51,58,59,52,45,38,31,39,46,53,60,61,54,47,55,62,63]
DC_L = ([0,1,5,1,1,1,1,1,1,0,0,0,0,0,0,0], list(range(12)))
DC_C = ([0,3,1,1,1,1,1,1,1,1,1,0,0,0,0,0], list(range(12)))
AC_L = ([0,2,1,3,3,2,4,3,5,5,4,4,0,0,1,0x7d], list(bytes.fromhex(
    '01020300041105122131410613516107227114328191a1082342b1c11552d1f02433627282090a161718191a25262728292a3435363738393a434445464748494a535455565758595a636465666768696a737475767778797a838485868788898a92939495969798999aa2a3a4a5a6a7a8a9aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae1e2e3e4e5e6e7e8e9eaf1f2f3f4f5f6f7f8f9fa')))
AC_C = ([0,2,1,2,4,4,3,4,7,5,4,4,0,1,2,0x77], list(bytes.fromhex(
    '000102031104052131061241510761711322328108144291a1b1c109233352f0156272d10a162434e125f11718191a262728292a35363738393a434445464748494a535455565758595a636465666768696a737475767778797a82838485868788898a92939495969798999aa2a3a4a5a6a7a8a9aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae2e3e4e5e6e7e8e9eaf2f3f4f5f6f7f8f9fa')))


def qtable(base, q):
    s = 5000 // q if q < 50 else 200 - 2 * q
    return [min(255, max(1, (b * s + 50) // 100)) for b in base]


def codes(bits, vals):
    c, k, tab = 0, 0, {}
    for l in range(1, 17):
        for _ in range(bits[l - 1]):
            tab[vals[k]] = (c, l); k += 1; c += 1
        c <<= 1
    return tab


STATS = {'max_block_bytes': 0}
FIX = lambda x: int(x * 65536 + 0.5)
C = dict(c1=2446, c2=3196, c3=4433, c4=6270, c5=7373, c6=9633, c7=12299, c8=15137, c9=16069, c10=16819, c11=20995, c12=25172)


def fdct(blk):  # jfdctint.c (libjpeg 6b / libjpeg-turbo), blk int64 [8][8] level-shifted
    d = blk.astype(np.int64).copy()
    ds = lambda x, n: (x + (1 << (n - 1))) >> n
    for p in range(2):
        out = np.zeros_like(d)
        for r in range(8):
            v = d[r] if p == 0 else d[:, r]
            t0, t7, t1, t6, t2, t5, t3, t4 = v[0]+v[7], v[0]-v[7], v[1]+v[6], v[1]-v[6], v[2]+v[5], v[2]-v[5], v[3]+v[4], v[3]-v[4]
            t10, t13, t11, t12 = t0+t3, t0-t3, t1+t2, t1-t2
            o = [0]*8
            if p == 0:
                o[0] = (t10+t11) << 2; o[4] = (t10-t11) << 2; sh = 11
            else:
                o[0] = ds(t10+t11, 2); o[4] = ds(t10-t11, 2); sh = 15
            z1 = (t12+t13)*C['c3']
            o[2] = ds(z1 + t13*C['c4'], sh); o[6] = ds(z1 - t12*C['c8'], sh)
            z1, z2, z3, z4 = t4+t7, t5+t6, t4+t6, t5+t7
            z5 = (z3+z4)*C['c6']
            t4 *= C['c1']; t5 *= C['c10']; t6 *= C['c12']; t7 *= C['c7']
            z1 *= -C['c5']; z2 *= -C['c11']; z3 *= -C['c9']; z4 *= -C['c2']
            z3 += z5; z4 += z5
            o[7] = ds(t4+z1+z3, sh); o[5] = ds(t5+z2+z4, sh); o[3] = ds(t6+z2+z3, sh); o[1] = ds(t7+z1+z4, sh)
            if p == 0: out[r] = o
            else: out[:, r] = o
        d = out
    return d


def quant(c, q):
    qv = q * 8
    a = abs(int(c)) + (qv >> 1)
    a = a // qv if a >= qv else 0
    return -a if c < 0 else a


def encode(rgb, q, sub420, rst):
    H, W, _ = rgb.shape
    r, g, b = [rgb[..., i].astype(np.int64) for i in range(3)]
    Y = (FIX(0.299)*r + FIX(0.587)*g + FIX(0.114)*b + 32768) >> 16
    Cb = (-FIX(0.16874)*r - FIX(0.33126)*g + FIX(0.5)*b + (128 << 16) + 32767) >> 16
    Cr = (FIX(0.5)*r - FIX(0.41869)*g - FIX(0.08131)*b + (128 << 16) + 32767) >> 16
    cdiv = lambda a, b: -(-a // b)
    hv = 2 if sub420 else 1
    mcux, mcuy = cdiv(W, 8*hv), cdiv(H, 8*hv)
    planes = []
    for ci, P in enumerate((Y, Cb, Cr)):
        if ci == 0 or not sub420:
            wb, hb = cdiv(W, 8), cdiv(H, 8)
            X = np.pad(P, ((0, 0), (0, wb*8 - W)), mode='edge')
        else:
            wb, hb = cdiv(cdiv(W, 2), 8), cdiv(cdiv(H, 2), 8)
            S = np.pad(P, ((0, H % 2), (0, wb*16 - W)), mode='edge')
            s = S[0::2, 0::2] + S[0::2, 1::2] + S[1::2, 0::2] + S[1::2, 1::2]
            bias = np.tile([1, 2], wb*8 // 2)
            X = (s + bias) >> 2
        rows_needed = (mcuy * (hv if (ci == 0 and sub420) else 1)) * 8
        X = np.pad(X, ((0, rows_needed - X.shape[0]), (0, 0)), mode='edge')
        planes.append((X, wb, hb))
    qt = [qtable(LUMA, q), qtable(CHROMA, q)]
    return planes, qt, (mcux, mcuy, hv)


def write(rgb, q, sub420, rst=None):
    """rgb: uint8 [H][W][3 or 4] (alpha ignored); rst: MCUs per restart interval, None = one MCU row (the definition)."""
    rgb = np.ascontiguousarray(rgb[:, :, :3])
    planes, qt, (mcux, mcuy, hv) = encode(rgb, q, sub420, rst)
    if rst is None:
        rst = mcux
    H, W, _ = rgb.shape
    dcs = [codes(*DC_L), codes(*DC_C)]
    acs = [codes(*AC_L), codes(*AC_C)]
    out = bytearray(b'\xff\xd8\xff\xe0\x00\x10JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00')
    for t in (0, 1):
        out += b'\xff\xdb\x00\x43' + bytes([t]) + bytes(qt[t][ZZ[k]] for k in range(64))
    samp = 0x22 if sub420 else 0x11
    out += b'\xff\xc0\x00\x11\x08' + H.to_bytes(2, 'big') + W.to_bytes(2, 'big') + bytes([3, 1, samp, 0, 2, 0x11, 1, 3, 0x11, 1])
    for cls, t, (bits, vals) in ((0, 0, DC_L), (1, 0, AC_L), (0, 1, DC_C), (1, 1, AC_C)):
        out += b'\xff\xc4' + (19 + len(vals)).to_bytes(2, 'big') + bytes([cls << 4 | t] + bits + vals)
    if rst:
        out += b'\xff\xdd\x00\x04' + rst.to_bytes(2, 'big')
    out += bytes.fromhex('ffda000c03010002110311003f00')
    acc, n = [0, 0], [0]
    def bitsout(v, l):
        for i in range(l - 1, -1, -1):
            acc[0] = (acc[0] << 1) | ((v >> i) & 1); acc[1] += 1
            if acc[1] == 8:
                out.append(acc[0]);
                if acc[0] == 0xFF: out.append(0)
                acc[0] = acc[1] = 0
    def flush():
        if acc[1]: bitsout((1 << (8 - acc[1])) - 1, 8 - acc[1])
    cache = {}
    def block(ci, bx, by):
        X, wb, hb = planes[ci]
        key = (ci, bx, by)
        if key not in cache:
            cache[key] = fdct(X[by*8:by*8+8, bx*8:bx*8+8] - 128).reshape(64)
        co = cache[key]
        t = 0 if ci == 0 else 1
        return [quant(co[ZZ[k]], qt[t][ZZ[k]]) for k in range(64)]
    pred = [0, 0, 0]
    mcu = 0
    for my in range(mcuy):
        for mx in range(mcux):
            if rst and mcu and mcu % rst == 0:
                flush(); out += bytes([0xFF, 0xD0 + ((mcu // rst - 1) & 7)]); pred = [0, 0, 0]
            blocks = []
            for ci in range(3):
                X, wb, hb = planes[ci]
                n = hv if (ci == 0 and sub420) else 1
                last = None
                for yy in range(n):
                    rowstart = None
                    for xx in range(n):
                        bx, by = mx*n + xx, my*n + yy
                        if by >= hb:
                            z = [0]*64; z[0] = prev_row_last[0]; blk = z
                        elif bx >= wb:
                            z = [0]*64; z[0] = last[0]; blk = z
                        else:
                            blk = block(ci, bx, by)
                        last = blk
                        blocks.append((ci, blk))
                    prev_row_last = last
            for ci, blk in blocks:
                start_bits = len(out) * 8 + acc[1]
                t = 0 if ci == 0 else 1
                diff = blk[0] - pred[ci]; pred[ci] = blk[0]
                s = abs(diff).bit_length()
                c, l = dcs[t][s]; bitsout(c, l)
                if s: bitsout(diff if diff >= 0 else diff - 1 + (1 << s), s)
                run = 0
                for k in range(1, 64):
                    v = blk[k]
                    if v == 0: run += 1; continue
                    while run > 15:
                        c, l = acs[t][0xF0]; bitsout(c, l); run -= 16
                    s = abs(v).bit_length()
                    c, l = acs[t][(run << 4) | s]; bitsout(c, l)
                    bitsout(v if v >= 0 else v - 1 + (1 << s), s)
                    run = 0
                if run:
                    c, l = acs[t][0]; bitsout(c, l)
                STATS['max_block_bytes'] = max(STATS['max_block_bytes'], (len(out) * 8 + acc[1] - start_bits + 7) // 8)
            mcu += 1
    flush()
    out += b'\xff\xd9'
    return bytes(out)


if __name__ == '__main__':
    rng = np.random.default_rng(0)
    fails = cases = 0
    for (h, w) in [(8, 8), (16, 16), (37, 53), (1, 1), (17, 33), (31, 9), (64, 48), (23, 101), (40, 130), (130, 17)]:
        for kind in ('noise', 'smooth'):
            if kind == 'noise':
                a = rng.integers(0, 256, (h, w, 3)).astype(np.uint8)
            else:
                yy, xx = np.mgrid[0:h, 0:w]
                a = np.stack([(xx*5 + yy*3) % 256, (yy*7) % 256, (xx*xx + yy) % 256], 2).astype(np.uint8)
            for q in (1, 10, 50, 75, 90, 100):
                for ss in (0, 2):
                    for rst in (None, 0, 1, 3):
                        kw = dict(restart_marker_rows=1) if rst is None else dict(restart_marker_blocks=rst) if rst else {}
                        b = io.BytesIO(); Image.fromarray(a).save(b, format='JPEG', quality=q, subsampling=ss, **kw)
                        cases += 1
                        if write(a, q, ss == 2, rst) != b.getvalue():
                            fails += 1
                            print('DIFF', h, w, kind, q, ss, rst)
    print(cases, 'cases,', fails, 'differ from Pillow; largest entropy-coded block:', STATS['max_block_bytes'], 'bytes')
