"""TEST INFRASTRUCTURE ONLY -- numpy + cv2 restatement of the reference `process_frame`.

Follows /root/reference/utils/color_correction/color_balance.cpp step by step (line numbers in the
comments) for every branch except the HSI one (702-774: float `acos` + `std::rand()` quickselect,
out of scope, SURVEY.md 8a P2).  tests/test_oracle_ref.py checks it byte-for-byte against the
compiled reference (oracle/ref_balance.py), which pins this restatement.

It exists (next to the compiled reference) because it exposes the intermediate statistics
(percentile bounds, means, gains, look-up tables) that the CUDA stats kernel is tested against.
"""
import numpy as np
import cv2


def percentile_min_max(channel, lower_perc=0.002, upper_perc=0.998):
    """color_balance.cpp:112-142.  The bounds are float32 products truncated to int."""
    n = int(channel.size)
    low_bound = int(np.float32(lower_perc) * np.float32(n))
    high_bound = n - int(np.float32(upper_perc) * np.float32(n))
    counts = np.bincount(channel.reshape(-1), minlength=256).astype(np.int64)
    return percentile_from_counts(counts, low_bound, high_bound)


def percentile_from_counts(counts, low_bound, high_bound):
    lo = hi = None
    for i in range(256):
        if low_bound < counts[i]:
            lo = i
            break
        low_bound -= int(counts[i])
    for i in range(255, -1, -1):
        if high_bound < counts[i]:
            hi = i
            break
        high_bound -= int(counts[i])
    return lo, hi


def constrain(val):
    """color_balance.cpp:13-23 with low=0, high=255: clamp in double, then truncate.  NaN (0 * inf, a zero
    channel mean) passes both comparisons and is undefined behaviour in the reference; defined as 0, as on the
    device (csrc/balance.cu, constrain255)."""
    val = np.asarray(val, dtype=np.float64)
    val = np.where(np.isnan(val), 0.0, val)
    return np.where(val < 0, 0, np.where(val > 255, 255, np.floor(val))).astype(np.uint8)


def _uchar_cast(val):
    """`(unsigned char)double` as g++ emits it on x86-64: cvttsd2si to a 32-bit int, then the low byte.  NaN and values
    outside the int range give INT_MIN there, whose low byte is 0.  Both are undefined behaviour in C++; this is what
    the compiled reference does and what the device defines (csrc/balance.cu, uchar_cast)."""
    val = np.asarray(val, dtype=np.float64)
    bad = np.isnan(val) | (val >= 2147483648.0) | (val <= -2147483649.0)
    return np.where(bad, 0, np.trunc(np.where(bad, 0.0, val)).astype(np.int64) & 0xFF).astype(np.uint8)


def sv_stretch(ch, lo, hi, zero_width_stretch="raise"):
    """color_balance.cpp:683-686 on a clipped S or V plane: int32 arithmetic, C division (operands are non-negative).
    A zero-width range divides by zero in the reference (integer SIGFPE): "raise" reports it; "zero" applies the
    device's definition (csrc/balance.cu, stats_sv_block), a table of 0 for that channel."""
    if hi == lo:
        if zero_width_stretch == "zero":
            return np.zeros_like(ch)
        raise ZeroDivisionError("reference divides by zero here (684-685, integer SIGFPE)")
    return (((ch.astype(np.int32) - lo) * 255) // (hi - lo)).astype(np.uint8)


def running_mean(values):
    """color_balance.cpp:459-470: m += (x - m) / k, strictly sequential in double."""
    m = 0.0
    for k, x in enumerate(np.asarray(values, dtype=np.float64).tolist(), start=1):
        m += (x - m) / k
    return m


def equalize_lut(x_gain, adaptive):
    """LUT over x=0..255 of the per-pixel gain expression (489-495)."""
    x = np.arange(256, dtype=np.float64)
    if adaptive:
        return constrain(x * (np.power((255. - x) / 255., 0.25) * (x_gain - 1.) + 1.))
    return constrain(x * x_gain)



# ---------------------------------------------------------------------------------------------
# HSI contrast branch (P2)
# ---------------------------------------------------------------------------------------------
f32 = np.float32
f64 = np.float64
PI = np.pi


def uchar_clip(x):
    """(int)f then clamp to 0..255; NaN / out-of-range float->int conversion gives INT_MIN on x86."""
    x=np.asarray(x,dtype=np.float32)
    bad=~np.isfinite(x) | (np.abs(x)>=2147483648.0)
    n=np.where(bad, -2147483648, np.trunc(np.where(bad,0,x))).astype(np.int64)
    return np.clip(n,0,255).astype(np.uint8)
def clip_f(ch, lo, hi):
    lo=f32(lo); hi=f32(hi)
    out=ch.copy()
    lt=ch<lo; gt=~lt&(ch>hi); nan=~lt&~gt&np.isnan(ch)
    out[lt]=lo; out[gt]=hi; out[nan]=lo
    return out
def hsi_branch(b, g, r):
    """color_balance.cpp:702-774 on flat uint8 planes (after the other stages); returns new (b, g, r).
    Every float / double conversion follows the compiled reference (0 differing bytes against oracle/_ref on
    frames of >= 128 k pixels; below that the reference's second quickselect starts at index (int)min_value and its
    result depends on std::rand()).  cos / acos are the double-precision libm functions, as in the reference."""
    n=b.size
    rf,gf,bf=r.astype(f32),g.astype(f32),b.astype(f32)
    I=((rf+gf).astype(f32)+bf).astype(f32).astype(f64)/3.0
    I=I.astype(f32)
    mn=np.minimum(np.minimum(r,g),b).astype(f32)
    with np.errstate(all='ignore'):
        S=np.where(I>0, (1.0-((mn/I).astype(f32).astype(f64))), 0.0).astype(f32)
        num=rf.astype(f64)-(0.5*g.astype(f64))-(0.5*b.astype(f64))
        ri,gi,bi=r.astype(np.int64),g.astype(np.int64),b.astype(np.int64)
        # (float)r*r + (float)g*g + (float)b*b - (float)(r*g) - (float)(r*b) - (float)(g*b)  : float arithmetic
        t=(rf*rf).astype(f32); t=(t+(gf*gf).astype(f32)).astype(f32); t=(t+(bf*bf).astype(f32)).astype(f32)
        t=(t-(ri*gi).astype(f32)).astype(f32); t=(t-(ri*bi).astype(f32)).astype(f32); t=(t-(gi*bi).astype(f32)).astype(f32)
        den=np.sqrt(t.astype(f64))
        H=np.arccos(num/den).astype(f32)
        H=np.where(b>g, (PI*2-H.astype(f64)).astype(f32), H)
    H=clip_f(H,0.,2.*PI); S=clip_f(S,0.,1.); I=clip_f(I,0.,255.)
    def pct(ch):
        lo=int(f32(0.002)*f32(n)); hi=int(f32(0.998)*f32(n))
        s=np.sort(ch)
        return s[lo], s[hi]
    smin,smax=pct(S); S=clip_f(S,smin,smax)
    imin,imax=pct(I); I=clip_f(I,imin,imax)
    with np.errstate(all='ignore'):
        s_mult=f32(1.0/f64(f32(smax-smin)))       # 750-751: float subtraction, double division
        i_mult=f32(255.0/f64(f32(imax-imin)))
        S=((S-smin).astype(f32)*s_mult).astype(f32); I=((I-imin).astype(f32)*i_mult).astype(f32)
    S=clip_f(S,0.,1.); I=clip_f(I,0.,255.)
    h,s,i=H,S,I
    hd,sd,idd=h.astype(f64),s.astype(f64),i.astype(f64)
    def cosh(x32):   # cos(h) with float argument
        return np.cos(x32.astype(f64))
    is_ = (i*s).astype(f32)           # i * s float
    ims = (i-is_).astype(f32)         # i - i*s
    ip2 = (i+((f32(2)*i).astype(f32)*s).astype(f32)).astype(f32)   # i + 2*i*s
    eps=1e-6
    feq0=np.abs(h-f32(0))<eps
    feq1=np.abs((h-f32(2.*PI/3.)).astype(f32))<eps
    feq2=np.abs((h-f32(4.*PI/3.)).astype(f32))<eps
    R=np.zeros(n,np.uint8);G=np.zeros(n,np.uint8);B=np.zeros(n,np.uint8)
    with np.errstate(all='ignore'):
        # sector 1
        c1=cosh(h)/np.cos(PI/3.-hd); v1=is_.astype(f64)*c1
        r1=uchar_clip((idd+v1).astype(f32)); g1=uchar_clip((idd+is_.astype(f64)*(1-c1)).astype(f32))
        c2=np.cos(hd-2.*PI/3.)/np.cos(PI-hd)
        g2=uchar_clip((idd+is_.astype(f64)*c2).astype(f32)); b2=uchar_clip((idd+is_.astype(f64)*(1-c2)).astype(f32))
        c3=np.cos(hd-4.*PI/3.)/np.cos(5.*PI/3.-hd)
        r3=uchar_clip((idd+is_.astype(f64)*(1-c3)).astype(f32)); b3=uchar_clip((idd+is_.astype(f64)*c3).astype(f32))
    lo=uchar_clip(ims); hi_=uchar_clip(ip2)
    m0=feq0
    m1=~m0&(0.<hd)&(hd<2.*PI/3.)
    m2=~m0&~m1&feq1
    m3=~m0&~m1&~m2&(2.*PI/3.<hd)&(hd<4.*PI/3.)
    m4=~m0&~m1&~m2&~m3&feq2
    m5=~(m0|m1|m2|m3|m4)
    R[m0]=hi_[m0];G[m0]=lo[m0];B[m0]=lo[m0]
    R[m1]=r1[m1];G[m1]=g1[m1];B[m1]=lo[m1]
    R[m2]=lo[m2];G[m2]=hi_[m2];B[m2]=lo[m2]
    R[m3]=lo[m3];G[m3]=g2[m3];B[m3]=b2[m3]
    R[m4]=lo[m4];G[m4]=lo[m4];B[m4]=hi_[m4]
    R[m5]=r3[m5];G[m5]=lo[m5];B[m5]=b3[m5]
    return B,G,R

def process_frame_np(img, equalize_rgb=True, rgb_contrast_correct=False,
                     hsv_contrast_correct=True, hsi_contrast_correct=False,
                     rgb_extrema_clipping=True, adaptive_cast_correction=False,
                     horizontal_blocks=1, vertical_blocks=1, sequential_mean=False,
                     return_stats=False, zero_width_stretch="raise"):
    """Returns the balanced BGR image (new array).  `sequential_mean=True` reproduces the running
    mean of 459-470 literally (python loop: small frames only); otherwise the exact mean is used,
    which the running mean equals to <=1.2e-12 (SURVEY.md A.7).  `zero_width_stretch`: what a zero-width S or V
    range does (sv_stretch): "raise" (the reference divides by zero) or "zero" (the device's definition)."""
    if zero_width_stretch not in ("raise", "zero"):
        raise ValueError("zero_width_stretch must be 'raise' or 'zero', not %r" % (zero_width_stretch,))
    if hsi_contrast_correct:                                               # 702-774: after every other stage
        rest = process_frame_np(img, equalize_rgb, rgb_contrast_correct, hsv_contrast_correct, False, rgb_extrema_clipping,
                                adaptive_cast_correction, horizontal_blocks, vertical_blocks, sequential_mean, return_stats,
                                zero_width_stretch)
        base, st = rest if return_stats else (rest, None)
        nb, ng, nr = hsi_branch(base[..., 0].reshape(-1), base[..., 1].reshape(-1), base[..., 2].reshape(-1))
        out = np.stack([nb, ng, nr], axis=-1).reshape(base.shape)
        return (out, st) if return_stats else out
    img = np.ascontiguousarray(img, dtype=np.uint8)
    height, width = img.shape[:2]
    n = height * width
    b = img[..., 0].reshape(-1).copy()                                      # 371-375
    g = img[..., 1].reshape(-1).copy()
    r = img[..., 2].reshape(-1).copy()
    stats = {}

    if rgb_extrema_clipping:                                               # 398-419 (order r, g, b)
        r_min, r_max = percentile_min_max(r)
        np.clip(r, r_min, r_max, out=r)
        g_min, g_max = percentile_min_max(g)
        np.clip(g, g_min, g_max, out=g)
        b_min, b_max = percentile_min_max(b)
        np.clip(b, b_min, b_max, out=b)
    else:                                                                  # 421-423
        r_min, r_max = int(r.min()), int(r.max())
        g_min, g_max = int(g.min()), int(g.max())
        b_min, b_max = int(b.min()), int(b.max())
    r_avg = float(int(r.sum(dtype=np.int64))) / n                            # 426-428
    g_avg = float(int(g.sum(dtype=np.int64))) / n
    b_avg = float(int(b.sum(dtype=np.int64))) / n
    stats.update(bgr_min=(b_min, g_min, r_min), bgr_max=(b_max, g_max, r_max),
                 bgr_avg=(b_avg, g_avg, r_avg), tiles=[])

    if equalize_rgb:                                                       # 441-544
        if width % horizontal_blocks or height % vertical_blocks:
            raise NotImplementedError("non-divisible tilings walk out of the row (SURVEY.md App. C)")
        bw, bh = width // horizontal_blocks, height // vertical_blocks
        r2, g2, b2 = r.reshape(height, width), g.reshape(height, width), b.reshape(height, width)
        for by in range(vertical_blocks):
            for bx in range(horizontal_blocks):
                sl = (slice(by * bh, (by + 1) * bh), slice(bx * bw, (bx + 1) * bw))
                if sequential_mean:
                    lr, lg, lb = running_mean(r2[sl].reshape(-1)), running_mean(g2[sl].reshape(-1)), \
                        running_mean(b2[sl].reshape(-1))
                else:
                    cnt = bw * bh
                    lr = float(int(r2[sl].sum(dtype=np.int64))) / cnt
                    lg = float(int(g2[sl].sum(dtype=np.int64))) / cnt
                    lb = float(int(b2[sl].sum(dtype=np.int64))) / cnt
                # 474: the unqualified abs() resolves to int abs(int) in the compiled reference (g++ 13,
                # <cmath>/<cstdlib> only): the difference is truncated toward zero before the comparison
                # (verified against oracle/_ref: a double fabs changes 18 683 bytes on a 4x2 tiling)
                if abs(int(lr - r_avg)) > r_avg / 6 or abs(int(lb - b_avg)) > b_avg / 6 or \
                        abs(int(lg - g_avg)) > g_avg / 6:
                    lr, lg, lb = r_avg, g_avg, b_avg
                with np.errstate(divide="ignore", invalid="ignore"):
                    if lr > lg and lr > lb:                                # 480: red cast
                        dom = "r"
                        g2[sl] = equalize_lut(np.float64(lr) / np.float64(lg), adaptive_cast_correction)[g2[sl]]
                        b2[sl] = equalize_lut(np.float64(lr) / np.float64(lb), adaptive_cast_correction)[b2[sl]]
                    elif lg > lr and lg > lb:                              # 501: green cast
                        dom = "g"
                        r2[sl] = equalize_lut(np.float64(lg) / np.float64(lr), adaptive_cast_correction)[r2[sl]]
                        b2[sl] = equalize_lut(np.float64(lg) / np.float64(lb), adaptive_cast_correction)[b2[sl]]
                    else:                                                  # 522: blue cast
                        dom = "b"
                        r2[sl] = equalize_lut(np.float64(lb) / np.float64(lr), adaptive_cast_correction)[r2[sl]]
                        g2[sl] = equalize_lut(np.float64(lb) / np.float64(lg), adaptive_cast_correction)[g2[sl]]
                stats["tiles"].append(dict(dom=dom, local=(lb, lg, lr)))

    if rgb_contrast_correct:                                               # 546-645
        chans = {"r": (r, r_min, r_max, r_avg), "g": (g, g_min, g_max, g_avg), "b": (b, b_min, b_max, b_avg)}
        if r_avg > g_avg:                                                  # 560-593
            if r_avg > b_avg:
                order = ("r", "g", "b") if g_avg > b_avg else ("r", "b", "g")
            else:
                order = ("b", "r", "g")
        else:                                                              # 594-627
            if g_avg > b_avg:
                order = ("g", "r", "b") if r_avg > b_avg else ("g", "b", "r")
            else:
                order = ("b", "g", "r")
        (mx, mx_min, mx_max, _), (md, md_min, md_max, _), (mn, mn_min, mn_max, _) = (chans[k] for k in order)
        desired_max = float((mn_max + md_max + mx_max) // 3)               # 629 (int division)
        with np.errstate(divide="ignore", invalid="ignore"):
            mn_ratio = np.float64(desired_max - mn_min) / np.float64(mn_max - mn_min)
            md_ratio = np.float64(desired_max) / np.float64(md_max - md_min)
            mx_ratio = np.float64(mx_max) / np.float64(mx_max - mx_min)
            mn[:] = _uchar_cast((mn.astype(np.int64) - mn_min) * mn_ratio)  # 634-640
            md[:] = _uchar_cast((md.astype(np.int64) - md_min) * md_ratio)
            mx[:] = _uchar_cast((mx.astype(np.int64) - mx_min) * mx_ratio)
        stats["rgb_cc"] = dict(order=order, ratios=(float(mn_ratio), float(md_ratio), float(mx_ratio)))

    if hsv_contrast_correct:                                               # 647-700
        bgr = np.stack([b, g, r], axis=-1).reshape(height, width, 3)
        hsv = cv2.cvtColor(bgr, cv2.COLOR_BGR2HSV)                         # 654
        h = hsv[..., 0].reshape(-1).copy()
        s = hsv[..., 1].reshape(-1).copy()
        v = hsv[..., 2].reshape(-1).copy()
        s_min, s_max = percentile_min_max(s)                               # 671-675
        np.clip(s, s_min, s_max, out=s)
        v_min, v_max = percentile_min_max(v)                               # 677-681
        np.clip(v, v_min, v_max, out=v)
        s = sv_stretch(s, s_min, s_max, zero_width_stretch)                # 683-686
        v = sv_stretch(v, v_min, v_max, zero_width_stretch)
        hsv2 = np.stack([h, s, v], axis=-1).reshape(height, width, 3)
        out = cv2.cvtColor(hsv2, cv2.COLOR_HSV2BGR)                        # 693
        stats.update(s_min=s_min, s_max=s_max, v_min=v_min, v_max=v_max)
    else:
        out = np.stack([b, g, r], axis=-1).reshape(height, width, 3)       # 776
    out = np.ascontiguousarray(out)
    return (out, stats) if return_stats else out
