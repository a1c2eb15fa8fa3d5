"""Host-side launch helpers: torch tensors in, C-ABI calls out (include/extdm_b200.h).

Every helper goes through a `Recorder`: in immediate mode the call is issued on the current CUDA
stream; in record mode it is appended to a launch list that a model runner replays (and captures into a
CUDA graph).  Nothing here computes with torch ops on the hot path -- torch only provides device memory.
"""
import ctypes as C

import torch

from . import lib as _lib

BF16 = torch.bfloat16


# ----------------------------------------------------------------------------- recorder
class Recorder:
    """Immediate or deferred issue of C-ABI launches (stream appended as the last argument)."""

    def __init__(self, record=False):
        self.record = record
        self.steps = []          # (cfunc, args, name)
        self.keep = []           # tensors / ctypes objects that must outlive the launch list
        self.meta = []           # per-launch algorithmic work (flops / bytes) for bench.py's roofline

    def emit(self, name, args, keep=(), meta=None):
        if self.record:
            self.keep.extend(keep)
            self.steps.append((getattr(_lib.load(), name), args, name))
            self.meta.append(meta or {})
        else:
            _lib.call(name, *args, C.c_void_p(torch.cuda.current_stream().cuda_stream))

    def run(self):
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        lib = _lib.load()
        for fn, args, name in self.steps:
            rc = fn(*args, stream)
            if rc != 0:
                raise _lib.ExtdmError(f"{name} failed ({rc}): {lib.extdm_last_error().decode()}")
        _lib._launches += len(self.steps)

    def __len__(self):
        return len(self.steps)

    def run_timed(self):
        """Eager replay with one CUDA-event pair per launch -> list of (name, meta, milliseconds)."""
        stream = torch.cuda.current_stream()
        sp = C.c_void_p(stream.cuda_stream)
        evs = []
        for fn, args, name in self.steps:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            rc = fn(*args, sp)
            b.record(stream)
            if rc != 0:
                raise _lib.ExtdmError(f"{name} failed ({rc})")
            evs.append((a, b))
        torch.cuda.synchronize()
        return [(name, m, a.elapsed_time(b)) for (_, _, name), m, (a, b) in zip(self.steps, self.meta, evs)]


IMMEDIATE = Recorder(record=False)


def _p(t):
    return C.c_void_p(0 if t is None else t.data_ptr())


def _chk(t, dtype, name):
    if t is None:
        return
    if not t.is_cuda or t.dtype != dtype or not t.is_contiguous():
        raise ValueError(f"{name}: expected contiguous CUDA {dtype}, got {t.dtype} cuda={t.is_cuda} "
                         f"contig={t.is_contiguous()}")


# ----------------------------------------------------------------------------- weight packing (load time)
def pack_conv_weight(w):
    """(Cout, Cin, [1,] kh, kw) fp32 -> (Cout, kh*kw*Cin) bf16, K index = (ky*kw + kx)*Cin + ci."""
    if w.dim() == 5:
        w = w[:, :, 0]
    co, ci, kh, kw = w.shape
    return w.permute(0, 2, 3, 1).reshape(co, kh * kw * ci).to(BF16).contiguous()


def pack_conv3d_weight(w):
    """(Cout, Cin, kt, kh, kw) fp32 -> (Cout, kt*kh*kw*Cin) bf16, K index = ((kt*kh + ky)*kw + kx)*Cin + ci."""
    co, ci, kt, kh, kw = w.shape
    return w.permute(0, 2, 3, 4, 1).reshape(co, kt * kh * kw * ci).to(BF16).contiguous()


def pack_linear_weight(w):
    return w.reshape(w.shape[0], -1).to(BF16).contiguous()


def pack_downsample_weight(w):
    """Conv3d (1,4,4)/s2/p1 weight (Cout, Cin, 1, 4, 4) -> 2x2 taps over the space-to-depth tensor:
    K index = (a*2+b)*4Cin + (py*2+px)*Cin + ci with ky = 2a+py, kx = 2b+px."""
    co, ci = w.shape[:2]
    w = w[:, :, 0].reshape(co, ci, 2, 2, 2, 2)             # co ci a py b px
    return w.permute(0, 2, 4, 3, 5, 1).reshape(co, 16 * ci).to(BF16).contiguous()


# output phase py -> [(input offset dy, kernel index ky)] for ConvTranspose (k=4, s=2, p=1): o = 2i - 1 + k
_UP_TAPS = {0: [(0, 1), (-1, 3)], 1: [(1, 0), (0, 2)]}


def pack_upsample_weight(w):
    """ConvTranspose3d weight (Cin, Cout, 1, 4, 4) -> 4 phase matrices (Cout, 4*Cin) bf16 + tap offsets."""
    ci, co = w.shape[:2]
    w = w[:, :, 0]
    out = {}
    for py in (0, 1):
        for px in (0, 1):
            mats, taps = [], []
            for dy, ky in _UP_TAPS[py]:
                for dx, kx in _UP_TAPS[px]:
                    mats.append(w[:, :, ky, kx].t())       # (co, ci)
                    taps.append((dx, dy, 0))
            out[(py, px)] = (torch.cat(mats, dim=1).to(BF16).contiguous(), taps)
    return out


def pack_upsample_weight_merged(w):
    """The four phase matrices stacked along the output rows -> ((4*Cout, 4*Cin) bf16, [taps of phase p], [(py, px)]):
    one launch of the phase-aware GEMM computes the whole ConvTranspose (upsample_cl)."""
    per = pack_upsample_weight(w)
    order = [(0, 0), (0, 1), (1, 0), (1, 1)]
    return torch.cat([per[ph][0] for ph in order], dim=0).contiguous(), [per[ph][1] for ph in order], order


def conv_taps(k):
    return [(kx - k // 2, ky - k // 2, 0) for ky in range(k) for kx in range(k)]


def conv3d_taps(k):
    return [(kx - k // 2, ky - k // 2, kt - k // 2) for kt in range(k) for ky in range(k) for kx in range(k)]


def std_box(H, W):
    """128-row tile as (bw, bh, bt) pixels."""
    bw = min(W, 128)
    bh = min(H, 128 // bw)
    bt = 128 // (bw * bh)
    return bw, bh, bt


# ----------------------------------------------------------------------------- GEMM
def gemm(rec, *, a0, c0, dims, strides0, box, start, count, taps, w, n, out, out_stride, out_base=0,
         a1=None, c1=0, strides1=None, out_fp32=False, col_group=None, col_group_stride=0, bias=None,
         res=None, res_fp32=False, res_base=0, res_stride=None, col_scale=None, col_shift=None, act=0,
         block_n=0, gn_partials=None, a1_offset=0, tf32=False, phases=None):
    """Generic launch of extdm_conv_gemm.  dims/strides: extents and element strides of D1..D4 of the A
    tensor(s); box/start/count: tile geometry; taps: list of (o1,o2,o3).
    phases: [(taps_p, out_offset_p), ...] -- several products over the same A tiles in one launch (ExtdmGemm.n_phase):
    phase p uses its own taps, the weight rows [p*n, (p+1)*n) and writes at out_base + out_offset_p."""
    if phases is not None:
        taps = phases[0][0]
        if any(len(tp) != len(taps) for tp, _ in phases):
            raise ValueError("gemm: every phase needs the same number of taps")
    g = _lib.ExtdmGemm()
    g.a0 = a0.data_ptr()
    g.a1 = 0 if a1 is None else a1.data_ptr() + 2 * a1_offset
    g.a0_channels, g.a1_channels = c0, (c1 if a1 is not None else 0)
    for i in range(4):
        g.a0_dim[i], g.a0_stride[i] = dims[i], strides0[i]
        g.a1_dim[i] = dims[i]
        g.a1_stride[i] = (strides1 or strides0)[i]
        g.box[i], g.start[i], g.count[i] = box[i], start[i], count[i]
        g.out_stride[i] = out_stride[i]
        g.res_stride[i] = (res_stride or out_stride)[i]
    g.ntaps = len(taps)
    all_taps = taps if phases is None else [t for tp, _ in phases for t in tp]
    for i, t in enumerate(all_taps):
        g.tap[i][0], g.tap[i][1], g.tap[i][2], g.tap[i][3] = t[0], t[1], t[2], 0
    n_phase = 1 if phases is None else len(phases)
    g.n_phase = n_phase
    for i in range(n_phase if phases is not None else 0):
        g.phase_out_offset[i] = phases[i][1]
    _chk(w, BF16, "gemm weight")
    if w.shape[1] != len(taps) * (c0 + (c1 if a1 is not None else 0)):
        raise ValueError(f"gemm: weight K {w.shape[1]} != taps*channels {len(taps)}*{c0}+{c1}")
    g.w, g.n, g.w_rows = w.data_ptr(), n, w.shape[0]
    g.out, g.out_fp32, g.out_base = out.data_ptr(), int(out_fp32), out_base
    g.col_group = col_group if col_group else max(n, 1)
    g.col_group_stride = col_group_stride
    g.bias = 0 if bias is None else bias.data_ptr()
    g.res = 0 if res is None else res.data_ptr()
    g.res_fp32, g.res_base = int(res_fp32), res_base
    g.col_scale = 0 if col_scale is None else col_scale.data_ptr()
    g.col_shift = 0 if col_shift is None else col_shift.data_ptr()
    g.act, g.block_n = act, block_n
    g.gn_partials = 0 if gn_partials is None else gn_partials.data_ptr()
    g.tf32 = int(tf32)
    rows = count[0] * count[1] * count[2] * count[3]
    ktot = len(taps) * (c0 + (c1 if a1 is not None else 0))
    if tf32:
        ktot //= 2                                       # channel counts are in 2-byte units: K in fp32 elements
    meta = dict(flops=2.0 * rows * n * ktot * n_phase, rows=rows, n=n, k=ktot, taps=len(taps), tf32=bool(tf32),
                bytes=2.0 * rows * (c0 + (c1 if a1 is not None else 0)) + n_phase * (2.0 * n * ktot
                + rows * n * (4.0 if out_fp32 else 2.0)))
    if n_phase > 1:
        meta["phases"] = n_phase
    rec.emit("extdm_conv_gemm", (C.byref(g),), keep=(g, a0, a1, w, out, bias, res, col_scale, col_shift, gn_partials),
             meta=meta)


def linear_rows(rec, x, w, n, out, *, bias=None, res=None, res_fp32=False, act=0, out_fp32=False, x2=None,
                block_n=0):
    """out[r, :n] = x[r, :] @ w.T (+bias, +res, act) for dense row-major x (rows, C) [+ x2 (rows, C2)]."""
    rows, c0 = x.numel() // x.shape[-1], x.shape[-1]
    c1 = 0 if x2 is None else x2.shape[-1]
    ld_out = out.shape[-1]
    gemm(rec, a0=x, c0=c0, a1=x2, c1=c1, dims=(rows, 1, 1, 1), strides0=(c0, rows * c0, rows * c0, rows * c0),
         strides1=None if x2 is None else (c1, rows * c1, rows * c1, rows * c1),
         box=(128, 1, 1, 1), start=(0, 0, 0, 0), count=(rows, 1, 1, 1), taps=[(0, 0, 0)], w=w, n=n, out=out,
         out_stride=(ld_out, 0, 0, 0), out_fp32=out_fp32, bias=bias, res=res, res_fp32=res_fp32,
         res_stride=None if res is None else (res.shape[-1], 0, 0, 0), act=act, block_n=block_n)


def conv_cl(rec, x, w, n, k, out, *, x2=None, bias=None, res=None, res_fp32=False, act=0, out_fp32=False,
            t_range=None, col_scale=None, col_shift=None, out_t_offset=0, res_t_offset=0, taps=None,
            out_scale=1, out_phase=(0, 0), block_n=0, gn_partials=None, x2_t_offset=0, tf32=False, out_pixel_offset=(0, 0)):
    """k x k 'same' convolution over channels-last x (B, T, H, W, C) [channel-concatenated with x2].
    out: (B, To, Ho, Wo, n') with n' >= n.  t_range=(t0, t1) restricts the frames computed; the output
    frame index is t + out_t_offset.  out_scale/out_phase write a strided output (ConvTranspose phases);
    out_pixel_offset (dy, dx) shifts the output pixel (writing the interior of a padded tensor)."""
    B, T, H, W, c0 = x.shape
    c1 = 0 if x2 is None else x2.shape[-1]
    bw, bh, bt = std_box(H, W)
    t0, t1 = t_range if t_range else (0, T)
    oB, oT, oH, oW, oC = out.shape
    s = out_scale
    ostr = (s * oC, s * oW * oC, oH * oW * oC, oT * oH * oW * oC)
    obase = out_t_offset * oH * oW * oC + ((out_phase[0] + out_pixel_offset[0]) * oW + out_phase[1] + out_pixel_offset[1]) * oC
    rstr, rbase = None, 0
    if res is not None:
        rB, rT, rH, rW, rC = res.shape
        rstr = (rC, rW * rC, rH * rW * rC, rT * rH * rW * rC)
        rbase = res_t_offset * rH * rW * rC
    # x2_t_offset: frame t of x pairs with frame t - x2_t_offset of x2 (a dense tensor holding only a frame range)
    gemm(rec, a0=x, c0=c0, a1=x2, c1=c1, dims=(W, H, T, B), a1_offset=-x2_t_offset * H * W * c1,
         strides0=(c0, W * c0, H * W * c0, T * H * W * c0),
         strides1=None if x2 is None else (c1, W * c1, H * W * c1, x2.shape[1] * H * W * c1),
         box=(bw, bh, bt, 1), start=(0, 0, t0, 0), count=(W, H, t1 - t0, B),
         taps=taps if taps is not None else conv_taps(k), w=w, n=n, out=out, out_stride=ostr, out_base=obase,
         out_fp32=out_fp32, bias=bias, res=res, res_fp32=res_fp32, res_base=rbase, res_stride=rstr,
         col_scale=col_scale, col_shift=col_shift, act=act, block_n=block_n, gn_partials=gn_partials, tf32=tf32)


def upsample_cl(rec, x, merged, n, out, *, bias=None):
    """ConvTranspose3d (1,4,4)/s2/p1 of channels-last x (B, T, H, W, C) -> out (B, T, 2H, 2W, n) as ONE launch: the four
    sub-pixel phases are 2x2-tap products over the same input tiles (merged = pack_upsample_weight_merged(weight))."""
    wm, taps, order = merged
    B, T, H, W, c0 = x.shape
    bw, bh, bt = std_box(H, W)
    oB, oT, oH, oW, oC = out.shape
    gemm(rec, a0=x, c0=c0, dims=(W, H, T, B), strides0=(c0, W * c0, H * W * c0, T * H * W * c0),
         box=(bw, bh, bt, 1), start=(0, 0, 0, 0), count=(W, H, T, B), taps=taps[0], w=wm, n=n, out=out,
         out_stride=(2 * oC, 2 * oW * oC, oH * oW * oC, oT * oH * oW * oC), bias=bias,
         phases=[(taps[i], (py * oW + px) * oC) for i, (py, px) in enumerate(order)])


def pack_conv_weight_f32(w, cin_pad=None, splits=None):
    """(Cout, Cin, kh, kw) fp32 -> (Cout, kh*kw*Cin') fp32 for the tf32 GEMM mode, K index = tap*Cin' + c.
    splits = [(c_begin, c_end, c_padded), ...] re-lays the input channels as several zero-padded groups
    (channel-concatenated sources whose widths are not multiples of 32)."""
    co, ci, kh, kw = w.shape
    if splits is None:
        splits = [(0, ci, cin_pad or ci)]
    parts = []
    for b, e, cp in splits:
        blk = torch.zeros(co, kh, kw, cp, device=w.device, dtype=torch.float32)
        blk[..., : e - b] = w[:, b:e].permute(0, 2, 3, 1)
        parts.append(blk)
    out = torch.cat(parts, dim=3).reshape(co, -1).contiguous()
    # round to the nearest tf32 (the tensor core would truncate the low 13 mantissa bits)
    bits = out.view(torch.int32)
    return ((bits + 0x1000) & ~0x1FFF).view(torch.float32)


def conv_cl_tf32(rec, x, w, n, k, out, *, x2=None, bias=None, act=0, taps=None, round_out=True):
    """k x k 'same' convolution of fp32 channels-last x (F, H, W, C) [| x2] in tf32 (fp32 accumulate), fp32 output
    (F, H, W, n') -- the LFAE conditioning convolutions (the reference's cuDNN path runs them in TF32 as well).
    w: pack_conv_weight_f32 layout; channel counts are multiples of 32.  round_out: the output feeds another tf32
    convolution (stored rounded to tf32); False for the heads whose logits are consumed in fp32."""
    for t in (x, x2, w, out):
        if t is not None and t.dtype != torch.float32:
            raise ValueError("conv_cl_tf32: fp32 tensors expected")
    # frames ride on the T axis so that one 128-row tile spans several small frames (the hourglass goes down to 1x1)
    v = lambda t: None if t is None else t.view(BF16).view(1, t.shape[0], t.shape[1], t.shape[2], 2 * t.shape[3])
    conv_cl(rec, v(x), w.view(BF16), n, k, out.view(1, *out.shape), x2=v(x2), bias=bias, act=act,
            out_fp32=True, taps=taps, tf32=2 if round_out else 1)


def conv_tiles_per_sample(T, H, W):
    """Number of 128-row GEMM tiles conv_cl cuts one sample's (T, H, W) volume into (= GroupNorm partials per sample)."""
    bw, bh, bt = std_box(H, W)
    return -(-W // bw) * -(-H // bh) * -(-T // bt)


def gn_parts_per_sample(T, H, W, Cc):
    """GroupNorm partial records (16 floats each) one sample's convolution epilogue writes: per (128-row tile, TMEM lane
    quarter) one record, or C/128 of them when a group is wider than a 16-column chunk (C = 256: 2, C = 512: 4) --
    include/extdm_b200.h: ExtdmGemm.gn_partials."""
    return conv_tiles_per_sample(T, H, W) * 4 * max(1, Cc // 128)


GN_CHUNKS = 32          # EXTDM_GN_CHUNKS


# ----------------------------------------------------------------------------- normalisation etc.
def groupnorm_silu(rec, x, stats_ws, gamma, beta, y, *, groups=8, scale_shift=None, ss_off=0, res=None, eps=1e-5,
                   n_part=None):
    """x, y, res: (B, P..., C) bf16 channels-last.  With n_part=None the statistics are computed here
    (stats_ws: float32 workspace >= B*32*groups*2); otherwise stats_ws already holds n_part partial sums per sample
    written by the producing convolution's epilogue (conv_cl(..., gn_partials=stats_ws))."""
    B, Cc = x.shape[0], x.shape[-1]
    P = x.numel() // (B * Cc)
    if n_part is None:
        rec.emit("extdm_groupnorm_stats", (_p(x), _p(stats_ws), B, P, Cc, groups), keep=(x, stats_ws))
        n_part = GN_CHUNKS
    ss_stride = 0 if scale_shift is None else scale_shift.shape[1]
    rec.emit("extdm_groupnorm_apply", (_p(x), _p(stats_ws), n_part, _p(gamma), _p(beta), _p(scale_shift), ss_stride,
                                       ss_off, _p(res), _p(y), B, P, Cc, groups, C.c_float(eps)),
             keep=(x, stats_ws, gamma, beta, scale_shift, res, y), meta=dict(bytes=(6.0 if res is not None else 4.0) * x.numel(), tag=f"C={Cc} P={P}"))


def chan_layernorm(rec, x, gamma, y, *, x2=None, t_range=None, t2_range=None, eps=1e-5):
    """Channel LayerNorm of frames t_range of x (B, T, H, W, C) [channel-concatenated with frames t2_range
    of x2 (B, T2, H, W, C)] -> dense y (B, nt, H, W, C[+C])."""
    B, T, H, W, Cc = x.shape
    t0, t1 = t_range if t_range else (0, T)
    hw = H * W
    n_inner = (t1 - t0) * hw
    x0p = C.c_void_p(x.data_ptr() + t0 * hw * Cc * 2)
    if x2 is not None:
        T2, C2 = x2.shape[1], x2.shape[-1]
        u0, u1 = t2_range if t2_range else (0, T2)
        if u1 - u0 != t1 - t0:
            raise ValueError("chan_layernorm: frame ranges of the two sources differ")
        x1p = C.c_void_p(x2.data_ptr() + u0 * hw * C2 * 2)
        s1 = T2 * hw * C2
    else:
        x1p, s1, C2 = C.c_void_p(0), 0, 0
    rec.emit("extdm_chan_layernorm", (x0p, T * hw * Cc, Cc, x1p, s1, C2, _p(gamma), _p(y), B, n_inner,
                                      C.c_float(eps)), keep=(x, x2, gamma, y))


def temporal_prenorm(rec, x, gamma, ln_w, ln_b, u, xz, eps=1e-5):
    Cc = x.shape[-1]
    rows = x.numel() // Cc
    rec.emit("extdm_temporal_prenorm", (_p(x), _p(gamma), _p(ln_w), _p(ln_b), _p(u), _p(xz), rows, Cc,
                                        C.c_float(eps)), keep=(x, gamma, ln_w, ln_b, u, xz))


def adaptor_workspace(B, Cc, device):
    n = _lib.load().extdm_adaptor_workspace_floats(B, Cc)
    return torch.empty(n, dtype=torch.float32, device=device)


def adaptor_normalize(rec, x, n_frames, y, mean_std, ws, eps=1e-5):
    """x: (B, Ttot, H, W, C); stats over frames [0, n_frames); y: (B, n_frames, H, W, C); mean_std (2, B, C)."""
    B, Tt, H, W, Cc = x.shape
    rec.emit("extdm_adaptor_normalize", (_p(x), Tt * H * W * Cc, _p(y), _p(mean_std), _p(ws), B, n_frames, H * W, Cc,
                                         C.c_float(eps)), keep=(x, y, mean_std, ws))


def space_to_depth(rec, x, z):
    B, T, H, W, Cc = x.shape
    rec.emit("extdm_space_to_depth", (_p(x), _p(z), B * T, H, W, Cc), keep=(x, z))


def im2col7_flow(rec, cond, x, a, t0, nt):
    B, _, tc, H, W = cond.shape
    tp = x.shape[2]
    rec.emit("extdm_im2col7_flow", (_p(cond), _p(x), _p(a), B, tc, tp, t0, nt, H, W), keep=(cond, x, a))


def im2col13x_flow(rec, x, out, t_off):
    """x (B, 3, tp, H, W) fp32 -> frames [t_off, t_off + tp) of out (B, T, H, W, 64) bf16: channel (dx + 6)*3 + c holds
    x[.., c, .., x + dx] (composite init_conv, csrc/unet_elementwise.cu)."""
    B, _, tp, H, W = x.shape
    rec.emit("extdm_im2col13x_flow", (_p(x), _p(out), B, tp, out.shape[1], t_off, H, W), keep=(x, out))


def init_corner_fix(rec, x, table, x0, t_off):
    """Corner add-back of the composite init_conv's ring correction: x (B, 3, tp, H, W) fp32, table (4, 9, 28, C) fp32,
    x0 (B, T, H, W, C) bf16 updated in place on frames [t_off, t_off + tp)."""
    B, _, tp, H, W = x.shape
    rec.emit("extdm_init_corner_fix", (_p(x), _p(table), _p(x0), B, tp, x0.shape[1], t_off, H, W, x0.shape[-1]),
             keep=(x, table, x0))


def upsample2_border(rec, fpad, top, bottom, left, right):
    """fpad (F.., h + 4, w + 4, C) with the interior written -> replicate-padded in place; border rows / columns of its x2
    bilinear up-sampling into top / bottom (F.., 2w + 6, C) and left / right (F.., 2h, C)."""
    hp, wp, Cc = fpad.shape[-3:]
    rec.emit("extdm_upsample2_border", (_p(fpad), _p(top), _p(bottom), _p(left), _p(right), fpad.numel() // (hp * wp * Cc),
                                        hp - 4, wp - 4, Cc), keep=(fpad, top, bottom, left, right))


def bilinear_resize_cl(rec, x, y):
    h, w, Cc = x.shape[-3:]
    H, W = y.shape[-3:-1]
    F = x.numel() // (h * w * Cc)
    rec.emit("extdm_bilinear_resize_cl", (_p(x), _p(y), F, h, w, H, W, Cc), keep=(x, y))


def time_mlp(rec, time, w1, b1, w2, b2, wss, bss, out, dim):
    scratch = torch.empty(time.shape[0], 4 * dim, dtype=torch.float32, device=out.device)
    rec.emit("extdm_time_mlp", (_p(time), _p(w1), _p(b1), _p(w2), _p(b2), _p(wss), _p(bss), _p(out), _p(scratch),
                                time.shape[0], dim, wss.shape[0]), keep=(time, w1, b1, w2, b2, wss, bss, out, scratch))


def head_project(rec, hf, ho, wf, bf, wo, bo, out, t0):
    B, T, H, W, Cc = hf.shape
    rec.emit("extdm_head_project", (_p(hf), _p(ho), _p(wf), _p(bf), _p(wo), _p(bo), _p(out), B, T, t0, H * W, Cc),
             keep=(hf, ho, wf, bf, wo, bo, out))


def head_project_gn(rec, h2f, rf, partf, gf, bf_, h2o, ro, parto, go, bo_, n_part, wf, bf, wo, bo, out, t0, eps=1e-5):
    B, T, H, W, Cc = h2f.shape
    rec.emit("extdm_head_project_gn", (_p(h2f), _p(rf), _p(partf), _p(gf), _p(bf_), _p(h2o), _p(ro), _p(parto), _p(go),
                                       _p(bo_), n_part, _p(wf), _p(bf), _p(wo), _p(bo), _p(out), B, T, t0, H * W, Cc,
                                       8, C.c_float(eps)),
             keep=(h2f, rf, partf, gf, bf_, h2o, ro, parto, go, bo_, wf, bf, wo, bo, out),
             meta=dict(bytes=8.0 * B * (T - t0) * H * W * Cc))


def window_attention(rec, qkv, out, bias_table, rcos, rsin, heads, dh, window, shift):
    B, T, H, W, _ = qkv.shape
    rec.emit("extdm_window_attention", (_p(qkv), _p(out), _p(bias_table), _p(rcos), _p(rsin), B, T, H, W, heads, dh,
                                        window[0], window[1], window[2], shift[0], shift[1], shift[2]),
             keep=(qkv, out, bias_table, rcos, rsin), meta=dict(bytes=8.0 * heads * dh * B * T * H * W,
                                                                tag=f"hid={heads * dh} {T}x{H}x{W}"))


def stw_fused_supported(C_, heads, dh, window):
    return bool(_lib.load().extdm_stw_fused_supported(C_, heads, dh, window[0], window[1], window[2]))


def stw_fused(rec, x, y, gamma, wqkv, wproj, proj_bias, bias_table, rcos, rsin, heads, dh, window, shift, eps=1e-5):
    B, T, H, W, Cc = x.shape
    rec.emit("extdm_stw_fused", (_p(x), _p(y), _p(gamma), _p(wqkv), _p(wproj), _p(proj_bias), _p(bias_table),
                                 _p(rcos), _p(rsin), B, T, H, W, Cc, heads, dh, window[0], window[1], window[2],
                                 shift[0], shift[1], shift[2], C.c_float(eps)),
             keep=(x, y, gamma, wqkv, wproj, proj_bias, bias_table, rcos, rsin),
             meta=dict(bytes=4.0 * x.numel(), tag=f"C={Cc} {T}x{H}x{W}"))


def stw_fused_pre_supported(C_, heads, dh, window):
    return bool(_lib.load().extdm_stw_fused_pre_supported(C_, heads, dh, window[0], window[1], window[2]))


def groupnorm_affine(rec, part, n_part, gamma, beta, ad, P, Cc, eps=1e-5):
    B = ad.shape[0]
    rec.emit("extdm_groupnorm_affine", (_p(part), n_part, _p(gamma), _p(beta), _p(ad), B, P, Cc, 8, C.c_float(eps)),
             keep=(part, gamma, beta, ad))


def stw_fused_pre(rec, h, res, ad, y, gamma, wqkv, wproj, proj_bias, bias_table, rcos, rsin, heads, dh, window, shift,
                  eps=1e-5):
    B, T, H, W, Cc = h.shape
    rec.emit("extdm_stw_fused_pre", (_p(h), _p(res), _p(ad), _p(y), _p(gamma), _p(wqkv), _p(wproj), _p(proj_bias),
                                     _p(bias_table), _p(rcos), _p(rsin), B, T, H, W, Cc, heads, dh, window[0],
                                     window[1], window[2], shift[0], shift[1], shift[2], C.c_float(eps)),
             keep=(h, res, ad, y, gamma, wqkv, wproj, proj_bias, bias_table, rcos, rsin),
             meta=dict(bytes=6.0 * h.numel(), tag=f"C={Cc} {T}x{H}x{W} +gn"))


def temporal_fused_supported(C_, heads, dh, T):
    return bool(_lib.load().extdm_temporal_fused_supported(C_, heads, dh, T))


def temporal_fused(rec, x, y, gamma, ln_w, ln_b, wqkv, wout, rel_bias, rcos, rsin, heads, dh, eps=1e-5):
    B, T, H, W, Cc = x.shape
    rec.emit("extdm_temporal_fused", (_p(x), _p(y), _p(gamma), _p(ln_w), _p(ln_b), _p(wqkv), _p(wout), _p(rel_bias),
                                      _p(rcos), _p(rsin), B, T, H * W, Cc, heads, dh, C.c_float(eps)),
             keep=(x, y, gamma, ln_w, ln_b, wqkv, wout, rel_bias, rcos, rsin),
             meta=dict(bytes=4.0 * x.numel(), tag=f"C={Cc} {T}x{H}x{W}"))


def temporal_attention(rec, qkv, out, rel_bias, rcos, rsin, heads, dh):
    B, T, H, W, _ = qkv.shape
    rec.emit("extdm_temporal_attention", (_p(qkv), _p(out), _p(rel_bias), _p(rcos), _p(rsin), B, T, H * W, heads, dh),
             keep=(qkv, out, rel_bias, rcos, rsin))


def cross_attention(rec, q, k, v, out, heads):
    """q (B, Lq, hid), k / v (B, Lk, hid) (row views allowed: last-dim stride 1), out (B, Lq, hid); dh = hid/heads."""
    B, Lq, hid = q.shape
    Lk = k.shape[1]
    rec.emit("extdm_cross_attention", (_p(q), _p(k), _p(v), _p(out), B, heads, hid // heads, Lq, Lk, q.stride(1),
                                       k.stride(1), out.stride(1)), keep=(q, k, v, out),
             meta=dict(flops=4.0 * B * Lq * Lk * hid, tag=f"Lq={Lq} Lk={Lk}"))


def maxpool2_frames_cl(rec, x, y, t_range):
    """MaxPool (1,2,2) of frames t_range of x (B, T, H, W, C) -> dense y (B, nt, H/2, W/2, C)."""
    B, T, H, W, Cc = x.shape
    t0, t1 = t_range
    xp = C.c_void_p(x.data_ptr() + t0 * H * W * Cc * 2)
    rec.emit("extdm_maxpool2_frames_cl", (xp, _p(y), B, t1 - t0, T * H * W * Cc, (t1 - t0) * (H // 2) * (W // 2) * Cc,
                                          H, W, Cc), keep=(x, y))


def bilinear_resize_frames_cl(rec, x, y, x_t_range, y_t0):
    """Resize frames x_t_range of x (B, Tx, h, w, C) into frames [y_t0, ...) of y (B, Ty, H, W, C)."""
    B, Tx, h, w, Cc = x.shape
    Ty, H, W = y.shape[1:4]
    t0, t1 = x_t_range
    xp = C.c_void_p(x.data_ptr() + t0 * h * w * Cc * 2)
    yp = C.c_void_p(y.data_ptr() + y_t0 * H * W * Cc * 2)
    rec.emit("extdm_bilinear_resize_frames_cl", (xp, yp, B, t1 - t0, Tx * h * w * Cc, Ty * H * W * Cc, h, w, H, W, Cc),
             keep=(x, y))


# ----------------------------------------------------------------------------- sampler
def ddim_threshold(rec, img, pred, c_recip, c_recipm1, q, s):
    B = img.shape[0]
    rec.emit("extdm_ddim_threshold", (_p(img), _p(pred), C.c_float(c_recip), C.c_float(c_recipm1), C.c_float(q),
                                      _p(s), B, img.numel() // B), keep=(img, pred, s))


def ddim_update(rec, img, pred, noise, s, c_recip, c_recipm1, sqrt_alpha_next, c, sigma, img_out, x_start_out=None):
    B = img.shape[0]
    rec.emit("extdm_ddim_update", (_p(img), _p(pred), _p(noise), _p(s), C.c_float(c_recip), C.c_float(c_recipm1),
                                   C.c_float(sqrt_alpha_next), C.c_float(c), C.c_float(sigma), _p(img_out),
                                   _p(x_start_out), B, img.numel() // B),
             keep=(img, pred, noise, s, img_out, x_start_out))


def ddim_update_seeded(rec, img, pred, seeds, step, s, c_recip, c_recipm1, sqrt_alpha_next, c, sigma, img_out,
                       x_start_out=None):
    """ddim_update with sigma * z, z the Philox draw of (seeds[b], step) (the generator of ddpm_update)."""
    if seeds is None:
        raise ValueError("ddim_update_seeded: seeds are required")
    _chk(seeds, torch.int64, "seeds")
    B = img.shape[0]
    if seeds.numel() != B or seeds.device != img.device:
        raise ValueError(f"ddim_update_seeded: seeds must be {B} int64 on {img.device}, got {seeds.numel()} on "
                         f"{seeds.device}")
    if (img.numel() // B) % 4:
        raise ValueError("ddim_update_seeded: elements per sample must be a multiple of 4")
    rec.emit("extdm_ddim_update_seeded", (_p(img), _p(pred), _p(seeds), int(step), _p(s), C.c_float(c_recip),
                                          C.c_float(c_recipm1), C.c_float(sqrt_alpha_next), C.c_float(c),
                                          C.c_float(sigma), _p(img_out), _p(x_start_out), B, img.numel() // B),
             keep=(img, pred, seeds, s, img_out, x_start_out))


def ddpm_threshold(rec, img, pred, rows, step, q, s):
    """As ddim_threshold, with (c_recip, c_recipm1) read from rows[step] on the device."""
    _chk(rows, torch.float32, "rows")
    _chk(step, torch.int32, "step")
    B = img.shape[0]
    rec.emit("extdm_ddpm_threshold", (_p(img), _p(pred), _p(rows), _p(step), C.c_float(q), _p(s), B, img.numel() // B),
             keep=(img, pred, rows, step, s))


def ddpm_update(rec, img, pred, rows, step, seeds, noise, s, img_out, x_start_out=None):
    """One ancestral step with the coefficients of rows[step]; noise (n_steps, *img.shape) or None (Philox of seeds)."""
    _chk(rows, torch.float32, "rows")
    _chk(step, torch.int32, "step")
    _chk(seeds, torch.int64, "seeds")
    _chk(noise, torch.float32, "noise")
    B = img.shape[0]
    rec.emit("extdm_ddpm_update", (_p(img), _p(pred), _p(rows), _p(step), _p(seeds), _p(noise), _p(s), _p(img_out),
                                   _p(x_start_out), B, img.numel() // B),
             keep=(img, pred, rows, step, seeds, noise, s, img_out, x_start_out))


def ddpm_fill_normal(rec, seeds, out):
    """out[b] = the x_T draw of video seed seeds[b]."""
    _chk(seeds, torch.int64, "seeds")
    _chk(out, torch.float32, "out")
    B = out.shape[0]
    rec.emit("extdm_ddpm_fill_normal", (_p(seeds), _p(out), B, out.numel() // B), keep=(seeds, out))


def ddpm_broadcast_row(rec, table, step, out):
    """out[b] = table[step] for every row b of out."""
    _chk(table, torch.float32, "table")
    _chk(step, torch.int32, "step")
    _chk(out, torch.float32, "out")
    if table.shape[-1] != out.shape[-1]:
        raise ValueError(f"ddpm_broadcast_row: rows of {table.shape[-1]} and {out.shape[-1]} floats")
    rec.emit("extdm_ddpm_broadcast_row", (_p(table), _p(step), _p(out), out.shape[0], out.shape[-1]),
             keep=(table, step, out))


def ddpm_advance(rec, step, times, time):
    """step += 1; time[:] = times[step] (while step < len(times))."""
    _chk(step, torch.int32, "step")
    _chk(times, torch.int64, "times")
    _chk(time, torch.int64, "time")
    rec.emit("extdm_ddpm_advance", (_p(step), _p(times), times.numel(), _p(time), time.numel()),
             keep=(step, times, time))


# ----------------------------------------------------------------------------- LFAE decode
def warp_blend_cl(rec, skip, prev, flow, occ, out, up2=False):
    """skip (Fs,H,W,C) bf16, prev (F,H,W,C) or None, flow (F,h,w,2) fp32, occ (F,1,h,w) fp32 or None."""
    Fs, H, W, Cc = skip.shape
    F, h, w = flow.shape[:3]
    rec.emit("extdm_warp_blend_cl", (_p(skip), _p(prev), _p(flow), _p(occ), _p(out), F, Fs, H, W, Cc, h, w, int(up2)),
             keep=(skip, prev, flow, occ, out))


def warp_image(rec, src, dec, flow, occ, prediction, deformed):
    Fs, _, H, W = src.shape
    F, h, w = flow.shape[:3]
    dstride = 0 if dec is None else dec.shape[-1]
    rec.emit("extdm_warp_image", (_p(src), _p(dec), dstride, _p(flow), _p(occ), _p(prediction), _p(deformed), F, Fs,
                                  H, W, h, w), keep=(src, dec, flow, occ, prediction, deformed))


def warp_taps(rec, flow, occ, H, W):
    """Index math of the warp kernels as tensors: (xy int32 (F,H,W,2), weights (F,H,W,4), gflow (F,H,W,3))."""
    F, h, w = flow.shape[:3]
    xy = torch.empty(F, H, W, 2, dtype=torch.int32, device=flow.device)
    wts = torch.empty(F, H, W, 4, dtype=torch.float32, device=flow.device)
    gf = torch.empty(F, H, W, 3, dtype=torch.float32, device=flow.device)
    rec.emit("extdm_warp_taps", (_p(flow), _p(occ), _p(xy), _p(wts), _p(gf), F, H, W, h, w),
             keep=(flow, occ, xy, wts, gf))
    return xy, wts, gf


def bn_relu_cl(rec, x, scale, shift, y):
    Cc = x.shape[-1]
    rec.emit("extdm_bn_relu_cl", (_p(x), _p(scale), _p(shift), _p(y), x.numel() // Cc, Cc), keep=(x, scale, shift, y))


def avgpool2_cl(rec, x, y):
    F, H, W, Cc = x.shape
    rec.emit("extdm_avgpool2_cl", (_p(x), _p(y), F, H, W, Cc), keep=(x, y))


def im2col7_image(rec, img, a):
    F, _, H, W = img.shape
    rec.emit("extdm_im2col7_image", (_p(img), _p(a), F, H, W), keep=(img, a))


def ncthw_to_cl(rec, x, y):
    B, Cc = x.shape[:2]
    rest = x.numel() // (B * Cc)
    rec.emit("extdm_ncthw_to_cl", (_p(x), _p(y), B, Cc, rest, 1), keep=(x, y))


def cl_to_ncthw(rec, x, y):
    B, Cc = y.shape[:2]
    rest = y.numel() // (B * Cc)
    rec.emit("extdm_cl_to_ncthw", (_p(x), _p(y), B, Cc, rest, 1), keep=(x, y))


# ----------------------------------------------------------------------------- LFAE conditioning stage (fp32)
def image_to_cl(rec, a, a_div, out, *, b=None, b_div=1, kern=None, stride=1):
    """NCHW fp32 image(s) -> (F, H/stride, W/stride, cpad) fp32 channels-last, optionally through the anti-alias filter."""
    F_, h, w, cpad = out.shape
    H, W = a.shape[2], a.shape[3]
    ks = 1 if kern is None else kern.shape[-1]
    rec.emit("extdm_image_to_cl", (_p(a), a.shape[1], a_div, _p(b) if b is not None else None,
                                   0 if b is None else b.shape[1], b_div, _p(kern) if kern is not None else None, ks,
                                   stride, _p(out), F_, H, W, cpad), keep=(a, b, kern, out), meta=dict(tag=f"{H}->{h}"))


def avgpool2_f32_cl(rec, x, y):
    F_, H, W, Cc = x.shape
    rec.emit("extdm_avgpool2_f32_cl", (_p(x), _p(y), F_, H, W, Cc), keep=(x, y),
             meta=dict(bytes=5.0 * y.numel() * 4))


def upsample2_f32_cl(rec, x, y):
    F_, H, W, Cc = x.shape
    rec.emit("extdm_upsample2_f32_cl", (_p(x), _p(y), F_, H, W, Cc), keep=(x, y),
             meta=dict(bytes=1.25 * y.numel() * 4))


def region_moments(rec, logits, K, crop, temperature, shift, covar):
    F_, h, w, ldc = logits.shape
    rec.emit("extdm_region_moments", (_p(logits), ldc, F_, K, h, w, crop, C.c_float(temperature), _p(shift), _p(covar)),
             keep=(logits, shift, covar))


def pca_affine(rec, covar, affine):
    """(n, 2, 2) covariances -> u diag(sqrt s) with cuSOLVER's (= torch.svd on CUDA) singular-vector signs."""
    rec.emit("extdm_pca_affine", (_p(covar), _p(affine), covar.numel() // 4), keep=(covar, affine))


def sparse_motion(rec, src, shift, covar, affine, bg, tc, revert_axis_swap, use_covar, region_var, inp, motion):
    F_, h, w, cpad = inp.shape
    K = shift.shape[1]
    rec.emit("extdm_sparse_motion", (_p(src), src.shape[-1], _p(shift), _p(covar), _p(affine),
                                     _p(bg) if bg is not None else None, F_, K, tc, h, w, int(revert_axis_swap),
                                     int(use_covar), C.c_float(region_var), _p(inp), cpad, _p(motion)),
             keep=(src, shift, covar, affine, bg, inp, motion))


def sparse_motion_src(rec, src, shift, covar, affine, bg, group, src_slot, revert_axis_swap, use_covar, region_var, inp,
                      motion):
    """sparse_motion with the source of frame f at slot src_slot of its group of `group` frames (one video each)."""
    F_, h, w, cpad = inp.shape
    K = shift.shape[1]
    rec.emit("extdm_sparse_motion_src", (_p(src), src.shape[-1], _p(shift), _p(covar), _p(affine),
                                         _p(bg) if bg is not None else None, F_, K, group, src_slot, h, w,
                                         int(revert_axis_swap), int(use_covar), C.c_float(region_var), _p(inp), cpad,
                                         _p(motion)),
             keep=(src, shift, covar, affine, bg, inp, motion))


def flow_compose(rec, head, motion, K, tc, grid, conf):
    F_, h, w, ldc = head.shape
    rec.emit("extdm_flow_compose", (_p(head), ldc, _p(motion), F_, K, tc, h, w, _p(grid),
                                    _p(conf) if conf is not None else None), keep=(head, motion, grid, conf))


def bg_head(rec, feat, fcw, fcb, bg_type, out):
    F_, hh, ww, Cc = feat.shape
    rec.emit("extdm_bg_head", (_p(feat), F_, hh * ww, Cc, _p(fcw), _p(fcb), fcw.shape[0], bg_type, _p(out)),
             keep=(feat, fcw, fcb, out))
