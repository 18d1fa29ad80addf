"""Host-side "programs" for the row-slab convolution kernel (csrc/conv_slab.cu): which input-row slabs
a tile needs, which taps reuse each slab, and how the master weights are laid out as [ncols x 64]
tiles.  Three users (all stride-1, same-size, bf16):
  * the fused MultiScaleBlock branches (enhanced_generator.py:52-71): 1x1 + 3x3 dil 1/2/4 in ONE launch
    writing the concatenated [N,H,W,C] tensor (+ the shared InstanceNorm statistics);
  * the 7x7 output conv + tanh (:137-138), N = 3 padded to 16;
  * the 7x7 input conv (:92) on the 3-channel image padded to 8 channels ("pixel-pair K").
"""
import ctypes

import torch

from . import _lib, ops
from ._lib import SHIFT_MAX_KBLOCKS, SLAB_MAX_KBLOCKS, SLAB_MAX_TAPS, ShiftDesc, SlabDesc


class SlabProgram:
    def __init__(self, Cin, Ntot, n_store, ncols, halo, pixel_pair, kblocks):
        """kblocks: list of (dy, cb, [(sx, acc_col, kstep, weight_key), ...])"""
        self.Cin, self.Ntot, self.n_store, self.ncols, self.halo, self.pixel_pair = Cin, Ntot, n_store, ncols, halo, pixel_pair
        self.kblocks = kblocks
        taps = [t for _, _, ts in kblocks for t in ts]
        if len(kblocks) > SLAB_MAX_KBLOCKS or len(taps) > SLAB_MAX_TAPS:
            raise ValueError("slab program too large")
        self.n_taps = len(taps)

    def fill(self, d):
        d.Cin, d.Ntot, d.n_store, d.ncols, d.halo, d.pixel_pair_k = (self.Cin, self.Ntot, self.n_store, self.ncols,
                                                                      self.halo, int(self.pixel_pair))
        d.n_kblocks, d.n_taps = len(self.kblocks), self.n_taps
        d.n_chains = 1   # measured on B200: independent accumulation chains do not speed up small-N MMAs
        seen, tp = set(), 0
        for kb, (dy, cb, taps) in enumerate(self.kblocks):
            d.kb_dy[kb], d.kb_cb[kb], d.kb_tap_begin[kb] = dy, cb, tp
            for sx, acc_col, kstep, _ in taps:
                d.tap_sx[tp], d.tap_acc_col[tp], d.tap_kstep[tp] = sx, acc_col, kstep
                d.tap_first[tp] = int(acc_col not in seen)
                seen.add(acc_col)
                tp += 1
        d.kb_tap_begin[len(self.kblocks)] = tp


def msb_max_taps(C):
    """Taps per k-block: at most 64 KB of weight tiles per k-block (C = 64: no split, the weights stay resident; C = 128:
    no split; C = 256: the 10-tap centre row is 8 + 2).  A finer split for C = 128 (4 + 4 + 2: twice the pipeline stages,
    two more slab loads per tile) measured slower on B200 (0.585 -> 0.626 ms per 16 images): the kernel is bound by
    L2 -> SM bytes, not by TMA latency.  csrc/conv_slab.cu: msb_maxt mirrors this for the straight-line issue code."""
    return max(1, (64 * 1024) // ((C // 4) * 128))


def msb_program(C, max_taps=None):
    """All four MultiScaleBlock branches; branch b writes accumulator columns [(b-1)C/4, bC/4)."""
    q = C // 4
    branches = [(1, 1), (3, 1), (3, 2), (3, 4)]   # (k, dilation) of branch1..4
    kblocks = []
    if max_taps is None:
        max_taps = msb_max_taps(C)
    # The centre row comes FIRST and its four un-shifted taps (the 1x1 branch and the centres of the three 3x3 branches) lead:
    # they read the same slab view and write the four adjacent accumulator slices, so the specialised kernels issue them as ONE
    # N = C MMA (csrc/conv_slab.cu: 28 -> 25 MMAs per K step) -- and as the first touch of every slice it needs no zeroing.
    for dy in (0, -4, -2, -1, 1, 2, 4):
        for cb in range(C // 64):
            taps = []
            for b, (k, dil) in enumerate(branches):
                for kh in range(k):
                    if (kh - k // 2) * dil != dy:
                        continue
                    for kw in range(k):
                        taps.append(((kw - k // 2) * dil, b * q, 0, (b, kh, kw, cb)))
            if dy == 0:
                taps = [t for t in taps if t[0] == 0] + [t for t in taps if t[0] != 0]
            for i in range(0, len(taps), max_taps):          # a long tap list re-loads the slab (rare: C=256 centre row)
                kblocks.append((dy, cb, taps[i:i + max_taps]))
    return SlabProgram(C, C, C, q, 4, False, kblocks)


def msb_weight_slab(prog, weights, dtype=torch.bfloat16):
    """weights: [w_branch1 [q,C,1,1], w_branch2..4 [q,C,3,3]] fp32 -> bf16 [n_taps*q, 64]."""
    rows = []
    for _, _, taps in prog.kblocks:
        for _, _, _, (b, kh, kw, cb) in taps:
            rows.append(weights[b][:, cb * 64:(cb + 1) * 64, kh, kw])
    return torch.cat(rows, 0).to(dtype).contiguous()


def msb_dgrad_program(C):
    """Data gradient of the four fused branches in ONE launch: the input is the concatenated branch gradient
    dB [N,H,W,C] (branch b = channels [bq, (b+1)q)), the output d(a1) [N,H,W,C] = sum over branches and taps of
    dB_b[y - dy][x - sx] W_b[:, :, kh, kw]^T.  Every tap is an N = C MMA group on the 64-channel block that holds
    the branch's slice (weight columns of other branches in that block are zero), instead of four small-Cin
    convs on the gather kernel with an accumulate pass each."""
    q = C // 4
    branches = [(1, 1), (3, 1), (3, 2), (3, 4)]
    max_taps = max(1, (64 * 1024) // (C * 128))
    kblocks = []
    for dy in (-4, -2, -1, 0, 1, 2, 4):
        for cb in range(C // 64):
            taps = []
            for b, (k, dil) in enumerate(branches):
                if (b * q) // 64 != cb:
                    continue
                for kh in range(k):
                    if -(kh - k // 2) * dil != dy:
                        continue
                    for kw in range(k):
                        taps.append((-(kw - k // 2) * dil, 0, 0, (b, kh, kw, cb)))
            for i in range(0, len(taps), max_taps):
                kblocks.append((dy, cb, taps[i:i + max_taps]))
    return SlabProgram(C, C, C, C, 4, False, kblocks)


def msb_dgrad_weight_slab(prog, weights, dtype=torch.bfloat16):
    """weights: [w_branch1 [q,C,1,1], w_branch2..4 [q,C,3,3]] fp32 -> bf16 [n_taps*C, 64]: tile row = input channel ci
    of the forward conv (= output channel of the dgrad), column kk = channel cb*64 + kk of dB."""
    C = prog.Cin
    q = C // 4
    rows = []
    for _, _, taps in prog.kblocks:
        for _, _, _, (b, kh, kw, cb) in taps:
            t = torch.zeros(C, 64, device=weights[b].device, dtype=torch.float32)
            k0 = b * q - cb * 64                           # first column of branch b inside this 64-channel block
            t[:, k0:k0 + min(q, 64)] = weights[b][:, :, kh, kw].t()[:, :min(q, 64)]
            rows.append(t)
    return torch.cat(rows, 0).to(dtype).contiguous()


def convT_phase_programs(Cin, Cout):
    """4x4 stride-2 pad-1 transposed conv (enhanced_generator.py:120-121, 127-128) = four sub-pixel phases, each a 2x2
    conv of the input plane (ops.ConvGeom.forward: phase (ph, pw) has padding (1-ph, 1-pw) and writes output pixels
    (2y+ph, 2x+pw)).  As a row-slab program a phase reads each input row slab ONCE for both horizontal taps: half the
    L2 -> SM bytes of the per-tap implicit GEMM, which is what bounds these layers.  Returns [(ph, pw, program)]."""
    progs = []
    for ph in range(2):
        for pw in range(2):
            kblocks = []
            for th in range(2):
                for cb in range(Cin // 64):
                    kblocks.append((th - (1 - ph), cb, [(tw - (1 - pw), 0, 0, (th, tw, cb)) for tw in range(2)]))
            progs.append((ph, pw, SlabProgram(Cin, Cout, Cout, Cout, 1, False, kblocks)))
    return progs


def convT_phase_weight_slabs(progs, wp, Cin, Cout):
    """wp: the packed phase weights of ops.ConvGeom('convT').pack_fwd, bf16 [4][Cout][2][2][Cin] flat ->
    one [n_taps*Cout, 64] slab per phase in program order."""
    w = wp.reshape(4, Cout, 2, 2, Cin)
    out = []
    for ph, pw, prog in progs:
        rows = [w[ph * 2 + pw, :, th, tw, cb * 64:(cb + 1) * 64] for _, _, taps in prog.kblocks for _, _, _, (th, tw, cb) in taps]
        out.append(torch.cat(rows, 0).contiguous())
    return out


def convT_slab(progs, x, w_slabs, bias, out, stats=None):
    """x [N,H,W,Cin] bf16 -> out [N,2H,2W,Cout] bf16 (all four phases; statistics accumulated over the four launches)."""
    ops._dev(x)
    N, H, W, Ci_total = x.shape
    for (ph, pw, prog), wsl in zip(progs, w_slabs):
        d = SlabDesc()
        d.dtype, d.N, d.H, d.W, d.Ci_total, d.ci_off = _lib.BF16, N, H, W, Ci_total, 0
        prog.fill(d)
        d.Co_total, d.co_off, d.act = out.shape[3], 0, ops.ACT_NONE
        d.out_stride, d.out_off_h, d.out_off_w = 2, ph, pw
        d.flags = _lib.CONV_STATS if stats is not None else 0
        _lib.call("msg_conv_slab", ctypes.byref(d), ops._p(x), ops._p(wsl), ops._p(bias), ops._p(out), ops._p(stats),
                  ops._stream())
    return out


def conv7_out_program(c):
    kblocks = []
    for kh in range(7):
        for cb in range(c // 64):
            kblocks.append((kh - 3, cb, [(kw - 3, 0, 0, (kh, kw, cb)) for kw in range(7)]))
    return SlabProgram(c, 16, 3, 16, 3, False, kblocks)


def conv7_out_weight_slab(prog, w, dtype=torch.bfloat16):
    """w: [3, c, 7, 7] fp32 -> bf16 [n_taps*16, 64] (filters 3..15 zero)."""
    rows = []
    for _, _, taps in prog.kblocks:
        for _, _, _, (kh, kw, cb) in taps:
            t = torch.zeros(16, 64, device=w.device, dtype=torch.float32)
            t[:3] = w[:, cb * 64:(cb + 1) * 64, kh, kw]
            rows.append(t)
    return torch.cat(rows, 0).to(dtype).contiguous()


def conv7_in_program(c):
    """7x7 conv on the image padded to 8 channels: one MMA (K=16) covers taps kw = 2j, 2j+1."""
    kblocks = [(kh - 3, 0, [(2 * j - 3, 0, j, (kh, j)) for j in range(4)]) for kh in range(7)]
    return SlabProgram(8, c, c, c, 3, True, kblocks)


def conv7_in_weight_slab(prog, w, dtype=torch.bfloat16):
    """w: [c, 3, 7, 7] fp32 -> bf16 [7*c, 64]; row (kh, co), k = j*16 + p*8 + ch  <->  w[co, ch, kh, 2j+p]."""
    c = w.shape[0]
    t = torch.zeros(7, c, 4, 2, 8, device=w.device, dtype=torch.float32)
    wp = torch.zeros(c, 8, 7, 8, device=w.device, dtype=torch.float32)
    wp[:, :3, :, :7] = w
    # wp[co, ch, kh, kw] -> t[kh, co, j, p, ch] with kw = 2j + p
    t.copy_(wp.reshape(c, 8, 7, 4, 2).permute(2, 0, 3, 4, 1))
    return t.reshape(7 * c, 64).to(dtype).contiguous()


def conv_slab(prog, x, w_slab, bias, out=None, co_off=0, stats=None, act=ops.ACT_NONE, nchw_out=None, ci_off=0):
    """x: [N,H,W,Ci_total] bf16.  Writes columns [co_off, co_off+n_store) of `out` [N,H,W,Co_total] bf16, or the
    fp32 NCHW tensor `nchw_out` [N,n_store,H,W]."""
    ops._dev(x)
    N, H, W, Ci_total = x.shape
    d = SlabDesc()
    d.dtype, d.N, d.H, d.W, d.Ci_total, d.ci_off = _lib.BF16, N, H, W, Ci_total, ci_off
    prog.fill(d)
    flags = 0
    if stats is not None:
        flags |= _lib.CONV_STATS
    if nchw_out is not None:
        flags |= _lib.CONV_OUT_NCHW_F32
        y, d.Co_total = nchw_out, prog.n_store
    else:
        if out is None:
            out = torch.empty((N, H, W, prog.n_store), device=x.device, dtype=x.dtype)
        y, d.Co_total = out, out.shape[3]
    d.co_off, d.act, d.flags = co_off, act, flags
    _lib.call("msg_conv_slab", ctypes.byref(d), ops._p(x), ops._p(w_slab), ops._p(bias), ops._p(y), ops._p(stats),
              ops._stream())
    return nchw_out if nchw_out is not None else out


# --------------------------------------------------------------------------------------------------
# "taps-as-N" programs (csrc/conv_shift.cu)
# --------------------------------------------------------------------------------------------------
class ShiftProgram:
    def __init__(self, Cin, Ntot, n_out, halo, kblocks, groups, tile_rows=1):
        """kblocks: [(dy, cb, col0, ncols, wrow)] or [(dy, cb, col0, ncols, wrow, first, same_slab)]: without explicit
        flags the first k-block must cover every accumulator column (it overwrites, the others accumulate);
        same_slab: re-use the slab of the previous k-block.
        groups: [(col0, span, out_col0, out_cols, [(shift, col), ...])] or [..., row] (output row inside a multi-row tile)"""
        self.Cin, self.Ntot, self.n_out, self.halo, self.kblocks, self.groups = Cin, Ntot, n_out, halo, kblocks, groups
        self.tile_rows = tile_rows
        if len(kblocks[0]) == 5:
            assert kblocks[0][2] == 0 and kblocks[0][3] == Ntot

    def fill(self, d):
        d.Cin, d.Ntot, d.n_out, d.halo = self.Cin, self.Ntot, self.n_out, self.halo
        d.n_kblocks, d.n_groups = len(self.kblocks), len(self.groups)
        d.tile_rows = self.tile_rows
        for i, kb in enumerate(self.kblocks):
            dy, cb, col0, ncols, wrow = kb[:5]
            first, same = (kb[5], kb[6]) if len(kb) == 7 else (int(i == 0), 0)
            d.kb_dy[i], d.kb_cb[i], d.kb_col0[i], d.kb_ncols[i], d.kb_wrow[i], d.kb_first[i] = dy, cb, col0, ncols, wrow, first
            d.kb_same_slab[i] = same
        t = 0
        for g, grp in enumerate(self.groups):
            col0, span, oc0, oc, terms = grp[:5]
            d.grp_row[g] = grp[5] if len(grp) == 6 else 0
            d.grp_col0[g], d.grp_span[g], d.grp_out_col0[g], d.grp_out_cols[g], d.grp_term_begin[g] = col0, span, oc0, oc, t
            for shift, col in terms:
                d.term_shift[t], d.term_col[t] = shift, col
                t += 1
        d.grp_term_begin[len(self.groups)] = t
        d.n_terms = t


def conv7_out_shift_program(c, tile_rows=2):
    """7x7 c->3 conv: per filter row ONE N=32 MMA (7 taps x 4 padded filters); 28*c/64 MMAs per output row.
    tile_rows = R: a tile is R output rows; input row y+dy (dy = -3..R+2) is loaded ONCE and feeds filter row dy+3-r of output
    row y+r (accumulator columns [32r, 32r+32)) for every r it reaches: R+6 slabs per R rows instead of 7R -- the kernel is
    bound by L2 -> SM slab bytes (ncu: ~24 B/clk/SM of TMA traffic, tensor pipe 16 %).  R = 2: 8 slabs per 2 rows (0.40 ms per
    16 images at 512^2 with two epilogue groups); R = 4: 10 slabs per 4 rows, but its 68 KB exchange tile leaves room for one
    epilogue group only and measures SLOWER (0.43 ms): the shifted-sum epilogue, not the slab traffic, sets the pace."""
    CB = c // 64
    terms = [(kw, kw * 4) for kw in range(7)]
    R = tile_rows
    while R > 1 and 7 * R * CB > SHIFT_MAX_KBLOCKS:
        R //= 2
    if R == 1:
        kblocks = [(kh - 3, cb, 0, 32, (kh * CB + cb) * 32) for kh in range(7) for cb in range(CB)]
        return ShiftProgram(c, 32, 3, 3, kblocks, [(0, 28, 0, 3, terms)])
    kblocks, seen = [], set()
    for dy in range(-3, R + 3):
        for cb in range(CB):
            same = 0
            for r in range(R):
                kh = dy + 3 - r
                if 0 <= kh <= 6:
                    kblocks.append((dy, cb, 32 * r, 32, (kh * CB + cb) * 32, int(r not in seen), same))
                    seen.add(r)
                    same = 1
    groups = [(32 * r, 28, 0, 3, terms, r) for r in range(R)]
    return ShiftProgram(c, 32 * R, 3, 3, kblocks, groups, tile_rows=R)


def conv7_out_shift_weights(prog, w, dtype=torch.bfloat16):
    """w [3, c, 7, 7] fp32 -> [7*CB*32, 64]: row (kh, cb, kw*4 + co) = w[co, cb*64:(cb+1)*64, kh, kw]."""
    c = w.shape[1]
    CB = c // 64
    t = torch.zeros(7, CB, 8, 4, 64, device=w.device, dtype=torch.float32)
    # w[co, cb*64+k, kh, kw] -> t[kh, cb, kw, co, k]
    t[:, :, :7, :3] = w.reshape(3, CB, 64, 7, 7).permute(3, 1, 4, 0, 2)
    return t.reshape(7 * CB * 32, 64).to(dtype).contiguous()


def msb64_shift_program():
    """MultiScaleBlock branches at C=64 (q=16): accumulator columns = b1 [0,16) | b2 sx=-1,0,1 [16,64) |
    b3 sx=-2,0,2 [64,112) | b4 sx=-4,0,4 [112,160).  Centre row first (N=160), then the six other rows (N=48)."""
    kblocks = [(0, 0, 0, 160, 0)]
    wrow = 160
    for b, dil in ((1, 1), (2, 2), (3, 4)):
        for kh in (0, 2):
            kblocks.append(((kh - 1) * dil, 0, 16 + 48 * (b - 1), 48, wrow))
            wrow += 48
    groups = [(0, 16, 0, 16, [(4, 0)])]
    for b, dil in ((1, 1), (2, 2), (3, 4)):
        groups.append((16 + 48 * (b - 1), 48, 16 * b, 16, [(4 - dil, 0), (4, 16), (4 + dil, 32)]))
    return ShiftProgram(64, 160, 64, 4, kblocks, groups)


def msb64_shift_weights(weights, dtype=torch.bfloat16):
    """weights: [w1 [16,64,1,1], w2..w4 [16,64,3,3]] fp32 -> [448, 64] in the program's row order."""
    rows = [weights[0][:, :, 0, 0]]
    for b in (1, 2, 3):
        rows += [weights[b][:, :, 1, kw] for kw in range(3)]          # centre filter row
    for b in (1, 2, 3):
        for kh in (0, 2):
            rows += [weights[b][:, :, kh, kw] for kw in range(3)]
    return torch.cat(rows, 0).to(dtype).contiguous()


def conv_shift(prog, x, w_rows, bias, out=None, co_off=0, stats=None, act=ops.ACT_NONE, nchw_out=None, ci_off=0):
    ops._dev(x)
    N, H, W, Ci_total = x.shape
    d = ShiftDesc()
    d.dtype, d.N, d.H, d.W, d.Ci_total, d.ci_off = _lib.BF16, N, H, W, Ci_total, ci_off
    prog.fill(d)
    flags = 0
    if stats is not None:
        flags |= _lib.CONV_STATS
    if nchw_out is not None:
        flags |= _lib.CONV_OUT_NCHW_F32
        y, d.Co_total = nchw_out, prog.n_out
    else:
        if out is None:
            out = torch.empty((N, H, W, prog.n_out), device=x.device, dtype=x.dtype)
        y, d.Co_total = out, out.shape[3]
    d.co_off, d.act, d.flags = co_off, act, flags
    _lib.call("msg_conv_shift", ctypes.byref(d), ops._p(x), ops._p(w_rows), ops._p(bias), ops._p(y), ops._p(stats),
              ops._stream())
    return nchw_out if nchw_out is not None else out


# ---------------------------------------------------------------------------------------------------------------------
# MultiScaleBlock branches at C = 64 as a ROW RING (csrc/msb_ring.cu)
#
# The per-tap slab kernel issues 25 MMAs of N = 16 per K step and output row, each ~40 cycles whatever N (the A operand
# read from shared memory bounds a small-N tcgen05.mma): shared-memory bound at 15-25 % of the tensor pipe, and it loads
# 7 input row slabs per output row.  Here a CTA walks DOWN a 128-pixel column strip: every input row is loaded ONCE, and
# for a horizontal shift sx the three vertical taps of a dilated 3x3 branch -- which send input row r to output rows
# r - d, r, r + d -- are ONE MMA of N = 48, because the accumulators of those three output rows sit in adjacent tensor
# memory columns: each branch keeps a ring of row accumulators per residue class (row mod d).  10 MMAs per K step and
# row instead of 25.  Finished rows are drained and their slots zeroed by the epilogue warps, so every MMA accumulates.
# The functions below ARE the schedule (the CUDA kernel restates them; tests/test_msb_ring_cpu.py runs them on tensors).
# ---------------------------------------------------------------------------------------------------------------------
RING_DIL = (0, 1, 2, 4)            # branch 1 (1x1) has no vertical extent
# Ring length per residue class of each branch, per PASS (= kernel launch).  C = 64: all four branches share the 512 tensor-memory
# columns (16 per row accumulator: 3*16 | 5*16 | 2*4*16 | 4*4*16 = 512).  C = 128 (32 columns per row accumulator) does not fit in
# one pass: branches 1 + 2 (4*32 + 2 sets of 6*32 = 512 columns), branch 3 (2*8*32 = 512) and branch 4 (4*4*32 = 512) run as
# three launches, each with its own resident weight stacks.
RING_PASSES = {64: (((0, 3), (1, 5), (2, 4), (3, 4)),),
               128: (((0, 4), (1, 6)), ((2, 8),), ((3, 4),))}
# How many steps (input rows) the MMA issuers may run ahead of the epilogue: the slot of the row a 3x3 branch finishes at step k is
# touched again at step k + (R - 2) d (the 1x1 branch: k + R), so the lead is at most the minimum of that over the pass.
RING_LEAD = {64: (3,), 128: (4, 8, 8)}


def ring_dup(C, ps, b):
    """accumulator sets of branch b in pass ps: the dilation-1 3x3 at C = 128 keeps one ring for even and one for odd INPUT rows (two
    issuers share the branch without touching the same columns; the epilogue adds the sets).  The second set follows the first."""
    return 2 if (C == 128 and ps == 0 and b == 1) else 1


def ring_layout(C, ps=0):
    """{branch: (ring length per residue class, first TMEM column)} of pass ps"""
    Q, col, out = C // 4, 0, {}
    for b, R in RING_PASSES[C][ps]:
        out[b] = (R, col)
        col += max(1, RING_DIL[b]) * R * Q * ring_dup(C, ps, b)
    assert col <= 512
    return out


def ring_col(b, y, C=64, ps=0):
    """TMEM column of the C/4-column accumulator of output row y of branch b."""
    d = max(1, RING_DIL[b])
    R, base = ring_layout(C, ps)[b]
    return base + ((y % d) * R + (y // d) % R) * (C // 4)


def ring_row_mmas(r, y0, y1, C=64, ps=0):
    """MMAs of input row r for a strip segment of output rows [y0, y1) in pass ps: a list of (branch, sx, first_entry, n_entries,
    col) -- the MMA multiplies the slab view shifted by sx with rows [Q * first_entry, Q * (first_entry + n_entries)) of the
    branch's weight stack for that sx (entries ordered by output row: r - d (ky = 2), r (ky = 1), r + d (ky = 0)) and accumulates
    into n_entries * Q columns starting at col (Q = C / 4).  Entries are merged while their ring slots are adjacent."""
    Q, out = C // 4, []
    lay = ring_layout(C, ps)
    if 0 in lay and y0 <= r < y1:
        out.append((0, 0, 0, 1, ring_col(0, r, C, ps)))
    for b in (1, 2, 3):
        if b not in lay:
            continue
        d = RING_DIL[b]
        rows = [r - d, r, r + d]
        run = []                                    # (entry, column)
        runs = []
        for e, y in enumerate(rows):
            if not (y0 <= y < y1):
                if run:
                    runs.append(run)
                run = []
                continue
            c = ring_col(b, y, C, ps)
            if run and c == run[-1][1] + Q:
                run.append((e, c))
            else:
                if run:
                    runs.append(run)
                run = [(e, c)]
        if run:
            runs.append(run)
        for sx in (-d, 0, d):
            for rn in runs:
                out.append((b, sx, rn[0][0], len(rn), rn[0][1]))
    return out


def ring_pass_rows(C, ps):
    """weight rows of pass ps (per 64-channel block): Q for the 1x1 branch, 9 * Q for a 3x3 branch"""
    Q = C // 4
    return sum(Q if b == 0 else 9 * Q for b, _ in RING_PASSES[C][ps])


def ring_stack_row(b, sx, C=64, ps=0):
    """first row (inside pass ps's block of one 64-channel slice) of the weight stack of (branch b >= 1, horizontal shift sx)"""
    Q, row = C // 4, 0
    for bb, _ in RING_PASSES[C][ps]:
        if bb == b:
            return row + (sx // RING_DIL[b] + 1) * 3 * Q
        row += Q if bb == 0 else 9 * Q
    raise KeyError(b)


def msb_ring_weights(weights, C=64, dtype=torch.bfloat16):
    """weights: [w1 [Q,C,1,1], w2..w4 [Q,C,3,3]] fp32 -> [sum over passes of (C/64) * rows(pass), 64]: per pass, per 64-channel block
    kb, the rows of its branches: Q rows of the 1x1 branch, then for every 3x3 branch and kx = 0..2 the 3Q-row stack
    [ky = 2 | ky = 1 | ky = 0] (the order of the output rows r - d, r, r + d an input row feeds)."""
    out = []
    for ps in range(len(RING_PASSES[C])):
        for kb in range(C // 64):
            sl = slice(kb * 64, (kb + 1) * 64)
            for b, _ in RING_PASSES[C][ps]:
                if b == 0:
                    out.append(weights[0][:, sl, 0, 0])
                else:
                    for kx in range(3):
                        out += [weights[b][:, sl, ky, kx] for ky in (2, 1, 0)]
    return torch.cat(out, 0).to(dtype).contiguous()


def msb64_ring_weights(weights, dtype=torch.bfloat16):
    return msb_ring_weights(weights, 64, dtype)


def msb_ring(x, w_stacks, bias, C=64, out=None, co_off=0, stats=None, ci_off=0):
    """The four MultiScaleBlock branches at C = 64 / 128 on the row-ring kernel: x [N,H,W,>=C] bf16 -> out [N,H,W,Co_total] bf16
    (C channels at co_off), IN statistics accumulated into stats.  w_stacks = msb_ring_weights(weights, C)."""
    ops._dev(x)
    N, H, W, Ci_total = x.shape
    if out is None:
        out = torch.empty((N, H, W, C), device=x.device, dtype=torch.bfloat16)
    rows = sum(ring_pass_rows(C, ps) for ps in range(len(RING_PASSES[C]))) * (C // 64)
    if tuple(w_stacks.shape) != (rows, 64) or w_stacks.dtype != torch.bfloat16:
        raise ValueError(f"msb_ring: w_stacks must be bf16 [{rows}, 64] (msb_ring_weights(weights, {C})), got {tuple(w_stacks.shape)}")
    d = _lib.MsbRingDesc()
    d.dtype, d.N, d.H, d.W, d.Ci_total, d.ci_off, d.Co_total, d.co_off = _lib.BF16, N, H, W, Ci_total, ci_off, out.shape[3], co_off
    d.flags = _lib.CONV_STATS if stats is not None else 0
    _lib.call("msg_msb_ring", ctypes.byref(d), C, ops._p(x), ops._p(w_stacks), ops._p(bias), ops._p(out), ops._p(stats), ops._stream())
    _lib.launches += len(RING_PASSES[C]) - 1        # one kernel per pass
    return out


def msb64_ring(x, w_stacks, bias, out=None, co_off=0, stats=None, ci_off=0):
    return msb_ring(x, w_stacks, bias, 64, out, co_off, stats, ci_off)


# ---------------------------------------------------------------------------------------------------------------------
# ConvTranspose2d(k = 4, stride 2, pad 1) as a ROW RING (csrc/convt_ring.cu): out[o, u] = sum in[i, j] w[ky, kx] with
# o = 2 i - 1 + ky, u = 2 j - 1 + kx.  One launch per horizontal output phase px = u mod 2 (and per 64 output channels); a CTA walks
# down a 128-pixel column strip of the input.  Input row r feeds the output rows 2r-1 .. 2r+2 (ky = 0..3), whose accumulators are
# adjacent 64-column slots of an eight-slot ring (slot = output row mod 8), so for each of the phase's two horizontal taps the four
# vertical taps are ONE MMA of N = 256 over the stack [ky = 0 | 1 | 2 | 3].  Input row r completes the output rows 2r-1 and 2r.
# The functions below ARE the schedule (the CUDA kernel restates them; tests/test_convt_ring_cpu.py runs them on tensors).
# ---------------------------------------------------------------------------------------------------------------------
CONVT_RING_KX = ((1, 3), (2, 0))        # [px] -> kx of the phase's two horizontal taps ...
CONVT_RING_DX = ((0, -1), (0, 1))       # ... and the input pixel they read relative to the output pixel pair (u = 2 j' + px)
CONVT_RING_SLOTS = 8
CONVT_RING_LEAD = 3                     # steps (input rows) the issuer may run ahead of the epilogue: a slot is touched again 3 rows later


def convt_ring_row_mmas(r, y0, y1):
    """MMAs input row r issues for the piece of input rows [y0, y1) (output rows [2 y0, 2 y1)), per horizontal tap:
    [(first entry e0 = ky, number of stacked entries, first TMEM column)]"""
    runs, run = [], []
    for e in range(4):
        o = 2 * r - 1 + e
        if not (2 * y0 <= o < 2 * y1):
            if run:
                runs.append(run)
            run = []
            continue
        c = (o % CONVT_RING_SLOTS) * 64
        if run and c == run[-1][1] + 64:
            run.append((e, c))
        else:
            if run:
                runs.append(run)
            run = [(e, c)]
    if run:
        runs.append(run)
    return [(rn[0][0], len(rn), rn[0][1]) for rn in runs]


def convt_ring_weights(w, dtype=torch.bfloat16):
    """w: ConvTranspose2d weight [Cin, Cout, 4, 4] -> [Cout/64][2 px][Cin/64][2 taps][4 ky][64 co][64 ci] as rows of 64"""
    Cin, Cout = w.shape[0], w.shape[1]
    out = []
    for g in range(Cout // 64):
        for px in range(2):
            for kb in range(Cin // 64):
                for t in range(2):
                    kx = CONVT_RING_KX[px][t]
                    for ky in range(4):
                        out.append(w[kb * 64:(kb + 1) * 64, g * 64:(g + 1) * 64, ky, kx].t())
    return torch.cat(out, 0).to(dtype).contiguous()


def convt_ring_supported(x, Cin, Cout):
    return x.dtype == torch.bfloat16 and Cin in (64, 128) and Cout % 64 == 0


def convt_ring(x, w_stacks, bias, Cout, out=None, co_off=0, stats=None, ci_off=0, Cin=None):
    """ConvTranspose2d(4, 2, 1): x [N,H,W,>=Cin] bf16 -> out [N,2H,2W,Co_total] bf16 (Cout channels at co_off), IN statistics
    accumulated into stats.  w_stacks = convt_ring_weights(weight)."""
    ops._dev(x)
    N, H, W, Ci_total = x.shape
    Cin = Ci_total if Cin is None else Cin
    if out is None:
        out = torch.empty((N, 2 * H, 2 * W, Cout), device=x.device, dtype=torch.bfloat16)
    rows = (Cout // 64) * 2 * (Cin // 64) * 512
    if tuple(w_stacks.shape) != (rows, 64) or w_stacks.dtype != torch.bfloat16:
        raise ValueError(f"convt_ring: w_stacks must be bf16 [{rows}, 64] (convt_ring_weights), got {tuple(w_stacks.shape)}")
    d = _lib.ConvtRingDesc()
    d.dtype, d.N, d.H, d.W, d.Cin, d.Cout = _lib.BF16, N, H, W, Cin, Cout
    d.Ci_total, d.ci_off, d.Co_total, d.co_off = Ci_total, ci_off, out.shape[3], co_off
    d.flags = _lib.CONV_STATS if stats is not None else 0
    _lib.call("msg_convt_ring", ctypes.byref(d), ops._p(x), ops._p(w_stacks), ops._p(bias), ops._p(out), ops._p(stats), ops._stream())
    _lib.launches += 2 * (Cout // 64) - 1           # one kernel per phase and 64 output channels
    return out


# ---------------------------------------------------------------------------------------------------------------------
# Output layer Conv2d(64, 3, 7, padding 3) + Tanh fused with the IN + ReLU + residual in front of it, as a ROW RING
# (csrc/out7_ring.cu).  Input row r feeds the output rows r-3 .. r+3 (ky = 6 .. 0): 16-column slots (3 channels padded) of a
# 32-slot ring, so for each horizontal tap (a shifted view of the slab) the 7 vertical taps are ONE MMA of N = 112 over the stack
# [ky = 6 | 5 | ... | 0]; input row r completes output row r-3.
# ---------------------------------------------------------------------------------------------------------------------
OUT7_RING_SLOTS = 32
OUT7_RING_LEAD = 6


def out7_ring_row_mmas(r, y0, y1):
    """MMAs input row r issues per horizontal tap for the piece of rows [y0, y1): [(first entry e0, entries, first TMEM column)];
    entry e = output row r - 3 + e = vertical tap ky = 6 - e"""
    runs, run = [], []
    for e in range(7):
        o = r - 3 + e
        if not (y0 <= o < y1):
            if run:
                runs.append(run)
            run = []
            continue
        c = (o % OUT7_RING_SLOTS) * 16
        if run and c == run[-1][1] + 16:
            run.append((e, c))
        else:
            if run:
                runs.append(run)
            run = [(e, c)]
    if run:
        runs.append(run)
    return [(rn[0][0], len(rn), rn[0][1]) for rn in runs]


def out7_ring_weights(w, dtype=torch.bfloat16):
    """w: Conv2d weight [3, 64, 7, 7] -> [7 kx][8 entries][16 co][64 ci] as rows of 64 (entry e < 7 = ky 6 - e, channels 3..15 and
    entry 7 zero)"""
    out = torch.zeros(7, 8, 16, 64, device=w.device, dtype=w.dtype)
    for kx in range(7):
        for e in range(7):
            out[kx, e, :3] = w[:, :, 6 - e, kx]
    return out.reshape(7 * 128, 64).to(dtype).contiguous()


def out7_ring(f, in_stats, residual, w_stacks, bias, nchw_out=None, in_affine=None):
    """y = tanh(conv7x7(residual + ReLU(IN(f))) + bias): f, residual [N,H,W,64] bf16, in_stats fp64 [N,64,2] (raw plane sums of f)
    -> fp32 [N,3,H,W].  in_affine: optional (gamma, beta, img_stride) of the IN (ops.instnorm_apply)."""
    ops._dev(f)
    N, H, W, Cf = f.shape
    if f.dtype != torch.bfloat16 or residual.dtype != torch.bfloat16 or residual.shape[:3] != f.shape[:3]:
        raise ValueError("out7_ring: f and residual must be bf16 NHWC tensors of the same plane")
    if tuple(w_stacks.shape) != (896, 64) or w_stacks.dtype != torch.bfloat16:
        raise ValueError(f"out7_ring: w_stacks must be bf16 [896, 64] (out7_ring_weights), got {tuple(w_stacks.shape)}")
    if nchw_out is None:
        nchw_out = torch.empty((N, 3, H, W), device=f.device, dtype=torch.float32)
    d = _lib.Out7RingDesc()
    d.dtype, d.N, d.H, d.W = _lib.BF16, N, H, W
    d.Cf_total, d.cf_off, d.Cr_total, d.cr_off, d.Cs_total, d.cs_off = Cf, 0, residual.shape[3], 0, in_stats.shape[1], 0
    if in_affine is None:
        _lib.call("msg_out7_ring", ctypes.byref(d), ops._p(f), ops._p(in_stats), ops._p(residual), ops._p(w_stacks), ops._p(bias),
                  ops._p(nchw_out), ops._stream())
    else:
        _lib.call("msg_out7_ring_affine", ctypes.byref(d), ops._p(f), ops._p(in_stats), *ops._aff(in_affine), ops._p(residual),
                  ops._p(w_stacks), ops._p(bias), ops._p(nchw_out), ops._stream())
    return nchw_out


# ---------------------------------------------------------------------------------------------------------------------
# Conv2d(64, Cout, 4, stride 2, padding 1) (+ the IN + ReLU in front of it) as a ROW RING (csrc/down_ring.cu):
# y[o, u] = sum a[2o - 1 + ky, 2u - 1 + kx] w[ky, kx].  A CTA walks down a strip of 128 output pixels; input row r arrives as its
# even-pixel and its odd-pixel slab (kx = 0, 2 read the odd slab at u - 1, u; kx = 1, 3 the even slab at u, u + 1) and feeds the two
# output rows (r - 1) // 2 and (r - 1) // 2 + 1 with the vertical taps ky = 3 - r % 2 and 1 - r % 2: adjacent 64-column slots of an
# eight-slot ring (slot = output row mod 8), ONE MMA of N = 128 per horizontal tap.  An even input row r completes output row r/2 - 1.
# ---------------------------------------------------------------------------------------------------------------------
DOWN_RING_LEAD = 8


def down_ring_row_mmas(r, y0, y1):
    """MMAs input row r issues per horizontal tap for the piece of OUTPUT rows [y0, y1): [(first entry e0, entries, first TMEM column)];
    entry e = output row (r - 1) // 2 + e, vertical tap ky = 3 - r % 2 - 2 e"""
    of = (r - 1) // 2
    runs, run = [], []
    for e in range(2):
        o = of + e
        if not (y0 <= o < y1):
            if run:
                runs.append(run)
            run = []
            continue
        c = (o % 8) * 64
        if run and c == run[-1][1] + 64:
            run.append((e, c))
        else:
            if run:
                runs.append(run)
            run = [(e, c)]
    if run:
        runs.append(run)
    return [(rn[0][0], len(rn), rn[0][1]) for rn in runs]


def down_ring_weights(w, dtype=torch.bfloat16):
    """w: Conv2d weight [Cout, 64, 4, 4] -> [Cout/64][4 kx][2 input-row parities][2 entries][64 co][64 ci] as rows of 64"""
    out = []
    for g in range(w.shape[0] // 64):
        for kx in range(4):
            for par in range(2):
                for e in range(2):
                    out.append(w[g * 64:(g + 1) * 64, :, 3 - par - 2 * e, kx])
    return torch.cat(out, 0).to(dtype).contiguous()


def down_ring(x, in_stats, w_stacks, bias, Cout, out=None, co_off=0, stats=None, ci_off=0, in_affine=None):
    """Conv2d(64, Cout, 4, 2, 1) of ReLU(IN(x)) (in_stats: fp64 [N,C,2] raw plane sums of x; None: x is used as it is; in_affine:
    optional (gamma, beta, img_stride) of the IN):
    x [N,H,W,>=64] bf16 -> out [N,H/2,W/2,Co_total] bf16 (Cout channels at co_off), IN statistics accumulated into stats."""
    ops._dev(x)
    N, H, W, Ci_total = x.shape
    if out is None:
        out = torch.empty((N, H // 2, W // 2, Cout), device=x.device, dtype=torch.bfloat16)
    rows = (Cout // 64) * 1024
    if tuple(w_stacks.shape) != (rows, 64) or w_stacks.dtype != torch.bfloat16:
        raise ValueError(f"down_ring: w_stacks must be bf16 [{rows}, 64] (down_ring_weights), got {tuple(w_stacks.shape)}")
    d = _lib.DownRingDesc()
    d.dtype, d.N, d.H, d.W, d.Cout = _lib.BF16, N, H, W, Cout
    d.Ci_total, d.ci_off, d.Co_total, d.co_off = Ci_total, ci_off, out.shape[3], co_off
    d.Cs_total, d.cs_off = (in_stats.shape[1], 0) if in_stats is not None else (0, 0)
    d.flags = _lib.CONV_STATS if stats is not None else 0
    if in_affine is None:
        _lib.call("msg_down_ring", ctypes.byref(d), ops._p(x), ops._p(in_stats), ops._p(w_stacks), ops._p(bias), ops._p(out),
                  ops._p(stats), ops._stream())
    else:
        _lib.call("msg_down_ring_affine", ctypes.byref(d), ops._p(x), ops._p(in_stats), *ops._aff(in_affine), ops._p(w_stacks),
                  ops._p(bias), ops._p(out), ops._p(stats), ops._stream())
    _lib.launches += Cout // 64 - 1                 # one kernel per 64 output channels
    return out
