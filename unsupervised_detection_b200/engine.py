"""Static launch-list executor for the hot path: bf16 NHWC activations in HBM, every op a call into libcis_b200.so.

Networks are described once (shapes are static), which produces three launch lists -- forward, backward for the recover
step and backward for the generator step -- that are then replayed (optionally inside a CUDA graph) every iteration.
PyTorch only owns device memory and streams here; there is no autograd and no torch compute on the hot path.
"""
import ctypes as C
import os

import numpy as np
import torch

from . import _lib
from ._lib import CisConv, CisWgrad, CisSrc, ACT_NONE, ACT_ELU, ACT_LEAKY


def ru(x, m):
    return (x + m - 1) // m * m


def same_pad(n_in, k, s=1, d=1):
    """TF 'SAME' padding split (SURVEY App. A.2)."""
    out = -(-n_in // s)
    total = max((out - 1) * s + (k - 1) * d + 1 - n_in, 0)
    return total // 2, total - total // 2


SIDE_STREAM = True
_SIDE = {}
MULTI_PARAM_OPS = os.environ.get('CIS_MULTI_PARAM', '1') == '1'   # per-layer pack / un-pack / BN launches batched into multi-job launches
DACT_COLSUM = os.environ.get('CIS_DACT_COLSUM', '1') == '1'       # activation derivative and bias-gradient partials of a layer in one launch
PLAN_MODEL = int(os.environ.get('CIS_PLAN_MODEL', '4'))           # MT choice of setup_halo: 1 wave model, 2 busiest-SM model, 3 smallest stack, 4 hybrid (default)
COLSUM_PIX = int(os.environ.get('CIS_COLSUM_PIX', '4'))            # pixels per thread of the column-sum passes (fewer = more blocks, <= 592)


def _side_stream(device, key=0):
    """Side lane of a plan replay.  `key` gives concurrently replayed plans (the pipelined PWC-Net branch) their own lane so the two
    branches do not serialise on one helper stream."""
    k = (str(device), key)
    if k not in _SIDE:
        _SIDE[k] = torch.cuda.Stream(device=device)
    return _SIDE[k]


class Plan(object):
    """An ordered list of C-ABI launches (and a few torch memsets) replayable on any stream."""

    def __init__(self, name=''):
        self.name = name
        self.ops = []
        self.keep = []  # ctypes structs / tensors that must outlive the plan

    def add(self, fname, *args, flops=0.0, lane=0):
        fn = getattr(_lib.load(), fname)
        self.ops.append((fn, args, fname, flops, lane))

    def add_py(self, fn, label='py'):
        self.ops.append((None, fn, label, 0.0, 0))

    def zero(self, t):
        self.keep.append(t)
        self.add('cis_zero', t.data_ptr(), t.numel() * t.element_size())

    def join(self):
        """Main lane waits for everything issued on the side lane so far."""
        self.ops.append((None, None, 'join', 0.0, 0))

    def run(self, stream=None, lane_key=0):
        """Lane 0 = the current stream; lane 1 = a side stream forked/joined with events (weight-gradient GEMMs run there,
        concurrently with the data-gradient chain).  Works eagerly and under CUDA-graph capture."""
        if stream is not None or not SIDE_STREAM or not any(op[4] for op in self.ops):
            st = stream if stream is not None else torch.cuda.current_stream().cuda_stream
            for fn, args, name, _, _ in self.ops:
                if fn is None:
                    if args is not None:
                        args()
                else:
                    rc = fn(*args, st)
                    if rc != 0:
                        _lib.check(rc, name)
            return
        main = torch.cuda.current_stream()
        side = _side_stream(main.device, lane_key)
        st0, st1 = main.cuda_stream, side.cuda_stream
        main_ahead, side_used = True, False
        for fn, args, name, _, lane in self.ops:
            if fn is None:
                if name == 'join':
                    if side_used:
                        ev = torch.cuda.Event()
                        ev.record(side)
                        main.wait_event(ev)
                        side_used = False
                elif args is not None:
                    args()
                    main_ahead = True
                continue
            if lane == 1:
                if main_ahead:
                    ev = torch.cuda.Event()
                    ev.record(main)
                    side.wait_event(ev)
                    main_ahead = False
                rc = fn(*args, st1)
                side_used = True
            else:
                rc = fn(*args, st0)
                main_ahead = True
            if rc != 0:
                _lib.check(rc, name)
        if side_used:
            ev = torch.cuda.Event()
            ev.record(side)
            main.wait_event(ev)

    def batch_param_ops(self, device):
        """A plan made only of the five parameter-space ops (BN fold, weight packs, gradient un-pack, BN chain rule), one launch per
        layer each -> one multi-job launch per kind (cis_param_multi), in dependency order: fold -> packs, un-pack -> chain rule."""
        from ._lib import CisParamJob, JOB_PACK, JOB_PACK_TILED, JOB_UNPACK, JOB_BN_FOLD, JOB_BN_CHAIN
        if not MULTI_PARAM_OPS or not self.ops:
            return self
        jobs = {k: [] for k in range(5)}
        for fn, a, name, _, _ in self.ops:
            j = CisParamJob()
            if name == 'cis_pack_weights':
                w, kmap, K_pad, rows, cout, sn, nmap, wp = a
                j.kind, blocks = JOB_PACK, -(-(rows * K_pad) // 256)
                ptrs, ints = [w, kmap, nmap, wp], [K_pad, rows, cout, sn]
            elif name == 'cis_pack_weights_tiled':
                w, kmap, cin8, ntaps, n_tiles, BN, cout, sn, nmap, out, layout = a
                j.kind, blocks = JOB_PACK_TILED, -(-(n_tiles * (-(-cin8 // 64)) * ntaps * BN * 64) // 256)
                if sn == 1:               # forward orientation: one block per BN x 64 tile (transposed through shared memory)
                    blocks = n_tiles * (-(-cin8 // 64)) * ntaps
                ptrs, ints = [w, kmap, nmap, out], [cin8, ntaps, n_tiles, BN, cout, sn, layout]
            elif name == 'cis_unpack_wgrad':
                dwp, kmap, K_pad, cout, nsplit, dw, colpart, nblocks, nch, db, layout = a
                j.kind, blocks = JOB_UNPACK, -(-(cout * K_pad + nch) // 256)
                ptrs, ints = [dwp, kmap, dw, colpart, db], [K_pad, cout, nsplit, nblocks, nch, layout]
            elif name == 'cis_bn_fold':
                w, bias, gamma, beta, nw, cout, w_eff, b_eff = a
                j.kind, blocks, j.n = JOB_BN_FOLD, -(-max(nw, cout) // 256), nw
                ptrs, ints = [w, bias, gamma, beta, w_eff, b_eff], [cout]
            elif name == 'cis_bn_chain':
                w, bias, gamma, dwe, dbe, nw, cout, dbias, dgamma, dbeta = a
                j.kind, blocks, j.n = JOB_BN_CHAIN, -(-cout // 8), nw          # one block per 8 output channels (csrc: kBnChainCo)
                ptrs, ints = [w, bias, gamma, dwe, dbe, dbias, dgamma, dbeta], [cout]
            else:
                return self          # something else in the plan: leave it as it is
            for q, v in enumerate(ptrs):
                j.p[q] = v
            for q, v in enumerate(ints):
                j.i[q] = v
            jobs[j.kind].append((j, blocks))
        out = Plan(self.name + '.multi')
        out.keep = self.keep
        for kind in (JOB_BN_FOLD, JOB_PACK_TILED, JOB_PACK, JOB_UNPACK, JOB_BN_CHAIN):
            if not jobs[kind]:
                continue
            arr = (CisParamJob * len(jobs[kind]))()
            first = 0
            for q, (j, blocks) in enumerate(jobs[kind]):
                j.i[7] = first
                arr[q] = j
                first += blocks
            tab = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(device)
            out.keep.append(tab)
            out.add('cis_param_multi', tab.data_ptr(), len(jobs[kind]), first)
        return out

    def count(self):
        """Kernel launches of one replay (a two-launch split-K conv counts twice)."""
        n = 0
        for fn, args, name, _, _ in self.ops:
            if fn is None or name == 'cis_zero':      # a memset node, not a kernel
                continue
            n += 1
            if name == 'cis_conv_igemm':
                d = args[0]._obj
                if d.splits > 1 and not d.sk_cluster:
                    n += 1
        return n

    def extend(self, other):
        self.ops += other.ops
        self.keep += other.keep


class Act(object):
    """A bf16 NHWC activation: a channel slice [c_off, c_off+C8) of a buffer [N,H,W,pitch]."""

    def __init__(self, N, H, W, C, device, buf=None, c_off=0, chanmap=None, n_mod=0, dep=frozenset(), name=''):
        if chanmap is not None and not C:
            C = max(chanmap) + 1
        self.N, self.H, self.W, self.C = N, H, W, C
        self.C8 = ru(C, 8) if chanmap is None else len(chanmap)
        if buf is None:
            buf = torch.zeros(N, H, W, self.C8, dtype=torch.bfloat16, device=device)
        self.buf = buf
        self.pitch = buf.shape[-1]
        self.c_off = c_off
        self.chanmap = list(chanmap) if chanmap is not None else list(range(C)) + [-1] * (self.C8 - C)
        self.n_mod = n_mod
        self.dep = frozenset(dep)
        self.name = name
        self.grad = None
        self.grad_written = {}   # mode -> bool
        self.device = device
        self.gen_rows = None     # batch rows processed by the generator-step backward (2B of 3B)

    @property
    def ptr(self):
        return self.buf.data_ptr()

    def src(self):
        return CisSrc(self.ptr, self.pitch, self.c_off, self.C8 // 8, self.n_mod)

    def rows(self, mode):
        return self.gen_rows if (mode == 'G' and self.gen_rows) else self.N

    def alias(self, n_mod):
        """Same storage seen as a batch-broadcast source (features shared by the three recover_net calls)."""
        a = Act(self.N, self.H, self.W, self.C, self.device, buf=self.buf, c_off=self.c_off, chanmap=self.chanmap, n_mod=n_mod,
                dep=self.dep, name=self.name + '.shared')
        a._owner = self
        a.grad_written = self.grad_written
        return a

    def get_grad(self):
        if getattr(self, '_owner', None) is not None:
            return self._owner.get_grad()
        if self.grad is None:
            self.grad = Act(self.N, self.H, self.W, self.C, self.device, chanmap=self.chanmap, name=self.name + '.grad')
        return self.grad

    def float(self):
        """Debug/test helper: real channels as fp32 [N,H,W,C] (a torch op, not on the hot path)."""
        idx = [i for i, m in enumerate(self.chanmap) if m >= 0]
        return self.buf[..., self.c_off:self.c_off + self.C8].float()[..., idx]


def _fill_taps(d, taps):
    d.ntaps = len(taps)
    for i, (a, b) in enumerate(taps):
        d.dh[i] = a
        d.dw[i] = b


def _fill_srcs(d, srcs):
    d.nsrc = len(srcs)
    for i, s in enumerate(srcs):
        d.src[i] = s.src()


def pick_bn(cout, cap=None):
    """(BN, n_tiles) of the GEMM N dimension.  `cap` (32 / 64) forces narrower n-tiles: more, smaller CTAs for layers whose pixel
    count yields only a handful of 128-row tiles (experiment CIS_SMALL_BN, DESIGN.md section 6 E2)."""
    if cout <= 16:
        return 16, 1
    if cout <= 32:
        return 32, 1
    if cap in (32, 64) and cout > cap:
        return cap, -(-cout // cap)
    if cout <= 64:
        return 64, 1
    return 128, -(-cout // 128)


def small_bn_cap(level):
    """CIS_SMALL_BN="cap:level" (default unset = off): PWC-Net layers of pyramid level >= `level` (12x20 and coarser for level 5)
    use n-tiles of `cap` columns.  Returns the cap for this level or None."""
    spec = os.environ.get('CIS_SMALL_BN', '')
    if not spec:
        return None
    cap, _, lvl = spec.partition(':')
    return int(cap) if level >= int(lvl or 5) else None



NUM_SMS = 148
HALO_ENABLED = True
WGRAD_TMA = True
MATERIALIZE_MISALIGNED_CONCAT = True


WGRAD_CTAS_PER_SM = int(os.environ.get('CIS_WGRAD_CTAS_PER_SM', '2'))   # split-K target: CTAs per SM of one weight-gradient launch
WGRAD_MAX_SLICE_MB = float(os.environ.get('CIS_WGRAD_MAX_SLICE_MB', '16'))  # 0 = no cap on splits x Cout x K_pad x 4 bytes per layer
WGRAD_HALO_MIN_CH = int(os.environ.get('CIS_WGRAD_HALO_MIN_CH', '16'))   # thinner inputs: the per-tap 64-channel padding costs more than the gather path
WGRAD_HALO = os.environ.get('CIS_WGRAD_HALO', '1') == '1'   # halo-resident swapped wgrad kernel (CisWgrad.tma = 2) where it fits


def wgrad_halo_fits(taps, cout, stride):
    """Eligibility of the halo-resident wgrad kernel (mirrors launch_wgrad_halo in csrc/conv_igemm.cu): stride 1, taps listed in
    increasing row-major order, (taps/2) x min(Cout16, 64) accumulator columns within TMEM, >= 2 pipeline stages in shared memory."""
    if stride != 1 or not taps:
        return False
    hoy, hox = min(a for a, _ in taps), min(b for _, b in taps)
    keys = [(a - hoy) * 1024 + (b - hox) for a, b in taps]
    if any(k1 <= k0 for k0, k1 in zip(keys, keys[1:])):
        return False
    wh, hh = 8 + max(b for _, b in taps) - hox, 8 + max(a for a, _ in taps) - hoy
    nh = 64 if cout > 64 else ru(cout, 16)
    if ((len(taps) + 1) // 2) * nh > 512 or wh > 256 or hh > 256:
        return False
    stage = ru(wh * hh * 128, 1024) + 8192
    return (200 * 1024) // stage >= 2


def _pow2_cols(c):
    for v in (32, 64, 128, 256, 512):
        if c <= v:
            return v
    return 1024


# split-K of launches that cover only a few SMs (low-resolution pyramid levels): 0 = off, 2 = on (two launches: private partial slices +
# a parallel finish kernel with a fixed summation order; measured r02: -0.4 ms per step)
SPLITK = int(os.environ.get('CIS_SPLITK', '2'))
SPLITK_CLUSTER = os.environ.get('CIS_SPLITK_CLUSTER', '0') == '1'   # reduce through a thread-block cluster (DSMEM) instead of the finish launch
SPLITK_MAX = int(os.environ.get('CIS_SPLITK_MAX', '16'))
SPLITK_NCTA = int(os.environ.get('CIS_SPLITK_NCTA', '64'))          # only launches with at most this many CTAs are split
SPLITK_MIN_UNITS = int(os.environ.get('CIS_SPLITK_MIN_UNITS', '18'))  # ... and at least this many serial pipeline steps per CTA
# smallest useful fraction of a launch's 16x8 output tiles for the halo kernel to take a stride-1 layer (below it: the K-dense gather
# kernel).  Low-resolution maps (6x10, 8x14, 4x7) only fill 20-45 % of their tiles, but the gather kernel's cp.async producers cost
# ~1450 clk per 64-wide K block against ~400 clk per 3-tap stage of the halo kernel (CIS_TRACE build, r02)
HALO_MIN_UTIL = float(os.environ.get('CIS_HALO_MIN_UTIL', '0.2'))
# experiment switch (default off = current behaviour): launches whose sources hold <= this many channels and that need >= 16 MMAs per
# tile on the compact thin halo (the 7x7 first layers: 28 MMAs of K = 16, where the K-dense gather kernel walks 7 blocks of K = 64)
# stay on the gather kernel -- an A/B lever for the thin-layer path, see DESIGN.md section 2.1
HALO_SKIP_THIN = int(os.environ.get('CIS_HALO_SKIP_THIN', '0'))


def setup_splitk(d, device, keep):
    """Launches whose grid would cover well under the 148 SMs (low-resolution pyramid levels) split their K loop over grid.z;
    see CisConv.splits.  Scratch and ticket buffers are per launch (launches on different lanes may overlap)."""
    if not SPLITK:
        return
    m_chunks = sum(d.src[i].chunks for i in range(d.nsrc))
    if d.halo:
        Hp0, Wp0 = -(-d.OH // d.dil), -(-d.OW // d.dil)
        tiles = (-(-Wp0 // 8)) * (-(-Hp0 // (16 * d.MT))) * d.dil * d.dil * d.N
        ncta, units, min_units, mt = tiles * d.n_tiles, -(-m_chunks // 8), 1, d.MT
    else:
        ncta, units, min_units, mt = (-(-(d.N * d.OH * d.OW) // 128)) * d.n_tiles, d.K_pad // 64, 4, 1
    steps = units * (d.ntaps if d.halo else 1)     # serial pipeline steps of one CTA (halo: one per (chunk, tap); generic: one per 64-wide K block)
    if ncta > SPLITK_NCTA or steps < SPLITK_MIN_UNITS:
        return
    splits = min(units // min_units, -(-2 * NUM_SMS // ncta), SPLITK_MAX, 8 if SPLITK_CLUSTER else 1 << 30)
    if splits < 2:
        return
    per = -(-units // splits)
    splits = -(-units // per)
    if splits < 2:
        return
    if SPLITK_CLUSTER and splits <= 8 and mt * 128 * d.BN * 4 + 1024 <= 226 * 1024:
        # the splits of a tile form a thread-block cluster and reduce through distributed shared memory: no scratch, no second launch
        d.splits, d.sk_scratch, d.sk_counters, d.sk_cluster = splits, None, None, 1
        return
    sc = torch.empty(ncta * mt * splits * 128 * d.BN, dtype=torch.float32, device=device)
    keep.append(sc)
    d.splits, d.sk_scratch, d.sk_counters = splits, sc.data_ptr(), None


def thin_items(rel, m_chunks):
    """The K=16 MMAs of a compact-thin-halo launch (CisConv.thin) for halo-relative taps `rel` (any order: the parity taps of data
    gradients and transposed convs come in descending order).  16 channels: one MMA per tap, K halves = channels 0-7 / 8-15 (the next
    8-channel plane).  8 channels: the second K half reads the NEXT pixel, so two x-adjacent taps share one MMA (taps are paired in
    row-major order); a tap left at the end of a row run pairs with a zero weight half, starting one pixel to its left when there is
    one (then the halo needs no extra column).  Returns [(dy, dx, (i0, c0), (i1, c1))]: the MMA's halo origin and, per
    K half, the index into `rel` (-1 = zero weights) and the first channel."""
    if m_chunks == 2:
        return [(a, b, (i, 0), (i, 8)) for i, (a, b) in enumerate(rel)]
    pos = {t: i for i, t in enumerate(rel)}
    used, items = set(), []
    for i in sorted(range(len(rel)), key=lambda q: rel[q]):
        a, b = rel[i]
        if i in used:
            continue
        used.add(i)
        j = pos.get((a, b + 1))
        if j is not None and j not in used:
            used.add(j)
            items.append((a, b, (i, 0), (j, 0)))
        elif b > 0:
            items.append((a, b - 1, (-1, 0), (i, 0)))
        else:
            items.append((a, b, (i, 0), (-1, 0)))
    return items


def _thin_footprint(HP, m_chunks, nmma, BN, nhs):
    """(shared memory bytes, operand bytes per CTA) of a compact-thin-halo CTA: nhs halo stages of m_chunks 16-byte-per-pixel planes,
    the whole weight set resident (BN x 32 B per MMA, one bulk copy)."""
    plane = ru(HP * 16, 128)
    smem = nhs * ru(m_chunks * plane, 1024) + HP * 4 + 1024 + nmma * BN * 32 + 1024
    return smem, m_chunks * HP * 16 + nmma * BN * 32


def setup_halo(d, taps, dil, n_tiles):
    """Switch a stride-1 gather descriptor to the halo-resident kernel when it pays off: taps become offsets relative to the
    halo origin in units of `dil`, MT (stacked 16x8 tiles per CTA) is chosen by a wave/overhead model.  Sources of <= 16 channels in
    all take the compact thin halo (CisConv.thin, see thin_items): returns the MMA list then, True for the 128-byte halo, False
    when the launch stays on the gather kernel."""
    if not HALO_ENABLED or d.sh != 1 or d.sw != 1:
        return False
    if any(a % dil or b % dil for a, b in taps):
        return False
    if dil > 1 and (d.OH != d.H or d.OW != d.W):
        return False
    th = [(a // dil, b // dil) for a, b in taps]
    hoy, hox = min(a for a, _ in th), min(b for _, b in th)
    rel = [(a - hoy, b - hox) for a, b in th]
    ey, ex = max(a for a, _ in rel), max(b for _, b in rel)
    Hp0, Wp0 = -(-d.OH // dil), -(-d.OW // dil)
    tiles_x = -(-Wp0 // 8)
    best = None
    ntaps = len(taps)
    m_chunks = sum(d.src[i].chunks for i in range(d.nsrc))
    thin = m_chunks <= 2 and dil == 1
    items = None
    if thin:
        items = thin_items(rel, m_chunks)
        if m_chunks == 1:                       # the second K half of every MMA reads one pixel to the right of its origin
            ex = max(ex, max(b for _, b, _, _ in items) + 1)
        ntaps = len(items)                      # MMAs per tile
    if HALO_SKIP_THIN and m_chunks * 8 <= HALO_SKIP_THIN and ntaps >= 16:
        return False
    nchunks = -(-m_chunks // 8)
    nhs = 2 if nchunks > 1 else 1
    force = int(os.environ.get('CIS_FORCE_MT128', '0')) if d.BN == 128 else 0
    for MT in (1, 2, 3, 4):
        if MT * d.BN > 512 or (force and MT != force):
            continue
        HP = (8 + ex) * (16 * MT + ey)
        fixed = nhs * ru(HP * 128, 1024) + HP * 4 + 1024
        smem = fixed + min(3, ntaps * nchunks) * d.BN * 128 + 1024
        if smem > 227 * 1024:          # (also the stack-height cap of the compact halo: taller stacks were not measured)
            continue
        if thin:
            smem, opb = _thin_footprint(HP, m_chunks, ntaps, d.BN, 1)
        tiles_y = -(-Hp0 // (16 * MT))
        util = (Hp0 * Wp0) / float(tiles_y * 16 * MT * tiles_x * 8)
        if util < (HALO_MIN_UTIL if dil == 1 else 0.5):      # dilated phases: no TMA halo path, d*d times the CTAs -> keep the old rule
            continue
        ncta = d.N * dil * dil * tiles_x * tiles_y * n_tiles
        cps = max(1, min((225 * 1024) // smem, 512 // _pow2_cols(MT * d.BN), 6))
        # per CTA: tensor time vs operand traffic (weights through the TMA engine ~40 B/clk/SM, halo through LDGSTS ~16 B/clk/SM),
        # plus a fixed prologue/epilogue latency that co-resident CTAs overlap
        t_mma = MT * 2.0 * d.BN * ntaps * nchunks
        t_mem = (d.BN * 128 * ntaps / 40.0 + HP * 128 / 16.0) * nchunks
        if thin:
            t_mem = opb / 40.0                  # halo planes and weights through the TMA engine
        t_cta = max(t_mma, t_mem) + (4000.0 + 1500.0 * MT) / cps
        cost = -(-ncta // (NUM_SMS * cps)) * cps * t_cta / min(cps, max(1.0, ncta / float(NUM_SMS)))
        if PLAN_MODEL == 2:
            # busiest SM: its CTAs' throughput-bound parts add up, their fixed latencies overlap cps at a time
            per_sm = -(-ncta // NUM_SMS)
            cost = per_sm * max(t_mma, t_mem) + (4000.0 + 1500.0 * MT) * (-(-per_sm // cps))
        if PLAN_MODEL == 3:
            cost = float(MT)            # smallest feasible stack
        if PLAN_MODEL == 4:
            # measured r02 (A/B of models 1-3 over every layer of the step): the smallest feasible stack wins everywhere EXCEPT on
            # big grids of short tiles (MMA loop below the fixed prologue + epilogue of a CTA), where the wave model's choice holds
            n1 = d.N * dil * dil * tiles_x * (-(-Hp0 // 16)) * n_tiles
            if not (2.0 * d.BN * ntaps * nchunks < 6000.0 and n1 > 4 * NUM_SMS):
                cost = float(MT)
        if best is None or cost < best[0] - 1e-9:
            best = (cost, MT, util)
    if best is None:
        return False
    d.halo, d.dil, d.MT, d.hoy, d.hox, d.ey, d.ex = 1, dil, best[1], hoy, hox, ey, ex
    if thin:
        d.thin = 1
        _fill_taps(d, [(a, b) for a, b, _, _ in items])
        return items
    _fill_taps(d, rel)
    return True


# stride-2 forward convolutions of >= 32-channel inputs on the 128-byte halo kernel (4 space-to-depth phase tensor maps, CisConv.nph = 4).
# Off by default: measured r02 neutral on those layers -- the K-dense gather kernel stays their stride-2 path.  Thin inputs (<= 16
# channels) always take the phases on the compact thin halo, where x-adjacent taps of a phase share one MMA.
S2_HALO = os.environ.get('CIS_S2_HALO', '0') == '1'


def setup_halo_s2(d, taps, n_tiles):
    """Stride-2 forward conv as a halo-kernel launch: input pixel (2*oh + u, 2*ow + v) of tap (u, v) is pixel (oh + u // 2, ow + v // 2)
    of the space-to-depth phase (u % 2, v % 2), so the conv is the sum over the 4 phases of stride-1 convs with the taps of that phase.
    Returns the tap permutation (phase-major) the pre-tiled weights must follow, or None when the launch stays on the gather kernel.
    Thin inputs (<= 16 channels, compact halo): the MMA list of thin_items per phase is left in d.thin_items, its K halves index `taps`."""
    if not HALO_ENABLED or d.sh != 2 or d.sw != 2:
        return None
    m_chunks = sum(d.src[i].chunks for i in range(d.nsrc))
    thin = m_chunks <= 2
    if not (thin or S2_HALO):
        return None
    if not thin and any(d.src[i].chunks % 8 for i in range(d.nsrc - 1)):   # TMA halo path only: a 64-channel chunk never straddles sources
        return None
    ph = [((u % 2) * 2 + (v % 2), u // 2, v // 2) for u, v in taps]
    order = sorted(range(len(taps)), key=lambda i: (ph[i][0], i))
    hoy, hox = min(a for _, a, _ in ph), min(b for _, _, b in ph)
    rel = [(ph[i][1] - hoy, ph[i][2] - hox) for i in order]
    ey, ex = max(a for a, _ in rel), max(b for _, b in rel)
    nchunks = -(-m_chunks // 8)
    nmma, items, bounds = len(taps), None, [0]
    if thin:
        items = []
        for q in range(4):
            idx = [k for k in range(len(order)) if ph[order[k]][0] == q]
            for a, b, h0, h1 in thin_items([rel[k] for k in idx], m_chunks):
                items.append((a, b) + tuple((order[idx[t]] if t >= 0 else -1, c) for t, c in (h0, h1)))
            bounds.append(len(items))
        if m_chunks == 1:
            ex = max(ex, max(b for _, b, _, _ in items) + 1)
        nmma = len(items)
        if HALO_SKIP_THIN and m_chunks * 8 <= HALO_SKIP_THIN and nmma >= 16:
            return None
    tiles_x = -(-d.OW // 8)
    best = None
    for MT in (1, 2, 3, 4):
        if MT * d.BN > 512:
            continue
        HP = (8 + ex) * (16 * MT + ey)
        smem = 2 * ru(HP * 128, 1024) + HP * 4 + 2048 + 2 * d.BN * 128
        if smem > 227 * 1024:
            continue
        if thin:
            smem, opb = _thin_footprint(HP, m_chunks, nmma, d.BN, 2)
        tiles_y = -(-d.OH // (16 * MT))
        util = (d.OH * d.OW) / float(tiles_y * 16 * MT * tiles_x * 8)
        if util < HALO_MIN_UTIL:
            continue
        ncta = d.N * tiles_x * tiles_y * n_tiles
        cps = max(1, min((225 * 1024) // smem, 512 // _pow2_cols(MT * d.BN), 4))
        t_mma = MT * 2.0 * d.BN * nmma * nchunks
        t_mem = (d.BN * 128 * len(taps) / 40.0 + 4 * HP * 128 / 40.0) * nchunks
        if thin:
            t_mem = 4 * opb / 40.0
        t_cta = max(t_mma, t_mem) + (4000.0 + 1500.0 * MT) / cps
        cost = -(-ncta // (NUM_SMS * cps)) * cps * t_cta / min(cps, max(1.0, ncta / float(NUM_SMS)))
        if best is None or cost < best[0] - 1e-9:
            best = (cost, MT)
    if best is None:
        return None
    d.halo, d.dil, d.MT, d.hoy, d.hox, d.ey, d.ex = 1, 1, best[1], hoy, hox, ey, ex
    d.sh = d.sw = 1                     # the phases absorb the stride; H x W stay the input size (tensor maps)
    d.nph = 4
    if thin:
        d.thin, d.thin_items = 1, items
        _fill_taps(d, [(a, b) for a, b, _, _ in items])
    else:
        _fill_taps(d, rel)
        for q in range(4):
            bounds.append(bounds[-1] + sum(1 for i in order if ph[i][0] == q))
    for q in range(5):
        d.ph_tap[q] = bounds[q]
    return order


GROUP_PARITY = os.environ.get('CIS_GROUP_PARITY', '1') == '1'   # the 4 output-parity launches of a stride-2 dgrad / transposed conv as one
GROUP_PARITY_MAX_TILES = int(os.environ.get('CIS_GROUP_PARITY_MAX_TILES', '1000000'))   # optional cap on the 16x8 tiles per parity (600: +0.4 % device-resident, within noise end to end)


def merge_parity_launches(descs):
    """Four (or fewer) halo-kernel descriptors that differ only in taps / halo origin / weights / output extent and offset -> ONE grouped
    descriptor (CisConv.nsub), or None when they cannot share a launch."""
    if not GROUP_PARITY or not (2 <= len(descs) <= 4):
        return None
    d0 = descs[0]
    same = ('N', 'H', 'W', 'BN', 'n_tiles', 'nsrc', 'act', 'DH', 'DW', 'osh', 'osw', 'out', 'out_pitch', 'out_coff', 'out_ch', 'outf', 'outf_pitch',
            'outf_coff', 'outf_ch', 'add_pre', 'add_pre_pitch', 'add_pre_coff', 'add_post', 'addf_pre', 'mode', 'bias', 'thin')
    for d in descs:
        if not d.halo or d.dil != 1 or d.splits > 1 or d.nph > 1 or any(getattr(d, f) != getattr(d0, f) for f in same):
            return None
        if any(bytes(d.src[i]) != bytes(d0.src[i]) for i in range(d0.nsrc)):
            return None
    if sum(d.ntaps for d in descs) > _lib.MAX_TAPS:
        return None
    # big grids are better off as separate launches (each becomes a persistent weight-resident launch when it qualifies): measured
    # layer by layer in r02 -- grouping wins below ~600 tiles per parity (one launch instead of four latency-bound ones), loses above
    if max(d.N * (-(-d.OH // 16)) * (-(-d.OW // 8)) for d in descs) > GROUP_PARITY_MAX_TILES:
        return None
    g = CisConv.from_buffer_copy(bytes(d0))
    g.MT, g.ey, g.ex = min(d.MT for d in descs), max(d.ey for d in descs), max(d.ex for d in descs)
    g.OH, g.OW = max(d.OH for d in descs), max(d.OW for d in descs)
    t = 0
    for i, d in enumerate(descs):
        for k in range(d.ntaps):
            g.dh[t + k], g.dw[t + k] = d.dh[k], d.dw[k]
        sb = g.sub[i]
        sb.tap0, sb.ntaps, sb.hoy, sb.hox, sb.OH, sb.OW, sb.oa, sb.ob, sb.wpack = t, d.ntaps, d.hoy, d.hox, d.OH, d.OW, d.oa, d.ob, d.wpack
        t += d.ntaps
    m_chunks = sum(g.src[i].chunks for i in range(g.nsrc))
    g.ntaps, g.nsub, g.splits, g.K_pad = t, len(descs), 0, ru(t * m_chunks * 8, 64)
    return g


class ParamStore(object):
    """One flat fp32 parameter buffer (+ grad, Adam m/v) per variable scope; names follow the TF variable layout
    (adversarial_learner.py:211-214 scopes 'MaskNet' / 'FlownetS'; model_pwcnet.py 'pwcnet')."""

    def __init__(self, device):
        self.device = device
        self.entries = []   # (name, shape, real_numel, offset, padded_numel)
        self.index = {}
        self.size = 0
        self.flat = None

    def declare(self, name, shape, padded=None):
        n = int(np.prod(shape))
        pn = ru(padded or n, 4)
        self.index[name] = len(self.entries)
        self.entries.append((name, tuple(shape), n, self.size, pn))
        self.size += pn

    def finalize(self, trainable):
        self.flat = torch.zeros(self.size, dtype=torch.float32, device=self.device)
        if trainable:
            self.grad = torch.zeros_like(self.flat)
            self.m = torch.zeros_like(self.flat)
            self.v = torch.zeros_like(self.flat)
            seg = [0]
            for _, _, n, off, _ in self.entries:
                seg.append(off + n)
            # segment i = [offset_i, offset_i + n_i): built as explicit (start,end) pairs flattened for the kernel
            self.seg_pairs = [(off, off + n) for _, _, n, off, _ in self.entries]

    def off(self, name):
        return self.entries[self.index[name]][3]

    def ptr(self, name, which='flat'):
        return getattr(self, which).data_ptr() + 4 * self.off(name)

    def view(self, name, which='flat'):
        _, shape, n, off, _ = self.entries[self.index[name]]
        return getattr(self, which)[off:off + n].view(shape)

    def load(self, params):
        for name, shape, n, off, _ in self.entries:
            if name not in params:
                raise KeyError('missing parameter ' + name)
            t = params[name].detach().to(torch.float32).reshape(-1)
            if t.numel() != n:
                raise ValueError('shape mismatch for %s: %d vs %d' % (name, t.numel(), n))
            self.flat[off:off + n].copy_(t)

    def export(self, which='flat'):
        return {name: getattr(self, which)[off:off + n].view(shape).clone() for name, shape, n, off, _ in self.entries}

    def real_count(self):
        return sum(e[2] for e in self.entries)


class ConvLayer(object):
    """One conv layer's static data: parameter views, packed bf16 operands (forward and data-gradient orientation),
    the fp32 packed weight-gradient buffer and the channel maps that tie packed K positions to HWIO indices."""

    def __init__(self, store, name, k, cin, cout, stride=1, dil=1, act=ACT_NONE, alpha=0.2, tag='', bn=False,
                 wname='kernel', bname='bias', transposed=False, bn_cap=None):
        self.store, self.name, self.k, self.cin, self.cout = store, name, k, cin, cout
        self.stride, self.dil, self.act, self.alpha, self.tag, self.bn = stride, dil, act, alpha, tag, bn
        self.transposed = transposed
        self.bn_cap = bn_cap
        self.BN, self.n_tiles = pick_bn(cout, bn_cap)
        self.npad = self.BN * self.n_tiles
        self.wkey, self.bkey = '%s/%s' % (name, wname), '%s/%s' % (name, bname)
        if transposed:
            store.declare(self.wkey, (k, k, cout, cin))
        else:
            store.declare(self.wkey, (k, k, cin, cout))
        store.declare(self.bkey, (cout,), padded=self.npad)
        if bn:
            store.declare('%s/gamma' % name, (cout,))
            store.declare('%s/beta' % name, (cout,))
        self.fwd_pack = None
        self.dgrad_packs = None
        self.device = store.device

    # ---- packed operands -------------------------------------------------------------------------------------
    def _kmap(self, taps_idx, chanmap, per_tap_stride, chan_stride):
        """kmap[k=(ti,pos)] = taps_idx[ti]*per_tap_stride + chanmap[pos]*chan_stride (or -1)."""
        m = len(chanmap)
        K = len(taps_idx) * m
        Kp = ru(max(K, (len(taps_idx) - 1) * m + ru(m, 64)), 64)   # halo kernel reads 64-channel chunks per tap
        km = np.full(Kp, -1, dtype=np.int32)
        cm = np.asarray(chanmap, dtype=np.int64)
        for ti, t in enumerate(taps_idx):
            v = np.where(cm >= 0, t * per_tap_stride + cm * chan_stride, -1)
            km[ti * m:(ti + 1) * m] = v
        return torch.from_numpy(km).to(self.device), Kp

    def setup_fwd(self, chanmap):
        """chanmap: packed input position -> original input channel (or -1)."""
        assert max(chanmap) == self.cin - 1, (self.name, max(chanmap), self.cin)
        self.in_chanmap = list(chanmap)
        kk = self.k * self.k
        if self.transposed:
            raise RuntimeError('use setup_transposed')
        kmap, Kp = self._kmap(range(kk), chanmap, self.cin * self.cout, self.cout)
        self.fwd_kmap, self.K_pad = kmap, Kp
        self.fwd_pack = torch.zeros(self.npad, Kp, dtype=torch.bfloat16, device=self.device)
        if self.bn:
            self.w_eff = torch.zeros(kk * self.cin * self.cout, dtype=torch.float32, device=self.device)
            self.b_eff = torch.zeros(self.npad, dtype=torch.float32, device=self.device)
            self.db_eff = torch.zeros(self.npad, dtype=torch.float32, device=self.device)

    def _alloc_tiles(self, ntaps, cin8, BN, n_tiles):
        nchunks = -(-cin8 // 64)
        return torch.zeros(n_tiles * nchunks * ntaps * BN * 64, dtype=torch.bfloat16, device=self.device)

    def _thin_tiles(self, items, tap_ids, chanmap, per_tap_stride, chan_stride, BN, n_tiles):
        """Compact-thin-halo operand (cis_pack_weights_tiled layout 1): one BN x 32 B tile per MMA of `items` (thin_items), its kmap
        (16 K positions per MMA: K half h = channels c_h .. c_h + 7 of tap tap_ids[i_h]) and the buffer."""
        km = np.full(len(items) * 16, -1, dtype=np.int32)
        for it, (_, _, h0, h1) in enumerate(items):
            for h, (t, c0) in enumerate((h0, h1)):
                if t < 0:
                    continue
                for e in range(8):
                    if c0 + e < len(chanmap) and chanmap[c0 + e] >= 0:
                        km[it * 16 + h * 8 + e] = tap_ids[t] * per_tap_stride + chanmap[c0 + e] * chan_stride
        return torch.from_numpy(km).to(self.device), torch.zeros(n_tiles * len(items) * BN * 16, dtype=torch.bfloat16, device=self.device)

    def fwd_tiles_buf(self, tap_order=None, items=None):
        """Pre-swizzled tile-major copy of the forward operand (halo kernel).  tap_order: the phase-major tap permutation of a
        stride-2 layer (setup_halo_s2); the tiles then follow that order.  items: the MMA list of a compact-thin-halo launch."""
        if getattr(self, 'fwd_tiles', None) is None:
            if items is not None:
                self.fwd_tiles_kmap, self.fwd_tiles = self._thin_tiles(items, range(self.k * self.k), self.in_chanmap, self.cin * self.cout,
                                                                       self.cout, self.BN, self.n_tiles)
            else:
                self.fwd_tiles = self._alloc_tiles(self.k * self.k, len(self.in_chanmap), self.BN, self.n_tiles)
                self.fwd_tiles_kmap = self.fwd_kmap
                if tap_order is not None:
                    self.fwd_tiles_kmap, _ = self._kmap(list(tap_order), self.in_chanmap, self.cin * self.cout, self.cout)
            self.fwd_tap_order, self.fwd_items = tap_order, items
        assert getattr(self, 'fwd_tap_order', None) == tap_order and getattr(self, 'fwd_items', None) == items, self.name
        return self.fwd_tiles

    def w_src_ptr(self):
        return self.w_eff.data_ptr() if self.bn else self.store.ptr(self.wkey)

    def bias_ptr(self):
        return self.b_eff.data_ptr() if self.bn else self.store.ptr(self.bkey)

    def plan_pack(self, plan, dgrad=False):
        """(Re)build the packed bf16 operands from the fp32 master weights."""
        s = self.store
        if self.bn:
            plan.add('cis_bn_fold', s.ptr(self.wkey), s.ptr(self.bkey), s.ptr(self.name + '/gamma'), s.ptr(self.name + '/beta'),
                     self.k * self.k * self.cin * self.cout, self.cout, self.w_eff.data_ptr(), self.b_eff.data_ptr())
        if self.fwd_pack is not None:
            if self.transposed:
                for pk in self.tr_packs:
                    if pk.get('wt') is not None and pk.get('items'):
                        plan.add('cis_pack_weights_tiled', self.w_src_ptr(), pk['tkmap'].data_ptr(), 16, len(pk['items']),
                                 self.n_tiles, self.BN, self.cout, self.cin, None, pk['wt'].data_ptr(), 1)
                    elif pk.get('wt') is not None:
                        plan.add('cis_pack_weights_tiled', self.w_src_ptr(), pk['kmap'].data_ptr(), len(self.in_chanmap), len(pk['taps']),
                                 self.n_tiles, self.BN, self.cout, self.cin, None, pk['wt'].data_ptr(), 0)
                    if pk.get('rows_used', True):
                        plan.add('cis_pack_weights', self.w_src_ptr(), pk['kmap'].data_ptr(), pk['K_pad'], self.npad, self.cout, self.cin,
                                 None, pk['w'].data_ptr())
            else:
                if getattr(self, 'fwd_tiles', None) is not None and self.fwd_items:
                    plan.add('cis_pack_weights_tiled', self.w_src_ptr(), self.fwd_tiles_kmap.data_ptr(), 16, len(self.fwd_items),
                             self.n_tiles, self.BN, self.cout, 1, None, self.fwd_tiles.data_ptr(), 1)
                elif getattr(self, 'fwd_tiles', None) is not None:
                    plan.add('cis_pack_weights_tiled', self.w_src_ptr(), self.fwd_tiles_kmap.data_ptr(), len(self.in_chanmap), self.k * self.k,
                             self.n_tiles, self.BN, self.cout, 1, None, self.fwd_tiles.data_ptr(), 0)
                if getattr(self, 'fwd_rows_used', True):
                    plan.add('cis_pack_weights', self.w_src_ptr(), self.fwd_kmap.data_ptr(), self.K_pad, self.npad, self.cout, 1,
                             None, self.fwd_pack.data_ptr())
        if dgrad and self.dgrad_packs:
            cout8 = ru(self.cout, 8)
            for pk in self.dgrad_packs:
                if pk.get('wt') is not None and pk.get('items'):
                    plan.add('cis_pack_weights_tiled', self.w_src_ptr(), pk['tkmap'].data_ptr(), 16, len(pk['items']), pk['n_tiles'], pk['BN'],
                             len(self.in_chanmap), self.cout, pk['nmap'].data_ptr(), pk['wt'].data_ptr(), 1)
                elif pk.get('wt') is not None:
                    plan.add('cis_pack_weights_tiled', self.w_src_ptr(), pk['kmap'].data_ptr(), cout8, len(pk['taps']), pk['n_tiles'], pk['BN'],
                             len(self.in_chanmap), self.cout, pk['nmap'].data_ptr(), pk['wt'].data_ptr(), 0)
                if pk.get('rows_used', True):
                    plan.add('cis_pack_weights', self.w_src_ptr(), pk['kmap'].data_ptr(), pk['K_pad'], pk['rows'], len(self.in_chanmap),
                             self.cout, pk['nmap'].data_ptr(), pk['w'].data_ptr())

    def plan_finalize(self, bp, mode):
        """Fixed-order sum of the private split-K slices of the packed fp32 weight gradient -> HWIO slot of the flat gradient
        buffer, same for the per-block bias-gradient partials (+ BN chain rule for the generator).  No atomics, nothing to zero."""
        if not hasattr(self, 'dwp') or mode not in getattr(self, 'wg_splits', {}):
            return
        s = self.store
        bp.add('cis_unpack_wgrad', self.dwp.data_ptr(), self.wg_kmap.data_ptr(), self.wg_K_pad, self.cout, self.wg_splits[mode],
               s.ptr(self.wkey, 'grad'), self.colpart.data_ptr(), self.col_blocks[mode], self.cout,
               (self.db_eff.data_ptr() if self.bn else s.ptr(self.bkey, 'grad')), 0 if self.wg_halo else 1)
        if self.bn:
            bp.add('cis_bn_chain', s.ptr(self.wkey), s.ptr(self.bkey), s.ptr(self.name + '/gamma'), s.ptr(self.wkey, 'grad'),
                   self.db_eff.data_ptr(), self.k * self.k * self.cin * self.cout, self.cout, s.ptr(self.bkey, 'grad'),
                   s.ptr(self.name + '/gamma', 'grad'), s.ptr(self.name + '/beta', 'grad'))

    # ---- tap tables ------------------------------------------------------------------------------------------
    def fwd_taps(self, H, W):
        pt, _ = same_pad(H, self.k, self.stride, self.dil)
        pl, _ = same_pad(W, self.k, self.stride, self.dil)
        return [(r * self.dil - pt, c * self.dil - pl) for r in range(self.k) for c in range(self.k)], pt, pl

    def setup_dgrad(self, H, W):
        """Packed weights for the data gradient on an input of size HxW: one launch for stride 1, four output-parity
        launches for stride 2 (each with the tap subset that lands on that parity)."""
        if self.dgrad_packs is not None:
            return
        _, pt, pl = self.fwd_taps(H, W)
        k, s, d = self.k, self.stride, self.dil
        g_chan = list(range(self.cout)) + [-1] * (ru(self.cout, 8) - self.cout)
        cin8 = len(self.in_chanmap)
        bn_, nt = pick_bn(cin8, self.bn_cap)
        rows = bn_ * nt
        nmap = torch.tensor(list(self.in_chanmap) + [-1] * (rows - cin8), dtype=torch.int32, device=self.device)
        packs = []
        for a in range(s):
            for b in range(s):
                tl, offs = [], []
                for r in range(k):
                    if (a + pt - r * d) % s:
                        continue
                    for c in range(k):
                        if (b + pl - c * d) % s:
                            continue
                        tl.append(r * k + c)
                        offs.append(((a + pt - r * d) // s, (b + pl - c * d) // s))
                # value = W[t, ci, co] -> flat (t*cin + ci)*cout + co ; K position (ti, co), row n = ci
                kmap, Kp = self._kmap(tl, g_chan, self.cin * self.cout, 1)
                packs.append(dict(a=a, b=b, taps=offs, tl=tl, chan=g_chan, kmap=kmap, K_pad=Kp, rows=rows, BN=bn_, n_tiles=nt, nmap=nmap,
                                  w=torch.zeros(rows, Kp, dtype=torch.bfloat16, device=self.device)))
        self.dgrad_packs = packs

    def setup_transposed(self, chanmap):
        """tf.layers.conv2d_transpose(k=4, s=2, 'same') as four output-parity stride-1 launches (model_pwcnet.py:286)."""
        assert self.transposed and self.k == 4
        self.in_chanmap = list(chanmap)
        packs = []
        for a in range(2):
            for b in range(2):
                tl, offs = [], []
                for ky in range(4):
                    if (a + 1 - ky) % 2:
                        continue
                    for kx in range(4):
                        if (b + 1 - kx) % 2:
                            continue
                        tl.append(ky * 4 + kx)
                        offs.append(((a + 1 - ky) // 2, (b + 1 - kx) // 2))
                # kernel [kh,kw,Cout,Cin]: flat ((t*Cout + co)*Cin + ci) ; K position (ti, ci), row n = co (stride Cin)
                kmap, Kp = self._kmap(tl, chanmap, self.cout * self.cin, 1)
                packs.append(dict(a=a, b=b, taps=offs, tl=tl, kmap=kmap, K_pad=Kp,
                                  w=torch.zeros(self.npad, Kp, dtype=torch.bfloat16, device=self.device)))
        self.tr_packs = packs
        self.fwd_pack = True


# ================================================================================================ graph builder
class Builder(object):
    """Builds the forward plan and records backward closures (reverse-mode, hand-scheduled)."""

    def __init__(self, device):
        self.device = device
        self.fwd = Plan('fwd')
        self.lane = 0        # lane given to forward launches (1 = side stream, see Plan.run)
        self.tape = []       # backward closures in forward order
        self.keep = []       # every buffer referenced by raw pointer from a descriptor must outlive the plans

    # ---- helpers
    def new_act(self, N, H, W, C, name='', dep=frozenset(), n_mod=0):
        a = Act(N, H, W, C, self.device, name=name, dep=dep, n_mod=n_mod)
        self.keep.append(a)
        return a

    def hold(self, obj):
        """Register a tensor / Act whose storage is referenced by raw pointer from a launch descriptor."""
        self.keep.append(obj)
        return obj

    def f32(self, *shape):
        return self.hold(torch.zeros(*shape, dtype=torch.float32, device=self.device))

    def conv(self, layer, srcs, out=None, post_add=None, addf=None, outf=None, outf_ch=0, mode=0, want_bf16=True, name=None,
             plan=None, out_rows=None):
        """y = act(conv(concat(srcs)) + bias [+ addf]) [+ post_add]; returns the output Act."""
        plan = plan or self.fwd
        if MATERIALIZE_MISALIGNED_CONCAT and len(srcs) > 1 and layer.tag and layer.stride == 1 and \
                any(s.C8 % 64 for s in srcs[:-1]):
            srcs = [self.concat(srcs, name=layer.name + '.cat')]
        s0 = srcs[0]
        N = out_rows or max(s.N for s in srcs)
        H, W = s0.H, s0.W
        for s in srcs:
            assert (s.H, s.W) == (H, W), (layer.name, [(q.H, q.W) for q in srcs])
        chanmap = []
        base = 0
        for s in srcs:
            chanmap += [(m + base if m >= 0 else -1) for m in s.chanmap]
            base += s.C
        if layer.fwd_pack is None:
            layer.setup_fwd(chanmap)
        else:
            assert layer.in_chanmap == chanmap, layer.name
        OH, OW = -(-H // layer.stride), -(-W // layer.stride)
        dep = frozenset().union(*[s.dep for s in srcs]) | ({layer.tag} if layer.tag else frozenset())
        if post_add is not None:
            dep = dep | post_add.dep
        if out is None and want_bf16:
            out = self.new_act(N, OH, OW, layer.cout, name=name or layer.name, dep=dep)
        if out is not None:
            out.dep = out.dep | dep
            gr = [s.gen_rows for s in srcs if s.gen_rows]
            if gr:
                out.gen_rows = gr[0]
        taps, _, _ = layer.fwd_taps(H, W)
        d = CisConv()
        d.N, d.H, d.W, d.OH, d.OW, d.sh, d.sw = N, H, W, OH, OW, layer.stride, layer.stride
        _fill_taps(d, taps)
        _fill_srcs(d, srcs)
        d.wpack, d.K_pad, d.BN, d.n_tiles = layer.fwd_pack.data_ptr(), layer.K_pad, layer.BN, layer.n_tiles
        d.bias, d.act, d.alpha = layer.bias_ptr(), layer.act, layer.alpha
        d.DH, d.DW, d.osh, d.osw, d.oa, d.ob = OH, OW, 1, 1, 0, 0
        if out is not None:
            d.out, d.out_pitch, d.out_coff, d.out_ch = out.ptr, out.pitch, out.c_off, out.C8
        if outf is not None:
            d.outf, d.outf_pitch, d.outf_coff, d.outf_ch = outf.data_ptr(), outf.shape[-1], 0, outf_ch or outf.shape[-1]
        if addf is not None:
            d.addf_pre, d.addf_pitch, d.addf_coff = addf.data_ptr(), addf.shape[-1], 0
            if outf is None:
                d.outf_ch = addf.shape[-1]
        if post_add is not None:
            d.add_post, d.add_post_pitch, d.add_post_coff = post_add.ptr, post_add.pitch, post_add.c_off
        d.mode = mode
        order = setup_halo_s2(d, taps, layer.n_tiles) if (layer.stride == 2 and layer.dil == 1) else None
        hl = layer.stride == 1 and order is None and setup_halo(d, taps, layer.dil, layer.n_tiles)
        if order is not None:
            d.wpack = layer.fwd_tiles_buf(order, getattr(d, 'thin_items', None)).data_ptr()
            layer.fwd_rows_used = getattr(layer, 'fwd_rows_used', False)
        elif hl:
            d.wpack = layer.fwd_tiles_buf(None, hl if hl is not True else None).data_ptr()
            layer.fwd_rows_used = getattr(layer, 'fwd_rows_used', False)
        else:
            layer.fwd_rows_used = True
        setup_splitk(d, self.device, plan.keep)
        plan.keep.append(d)
        plan.keep += [srcs, out, outf, addf, post_add, layer]
        plan.add('cis_conv_igemm', C.byref(d), flops=2.0 * N * OH * OW * layer.k * layer.k * layer.cin * layer.cout, lane=self.lane)
        if layer.tag:
            self.tape.append(lambda bp, m, L=layer, S=list(srcs), O=out, P=post_add: self._conv_bwd(bp, m, L, S, O, P))
        return out

    def _conv_bwd(self, bp, mode, layer, srcs, out, post_add):
        if out is None or mode not in out.dep or not out.grad_written.get(mode):
            return
        G = out.get_grad()
        nb = out.rows(mode)
        npix = nb * out.H * out.W
        if post_add is not None and mode in post_add.dep:
            pg = post_add.get_grad()
            bp.add('cis_add_slice', pg.ptr, pg.pitch, pg.c_off, G.ptr, G.pitch, G.c_off, npix, G.C8 // 8, 1,
                   1 if post_add.grad_written.get(mode) else 0)
            post_add.grad_written[mode] = True
        if layer.tag == mode:
            chunks = -(-layer.cout // 8)
            ppb = (256 // chunks) * COLSUM_PIX                      # pixels per colsum block (P pixel lanes x COLSUM_PIX pixels each)
            if not hasattr(layer, 'col_blocks'):
                layer.col_blocks = {}
            layer.col_blocks[mode] = max(1, min(592, -(-npix // ppb)))
            if getattr(layer, 'colpart', None) is None:
                layer.colpart = torch.empty(592 * layer.cout, dtype=torch.float32, device=self.device)
        res = (post_add.ptr, post_add.pitch, post_add.c_off) if post_add is not None else (None, 0, 0)
        fused_colsum = bool(DACT_COLSUM and layer.act != ACT_NONE and layer.tag == mode)
        if fused_colsum:      # activation derivative + bias-gradient partials in one pass over the gradient
            bp.add('cis_dact_colsum', G.ptr, G.pitch, G.c_off, out.ptr, out.pitch, out.c_off, res[0], res[1], res[2], npix, layer.cout,
                   layer.act, layer.alpha, layer.colpart.data_ptr(), layer.col_blocks[mode])
        elif layer.act != ACT_NONE:
            bp.add('cis_dact_mul', G.ptr, G.pitch, G.c_off, out.ptr, out.pitch, out.c_off, res[0], res[1], res[2], npix, G.C8 // 8,
                   layer.act, layer.alpha)
        s0 = srcs[0]
        H, W = s0.H, s0.W
        taps, _, _ = layer.fwd_taps(H, W)
        if layer.tag == mode:   # weight + bias gradients
            if not hasattr(layer, 'dwp'):
                # TMA operand path (8x8 pixel tiles) for stride-1 layers whose concat sources are 64-channel aligned
                layer.wg_tma = bool(WGRAD_TMA and layer.stride == 1 and len(layer.in_chanmap) >= 32 and
                                    all(s_.C8 % 64 == 0 for s_ in srcs[:-1]))   # thin inputs: per-tap 64-channel padding would waste the loads
                # (thin inputs are excluded like for the TMA path: every tap is padded to a 64-channel column group there)
                layer.wg_halo = bool(WGRAD_HALO and len(layer.in_chanmap) >= WGRAD_HALO_MIN_CH and wgrad_halo_fits(taps, layer.cout, layer.stride) and
                                     all(s_.C8 % 64 == 0 for s_ in srcs[:-1]))
                if layer.wg_tma or layer.wg_halo:
                    cin8 = len(layer.in_chanmap)
                    nch64 = -(-cin8 // 64)
                    ncol = layer.k * layer.k * nch64 * 64
                    layer.wg_K_pad = ru(ncol, 128)
                    km = np.full(layer.wg_K_pad, -1, dtype=np.int32)
                    fk = layer.fwd_kmap.cpu().numpy()
                    for t in range(layer.k * layer.k):
                        for pos in range(cin8):
                            km[(t * nch64 + pos // 64) * 64 + pos % 64] = fk[t * cin8 + pos]
                    layer.wg_kmap = torch.from_numpy(km).to(self.device)
                else:
                    layer.wg_K_pad, layer.wg_kmap = layer.K_pad, layer.fwd_kmap
                layer.dwp, layer.wg_splits = None, {}
            w = CisWgrad()
            w.N, w.H, w.W, w.OH, w.OW, w.sh, w.sw = nb, H, W, out.H, out.W, layer.stride, layer.stride
            _fill_taps(w, taps)
            _fill_srcs(w, srcs)
            w.g, w.g_pitch, w.g_coff, w.g_chunks = G.ptr, G.pitch, G.c_off, G.C8 // 8
            w.Cout, w.K_pad = layer.cout, layer.wg_K_pad
            w.tma = 2 if layer.wg_halo else (1 if layer.wg_tma else 0)
            nkb = (nb * (-(-out.H // 8)) * (-(-out.W // 8))) if w.tma else -(-npix // 64)
            ntile = -(-layer.wg_K_pad // 128)
            if w.tma == 2:      # grid.x = 64-channel chunks of the input, grid.z = 64-channel halves of Cout
                ntile = (-(-len(layer.in_chanmap) // 64)) * (2 if layer.cout > 64 else 1)
            splits = max(1, min(nkb // 8 if nkb >= 8 else 1, max(1, (WGRAD_CTAS_PER_SM * NUM_SMS) // ntile)))
            if WGRAD_MAX_SLICE_MB > 0:      # the private slices are written once and read once more by the un-pack job: bound their volume
                splits = max(1, min(splits, int(WGRAD_MAX_SLICE_MB * 1e6 / (layer.cout * layer.wg_K_pad * 4.0))))
            splits = -(-nkb // (-(-nkb // splits)))        # every split owns >= 1 reduction block (its slice is written, not accumulated)
            w.splits = splits
            layer.wg_splits[mode] = splits
            if layer.dwp is None or layer.dwp.numel() < splits * layer.cout * layer.wg_K_pad:
                assert not getattr(layer, 'wgrad_modes', None), 'slice buffer must be sized by the first (largest) mode'
                layer.dwp = torch.empty(max(layer.wg_splits.values()) * layer.cout * layer.wg_K_pad, dtype=torch.float32, device=self.device)
            w.dwp = layer.dwp.data_ptr()
            bp.keep.append(w)
            bp.add('cis_conv_wgrad', C.byref(w), flops=2.0 * npix * layer.k * layer.k * layer.cin * layer.cout, lane=1)
            layer.wgrad_modes = getattr(layer, 'wgrad_modes', set()) | {mode}
            if not fused_colsum:
                bp.add('cis_colsum', G.ptr, G.pitch, G.c_off, npix, layer.cout, layer.colpart.data_ptr(), layer.col_blocks[mode], lane=1)
        need = [s for s in srcs if mode in s.dep]
        if not need:
            return
        layer.setup_dgrad(H, W)
        layer.dgrad_used = True
        cin8 = len(layer.in_chanmap)
        single = (len(srcs) == 1 and srcs[0].n_mod == 0)
        if single:
            tgt = srcs[0].get_grad()
            acc = bool(srcs[0].grad_written.get(mode))
        else:
            if not hasattr(layer, 'dcat'):
                layer.dcat = Act(max(s.N for s in srcs), H, W, cin8, self.device, chanmap=layer.in_chanmap, name=layer.name + '.dcat')
            tgt, acc = layer.dcat, False
        emitted = []
        for pk in layer.dgrad_packs:
            s = layer.stride
            oh = -(-(H - pk['a']) // s)
            ow = -(-(W - pk['b']) // s)
            if oh <= 0 or ow <= 0:
                continue
            d = CisConv()
            d.N, d.H, d.W, d.OH, d.OW, d.sh, d.sw = nb, out.H, out.W, oh, ow, 1, 1
            _fill_taps(d, pk['taps'])
            d.nsrc = 1
            d.src[0] = G.src()
            d.wpack, d.K_pad, d.BN, d.n_tiles = pk['w'].data_ptr(), pk['K_pad'], pk['BN'], pk['n_tiles']
            d.bias, d.act = None, ACT_NONE
            d.DH, d.DW, d.osh, d.osw, d.oa, d.ob = H, W, s, s, pk['a'], pk['b']
            d.out, d.out_pitch, d.out_coff, d.out_ch = tgt.ptr, tgt.pitch, tgt.c_off, tgt.C8
            if acc:
                d.add_pre, d.add_pre_pitch, d.add_pre_coff = tgt.ptr, tgt.pitch, tgt.c_off
            hl = setup_halo(d, pk['taps'], layer.dil if s == 1 else 1, pk['n_tiles'])
            if hl:
                items = hl if hl is not True else None
                if pk.get('wt') is None:
                    pk['items'] = items
                    if items:
                        pk['tkmap'], pk['wt'] = layer._thin_tiles(items, pk['tl'], pk['chan'], layer.cin * layer.cout, 1, pk['BN'], pk['n_tiles'])
                    else:
                        pk['wt'] = layer._alloc_tiles(len(pk['taps']), ru(layer.cout, 8), pk['BN'], pk['n_tiles'])
                assert pk['items'] == items, layer.name
                d.wpack = pk['wt'].data_ptr()
                pk['rows_used'] = pk.get('rows_used', False)
            else:
                pk['rows_used'] = True
            emitted.append((d, 2.0 * nb * oh * ow * len(pk['taps']) * layer.cin * layer.cout))
        grp = merge_parity_launches([d for d, _ in emitted]) if len(emitted) > 1 else None
        if grp is not None:
            bp.keep.append(grp)
            bp.add('cis_conv_igemm', C.byref(grp), flops=sum(f for _, f in emitted))
        else:
            for d, fl in emitted:
                setup_splitk(d, self.device, bp.keep)
                bp.keep.append(d)
                bp.add('cis_conv_igemm', C.byref(d), flops=fl)
        if single:
            srcs[0].grad_written[mode] = True
        else:
            # gradient of the virtual concat -> the sources' gradient slices, ONE launch (same-size case of the fused resize-concat
            # transpose: slices the channels, folds the replicas of batch-broadcast sources, accumulates where a gradient exists)
            want = [1 if mode in s_.dep else 0 for s_ in srcs]
            garr, acc = [], []
            for s_, w_ in zip(srcs, want):
                if w_:
                    sg = s_.get_grad()
                    garr.append(CisSrc(sg.ptr, sg.pitch, sg.c_off, s_.C8 // 8, s_.n_mod))
                    acc.append(1 if s_.grad_written.get(mode) else 0)
                    s_.grad_written[mode] = True
                else:
                    garr.append(CisSrc(None, 8, 0, s_.C8 // 8, s_.n_mod))
                    acc.append(0)
            ga = (CisSrc * len(srcs))(*garr)
            wa, aa = (C.c_int32 * len(srcs))(*want), (C.c_int32 * len(srcs))(*acc)
            bp.keep += [ga, wa, aa]
            bp.add('cis_resize_concat_bf16_bwd', tgt.ptr, tgt.pitch, 0, nb, H, W, ga, wa, aa, len(srcs), H, W)

    # ---- fused resize + concat: ONE launch brings up to 4 same-resolution sources (batch-broadcast ones included) to OH x OW and lays
    # them side by side in one buffer, ONE launch takes the gradient back (folding the broadcast replicas); replaces a resize launch
    # per source plus a copy per source and replica (recover decoder: `deconv` inputs, nets.py:80-104; misaligned virtual concats)
    def resize_concat(self, srcs, OH=None, OW=None, name='cat'):
        srcs = list(srcs)
        assert 1 <= len(srcs) <= 4
        N = max(s.N for s in srcs)
        H, W = srcs[0].H, srcs[0].W
        OH, OW = OH or H, OW or W
        for s in srcs:
            assert (s.H, s.W) == (H, W) and (s.n_mod == 0 or N % s.n_mod == 0)
        chanmap, base = [], 0
        for s in srcs:
            chanmap += [(m + base if m >= 0 else -1) for m in s.chanmap]
            base += s.C
        dep = frozenset().union(*[s.dep for s in srcs])
        cat = Act(N, OH, OW, base, self.device, chanmap=chanmap, dep=dep, name=name)
        gr = [s.gen_rows for s in srcs if s.gen_rows]
        if gr:
            cat.gen_rows = gr[0]
        arr = (CisSrc * len(srcs))(*[s.src() for s in srcs])
        self.keep += [srcs, cat, arr]
        self.fwd.add('cis_resize_concat_bf16', arr, len(srcs), N, H, W, cat.ptr, cat.pitch, cat.c_off, OH, OW, lane=self.lane)

        def bwd(bp, mode):
            if mode not in cat.dep or not cat.grad_written.get(mode):
                return
            g = cat.get_grad()
            nb = cat.rows(mode)
            want = [1 if mode in s_.dep else 0 for s_ in srcs]
            if not any(want):
                return
            garr, acc = [], []
            for s_, w_ in zip(srcs, want):
                if w_:
                    sg = s_.get_grad()
                    garr.append(CisSrc(sg.ptr, sg.pitch, sg.c_off, s_.C8 // 8, s_.n_mod))
                    acc.append(1 if s_.grad_written.get(mode) else 0)
                    s_.grad_written[mode] = True
                else:
                    garr.append(CisSrc(None, 8, 0, s_.C8 // 8, s_.n_mod))
                    acc.append(0)
            ga = (CisSrc * len(srcs))(*garr)
            wa, aa = (C.c_int32 * len(srcs))(*want), (C.c_int32 * len(srcs))(*acc)
            bp.keep += [ga, wa, aa]
            bp.add('cis_resize_concat_bf16_bwd', g.ptr, g.pitch, g.c_off, nb, OH, OW, ga, wa, aa, len(srcs), H, W)
        self.tape.append(bwd)
        return cat

    def concat(self, srcs, name='cat'):
        """Materialised concat (only where the virtual concat is not 64-channel aligned, so the TMA operand paths apply)."""
        return self.resize_concat(srcs, name=name)

    # ---- transposed conv (PWC-Net up_flow / up_feat), forward only
    def conv_transpose(self, layer, src, out=None, outf=None, plan=None, name=None):
        plan = plan or self.fwd
        if layer.fwd_pack is None:
            layer.setup_transposed(src.chanmap)
        N, H, W = src.N, src.H, src.W
        if out is None:
            out = self.new_act(N, 2 * H, 2 * W, layer.cout, name=name or layer.name, dep=src.dep)
        emitted = []
        for pk in layer.tr_packs:
            d = CisConv()
            d.N, d.H, d.W, d.OH, d.OW, d.sh, d.sw = N, H, W, H, W, 1, 1
            _fill_taps(d, pk['taps'])
            _fill_srcs(d, [src])
            d.wpack, d.K_pad, d.BN, d.n_tiles = pk['w'].data_ptr(), pk['K_pad'], layer.BN, layer.n_tiles
            d.bias, d.act = layer.bias_ptr(), ACT_NONE
            d.DH, d.DW, d.osh, d.osw, d.oa, d.ob = 2 * H, 2 * W, 2, 2, pk['a'], pk['b']
            d.out, d.out_pitch, d.out_coff, d.out_ch = out.ptr, out.pitch, out.c_off, layer.cout
            if outf is not None:
                d.outf, d.outf_pitch, d.outf_coff, d.outf_ch = outf.data_ptr(), outf.shape[-1], 0, layer.cout
            hl = setup_halo(d, pk['taps'], 1, layer.n_tiles)
            if hl:
                items = hl if hl is not True else None
                if pk.get('wt') is None:
                    pk['items'] = items
                    if items:
                        pk['tkmap'], pk['wt'] = layer._thin_tiles(items, pk['tl'], layer.in_chanmap, layer.cout * layer.cin, 1, layer.BN,
                                                                  layer.n_tiles)
                    else:
                        pk['wt'] = layer._alloc_tiles(len(pk['taps']), len(layer.in_chanmap), layer.BN, layer.n_tiles)
                assert pk['items'] == items, layer.name
                d.wpack = pk['wt'].data_ptr()
                pk['rows_used'] = pk.get('rows_used', False)
            else:
                pk['rows_used'] = True
            plan.keep += [src, out, outf, layer]
            emitted.append((d, 2.0 * N * H * W * len(pk['taps']) * layer.cin * layer.cout))
        grp = merge_parity_launches([d for d, _ in emitted])
        if grp is not None:
            plan.keep.append(grp)
            plan.add('cis_conv_igemm', C.byref(grp), flops=sum(f for _, f in emitted), lane=self.lane)
        else:
            for d, fl in emitted:
                setup_splitk(d, self.device, plan.keep)
                plan.keep.append(d)
                plan.add('cis_conv_igemm', C.byref(d), flops=fl)
        return out

    # ---- resampling ops
    def resize_bilinear(self, src, OH, OW, name=''):
        """tf.image.resize_images legacy bilinear (convolution_utils.py:88); identity when the size matches."""
        if (src.H, src.W) == (OH, OW):
            return src
        out = Act(src.N, OH, OW, src.C, self.device, chanmap=src.chanmap, n_mod=src.n_mod, dep=src.dep, name=name or src.name + '.rs')
        out.gen_rows = src.gen_rows
        self.keep += [src, out]
        self.fwd.add('cis_resize_bilinear_bf16', src.ptr, src.pitch, src.c_off, src.N, src.H, src.W, out.ptr, out.pitch, out.c_off, OH, OW,
                     src.C8 // 8)

        def bwd(bp, mode):
            if mode not in out.dep or not out.grad_written.get(mode):
                return
            g, sg = out.get_grad(), src.get_grad()
            bp.add('cis_resize_bilinear_bf16_bwd', g.ptr, g.pitch, g.c_off, out.rows(mode), OH, OW, sg.ptr, sg.pitch, sg.c_off, src.H, src.W,
                   src.C8 // 8, 1 if src.grad_written.get(mode) else 0)
            src.grad_written[mode] = True
        self.tape.append(bwd)
        return out

    def upsample_nn2x(self, src, name=''):
        """tf.image.resize_nearest_neighbor(align_corners=True) x2 (convolution_utils.py:71)."""
        assert src.c_off == 0 and src.pitch == src.C8
        out = Act(src.N, 2 * src.H, 2 * src.W, src.C, self.device, chanmap=src.chanmap, dep=src.dep, name=name or src.name + '.up')
        self.keep += [src, out]
        self.fwd.add('cis_upsample_nn2x', src.ptr, src.N, src.H, src.W, src.pitch, out.ptr)

        def bwd(bp, mode):
            if mode not in out.dep or not out.grad_written.get(mode):
                return
            g, sg = out.get_grad(), src.get_grad()
            bp.add('cis_upsample_nn2x_bwd', g.ptr, src.N, src.H, src.W, src.pitch, sg.ptr, 1 if src.grad_written.get(mode) else 0)
            src.grad_written[mode] = True
        self.tape.append(bwd)
        return out

    def build_backward(self, mode, seeds):
        """seeds: Acts whose .grad has been written by the loss backward.  Returns the backward Plan for `mode`."""
        bp = Plan('bwd_' + mode)
        for a in seeds:
            a.grad_written[mode] = True
        for fn in reversed(self.tape):
            fn(bp, mode)
        return bp
