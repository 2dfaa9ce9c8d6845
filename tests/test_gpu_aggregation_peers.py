"""The aggregation kernels of csrc/fedavg.cu at 2 to 8 ranks on ONE GPU, against a float64 reference.

K2 (``fedavg_round_kernel``), K3 (``small_allreduce_kernel``) and the fused GLM tail (``glm_aggregate_update_kernel``)
only see raw pointers: every rank's buffers and signal pad arrive as a ``PeerTable``.  So one process can play a whole
federation.  ``SymmetricHeap`` is replaced by an emulation in which every rank owns ordinary device tensors and every
rank's ``peer_ptrs`` name all ranks' tensors; the ranks then launch one after another on one stream.  Before rank r
launches, the flags that the ranks still to come would raise in r's pad are raised for them, so every wait succeeds at
its first poll.  The reducer slices are disjoint (sharded) or there is a single reducer (central), so reducer r reads
its slice of every upload before any other kernel writes that slice: the sequential run computes exactly what the
concurrent one does.  The real engine code runs: ``slice_bounds``, ``_reshard``, ``mark_dead``, the argument plumbing
of ``fedavg_round`` and every template instantiation of the kernel (WMAX = 2, 4, 8).

What this cannot check, and what stays with ``dist_comm_check.py`` under torchrun on several GPUs:
* multicast: ``multimem.ld_reduce`` / ``multimem.st`` and the ``s_use_mc`` branch need a multicast object over at
  least 2 GPUs (the emulated heap hands out none, so every round here takes the P2P path);
* cross-GPU memory ordering: the ranks run in stream order, so a missing fence cannot show;
* K1 (``bcast_push_gemm_bf16``).

Every check compares with a float64 evaluation of the documented formulas (``reference_round``), within a bound
derived from the number of fp32 operations per element; elements that must not be read hold NaN, elements that must
not be written hold a sentinel bit pattern and are compared bit for bit.
"""
from __future__ import annotations

import functools
import itertools
import struct

import numpy as np
import pytest
import torch

from vantage6_b200.parallel import fedavg as fedavg_mod
from vantage6_b200.parallel.fedavg import UPLOAD_MODES, FedAvgEngine, ServerOptConfig, SmallAggregator
from vantage6_b200.parallel.symm import PAD_WORDS, SymmBuffer

# signal-pad words (csrc/api.h)
PAD_UPLOAD, PAD_BCAST, PAD_SMALL, PAD_STATUS, PAD_MISSING, PAD_NI, PAD_RFAIL, PAD_RMISS = 0, 32, 96, 129, 130, 136, 144, 152
# A flag the harness raises for a rank that has not launched yet holds epoch + RAISED: the kernels wait for >= epoch,
# and the owner's kernel later stores exactly the epoch.  So a flag equal to the epoch after a round was stored by a kernel.
RAISED = 1 << 16
# NaN bit patterns: poison when an element that must not be read is read, and proof that an element that must not be
# written was not (compared as integers, since NaN != NaN)
SENT32, SENT16 = 0x7FC0DEAD, 0x7FC1
U = 2.0 ** -24
N8 = [3.0, 1.5, 7.0, 2.0, 5.0, 0.25, 11.0, 4.0]           # unequal sample counts, exact in fp32
LR = {"fedavg": 0.7, "fedavgm": 0.5, "fedadam": 0.05}
DEV = "cuda:0"


def _f32(x: float) -> float:
    return float(np.float32(x))


def _f32_bits(x: float) -> int:
    return struct.unpack("<i", struct.pack("<f", x))[0]


def _ints(t: torch.Tensor) -> torch.Tensor:
    return t.view(torch.int16 if t.element_size() == 2 else torch.int32)


def _poison(t: torch.Tensor) -> None:
    _ints(t).fill_(SENT16 if t.element_size() == 2 else SENT32)


def _is_sentinel(t: torch.Tensor) -> bool:
    return bool((_ints(t) == (SENT16 if t.element_size() == 2 else SENT32)).all())


def assert_within(name: str, got: torch.Tensor, want: torch.Tensor, tol: torch.Tensor) -> None:
    got = got.double()
    bad = ~((got - want).abs() <= tol)                    # NaN counts as outside
    if bool(bad.any()):
        i = int(bad.nonzero()[0, 0])
        raise AssertionError(f"{name}: {int(bad.sum())} of {bad.numel()} elements outside the bound; first at [{i}]: "
                             f"got {got[i].item()!r}, want {want[i].item()!r} +- {tol[i].item():.3g}")


# ---------------------------------------------------------------------------------------------------- float64 reference
def reference_round(xs, n, *, prescaled: bool, delta: bool, opt: ServerOptConfig, t: int, wg, m, v) -> dict:
    """One FedAvg server round in float64 over the whole vector, as ``parallel/fedavg.py`` documents it, and the bound
    on what an fp32 evaluation of the same formulas may deviate from it, per element.

    ``xs[p]``: rank p's upload (ignored when ``n[p] == 0``); ``n``: the sample counts (0 = not reporting); ``wg, m, v``:
    the server state at the start of the round; ``t``: the server step the bias corrections use.  The optimizer's
    scalars enter as the fp32 values the kernel receives."""
    lr, b1, b2, eps = _f32(opt.lr), _f32(opt.beta1), _f32(opt.beta2), _f32(opt.eps)
    bias1, bias2 = _f32(1.0 / (1.0 - opt.beta1 ** t)), _f32(1.0 / (1.0 - opt.beta2 ** t))
    rep = [p for p in range(len(n)) if n[p] > 0]
    tot = float(sum(n[p] for p in rep))
    terms = [xs[p] if prescaled else n[p] * xs[p] for p in rep]
    mean = sum(terms) / tot
    S = sum(x.abs() for x in terms) / tot
    d = mean if delta else mean - wg
    # Error bound, to first order.  An fp32 rounding errs by at most 2^-24 of its result; the extension is built with
    # --use_fast_math, so 1/x, a/b and sqrtf are approximate (MUFU.RCP / MUFU.SQRT, within 2 ulp) and every operation
    # below counts u = 2^-23.  With W reporting ranks and S = sum_p |n_p x_p| / sum_p n_p:
    #   mean     W fmaf over the contributors, sum of the n_p, 1/sum, the final multiply   e_mean <= (2W + 2) u S
    #   d        minus w_global in weights_f32 mode                                        e_d = e_mean + u |d|
    #   FedAvg   w' = fmaf(lr, d, w)                                                       e_w = lr e_d + u |w'|
    #   FedAvgM  m' = fmaf(b1, m, d),  w' = fmaf(lr, m', w)      e_m = e_d + u |m'|,       e_w = lr e_m + u |w'|
    #   FedAdam  m' = b1 m + (1-b1) d                            e_m = (1-b1) e_d + 2u (b1 |m| + (1-b1) |d|)
    #            v' = b2 v + (1-b2) d d                          e_v = 2 (1-b2) |d| e_d + 3u (b2 v + (1-b2) d^2)
    #            w' = w + lr (m' bias1) / (sqrt(v' bias2) + eps), propagated term by term below
    # The tolerance is twice the bound (second-order terms; the compiler's freedom to contract a*b+c).
    u = 2 * U
    e_d = (2 * len(rep) + 2) * u * S + u * d.abs()
    m1, v1, e_m, e_v = m, v, torch.zeros_like(d), torch.zeros_like(d)
    if opt.name == "fedavg":
        w1 = wg + lr * d
        e_w = lr * e_d + u * w1.abs()
    elif opt.name == "fedavgm":
        m1 = b1 * m + d
        e_m = e_d + u * m1.abs()
        w1 = wg + lr * m1
        e_w = lr * e_m + u * w1.abs()
    else:
        m1 = b1 * m + (1 - b1) * d
        v1 = b2 * v + (1 - b2) * d * d
        e_m = (1 - b1) * e_d + 2 * u * (b1 * m.abs() + (1 - b1) * d.abs())
        e_v = 2 * (1 - b2) * d.abs() * e_d + 3 * u * (b2 * v + (1 - b2) * d * d)
        mh, vh = m1 * bias1, v1 * bias2
        e_mh, e_vh = bias1 * e_m + u * mh.abs(), bias2 * e_v + u * vh
        s = vh.sqrt()
        e_s = torch.minimum(e_vh / (2 * s).clamp_min(1e-300), e_vh.sqrt()) + u * s      # sqrt is 1/2-Hoelder near 0
        D = s + eps
        q = mh / D
        e_q = e_mh / D + mh.abs() * (e_s + u * D) / (D * D) + u * q.abs()
        w1 = wg + lr * q
        e_w = lr * e_q + u * w1.abs()
    floor = 1e-37                                            # below the fp32 normal range (the kernels flush denormals)
    return dict(w=w1, m=m1, v=v1, tol_w=2 * e_w + floor, tol_m=2 * e_m + floor, tol_v=2 * e_v + floor)


@pytest.mark.parametrize("upload", UPLOAD_MODES)
@pytest.mark.parametrize("opt", ["fedavg", "fedavgm", "fedadam"])
def test_reference_matches_collective_plane_world1(opt, upload):
    """The float64 reference and its bound against the CPU collective plane (plain torch fp32 math) of one rank."""
    torch.manual_seed(5)
    n = 1003
    e = FedAvgEngine(n, 0, 1, "cpu", data_plane="collective", server_opt=ServerOptConfig(opt, LR[opt]), upload=upload)
    e.w.copy_(torch.randn(e.n))
    e.initialize_global()
    torch.testing.assert_close(e.w_global, e.w, rtol=0, atol=0)
    for rnd in range(3):
        prescaled = upload != "weights_f32" and rnd == 2
        wg, m, v = e.w_global.double(), e.opt_m.double(), e.opt_v.double()
        if upload == "weights_f32":
            e.w.add_(0.1 * torch.randn(e.n))
        else:
            e.upload.copy_((0.1 * torch.randn(e.n) * (5.0 if prescaled else 1.0)).to(e.upload.dtype))
        xs = [e.upload.double()]
        e.aggregate([5.0], prescaled=prescaled)
        if opt == "fedavg":
            m = v = torch.zeros(e.n, dtype=torch.float64)
        ref = reference_round(xs, [5.0], prescaled=prescaled, delta=upload != "weights_f32", opt=e.opt, t=e.server_step,
                              wg=wg, m=m, v=v)
        assert_within(f"round {rnd} w_global", e.w_global, ref["w"], ref["tol_w"])
        if opt != "fedavg":
            assert_within(f"round {rnd} m", e.opt_m, ref["m"], ref["tol_m"])
        if opt == "fedadam":
            assert_within(f"round {rnd} v", e.opt_v, ref["v"], ref["tol_v"])
        assert torch.equal(e.w, e.w_global)


def test_reference_bound_is_tight_enough_to_see_one_wrong_weight():
    """The bound is not so loose that a plausible slip passes: off-by-one-rank weights move the mean far outside it."""
    torch.manual_seed(6)
    xs = [torch.randn(4096, dtype=torch.float64) for _ in range(5)]
    z = torch.zeros(4096, dtype=torch.float64)
    for name in ("fedavg", "fedavgm", "fedadam"):
        opt = ServerOptConfig(name, LR[name])
        ref = reference_round(xs, N8[:5], prescaled=False, delta=True, opt=opt, t=1, wg=z, m=z, v=z)
        bad = reference_round(xs, N8[:4] + [N8[0]], prescaled=False, delta=True, opt=opt, t=1, wg=z, m=z, v=z)
        assert float(((bad["w"] - ref["w"]).abs() > ref["tol_w"]).double().mean()) > 0.9, name


# ---------------------------------------------------------------------------------------------------- emulated heap
class _Fabric:
    """The memory of one emulated federation: allocation k of every rank, created when the first rank asks for it."""

    def __init__(self, world: int):
        self.world = world
        self.allocs: list = []

    def get(self, k: int, nbytes: int) -> list:
        if k == len(self.allocs):
            self.allocs.append([torch.zeros(nbytes, dtype=torch.uint8, device=DEV) for _ in range(self.world)])
        bufs = self.allocs[k]
        assert bufs[0].numel() == nbytes, "the ranks of one federation must allocate the same sizes in the same order"
        return bufs


class _EmulatedHeap:
    """Stands in for ``SymmetricHeap``: rank r's k-th ``alloc`` returns its own zeroed tensor of allocation k, with the
    device addresses of all ranks' tensors of allocation k as ``peer_ptrs`` and no multicast address."""

    def __init__(self, fabric: _Fabric, rank: int, world: int, device=None, *args, **kwargs):
        assert world == fabric.world
        self.fabric, self.rank, self.world = fabric, rank, world
        self.multicast = False
        self._k = 0

    def alloc(self, nbytes: int, multicast: bool = True) -> SymmBuffer:
        nbytes = (nbytes + 15) // 16 * 16
        bufs = self.fabric.get(self._k, nbytes)
        self._k += 1
        return SymmBuffer(local=bufs[self.rank], peer_ptrs=[b.data_ptr() for b in bufs], mc_ptr=0, nbytes=nbytes)

    def host_barrier(self) -> None:
        pass

    def close(self) -> None:
        pass


@pytest.fixture
def federation(monkeypatch):
    """``new(world)`` starts an emulated federation: every FedAvgEngine / SmallAggregator (and so FederatedGLM) built
    after the call allocates its symmetric buffers from it.  Build the ranks in rank order."""
    from vantage6_b200.ops import native

    native()                        # loud failure if the extension is missing
    torch.cuda.set_device(0)

    def new(world: int) -> _Fabric:
        fabric = _Fabric(world)
        monkeypatch.setattr(fedavg_mod, "SymmetricHeap", functools.partial(_EmulatedHeap, fabric))
        return fabric

    yield new
    torch.cuda.synchronize()


def _raise_flags(pad: torch.Tensor, words: list) -> None:
    if words:
        idx, val = zip(*words)
        pad[torch.tensor(idx, device=pad.device)] = torch.tensor(val, dtype=torch.int32, device=pad.device)


def run_round(engines, live, weights, *, dynamic=False, prescaled=False, round0=False, absent=None) -> int:
    """One round of the emulated federation; returns its epoch.  Every live rank except ``absent`` launches, in rank
    order, on the current stream.  Before rank r launches, r's pad receives the words the live ranks still to launch
    would have stored there: PAD_UPLOAD (and PAD_NI, the float bits of n_p, with ``dynamic`` weights) when r is a
    reducer, PAD_BCAST of every such rank that is a reducer.  ``absent`` stays silent: nobody raises its flags."""
    launch = [r for r in live if r != absent]
    epoch = engines[launch[0]].epoch + 1
    reducers = engines[launch[0]].reducers
    for i, r in enumerate(launch):
        words = []
        for p in launch[i + 1:]:
            if r in reducers:
                words.append((PAD_UPLOAD + p, epoch + RAISED))
                if dynamic:
                    words.append((PAD_NI + p, _f32_bits(weights[p])))
            if p in reducers:
                words.append((PAD_BCAST + p, epoch + RAISED))
        _raise_flags(engines[r].pad, words)
        if round0:
            engines[r].initialize_global()
        elif dynamic:
            engines[r].aggregate(weights[r], prescaled=prescaled)
        else:
            engines[r].aggregate(list(weights), prescaled=prescaled)
    return epoch


class _Fed:
    """W emulated FedAvgEngines plus the checks that every round must pass."""

    def __init__(self, engines):
        self.e = engines
        self.W = len(engines)
        self.n = engines[0].n
        self.dead: dict = {}                 # rank -> bit snapshots of its buffers and pad at the time it died
        self.gen = torch.Generator(device=DEV).manual_seed(1234 + self.W)

    @property
    def live(self):
        return [r for r in range(self.W) if r not in self.dead]

    def slices(self):
        """(rank, lo, hi) of every live reducer with a non-empty slice; they tile [0, n)."""
        out = [(r, self.e[r].lo, self.e[r].hi) for r in self.live if self.e[r].is_reducer and self.e[r].hi > self.e[r].lo]
        cover = torch.zeros(self.n, dtype=torch.int32)
        for _, lo, hi in out:
            cover[lo:hi] += 1
        assert bool((cover == 1).all()), "reducer slices do not tile the model"
        return out

    def state(self):
        """The server state (w_global, m, v) assembled from the owners' slices, as float64."""
        wg, m, v = (torch.zeros(self.n, dtype=torch.float64, device=DEV) for _ in range(3))
        for r, lo, hi in self.slices():
            e = self.e[r]
            wg[lo:hi] = e.w_global[lo:hi].double()
            if e.opt_m.numel() >= self.n:
                m[lo:hi] = e.opt_m[lo:hi].double()
            if e.opt_v.numel() >= self.n:
                v[lo:hi] = e.opt_v[lo:hi].double()
        return wg, m, v

    def _outside(self, e):
        """The parts of this rank's server-state buffers that lie outside its slice (must never be written)."""
        for t in (e.w_global, e.opt_m, e.opt_v):
            lo, hi = (e.lo, e.hi) if e.is_reducer else (0, 0)
            yield t[:lo]
            yield t[hi:]

    def _shadow_owned(self, e) -> torch.Tensor:
        """Elements of e.shadow that K2 writes: all but the shadow_skip range, which only its owner writes."""
        own = torch.ones(self.n, dtype=torch.bool, device=DEV)
        slo, shi = e.shadow_skip
        own[slo:shi] = False
        for r, lo, hi in self.slices():
            if r == e.rank:
                a, b = max(lo, slo), min(hi, shi)
                if b > a:
                    own[a:b] = True
        return own

    def kill(self, p: int, hint=None) -> None:
        """mark_dead(p) on every survivor; then check the re-partitioned server state: the same global model, the
        moments kept where the owner did not change and zero where it did."""
        wg0, m0, v0 = self.state()
        old = {r: (lo, hi) for r, lo, hi in self.slices()}
        for r in self.live:
            if r != p:
                self.e[r].mark_dead(p, master_hint=hint)
        e = self.e[p]
        for t in (e.w, e.upload, e.shadow):
            if t is not None:
                _poison(t)
        self.dead[p] = [(t, _ints(t).clone()) for t in (e.w, e.upload, e.shadow, e.pad) if t is not None]
        wg, m, v = self.state()
        assert torch.equal(wg, wg0), "mark_dead lost the global model"
        kept = torch.zeros(self.n, dtype=torch.bool, device=DEV)
        for r, lo, hi in self.slices():
            if r in old:
                a, b = max(lo, old[r][0]), min(hi, old[r][1])
                if b > a:
                    kept[a:b] = True
        for got, was in ((m, m0), (v, v0)):
            assert torch.equal(got, torch.where(kept, was, torch.zeros_like(was))), "moments after mark_dead"

    def _prepare(self, weights, *, prescaled, round0):
        """Write this round's uploads (NaN for every rank that must not be read) and the sentinels; return what the
        reference needs."""
        live = self.live
        eff = [float(weights[p]) if p in live else 0.0 for p in range(self.W)]
        wg, m, v = self.state()
        g32 = wg.float()
        xs = [None] * self.W
        for p in live:
            e = self.e[p]
            up = e.w if (round0 or e.upload_mode == "weights_f32") else e.upload
            if eff[p] > 0:
                noise = torch.randn(self.n, device=DEV, generator=self.gen)
                if round0:
                    up.copy_(noise)
                elif e.upload_mode == "weights_f32":
                    up.copy_(g32 + 0.1 * noise)
                else:
                    up.copy_((0.1 * noise * (eff[p] if prescaled else 1.0)).to(up.dtype))
                xs[p] = up.double()
            else:
                _poison(up)
            for t in self._outside(e):
                _poison(t)
            if e.shadow is not None:
                _poison(e.shadow)
        return eff, xs, (wg, m, v)

    def _check_dead(self):
        for p, snaps in self.dead.items():
            for t, was in snaps:
                assert torch.equal(_ints(t), was), f"a buffer or the pad of dead rank {p} was written"

    def round(self, weights, *, dynamic=False, prescaled=False, round0=False) -> None:
        """One round through run_round, then every check: the float64 reference, identical global model on every live
        rank, the bf16 shadow, untouched sentinels, the protocol words and the status words."""
        live = self.live
        eff, xs, (wg, m, v) = self._prepare(weights, prescaled=prescaled, round0=round0)
        epoch = run_round(self.e, live, weights, dynamic=dynamic, prescaled=prescaled, round0=round0)
        torch.cuda.synchronize()
        e0 = self.e[live[0]]
        opt = ServerOptConfig("fedavg", 1.0) if round0 else e0.opt
        delta = not round0 and e0.upload_mode != "weights_f32"
        ref = reference_round(xs, eff, prescaled=prescaled, delta=delta, opt=opt, t=max(e0.server_step, 1), wg=wg, m=m, v=v)
        wg1, m1, v1 = self.state()
        tag = f"epoch {epoch}"
        assert_within(f"{tag} w_global", wg1, ref["w"], ref["tol_w"])
        if opt.name != "fedavg":
            assert_within(f"{tag} server momentum", m1, ref["m"], ref["tol_m"])
        if opt.name == "fedadam":
            assert_within(f"{tag} Adam second moment", v1, ref["v"], ref["tol_v"])
        g32 = wg1.float()
        reducers = e0.reducers
        for r in live:
            e = self.e[r]
            assert torch.equal(_ints(e.w), _ints(g32)), f"{tag}: rank {r} holds another global model"
            for t in self._outside(e):
                assert _is_sentinel(t), f"{tag}: rank {r} wrote server state outside its slice"
            if e.shadow is not None:
                want = g32.to(torch.bfloat16)
                own = self._shadow_owned(e)
                assert torch.equal(_ints(e.shadow)[own], _ints(want)[own]), f"{tag}: rank {r} bf16 shadow"
                # initialize_global() copies w into the whole shadow once its K2 returns.  Run concurrently, step (6)
                # holds that until every reducer has pushed; run in stream order, the reducers after r push later and
                # refresh only the elements K2 writes, so another owner's skip range holds a stale copy here.
                if not round0:
                    assert _is_sentinel(e.shadow[~own]), f"{tag}: rank {r} shadow written inside another owner's skip range"
            pad = e.pad.cpu()
            assert int(pad[PAD_STATUS]) == 0 and int(pad[PAD_MISSING]) == 0, f"{tag}: rank {r} reports a failure"
            for p in live:
                if r in reducers:
                    assert int(pad[PAD_UPLOAD + p]) == epoch, f"{tag}: PAD_UPLOAD[{p}] in reducer {r}'s pad"
                    if dynamic:
                        assert int(pad[PAD_NI + p]) == _f32_bits(weights[p]), f"{tag}: PAD_NI[{p}] in reducer {r}'s pad"
                if p in reducers:
                    assert int(pad[PAD_BCAST + p]) == epoch, f"{tag}: PAD_BCAST[{p}] in rank {r}'s pad"
            assert int(e._cta_counter[0]) == 0, f"{tag}: rank {r} CTA counter not reset"
        self._check_dead()

    def failed_round(self, weights, absent: int) -> None:
        """A round in which live rank ``absent`` never launches: every launched rank must report it, and nothing of a
        failed reducer's slice may be pushed."""
        live = self.live
        central = self.e[live[0]].server_mode == "central"
        self._prepare(weights, prescaled=False, round0=False)
        before = {}
        for r in live:
            e = self.e[r]
            bufs = [e.w, e.w_global, e.opt_m, e.opt_v] + ([e.shadow] if e.shadow is not None else [])
            before[r] = [(t, _ints(t).clone()) for t in bufs]
        epoch = run_round(self.e, live, weights, absent=absent)
        torch.cuda.synchronize()
        for r in live:
            if r == absent:
                continue
            e = self.e[r]
            st, miss = e.poll_status(), e.missing_mask()
            assert st != 0 and miss == 1 << absent, f"epoch {epoch}: rank {r} status {st}, missing {miss:#x}"
            if central and absent != 0 and r != 0:
                # a non-reducer's own wait succeeded; it learns of the failure from the server's PAD_RFAIL / PAD_RMISS
                assert st == 2, f"rank {r} did not see the server's failure report"
            else:
                assert st == 1, f"rank {r}: its own wait should have timed out"
            assert int(e._cta_counter[0]) == 0
        for r, snaps in before.items():
            for t, was in snaps:
                assert torch.equal(_ints(t), was), f"epoch {epoch}: rank {r} was written in a failed round"
        self._check_dead()


# ---------------------------------------------------------------------------------------------------- K2 cases
def _case(W, mode, upload, opt, weights, n, *, dead=None, shadow=False, skip=False, sm2=False):
    return pytest.param(dict(W=W, mode=mode, upload=upload, opt=opt, weights=weights, n=n, dead=dead, shadow=shadow or skip,
                             skip=skip, sm2=sm2),
                         id=f"W{W}-{mode}-{upload}-{opt}-{weights}-n{n}" + (f"-dead{dead}" if dead is not None else "")
                         + ("-skip" if skip else "-shadow" if shadow else "") + ("-sm2" if sm2 else ""))


# WMAX 2 (U 4): W 2; WMAX 4 (U 2): W 3, 4; WMAX 8 (U 1): W 5, 8.  Every upload mode meets every optimizer; n = 8 at W = 8
# leaves seven reducers an empty slice; 100_003 leaves a vector tail; 3_000_017 takes several grid-stride iterations at
# the default grid (central, or two to four reducers).
K2_CASES = [
    _case(2, "sharded", "weights_f32", "fedavg", "vector", 1000),
    _case(2, "central", "delta_bf16", "fedadam", "dynamic", 3_000_017, shadow=True),
    _case(2, "sharded", "delta_f32", "fedavgm", "prescaled", 100_003, skip=True),
    _case(3, "sharded", "delta_f32", "fedadam", "zero", 100_003, shadow=True),
    _case(3, "central", "weights_f32", "fedavgm", "equal", 1000, dead=2),
    _case(4, "sharded", "delta_bf16", "fedadam", "prescaled", 3_000_017),
    _case(4, "central", "delta_f32", "fedavg", "dynamic", 100_003, sm2=True),
    _case(4, "sharded", "weights_f32", "fedadam", "vector", 100_003, dead=1, skip=True),
    _case(5, "sharded", "delta_bf16", "fedavgm", "vector", 100_003, skip=True),
    _case(5, "central", "weights_f32", "fedadam", "dynamic", 3_000_017, dead=3, shadow=True),
    _case(5, "sharded", "delta_f32", "fedavg", "dynamic_zero", 1000),
    _case(8, "sharded", "delta_f32", "fedadam", "vector", 8, shadow=True),
    _case(8, "sharded", "weights_f32", "fedavgm", "equal", 100_003, dead=5),
    _case(8, "central", "delta_bf16", "fedavg", "zero", 100_003, skip=True),
    _case(8, "sharded", "delta_bf16", "fedadam", "dynamic", 1000, dead=6, shadow=True),
    _case(8, "central", "delta_f32", "fedavgm", "prescaled", 100_003, sm2=True),
]


def _weights(kind: str, W: int):
    """(per-rank sample counts, dynamic, prescaled) of a weight scheme."""
    n = list(N8[:W])
    if kind == "equal":
        return [4.0] * W, True, False
    if kind in ("zero", "dynamic_zero"):
        n[1] = 0.0                    # alive (waited for, pushed to) but not reporting
    return n, kind in ("dynamic", "dynamic_zero"), kind == "prescaled"


def _engines(new, W, n, *, mode, upload, opt="fedavg", shadow=False, skip=False):
    new(W)
    shadow_skip = ((n // 4) // 8 * 8, (n // 2 + 7) // 8 * 8) if skip else (0, 0)
    return [FedAvgEngine(n, r, W, DEV, data_plane="native", server_mode=mode, server_opt=ServerOptConfig(opt, LR[opt]),
                         upload=upload, shadow_bf16=shadow, shadow_skip=shadow_skip, timeout_ms=0.05) for r in range(W)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", K2_CASES)
def test_fedavg_round_peers_match_float64(federation, case):
    """Round 0 (initialize_global) and three rounds of K2 at W ranks against the float64 reference."""
    W = case["W"]
    engines = _engines(federation, W, case["n"], mode=case["mode"], upload=case["upload"], opt=case["opt"],
                       shadow=case["shadow"], skip=case["skip"])
    if case["sm2"]:
        for e in engines:
            e.sm_count = 2                  # a two-CTA grid: the grid-stride loop runs many times
    fed = _Fed(engines)
    fed.round([1.0] + [0.0] * (W - 1), round0=True)
    if case["dead"] is not None:
        fed.kill(case["dead"])
    weights, dynamic, prescaled = _weights(case["weights"], W)
    for _ in range(3):
        fed.round(weights, dynamic=dynamic, prescaled=prescaled)
    for e in engines:
        e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("W,mode,absent,upload,opt", [
    (4, "sharded", 2, "delta_f32", "fedadam"),
    (5, "central", 3, "weights_f32", "fedavgm"),
    (3, "central", 0, "delta_bf16", "fedavg"),            # the server itself is missing: the role moves to rank 1
    (8, "sharded", 0, "weights_f32", "fedadam"),
])
def test_fedavg_round_missing_rank_reported_then_excluded(federation, W, mode, absent, upload, opt):
    """A rank alive by live_mask that never launches: every reducer's wait ends on its timeout, every launched rank
    reports it, nothing is pushed; after clear_status + mark_dead the next round matches the reference without it."""
    engines = _engines(federation, W, 100_003, mode=mode, upload=upload, opt=opt, shadow=True)
    fed = _Fed(engines)
    fed.round([1.0] + [0.0] * (W - 1), round0=True)
    weights = list(N8[:W])
    fed.round(weights)
    g = fed.state()[0].float()
    fed.failed_round(weights, absent)
    for r in fed.live:
        if r != absent:
            engines[r].clear_status()
    # weights_f32: w holds the local weights of the failed round, so the global model is handed over explicitly
    fed.kill(absent, hint=g if upload == "weights_f32" else None)
    for _ in range(2):
        fed.round(weights)
    for e in engines:
        e.close()


# ---------------------------------------------------------------------------------------------------- K3
@pytest.mark.gpu
@pytest.mark.parametrize("n_floats", [4, 1000, 16384])
@pytest.mark.parametrize("W", [2, 5, 8])
def test_small_allreduce_peers_match_float64(federation, W, n_floats):
    """K3 at W ranks: weighted sum over the slots of every reporting rank (a weight-0 rank's slot holds NaN), with and
    without normalisation, over both slot parities."""
    federation(W)
    aggs = [SmallAggregator(n_floats, r, W, DEV, timeout_ms=0.05) for r in range(W)]
    pads = [a._pad_buf.view(torch.int32, PAD_WORDS) for a in aggs]
    gen = torch.Generator(device=DEV).manual_seed(77 + W)
    zero = list(N8[:W])
    zero[W - 1] = 0.0
    for weights, normalize in ((zero, True), (list(N8[:W]), False), ([2.0] * W, True)):
        epoch = aggs[0].epoch + 1
        xs = []
        for r, a in enumerate(aggs):
            if weights[r] > 0:
                a.slot().copy_(torch.randn(a.n, device=DEV, generator=gen))
            else:
                _poison(a.slot())
            xs.append(a.slot().double())
            _poison(a.out)
        for r, a in enumerate(aggs):
            _raise_flags(pads[r], [(PAD_SMALL + p, epoch + RAISED) for p in range(r + 1, W)])
            a.allreduce(weights, normalize=normalize)
        torch.cuda.synchronize()
        inv = _f32(1.0 / sum(weights)) if normalize else 1.0
        rep = [p for p in range(W) if weights[p] > 0]
        want = sum(weights[p] * xs[p] for p in rep) * inv
        # len(rep) fmaf and one multiply, each within 2^-24 of its result: twice that, relative to sum |w_p x_p| * inv
        tol = 2 * (len(rep) + 1) * U * sum(weights[p] * xs[p].abs() for p in rep) * inv + 1e-37
        for r, a in enumerate(aggs):
            assert_within(f"epoch {epoch} rank {r} out", a.out, want, tol)
            pad = pads[r].cpu()
            assert int(pad[PAD_STATUS]) == 0, f"epoch {epoch}: rank {r} reports a timeout"
            assert [int(pad[PAD_SMALL + p]) for p in range(W)] == [epoch] * W
    for a in aggs:
        a.close()


# ---------------------------------------------------------------------------------------------------- fused GLM tail
def _fold_f32(part: np.ndarray, nparts: int, F: int, rows: float, n: int) -> np.ndarray:
    """The kernel's fold of the per-CTA partials into a payload slot, in the same fixed order and in fp32."""
    out = np.zeros(n, dtype=np.float32)
    p = part.reshape(nparts, F + 2)
    acc = np.zeros(F + 2, dtype=np.float32)
    for i in range(nparts):
        acc += p[i]
    out[: F + 2] = acc
    out[F + 2] = rows
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("W,nparts,F", [((2, 5, 8)[i % 3], np_, F) for i, (np_, F) in
                                        enumerate(itertools.product((1, 7, 592), (1, 29, 256)))])
def test_glm_aggregate_update_peers_match_float64(federation, W, nparts, F):
    """The fused GLM tail through its binding at W ranks, two iterations (both slot parities): each rank's folded
    slot, the summed payload, the coefficients and the loss, against float64."""
    from vantage6_b200.ops import native, stream_ptr
    from vantage6_b200.ops.glm import payload_len

    C = native()
    federation(W)
    aggs = [SmallAggregator(payload_len(F), r, W, DEV, timeout_ms=0.05) for r in range(W)]
    n = aggs[0].n
    pads = [a._pad_buf.view(torch.int32, PAD_WORDS) for a in aggs]
    lr = 0.5
    rng = np.random.default_rng(nparts * 1000 + F)
    w0 = torch.tensor(rng.standard_normal(F + 1), dtype=torch.float32, device=DEV)
    ws = [w0.clone() for _ in range(W)]
    losses = [torch.zeros((), dtype=torch.float32, device=DEV) for _ in range(W)]
    u = 2 * U
    for it in range(2):
        parts = [rng.standard_normal(nparts * (F + 2)).astype(np.float32) for _ in range(W)]
        rows = [float(100 + 37 * r + it) for r in range(W)]
        folds = [_fold_f32(parts[r], nparts, F, rows[r], n) for r in range(W)]
        parts_dev = [torch.from_numpy(p).to(DEV) for p in parts]
        epoch = aggs[0].epoch + 1
        par = epoch & 1
        w_prev = [w.double() for w in ws]
        for a in aggs:
            _poison(a.slots[par])
            _poison(a.out)
        for r, a in enumerate(aggs):
            # every kernel folds only its own slot: the slots of the ranks still to launch get their fold now
            for p in range(r + 1, W):
                aggs[p].slots[par].copy_(torch.from_numpy(folds[p]).to(DEV))
            _raise_flags(pads[r], [(PAD_SMALL + p, epoch + RAISED) for p in range(r + 1, W)])
            a.epoch += 1
            C.glm_aggregate_update(a._slots.peer(par * n * 4), a._pad_buf.peer(), [1.0] * W, a.out.data_ptr(), n, r, W,
                                   a.epoch, a.timeout_cycles, parts_dev[r].data_ptr(), nparts, F, rows[r], lr,
                                   ws[r].data_ptr(), losses[r].data_ptr(), stream_ptr())
        torch.cuda.synchronize()
        part64 = [torch.from_numpy(p.astype(np.float64)).view(nparts, F + 2).to(DEV) for p in parts]
        G = sum(p.sum(0) for p in part64)
        A = sum(p.abs().sum(0) for p in part64)
        N = sum(rows)
        # fold: nparts additions per rank; sum over ranks: W more -> e_G <= (nparts + W) u A; then x lr, x 1/N, minus
        e_G = (nparts + W) * u * A
        for r, a in enumerate(aggs):
            slot = a.slots[par].double()
            f64 = part64[r].sum(0)
            assert_within(f"iteration {it} rank {r} folded slot", slot[: F + 2], f64, 2 * nparts * u * part64[r].abs().sum(0) + 1e-37)
            assert float(slot[F + 2]) == rows[r] and bool((slot[F + 3:] == 0).all()), f"rank {r} slot tail"
            assert_within(f"iteration {it} rank {r} summed payload", a.out[: F + 2], G, 2 * e_G + 1e-37)
            assert float(a.out[F + 2]) == N and bool((a.out[F + 3:] == 0).all()), f"rank {r} summed row count / pad"
            want_w = w_prev[r] - lr * G[: F + 1] / N
            tol_w = 2 * (lr * (e_G[: F + 1] + 3 * u * G[: F + 1].abs()) / N + u * want_w.abs()) + 1e-37
            assert_within(f"iteration {it} rank {r} coefficients", ws[r], want_w, tol_w)
            want_l = G[F + 1:F + 2] / N
            assert_within(f"iteration {it} rank {r} loss", losses[r].reshape(1), want_l,
                          2 * (e_G[F + 1:F + 2] + 2 * u * want_l.abs() * N) / N + 1e-37)
            pad = pads[r].cpu()
            assert int(pad[PAD_STATUS]) == 0 and [int(pad[PAD_SMALL + p]) for p in range(W)] == [epoch] * W
    for a in aggs:
        a.close()
