"""The LPG reverse pass kernel by kernel (no agent adjoint, no meta loss): the tensor-core chain
toued_cotangent_max -> toued_gru_backward_tc -> toued_lpg_wgrad_tc -> toued_lpg_wgrad_embed -> toued_reduce_partials and
its exact-fp32 SIMT twin toued_gru_backward -> toued_lpg_wgrad, issued as meta/train.py issues them, on one forward of a
seeded rollout and on seeded synthetic (or real) cotangents d pi_hat [L][R], d y_hat [L][R][8].

  R1  SIMT chain vs fp64 autograd of oracle/lpg.py (fp32 arithmetic only)
  R2  tensor-core chain vs the SIMT chain fed the tensor-core forward's own activations (h16, gate planes): the error of
      the reverse pass alone (fp16 Wh, fp16 dG, the hi / lo carry injection); tolerances measured, DESIGN.md section 6
  R3  tensor-core chain vs fp64 end to end, at the meta-gradient tolerances of test_13 / test_15

Errors are reported per parameter block as relative L2 and as max |error| / max |reference|.  Also: bitwise
reproducibility, exact power-of-two scale equivariance, accumulation of two updates with separate scales, the
{max, status} word of toued_cotangent_max, the fp16 range status of the BPTT kernel, and NaN propagation."""
import numpy as np
import pytest
import torch

from helpers import Case, to_oracle_traj
from oracle.agents import tab_forward
from oracle.lpg import lpg_forward
from test_13_tc_gpu import _fac_plane, _from_rb32

pytestmark = pytest.mark.gpu

# Stated tolerances, each bounding both relative L2 and max |error| / max |reference| of a parameter block.  Measured
# worst cases on a B200 over the shape matrix, the real-cotangent cases and the saturation control are in DESIGN.md
# section 6 (R1 1.9e-5: the scalar e_b1, a sum that cancels; R2 8.4e-4 GRU, 4e-6 heads, 1.9e-3 embedding, dx 2.3e-4).
R1_TOL = 5e-5                 # fp32 SIMT chain vs fp64
R2_TOL = {"Wh": 2e-3, "Wi": 2e-3, "bi": 2e-3, "bhn": 2e-3,          # GRU blocks: fp16 dG, Wh and x operands
          "w_pi": 2e-5, "W_y": 2e-5, "b_y": 2e-5, "b_pi": 2e-5,     # heads: fp16 hi / lo cotangents, exact relu(h16)
          "e_w0": 5e-3, "e_b0": 5e-3, "e_w1": 5e-3, "e_b1": 5e-3,   # embedding MLP: sums of dx that cancel over tokens
          "all": 2e-3}
R2_DX_TOL = 1e-3              # dx / S vs the SIMT dx (dl / S is bit-identical to the SIMT dl)
# End to end: the meta-gradient tolerances of test_13 / test_15, for real cotangents.  Synthetic cotangents of random
# sign cancel in every parameter sum, and the tensor-core FORWARD's fp16 rounding (not the reverse pass: R2) then
# reaches 1.4e-2 relative L2 of the whole gradient; there only that is asserted, against R3_SYNTH_L2.
R3_L2, R3_BLOCK, R3_SYNTH_L2 = 1e-2, 2e-2, 2e-2
FWD_TOL = 3e-3                # tensor-core forward vs fp32 kernel (test_13)
STATUS_NONFINITE_COT, STATUS_FP16_RANGE = 1, 2      # include/toued.h TOUED_STATUS_*


def _lib():
    from to_ued_b200 import _lib as L
    return L


class Fwd:
    """One rollout of a Case, LPG inputs and both forwards (fp32 SIMT and tensor-core) on it."""

    def __init__(self, c, zero_done=False):
        from to_ued_b200.agents.lpg_agent import Tape
        L_, p = _lib(), _lib().ptr
        s = L_.stream_ptr()
        self._shape(c)
        ag, ro = c.agent_state()
        traj, _, _, _ = ro.batch_rollout(c.keys, ag.actor_state, ag.level.packed, ag.env_obs, ag.env_state)
        self.lpg = torch.from_numpy(c.lpg).cuda()
        self.critic, self.step = ag.critic_state.params, ag.actor_state.step
        self.tapes = {}
        for prec in ("fp32", "tc"):
            t = Tape(c.n, c.w, c.L, c.D, 1, "cuda", precision=prec)
            t.obs[0].copy_(traj.obs); t.action[0].copy_(traj.action); t.reward[0].copy_(traj.reward)
            t.done[0].copy_(traj.done)
            if zero_done:
                t.done[0].zero_()
            L_.call("toued_lpg_prepare", p(t.obs[0]), p(t.action[0]), p(t.reward[0]), p(t.done[0]),
                    p(ag.actor_state.params), p(self.critic), p(self.lpg), p(self.step), p(ag.level.packed), p(t.x[0]),
                    p(t.ximg[0]) if t.ximg is not None else None, c.n, c.w, c.L, c.D, self.cond, 0, s)
            self.tapes[prec] = t
        self.traj = to_oracle_traj(self.tapes["fp32"].transition(0))
        self.actor64 = torch.tensor(c.actor, dtype=torch.float64)
        self.critic64 = torch.tensor(c.critic, dtype=torch.float64)
        self.steps64, self.life = torch.tensor(c.steps.astype(np.int64)), c.life
        self.run_forward()

    def _shape(self, c):
        self.c, self.n, self.w, self.L, self.D = c, c.n, c.w, c.L, c.D
        self.R, self.cond = c.n * c.w, int(c.layout.lifetime_conditioning)

    @classmethod
    def from_meta_step(cls, c, tape):
        """Update 0 of a finished tensor-core meta-step (tape slot 0: rollout, inputs, activations, tables)."""
        f = cls.__new__(cls)
        f._shape(c)
        f.lpg, f.critic, f.tapes = torch.from_numpy(c.lpg).cuda(), tape.critic[0], {"tc": tape}
        f.traj = to_oracle_traj(tape.transition(0))
        f.actor64, f.critic64 = tape.actor[0][..., :5].double().cpu(), tape.critic[0].double().cpu()
        f.steps64, f.life = tape.step_in[0].long().cpu(), c.life
        return f

    def run_forward(self):
        L_, p, s = _lib(), _lib().ptr, _lib().stream_ptr()
        t = self.tapes["fp32"]
        L_.call("toued_gru_forward", p(t.x[0]), p(t.done[0]), p(self.lpg), p(t.h[0]), p(t.gates[0]), p(t.pi_hat[0]),
                p(t.y_hat[0]), self.n, self.w, self.L, self.cond, 0, s)
        t = self.tapes["tc"]
        L_.call("toued_pack_wh_forward", p(self.lpg), p(t.wh_img), self.cond, s)
        L_.call("toued_gru_forward_tc", p(t.x[0]), p(t.done[0]), p(self.lpg), p(t.wh_img), p(t.h16[0]), p(t.fac[0]),
                p(t.hpimg[0]), p(t.pi_hat[0]), p(t.y_hat[0]), self.n, self.w, self.L, self.cond, s)

    def tc_activations(self):
        """h and the gate planes (r, |z|, n, hn) of the tensor-core forward as the SIMT chain's fp32 inputs."""
        t = self.tapes["tc"]
        h = _from_rb32(t.h16[0], self.L, self.R).float().contiguous()
        planes = [_fac_plane(t.fac[0], i, self.L, self.R) for i in range(4)]
        planes[1] = planes[1].abs()
        return h, torch.stack(planes).float().contiguous()


def _new_partials():
    return torch.zeros(_lib().lib().toued_lpg_wgrad_workspace_floats(), dtype=torch.float32, device="cuda")


def _reduce(f, partials, tc):
    L_ = _lib()
    n_wh, n_sm = (L_.lib().toued_wgrad_tc_splits(), L_.lib().toued_wgrad_tc_small_splits()) if tc else \
        (L_.lib().toued_lpg_wgrad_splits(0), L_.lib().toued_lpg_wgrad_splits(1))
    grad = torch.empty(f.c.layout.size, dtype=torch.float32, device="cuda")
    L_.call("toued_reduce_partials", L_.ptr(partials), L_.ptr(grad), f.cond, n_wh, n_sm, L_.stream_ptr())
    return grad


def simt_chain(f, d_pi, d_y, h=None, gates=None, y_hat=None):
    """toued_transpose_wh -> toued_gru_backward -> toued_lpg_wgrad -> toued_reduce_partials (meta/train.py, fp32 path).
    Activations default to the fp32 forward's.  Returns (grad, dl, dx)."""
    L_, p, s = _lib(), _lib().ptr, _lib().stream_ptr()
    t = f.tapes["tc"]                                               # rollout and LPG inputs (the same in both tapes)
    if h is None:
        h, gates, y_hat = f.tapes["fp32"].h[0], f.tapes["fp32"].gates[0], f.tapes["fp32"].y_hat[0]
    g = gates.clone()                                               # toued_gru_backward overwrites it with dgates
    whT = torch.empty((768, 256), dtype=torch.float32, device="cuda")
    dl = torch.empty((f.L, f.R, 8), dtype=torch.float32, device="cuda")
    dx = torch.empty((f.L, f.R, 2), dtype=torch.float32, device="cuda")
    part = _new_partials()
    L_.call("toued_transpose_wh", p(f.lpg), p(whT), s)
    L_.call("toued_gru_backward", p(t.done[0]), p(f.lpg), p(whT), p(h), p(g), p(y_hat), p(d_pi), p(d_y), p(dl), p(dx),
            f.n, f.w, f.L, f.cond, s)
    L_.call("toued_lpg_wgrad", p(t.obs[0]), p(t.done[0]), p(f.critic), p(f.lpg), p(t.x[0]), p(h), p(g), p(d_pi), p(dl),
            p(dx), p(part), f.n, f.w, f.L, f.D, f.cond, 0, s)
    return _reduce(f, part, False), dl, dx


def tc_chain_into(f, d_pi, d_y, cotmax, partials, accumulate):
    """One update's tensor-core reverse pass into `partials` (meta/train.py backward_step); returns (dl, dx) in units of S."""
    L_, p, s = _lib(), _lib().ptr, _lib().stream_ptr()
    t = f.tapes["tc"]
    Rp = (f.R + 63) // 64 * 64
    whb = torch.empty(256 * 768, dtype=torch.float16, device="cuda")
    dgimg = torch.zeros(f.L * Rp * 1024 * 2, dtype=torch.uint8, device="cuda")
    dl = torch.empty((f.L, f.R, 8), dtype=torch.float32, device="cuda")
    dx = torch.empty((f.L, f.R, 2), dtype=torch.float32, device="cuda")
    off_small = L_.lib().toued_lpg_wgrad_workspace_offset(1)
    L_.call("toued_pack_wh_backward", p(f.lpg), p(whb), s)
    L_.call("toued_cotangent_max", p(d_pi), p(d_y), f.n, f.w, f.L, p(cotmax), s)
    L_.call("toued_gru_backward_tc", p(t.done[0]), p(f.lpg), p(whb), p(t.h16[0]), p(t.fac[0]), p(t.y_hat[0]), p(d_pi),
            p(d_y), p(dgimg), p(dl), p(dx), p(cotmax), f.n, f.w, f.L, f.cond, s)
    L_.call("toued_lpg_wgrad_tc", p(t.hpimg[0]), p(dgimg), p(t.ximg[0]), p(t.h16[0]), p(d_pi), p(dl), p(partials),
            p(partials[off_small:]), p(cotmax), f.n, f.w, f.L, accumulate, s)
    L_.call("toued_lpg_wgrad_embed", p(t.obs[0]), p(t.done[0]), p(f.critic), p(f.lpg), p(dx), p(partials), p(cotmax),
            f.n, f.w, f.L, f.D, f.cond, accumulate, s)
    return dl, dx


def scale_of(cotmax):
    """tc.cuh::cot_scale_from_max on the host."""
    bits = int(cotmax[0].item()) & 0xFFFFFFFF
    if bits == 0 or bits >= 0x7F800000:
        return 1.0
    return 2.0 ** min(max(3 - ((bits >> 23) - 127), -100), 100)


def tc_chain(f, d_pi, d_y):
    """Returns (grad, dl / S, dx / S, cotmax word pair)."""
    cm = torch.zeros(2, dtype=torch.int32, device="cuda")
    part = _new_partials()
    dl, dx = tc_chain_into(f, d_pi, d_y, cm, part, 0)
    grad = _reduce(f, part, True)
    torch.cuda.synchronize()
    S = scale_of(cm)
    return grad, dl / S, dx / S, cm.cpu()


def fp64_reference(f, d_pi, d_y, lpg=None, hidden=None, nan_at=None):
    """fp64 autograd of oracle lpg_forward on the same trajectory and tables (oracle/agents.py lpg_agent_train_step:
    pi and y_t detached, gradient w.r.t. the flat LPG parameters).  ``hidden``: also return d/dh_t of every step;
    ``nan_at`` = (t, row): a NaN policy input at that token."""
    dt = torch.float64
    tr, N, W, L = f.traj, f.n, f.w, f.L
    reward, done = torch.as_tensor(tr.reward).to(dt), torch.as_tensor(tr.done).to(dt)
    action = torch.as_tensor(tr.action.astype(np.int64))
    oi, ot = tr.obs_idx, tr.obs_time
    pi = torch.gather(tab_forward(f.actor64, oi[:, :L], ot[:, :L]) + 1e-8, -1, action[..., None])[..., 0]
    y_t = tab_forward(f.critic64, oi[:, :L], ot[:, :L])
    y_tp1 = tab_forward(f.critic64, oi[:, 1:], ot[:, 1:])
    seq = lambda a: a.transpose(1, 2).reshape((N * W, L) + a.shape[3:])
    pis = seq(pi)
    if nan_at is not None:
        pis[nan_at[1], nan_at[0]] = float("nan")
    flat = torch.tensor(f.c.lpg if lpg is None else lpg, dtype=dt).requires_grad_()
    hs = [] if hidden is not None else None
    life = torch.as_tensor(np.asarray(f.life))
    pi_hat, y_hat = lpg_forward(f.c.layout, flat, seq(reward), seq(done), pis, seq(y_t), seq(y_tp1),
                                f.steps64.repeat_interleave(W), life.repeat_interleave(W), hidden=hs)
    # the kernels' cotangents are time-major [L][R]; the oracle's sequences are [R][L]
    cp = d_pi.double().cpu().T
    cy = d_y.double().cpu().transpose(0, 1)
    gs = torch.autograd.grad((pi_hat, y_hat), [flat] + (hs or []), (cp, cy))
    if hidden is not None:
        hidden.extend(gs[1:])
    return gs[0].numpy(), pi_hat.detach(), y_hat.detach()


def block_errors(c, g, ref):
    g = np.asarray(g.detach().cpu() if torch.is_tensor(g) else g, np.float64)
    ref = np.asarray(ref.detach().cpu() if torch.is_tensor(ref) else ref, np.float64)
    out = {}
    for name, (off, cnt, _) in c.layout.offsets.items():
        a, b = g[off:off + cnt], ref[off:off + cnt]
        out[name] = (np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30), np.abs(a - b).max() / (np.abs(b).max() + 1e-30))
    out["all"] = (np.linalg.norm(g - ref) / (np.linalg.norm(ref) + 1e-30), np.abs(g - ref).max() / (np.abs(ref).max() + 1e-30))
    return out


def r2_failures(errs):
    return [f"{k} {l2:.2e}/{mx:.2e}" for k, (l2, mx) in errs.items() if not (l2 < R2_TOL[k] and mx < R2_TOL[k])]


def _fmt(tag, errs):
    return f"{tag}: " + " ".join(f"{k}={v[0]:.1e}/{v[1]:.1e}" for k, v in errs.items())


def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


def synthetic_cotangents(f, seed, scale=1e-3):
    g = torch.Generator(device="cpu").manual_seed(seed)
    d_pi = (torch.randn(f.L, f.R, generator=g) * scale).cuda()
    d_y = (torch.randn(f.L, f.R, 8, generator=g) * scale).cuda()
    return d_pi, d_y


def make_case(n, w, L, cond, seed=11, scale=None):
    steps = (np.arange(n) * 37 % 250).astype(np.int32) if cond else None
    c = Case("all_vrandlife" if cond else "all_shortlife", n=n, w=w, L=L, seed=seed, cond=cond, table_scale=0.3,
             steps=steps)
    for name, fac in (scale or {}).items():
        off, cnt, _ = c.layout.offsets[name]
        c.lpg[off:off + cnt] *= fac
    return c


# (n, W, L, cond); see the module docstring of each geometry in the ids
SHAPES = [
    pytest.param(4, 64, 20, False, id="R256-production-tiles"), pytest.param(4, 64, 20, True, id="R256-cond"),
    pytest.param(3, 8, 20, False, id="R24-one-partial-tile"), pytest.param(3, 8, 20, True, id="R24-cond"),
    pytest.param(9, 8, 20, False, id="R72-ragged-second-block"), pytest.param(9, 8, 20, True, id="R72-cond"),
    pytest.param(5, 32, 20, False, id="R160-two-ctas-R%64=32"), pytest.param(5, 32, 20, True, id="R160-cond"),
    pytest.param(1, 1, 20, False, id="R1-minimum"),
    pytest.param(1, 128, 20, False, id="W128"),
    pytest.param(4, 64, 1, False, id="L1"), pytest.param(4, 64, 2, False, id="L2"),
    pytest.param(3, 16, 33, False, id="L33-odd"),
    pytest.param(2, 64, 64, False, id="L64-WL4096"),
]


@pytest.mark.parametrize("n,w,L,cond", SHAPES)
def test_reverse_pass_per_kernel_chain(built_lib, n, w, L, cond):
    c = make_case(n, w, L, cond)
    f = Fwd(c)
    d_pi, d_y = synthetic_cotangents(f, seed=n * 1000 + w * 10 + L)
    torch.cuda.synchronize()
    # tensor-core forward vs the fp32 kernel (test_13's tolerance)
    t32, ttc = f.tapes["fp32"], f.tapes["tc"]
    e_pi, e_y = _rel(ttc.pi_hat[0], t32.pi_hat[0]), _rel(ttc.y_hat[0], t32.y_hat[0])
    assert e_pi < FWD_TOL and e_y < FWD_TOL, f"forward: pi_hat {e_pi:.2e} y_hat {e_y:.2e}"
    # R1
    g32, dl32, dx32 = simt_chain(f, d_pi, d_y)
    g64, _, _ = fp64_reference(f, d_pi, d_y)
    r1 = block_errors(c, g32, g64)
    # R2
    h, gates = f.tc_activations()
    g32tc, dl32tc, dx32tc = simt_chain(f, d_pi, d_y, h, gates, ttc.y_hat[0])
    gtc, dltc, dxtc, cm = tc_chain(f, d_pi, d_y)
    r2 = block_errors(c, gtc, g32tc)
    e_dl, e_dx = _rel(dltc, dl32tc), _rel(dxtc, dx32tc)
    # R3, and the share of the tensor-core forward in it (the exact SIMT reverse pass on its activations vs fp64)
    r3, r3f = block_errors(c, gtc, g64), block_errors(c, g32tc, g64)
    print(f"\n[n={n} W={w} L={L} cond={cond}] forward pi_hat {e_pi:.1e} y_hat {e_y:.1e}; status {int(cm[1])}\n  "
          + _fmt("R1", r1) + "\n  " + _fmt("R2", r2) + f" dl={e_dl:.1e} dx={e_dx:.1e}\n  " + _fmt("R3", r3)
          + "\n  " + _fmt("R3 of the forward alone", r3f))
    assert int(cm[1]) == 0, "status set on an ordinary reverse pass"
    # bitwise reproducible
    gtc2, dltc2, dxtc2, _ = tc_chain(f, d_pi, d_y)
    assert torch.equal(gtc, gtc2) and torch.equal(dltc, dltc2) and torch.equal(dxtc, dxtc2), "tensor-core chain not reproducible"
    for name, (l2, mx) in r1.items():
        assert l2 < R1_TOL and mx < R1_TOL, f"R1 block {name}: {l2:.2e} / {mx:.2e}"
    assert not r2_failures(r2), f"R2: {r2_failures(r2)}"
    assert e_dl < 1e-6 and e_dx < R2_DX_TOL, f"R2 dl {e_dl:.2e} dx {e_dx:.2e}"
    assert r3["all"][0] < R3_SYNTH_L2, f"R3 relative L2 {r3['all'][0]:.2e}"


def test_reverse_pass_bench_chunk_geometry(built_lib):
    """R = 16384 (256 agents x 64 workers, the benchmark's chunk): R2 only (the fp64 reference is too slow here)."""
    c = make_case(256, 64, 20, False)
    f = Fwd(c)
    d_pi, d_y = synthetic_cotangents(f, seed=5)
    e_pi, e_y = _rel(f.tapes["tc"].pi_hat[0], f.tapes["fp32"].pi_hat[0]), _rel(f.tapes["tc"].y_hat[0], f.tapes["fp32"].y_hat[0])
    assert e_pi < FWD_TOL and e_y < FWD_TOL, f"forward: pi_hat {e_pi:.2e} y_hat {e_y:.2e}"
    h, gates = f.tc_activations()
    g32tc, dl32, dx32 = simt_chain(f, d_pi, d_y, h, gates, f.tapes["tc"].y_hat[0])
    gtc, dltc, dxtc, cm = tc_chain(f, d_pi, d_y)
    r2 = block_errors(c, gtc, g32tc)
    print("\n[R=16384] " + _fmt("R2", r2) + f" dl={_rel(dltc, dl32):.1e} dx={_rel(dxtc, dx32):.1e}")
    assert int(cm[1]) == 0
    gtc2, _, _, _ = tc_chain(f, d_pi, d_y)
    assert torch.equal(gtc, gtc2)
    assert not r2_failures(r2), f"R2: {r2_failures(r2)}"
    assert _rel(dltc, dl32) < 1e-6 and _rel(dxtc, dx32) < R2_DX_TOL


@pytest.mark.parametrize("cond", [False, True])
def test_reverse_pass_real_cotangents(built_lib, monkeypatch, cond):
    """Cotangents and activations of update 0 of a real meta-step (agent adjoint of the tensor-core path)."""
    import to_ued_b200
    from test_14_meta_grad_gpu import _run
    monkeypatch.setattr(to_ued_b200, "GRU_PRECISION", "tc")
    c = make_case(3, 64, 20, cond, seed=7)
    (_, _, _, met), ws = _run(c, 2)
    tape = ws.tape
    d_pi, d_y = ws.d_pi_hat2[0].clone(), ws.d_y_hat2[0].clone()
    f = Fwd.from_meta_step(c, tape)
    h, gates = f.tc_activations()
    g32tc, _, _ = simt_chain(f, d_pi, d_y, h, gates, tape.y_hat[0])
    gtc, _, _, cm = tc_chain(f, d_pi, d_y)
    g64, _, _ = fp64_reference(f, d_pi, d_y)
    r2, r3 = block_errors(c, gtc, g32tc), block_errors(c, gtc, g64)
    print(f"\n[real cotangents cond={cond}] max |cot| {float(torch.max(d_pi.abs().max(), d_y.abs().max())):.2e}\n  "
          + _fmt("R2", r2) + "\n  " + _fmt("R3", r3))
    assert int(cm[1]) == 0
    assert not r2_failures(r2), f"R2: {r2_failures(r2)}"
    assert r3["all"][0] < R3_L2
    for name, (l2, mx) in r3.items():
        assert mx < R3_BLOCK, f"R3 block {name}: {mx:.2e}"


@pytest.mark.parametrize("n,w", [(4, 64), (9, 8)])
def test_two_updates_accumulate_with_their_own_scales(built_lib, n, w):
    """Two reverse passes into the same partials (accumulate 0 then 1), cotangents 2^20 apart, one cotmax word pair
    each: the result is the sum of the two single-update results (a consumer that read the other update's S would be
    off by 2^20)."""
    c = make_case(n, w, 20, False)
    f = Fwd(c)
    a_pi, a_y = synthetic_cotangents(f, seed=1)
    b_pi, b_y = synthetic_cotangents(f, seed=2, scale=1e-3 * 2.0 ** 20)
    ga, _, _, _ = tc_chain(f, a_pi, a_y)
    gb, _, _, _ = tc_chain(f, b_pi, b_y)
    part = _new_partials()
    cms = torch.zeros((2, 2), dtype=torch.int32, device="cuda")
    tc_chain_into(f, a_pi, a_y, cms[0], part, 0)
    tc_chain_into(f, b_pi, b_y, cms[1], part, 1)
    g = _reduce(f, part, True)
    torch.cuda.synchronize()
    want = ga.double() + gb.double()
    errs = block_errors(c, g, want)
    print("\n" + _fmt("accumulated vs sum", errs))
    for name, (l2, mx) in errs.items():
        assert l2 < 1e-5 and mx < 1e-5, f"block {name}: {l2:.2e} / {mx:.2e}"


@pytest.mark.parametrize("n,w", [(4, 64), (9, 8)])
def test_power_of_two_scale_equivariance_is_exact(built_lib, n, w):
    """S is a power of two derived from max |cotangent|: scaling the cotangents by 2^e scales gradient, dl / S and
    dx / S by exactly 2^e (the fp16 operands are bit-identical)."""
    c = make_case(n, w, 20, False)
    f = Fwd(c)
    d_pi, d_y = synthetic_cotangents(f, seed=3)
    g0, dl0, dx0, _ = tc_chain(f, d_pi, d_y)
    for e in (-40, -8, 8, 40):
        k = 2.0 ** e
        g, dl, dx, cm = tc_chain(f, d_pi * k, d_y * k)
        assert int(cm[1]) == 0
        assert torch.equal(g, g0 * k), f"2^{e}: gradient not exactly scaled"
        assert torch.equal(dl, dl0 * k) and torch.equal(dx, dx0 * k), f"2^{e}: dl / dx not exactly scaled"


def test_cotangent_max_word_pair(built_lib):
    L_, p = _lib(), _lib().ptr
    n, w, L = 9, 8, 33                                        # 2376 tokens: not a multiple of the kernel's grid stride
    R = n * w

    def run(d_pi, d_y, status=0):
        cm = torch.tensor([0x12345, status], dtype=torch.int32, device="cuda")
        L_.call("toued_cotangent_max", p(d_pi), p(d_y), n, w, L, p(cm), L_.stream_ptr())
        torch.cuda.synchronize()
        return int(cm[0].item()) & 0xFFFFFFFF, int(cm[1].item())

    g = torch.Generator(device="cpu").manual_seed(0)
    d_pi, d_y = torch.randn(L, R, generator=g).cuda(), torch.randn(L, R, 8, generator=g).cuda()
    d_y[-1, -1, -1] = -1e3                                     # the maximum at the very last token of d_y_hat
    bits = int(np.float32(1e3).view(np.uint32))
    assert run(d_pi, d_y) == (bits, 0)
    assert run(d_pi, d_y, status=4) == (bits, 4), "status word must be sticky"
    assert run(torch.zeros_like(d_pi), torch.zeros_like(d_y)) == (0, 0)
    assert scale_of(torch.tensor([0, 0])) == 1.0
    for where, v in (("pi", float("nan")), ("pi", float("inf")), ("y", float("-inf")), ("y", float("nan"))):
        a, b = d_pi.clone(), d_y.clone()
        if where == "pi":
            a[L // 2, R - 1] = v
        else:
            b[L - 1, R - 1, 7] = v
        mx, st = run(a, b)
        assert mx == 0x7F800000 and st == STATUS_NONFINITE_COT, f"{where} {v}: max {mx:#x} status {st}"


SATURATION = [
    pytest.param({"Wh": 8.0, "w_pi": 16.0, "W_y": 16.0}, 20, id="Wh8-heads16-L20"),
    pytest.param({"Wh": 4.0, "w_pi": 16.0, "W_y": 16.0}, 64, id="Wh4-heads16-L64"),
    pytest.param({"Wh": 3.0}, 20, id="Wh3-control"),
]


@pytest.mark.parametrize("scale,L", SATURATION)
def test_fp16_saturation_is_reported(built_lib, scale, L):
    """The reverse pass has ~2^12 of headroom over max |cotangent| (tc.cuh).  A chain whose |dh| grows past it must set
    TOUED_STATUS_FP16_RANGE; one that stays far below must not, and must then meet R2.  Never a wrong result with the
    status clear."""
    c = make_case(2, 64, L, False, scale=scale)
    f = Fwd(c, zero_done=True)
    d_pi, d_y = synthetic_cotangents(f, seed=9)
    hidden = []
    fp64_reference(f, d_pi, d_y, hidden=hidden)
    growth = float(max(x.abs().max() for x in hidden) / torch.max(d_pi.abs().max(), d_y.abs().max()).double().cpu())
    h, gates = f.tc_activations()
    g32tc, _, _ = simt_chain(f, d_pi, d_y, h, gates, f.tapes["tc"].y_hat[0])
    gtc, _, _, cm = tc_chain(f, d_pi, d_y)
    st = int(cm[1])
    r2 = block_errors(c, gtc, g32tc)
    ok = not r2_failures(r2)
    print(f"\n[{scale} L={L}] growth max|dh|/max|cot| = {growth:.3g}, status {st}, R2 within tolerance: {ok}\n  " + _fmt("R2", r2))
    if growth > 2.0 ** 14:
        assert st & STATUS_FP16_RANGE, f"growth {growth:.3g} but no saturation status"
    if growth < 2.0 ** 10:
        assert st == 0, f"growth {growth:.3g} but status {st}"
        assert ok, "R2 fails without saturation"
    assert ok or st & STATUS_FP16_RANGE, "wrong tensor-core gradient with the status clear"


@pytest.mark.parametrize("v", [float("nan"), float("inf")])
def test_nonfinite_cotangent_is_never_silent(built_lib, v):
    c = make_case(4, 64, 20, False)
    f = Fwd(c)
    d_pi, d_y = synthetic_cotangents(f, seed=4)
    d_pi[7, 100] = v
    g, _, _, cm = tc_chain(f, d_pi, d_y)
    finite = bool(torch.isfinite(g).all())
    print(f"\n[d_pi_hat = {v}] gradient finite: {finite}, status {int(cm[1])}")
    assert not finite or int(cm[1]) & STATUS_NONFINITE_COT, "finite gradient with the status clear"
    assert int(cm[1]) & STATUS_NONFINITE_COT


def test_nan_input_propagates_through_both_forwards(built_lib):
    """A NaN in one sequence's LPG input row: that sequence's pi_hat / y_hat are non-finite at that step in both
    precisions (as in fp64), every other sequence is bitwise unchanged."""
    c = make_case(4, 64, 20, False)
    f = Fwd(c)
    clean = {k: (t.pi_hat[0].clone(), t.y_hat[0].clone()) for k, t in f.tapes.items()}
    t0, r0 = 11, 133
    for t in f.tapes.values():
        t.x[0][t0, r0, 2] = float("nan")                        # the pi column of token (t0, r0)
    f.run_forward()
    torch.cuda.synchronize()
    other = torch.ones(f.L, f.R, dtype=torch.bool, device="cuda")
    other[:, r0] = False
    for k, t in f.tapes.items():
        pi, y = t.pi_hat[0], t.y_hat[0]
        assert not torch.isfinite(pi[t0, r0]), f"{k}: pi_hat finite after a NaN input"
        assert not torch.isfinite(y[t0, r0]).all(), f"{k}: y_hat finite after a NaN input"
        assert torch.equal(pi[other], clean[k][0][other]) and torch.equal(y[other], clean[k][1][other]), \
            f"{k}: other sequences changed"
    # as in the fp64 oracle (its sequences are [R][L])
    d_pi, d_y = synthetic_cotangents(f, seed=0)
    _, pi64, y64 = fp64_reference(f, d_pi, d_y, nan_at=(t0, r0))
    assert not torch.isfinite(pi64[r0, t0]) and not torch.isfinite(y64[r0, t0]).all()
    assert torch.isfinite(pi64[:r0]).all() and torch.isfinite(pi64[r0 + 1:]).all()
