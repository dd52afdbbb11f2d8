"""Diagnostic (not a pytest file): checksum the outputs of one BASELINE-size tensor-core meta-gradient step.

    TOUED_LIB_VARIANT=<variant> python tests/diag_probe.py [--poison nan|big|rand] [n_agents]

Used with the schedule-fuzz library variant (csrc/build.py::VARIANTS) to show that the warp-specialised kernels give
bit-identical results whatever the relative progress of their warps, and with --poison to show that no kernel reads
uninitialised workspace memory (the caching allocator's free blocks are filled with a pattern before the workspaces
are allocated)."""
import hashlib
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from diag_nondeterminism import run  # noqa: E402
from helpers import Case  # noqa: E402


def sha(t):
    return hashlib.sha1(t.detach().contiguous().cpu().numpy().tobytes()).hexdigest()[:12]


def main():
    args = sys.argv[1:]
    poison = None
    if "--poison" in args:
        i = args.index("--poison")
        poison = args[i + 1]
        del args[i:i + 2]
    n = int(args[0]) if args else 512
    if poison:
        blocks = []
        for _ in range(40):                                     # 40 GiB of cached blocks with a pattern
            b = torch.empty(256 * 1024 * 1024, dtype=torch.int32, device="cuda")
            if poison == "nan":
                b.fill_(0x7FC00000)
            elif poison == "big":
                b.view(torch.float32).fill_(1e30)
            else:
                b.random_(-2 ** 31, 2 ** 31 - 1)
            blocks.append(b)
        del blocks, b                                           # back to the caching allocator, contents intact
        torch.cuda.synchronize()
    c = Case("all_shortlife", n=n, seed=3)
    out, cache = run(c, 5, 2)
    g = out[3]["_grad"]
    tapes = [ws.tape for ws in cache.values()]
    print(f"variant={os.environ.get('TOUED_LIB_VARIANT', '') or 'production'} poison={poison} "
          f"grad={sha(g)} finite={bool(torch.isfinite(g).all())} |g|={float(g.norm()):.6e} "
          f"pi_hat={sha(torch.stack([t.pi_hat for t in tapes]))} actor={sha(out[1].actor_state.params)}", flush=True)


if __name__ == "__main__":
    main()
