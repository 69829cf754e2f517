"""Roofline figures of gp_var_toeplitz_kernel (DESIGN.md section 4.2c), from the shapes and a measured phase time.

bench.py's roofline block still counts the N^2 M flop of gp_var_kernel's forward substitution, which the recurrence does
not do; its `achieved` and `frac` are no longer a share of anything.  The two honest bounds of the recurrence are:
  - HBM: the packed factor (tiles_in_lower(nt) * 512 bytes per window) is read once by the back substitution;
  - FP64 pipe: 4 FMA per factor entry pair and right-hand side of the back substitution, 3 n FMA per chain point.
With --grouped, the shared-covariance path (DESIGN.md section 4.2d) instead: one window's factor and recurrence for the
whole batch, and per member the forward solve for z (one FMA per factor entry), the back substitution for alpha (one
right-hand side) and n FMA per chain point for the mean; HBM carries y in and mean, variance, LML and status out.  The
members of a CTA (TG_WARPS of them) share one shared-memory copy of each tile column, so L2 delivers the factor twice
(z, alpha) per member CTA, plus the L_jj tiles with the z pass.  --ms is then the step time (fit and variance phases together: the member kernel does both).
Usage: python tools/var_toeplitz_roofline.py --ms <variance phase ms> [--B 4096 --N 256 --M 600] [--grouped]
       [--hbm-tbs 7.7] [--fp64-tflops 33.9]   (data-sheet HBM bandwidth; DFMA issue peak of profiles/fp64_peak_r01.json)"""
import argparse
import json


def figures(B, N, M, ms, hbm_tbs, fp64_tflops):
    nt = (N + 7) // 8
    tiles = nt * (nt + 1) // 2
    factor_bytes = tiles * 512 * B
    chain = M + 1 if M > 0 else 0                 # the benchmark grid x_{N-1} + 1 + j: chain from m0 = N - 1
    fma_back = tiles * 64 * 2 * B                 # two right-hand sides, one FMA per factor entry each
    fma_chain = 3 * N * chain * B
    fma = fma_back + fma_chain
    t = ms * 1e-3
    return {
        "B": B, "N": N, "M": M, "phase_ms": ms,
        "factor_bytes": factor_bytes, "hbm_tb_per_s": factor_bytes / t * 1e-12,
        "hbm_frac": factor_bytes / t * 1e-12 / hbm_tbs,
        "fma": fma, "fp64_tflops": 2 * fma / t * 1e-12, "fp64_frac": 2 * fma / t * 1e-12 / fp64_tflops,
        "lower_bound_ms": 1e3 * max(factor_bytes / (hbm_tbs * 1e12), 2 * fma / (fp64_tflops * 1e12)),
    }


TG_WARPS = 8   # members per CTA of gp_toep_member_kernel


def grouped_figures(B, N, M, ms, hbm_tbs, fp64_tflops):
    nt = (N + 7) // 8
    tiles = nt * (nt + 1) // 2
    chain = M + 1 if M > 0 else 0
    one = tiles * 64 * 2 + 3 * N * chain                        # the group's own back substitution and recurrence
    member = tiles * 64 + tiles * 64 + N * chain                # z, alpha, the mean
    fma = one + member * B
    hbm_bytes = tiles * 512 + B * (8 * N + 16 * M + 12)         # one factor; y in; mean, variance, LML, status out
    t = ms * 1e-3
    return {
        "B": B, "N": N, "M": M, "step_ms": ms, "grouped": True,
        "hbm_bytes": hbm_bytes, "hbm_tb_per_s": hbm_bytes / t * 1e-12, "hbm_frac": hbm_bytes / t * 1e-12 / hbm_tbs,
        "l2_factor_bytes": (tiles * 2 + nt) * 512 * -(-B // TG_WARPS),   # twice per member CTA, L_jj once
        "fma": fma, "fp64_tflops": 2 * fma / t * 1e-12, "fp64_frac": 2 * fma / t * 1e-12 / fp64_tflops,
        "lower_bound_ms": 1e3 * max(hbm_bytes / (hbm_tbs * 1e12), 2 * fma / (fp64_tflops * 1e12)),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ms", type=float, required=True)
    ap.add_argument("--B", type=int, default=4096)
    ap.add_argument("--N", type=int, default=256)
    ap.add_argument("--M", type=int, default=600)
    ap.add_argument("--hbm-tbs", type=float, default=7.7)
    ap.add_argument("--fp64-tflops", type=float, default=33.9)
    ap.add_argument("--grouped", action="store_true")
    a = ap.parse_args()
    f = grouped_figures if a.grouped else figures
    print(json.dumps(f(a.B, a.N, a.M, a.ms, a.hbm_tbs, a.fp64_tflops), indent=1))


if __name__ == "__main__":
    main()
