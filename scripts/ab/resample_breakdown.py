#!/usr/bin/env python
"""Builds of an older commit's library (the whole-pool resampling event) whose instrumented kernel times other
sub-phases of the event in the timer slots, for scripts/gpu_resample.sh:
  python scripts/ab/resample_breakdown.py COMMIT      -> build/ab/lib_parent_t{A,B,C}.so
  tA: [4] plan + barrier, [5] row maps, [7] clear pass + barrier
  tB: [4] recount + barrier, [5] mark pass + barrier, [7] rebuild scan + barrier
  tC: no event sub-phases; [7] the P-CTAs' redone propose + commit; on the E-CTAs in the phase after an event,
      [5] the evaluation (its free-id cache empty) and [4] the refill after it
Needs the current tree built (the group and wide cubins are embedded as they are)."""
import os
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
PKG = os.path.join(ROOT, "particlemdi.jl_b200")


def variants(src):
    clear_sync = ("    for (int sl = threadIdx.x; sl < ns; sl += PMDI_NT) T.lw_s[sl] = 1.0;  // logweight .= 1.0 "
                  "(src/pmdi.jl:319)\n  if (!spec_gsync(sp, sm)) return false;\n")
    recount_sync = ("  if (gt == 0) {\n    *sp.gcnt = 0;\n    for (int k = 0; k < K; ++k) __stcg(sp.pd[k].ctr + 1, 0);\n  }\n"
                    "  if (!spec_gsync(sp, sm)) return false;\n")
    mark_sync = ("      __stcg(pd.mark + ldcg_info(pd.info + (size_t)(parn ^ 1) * pd.cap + c).z, 1);\n    }\n  }\n"
                 "  if (!spec_gsync(sp, sm)) return false;\n")
    final7 = "  if (!spec_xsync(sp, sm)) return false;  // no rank recycles a row while a peer may still be pulling it\n  RS_MARK(7)\n"
    redo = "          for (int u = warp; u < nu; u += NW) spec_commit<DBG, GRP>(sp, sm, T, u, t, ns);\n        }\n"
    ev = ("      if (t + 1 < steps) spec_eval<DBG>(sp, sm, T, e, t + 1, xring, obs_ok, t - 1);\n      PHASE_MARK(1)\n"
          "      SWEEP_TRACE(t, 52)\n      spec_refill(sp, sm, T);\n")
    e_res = "          if (!spec_resample<GRP>(sp, sm, T, ns, t - 1, s_tmp, false, e)) return;\n          PHASE_MARK(6)\n"
    for s in (clear_sync, recount_sync, mark_sync, final7, redo, ev, e_res):
        assert src.count(s) == 1, s[:60]
    a = src.replace(clear_sync, clear_sync + "  RS_MARK(7)\n").replace(final7, final7.replace("  RS_MARK(7)\n", ""))
    b = src.replace("  RS_MARK(4)\n", "").replace("  RS_MARK(5)\n", "")
    b = (b.replace(clear_sync, clear_sync + "  if (tm) t_ = globaltimer_ns();\n")
          .replace(recount_sync, recount_sync + "  RS_MARK(4)\n").replace(mark_sync, mark_sync + "  RS_MARK(5)\n"))
    c = src.replace("  const bool tm = sp.phase_ns != nullptr && threadIdx.x == 0;", "  const bool tm = false;")
    c = c.replace(redo, redo.replace("        }\n", "          PHASE_MARK(7)\n        }\n"))
    c = c.replace(ev, "      if (t + 1 < steps) spec_eval<DBG>(sp, sm, T, e, t + 1, xring, obs_ok, t - 1);\n"
                      "      if (after_ev) { PHASE_MARK(5) } else { PHASE_MARK(1) }\n      spec_refill(sp, sm, T);\n"
                      "      if (after_ev) { PHASE_MARK(4) }\n      after_ev = false;\n")
    c = c.replace(e_res, e_res + "          after_ev = true;\n")
    c = c.replace("  int obs_ok = -1;\n", "  int obs_ok = -1;\n  bool after_ev = false;\n")
    return {"tA": a, "tB": b, "tC": c}


def main():
    commit = sys.argv[1]
    out = os.path.join(ROOT, "build", "ab")
    os.makedirs(out, exist_ok=True)
    with tempfile.TemporaryDirectory() as tmp:
        arch = subprocess.run(["git", "-C", ROOT, "archive", commit, "particlemdi.jl_b200/csrc", "include"],
                              check=True, capture_output=True).stdout
        subprocess.run(["tar", "-x", "-C", tmp], input=arch, check=True)
        csrc = os.path.join(tmp, "particlemdi.jl_b200", "csrc")
        shutil.copy(os.path.join(PKG, "csrc", "pmdi_embedded.inc"), csrc)
        src = open(os.path.join(csrc, "spec_kernel.cuh")).read()
        procs = []
        for name, text in variants(src).items():
            d = os.path.join(tmp, name)
            shutil.copytree(os.path.join(tmp, "particlemdi.jl_b200"), os.path.join(d, "particlemdi.jl_b200"))
            shutil.copytree(os.path.join(tmp, "include"), os.path.join(d, "include"))
            vc = os.path.join(d, "particlemdi.jl_b200", "csrc")
            open(os.path.join(vc, "spec_kernel.cuh"), "w").write(text)
            procs.append(subprocess.Popen(
                ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler",
                 "-fPIC", "-shared", f'-DPMDI_GROUP_CUBIN="{os.path.join(PKG, "pmdi_spec_group.cubin")}"',
                 f'-DPMDI_WIDE_CUBIN="{os.path.join(PKG, "pmdi_sweep_wide.cubin")}"',
                 "-o", os.path.join(out, f"lib_parent_{name}.so"), os.path.join(vc, "pmdi_cuda.cu")]))
        if any(p.wait() for p in procs):
            sys.exit("a build failed")
    print("built", ", ".join(f"build/ab/lib_parent_{n}.so" for n in ("tA", "tB", "tC")))


if __name__ == "__main__":
    main()
