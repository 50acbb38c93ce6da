#!/usr/bin/env python3
"""Build the UNMODIFIED reference HiGHS (CPU pdlp = vendored cuPDLP-C) into oracle/_ref/.

TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is on the product path.

This is our own recipe, not the reference's build system: it reads the source
*lists* from /root/reference/cmake/sources.cmake, writes a hand-made HConfig.h
(the only "generated" header; it is six #defines) into oracle/_ref/include, and
compiles every translation unit where it lies under /root/reference with
gcc/g++ -O3 through a ninja file that this script emits.  No reference source is
copied into this repository; the outputs (objects, libhighs_ref.so,
ref_driver) live only in oracle/_ref/, which is git-ignored but travels to the
GPU box with the gpurun snapshot.

Usage:  python oracle/build_ref.py            # build lib + driver (idempotent)
        python oracle/build_ref.py --force
The GPU box has no /root/reference: there the prebuilt oracle/_ref/ is used.
"""
import os
import re
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("HIGHS_REFERENCE", "/root/reference")
OUT = os.path.join(HERE, "_ref")

# lists that make up the default (`sources`) library: highs/CMakeLists.txt:7
LISTS = ["highs_sources", "cupdlp_sources", "ipx_sources", "basiclu_sources",
         "hipo_sources", "factor_highs_sources", "hipo_util_sources"]

INCLUDE_SUBDIRS = ["extern", "highs", "highs/interfaces", "highs/io", "highs/io/filereader",
                   "highs/ipm", "highs/ipm/ipx", "highs/ipm/basiclu", "highs/lp_data",
                   "highs/mip", "highs/model", "highs/parallel", "highs/pdlp",
                   "highs/pdlp/cupdlp", "highs/pdlp/hipdlp", "highs/presolve",
                   "highs/qpsolver", "highs/simplex", "highs/test_kkt", "highs/util",
                   "highs/hipo", "highs/hipo/auxiliary", "highs/hipo/factorhighs",
                   "highs/hipo/ipm"]

HCONFIG = """#ifndef HCONFIG_H_
#define HCONFIG_H_
/* hand-written for the oracle build (oracle/build_ref.py); mirrors a Release,
 * FAST_BUILD, CUPDLP_CPU, 32-bit HighsInt configuration of HConfig.h.in */
#define FAST_BUILD
#define CUPDLP_CPU
#define HIGHS_SHARED_EXTRAS_LIBRARY /* extras (HiPO orderings) dlopen()ed if present; unused by pdlp */
#define CMAKE_BUILD_TYPE "Release"
#define HIGHS_HAVE_MM_PAUSE
#define HIGHS_HAVE_BUILTIN_CLZ
#define HIGHS_GITHASH "oracle"
#define HIGHS_VERSION_MAJOR 1
#define HIGHS_VERSION_MINOR 15
#define HIGHS_VERSION_PATCH 1
#endif
"""


def parse_lists(path):
    txt = open(path).read()
    out = {}
    for m in re.finditer(r"set\((\w+)\s+([^)]*)\)", txt):
        name, body = m.group(1), m.group(2)
        out[name] = [t for t in body.split() if not t.startswith("#")]
    return out


def main():
    force = "--force" in sys.argv
    lib = os.path.join(OUT, "libhighs_ref.so")
    drv = os.path.join(OUT, "ref_driver")
    if not os.path.isdir(REF):
        if os.path.exists(lib):
            print("oracle/_ref: reference tree absent, using prebuilt", lib)
            return 0
        print("oracle/_ref: no reference tree and no prebuilt library", file=sys.stderr)
        return 1
    os.makedirs(os.path.join(OUT, "include"), exist_ok=True)
    os.makedirs(os.path.join(OUT, "obj"), exist_ok=True)
    hc = os.path.join(OUT, "include", "HConfig.h")
    if not os.path.exists(hc) or open(hc).read() != HCONFIG:
        open(hc, "w").write(HCONFIG)
    lists = parse_lists(os.path.join(REF, "cmake", "sources.cmake"))
    srcs = []
    for l in LISTS:
        for s in lists.get(l, []):
            if s.endswith((".c", ".cc", ".cpp")):
                p = os.path.join(REF, "highs", s)
                if os.path.exists(p):
                    srcs.append(p)
    incs = " ".join("-I" + os.path.join(REF, d) for d in INCLUDE_SUBDIRS)
    incs += " -I" + os.path.join(OUT, "include")
    common = "-O3 -DNDEBUG -fPIC -w " + incs
    nj = [
        "cxx = g++", "cc = gcc",
        f"cxxflags = -std=c++11 {common}",
        f"cflags = {common} -Wno-implicit-function-declaration",
        "rule cxx\n  command = $cxx $cxxflags -MMD -MF $out.d -c $in -o $out\n  depfile = $out.d\n  deps = gcc",
        "rule cc\n  command = $cc $cflags -MMD -MF $out.d -c $in -o $out\n  depfile = $out.d\n  deps = gcc",
        "rule link\n  command = g++ -shared -o $out $in -lpthread -lm -ldl",
        "rule exe\n  command = g++ -std=c++11 -O2 $cxxincs $in -o $out -L$libdir -lhighs_ref '-Wl,-rpath,$$ORIGIN' -lpthread",
    ]
    objs = []
    for s in srcs:
        o = os.path.join(OUT, "obj", os.path.relpath(s, REF).replace("/", "_") + ".o")
        objs.append(o)
        nj.append(f"build {o}: {'cc' if s.endswith('.c') else 'cxx'} {s}")
    nj.append(f"build {lib}: link {' '.join(objs)}")
    nj.append(f"build {drv}: exe {os.path.join(HERE, 'ref_driver.cpp')} | {lib}\n"
              f"  cxxincs = {incs} -w\n  libdir = {OUT}")
    # --- drop-in demonstration (INTEGRATION.md): the same objects MINUS the reference wrapper
    # (CupdlpWrapper.cpp), PLUS highs_b200/csrc/highs_shim.cpp, linked against libb200pdlp.so.
    shim_src = os.path.join(os.path.dirname(HERE), "highs_b200", "csrc", "highs_shim.cpp")
    eng_dir = os.path.join(os.path.dirname(HERE), "highs_b200")
    lib2 = os.path.join(OUT, "libhighs_b200.so")
    drv2 = os.path.join(OUT, "ref_driver_b200")
    shim_o = os.path.join(OUT, "obj", "highs_shim.o")
    # (the vendored cuPDLP-C objects stay in the library only because HiPDLP -- solver=hipdlp -- uses
    #  their logging utilities, e.g. debugPdlpRestartLog; nothing on the solver=pdlp path calls them)
    keep = [o for o, s_ in zip(objs, srcs) if not s_.endswith("pdlp/CupdlpWrapper.cpp")]
    nj.append("rule cxxshim\n  command = g++ -std=c++11 $cxxflags_shim -c $in -o $out")
    nj.append(f"build {shim_o}: cxxshim {shim_src}\n  cxxflags_shim = {common} -I{os.path.join(os.path.dirname(HERE), 'include')}")
    # the engine is found relative to oracle/_ref/ (not by absolute path), so a tree copied elsewhere still runs; an oracle/_ref/
    # reached through a symlink needs oracle.binding.driver_env() (LD_LIBRARY_PATH), since $ORIGIN resolves symlinks
    nj.append("rule linkshim\n  command = g++ -shared -o $out $in -L$engdir -lb200pdlp '-Wl,-rpath,$$ORIGIN/../../highs_b200' -lpthread -lm -ldl")
    nj.append(f"build {lib2}: linkshim {' '.join(keep)} {shim_o}\n  engdir = {eng_dir}")
    nj.append("rule exeshim\n  command = g++ -std=c++11 -O2 $cxxincs $in -o $out -L$libdir -lhighs_b200 -L$engdir -lb200pdlp '-Wl,-rpath,$$ORIGIN' '-Wl,-rpath,$$ORIGIN/../../highs_b200' -lpthread")
    nj.append(f"build {drv2}: exeshim {os.path.join(HERE, 'ref_driver.cpp')} | {lib2}\n"
              f"  cxxincs = {incs} -w\n  libdir = {OUT}\n  engdir = {eng_dir}")
    # --- the same with the HiPDLP wrapper replaced as well (solver=hipdlp -> the engine's Halpern mode); kept in a THIRD
    # library so that the validated solver=pdlp drop-in above is untouched while the HiPDLP device mode is unvalidated
    shim2_src = os.path.join(os.path.dirname(HERE), "highs_b200", "csrc", "highs_shim_hipdlp.cpp")
    shim2_o = os.path.join(OUT, "obj", "highs_shim_hipdlp.o")
    lib3 = os.path.join(OUT, "libhighs_b200_hipdlp.so")
    drv3 = os.path.join(OUT, "ref_driver_b200_hipdlp")
    keep3 = [o for o, s_ in zip(objs, srcs) if not s_.endswith("pdlp/CupdlpWrapper.cpp") and not s_.endswith("pdlp/HiPdlpWrapper.cpp")]
    nj.append(f"build {shim2_o}: cxxshim {shim2_src}\n  cxxflags_shim = {common} -I{os.path.join(os.path.dirname(HERE), 'include')}")
    nj.append(f"build {lib3}: linkshim {' '.join(keep3)} {shim_o} {shim2_o}\n  engdir = {eng_dir}")
    nj.append("rule exeshim3\n  command = g++ -std=c++11 -O2 $cxxincs $in -o $out -L$libdir -lhighs_b200_hipdlp -L$engdir -lb200pdlp '-Wl,-rpath,$$ORIGIN' '-Wl,-rpath,$$ORIGIN/../../highs_b200' -lpthread")
    nj.append(f"build {drv3}: exeshim3 {os.path.join(HERE, 'ref_driver.cpp')} | {lib3}\n"
              f"  cxxincs = {incs} -w\n  libdir = {OUT}\n  engdir = {eng_dir}")
    if "--shim" in sys.argv and os.path.exists(os.path.join(eng_dir, "libb200pdlp.so")):
        nj.append(f"default {lib} {drv} {lib2} {drv2} {lib3} {drv3}")
    else:
        nj.append(f"default {lib} {drv}")
    njp = os.path.join(OUT, "build.ninja")
    open(njp, "w").write("\n".join(nj) + "\n")
    if force:
        subprocess.call(["ninja", "-f", njp, "-t", "clean"], cwd=OUT)
    return subprocess.call(["ninja", "-f", njp], cwd=OUT)


if __name__ == "__main__":
    sys.exit(main())
