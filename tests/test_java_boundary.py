"""The Java side of the drop-in boundary (java/net/preibisch/simulation/gpu/*.java, jni/mvsim_jni.c) without a JDK:

  * every `static native` method of Mvsim.java has a stub Java_net_preibisch_simulation_gpu_Mvsim_<name> in jni/mvsim_jni.c
    with the same number of parameters (+ JNIEnv*, jclass), and vice versa;
  * jni/mvsim_jni.c compiles warning-free against a stand-in <jni.h> (tests/jni_stub) and include/mvsim.h -- i.e. every call
    into the C ABI has the header's arity and types -- and links against libmvsim.so with no undefined symbol;
  * every mvsim_* function the stubs call is declared in include/mvsim.h and exported by libmvsim.so;
  * the facades carry the reference's public static signatures (S/SimulateMultiViewDataset.java:80,104,181,195,233,253,318 and
    S/Tools.java:73,112,143) verbatim -- REFERENCE_SIGNATURES holds those lines of the reference -- and no body is elided.
"""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
JAVA = os.path.join(ROOT, "java", "net", "preibisch", "simulation", "gpu")
JNI_C = os.path.join(ROOT, "jni", "mvsim_jni.c")
HEADER = os.path.join(ROOT, "include", "mvsim.h")
LIB = os.path.join(ROOT, "multiview-simulation_b200", "libmvsim.so")


def _strip_comments(src):
    src = re.sub(r"/\*.*?\*/", " ", src, flags=re.S)
    return re.sub(r"//[^\n]*", " ", src)


def _split_args(arglist):
    arglist = arglist.strip()
    if not arglist or arglist == "void":
        return []
    depth, cur, out = 0, "", []
    for ch in arglist.replace("->", "."):
        if ch in "(<[":
            depth += 1
        elif ch in ")>]":
            depth -= 1
        if ch == "," and depth == 0:
            out.append(cur.strip())
            cur = ""
        else:
            cur += ch
    out.append(cur.strip())
    return out


def java_natives():
    src = _strip_comments(open(os.path.join(JAVA, "Mvsim.java")).read())
    return {m.group(1): _split_args(m.group(2)) for m in re.finditer(r"static\s+native\s+[\w\[\]<>]+\s+(\w+)\s*\(([^)]*)\)\s*;", src)}


def jni_stubs():
    src = _strip_comments(open(JNI_C).read())
    return {m.group(1): _split_args(m.group(2)) for m in re.finditer(r"MVSIM_JNI\(\s*\w+\s*,\s*(\w+)\s*\)\s*\(([^)]*)\)", src)}


def header_prototypes():
    src = _strip_comments(open(HEADER).read())
    return {m.group(1): _split_args(m.group(2)) for m in re.finditer(r"\b(mvsim_\w+)\s*\(([^;{]*?)\)\s*;", src)}


def test_every_native_method_has_a_stub_of_matching_arity():
    natives, stubs = java_natives(), jni_stubs()
    assert len(natives) >= 20
    assert set(natives) == set(stubs)
    for name, params in natives.items():
        assert len(stubs[name]) == len(params) + 2, (name, params, stubs[name])      # + JNIEnv*, jclass
        assert stubs[name][0].startswith("JNIEnv") and stubs[name][1].startswith("jclass")
    # Java type -> JNI type, position by position
    jmap = {"int": "jint", "long": "jlong", "float": "jfloat", "double": "jdouble", "boolean": "jboolean", "long[]": "jlongArray", "int[]": "jintArray",
            "double[]": "jdoubleArray", "FloatBuffer": "jobject", "ByteBuffer": "jobject", "Buffer": "jobject", "FloatBuffer[]": "jobjectArray"}
    for name, params in natives.items():
        for jp, cp in zip(params, stubs[name][2:]):
            assert cp.split()[0] == jmap[jp.replace("final ", "").split()[0]], (name, jp, cp)


def test_stubs_call_the_c_abi_with_the_headers_arity():
    protos = header_prototypes()
    src = _strip_comments(open(JNI_C).read())
    called = {}
    for m in re.finditer(r"\b(mvsim_[a-z_0-9]+)\s*\(", src):
        name = m.group(1)
        if name in ("mvsim_ctx", "mvsim_view_params"):
            continue
        depth, i = 1, m.end()
        while depth:
            depth += {"(": 1, ")": -1}.get(src[i], 0)
            i += 1
        called.setdefault(name, []).append(_split_args(src[m.end():i - 1]))
    assert len(called) >= 20
    exported = subprocess.run(["nm", "-D", "--defined-only", LIB], capture_output=True, text=True, check=True).stdout
    for name, calls in called.items():
        assert name in protos, f"{name} is not declared in include/mvsim.h"
        assert re.search(rf"\bT {name}\b", exported), f"{name} is not exported by libmvsim.so"
        for args in calls:
            assert len(args) == len(protos[name]), (name, args, protos[name])
    # the path's entry points are all bound
    for need in ("mvsim_axis_rotation", "mvsim_rotate_axis", "mvsim_attenuate", "mvsim_psf_normalize", "mvsim_convolve", "mvsim_adjust",
                 "mvsim_extract_slices", "mvsim_poisson", "mvsim_simulate_view", "mvsim_simulate_views", "mvsim_alloc_pinned", "mvsim_free_pinned"):
        assert need in called, need


def test_stubs_compile_against_the_header_and_link_against_the_library(tmp_path):
    out = tmp_path / "libmvsim_jni_check.so"
    cmd = ["gcc", "-std=c11", "-Wall", "-Wextra", "-Werror", "-shared", "-fPIC", "-I", os.path.join(ROOT, "tests", "jni_stub"), "-I", os.path.join(ROOT, "include"),
           JNI_C, "-L", os.path.dirname(LIB), "-lmvsim", "-Wl,--no-undefined", "-o", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    syms = subprocess.run(["nm", "-D", "--defined-only", str(out)], capture_output=True, text=True, check=True).stdout
    for name in java_natives():
        assert f"Java_net_preibisch_simulation_gpu_Mvsim_{name}" in syms


# the reference's signatures, normalised to single spaces (file:line in the reference)
REFERENCE_SIGNATURES = {
    "SimulateMultiViewDatasetGPU.java": [
        ("SimulateMultiViewDataset.java", 80, "public static AffineModel3D axisRotation( final Interval in, final int axis, final int degrees )"),
        ("SimulateMultiViewDataset.java", 104, "public static Img< FloatType > rotateAroundAxis( final RandomAccessibleInterval< FloatType > in, final int axis, final int degrees )"),
        ("SimulateMultiViewDataset.java", 181, "public static Img< FloatType > extractSlices( final RandomAccessibleInterval< FloatType > randomAccessible, final int inc, final float poissonSNR )"),
        ("SimulateMultiViewDataset.java", 195, "public static Img< FloatType > extractSlices( final RandomAccessibleInterval< FloatType > randomAccessible, final int inc, final float poissonSNR, final Random rnd )"),
        ("SimulateMultiViewDataset.java", 233, "public static Img< FloatType > poissonProcess( final RandomAccessibleInterval< FloatType > in, final float poissonSNR, final Random rnd )"),
        ("SimulateMultiViewDataset.java", 253, "public static Img< FloatType > convolve( final Img< FloatType > img, final Img< FloatType > psf, final ExecutorService service )"),
        ("SimulateMultiViewDataset.java", 318, "public static Img< FloatType > attenuate3d( final RandomAccessibleInterval< FloatType > randomAccessible, final double delta )"),
    ],
    "ToolsGPU.java": [
        ("Tools.java", 73, "public static void poissonProcess( final RandomAccessibleInterval< FloatType > img, final double SNR, final Random rnd )"),
        ("Tools.java", 112, "final public static void normImage( final Iterable< FloatType > img )"),
        ("Tools.java", 143, "public static double adjustImage( final IterableInterval< FloatType > image, final float minValue, final float targetAverage )"),
    ],
}


def _norm(s):
    s = re.sub(r"\s+", " ", s.strip())
    s = re.sub(r"<\s*", "< ", s)
    s = re.sub(r"\s*>", " >", s)
    return re.sub(r"\s+", " ", s)


def test_facades_carry_the_references_signatures_and_complete_bodies():
    for fname, sigs in REFERENCE_SIGNATURES.items():
        src = open(os.path.join(JAVA, fname)).read()
        flat = _norm(src)
        for _, _, sig in sigs:
            assert _norm(sig) in flat, f"{fname}: missing {sig}"
        # no elided bodies: no comment-only or empty method bodies, no "..." placeholders
        code = _strip_comments(src)
        assert "..." not in code
        assert not re.search(r"\)\s*\{\s*\}", code.replace("private Mvsim() {}", "")), f"{fname}: empty method body"
    # the generic (cursor-copy) path for views such as Views.zeroMin( Views.interval( con, min, max ) ) (S/SimulateTileStitching.java:153)
    facade = open(os.path.join(JAVA, "SimulateMultiViewDatasetGPU.java")).read()
    assert "Views.flatIterable( rai ).cursor()" in facade and "getCurrentStorageArray()" in facade
    for fused in ("public static Img< FloatType > simulateView(", "public static List< Img< FloatType > > simulateViews("):
        assert fused in facade
    # every native used by the facades exists
    natives = java_natives()
    for fname in REFERENCE_SIGNATURES:
        for m in re.finditer(r"Mvsim\.(\w+)\s*\(", _strip_comments(open(os.path.join(JAVA, fname)).read())):
            assert m.group(1) in natives or m.group(1) in ("pinnedFloats",), m.group(1)


def test_java_sources_are_balanced():
    """Cheap syntax guard (no javac here): braces / parentheses balance and every statement-level line ends properly."""
    for fname in os.listdir(JAVA):
        code = _strip_comments(open(os.path.join(JAVA, fname)).read())
        code = re.sub(r'"(\\.|[^"\\])*"', '""', code)
        for a, b in ("{}", "()", "[]"):
            assert code.count(a) == code.count(b), (fname, a, code.count(a), code.count(b))
        assert re.search(r"^package net\.preibisch\.simulation\.gpu;", code.strip(), flags=re.M)
