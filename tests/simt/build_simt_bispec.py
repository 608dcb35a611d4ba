"""Builds tests/simt/_build/libapk_simt_bispec.so: the device part of astrild_b200/csrc/bispec.cu (shell fill,
triple-product reduction in float32 and float64, fold), unchanged, compiled by g++ against tests/simt/simt.h with the
helpers of build_simt.py.  Tests only."""
import os

import build_simt as bs


def bispec_device_part(path: str) -> str:
    """bispec.cu without its host code and C entry points (everything from ``using namespace apk;`` on); the dynamic
    shared memory declaration points at the emulator's buffer, and APK_SIMT selects plain copies for cp.async."""
    text = open(path).read()
    text = text[:text.index("using namespace apk;")]
    assert text.count(bs.DYN_SMEM_DECL) == 1
    return text.replace(bs.DYN_SMEM_DECL, "unsigned char *smem_raw = simt::dyn_smem;")


def build_bispec(force: bool = False) -> str:
    """-> tests/simt/_build/libapk_simt_bispec.so (bk_fill_kernel, bk_reduce_kernel<float/double>, bk_fold_kernel on
    CPU fibers)"""
    so = os.path.join(bs.OUT_DIR, "libapk_simt_bispec.so")
    srcs = [os.path.join(bs.CSRC, f) for f in ("bispec.cu", "apk_common.cuh")]
    srcs += [os.path.join(bs.HERE, f) for f in ("simt.h", "bispec_host.cpp", "build_simt.py", "build_simt_bispec.py")]
    if not force and bs._fresh(so, srcs):
        return so
    os.makedirs(bs.OUT_DIR, exist_ok=True)
    with open(os.path.join(bs.OUT_DIR, "bispec_kernels.inc"), "w") as f:
        f.write(bispec_device_part(srcs[0]))
    return bs._gxx("bispec_host.cpp", bs.OUT_DIR, so)


if __name__ == "__main__":
    print(build_bispec(force=True))
