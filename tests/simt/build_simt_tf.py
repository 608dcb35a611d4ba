"""Builds tests/simt/_build/libapk_simt_tf.so: the device part of astrild_b200/csrc/tf.cu (moment tile kernel, combine)
and the brick partition kernels of deposit_sorted.cu, unchanged, compiled by g++ against tests/simt/simt.h with the
helpers of build_simt.py.  Tests only."""
import os

import build_simt as bs


def tf_device_part(path: str) -> str:
    """tf.cu without its host code and C entry points (everything from ``using namespace apk;`` on); the dynamic shared
    memory declaration points at the emulator's buffer."""
    text = open(path).read()
    text = text[:text.index("using namespace apk;")]
    assert text.count(bs.DYN_SMEM_DECL) == 1
    return text.replace(bs.DYN_SMEM_DECL, "unsigned char *smem_raw = simt::dyn_smem;")


def build_tf(force: bool = False) -> str:
    """-> tests/simt/_build/libapk_simt_tf.so (NGP partition, tf_moment_tile_kernel, tf_combine_kernel on CPU fibers)"""
    so = os.path.join(bs.OUT_DIR, "libapk_simt_tf.so")
    srcs = [os.path.join(bs.CSRC, f) for f in ("tf.cu", "deposit_sorted.cu", "brick_common.cuh", "apk_common.cuh",
                                               "deposit_common.cuh")]
    srcs += [os.path.join(bs.HERE, f) for f in ("simt.h", "tf_host.cpp", "build_simt.py", "build_simt_tf.py")]
    if not force and bs._fresh(so, srcs):
        return so
    os.makedirs(bs.OUT_DIR, exist_ok=True)
    with open(os.path.join(bs.OUT_DIR, "deposit_sorted_kernels.inc"), "w") as f:
        f.write(bs.device_part(srcs[1]))
    with open(os.path.join(bs.OUT_DIR, "tf_kernels.inc"), "w") as f:
        f.write(tf_device_part(srcs[0]))
    return bs._gxx("tf_host.cpp", bs.OUT_DIR, so)


if __name__ == "__main__":
    print(build_tf(force=True))
