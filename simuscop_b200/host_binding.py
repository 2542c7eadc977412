"""ctypes binding of libsimuscop_host.so (include/simuscop_host.h): the C++ front end that turns a
reference-style configuration file into the haplotype store and read plan of a device handle."""
import ctypes as C

from . import cuda_binding
from .paths import LIB_HOST

_lib = None


def lib():
    global _lib
    if _lib is None:
        cuda_binding.lib()          # libsimuscop_cuda.so first (the host library links against it)
        L = C.CDLL(LIB_HOST)
        L.ssh_open.argtypes = [C.c_char_p, C.c_uint64, C.POINTER(C.c_void_p)]
        L.ssh_close.argtypes = [C.c_void_p]
        L.ssh_num_samples.argtypes = [C.c_void_p]
        L.ssh_sample_stem.argtypes = [C.c_void_p, C.c_int]
        L.ssh_sample_stem.restype = C.c_char_p
        L.ssh_paired.argtypes = [C.c_void_p]
        L.ssh_read_length.argtypes = [C.c_void_p]
        L.ssh_output_dir.argtypes = [C.c_void_p]
        L.ssh_output_dir.restype = C.c_char_p
        L.ssh_prepare_sample.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_char_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.ssh_write_truth_vcf.argtypes = [C.c_void_p, C.c_int, C.c_char_p]
        L.ssh_run.argtypes = [C.c_void_p, C.c_int]
        _lib = L
    return _lib


class Job:
    def __init__(self, config_path, seed):
        self.j = C.c_void_p()
        rc = lib().ssh_open(config_path.encode(), seed, C.byref(self.j))
        if rc:
            raise RuntimeError("ssh_open failed (%d)" % rc)

    def close(self):
        if self.j:
            lib().ssh_close(self.j)
            self.j = C.c_void_p()

    @property
    def num_samples(self):
        return lib().ssh_num_samples(self.j)

    @property
    def paired(self):
        return bool(lib().ssh_paired(self.j))

    @property
    def read_length(self):
        return lib().ssh_read_length(self.j)

    def prepare(self, sample, gen, dump_path=None):
        """Uploads sample `sample` (haplotype store + plan) into the cuda_binding.Generator `gen`."""
        pp, ep = C.c_int64(), C.c_int64()
        rc = lib().ssh_prepare_sample(self.j, sample, gen.h, dump_path.encode() if dump_path else None,
                                      C.byref(pp), C.byref(ep))
        if rc:
            raise cuda_binding.SscError("ssh_prepare_sample failed (%d): %s" % (
                rc, cuda_binding.lib().ssc_last_error().decode(errors="replace")))
        gen.planned, gen.emitted = pp.value, ep.value
        return pp.value, ep.value

    def write_truth_vcf(self, sample, path):
        """Writes the truth VCF of `sample` (after prepare() of that sample) to `path`."""
        rc = lib().ssh_write_truth_vcf(self.j, sample, path.encode())
        if rc:
            raise RuntimeError("ssh_write_truth_vcf failed (%d)" % rc)
