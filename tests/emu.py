"""ctypes handle on tests/cpu_emu/libemu.so (TEST-ONLY host emulation of the kernels' loops)."""
import ctypes as C
import os
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
dp = C.POINTER(C.c_double)


class Emu:
    def __init__(self, cfg):
        self.lib = C.CDLL(os.path.join(HERE, "cpu_emu", "libemu.so"))
        self.lib.emu_error.restype = C.c_char_p
        self.lib.emu_set_radius.argtypes = [C.c_double]
        self.lib.emu_set_cloudtop.argtypes = [C.c_double]
        self.lib.emu_set_scattering.argtypes = [C.c_int, C.c_double]
        if self.lib.emu_init(cfg.encode()) != 0:
            raise RuntimeError(self.lib.emu_error().decode())
        self.nwave, self.nlayer = self.lib.emu_nwave(), self.lib.emu_nlayer()

    def set_radius(self, r):
        self.lib.emu_set_radius(r)

    def set_cloudtop(self, t):
        self.lib.emu_set_cloudtop(t)

    def set_scattering(self, f, v):
        self.lib.emu_set_scattering(f, v)

    def set_lbl_ext(self, ext):
        """line-by-line mode (cfg without opacityfile): ext[layer][wave] of the next run() calls"""
        ext = np.ascontiguousarray(ext, dtype=np.float64)
        assert ext.shape == (self.nlayer, self.nwave)
        self.lib.emu_set_lbl_ext(ext.ctypes.data_as(dp))

    def wn(self):
        out = np.zeros(self.nwave)
        self.lib.emu_wn(out.ctypes.data_as(dp))
        return out

    def run(self, model):
        nw, nl = self.nwave, self.nlayer
        model = np.ascontiguousarray(model, dtype=np.float64)
        out = dict(spectrum=np.zeros(nw), tau=np.zeros((nw, nl)), last=np.zeros(nw, dtype=np.int32),
                   radius=np.zeros(nl), ext=np.zeros((nl, nw)))
        out["status"] = self.lib.emu_run(
            model.ctypes.data_as(dp), out["spectrum"].ctypes.data_as(dp), out["tau"].ctypes.data_as(dp),
            out["last"].ctypes.data_as(C.POINTER(C.c_int)), out["radius"].ctypes.data_as(dp),
            out["ext"].ctypes.data_as(dp))
        return out

    def run_build(self, model, ahead):
        """One eclipse model through the throughput kernel's build for this configuration
        (emu_run_build): -> spectrum, status, (NMOL, NCIA) of the build that ran."""
        model = np.ascontiguousarray(model, dtype=np.float64)
        spec = np.zeros(self.nwave)
        build = np.zeros(2, dtype=np.int32)
        st = self.lib.emu_run_build(model.ctypes.data_as(dp), int(ahead), spec.ctypes.data_as(dp),
                                    build.ctypes.data_as(C.POINTER(C.c_int)))
        if st < 0:
            raise RuntimeError("emu_run_build: not an eclipse configuration")
        return spec, st, tuple(int(b) for b in build)
