"""oracle/oracle.py -- TEST INFRASTRUCTURE ONLY.

ctypes front-end of liboracle.so (oracle/transit_oracle.c) plus small, independent
Python/numpy readers of the reference's input formats, so that the oracle shares no parsing
code with the product library.  Only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs may import this module.

The band-integration oracle (`resample`, `bandintegrate`) restates code/wine.py:127-199 and
code/BARTfunc.py:386-396 in numpy.
"""
import ctypes as C
import os
import struct
import subprocess
import numpy as np

_trapz = getattr(np, "trapezoid", None) or np.trapz

HERE = os.path.dirname(os.path.abspath(__file__))
LIBPATH = os.path.join(HERE, "liboracle.so")
REFLIB = os.path.join(HERE, "_ref", "libtransit_ref.so")
dp = C.POINTER(C.c_double)
ip = C.POINTER(C.c_int)


def build(force=False):
    """Compile liboracle.so (and oracle/_ref when /root/reference is present)."""
    if force or not os.path.exists(LIBPATH) or \
            os.path.getmtime(LIBPATH) < os.path.getmtime(os.path.join(HERE, "transit_oracle.c")):
        subprocess.check_call(["make", "-s", "-C", HERE, "liboracle.so"])
    if os.path.isdir("/root/reference/modules/transit/transit/src") and \
            (force or not os.path.exists(REFLIB)):
        subprocess.check_call(["make", "-s", "-C", HERE, "ref"])


class OrcConfig(C.Structure):
    _fields_ = [
        ("nlayer", C.c_int), ("nspec", C.c_int), ("nwave", C.c_int),
        ("press", dp), ("pfct", C.c_double), ("rfct", C.c_double),
        ("mass", dp), ("pol", dp), ("wn", dp),
        ("gsurf", C.c_double), ("p0", C.c_double), ("r0", C.c_double),
        ("ntemp", C.c_int), ("ngmol", C.c_int),
        ("gtemp", dp), ("gmol_spec", ip), ("grid", dp),
        ("ncia", C.c_int), ("cia_nwn", ip), ("cia_nt", ip),
        ("cia_wn", C.POINTER(dp)), ("cia_t", C.POINTER(dp)), ("cia_tab", C.POINTER(dp)),
        ("cia_nspec", ip), ("cia_spec", ip),
        ("toomuch", C.c_double), ("nangle", C.c_int), ("angles_deg", dp),
        ("starrad_cm", C.c_double), ("transparent", C.c_int),
        ("cloud_flag", C.c_int), ("cloudext", C.c_double), ("cloudtop", C.c_double),
        ("cloudbot", C.c_double),
        ("scat_flag", C.c_int), ("scat_logext", C.c_double),
        ("modlevel", C.c_int),
    ]


class OrcInter(C.Structure):
    _fields_ = [("radius", dp), ("temp", dp), ("mm", dp), ("dens", dp), ("ext", dp),
                ("cia", dp), ("tau", dp), ("last", C.POINTER(C.c_long)), ("intens", dp)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(LIBPATH)
        _lib.orc_forward.argtypes = [C.POINTER(OrcConfig), C.c_int, dp, dp, C.POINTER(OrcInter)]
        _lib.orc_forward.restype = C.c_int
        _lib.orc_simps_path.restype = C.c_double
        _lib.orc_simps_path.argtypes = [dp, dp, C.c_int]
        _lib.orc_totaltau1.restype = C.c_double
        _lib.orc_totaltau1.argtypes = [C.c_double, dp, dp, C.c_long]
        _lib.orc_modulation1.restype = C.c_double
        _lib.orc_modulation1.argtypes = [dp, C.c_long, C.c_double, dp, C.c_long, C.c_double,
                                         C.c_double, C.c_int]
        _lib.orc_voigtn.argtypes = [C.c_int, C.c_double, C.c_double, C.c_double,
                                    C.POINTER(C.c_float), C.c_int]
        _lib.orc_profile_halfsize.restype = C.c_long
        _lib.orc_profile_halfsize.argtypes = [C.c_double, C.c_double, C.c_double, C.c_float,
                                              C.c_long]
    return _lib


def _d(a):
    return a.ctypes.data_as(dp)


# ----------------------------------------------------------------------------------------
# Independent readers of the reference's input formats
def read_cfg(path):
    """`key value` lines, '#' comments (procopt.c:649-704).  Returns the raw dict."""
    out = {}
    with open(path) as f:
        for line in f:
            line = line.rstrip("\n")
            if not line or line.startswith("#"):
                continue
            parts = line.split(None, 1)
            out[parts[0]] = parts[1].strip() if len(parts) > 1 else ""
    return out


def read_molecules(path):
    tab = {}
    with open(path) as f:
        for line in f:
            if not line.strip() or line.lstrip().startswith("#"):
                continue
            p = line.split()
            tab[p[1]] = dict(id=int(p[0]), mass=float(p[2]), radius=float(p[3]) / 2.0 * 1e-8,
                             pol=float(p[5]))
    return tab


def read_atm(path):
    """TEA-format atmosphere file (readatm.c:255-620)."""
    species, rows = None, []
    rfct = pfct = tfct = 1.0
    with open(path) as f:
        lines = f.readlines()
    i = 0
    while i < len(lines):
        s = lines[i].strip()
        if s.startswith("#SPECIES"):
            species = lines[i + 1].split()
            i += 2
            continue
        if s.startswith("ur"):
            rfct = float(s[2:])
        elif s.startswith("up"):
            pfct = float(s[2:])
        elif s.startswith("ut"):
            tfct = float(s[2:])
        elif s and not s.startswith("#") and not s.startswith("q") and species is not None \
                and (s[0].isdigit() or s[0] in "+-."):
            rows.append([float(v) for v in s.split()])
        i += 1
    a = np.array(rows)
    c = np.ascontiguousarray
    return dict(species=species, radius=c(a[:, 0]), press=c(a[:, 1]), temp=c(a[:, 2]), q=c(a[:, 3:]),
                rfct=rfct, pfct=pfct, tfct=tfct)


def read_cia(path):
    species, temps, rows = None, None, []
    with open(path) as f:
        for line in f:
            s = line.strip()
            if not s or s.startswith("#"):
                continue
            if s[0] == "i":
                species = s.split()[1:]
            elif s[0] == "t":
                temps = np.array([float(v.rstrip("kK")) for v in s.split()[1:]])
            else:
                rows.append([float(v) for v in s.split()])
    a = np.array(rows)
    return dict(species=species, temps=temps, wn=np.ascontiguousarray(a[:, 0]),
                tab=np.ascontiguousarray(a[:, 1:]))


def read_opacity(path):
    with open(path, "rb") as f:
        nmol, nT, nlayer, nw = struct.unpack("4l", f.read(32))
        molids = np.frombuffer(f.read(4 * nmol), dtype=np.int32).copy()
        temps = np.frombuffer(f.read(8 * nT), dtype=np.float64).copy()
        press = np.frombuffer(f.read(8 * nlayer), dtype=np.float64).copy()
        wn = np.frombuffer(f.read(8 * nw), dtype=np.float64).copy()
        off = f.tell()
    o = np.fromfile(path, dtype=np.float64, offset=off).reshape(nlayer, nT, nmol, nw)
    return dict(molids=molids, temps=temps, press=press, wn=wn, o=o)


def wn_grid(lo, hi, d):
    n = int(((1.0 + 1e-8) * hi - lo) / d + 1)
    return lo + np.arange(n) * d


class Oracle:
    """One configuration (the state transit_init leaves behind) for orc_forward."""

    def __init__(self, cfgpath):
        cfg = read_cfg(cfgpath)
        self.cfg = cfg
        key = lambda k, d=None: next((v for kk, v in cfg.items() if k.startswith(kk) or
                                      kk.startswith(k)), d) if k not in cfg else cfg[k]
        self.eclipse = cfg.get("solution", "eclipse") == "eclipse"
        atm = read_atm(cfg["atm"])
        mols = read_molecules(cfg["molfile"])
        self.atm = atm
        self.species = atm["species"]
        ns = len(self.species)
        self.mass = np.array([mols[s]["mass"] for s in self.species])
        self.pol = np.array([mols[s]["pol"] for s in self.species])
        self.radius_cm = np.array([mols[s]["radius"] for s in self.species])
        self.ids = [mols[s]["id"] for s in self.species]
        self.press = np.ascontiguousarray(atm["press"])
        if "wnlow" in cfg:
            lo, hi = float(cfg["wnlow"]), float(cfg["wnhigh"])
        else:
            fct = float(cfg.get("wlfct", 1e-4))
            lo, hi = 1.0 / (float(cfg["wlhigh"]) * fct), 1.0 / (float(cfg["wllow"]) * fct)
        self.wn = wn_grid(lo, hi, float(cfg["wndelt"]))
        c = OrcConfig()
        c.nlayer, c.nspec, c.nwave = len(self.press), ns, len(self.wn)
        c.press, c.pfct, c.rfct = _d(self.press), atm["pfct"], atm["rfct"]
        c.mass, c.pol, c.wn = _d(self.mass), _d(self.pol), _d(self.wn)
        c.gsurf = float(cfg["gsurf"])
        c.p0 = float(cfg["refpress"])
        c.r0 = float(cfg["refradius"])
        self.lbl = None
        if cfg.get("opacityfile"):
            op = read_opacity(cfg["opacityfile"])
            self.op = op
            self.grid = np.ascontiguousarray(op["o"])
            self.gtemp = op["temps"]
            self.gmol_spec = np.array([self.ids.index(int(m)) for m in op["molids"]], dtype=np.int32)
            c.ntemp, c.ngmol = len(self.gtemp), len(self.gmol_spec)
            c.gtemp, c.gmol_spec, c.grid = _d(self.gtemp), self.gmol_spec.ctypes.data_as(ip), \
                _d(self.grid)
        else:
            # no opacity file (opacity.c:28-36): line-by-line extinction per layer, tau.c:163-175
            self.B = BuilderOracle(cfgpath, grid_temps=False)
            lb, keep = self.B.lbl_struct()
            isos = self.B.tli["isos"]
            self._iso_nt = np.array([len(i["T"]) for i in isos], dtype=np.int32)
            self._iso_T = [np.ascontiguousarray(i["T"], dtype=np.float64) for i in isos]
            self._iso_Z = [np.ascontiguousarray(i["Z"], dtype=np.float64) for i in isos]
            f = OrcLblFwd()
            f.lbl = C.pointer(lb)
            f.iso_nt = self._iso_nt.ctypes.data_as(ip)
            Tp = (dp * len(isos))(*[_d(t) for t in self._iso_T])
            Zp = (dp * len(isos))(*[_d(z) for z in self._iso_Z])
            f.iso_T, f.iso_Z = Tp, Zp
            self._lblkeep = (lb, keep, Tp, Zp)
            self.lbl = f
        files = [f for f in cfg.get("csfile", "").split(",") if f]
        self.cia = [read_cia(f) for f in files]
        n = len(self.cia)
        c.ncia = n
        self._keep = []
        if n:
            self.cia_nwn = np.array([len(t["wn"]) for t in self.cia], dtype=np.int32)
            self.cia_nt = np.array([len(t["temps"]) for t in self.cia], dtype=np.int32)
            self.cia_nspec = np.array([len(t["species"]) for t in self.cia], dtype=np.int32)
            spec = np.zeros(2 * n, dtype=np.int32)
            for i, t in enumerate(self.cia):
                for k, s in enumerate(t["species"]):
                    spec[2 * i + k] = self.species.index(s)
            self.cia_spec = spec
            wnp = (dp * n)(*[_d(t["wn"]) for t in self.cia])
            tp = (dp * n)(*[_d(t["temps"]) for t in self.cia])
            tabp = (dp * n)(*[_d(t["tab"]) for t in self.cia])
            self._keep += [wnp, tp, tabp]
            c.cia_nwn, c.cia_nt = self.cia_nwn.ctypes.data_as(ip), self.cia_nt.ctypes.data_as(ip)
            c.cia_wn, c.cia_t, c.cia_tab = wnp, tp, tabp
            c.cia_nspec, c.cia_spec = self.cia_nspec.ctypes.data_as(ip), spec.ctypes.data_as(ip)
        c.toomuch = float(cfg.get("toomuch", 20))
        self.angles = np.array([float(v) for v in cfg.get("raygrid", "0 20 40 60 80").split()])
        c.nangle, c.angles_deg = len(self.angles), _d(self.angles)
        c.starrad_cm = float(cfg.get("starrad", 1.125)) * 6.957e10
        c.transparent = 0
        c.modlevel = int(cfg.get("modlevel", 1))
        c.cloud_flag, c.cloudext, c.cloudtop, c.cloudbot = 0, 0.0, 0.0, 0.0
        if "cloudtop" in cfg:
            self.set_cloudtop(float(cfg["cloudtop"]), c)
        c.scat_flag, c.scat_logext = 0, 0.0
        if "scattering" in cfg:
            if cfg["scattering"] == "polar":
                c.scat_flag = 2
            else:
                c.scat_flag, c.scat_logext = 1, float(cfg["scattering"])
        self.c = c

    # transit.c:98-115
    def set_radius(self, r):
        self.c.r0 = r

    def set_cloudtop(self, top, c=None):
        c = c or self.c
        c.cloud_flag, c.cloudext, c.cloudtop, c.cloudbot = 1, 100.0, top, top + 10

    def set_scattering(self, flag, logext):
        self.c.scat_flag, self.c.scat_logext = flag, logext

    def status(self, model):
        """The rejection code (REJ_TGRID 1, REJ_TCIA 2, as bart_b200.api names them) of a model whose
        layer temperatures leave the opacity grid's or a CIA table's range, where the reference
        exits (extinction.c:534-581, crosssec.c:293-309); 0 otherwise."""
        T = np.asarray(model, dtype=np.float64)[:self.c.nlayer]
        st = 0
        if self.lbl is None and ((T < self.gtemp[0]).any() or (T > self.gtemp[-1]).any()):
            st |= 1
        for t in self.cia:
            if (T < t["temps"][0]).any() or (T > t["temps"][-1]).any():
                st |= 2
        return st

    def run(self, model, inter=False):
        """The spectrum of one model (with inter: a dict of the intermediate arrays, its "status"
        and "spectrum").  A model the reference would exit on (status() != 0) is not computed:
        its spectrum is -1, as the product reports a rejected model."""
        model = np.ascontiguousarray(model, dtype=np.float64)
        nl, nw, ns = self.c.nlayer, self.c.nwave, self.c.nspec
        spec = np.zeros(nw)
        st = self.status(model)
        if st:
            spec[:] = -1.0
            return dict(status=st, spectrum=spec) if inter else spec
        if not inter:
            self._forward(model, spec, None)
            return spec
        it = OrcInter()
        out = dict(radius=np.zeros(nl), temp=np.zeros(nl), mm=np.zeros(nl),
                   density=np.zeros((ns, nl)), ext=np.zeros((nl, nw)), cia=np.zeros((nw, nl)),
                   tau=np.zeros((nw, nl)), last=np.zeros(nw, dtype=np.int64))
        it.radius, it.temp, it.mm, it.dens = _d(out["radius"]), _d(out["temp"]), \
            _d(out["mm"]), _d(out["density"])
        it.ext, it.cia, it.tau = _d(out["ext"]), _d(out["cia"]), _d(out["tau"])
        it.last = out["last"].ctypes.data_as(C.POINTER(C.c_long))
        if self.eclipse:
            out["intens"] = np.zeros((self.c.nangle, nw))
            it.intens = _d(out["intens"])
        self._forward(model, spec, C.byref(it))
        out["spectrum"], out["status"] = spec, 0
        return out

    def _forward(self, model, spec, it):
        if self.lbl is None:
            lib().orc_forward(C.byref(self.c), int(self.eclipse), _d(model), _d(spec), it)
        else:
            L = lib()
            L.orc_forward_lbl.argtypes = [C.POINTER(OrcConfig), C.POINTER(OrcLblFwd), C.c_int, dp, dp,
                                          C.POINTER(OrcInter)]
            L.orc_forward_lbl(C.byref(self.c), C.byref(self.lbl), int(self.eclipse), _d(model),
                              _d(spec), it)

    def run_batch(self, models):
        return np.stack([self.run(m) for m in np.atleast_2d(models)])


# ----------------------------------------------------------------------------------------
# Stage (c): band integration (code/wine.py:16-66,127-199; code/BARTfunc.py:386-396)
def readfilter(path):
    with open(path) as f:
        lines = f.readlines()
    while lines[0].startswith("#") or not lines[0].strip():
        lines.pop(0)
    n = len(lines)
    wl = np.zeros(n)
    tr = np.zeros(n)
    for i in range(n):
        a, b = lines[i].strip().split()[0:2]
        wl[n - 1 - i], tr[n - 1 - i] = float(a), float(b)
    return 1.0 / (wl * 1e-4), tr


def resample(specwn, filterwn, filtertr, starwn, starfl):
    idx = np.where((specwn < filterwn[-1]) & (filterwn[0] < specwn))[0]
    ifilter = np.interp(specwn[idx], filterwn, filtertr)
    istarfl = np.interp(specwn[idx], starwn, starfl)
    nifilter = ifilter / _trapz(ifilter, specwn[idx])
    return nifilter, istarfl, idx


def bandintegrate(spectrum, specwn, nifilter, idx):
    return _trapz(spectrum * nifilter, specwn[idx])


def bandflux(spectrum, specwn, filters, star=None, rprs=None):
    """filters: list of (nifilter, istarfl, idx).  Eclipse when `star` is truthy."""
    out = np.zeros(len(filters))
    for i, (nif, istar, idx) in enumerate(filters):
        if star:
            out[i] = bandintegrate(spectrum[idx] / istar * rprs * rprs, specwn, nif, idx)
        else:
            out[i] = bandintegrate(spectrum[idx], specwn, nif, idx)
    return out


# ----------------------------------------------------------------------------------------
# Stage (d): line-by-line opacity-grid builder oracle (opacity.c:218-427 driving
# orc_voigtn / orc_computemolext of transit_oracle.c)
class OrcLbl(C.Structure):
    _fields_ = [
        ("nlines", C.c_long), ("wl_um", dp), ("elow", dp), ("gf", dp),
        ("isoid", C.POINTER(C.c_short)), ("niso", C.c_int), ("iso_mass", dp), ("iso_ratio", dp),
        ("iso_spec", ip), ("iso_gmol", ip), ("ngmol", C.c_int), ("nspec", C.c_int),
        ("spec_mass", dp), ("spec_radius", dp), ("wn_lo", C.c_double), ("dwn", C.c_double),
        ("nwave", C.c_long), ("osamp", C.c_int), ("nowns", C.c_long),
        ("nDop", C.c_int), ("nLor", C.c_int), ("aDop", dp), ("aLor", dp),
        ("profsize", C.POINTER(C.c_long)), ("profile", C.POINTER(C.POINTER(C.c_float))),
        ("ethresh", C.c_double),
    ]


class OrcLblFwd(C.Structure):
    _fields_ = [("lbl", C.POINTER(OrcLbl)), ("iso_nt", ip), ("iso_T", C.POINTER(dp)),
                ("iso_Z", C.POINTER(dp))]


def read_tli(path):
    """TLI v6 (readlineinfo.c:87-244, 416-537)."""
    with open(path, "rb") as f:
        buf = f.read()
    pos = 4
    ver, _, _ = struct.unpack_from("3h", buf, pos); pos += 6
    assert ver == 6
    wl_ini, wl_fin = struct.unpack_from("2d", buf, pos); pos += 16
    (ndb,) = struct.unpack_from("h", buf, pos); pos += 2
    isos = []
    for d in range(ndb):
        (n,) = struct.unpack_from("h", buf, pos); pos += 2
        dbname = buf[pos:pos + n].decode(); pos += n
        (n,) = struct.unpack_from("h", buf, pos); pos += 2
        molname = buf[pos:pos + n].decode(); pos += n
        nT, niso = struct.unpack_from("hh", buf, pos); pos += 4
        T = np.frombuffer(buf, dtype="<f8", count=nT, offset=pos).copy(); pos += 8 * nT
        for i in range(niso):
            (n,) = struct.unpack_from("h", buf, pos); pos += 2
            name = buf[pos:pos + n].decode(); pos += n
            mass, ratio = struct.unpack_from("2d", buf, pos); pos += 16
            Z = np.frombuffer(buf, dtype="<f8", count=nT, offset=pos).copy(); pos += 8 * nT
            isos.append(dict(db=dbname, mol=molname, name=name, mass=mass, ratio=ratio, T=T, Z=Z))
    (nlines,) = struct.unpack_from("Q", buf, pos); pos += 8
    (niso_l,) = struct.unpack_from("i", buf, pos); pos += 4
    per = struct.unpack_from("%dQ" % niso_l, buf, pos); pos += 8 * niso_l
    wl = np.frombuffer(buf, dtype="<f8", count=nlines, offset=pos).copy(); pos += 8 * nlines
    isoid = np.frombuffer(buf, dtype="<i2", count=nlines, offset=pos).copy(); pos += 2 * nlines
    elow = np.frombuffer(buf, dtype="<f8", count=nlines, offset=pos).copy(); pos += 8 * nlines
    gf = np.frombuffer(buf, dtype="<f8", count=nlines, offset=pos).copy()
    return dict(isos=isos, per=per, wl=wl, isoid=isoid, elow=elow, gf=gf, wl_ini=wl_ini, wl_fin=wl_fin)


def select_lines(tli, wnlow, wnhigh):
    """Per-isotope slice by the reference's binary search + linear refinement
    (readlineinfo.c:16-77, 496-525)."""
    iniw, finw = 1.0 / wnhigh / 1e-4, 1.0 / wnlow / 1e-4
    keep = []
    off = 0
    for n in tli["per"]:
        w = tli["wl"][off:off + n]
        if n > 0:
            lo, hi = 0, n - 1
            while True:
                loc = (hi + lo) // 2
                if iniw > w[loc]:
                    lo = loc
                else:
                    hi = loc
                if hi - lo <= 1:
                    break
            first = hi
            while first > 0 and not (w[first - 1] < iniw):
                first -= 1
            lo, hi = 0, n - 1
            while True:
                loc = (hi + lo) // 2
                if finw > w[loc]:
                    lo = loc
                else:
                    hi = loc
                if hi - lo <= 1:
                    break
            last = lo
            while last < n - 1 and not (w[last + 1] > finw):
                last += 1
            if last >= first:
                keep.append(np.arange(off + first, off + last + 1))
        off += n
    idx = np.concatenate(keep) if keep else np.zeros(0, dtype=int)
    return idx


class BuilderOracle:
    """calcprofiles + calcopacity restated: builds o[layer][temp][mol][wave] on the CPU."""

    def __init__(self, cfgpath, with_profiles=True, grid_temps=True):
        L = lib()
        L.orc_computemolext.argtypes = [C.POINTER(OrcLbl), C.c_double, dp, dp, dp,
                                        C.POINTER(C.c_long), C.POINTER(C.c_long)]
        L.orc_spline_init.argtypes = [dp, dp, dp, C.c_long]
        L.orc_splinterp_pt.restype = C.c_double
        L.orc_splinterp_pt.argtypes = [dp, C.c_long, dp, dp, C.c_double]
        cfg = read_cfg(cfgpath)
        self.cfg = cfg
        atm = read_atm(cfg["atm"])
        mols = read_molecules(cfg["molfile"])
        self.atm = atm
        species = atm["species"]
        self.spec_mass = np.array([mols[s]["mass"] for s in species])
        self.spec_radius = np.array([mols[s]["radius"] for s in species])
        ids = [mols[s]["id"] for s in species]
        lo, hi, d = float(cfg["wnlow"]), float(cfg["wnhigh"]), float(cfg["wndelt"])
        self.wn = wn_grid(lo, hi, d)
        self.osamp = int(float(cfg.get("wnosamp", 2160)))
        self.nowns = (len(self.wn) - 1) * self.osamp + 1
        self.odwn = d / self.osamp
        self.dwn = d
        self.temps = wn_grid(float(cfg.get("tlow", 500)), float(cfg.get("thigh", 3000)),
                             float(cfg.get("tempdelt", 100))) if grid_temps else np.zeros(0)
        tli = read_tli(cfg["linedb"])
        self.tli = tli
        idx = select_lines(tli, lo, hi)
        self.line_idx = idx
        self.wl = np.ascontiguousarray(tli["wl"][idx])
        self.elow = np.ascontiguousarray(tli["elow"][idx])
        self.gf = np.ascontiguousarray(tli["gf"][idx])
        self.isoid = np.ascontiguousarray(tli["isoid"][idx])
        isos = tli["isos"]
        self.niso = len(isos)
        self.iso_mass = np.array([i["mass"] for i in isos])
        self.iso_ratio = np.array([i["ratio"] for i in isos])
        self.iso_spec = np.array([species.index(i["mol"]) for i in isos], dtype=np.int32)
        gm, gmol = [], []
        for i in isos:
            mid = ids[species.index(i["mol"])]
            if mid not in gm:
                gm.append(mid)
            gmol.append(gm.index(mid))
        self.gmol_id = gm
        self.iso_gmol = np.array(gmol, dtype=np.int32)
        # Z(T grid) by natural spline (opacity.c:325-339)
        self.ziso = np.zeros((self.niso, len(self.temps)))
        for k, i in enumerate(isos):
            z = np.zeros(len(i["T"]))
            L.orc_spline_init(_d(z), _d(i["T"]), _d(i["Z"]), len(i["T"]))
            for t, T in enumerate(self.temps):
                self.ziso[k, t] = L.orc_splinterp_pt(_d(z), len(i["T"]), _d(i["T"]), _d(i["Z"]), float(T))
        # Voigt table (calcprofiles)
        self.nDop, self.nLor = int(cfg.get("ndop", 60)), int(cfg.get("nlor", 60))
        f32 = np.float32
        dmin, dmax = f32(cfg.get("dmin", 1e-3)), f32(cfg.get("dmax", 0.25))
        lmin, lmax = f32(cfg.get("lmin", 1e-4)), f32(cfg.get("lmax", 10.0))

        def logspace(a, b, n):
            l0, l1 = np.log10(float(a)), np.log10(float(b))
            st = (l1 - l0) / (n - 1.0)
            return np.array([10.0 ** (l0 + i * st) for i in range(n)])
        self.aDop, self.aLor = logspace(dmin, dmax, self.nDop), logspace(lmin, lmax, self.nLor)
        self.ta = f32(cfg.get("nwidth", 20))
        self.ethresh = float(cfg.get("ethresh", cfg.get("ethreshold", 1e-8)))
        self.profsize = np.zeros(self.nDop * self.nLor, dtype=np.int64)
        self.profiles = [None] * (self.nDop * self.nLor)
        if with_profiles:
            for i in range(self.nDop):
                for j in range(self.nLor):
                    p = i * self.nLor + j
                    if self.aDop[i] * 10.0 < self.aLor[j] and i != 0:
                        self.profsize[p] = self.profsize[p - self.nLor]
                        self.profiles[p] = self.profiles[p - self.nLor]
                        continue
                    self.profiles[p], self.profsize[p] = self.profile(i, j)

    def profile(self, i, j):
        L = lib()
        dop, lor = float(np.float32(self.aDop[i])), float(np.float32(self.aLor[j]))
        ps = L.orc_profile_halfsize(self.odwn, dop, lor, self.ta, self.nowns)
        n = 2 * ps + 1
        out = np.zeros(n, dtype=np.float32)
        L.orc_voigtn(n, self.odwn * ps, lor, dop, out.ctypes.data_as(C.POINTER(C.c_float)),
                     1 if n > 99999 else 0)
        return out, ps

    def lbl_struct(self):
        """(OrcLbl, objects to keep alive)"""
        nw = len(self.wn)
        ng = len(self.gmol_id)
        lb = OrcLbl()
        lb.nlines = len(self.wl)
        lb.wl_um, lb.elow, lb.gf = _d(self.wl), _d(self.elow), _d(self.gf)
        lb.isoid = self.isoid.ctypes.data_as(C.POINTER(C.c_short))
        lb.niso, lb.iso_mass, lb.iso_ratio = self.niso, _d(self.iso_mass), _d(self.iso_ratio)
        lb.iso_spec, lb.iso_gmol = self.iso_spec.ctypes.data_as(ip), self.iso_gmol.ctypes.data_as(ip)
        lb.ngmol, lb.nspec = ng, len(self.spec_mass)
        lb.spec_mass, lb.spec_radius = _d(self.spec_mass), _d(self.spec_radius)
        lb.wn_lo, lb.dwn, lb.nwave, lb.osamp, lb.nowns = self.wn[0], self.dwn, nw, self.osamp, self.nowns
        lb.nDop, lb.nLor, lb.aDop, lb.aLor = self.nDop, self.nLor, _d(self.aDop), _d(self.aLor)
        psz = self.profsize.astype(np.int64)
        lb.profsize = psz.ctypes.data_as(C.POINTER(C.c_long))
        ptrs = (C.POINTER(C.c_float) * len(self.profiles))(
            *[p.ctypes.data_as(C.POINTER(C.c_float)) for p in self.profiles])
        lb.profile = ptrs
        lb.ethresh = self.ethresh
        return lb, (psz, ptrs)

    def total(self, temp, density, Z):
        """computemolext(permol=0) of one layer: k[nwave] (extinction.c:281-529)"""
        L = lib()
        L.orc_computemolext_total.argtypes = [C.POINTER(OrcLbl), C.c_double, dp, dp, dp,
                                              C.POINTER(C.c_long)]
        lb, keep = self.lbl_struct()
        k = np.zeros(len(self.wn))
        density = np.ascontiguousarray(density, dtype=np.float64)
        Z = np.ascontiguousarray(Z, dtype=np.float64)
        L.orc_computemolext_total(C.byref(lb), float(temp), _d(density), _d(Z), _d(k), None)
        return k

    def build(self, layers=None, temps=None, trace=False):
        L = lib()
        atm = self.atm
        nl = len(atm["press"])
        layers = range(nl) if layers is None else layers
        temps = range(len(self.temps)) if temps is None else temps
        nw = len(self.wn)
        ng = len(self.gmol_id)
        lb, _keep = self.lbl_struct()
        out = np.zeros((len(list(layers)), len(list(temps)), ng, nw))
        tr = np.zeros(len(self.wl), dtype=np.int64) if trace else None
        for a, r in enumerate(layers):
            for b, t in enumerate(temps):
                T = float(self.temps[t])
                dens = 1.66053886e-24 * atm["q"][r] * (atm["press"][r] * atm["pfct"]) / 1.380658e-16 / T \
                    * self.spec_mass
                dens = np.ascontiguousarray(dens)
                Z = np.ascontiguousarray(self.ziso[:, t])
                k = np.zeros((ng, nw))
                L.orc_computemolext(C.byref(lb), T, _d(dens), _d(Z), _d(k),
                                    tr.ctypes.data_as(C.POINTER(C.c_long)) if trace else None, None)
                out[a, b] = k
        self.trace = tr
        return out
