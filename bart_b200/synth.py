"""Synthetic, seed-fixed inputs of the shapes BASELINE.json names (SURVEY.md section 8d).

Everything the transit forward model reads from disk is produced here in the reference's own
file formats, so the same files can be fed to (i) this package's C/CUDA library, (ii) the
oracle restatement and (iii) the compiled reference (oracle/_ref) for parity:

* atmosphere file  (TEA format parsed by readatm.c:255-620 of the reference)
* molecules.dat    (readatm.c:625-717)
* CIA table        (crosssec.c:9-268)
* TLI v6 line list (readlineinfo.c:87-244,416-537; writer of record pylineread.py:185-428)
* opacity grid     (opacity.c:406-421 / 432-503: 4 longs, int molID[], double T[], p[], wn[],
                    double o[layer][temp][mol][wave])
* filter files     (wine.py:16-66: two columns, wavelength in micron ascending, transmission)
* transit cfg      (`key value` lines, procopt.c:649-704)

No network, no reference data needed: the GPU box regenerates bit-identical inputs from the
seed (numpy Generator streams are stable across platforms for a given numpy version).
"""
import os
import struct
import numpy as np

# Physical data for the species used by the BART example configurations.  Columns follow the
# reference's molecules.dat layout: ID, name, mass (g/mol), diameter (A), source tag,
# polarizability (A^3), long name.
MOLECULES = [
    (101, "H2O", 18.01528, 3.2, "01", 1.501, "Water"),
    (102, "CH4", 16.0425, 4.0, "01", 2.448, "Methane"),
    (103, "CO", 28.0101, 2.8, "01", 1.953, "Carbon Monoxide"),
    (104, "CO2", 44.0095, 2.8, "01", 2.507, "Carbon Dioxide"),
    (105, "H2", 2.01588, 2.89, "02", 0.787, "Molecular Hydrogen"),
    (106, "NH3", 17.03052, 3.6, "01", 2.103, "Ammonia"),
    (110, "N2", 28.01340, 3.64, "02", 1.710, "Molecular Nitrogen"),
    (1, "H", 1.007940, 2.4, "01", 0.667, "Hydrogen"),
    (2, "He", 4.0026020, 2.0, "01", 0.208, "Helium"),
    (6, "C", 12.0107, 1.7, "04", 1.760, "Carbon"),
    (7, "N", 14.0067, 1.55, "04", 1.100, "Nitrogen"),
    (8, "O", 15.9994, 1.52, "04", 0.802, "Oxygen"),
]
MOL_BY_NAME = {m[1]: m for m in MOLECULES}

SPECIES = ["H", "He", "C", "N", "O", "H2", "CO", "CO2", "CH4", "H2O"]
# examples/WASP-12b/BART.cfg:69 `uniform`, H2 trimmed so that the sum is exactly 1
UNIFORM = [1e-9, 0.15, 1e-9, 1e-9, 1e-9, 0.8496, 1e-4, 1e-4, 1e-4, 1e-4]

KB = 1.380658e-16
AMU = 1.66053886e-24


def write_molecules(path):
    with open(path, "w") as f:
        f.write("# Molecular info (synthetic copy of the physical constants)\n")
        f.write("# ID    Molecule  Mass         Diameter  Diameter  Polarizability Long\n")
        f.write("#       Name      g/mol        Angstrom  source    Angstrom^3     name\n")
        for mid, name, mass, diam, src, pol, longname in MOLECULES:
            f.write(" %3d    %-8s %10.6f   %5.2f      %s        %6.3f         %s\n"
                    % (mid, name, mass, diam, src, pol, longname))
    return path


def pressure_grid(nlayer=100, p_bottom=100.0, p_top=1e-5):
    """Bottom -> top, bar, log-spaced (BART.py:88-98 defaults)."""
    return np.logspace(np.log10(p_bottom), np.log10(p_top), nlayer)


def temperature_profile(press, t_deep=1650.0, t_top=1240.0, p_knee=0.3, width=1.0):
    """Smooth monotone profile, hot below the knee, in [t_top, t_deep]."""
    x = (np.log10(press) - np.log10(p_knee)) / width
    return t_top + (t_deep - t_top) * 0.5 * (1.0 + np.tanh(x))


def hydrostatic_radius_km(press, temp, mu, gsurf=1000.0, r0_km=92000.0):
    """Rough hydrostatic radii for the file's radius column (the forward model recomputes them
    every call, readatm.c:787-865; the file values only need to be monotone)."""
    rad = np.zeros_like(press)
    rad[0] = r0_km
    for i in range(1, len(press)):
        H = KB * 0.5 * (temp[i] + temp[i - 1]) / (0.5 * (mu[i] + mu[i - 1]) * AMU * gsurf)
        rad[i] = rad[i - 1] + H * np.log(press[i - 1] / press[i]) / 1e5
    return rad


def write_atm(path, press, temp, abund, species=SPECIES, gsurf=1000.0, r0_km=92000.0):
    """TEA-style atmosphere file; layers bottom -> top, p in bar, radius in km."""
    masses = np.array([MOL_BY_NAME[s][2] for s in species])
    abund = np.asarray(abund, dtype=float)
    if abund.ndim == 1:
        abund = np.tile(abund, (len(press), 1))
    mu = abund @ masses
    rad = hydrostatic_radius_km(press, temp, mu, gsurf, r0_km)
    with open(path, "w") as f:
        f.write("# Synthetic atmosphere (bart_b200.synth)\n")
        f.write("# Units: pressure (bar), temperature (K), abundance (unitless).\n\n")
        f.write("#Values units:\nur 1e5\nup 1e6\nq number\n\n")
        f.write("#SPECIES\n" + " ".join(species) + "\n\n")
        f.write("#TEADATA\n")
        f.write("#Radius    Pressure   Temp       " + " ".join("%-10s" % s for s in species) + "\n")
        for i in range(len(press)):
            # a leading blank like TEA's files: the reference's reader drops the first character of
            # the first data row (readatm.c:425-470), which only the executable's path ever sees
            f.write(" %10.3f %.4e %7.2f " % (rad[i], press[i], temp[i])
                    + " ".join("%.4e" % q for q in abund[i]) + " \n")
    return path


def write_cia(path, pair=("H2", "H2"), temps=None, wn=None, seed=7):
    """Synthetic CIA table: smooth, positive, band-shaped in wn, slowly varying in T
    (cm-1 amagat-2), same layout as the reference's CIA_H2H2_400-7000K.dat."""
    if temps is None:
        temps = np.array([400, 500, 600, 700, 800, 900, 1000, 2000, 3000, 4000, 5000,
                          6000, 7000], dtype=float)
    if wn is None:
        wn = np.arange(20.0, 17001.0, 20.0)
    rng = np.random.default_rng(seed)
    centers = np.array([600.0, 4200.0, 8100.0, 12000.0])
    amps = np.array([3e-6, 1.2e-6, 8e-8, 4e-9])
    widths = np.array([500.0, 700.0, 900.0, 1100.0])
    tab = np.zeros((len(wn), len(temps)))
    for c, a, w in zip(centers, amps, widths):
        for j, T in enumerate(temps):
            ww = w * np.sqrt(T / 1000.0)
            tab[:, j] += a * (T / 1000.0) ** 0.5 * np.exp(-0.5 * ((wn - c) / ww) ** 2)
    tab *= 1.0 + 0.02 * rng.standard_normal(tab.shape)
    tab += 1e-12
    with open(path, "w") as f:
        f.write("# Synthetic %s-%s CIA table (bart_b200.synth)\n\n" % pair)
        f.write("i %s %s\n" % pair)
        f.write("t " + " ".join("%10d" % int(t) for t in temps) + "\n\n")
        f.write("# Wavenumber in cm-1, CIA coefficients in cm-1 amagat-2:\n")
        for i in range(len(wn)):
            f.write("%10.2f    " % wn[i] + " ".join("%.4e" % v for v in tab[i]) + "\n")
    return path


def write_filter(path, wl_lo, wl_hi, npts=100, edge=0.1, shape="trapezoid"):
    """Two-column filter file, wavelength (micron) ascending (wine.py:16-66)."""
    wl = np.linspace(wl_lo, wl_hi, npts)
    x = (wl - wl_lo) / (wl_hi - wl_lo)
    if shape == "trapezoid":
        tr = np.clip(np.minimum(x, 1 - x) / edge, 0.0, 1.0)
    else:
        tr = np.where((x > edge) & (x < 1 - edge), 1.0, 0.0)
    with open(path, "w") as f:
        f.write("# Synthetic filter\n# Wavelength (um)   Transmission\n")
        for a, b in zip(wl, tr):
            f.write("  %.8f        %.6f\n" % (a, b))
    return path


def partition_function(T, mass):
    """Smooth, increasing Z(T) of the magnitude HITRAN lists for CH4-like rotors."""
    return 0.6 * mass ** 0.25 * T ** 1.5 * (1.0 + (T / 1500.0) ** 3)


def write_tli(path, wn_lo, wn_hi, nlines, dbs=None, seed=12345, tli_T=None):
    """TLI v6 with HITRAN-2012-shaped content.  `dbs` is a list of
    (dbname, molname, [(isoname, mass, ratio), ...]).  Lines: nu ~ U(wn_lo, wn_hi) per isotope,
    stored as wavelength (micron) ascending inside each isotope block; gf = 10^U(-12,-6);
    elow ~ U(0, 3000) cm-1.  Returns the arrays written (for the oracle)."""
    if dbs is None:
        dbs = [("HITRAN CH4", "CH4", [("61", 16.0313, 0.98827), ("62", 17.03466, 0.0111031)])]
    if tli_T is None:
        tli_T = np.arange(70.0, 3001.0, 10.0)
    rng = np.random.default_rng(seed)
    niso_tot = sum(len(d[2]) for d in dbs)
    # split the lines between isotopes proportionally to sqrt(ratio) (minor ones get fewer)
    w = np.array([np.sqrt(iso[2]) for d in dbs for iso in d[2]])
    counts = np.maximum(1, np.floor(nlines * w / w.sum()).astype(np.int64))
    counts[0] += nlines - counts.sum()
    wl_all, iso_all, el_all, gf_all = [], [], [], []
    for k in range(niso_tot):
        nu = np.sort(rng.uniform(wn_lo, wn_hi, counts[k]))[::-1]   # descending nu
        wl = 1e4 / nu                                              # ascending wavelength (um)
        wl_all.append(wl)
        iso_all.append(np.full(counts[k], k, dtype=np.int16))
        el_all.append(rng.uniform(0.0, 3000.0, counts[k]))
        gf_all.append(10.0 ** rng.uniform(-12.0, -6.0, counts[k]))
    wl_all = np.concatenate(wl_all)
    iso_all = np.concatenate(iso_all)
    el_all = np.concatenate(el_all)
    gf_all = np.concatenate(gf_all)
    wl_ini = 1e4 / wn_hi
    wl_fin = 1e4 / wn_lo
    with open(path, "wb") as f:
        f.write(b"\xff\xb6\xb3\xab")
        f.write(struct.pack("3h", 6, 6, 2))
        f.write(struct.pack("2d", wl_ini, wl_fin))
        f.write(struct.pack("h", len(dbs)))
        for dbname, molname, isos in dbs:
            f.write(struct.pack("h", len(dbname)) + dbname.encode())
            f.write(struct.pack("h", len(molname)) + molname.encode())
            f.write(struct.pack("hh", len(tli_T), len(isos)))
            f.write(np.asarray(tli_T, dtype="<f8").tobytes())
            for isoname, mass, ratio in isos:
                f.write(struct.pack("h", len(isoname)) + isoname.encode())
                f.write(struct.pack("d", mass))
                f.write(struct.pack("d", ratio))
                f.write(partition_function(np.asarray(tli_T), mass).astype("<f8").tobytes())
        f.write(struct.pack("Q", len(wl_all)))
        f.write(struct.pack("i", niso_tot))
        f.write(struct.pack("%dQ" % niso_tot, *[int(c) for c in counts]))
        f.write(wl_all.astype("<f8").tobytes())
        f.write(iso_all.astype("<i2").tobytes())
        f.write(el_all.astype("<f8").tobytes())
        f.write(gf_all.astype("<f8").tobytes())
    return dict(wl=wl_all, isoid=iso_all, elow=el_all, gf=gf_all, counts=counts,
                tli_T=np.asarray(tli_T), dbs=dbs)


def synth_opacity_grid(nlayer, temps, molids, wn, press_bar, seed=2026, dtype=np.float64):
    """Seed-fixed grid o[layer][temp][mol][wave] (cm2/g): band envelopes + line-like spikes
    in wn, Boltzmann-like growth in T, pressure-broadening-like smoothing factor per layer."""
    rng = np.random.default_rng(seed)
    nT, nmol, nw = len(temps), len(molids), len(wn)
    o = np.empty((nlayer, nT, nmol, nw), dtype=dtype)
    x = (wn - wn[0]) / max(wn[-1] - wn[0], 1.0)
    tt = (np.asarray(temps) / 1000.0)[:, None]
    for m in range(nmol):
        nb = 4
        centers = rng.uniform(0.0, 1.0, nb)
        widths = rng.uniform(0.05, 0.2, nb)
        amps = rng.uniform(-1.0, 2.0, nb)
        env = np.full(nw, -4.0)
        for c, w, a in zip(centers, widths, amps):
            env = np.maximum(env, a - 3.0 * ((x - c) / w) ** 2)
        spikes = rng.uniform(-1.5, 1.0, nw)
        hot = rng.uniform(0.2, 1.5, nw)          # hot-band growth differs per wavenumber
        base = env + spikes                       # log10 at 1000 K
        logo_T = base[None, :] + hot[None, :] * (tt - 1.0)       # [nT][nw]
        for r in range(nlayer):
            pfac = 0.15 * np.log10(press_bar[r] / 1e-5) / 7.0    # mild layer dependence
            noise = 0.05 * rng.standard_normal((nT, nw))
            o[r, :, m, :] = 10.0 ** (logo_T * (1.0 - pfac) + noise)
    return o


def write_opacity(path, molids, temps, press_barye, wn, o):
    """opacity.c:406-421 byte layout (native endian, LP64)."""
    nlayer, nT, nmol, nw = o.shape
    with open(path, "wb") as f:
        f.write(struct.pack("4l", nmol, nT, nlayer, nw))
        f.write(np.asarray(molids, dtype=np.int32).tobytes())
        f.write(np.asarray(temps, dtype=np.float64).tobytes())
        f.write(np.asarray(press_barye, dtype=np.float64).tobytes())
        f.write(np.asarray(wn, dtype=np.float64).tobytes())
        f.write(np.ascontiguousarray(o, dtype=np.float64).tobytes())
    return path


def read_opacity(path, mmap=True):
    with open(path, "rb") as f:
        nmol, nT, nlayer, nw = struct.unpack("4l", f.read(32))
        molids = np.frombuffer(f.read(4 * nmol), dtype=np.int32).copy()
        temps = np.frombuffer(f.read(8 * nT), dtype=np.float64).copy()
        press = np.frombuffer(f.read(8 * nlayer), dtype=np.float64).copy()
        wn = np.frombuffer(f.read(8 * nw), dtype=np.float64).copy()
        off = f.tell()
    if mmap:
        o = np.memmap(path, dtype=np.float64, mode="r", offset=off,
                      shape=(nlayer, nT, nmol, nw))
    else:
        o = np.fromfile(path, dtype=np.float64, offset=off).reshape(nlayer, nT, nmol, nw)
    return dict(molids=molids, temps=temps, press=press, wn=wn, o=o)


def wn_grid(wnlow, wnhigh, wndelt):
    """makesample1 (makesample.c:77-104): n = floor(((1+1e-8) f - i)/d) + 1, v = i + k d."""
    n = int(((1.0 + 1e-8) * wnhigh - wnlow) / wndelt + 1)
    return wnlow + np.arange(n) * wndelt


SHAPES = {
    # name: wnlow, wnhigh, wndelt, grid molecules (ID order as a TLI would give), nfilters
    "demo": dict(wnlow=2500.0, wnhigh=5000.0, wndelt=1.0, mols=["CH4"], toomuch=10.0),
    "w12": dict(wnlow=910.0, wnhigh=3333.0, wndelt=1.0, mols=["H2O", "CO2", "CO", "CH4"],
                toomuch=10.0),
    "tiny": dict(wnlow=2500.0, wnhigh=2700.0, wndelt=1.0, mols=["CH4"], toomuch=10.0),
    "small4": dict(wnlow=2000.0, wnhigh=2600.0, wndelt=1.0, mols=["H2O", "CO2", "CO", "CH4"],
                   toomuch=10.0),
}


def read_tea_atm(path):
    """Parse a TEA-style atmosphere file (the layout readatm.c:425-470 reads): -> species, radius,
    pressure (file units), temperature, abundances[layer][species].  For building proposal models
    from an atmosphere file that was not written by write_atm."""
    species, rows, section = None, [], None
    for line in open(path):
        t = line.strip()
        if not t:
            continue
        if t.startswith("#"):
            section = t[1:].strip().upper()
            continue
        if section == "SPECIES" and species is None:
            species = t.split()
            continue
        parts = t.split()
        try:
            vals = [float(x) for x in parts]
        except ValueError:
            continue                                     # unit keywords: ur / up / q ...
        if species is not None and len(vals) == 3 + len(species):
            rows.append(vals)
    a = np.array(rows)
    return species, a[:, 0], a[:, 1], a[:, 2], a[:, 3:]


def make_case(workdir, shape="demo", solution="eclipse", seed=12345, nlayer=100,
              tlow=400.0, thigh=3000.0, tempdelt=100.0, with_cia=True, with_grid=True,
              nlines=0, wnosamp=2160, extra_cfg=None, nfilters=None, overrides=None,
              cia_path=None, starrad=1.155, refpress=0.1, gsurf=1165.02,
              refradius_km=123820.0, ethresh=1e-6, nwidth=20, outputs=False, verb=0,
              no_opacity=False, cia_h2he=False, atm_path=None, mol_path=None, species=None,
              abund=None):
    """Create every input file of one configuration under `workdir`; returns paths + arrays.
    `species` / `abund`: the atmosphere's species and their uniform abundances (default SPECIES /
    UNIFORM); every grid molecule of the shape must be one of the species."""
    os.makedirs(workdir, exist_ok=True)
    sh = dict(SHAPES[shape]) if isinstance(shape, str) else dict(shape)
    if overrides:
        sh.update(overrides)
    P = lambda n: os.path.join(workdir, n)
    wn = wn_grid(sh["wnlow"], sh["wnhigh"], sh["wndelt"])
    press = pressure_grid(nlayer)
    temp = temperature_profile(press)
    species = list(SPECIES if species is None else species)
    abund = np.array(UNIFORM if abund is None else abund, dtype=float)
    case = dict(workdir=workdir, shape=sh, wn=wn, press_bar=press, temp=temp,
                abund=np.tile(abund, (nlayer, 1)), species=species, solution=solution,
                nlayer=nlayer)
    case["molfile"] = mol_path or write_molecules(P("molecules.dat"))
    if atm_path:          # an existing atmosphere file (e.g. the reference's shipped demo atmosphere)
        sp, _, press, temp, ab = read_tea_atm(atm_path)
        nlayer = len(press)
        case.update(press_bar=press, temp=temp, abund=ab, species=list(sp), nlayer=nlayer, atm=atm_path)
    else:
        case["atm"] = write_atm(P("atm.dat"), press, temp, abund, species=species, gsurf=gsurf,
                                r0_km=refradius_km * 0.97)
    if with_cia:
        case["cia"] = cia_path or write_cia(P("CIA_H2H2_synth.dat"))
        if cia_h2he:      # a second, two-species table like examples/WASP-12b/BART.cfg's H2-He file
            t2 = np.array([1000, 1500, 2000, 2500, 3000, 4000, 5000], dtype=float)
            case["cia"] += "," + write_cia(P("CIA_H2He_synth.dat"), pair=("H2", "He"), temps=t2,
                                           wn=np.arange(50.0, 12001.0, 25.0), seed=8)
    molids = [MOL_BY_NAME[m][0] for m in sh["mols"]]
    temps = np.arange(tlow, thigh + 0.5 * tempdelt, tempdelt)
    case["grid_temps"] = temps
    case["grid_molids"] = molids
    case["opacity"] = P("opacity.dat")
    if with_grid:
        o = synth_opacity_grid(nlayer, temps, molids, wn, press, seed=seed + 1)
        write_opacity(case["opacity"], molids, temps, press * 1e6, wn, o)
        case["grid"] = o
    # TLI: always present (header is read at every init, readlineinfo.c:544-614)
    dbs = []
    iso_table = {"CH4": [("61", 16.0313, 0.98827), ("62", 17.03466, 0.0111031)],
                 "H2O": [("161", 18.010565, 0.997317), ("181", 20.014811, 0.00199983)],
                 "CO2": [("626", 43.98983, 0.98420)],
                 "CO": [("26", 27.994915, 0.98654), ("36", 28.99827, 0.01108)],
                 "NH3": [("4111", 17.026549, 0.995872)]}
    for m in sh["mols"]:
        dbs.append(("HITRAN " + m, m, iso_table[m]))
    case["tli"] = P("lines.tli")
    case["lines"] = write_tli(case["tli"], sh["wnlow"], sh["wnhigh"], max(nlines, len(dbs) * 4),
                              dbs=dbs, seed=seed)
    # filters
    if nfilters is None:
        nfilters = 10 if len(sh["mols"]) == 1 else 4
    wl_lo, wl_hi = 1e4 / wn[-1], 1e4 / wn[0]
    edges = np.linspace(wl_lo * 1.002, wl_hi * 0.998, nfilters + 1)
    case["filters"] = [write_filter(P("filter%02d.dat" % i), edges[i], edges[i + 1])
                       for i in range(nfilters)]
    # transit cfg (the file makecfg.makeTransit would write, makecfg.py:23-108)
    lines = ["atm %s" % case["atm"], "molfile %s" % case["molfile"], "linedb %s" % case["tli"]]
    if not no_opacity:      # without it transit computes the extinction line by line (tau.c:163-175)
        lines.append("opacityfile %s" % case["opacity"])
    if with_cia:
        lines.append("csfile %s" % case["cia"])
    lines += ["wnlow %.10g" % sh["wnlow"], "wnhigh %.10g" % sh["wnhigh"],
              "wndelt %.10g" % sh["wndelt"], "wnosamp %d" % wnosamp, "wlfct 1e-4", "wnfct 1.0",
              "solution %s" % solution, "raygrid 0 20 40 60 80",
              "toomuch %.10g" % sh["toomuch"], "ethresh %g" % ethresh, "nwidth %d" % nwidth,
              "tlow %.10g" % tlow, "thigh %.10g" % thigh, "tempdelt %.10g" % tempdelt,
              "refpress %.10g" % refpress, "refradius %.10g" % refradius_km,
              "gsurf %.10g" % gsurf, "starrad %.10g" % starrad, "verb %d" % verb]
    if outputs:
        lines += ["outspec %s" % P("outspec.dat")]
    else:
        lines += ["outspec /dev/null"]
    if extra_cfg:
        lines += list(extra_cfg)
    case["cfg"] = P("transit.cfg")
    with open(case["cfg"], "w") as f:
        f.write("# synthetic transit configuration (bart_b200.synth)\n")
        f.write("\n".join(lines) + "\n")
    case["refpress"], case["gsurf"], case["refradius_km"] = refpress, gsurf, refradius_km
    case["starrad"] = starrad
    return case


def make_models(case, M, seed=99, molfit=("CH4",), tmin=400.0, tmax=3000.0, radius_jitter=0.0):
    """M proposal models in the layout run_transit() takes (BARTfunc.py:213-222,333-363):
    profiles[m] = [T(layer 0..n-1), q_species0(layers), q_species1(layers), ...], layers
    bottom -> top.  T profiles are smooth random members of the family above; abundances of the
    `molfit` species are scaled by 10^U(-2, 1.5) and H2/He renormalised as BARTfunc does."""
    rng = np.random.default_rng(seed)
    press = case["press_bar"]
    species = case["species"]
    nlayer = len(press)
    nspec = len(species)
    base = case["abund"]
    iH2, iHe = species.index("H2"), species.index("He")
    imetals = [i for i, s in enumerate(species) if s not in ("H2", "He")]
    ratio = base[:, iH2] / base[:, iHe]
    out = np.zeros((M, (nspec + 1) * nlayer))
    for m in range(M):
        while True:
            t_deep = rng.uniform(1300.0, 2800.0)
            t_top = rng.uniform(600.0, min(t_deep, 2000.0))
            if rng.uniform() < 0.25:           # thermal inversion
                t_deep, t_top = t_top, t_deep
            knee = 10.0 ** rng.uniform(-2.5, 0.5)
            width = rng.uniform(0.4, 1.5)
            T = temperature_profile(press, t_deep, t_top, knee, width)
            T = T + 15.0 * np.sin(np.log10(press) * rng.uniform(1.0, 3.0) + rng.uniform(0, 6.28))
            if T.min() > max(tmin, 1.0) + 5 and T.max() < tmax - 5:
                break
        q = base.copy()
        for name in molfit:
            q[:, species.index(name)] *= 10.0 ** rng.uniform(-2.0, 1.5)
        rest = 1.0 - q[:, imetals].sum(axis=1)
        q[:, iH2] = ratio * rest / (1.0 + ratio)
        q[:, iHe] = rest / (1.0 + ratio)
        prof = np.vstack([T[None, :], q.T])
        out[m] = prof.ravel()
    return out


def write_synth_opacity_stream(path, nlayer, temps, molids, wn, press_bar, seed=2026):
    """Large grids (the high-resolution sweep: 1e5-1e6 wavenumbers, several GB): the same
    envelope/spike/hot-band model as synth_opacity_grid without the per-cell noise, written layer
    by layer so that the array never has to sit in host memory."""
    rng = np.random.default_rng(seed)
    nT, nmol, nw = len(temps), len(molids), len(wn)
    x = (wn - wn[0]) / max(wn[-1] - wn[0], 1.0)
    tt = (np.asarray(temps) / 1000.0)[:, None]
    logo = np.empty((nmol, nT, nw))
    for m in range(nmol):
        centers = rng.uniform(0.0, 1.0, 4)
        widths = rng.uniform(0.05, 0.2, 4)
        amps = rng.uniform(-1.0, 2.0, 4)
        env = np.full(nw, -4.0)
        for c, w, a in zip(centers, widths, amps):
            env = np.maximum(env, a - 3.0 * ((x - c) / w) ** 2)
        base = env + rng.uniform(-1.5, 1.0, nw)
        hot = rng.uniform(0.2, 1.5, nw)
        logo[m] = base[None, :] + hot[None, :] * (tt - 1.0)
    with open(path, "wb") as f:
        f.write(struct.pack("4l", nmol, nT, nlayer, nw))
        f.write(np.asarray(molids, dtype=np.int32).tobytes())
        f.write(np.asarray(temps, dtype=np.float64).tobytes())
        f.write((np.asarray(press_bar) * 1e6).astype(np.float64).tobytes())
        f.write(np.asarray(wn, dtype=np.float64).tobytes())
        for r in range(nlayer):
            pfac = 0.15 * np.log10(press_bar[r] / 1e-5) / 7.0
            # [T][mol][wave] for this layer
            f.write(np.ascontiguousarray(np.transpose(10.0 ** (logo * (1.0 - pfac)), (1, 0, 2))).tobytes())
    return path


def make_hr_case(workdir, nwave=100001, ntemp=20, solution="eclipse", seed=2026):
    """High-resolution sweep shape (BASELINE.json configs[4]): nwave samples over 910-3333 cm-1,
    100 layers, ntemp grid temperatures from 400 K in 100 K steps, 4 molecules + H2-H2 CIA."""
    wnlow, wnhigh = 910.0, 3333.0
    wndelt = (wnhigh - wnlow) / (nwave - 1)
    thigh = 400.0 + 100.0 * (ntemp - 1)
    sh = dict(wnlow=wnlow, wnhigh=wnhigh, wndelt=wndelt, mols=["H2O", "CO2", "CO", "CH4"], toomuch=10.0)
    case = make_case(workdir, shape=sh, solution=solution, seed=seed, thigh=thigh, with_grid=False)
    wn = case["wn"]
    write_synth_opacity_stream(case["opacity"], case["nlayer"], case["grid_temps"], case["grid_molids"],
                               wn, case["press_bar"], seed=seed + 1)
    return case
