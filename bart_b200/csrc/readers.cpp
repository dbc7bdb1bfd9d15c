// readers.cpp -- input formats of the transit forward model, parsed once at init on the host.
// Each reader follows the byte/field layout the reference reads (cited per function); none of
// this runs per model.
#include "host.hpp"
#include <sys/mman.h>
#include <sys/stat.h>
#include <fcntl.h>
#include <unistd.h>
#include <cmath>
#include <cstring>
#include <cstdlib>
#include <cctype>
#include <fstream>
#include <sstream>
#include <algorithm>
#include <thread>
#include <atomic>

namespace bart {

namespace {
std::vector<std::string> split_ws(const std::string &s) {
  std::vector<std::string> out;
  std::istringstream is(s);
  std::string w;
  while (is >> w) out.push_back(w);
  return out;
}
bool blank(const std::string &s) {
  for (char c : s) if (!isspace((unsigned char)c)) return false;
  return true;
}
}  // namespace

// ---------------------------------------------------------------------------------------
// Atmosphere file.  Reference: transit/src/readatm.c:255-404 (keywords: `#SPECIES`, q, z, ur/up/ut,
// n) and 425-620 (data rows: radius pressure temperature abundances..., '#' and blank lines
// skipped, layers re-sorted bottom -> top when given top -> bottom).
void read_atmosphere(const std::string &path, Atmosphere &a) {
  if (path.empty() || path == "-") fail("getatm() :: No atmospheric file specified.");
  std::ifstream in(path);
  if (!in) fail("Atmospheric info file '%s' cannot be opened.", path.c_str());
  std::string line;
  double zerorad = 0.0;
  bool in_data = false;
  std::vector<std::vector<double>> rows;
  while (std::getline(in, line)) {
    if (!line.empty() && line.back() == '\r') line.pop_back();
    if (blank(line)) continue;
    if (!in_data) {
      char c = line[0];
      if (c == '#') {
        std::vector<std::string> w = split_ws(line.substr(1));
        if (!w.empty() && w[0] == "SPECIES") {
          if (!std::getline(in, line)) fail("readatm :: EOF after #SPECIES in '%s'", path.c_str());
          a.species = split_ws(line);
        }
        continue;
      }
      if (c == 'q') {
        size_t p = 1;
        while (p < line.size() && line[p] == ' ') p++;
        char t = p < line.size() ? (char)(line[p] | 0x20) : 0;
        if (t == 'n') a.mass_abund = false;
        else if (t == 'm') a.mass_abund = true;
        else warn(1, "'q' option in the atmosphere file can only be followed by 'm' or 'n'.");
        continue;
      }
      if (c == 'z') { zerorad = atof(line.c_str() + 1); continue; }
      if (c == 'u') {
        char k = line.size() > 1 ? line[1] : 0;
        double v = atof(line.c_str() + 2);
        if (k == 'r') a.rfct = v; else if (k == 'p') a.pfct = v; else if (k == 't') a.tfct = v;
        else fail("Invalid unit factor indication in atmosphere file.");
        continue;
      }
      if (c == 'n') continue;
      in_data = true;                      // first non-keyword line starts the data block
    }
    if (line[0] == '#') continue;
    std::vector<std::string> w = split_ws(line);
    std::vector<double> r;
    for (auto &s : w) {
      char *e; double v = strtod(s.c_str(), &e);
      if (e == s.c_str()) fail("Atmosphere file '%s': invalid field '%s'", path.c_str(), s.c_str());
      if (v < 0) fail("Atmosphere file '%s': negative value (%g).", path.c_str(), v);
      r.push_back(v);
    }
    rows.push_back(r);
  }
  if (a.species.empty())
    fail("No species were found in the atmospheric file, make sure to specify them with the "
         "comment/header in the previous line '#SPECIES'.");
  const int ns = a.nspec();
  const int nl = (int)rows.size();
  if (nl < 1) fail("readatm :: no t,p data points in '%s'", path.c_str());
  a.radius.resize(nl); a.press.resize(nl); a.temp.resize(nl);
  a.q.assign((size_t)ns * nl, 0.0);
  for (int r = 0; r < nl; r++) {
    if ((int)rows[r].size() < 3 + ns)
      fail("Atmosphere file '%s': a data line contains %d abundance values, when there were %d "
           "expected.", path.c_str(), (int)rows[r].size() - 3, ns);
    a.radius[r] = rows[r][0] + zerorad;
    a.press[r] = rows[r][1];
    a.temp[r] = rows[r][2];
    for (int j = 0; j < ns; j++) a.q[(size_t)j * nl + r] = rows[r][3 + j];
  }
  bool sorted = true, reversed = true;
  for (int i = 0; i < nl - 1; i++) {
    if (a.radius[i] >= a.radius[i + 1] || a.press[i] <= a.press[i + 1]) sorted = false;
    if (a.radius[i] <= a.radius[i + 1] || a.press[i] >= a.press[i + 1]) reversed = false;
  }
  if (nl > 1 && !sorted && !reversed)
    fail("The atmospheric layers are neither sorted from the bottom up, nor from the top down.");
  if (nl > 1 && reversed) {
    warn(1, "The atmospheric layers are in reversed order (top-bottom). Resorting to be from the "
            "bottom-up.");
    std::reverse(a.radius.begin(), a.radius.end());
    std::reverse(a.press.begin(), a.press.end());
    std::reverse(a.temp.begin(), a.temp.end());
    for (int j = 0; j < ns; j++)
      std::reverse(a.q.begin() + (size_t)j * nl, a.q.begin() + (size_t)(j + 1) * nl);
  }
}

// ---------------------------------------------------------------------------------------
// molecules.dat.  Reference: transit/src/readatm.c:625-717 -- columns ID, name, mass, diameter
// (Angstrom; radius = diameter/2), source tag, polarizability; the table ends at the first
// blank or comment line after its first data row.
void read_molecules(const std::string &path, const Atmosphere &a, Molecules &m) {
  std::ifstream in(path);
  if (!in) fail("Molecular info file '%s' cannot be opened.", path.c_str());
  struct Row { int id; std::string name; double mass, radius, pol; };
  std::vector<Row> rows;
  std::string line;
  bool started = false;
  while (std::getline(in, line)) {
    bool skip = blank(line) || line[0] == '#';
    if (skip) { if (started) break; else continue; }
    started = true;
    std::vector<std::string> w = split_ws(line);
    if (w.size() < 4) continue;
    Row r;
    r.id = (int)strtol(w[0].c_str(), nullptr, 10);
    r.name = w[1];
    r.mass = strtod(w[2].c_str(), nullptr);
    r.radius = strtod(w[3].c_str(), nullptr) / 2.0;
    r.pol = w.size() > 5 ? strtod(w[5].c_str(), nullptr) : 0.0;
    rows.push_back(r);
  }
  const int ns = a.nspec();
  m.id.resize(ns); m.mass.resize(ns); m.radius_cm.resize(ns); m.pol.resize(ns);
  for (int i = 0; i < ns; i++) {
    int j = -1;
    for (size_t k = 0; k < rows.size(); k++) if (rows[k].name == a.species[i]) { j = (int)k; break; }
    if (j < 0)
      fail("The atmospheric species '%s' is not present in the list of known species:\n '%s'.",
           a.species[i].c_str(), path.c_str());
    m.id[i] = rows[j].id; m.mass[i] = rows[j].mass;
    m.radius_cm[i] = rows[j].radius * kANGSTROM; m.pol[i] = rows[j].pol;
  }
}

// ---------------------------------------------------------------------------------------
// TLI v6.  Reference: transit/src/readlineinfo.c:87-244 (header), 416-537 (line data); writer of
// record modules/transit/pylineread/src/pylineread.py:185-428.
namespace {
template <class T> T rd(FILE *f) {
  T v;
  if (fread(&v, sizeof(T), 1, f) != 1) fail("TLI file: unexpected end of file");
  return v;
}
std::string rdstr(FILE *f) {
  unsigned short n = rd<unsigned short>(f);
  std::string s(n, '\0');
  if (n && fread(&s[0], 1, n, f) != n) fail("TLI file: unexpected end of file");
  return s;
}
}  // namespace

void read_tli_header(const std::string &path, Tli &t) {
  t = Tli();
  if (path.empty()) { warn(1, "No TLI file set."); return; }
  const File f(path.c_str(), "rb");
  if (!f) fail("Line info file '%s' is not found.", path.c_str());
  (void)rd<int32_t>(f);                                     // endianness magic
  unsigned short ver = rd<unsigned short>(f);
  unsigned short lrv = rd<unsigned short>(f), lrr = rd<unsigned short>(f);
  if (ver != 6)
    fail("The version of the TLI file: %i (lineread v%i.%i) is not compatible with this version "
         "of transit, which can only read version 6.", ver, lrv, lrr);
  t.wl_ini = rd<double>(f);
  t.wl_fin = rd<double>(f);
  unsigned short ndb = rd<unsigned short>(f);
  int niso = 0;
  for (int i = 0; i < ndb; i++) {
    TliDb db;
    db.name = rdstr(f);
    db.molname = rdstr(f);
    unsigned short nT = rd<unsigned short>(f), nI = rd<unsigned short>(f);
    db.T.resize(nT);
    if (fread(db.T.data(), sizeof(double), nT, f) != nT) fail("TLI file: truncated");
    t.tmin = std::max(t.tmin, db.T.front());
    t.tmax = std::min(t.tmax, db.T.back());
    db.first_iso = niso; db.niso = nI;
    for (int j = 0; j < nI; j++) {
      t.iso_name.push_back(rdstr(f));
      t.iso_mass.push_back(rd<double>(f));
      t.iso_ratio.push_back(rd<double>(f));
      std::vector<double> Z(nT);
      if (fread(Z.data(), sizeof(double), nT, f) != nT) fail("TLI file: truncated");
      t.iso_Z.push_back(Z);
      t.iso_db.push_back(i);
    }
    niso += nI;
    t.db.push_back(db);
  }
  t.data_offset = ftell(f);
  t.present = true;
}

// Lines inside [wnlow, wnhigh], per isotope block, by the same boundary rule as the reference's
// on-disk binary search + linear refinement (readlineinfo.c:16-77, 496-525): first record with
// wl >= iniw ... last record with wl <= finw, but never an empty slice (the reference always
// reads at least the record its search lands on).
// The line block is memory-mapped: the per-isotope binary searches touch O(log n) pages of the
// wavelength array and only the selected slices of the four columns are copied, so a 1e8-line TLI
// (2.6 GB) costs what its in-range part costs.  Selection = readdatarng (readlineinfo.c:416-537).
bool parallel_pread(int fd, void *dst, size_t bytes, long long off) {
  auto part = [fd](char *d, size_t n, long long o) {
    while (n > 0) {
      const ssize_t got = pread(fd, d, n, (off_t)o);
      if (got <= 0) return false;
      d += got; o += got; n -= (size_t)got;
    }
    return true;
  };
  int nthr = 4;
  if (const char *e = getenv("BART_IO_THREADS")) nthr = std::max(1, std::min(16, atoi(e)));
  if (bytes < ((size_t)4 << 20) || nthr == 1) return part((char *)dst, bytes, off);
  const size_t per = ((bytes + nthr - 1) / nthr + 4095) & ~(size_t)4095;
  std::atomic<bool> ok(true);
  std::vector<std::thread> th;
  for (int k = 0; k < nthr; k++) {
    const size_t b0 = (size_t)k * per;
    if (b0 >= bytes) break;
    const size_t n = std::min(per, bytes - b0);
    th.emplace_back([&, b0, n] { if (!part((char *)dst + b0, n, off + (long long)b0)) ok = false; });
  }
  for (auto &t : th) t.join();
  return ok;
}

namespace {
struct Mapping {                          // read-only mmap of a whole file, unmapped when it goes
  void *p;
  size_t size;
  Mapping(int fd, size_t n) : p(mmap(nullptr, n, PROT_READ, MAP_PRIVATE, fd, 0)), size(n) {}
  ~Mapping() { if (p != MAP_FAILED) munmap(p, size); }
  Mapping(const Mapping &) = delete;
  Mapping &operator=(const Mapping &) = delete;
};
}  // namespace

void map_tli_lines(const std::string &path, const Tli &t, double wnlow, double wnhigh, TliLineMap &m) {
  const Fd fd(path.c_str(), O_RDONLY);
  if (fd < 0) fail("Data file '%s' not found.", path.c_str());
  struct stat st;
  if (fstat(fd, &st) != 0) fail("Data file '%s': cannot stat.", path.c_str());
  const size_t fsize = (size_t)st.st_size;
  const Mapping map(fd, fsize);
  if (map.p == MAP_FAILED) fail("Data file '%s': mmap failed.", path.c_str());
  const char *base = (const char *)map.p;
  auto need = [&](long long off, long long bytes) {
    if (off < 0 || bytes < 0 || (size_t)(off + bytes) > fsize) fail("TLI file: truncated");
  };
  long long pos = t.data_offset;
  need(pos, 12);
  long long nlines; int niso;
  memcpy(&nlines, base + pos, 8); pos += 8;
  memcpy(&niso, base + pos, 4); pos += 4;
  need(pos, (long long)niso * 8);
  std::vector<long long> per(niso);
  memcpy(per.data(), base + pos, (size_t)niso * 8); pos += (long long)niso * 8;
  const long long start = pos;
  m = TliLineMap();
  m.nlines = nlines;
  m.wl_off = start; m.iso_off = start + nlines * 8; m.el_off = m.iso_off + nlines * 2;
  m.gf_off = m.el_off + nlines * 8;
  need(m.gf_off, nlines * 8);
  // the columns are not 8-byte aligned in the file in general: copy through memcpy
  auto wl_at = [&](long long i) { double v; memcpy(&v, base + start + i * 8, 8); return v; };
  const double iniw = 1.0 / wnhigh / 1e-4, finw = 1.0 / wnlow / 1e-4;   // micron
  long long off = 0;
  for (int i = 0; i < niso; i++) {
    const long long n = per[i];
    long long first = 0, nread = 0;
    if (n > 0) {
      auto w = [&](long long k) { return wl_at(off + k); };
      // datafileBS(..., up=0): binary search then walk down while the previous record >= target
      long long lo = 0, hi = n - 1;
      do { long long loc = (hi + lo) / 2; if (iniw > w(loc)) lo = loc; else hi = loc; } while (hi - lo > 1);
      first = hi;
      while (first > 0 && !(w(first - 1) < iniw)) first--;
      // datafileBS(..., up=1): walk up while the next record <= target
      lo = 0; hi = n - 1;
      do { long long loc = (hi + lo) / 2; if (finw > w(loc)) lo = loc; else hi = loc; } while (hi - lo > 1);
      long long last = lo;
      while (last < n - 1 && !(w(last + 1) > finw)) last++;
      nread = std::max<long long>(0, last - first + 1);
    }
    m.first.push_back(off + first);
    m.count.push_back(nread);
    m.total += nread;
    off += n;
  }
}

void read_tli_lines(const std::string &path, Tli &t, double wnlow, double wnhigh) {
  TliLineMap m;
  map_tli_lines(path, t, wnlow, wnhigh, m);
  const Fd fd(path.c_str(), O_RDONLY);
  if (fd < 0) fail("Data file '%s' not found.", path.c_str());
  t.wl.assign((size_t)m.total, 0.0); t.elow.assign((size_t)m.total, 0.0); t.gf.assign((size_t)m.total, 0.0);
  t.isoid.assign((size_t)m.total, 0);
  auto rd = [&](void *dst, long long off, long long bytes) {
    char *d = (char *)dst;
    while (bytes > 0) {
      const ssize_t got = pread(fd, d, (size_t)bytes, (off_t)off);
      if (got <= 0) fail("TLI file: read failed");
      d += got; off += got; bytes -= got;
    }
  };
  size_t b0 = 0;
  for (size_t i = 0; i < m.count.size(); i++) {
    const long long f = m.first[i], n = m.count[i];
    if (n <= 0) continue;
    rd(t.wl.data() + b0, m.wl_off + f * 8, n * 8);
    rd(t.isoid.data() + b0, m.iso_off + f * 2, n * 2);
    rd(t.elow.data() + b0, m.el_off + f * 8, n * 8);
    rd(t.gf.data() + b0, m.gf_off + f * 8, n * 8);
    b0 += (size_t)n;
  }
}

// ---------------------------------------------------------------------------------------
// CIA table.  Reference: transit/src/crosssec.c:83-252 -- `i A [B]` species line, `t T1 T2 ...`
// temperatures (optional trailing K), then rows `wavenumber v(T1) v(T2) ...`.
void read_cia(const std::string &path, CiaTable &c) {
  std::ifstream in(path);
  if (!in) fail("Cannot read cross-section file '%s'.", path.c_str());
  c = CiaTable();
  c.file = path;
  std::string line;
  while (std::getline(in, line)) {
    if (blank(line) || line[0] == '#') continue;
    size_t p = 0;
    while (p < line.size() && isspace((unsigned char)line[p])) p++;
    char k = line[p];
    if (k == 'i' && c.wn.empty() && isspace((unsigned char)line[p + 1])) {
      c.species = split_ws(line.substr(p + 1));
      if (c.species.size() != 1 && c.species.size() != 2)
        fail("Wrong header in cross section file '%s', The 'i'-line should contain either one "
             "or two species.", path.c_str());
      continue;
    }
    if (k == 't' && c.wn.empty() && isspace((unsigned char)line[p + 1])) {
      for (auto &s : split_ws(line.substr(p + 1))) c.temp.push_back(strtod(s.c_str(), nullptr));
      continue;
    }
    if (c.temp.empty()) fail("File '%s' has data before the temperature line.", path.c_str());
    std::vector<std::string> w = split_ws(line);
    if (w.size() < c.temp.size() + 1)
      fail("Less fields (%d) than expected (%d) were read for the %dth wavenumber in the "
           "cross-section file '%s'.", (int)w.size() - 1, (int)c.temp.size(), (int)c.wn.size() + 1,
           path.c_str());
    c.wn.push_back(strtod(w[0].c_str(), nullptr));
    for (size_t i = 0; i < c.temp.size(); i++) c.tab.push_back(strtod(w[i + 1].c_str(), nullptr));
  }
  if (c.wn.empty()) fail("File '%s' finished before opacity info.", path.c_str());
}

// ---------------------------------------------------------------------------------------
// Opacity grid file.  Reference: transit/src/opacity.c:406-421 (write), 432-503 (read):
// long Nmol, Ntemp, Nlayer, Nwave; int molID[Nmol]; double temp[Ntemp]; double press[Nlayer]
// (barye); double wns[Nwave]; double o[Nlayer][Ntemp][Nmol][Nwave] (cm2/g), native endian.
bool read_opacity_header(const std::string &path, OpacityGrid &g) {
  const File f(path.c_str(), "rb");
  if (!f) return false;
  long dims[4];
  if (fread(dims, sizeof(long), 4, f) != 4) fail("Opacity file '%s' is truncated.", path.c_str());
  g.nmol = dims[0]; g.ntemp = dims[1]; g.nlayer = dims[2]; g.nwave = dims[3];
  if (g.nmol <= 0 || g.ntemp <= 1 || g.nlayer <= 0 || g.nwave <= 0 || g.nmol > 1000 ||
      g.ntemp > 100000 || g.nlayer > 100000)
    fail("Opacity file '%s' has an invalid header.", path.c_str());
  g.molid.resize(g.nmol); g.temp.resize(g.ntemp); g.press.resize(g.nlayer); g.wn.resize(g.nwave);
  bool ok = fread(g.molid.data(), sizeof(int), g.nmol, f) == (size_t)g.nmol &&
            fread(g.temp.data(), 8, g.ntemp, f) == (size_t)g.ntemp &&
            fread(g.press.data(), 8, g.nlayer, f) == (size_t)g.nlayer &&
            fread(g.wn.data(), 8, g.nwave, f) == (size_t)g.nwave;
  g.data_offset = ftell(f);
  if (!ok) fail("Opacity file '%s' is truncated.", path.c_str());
  return true;
}

void write_opacity_file(const std::string &path, const OpacityGrid &g, const double *o) {
  const File f(path.c_str(), "wb");
  if (!f) fail("Opacity filename '%s' cannot be opened for writing.", path.c_str());
  long dims[4] = {g.nmol, g.ntemp, g.nlayer, g.nwave};
  fwrite(dims, sizeof(long), 4, f);
  fwrite(g.molid.data(), sizeof(int), g.nmol, f);
  fwrite(g.temp.data(), 8, g.ntemp, f);
  fwrite(g.press.data(), 8, g.nlayer, f);
  fwrite(g.wn.data(), 8, g.nwave, f);
  size_t n = (size_t)g.nlayer * g.ntemp * g.nmol * g.nwave;
  if (fwrite(o, 8, n, f) != n) fail("Short write on opacity file '%s'.", path.c_str());
}

// ---------------------------------------------------------------------------------------
// Natural cubic spline (reference: pu/src/spline.c:12-48 Thomas solve, 131-183 evaluation) and the
// nearest-index search (pu/src/iomisc.c:1088-1108).  Init-time only.
int nearest_index(const double *a, double v, int lo, int hi) {
  while (hi - lo > 1) {
    int mid = (hi + lo) / 2;
    if (a[mid] > v) hi = mid; else lo = mid;
  }
  if (hi == lo) return lo;
  return std::fabs(a[hi] - v) < std::fabs(a[lo] - v) ? hi : lo;
}

void spline_second_derivs(const double *x, const double *y, long n, double *z) {
  std::vector<double> h(n - 1), b(n - 1), u(n - 1, 0.0), v(n - 1, 0.0);
  for (long i = 0; i < n - 1; i++) { h[i] = x[i + 1] - x[i]; b[i] = (y[i + 1] - y[i]) / h[i]; }
  if (n > 2) {
    u[1] = 2 * (h[1] + h[0]);
    v[1] = 6 * (b[1] - b[0]);
    for (long i = 2; i < n - 1; i++) {
      u[i] = 2 * (h[i] + h[i - 1]) - h[i - 1] * h[i - 1] / u[i - 1];
      v[i] = 6 * (b[i] - b[i - 1]) - v[i - 1] * h[i - 1] / u[i - 1];
    }
  }
  z[0] = z[n - 1] = 0.0;
  for (long i = n - 2; i > 0; i--) z[i] = (v[i] - h[i] * z[i + 1]) / u[i];
}

double spline_eval(const double *z, long n, const double *x, const double *y, double xo) {
  int k = nearest_index(x, xo, 0, (int)n - 1);
  if (k == n - 1 || xo < x[k]) k--;
  if (x[k] == xo) return y[k];
  double h = x[k + 1] - x[k];
  if (!(h > 0)) return 0.0;
  double dx = xo - x[k];
  double a = (z[k + 1] - z[k]) / (6 * h), b = 0.5 * z[k];
  double c = (y[k + 1] - y[k]) / h - h / 6 * (z[k + 1] + 2 * z[k]);
  return y[k] + dx * (c + dx * (b + dx * a));
}

// CIA tables pre-folded through the wavenumber spline (see transit.cu setup_cia): P[k][w] is the
// natural-spline-in-wavenumber interpolant of table column k at spectrum sample w, Q[k][w] the
// same for the column of temperature second derivatives.  Reference steps being folded:
// bicubicinterpolate, crosssec.c:404-420.
void fold_cia_table(const CiaTable &c, const std::vector<double> &wn, std::vector<double> &P,
                    std::vector<double> &Q) {
  const int nx = (int)c.wn.size(), nt = (int)c.temp.size(), nw = (int)wn.size();
  std::vector<double> zT((size_t)nx * nt);
  for (int i = 0; i < nx; i++)
    spline_second_derivs(c.temp.data(), &c.tab[(size_t)i * nt], nt, &zT[(size_t)i * nt]);
  P.assign((size_t)nt * nw, 0.0);
  Q.assign((size_t)nt * nw, 0.0);
  std::vector<double> col(nx), z(nx);
  for (int k = 0; k < nt; k++)
    for (int pass = 0; pass < 2; pass++) {
      for (int i = 0; i < nx; i++) col[i] = pass == 0 ? c.tab[(size_t)i * nt + k] : zT[(size_t)i * nt + k];
      spline_second_derivs(c.wn.data(), col.data(), nx, z.data());
      std::vector<double> &dst = pass == 0 ? P : Q;
      for (int w = 0; w < nw; w++)
        dst[(size_t)k * nw + w] = spline_eval(z.data(), nx, c.wn.data(), col.data(), wn[w]);
    }
}

// Sampling: reference transit/src/makesample.c:27-120.  n = (long)(((1+1e-8) f - i)/d + 1), then
// oversampled n = (n-1) o + 1, v[k] = i + k (d/o).
std::vector<double> make_sampling(double lo, double hi, double d, int osamp) {
  if (hi < lo) fail("Hinted final value for wavenumber sampling (%g) is smaller than hinted "
                    "initial value %.8g.", hi, lo);
  if (d == 0) fail("Spacing (%g) was not hinted in wavenumber sampling.", d);
  if (osamp <= 0) fail("Invalid hinted oversampling for wavenumber sampling.");
  double excess = d < 0 ? -1e-8 : 1e-8;
  long long n = (long long)(((1.0 + excess) * hi - lo) / d + 1);
  if (n < 0) n = -n;
  n = (n - 1) * osamp + 1;
  double osd = d / (double)osamp;
  std::vector<double> v((size_t)n);
  for (long long k = 0; k < n; k++) v[(size_t)k] = lo + k * osd;
  return v;
}

}  // namespace bart
