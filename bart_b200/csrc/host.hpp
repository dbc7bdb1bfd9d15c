// host.hpp -- internal host-side state of libbart_b200 (not part of the C ABI).
#pragma once
#include <string>
#include <vector>
#include <cstdio>
#include <cstdint>
#include <fcntl.h>
#include <unistd.h>

namespace bart {

// ---- physical constants, CGS (reference: transit/include/constants_tr.h:20-46) ----
constexpr double kPI = 3.141592653589793;
constexpr double kDEG = kPI / 180.0;
constexpr double kAMU = 1.66053886e-24;
constexpr double kLS = 2.99792458e10;
constexpr double kKB = 1.380658e-16;
constexpr double kH = 6.6260755e-27;
constexpr double kEC = 4.8032068e-10;
constexpr double kME = 9.1093897e-28;
constexpr double kAMAGAT = 2.68678e19;
constexpr double kE0H2 = 4.911e-23;
constexpr double kNAVO = 6.02214076e23;
constexpr double kMICRON = 1e-4;
constexpr double kANGSTROM = 1e-8;
constexpr double kSUNRADIUS = 6.957e10;
constexpr double kSIGCTE = kPI * kEC * kEC / kLS / kLS / kME / kAMU;
constexpr double kEXPCTE = kH * kLS / kKB;
constexpr double kSQRTLN2 = 0.83255461115769775635;

// ---- error handling ----
void fail(const char *fmt, ...);          // records message; exits in mode 0 (reference behaviour)
void warn(int level, const char *fmt, ...);
extern int g_verb;

// ---- file owners: closed when the owner goes, so a fail() that throws leaks no handle ----
struct Fd {                               // open(); fd < 0 when that failed
  int fd;
  Fd(const char *path, int flags, mode_t mode = 0) : fd(open(path, flags, mode)) {}
  ~Fd() { if (fd >= 0) close(fd); }
  Fd(const Fd &) = delete;
  Fd &operator=(const Fd &) = delete;
  operator int() const { return fd; }
};
struct File {                             // fopen(); null when that failed
  FILE *f;
  File(const char *path, const char *mode) : f(fopen(path, mode)) {}
  ~File() { if (f) fclose(f); }
  File(File &&o) noexcept : f(o.f) { o.f = nullptr; }
  File(const File &) = delete;
  File &operator=(const File &) = delete;
  operator FILE *() const { return f; }
};

// ---- options (reference: transit/src/argum.c:112-320 table, 372-739 handling) ----
struct Options {
  std::string atm, linedb, outtoomuch, outsample, outspec = "outspectrum", outintens;
  std::string molfile = "../inputs/molecules.dat", opacityfile, saveext;
  bool savefiles = false;
  double raddelt = -1, radlow = 0, radhigh = 0, radfct = 0;
  double allowq = 0.00001f;
  double refpress = 0, refradius = 0, gsurf = 0;
  std::string qmol, qscale;
  double wllow = 0, wlhigh = 0, wlfct = 1e-4;
  double wnlow = 0, wnhigh = 0, wndelt = 0, wnfct = 0;
  int wnosamp = 2160;
  int ndop = 60, nlor = 60;
  float dmin = 1e-3f, dmax = 0.25f, lmin = 1e-4f, lmax = 10.0f;   // float like the hint struct
  float nwidth = 20;
  double ethreshold = 1e-8;
  int cloud_flag = 0;
  double cloudext = 0, cloudtop = 0, cloudbot = 0;
  int scat_flag = 0;
  double scat_logext = 0;
  std::vector<std::string> csfiles;
  double tlow = 500, thigh = 3000, tempdelt = 100;
  bool justOpacity = false, shareOpacity = false;
  std::string solution = "eclipse";
  double toomuch = 20;
  int taulevel = 1, modlevel = 1;
  double starrad = 1.125;
  bool transparent = false;
  std::string raygrid = "0 20 40 60 80";
  int verb = 2;
};
void parse_options(int argc, char **argv, Options &o);

// ---- inputs ----
struct Atmosphere {   // reference: transit/src/readatm.c:23-114,255-620
  std::vector<std::string> species;
  std::vector<double> radius, press, temp;      // [nlayer], file units, bottom -> top
  std::vector<double> q;                        // [nspec][nlayer]
  double rfct = 1, pfct = 1, tfct = 1;
  bool mass_abund = false;
  int nlayer() const { return (int)press.size(); }
  int nspec() const { return (int)species.size(); }
};
void read_atmosphere(const std::string &path, Atmosphere &a);

struct Molecules {    // per atmosphere species; reference: readatm.c:625-717
  std::vector<int> id;
  std::vector<double> mass, radius_cm, pol;
};
void read_molecules(const std::string &path, const Atmosphere &a, Molecules &m);

struct TliDb {
  std::string name, molname;
  std::vector<double> T;
  int first_iso = 0, niso = 0;
};
struct Tli {          // reference: transit/src/readlineinfo.c:87-244,416-537
  bool present = false;
  double wl_ini = 0, wl_fin = 0;
  std::vector<TliDb> db;
  std::vector<std::string> iso_name;
  std::vector<double> iso_mass, iso_ratio;
  std::vector<int> iso_db;
  std::vector<std::vector<double>> iso_Z;       // [niso][nT of its db]
  double tmin = 0.0, tmax = 70000.0;
  long long data_offset = 0;
  // line data (only loaded by the grid builder)
  std::vector<double> wl, elow, gf;
  std::vector<short> isoid;
  int niso() const { return (int)iso_name.size(); }
};
void read_tli_header(const std::string &path, Tli &t);
void read_tli_lines(const std::string &path, Tli &t, double wnlow, double wnhigh);
// Where the in-range lines sit in the file (readdatarng's per-isotope binary searches,
// readlineinfo.c:416-537) without reading them: byte offsets of the four columns and, per isotope,
// the first record and the record count of its slice.
struct TliLineMap {
  long long nlines = 0;                     // records in the file
  long long wl_off = 0, iso_off = 0, el_off = 0, gf_off = 0;   // column starts (bytes)
  std::vector<long long> first, count;      // per isotope with lines in the file
  long long total = 0;                      // sum of count
};
void map_tli_lines(const std::string &path, const Tli &t, double wnlow, double wnhigh, TliLineMap &m);
// pread of `bytes` at file offset `off` into `dst`, split over a few threads (one thread copies out
// of the page cache at 2-3 GB/s; the staging buffers of the grid and line-list uploads are filled
// several times faster this way).  Returns false on a short read.
bool parallel_pread(int fd, void *dst, size_t bytes, long long off);

struct CiaTable {     // reference: transit/src/crosssec.c:9-268
  std::string file;
  std::vector<std::string> species;
  std::vector<double> temp, wn, tab;            // tab[nwn][nt]
};
void read_cia(const std::string &path, CiaTable &c);
void fold_cia_table(const CiaTable &c, const std::vector<double> &wn, std::vector<double> &P,
                    std::vector<double> &Q);

struct OpacityGrid {  // reference: transit/src/opacity.c:406-421,432-503
  long nmol = 0, ntemp = 0, nlayer = 0, nwave = 0;
  std::vector<int> molid;
  std::vector<double> temp, press, wn;
  long long data_offset = 0;
};
bool read_opacity_header(const std::string &path, OpacityGrid &g);
void write_opacity_file(const std::string &path, const OpacityGrid &g, const double *o);

// natural cubic spline helpers (reference: pu/src/spline.c) used at init only
void spline_second_derivs(const double *x, const double *y, long n, double *z);
double spline_eval(const double *z, long n, const double *x, const double *y, double xo);
int nearest_index(const double *a, double v, int lo, int hi);   // pu/src/iomisc.c:1088-1108

std::vector<double> make_sampling(double lo, double hi, double d, int osamp);  // makesample.c:77-104

}  // namespace bart
