// fits.cpp — lens-plane output: file naming (densitymaps.cpp:636-649) and a minimal FITS writer for what writeMaps
// (densitymaps.cpp:530-630) produces with CCfits: one primary HDU, BITPIX -32, NAXIS1 = NAXIS2 = npix, pixel
// [gx + npix*gy] big-endian IEEE float, plus the reference's keys.  Keywords longer than 8 characters or in lower
// case (DlLOW, DlUP, PHYSICALSIZE, PIXELUNIT, OMEGAMATTER, OMEGALAMBDA, nparttype0-5, m0-5) are written as ESO
// HIERARCH cards, which is what CFITSIO emits for them; astropy (Lens/kslicer.py:39-40,84-86) reads them
// transparently and case-insensitively.
#include "slicer_host.h"

#include <cctype>
#include <cstring>
#include <fstream>
#include <iostream>

namespace slicer
{

std::string fileOutput(const InputParams &p, const std::string &snappl, int label)
{
  char lab[32];
  snprintf(lab, sizeof(lab), "%i", label);
  if (p.simType == "Gadget" && !p.partinplanes)
    return p.directory + p.simulation + "." + snappl + ".plane_" + p.snpix + "_" + p.suffix + ".fits";
  if (p.simType == "Gadget" && p.partinplanes)
    return p.directory + p.simulation + "." + snappl + ".ptype" + lab + "_plane_" + p.snpix + "_" + p.suffix + ".fits";
  throw SliceError{"Output name format not recognized"};
}

static void card(std::string &hdr, const std::string &text)
{
  std::string c = text;
  c.resize(80, ' ');
  hdr += c;
}

static bool plain_keyword(const std::string &k)
{
  if (k.size() > 8)
    return false;
  for (char ch : k)
    if (!(isupper((unsigned char)ch) || isdigit((unsigned char)ch) || ch == '_' || ch == '-'))
      return false;
  return true;
}

static std::string value_card(const std::string &key, const std::string &value, const std::string &comment)
{
  char buf[128];
  if (plain_keyword(key))
    snprintf(buf, sizeof(buf), "%-8s= %20s", key.c_str(), value.c_str());
  else
    snprintf(buf, sizeof(buf), "HIERARCH %s = %s", key.c_str(), value.c_str());
  std::string c = buf;
  if (!comment.empty() && c.size() + 3 + comment.size() <= 80)
    c += " / " + comment;
  return c;
}

void writeFitsImage(const std::string &file, const float *map, int npix, const std::vector<std::pair<std::string, double>> &dkeys,
                    const std::vector<std::pair<std::string, long long>> &ikeys, const std::vector<std::string> &order)
{
  if (std::ifstream(file.c_str()))
    throw SliceError{"file exists: " + file}; // CFITSIO refuses to overwrite: FITS::CantCreate
  FILE *f = fopen(file.c_str(), "wb");
  if (!f)
    throw SliceError{"cannot create " + file};
  std::string hdr;
  card(hdr, value_card("SIMPLE", "T", "file does conform to FITS standard"));
  card(hdr, value_card("BITPIX", "-32", "number of bits per data pixel"));
  card(hdr, value_card("NAXIS", "2", "number of data axes"));
  card(hdr, value_card("NAXIS1", std::to_string(npix), "length of data axis 1"));
  card(hdr, value_card("NAXIS2", std::to_string(npix), "length of data axis 2"));
  card(hdr, value_card("EXTEND", "T", "FITS dataset may contain extensions"));
  for (const std::string &k : order)
  {
    char v[64];
    bool found = false;
    for (auto &d : dkeys)
      if (d.first == k)
      {
        snprintf(v, sizeof(v), "%.17G", d.second);
        if (!strchr(v, '.') && !strchr(v, 'E') && !strchr(v, 'N') && !strchr(v, 'I'))
          strcat(v, "."); // FITS real values carry a decimal point
        found = true;
      }
    for (auto &i : ikeys)
      if (i.first == k)
      {
        snprintf(v, sizeof(v), "%lld", i.second);
        found = true;
      }
    if (found)
      card(hdr, value_card(k, v, k == "PIXELUNIT" ? "Mass unit in M_Sun" : (k == "DlLOW" || k == "DlUP") ? "comoving distance in Mpc" : ""));
  }
  card(hdr, "END");
  hdr.resize((hdr.size() + 2879) / 2880 * 2880, ' ');
  bool ok = fwrite(hdr.data(), 1, hdr.size(), f) == hdr.size();
  const size_t n = (size_t)npix * npix;
  std::vector<uint32_t> row((size_t)npix); // FITS is big-endian: one vectorisable byte swap per row, one write per row
  for (int gy = 0; gy < npix && ok; gy++)
  {
    const float *src = map + (size_t)npix * gy;
    for (int gx = 0; gx < npix; gx++)
    {
      uint32_t u;
      memcpy(&u, src + gx, 4);
      row[gx] = __builtin_bswap32(u);
    }
    ok = fwrite(row.data(), 4, row.size(), f) == row.size();
  }
  const size_t pad = (2880 - (n * 4) % 2880) % 2880;
  if (ok && pad)
  {
    std::vector<unsigned char> z(pad, 0);
    ok = fwrite(z.data(), 1, pad, f) == pad;
  }
  ok = (fclose(f) == 0) && ok;
  if (!ok)
    throw SliceError{"short write on " + file};
}

// densitymaps.cpp:530-630.  ntotxyi are the real per-type accepted counts (the reference always writes 0 because of
// densitymaps.cpp:497, and therefore writes NO per-type file at all with partinplanes: here the documented intent
// of README.md:74 is implemented — one file per type that has particles in the plane).
void writeMaps(const InputParams &p, const Header &data, const Lens &lens, int isnap, double zsim, const std::string &snappl,
               const std::valarray<float> &mapxytotrecv, const std::valarray<float> *mapxytotirecv, const long long *ntotxyi, int myid)
{
  if (myid != 0)
    return;
  std::vector<std::pair<std::string, double>> d = {{"REDSHIFT", zsim},
                                                   {"PHYSICALSIZE", p.fov},
                                                   {"PIXELUNIT", 1.e+10 / data.h},
                                                   {"DlLOW", lens.ld[isnap] / data.h},
                                                   {"DlUP", lens.ld2[isnap] / data.h},
                                                   {"HUBBLE", data.h},
                                                   {"OMEGAMATTER", data.om0},
                                                   {"OMEGALAMBDA", data.oml}};
  if (!p.partinplanes)
  {
    std::vector<std::pair<std::string, long long>> k;
    std::vector<std::string> order = {"REDSHIFT", "PHYSICALSIZE", "PIXELUNIT", "DlLOW", "DlUP"};
    for (int i = 0; i < 6; i++)
    {
      k.push_back({"nparttype" + std::to_string(i), ntotxyi[i]});
      order.push_back("nparttype" + std::to_string(i));
    }
    order.insert(order.end(), {"HUBBLE", "OMEGAMATTER", "OMEGALAMBDA"});
    for (int i = 0; i < 6; i++)
    {
      d.push_back({"m" + std::to_string(i), data.massarr[i]});
      order.push_back("m" + std::to_string(i));
    }
    const std::string fileoutput = fileOutput(p, snappl);
    std::cout << "Saving the maps on: " + fileoutput + "\n" << std::flush; // one insertion: planes are written on several threads
    writeFitsImage(fileoutput, &mapxytotrecv[0], p.npix, d, k, order);
    return;
  }
  for (int i = 0; i < 6; i++)
    if (ntotxyi[i] > 0)
    {
      std::vector<std::pair<std::string, double>> di = d;
      di.push_back({"m" + std::to_string(i), data.massarr[i]});
      std::vector<std::pair<std::string, long long>> k = {{"nparttype0", ntotxyi[i]}};
      writeFitsImage(fileOutput(p, snappl, i), &mapxytotirecv[i][0], p.npix, di, k,
                     {"REDSHIFT", "PHYSICALSIZE", "PIXELUNIT", "DlLOW", "DlUP", "nparttype0", "HUBBLE", "OMEGAMATTER", "OMEGALAMBDA",
                      "m" + std::to_string(i)});
    }
}

} // namespace slicer
