// rpsf_bands.cuh — the row bands of a plan: where the row pass (K1) leaves the row spectra that the column pass (K2) and
// the kernel gradient (kgrad) read.
//
// The row FFT of a patch row is FFT_x(w_x ⊙ frame_row[cx : cx + P]); only the row window w_y tells two patches with the
// same corner column apart, and it is applied after the transform.  So K1 transforms each frame row once per band (a
// corner column, see below), stores it without w_y, and K2 / kgrad multiply by w_y as they load a patch's rows.  For
// calculate_covering, where two patches sit on every row of a patch column, that is 0.53 of the row FFTs per frame.
//
// K1 transforms rows in pairs (row_a + i row_b), and the split into two half-spectra rounds differently for another
// partner row, so a band only holds patches whose corner rows share one parity: every patch keeps the row pairs it had
// with a spectrum of its own.  The last row of a window of odd length was paired with a zero row; such patches get a
// band each, whose row past the window is a zero row again.
//
// Band buffer: [frame][band-buffer row][P/2] complex, packed Hermitian rows (bin 0 holds (DC.re, Nyquist.re)).  A band
// occupies the rows [base, base + rows); its row base + i is frame row row0 + i.
#pragma once
#include <algorithm>
#include <map>
#include <tuple>
#include <vector>
#include "rpsf_fft.cuh"

namespace rpsf {

// Rows per K1 work item: the row pairs of one warp of the streaming K1 (rpsf_stream.cuh asserts it)
template <int P> __host__ __device__ constexpr int band_quantum() { return 2 * (32 / Split<P>::N1); }

// K1 work item: band_quantum consecutive rows of one band
struct BandItem {
  int row;          // plan-frame row of the first row (the coordinates of the patch corners)
  int cx;           // corner column of the band
  int buf_row;      // band-buffer row of the first row, within a frame
  unsigned live;    // bit r: row `row + r` lies in the window of a patch of the band; the other rows are zero rows
};

// What the kernels get of a plan's bands (device pointers)
struct RowBands {
  const BandItem* items;   // one frame's items, in (row, corner column) order: K1 walks the frame top to bottom
  const int* patch_row;    // per active patch: band-buffer row of its patch row 0, band.base + cy - band.row0
  int n_items;             // per frame
  int frame_rows;          // band-buffer rows per frame
};

// Host side: the bands of a plan's active patches (corners in plan coordinates, the plan's order)
struct BandLayout {
  std::vector<BandItem> items;
  std::vector<int> patch_row;
  int frame_rows = 0;
  int n_bands = 0;
};

inline BandLayout build_row_bands(const std::vector<int2>& corners, int win_len, int quantum) {
  BandLayout out;
  out.patch_row.assign(corners.size(), 0);
  // key: corner column, corner-row parity, and for odd windows the corner row itself (a band per patch)
  std::map<std::tuple<int, int, int>, std::vector<int>> bands;
  for (size_t a = 0; a < corners.size(); ++a) {
    const int2 c = corners[a];
    bands[std::make_tuple(c.y, ((c.x % 2) + 2) % 2, (win_len % 2) ? c.x : 0)].push_back((int)a);
  }
  out.n_bands = (int)bands.size();
  std::vector<std::pair<int, BandItem>> order;       // (band, item), sorted below
  int base = 0, band = 0;
  for (const auto& kv : bands) {
    int row0 = corners[kv.second[0]].x, end = row0;
    for (int a : kv.second) { row0 = std::min(row0, corners[a].x); end = std::max(end, corners[a].x + win_len); }
    const int rows = (end - row0 + quantum - 1) / quantum * quantum;
    std::vector<char> live(rows, 0);
    for (int a : kv.second) {
      std::fill(live.begin() + (corners[a].x - row0), live.begin() + (corners[a].x - row0 + win_len), 1);
      out.patch_row[a] = base + corners[a].x - row0;
    }
    for (int q = 0; q < rows; q += quantum) {
      unsigned mask = 0;
      for (int r = 0; r < quantum; ++r) mask |= live[q + r] ? 1u << r : 0u;
      if (mask) order.push_back({band, BandItem{row0 + q, std::get<0>(kv.first), base + q, mask}});
    }
    base += rows;
    ++band;
  }
  std::stable_sort(order.begin(), order.end(), [](const std::pair<int, BandItem>& u, const std::pair<int, BandItem>& v) {
    return u.second.row != v.second.row ? u.second.row < v.second.row : u.first < v.first;
  });
  for (const auto& e : order) out.items.push_back(e.second);
  out.frame_rows = base;
  return out;
}

}  // namespace rpsf
