// extern "C" wrapper so the Python tests can feed REAL operator patterns (from the oracle) to the cost model.
#include "mxg_ilv_model.h"

extern "C" int ilv_model_eval(const int32_t* rowPat, const int32_t* patOff, const int32_t* delta, int64_t rowBegin, int64_t rowEnd,
                              int xBytes, int patEntryBytes, double out[5]) {
  mxg::IlvCost c = mxg::ilvCostModel(rowPat, patOff, [delta](int32_t q) { return delta[q]; }, rowBegin, rowEnd, xBytes, patEntryBytes);
  out[0] = c.pat[0]; out[1] = c.pat[1]; out[2] = c.col[0]; out[3] = c.col[1]; out[4] = c.tiles;
  return 0;
}
extern "C" int ilv_model_wins(const double cost[5]) {
  mxg::IlvCost c;
  c.pat[0] = cost[0]; c.pat[1] = cost[1]; c.col[0] = cost[2]; c.col[1] = cost[3]; c.tiles = int(cost[4]);
  return mxg::ilvWins(c) ? 1 : 0;
}
