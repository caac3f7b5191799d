// host_tables.cpp — map loading and the small host-built tables.
//
// Replaces load_settlements (data/settlements_loader.rs:23-42), load_generators
// (data/generators_loader.rs:47-207), the coastline include (utils/map_handler.rs:360-375) and
// initialize_map (main.rs:74-125). Everything the device path needs from libm (pow, exp) is evaluated
// here for the 26 year offsets, 15 types, 3 multipliers and 4 offset types that can occur:
// config/const_funcs.rs:13-106,186-203,269-351; config/tech_type.rs:53-200; models/generator.rs:184-342,
// 451-626; models/carbon_offset.rs:188-232.
#include "host_tables.hpp"
#include "json_min.hpp"
#include "common.hpp"
#include <algorithm>
#include <cmath>
#include <cstring>
#include <sstream>

namespace {

enum { OnshoreWind, OffshoreWind, DomesticSolar, CommercialSolar, UtilitySolar, Nuclear, CoalPlant, GasCombinedCycle,
       GasPeaker, Biomass, HydroDam, PumpedStorage, BatteryStorage, TidalGenerator, WaveEnergy };

// f64::powi lowers to compiler-rt's __powidf2 (square-and-multiply), which is not pow()
double rust_powi(double a, int b) {
  const bool recip = b < 0;
  double r = 1;
  for (;;) {
    if (b & 1) r *= a;
    b /= 2;
    if (b == 0) break;
    a *= a;
  }
  return recip ? 1 / r : r;
}
double inflation(int yi) { return rust_powi(1.0 + 0.0185, yi); }  // const_funcs.rs:13-15

const double kBaseCost[EG_NT] = {1500000.0, 4000000.0, 10000000.0, 40000000.0, 240000000.0, 15000000000.0, 1500000000.0,
                                 560000000.0, 500000000.0, 150000000.0, 2500000000.0, 1200000000.0, 150000000.0,
                                 1000000000.0, 800000000.0};  // generator.rs:244-293
const double kRate[EG_NT] = {0.99, 0.99, 0.97, 0.97, 0.97, 0.99, 1.10, 1.04, 1.04, 0.99, 1.06, 1.06, 0.97, 0.95, 0.95};  // generator.rs:184-202
const double kPower[EG_NT] = {500.0, 800.0, 10.0, 50.0, 300.0, 1500.0, 1000.0, 800.0, 400.0, 50.0, 1200.0, 600.0, 500.0, 200.0, 100.0};
const double kCo2Rate[EG_NT] = {0, 0, 0, 0, 0, 0, 6300.0, 3500.0, 4800.0, 1500.0, 0, 0, 0, 0, 0};  // constants.rs:125-128
const double kOpinionBase[EG_NT] = {0.83, 0.83, 0.89, 0.89, 0.89, 0.43, 0.41, 0.42, 0.42, 0.60, 0.89, 0.89, 0.85, 0.75, 0.75};  // const_funcs.rs:80-90
const double kOpinionChange[EG_NT] = {0.005, 0.005, 0.008, 0.008, 0.008, 0.002, -0.015, -0.008, -0.008, 0.001, 0.004, 0.004, 0.003, 0.005, 0.005};
const double kRadius[EG_NT] = {5000.0, 5000.0, 3000.0, 3000.0, 3000.0, 12000.0, 8000.0, 8000.0, 3000.0, 3000.0, 7000.0, 7000.0, 3000.0, 6000.0, 6000.0};
const double kRadii[EG_N_RCLASS] = {3000.0, 5000.0, 6000.0, 7000.0, 8000.0, 12000.0};

bool is_water_type(int t) { return t == OffshoreWind || t == TidalGenerator || t == WaveEnergy; }  // generator.rs:142-154
bool is_intermittent(int t) { return t <= UtilitySolar; }
bool is_storage(int t) { return t == PumpedStorage || t == BatteryStorage; }

double location_modifier(int t) {  // const_funcs.rs:37-54 with the arguments of generator.rs:583-590
  double m = 1.0;
  if (t == DomesticSolar || t == CommercialSolar) m *= 1.1;  // can_be_urban -> URBAN_SOLAR_BONUS
  else if (t == GasPeaker) m *= 0.7;                          // URBAN_PEAKER_PENALTY
  if (is_water_type(t)) m *= 1.15;                            // COASTAL_BONUS
  return m;
}

double type_opinion(int t, int yi) {  // const_funcs.rs:78-93
  double v = kOpinionBase[t] + kOpinionChange[t] * (double)yi;
  return std::min(std::max(v, 0.0), 1.0);
}
double cost_opinion(double cost, int yi) {  // const_funcs.rs:95-106
  const double adjusted_max = 1384000000.0 * inflation(yi);
  const double n = cost / adjusted_max;
  return n <= 1.0 ? 1.0 - n : 0.5 * std::exp(-0.5 * (n - 1.0));
}
double carbon_price(int year) {  // const_funcs.rs:186-203
  if (year < 2030) return 75.0;
  if (year < 2040) return 75.0 + ((double)(year - 2030) / (double)(2040 - 2030)) * (130.0 - 75.0);
  if (year <= 2050) return 130.0 + ((double)(year - 2040) / (double)(2050 - 2040)) * (300.0 - 130.0);
  return 300.0;
}

// planning/construction durations for a plant registered in `year` (tech_type.rs:70-200, const_funcs.rs:269-295)
double lerp_duration(int year, double base_2025, double end_2050) {
  const int clamped = std::min(std::max(year, 2025), 2050);
  const double t = ((double)clamped - 2025.0) / (2050.0 - 2025.0);
  return std::max(base_2025 + t * (end_2050 - base_2025), end_2050);
}
void tech_durations(int t, int year, double* planning, double* construction) {
  double p0, p1, c0, c1;
  switch (t) {
    case OnshoreWind: p0 = 1.5; p1 = 0.5; c0 = 1.25; c1 = 0.75; break;
    case OffshoreWind: p0 = 3.0; p1 = 1.0; c0 = 3.0; c1 = 2.0; break;
    case DomesticSolar: case CommercialSolar: case UtilitySolar: p0 = 1.0; p1 = 0.3; c0 = 0.5; c1 = 0.25; break;
    case GasCombinedCycle: case GasPeaker: p0 = 2.0; p1 = 1.0; c0 = 2.5; c1 = 2.0; break;
    case CoalPlant: p0 = 2.0; p1 = 1.0; c0 = 3.0; c1 = 3.0; break;
    case Nuclear: p0 = 5.0; p1 = 3.0; c0 = 7.0; c1 = 4.0; break;
    case HydroDam: p0 = 2.5; p1 = 1.5; c0 = 4.0; c1 = 3.5; break;
    case PumpedStorage: case BatteryStorage: p0 = 1.5; p1 = 0.8; c0 = 1.0; c1 = 0.5; break;
    case Biomass: p0 = 2.0; p1 = 1.0; c0 = 2.0; c1 = 1.5; break;
    default: p0 = 3.0; p1 = 1.5; c0 = 2.0; c1 = 1.5; break;  // Tidal, Wave
  }
  *planning = lerp_duration(year, p0, p1);
  *construction = lerp_duration(year, c0, c1);
}

bool lat_lon_to_grid(double lat, double lon, double* x, double* y) {  // const_funcs.rs:124-136
  if (lat < 51.4 || lat > 55.4 || lon < -10.6 || lon > -5.9) return false;
  *x = std::min(std::max((lon - (-10.6)) * 10638.297872340427, 0.0), 50000.0);
  *y = std::min(std::max((lat - 51.4) * 12500.0, 0.0), 50000.0);
  return true;
}

int fuel_to_type(std::string fuel) {  // generators_loader.rs:47-57
  for (char& c : fuel) c = (char)std::tolower((unsigned char)c);
  if (fuel == "gas") return GasCombinedCycle;
  if (fuel == "coal") return CoalPlant;
  if (fuel == "wind") return OnshoreWind;
  if (fuel == "hydro") return HydroDam;
  if (fuel == "oil") return GasPeaker;
  if (fuel == "biomass") return Biomass;
  return -1;
}

double normalized_size(double capacity, int t) {  // generators_loader.rs:118-131
  double max_power;
  switch (t) {
    case OnshoreWind: max_power = 500.0; break;
    case OffshoreWind: max_power = 800.0; break;
    case CoalPlant: max_power = 1000.0; break;
    case GasCombinedCycle: max_power = 800.0; break;
    case GasPeaker: max_power = 400.0; break;
    case HydroDam: max_power = 1200.0; break;
    case Biomass: max_power = 50.0; break;
    default: max_power = 800.0; break;
  }
  return std::min(std::max(capacity / max_power, 0.1), 1.0);
}

std::string trim(const std::string& s) {
  size_t a = s.find_first_not_of(" \t\r\n"), b = s.find_last_not_of(" \t\r\n");
  return a == std::string::npos ? std::string() : s.substr(a, b - a + 1);
}

}  // namespace

void eg_host_tech_durations(int type, int year, double* planning, double* construction) { tech_durations(type, year, planning, construction); }

int eg_host_map_load(EgHostMap* m, const char* settlements_json, const char* generators_csv, const char* coastline_json) {
  *m = EgHostMap();
  std::string text;
  // settlements.json — SettlementsList { settlements: [ { name, lat, lon, population, .. } ] }
  if (!egjson::read_file(settlements_json, &text)) return eg_fail(EG_ERR_IO, std::string("cannot read ") + settlements_json);
  try {
    egjson::Value root = egjson::Parser(text).parse();
    const egjson::Value* list = root.get("settlements");
    if (!list || list->kind != egjson::Value::Array) return eg_fail(EG_ERR_IO, "settlements.json: missing 'settlements' array");
    for (const egjson::Value& s : list->arr) {
      const egjson::Value *lat = s.get("lat"), *lon = s.get("lon"), *pop = s.get("population");
      if (!lat || !lon || !pop) return eg_fail(EG_ERR_IO, "settlements.json: entry without lat/lon/population");
      // SettlementData { lat: f64, lon: f64, population: u32 } (settlements_loader.rs:8-16): serde fails on other types
      if (lat->kind != egjson::Value::Number || lon->kind != egjson::Value::Number || pop->kind != egjson::Value::Number ||
          !(pop->num >= 0.0 && pop->num <= 4294967295.0) || pop->num != std::floor(pop->num))
        return eg_fail(EG_ERR_IO, "settlements.json: lat/lon must be numbers and population a u32");
      double x, y;
      if (!lat_lon_to_grid(lat->num, lon->num, &x, &y)) continue;  // reference warns and skips (settlements_loader.rs:38-40)
      m->sx.push_back(x);
      m->sy.push_back(y);
      m->spop.push_back((uint32_t)pop->num);
      const egjson::Value* name = s.get("name");
      m->sname.push_back(name && name->kind == egjson::Value::String ? name->str : "Settlement_" + std::to_string(m->sname.size()));
    }
  } catch (const std::exception& ex) {
    return eg_fail(EG_ERR_IO, std::string(settlements_json) + ": " + ex.what());
  }
  // ireland_generators.csv — capacity_mw,latitude,longitude,primary_fuel with a header row
  if (!egjson::read_file(generators_csv, &text)) return eg_fail(EG_ERR_IO, std::string("cannot read ") + generators_csv);
  {
    std::istringstream in(text);
    std::string line;
    bool header = true;
    while (std::getline(in, line)) {
      if (trim(line).empty()) continue;
      if (header) { header = false; continue; }
      std::vector<std::string> f;
      std::stringstream ls(line);
      std::string cell;
      while (std::getline(ls, cell, ',')) f.push_back(trim(cell));
      if (f.size() < 4) return eg_fail(EG_ERR_IO, std::string(generators_csv) + ": row with fewer than 4 fields");
      char* end = nullptr;
      const double cap = std::strtod(f[0].c_str(), &end);
      if (end == f[0].c_str()) return eg_fail(EG_ERR_IO, "Invalid capacity: Invalid capacity format");
      double lat = std::strtod(f[1].c_str(), &end);
      if (end == f[1].c_str()) return eg_fail(EG_ERR_IO, "Invalid coordinate: Invalid latitude format");
      double lon = std::strtod(f[2].c_str(), &end);
      if (end == f[2].c_str()) return eg_fail(EG_ERR_IO, "Invalid coordinate: Invalid longitude format");
      const int t = fuel_to_type(f[3]);
      if (t < 0) return eg_fail(EG_ERR_IO, "Invalid fuel type: " + f[3]);
      // transform_coordinates (generators_loader.rs:59-116): out-of-range inputs are clamped, not rejected
      lat = std::min(std::max(lat, 51.4), 55.4);
      lon = std::min(std::max(lon, -10.6), -5.9);
      double x, y;
      if (!lat_lon_to_grid(lat, lon, &x, &y)) return eg_fail(EG_ERR_IO, "Invalid coordinate: Failed to transform coordinates");
      m->ex.push_back(x);
      m->ey.push_back(y);
      m->etype.push_back((uint8_t)t);
      m->ecap.push_back(cap);
    }
  }
  // coastline_points.json — { "grid_coords": [[x, y], ..] }
  if (!egjson::read_file(coastline_json, &text)) return eg_fail(EG_ERR_IO, std::string("cannot read ") + coastline_json);
  try {
    egjson::Value root = egjson::Parser(text).parse();
    const egjson::Value* pts = root.get("grid_coords");
    if (!pts || pts->kind != egjson::Value::Array) return eg_fail(EG_ERR_IO, "coastline_points.json: Invalid coastline format");
    for (const egjson::Value& pnt : pts->arr) {
      if (pnt.kind != egjson::Value::Array || pnt.arr.size() < 2) return eg_fail(EG_ERR_IO, "coastline_points.json: Invalid point format");
      m->cx.push_back(std::min(std::max(pnt.arr[0].num, 0.0), 50000.0));
      m->cy.push_back(std::min(std::max(pnt.arr[1].num, 0.0), 50000.0));
    }
  } catch (const std::exception& ex) {
    return eg_fail(EG_ERR_IO, std::string(coastline_json) + ": " + ex.what());
  }
  m->grid_n = 51;      // distinct points of the 100x100 scan after Coordinate::new clamps at 50 km
  m->step = 1000.0;    // grid_step, metal_location_search.rs:113
  return EG_OK;
}

int eg_host_map_set(EgHostMap* m, const eg_map_desc* d) {
  *m = EgHostMap();
  if (!d) return eg_fail(EG_ERR_INVALID, "eg_map_set: desc is NULL");
  auto clampc = [](double v) { return std::min(std::max(v, 0.0), 50000.0); };
  for (uint32_t i = 0; i < d->n_settlements; i++) {
    m->sx.push_back(clampc(d->settlement_x[i]));
    m->sy.push_back(clampc(d->settlement_y[i]));
    m->spop.push_back(d->settlement_pop[i]);
  }
  for (uint32_t i = 0; i < d->n_existing; i++) {
    if (d->existing_type[i] >= EG_NT) return eg_fail(EG_ERR_INVALID, "eg_map_set: generator type out of range");
    m->ex.push_back(clampc(d->existing_x[i]));
    m->ey.push_back(clampc(d->existing_y[i]));
    m->etype.push_back(d->existing_type[i]);
    m->ecap.push_back(d->existing_capacity_mw[i]);
  }
  for (uint32_t i = 0; i < d->n_coast; i++) {
    m->cx.push_back(clampc(d->coast_x[i]));
    m->cy.push_back(clampc(d->coast_y[i]));
  }
  m->grid_n = (int)d->grid_n;
  m->step = d->grid_step;
  return EG_OK;
}

int eg_host_map_validate(const EgHostMap& m) {
  if (m.grid_n < 2 || m.grid_n > 255) return eg_fail(EG_ERR_INVALID, "map: grid_n must be in [2, 255]");
  if (!(m.step >= 1.0) || m.step != std::floor(m.step)) return eg_fail(EG_ERR_INVALID, "map: grid_step must be a positive integer number of metres");
  if ((double)(m.grid_n - 1) * m.step > 50000.0) return eg_fail(EG_ERR_INVALID, "map: candidate grid exceeds the 50 km map (Coordinate::new would clamp it)");
  if ((size_t)m.grid_n * m.grid_n > 65535) return eg_fail(EG_ERR_INVALID, "map: more than 65535 candidate sites");
  return EG_OK;
}

void eg_host_build_tables(const EgHostMap& m, EgHostTables* out) {
  EgSmallTables& T = out->small;
  std::memset(&T, 0, sizeof(T));
  const size_t S = m.sx.size(), E = m.ex.size();

  // ---- per-type constants of a plant built by the simulation (actions.rs:43-72; quirk Q3: size does not scale output)
  static const uint8_t pclass_of_type[EG_NT] = {1, 2, 0, 0, 0, 6, 5, 5, 0, 0, 4, 4, 0, 3, 3};
  static const uint8_t rclass_of_pclass[EG_N_PCLASS] = {0, 1, 1, 2, 3, 4, 5};
  static const uint8_t water_of_pclass[EG_N_PCLASS] = {0, 0, 1, 1, 0, 0, 0};
  for (int t = 0; t < EG_NT; t++) {
    const double base_output = kPower[t] * 0.99 * 1.0;  // power_out * efficiency * operation_percentage
    T.net_mw[t] = is_intermittent(t) ? base_output * (t <= OffshoreWind ? 0.35 : 0.20) : base_output;  // generator.rs:538-552
    const double co2_out = kCo2Rate[t] * (100.0 / 100.0);
    T.co2[t] = co2_out * 1.0 * (1.0 - (0.99 - 0.99));    // generator.rs:625
    T.loc_mod[t] = location_modifier(t);
    T.acc_class[t] = is_intermittent(t) ? EG_ACC_INTERMITTENT : (is_storage(t) ? EG_ACC_STORAGE : EG_ACC_PLAIN);
    T.pclass[t] = pclass_of_type[t];
    for (int y = 0; y < EG_NY; y++) {
      T.base_cost[t][y] = kBaseCost[t] * std::pow(kRate[t], (double)y);  // generator.rs:295-297
      T.tech[t][y] = std::pow(kRate[t], (double)y);                       // const_funcs.rs:33-34
      T.op_type[y][t] = 0.12 * type_opinion(t, y);
    }
  }
  for (int pc = 0; pc < EG_N_PCLASS; pc++) { T.rclass_of_pclass[pc] = rclass_of_pclass[pc]; T.water_of_pclass[pc] = water_of_pclass[pc]; }
  T.mult[0] = std::min(std::max(100.0 / 100.0, 1.0), 5.0);
  T.mult[1] = std::min(std::max(120.0 / 100.0, 1.0), 5.0);
  T.mult[2] = std::min(std::max(150.0 / 100.0, 1.0), 5.0);
  T.size_factor = 1.0 - ((double)(float)(100.0 / 100.0) * 0.1);  // metal_location_search.rs:166 with size 1.0 as f32
  // offsets in canonical order Forest, Wetland, ActiveCapture, CarbonCredit (actions.rs:134-172, carbon_offset.rs:212-217)
  const double off_size[4] = {500.0, 300.0, 100.0, 1000.0}, off_rate[4] = {25.0, 40.0, 500.0, 100.0};
  const double off_cost[4] = {1000000.0, 1000000.0, 1000000000.0, 50000000.0};
  for (int o = 0; o < 4; o++) {
    T.off_amount[o] = (off_size[o] * off_rate[o]) * 0.85;
    T.off_base_cost[o] = off_cost[o];
    T.natural_offset[o] = (o == 0 || o == 1) ? 1 : 0;
  }
  for (int d = 0; d < EG_NY; d++) T.maturity[d] = std::min(std::max(1.0 - std::exp(-0.1 * (double)d), 0.0), 1.0);  // carbon_offset.rs:226-227

  // ---- CONSTRUCTION_COST_WEIGHT * cost opinion of a simulation-built plant
  // (the cost re-priced at the year before the build year is read too: yearly capital cost, map_handler.rs:968-985)
  out->plant_terms.assign((size_t)EG_OPC_SIZE * 2, 0.0);
  for (int y = 0; y < EG_NY; y++)
    for (int t = 0; t < EG_NT; t++)
      for (int mi = 0; mi < EG_N_MULTS; mi++)
        for (int b = 0; b < EG_NY; b++) {
          const double cost = T.base_cost[t][b] * inflation(y) * T.tech[t][y] * T.loc_mod[t] * T.mult[mi];
          out->plant_terms[(size_t)EG_OPC_INDEX(y, t, mi, b) * 2] = 0.82 * cost_opinion(cost, y);
          out->plant_terms[(size_t)EG_OPC_INDEX(y, t, mi, b) * 2 + 1] = cost;
        }

  // ---- settlements: population growth and demand (simulation.rs:107-120, map_handler.rs:813-827)
  out->pop.assign((size_t)EG_NY * S, 0);
  for (size_t s = 0; s < S; s++) out->pop[s] = m.spop[s];
  for (int y = 1; y < EG_NY; y++)
    for (size_t s = 0; s < S; s++) out->pop[(size_t)y * S + s] = (uint32_t)std::round((double)out->pop[(size_t)(y - 1) * S + s] * 1.01);

  // ---- plants that exist before the simulation: registered in 2024 with construction delays on (quirk Q1)
  std::vector<double> settle_op(E, 1.0), planning(E), construction(E), size(E);
  for (size_t g = 0; g < E; g++) {
    double sum = 0.0;
    for (size_t s = 0; s < S; s++) {
      const double dx = m.sx[s] - m.ex[g], dy = m.sy[s] - m.ey[g];
      sum += 1.0 / (1.0 + std::sqrt(dx * dx + dy * dy) / 10000.0);
    }
    settle_op[g] = S ? sum / (double)S : 1.0;
    double p, c;
    tech_durations(m.etype[g], 2024, &p, &c);
    const double opinion_factor = 1.0 - (0.65 * 0.5);            // calculate_public_opinion_at_location == 0.65
    planning[g] = std::max(p * opinion_factor * 1.0, 0.25);        // const_funcs.rs:276-282
    construction[g] = std::max(c * 1.0, 0.1);                      // const_funcs.rs:291-294
    size[g] = normalized_size(m.ecap[g], m.etype[g]);
  }
  std::vector<int> status(E, 0), start(E, 0);  // 0 Planned, 1 Granted, 2 UnderConstruction, 3 Operational
  out->ex_online_year.assign(E, 0);
  for (int y = 0; y < EG_NY; y++) {
    const int year = EG_BASE_YEAR + y;
    EgYearRow& row = T.year[y];
    for (size_t g = 0; g < E; g++) {  // Generator::update_construction_status, generator.rs:482-517
      if (status[g] == 0) { if ((double)(year - 2024) >= planning[g]) status[g] = 1; }
      else if (status[g] == 1) { status[g] = 2; start[g] = year; }
      else if (status[g] == 2) { if ((double)(year - start[g]) >= construction[g]) status[g] = 3; }
      if (status[g] == 3 && !out->ex_online_year[g]) out->ex_online_year[g] = year;
    }
    double usage = 0.0;
    uint32_t pop_total = 0;
    const double per_capita = 0.001 * std::pow(1.0 + 0.02, (double)y);  // const_funcs.rs:17-26
    for (size_t s = 0; s < S; s++) {
      const uint32_t p = out->pop[(size_t)y * S + s];
      pop_total += p;
      usage += (double)p * per_capita;
    }
    row.usage_total = usage * (1.0 + ((double)year - 2024.0) * 0.02);
    row.pop_total = pop_total;
    row.inflation = inflation(y);
    row.carbon_price = carbon_price(year);
    row.ex_gen[0] = row.ex_gen[1] = row.ex_gen[2] = 0.0;
    row.ex_co2 = 0.0;
    row.ex_opinion_sum = 0.0;
    row.ex_active = 0;
    for (size_t g = 0; g < E; g++) {
      const int t = m.etype[g];
      const bool active = status[g] == 3;
      double output = 0.0;
      if (active) {
        const double base_output = m.ecap[g] * 0.99 * 1.0;
        output = is_intermittent(t) ? base_output * (t <= OffshoreWind ? 0.35 : 0.20) : base_output;
      }
      row.ex_gen[is_intermittent(t) ? EG_ACC_INTERMITTENT : (is_storage(t) ? EG_ACC_STORAGE : EG_ACC_PLAIN)] += output;
      if (!active) continue;
      const double co2_out = kCo2Rate[t] * size[g];                 // calc_initial_co2_output, const_funcs.rs:113-122
      row.ex_co2 += co2_out * 1.0 * (1.0 - (0.99 - 0.99));
      // base_cost stored by load_generators is get_base_cost(2025) with no modifier (generators_loader.rs:175-182)
      const double stored_base = ((kBaseCost[t] * std::pow(kRate[t], 0.0)) * inflation(0) * std::pow(kRate[t], 0.0)) * 1.0;
      const double cost = (stored_base * inflation(y) * std::pow(kRate[t], (double)y) * location_modifier(t)) * 1.0;
      row.ex_opinion_sum += 0.03 * settle_op[g] + 0.12 * type_opinion(t, y) + 0.82 * cost_opinion(cost, y);
      row.ex_active++;
    }
    row.prefix_changed = 1;
    if (y > 0) {
      const EgYearRow& prev = T.year[y - 1];
      row.prefix_changed = std::memcmp(prev.ex_gen, row.ex_gen, sizeof(row.ex_gen)) != 0 || std::memcmp(&prev.ex_co2, &row.ex_co2, sizeof(double)) != 0;
    }
  }

  // ---- distance/radius factors between candidate sites. Sites lie on an integer grid, so dx*dx + dy*dy of the
  // reference's distance_to is exactly step^2 * d2 with d2 = di^2 + dj^2, and the factor is a function of d2 alone.
  const int kmax = (int)std::floor(12000.0 / m.step) + 1;
  out->kmax = kmax;
  int stride = 1;
  for (int rc = 0; rc < EG_N_RCLASS; rc++) {
    int d2 = 0;
    while (std::sqrt((double)d2 * m.step * m.step) < kRadii[rc]) d2++;
    out->r2_limit[rc] = d2;
    stride = std::max(stride, d2 + 1);  // entry r2_limit[rc] of every class stays 1.0: what a plant out of range multiplies by
  }
  out->r2_stride = stride;
  for (int rc = 0, off = 0; rc <= EG_N_RCLASS; rc++) {
    out->r2_limit[EG_N_RCLASS + rc] = off;
    if (rc < EG_N_RCLASS) off += out->r2_limit[rc] + 1;  // the kernel's copy ends every class with a factor of 1.0 (out of range)
  }
  out->near_factor.assign((size_t)EG_N_RCLASS * stride, 1.0);
  for (int rc = 0; rc < EG_N_RCLASS; rc++)
    for (int d2 = 0; d2 < out->r2_limit[rc]; d2++) {
      const double distance = std::sqrt((double)d2 * m.step * m.step);
      out->near_factor[(size_t)rc * stride + d2] = distance / kRadii[rc];
    }
  // the kernel's one-instruction cell distance needs coordinates below 64, its two-instruction form |g|^2 < 65536 (181 sites per
  // axis); both read the factors from a block-shared copy of the table (entries inside the radii: a few KB on maps with cells of
  // 750 m or more, 27 KB on the 10x grid)
  for (int ty = 0; ty < EG_NT; ty++) {
    T.type_sums[ty][0] = T.type_sums[ty][1] = T.type_sums[ty][2] = 0.0;
    T.type_sums[ty][T.acc_class[ty] == EG_ACC_PLAIN ? 0 : (T.acc_class[ty] == EG_ACC_INTERMITTENT ? 1 : 2)] = T.net_mw[ty];
    T.type_sums[ty][3] = T.co2[ty];
    const int pc = T.pclass[ty], rc = T.rclass_of_pclass[pc];
    const int table_off = out->r2_limit[EG_N_RCLASS + rc];
    T.place_info[ty][0] = (uint32_t)pc | ((uint32_t)rc << 4) | ((uint32_t)(T.water_of_pclass[pc] != 0) << 8) | ((uint32_t)(table_off & 0xFFFF) << 16);
    T.place_info[ty][1] = (uint32_t)out->r2_limit[rc];
  }
  {
    const int entries = out->r2_limit[2 * EG_N_RCLASS];
    out->near_geom = (m.grid_n <= 64 && entries <= EG_COMPACT_MAX_FACTORS) ? 0 : ((m.grid_n <= 181 && entries <= EG_MEDIUM_MAX_FACTORS) ? 1 : 2);
  }
  (void)kRadius;
}
