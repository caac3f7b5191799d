// report_files.cpp — output files from host data: the best run's CSV files and the location analysis cache and report.
#include <sys/stat.h>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include "common.hpp"
#include "eg_math.hpp"
#include "host_tables.hpp"
#include "json_min.hpp"
#include "weights.hpp"

namespace {

// Rust's `{}` for f64: shortest digits that round-trip, never scientific notation
std::string rust_display(double v) {
  char buf[400];
  for (int prec = 1; prec <= 17; prec++) {
    std::snprintf(buf, sizeof(buf), "%.*g", prec, v);
    if (std::strtod(buf, nullptr) == v) break;
  }
  if (!std::strpbrk(buf, "eE")) return buf;
  // re-print without exponent: enough fixed digits to round-trip
  for (int prec = 0; prec <= 340; prec++) {
    std::snprintf(buf, sizeof(buf), "%.*f", prec, v);
    if (std::strtod(buf, nullptr) == v) break;
  }
  return buf;
}

std::string fixed(double v, int prec) {
  char buf[400];
  std::snprintf(buf, sizeof(buf), "%.*f", prec, v);
  return buf;
}

// uniform in [0,1) for the exported offset coordinates: Philox4x32-10, counter (index, axis, 0, "CSVO")
double csv_uniform(uint32_t index, uint32_t axis) {
  uint32_t x[4] = {index, axis, 0u, 0x4353564Fu};
  egm::philox4x32_10(x, 0x45495247u, 0x52494442u);
  return egm::uniform53(x[0], x[1]);
}

bool mkdir_p(const std::string& p) {
  std::string cur;
  for (size_t i = 0; i <= p.size(); i++) {
    if ((i == p.size() || p[i] == '/') && !cur.empty()) {
      struct stat st;
      if (stat(cur.c_str(), &st) != 0 && mkdir(cur.c_str(), 0777) != 0 && stat(cur.c_str(), &st) != 0) return false;
    }
    if (i < p.size()) cur += p[i];
  }
  return true;
}

// f64::powi lowers to repeated squaring (compiler-rt __powidf2); reproduced for the non-negative exponents used here
double powi(double a, int b) { double r = 1.0; for (;;) { if (b & 1) r *= a; b /= 2; if (b == 0) break; a *= a; } return r; }

}  // namespace

int eg_write_best_run_csv(const char* output_dir, const eg_weights* w, const EgHostMap& hmap, const EgHostTables& htab, const eg_traj& traj,
                          const int* row, const eg_result& res, const eg_yearly& yearly, const eg_sites& sites, char* written_dir) {
  char ts[32];
  const std::time_t t = std::time(nullptr);
  std::tm tmv;
  localtime_r(&t, &tmv);
  std::strftime(ts, sizeof(ts), "%Y%m%d_%H%M%S", &tmv);  // CsvExporter::new, csv_export.rs:114-128
  const std::string dir = std::string(output_dir) + "/" + ts;
  if (!mkdir_p(dir + "/yearly_details")) return eg_fail(EG_ERR_IO, "cannot create " + dir);
  const EgSmallTables& T = htab.small;

  {  // simulation_summary.csv, csv_export.rs:215-432
    std::FILE* f = std::fopen((dir + "/simulation_summary.csv").c_str(), "w");
    if (!f) return eg_fail(EG_ERR_IO, "cannot write simulation_summary.csv in " + dir);
    std::fprintf(f, "Simulation Summary\nTimestamp,%s\n\n", ts);
    std::fprintf(f, "Final Metrics\nFinal Net Emissions (tonnes CO2),%s\n", rust_display(res.net_emissions).c_str());
    std::fprintf(f, "Average Public Opinion (%%),%s\n", fixed(res.public_opinion * 100.0, 2).c_str());
    std::fprintf(f, "Total Cost (\xE2\x82\xAC),%s\n", fixed(res.total_cost, 2).c_str());
    std::fprintf(f, "Power Reliability (%%),%s\n\n", fixed(res.power_reliability * 100.0, 2).c_str());
    std::fprintf(f, "Actions Taken\nYear,Action Type,Generator Type,Generator ID,Operation %%,Offset Type,Estimated Cost (\xE2\x82\xAC)\n");
    for (int y = 0; y < EG_NY; y++) {
      // SimulationResult.actions holds the additional actions only (simulation.rs:193, iteration.rs:90)
      for (int i = traj.n_deficit[y]; i < traj.n_deficit[y] + traj.n_additional[y]; i++) {
        const int a = traj.actions[row[y] + i];
        const int year = EG_BASE_YEAR + y;
        if (a < 45) {
          const int tp = a / 3, m = a % 3;
          // calc_generator_cost(type, base_cost(year), year, can_be_urban, requires_water, requires_water) * multiplier / 100
          const double cost = htab.plant_terms[(size_t)EG_OPC_INDEX(y, tp, 0, y) * 2 + 1] * T.mult[m];
          std::fprintf(f, "%d,AddGenerator,%s,,,,%s\n", year, kGenNames[tp], fixed(cost, 2).c_str());
        } else if (a < 57) {
          const int o = (a - 45) / 3, m = (a - 45) % 3;
          const double cost = (T.off_base_cost[o] * T.year[y].inflation) * T.mult[m];
          std::fprintf(f, "%d,AddCarbonOffset,,,,%s,%s\n", year, kOffsetNames[o], fixed(cost, 2).c_str());
        } else if (a == EG_ACT_UPGRADE) std::fprintf(f, "%d,UpgradeEfficiency,,,,,0.00\n", year);   // empty id: no generator found
        else if (a == EG_ACT_ADJUST) std::fprintf(f, "%d,AdjustOperation,,,0,,0.00\n", year);
        else if (a == EG_ACT_CLOSE) std::fprintf(f, "%d,CloseGenerator,,,,,0.00\n", year);
        else std::fprintf(f, "%d,DoNothing,,,,,0.00\n", year);
      }
    }
    std::fprintf(f, "\nYearly Summary Metrics\n");
    std::fprintf(f, "Year,Population,PowerUsage,PowerGeneration,PowerBalance,PublicOpinion,YearlyCapitalCost,TotalCapitalCost,Inflation,CO2Emissions,"
                    "CarbonOffset,NetEmissions,YearlyRevenue,TotalRevenue,ActiveGenerators,YearlyUpgradeCosts,YearlyClosureCosts,YearlyTotalCost,TotalCost\n");
    for (int y = 0; y < EG_NY; y++) {
      const eg_year_metrics& m = yearly.y[y];
      std::fprintf(f, "%d,%u,%.2f,%.2f,%.2f,%.4f,%.2f,%.2f,%.4f,%.2f,%.2f,%.2f,%.2f,%.2f,%u,%.2f,%.2f,%.2f,%.2f\n", EG_BASE_YEAR + y, m.total_population,
                   m.total_power_usage, m.total_power_generation, m.power_balance, m.average_public_opinion, m.yearly_capital_cost,
                   m.total_capital_cost, m.inflation_factor, m.total_co2_emissions, m.total_carbon_offset, m.net_co2_emissions,
                   m.yearly_carbon_credit_revenue, m.total_carbon_credit_revenue, m.active_generators, 0.0, 0.0, m.yearly_total_cost, m.total_cost);
    }
    std::fclose(f);
  }
  if (!w->history.empty()) {  // improvement_history.csv, csv_export.rs:155-212
    std::FILE* f = std::fopen((dir + "/improvement_history.csv").c_str(), "w");
    if (!f) return eg_fail(EG_ERR_IO, "cannot write improvement_history.csv in " + dir);
    std::fprintf(f, "Iteration,Score,Net Emissions (tonnes),Total Cost (\xE2\x82\xAC),Public Opinion (%%),Power Reliability (%%),Score Improvement (%%),Timestamp\n");
    double prev = 0.0;
    for (size_t i = 0; i < w->history.size(); i++) {
      const EgImprovement& h = w->history[i];
      const double imp = (i > 0 && prev > 0.0) ? ((h.score - prev) / prev) * 100.0 : 0.0;
      std::fprintf(f, "%u,%.6f,%.2f,%.2f,%.2f,%.2f,%.2f,%s\n", h.iteration, h.score, h.net_emissions, h.total_cost, h.public_opinion * 100.0,
                   h.power_reliability * 100.0, imp, h.timestamp.c_str());
      prev = h.score;
    }
    std::fclose(f);
  }
  {  // yearly_details/settlements.csv, csv_export.rs:456-530 (population and usage re-derived from the 2025 values, as there)
    std::FILE* f = std::fopen((dir + "/yearly_details/settlements.csv").c_str(), "w");
    if (!f) return eg_fail(EG_ERR_IO, "cannot write settlements.csv in " + dir);
    std::fprintf(f, "Year,Name,Longitude,Latitude,Population,PowerUsage\n");
    const EgHostMap& m = hmap;
    for (int y = 0; y < EG_NY; y++) {
      for (size_t s = 0; s < m.sx.size(); s++) {
        const double xv = std::min(std::max(m.sx[s], 0.0), 50000.0), yv = std::min(std::max(m.sy[s], 0.0), 50000.0);
        const double lon = -10.6 + ((-5.9 - -10.6) * (xv / 50000.0)), lat = 51.4 + ((55.4 - 51.4) * (yv / 50000.0));  // transform_grid_to_lat_lon, csv_export.rs:42-83
        const uint32_t pop = (uint32_t)std::round((double)m.spop[s] * powi(1.01, y));
        const double usage = ((double)m.spop[s] * 0.001) * powi(1.02, y);  // settlement power usage of the loader: population x 1 kW in MW
        std::fprintf(f, "%d,%s,%.6f,%.6f,%u,%s\n", EG_BASE_YEAR + y, s < m.sname.size() ? m.sname[s].c_str() : ("Settlement_" + std::to_string(s)).c_str(),
                     lon, lat, pop, rust_display(usage).c_str());
      }
    }
    std::fclose(f);
  }
  {  // yearly_details/generators.csv, csv_export.rs:532-984
    // `Generator.eol` holds a lifespan in years, so the exporter's first pass (`year > eol`, :701) skips every plant of the
    // map and all rows come from its second pass (:813-979): one row per generator listed as active in that year's
    // metrics, with type, commissioning year and end of life parsed back out of the id and the remaining columns filled
    // from per-type defaults; plants added during the run get the id-hash coordinates of :867-869, pre-existing plants
    // their real ones. Row order inside a year is HashMap order there; here: pre-existing plants, then build order.
    std::FILE* f = std::fopen((dir + "/yearly_details/generators.csv").c_str(), "w");
    if (!f) return eg_fail(EG_ERR_IO, "cannot write generators.csv in " + dir);
    std::fprintf(f, "Year,Generator ID,Type,Longitude,Latitude,Power Output (MW),Efficiency (%%),Operation (%%),CO2 Output (tonnes),Is Active,"
                    "Commissioning Year,End of Life Year,Size,Capital Cost (\xE2\x82\xAC),Operating Cost (\xE2\x82\xAC),Total Annual Cost (\xE2\x82\xAC),"
                    "Reliability Factor,Planning Time (years),Construction Time (years),Construction Speed\n");
    static const double kDefPower[EG_NT] = {50.0, 200.0, 0.01, 0.5, 50.0, 1000.0, 500.0, 400.0, 100.0, 50.0, 250.0, 200.0, 50.0, 30.0, 20.0};
    static const double kDefCo2PerKwh[EG_NT] = {0, 0, 0, 0, 0, 0, 3.0, 0.4, 0.5, 0.1, 0, 0, 0, 0, 0};
    static const double kDefCostPerMw[EG_NT] = {1500000.0, 3500000.0, 1000000.0, 800000.0, 600000.0, 6000000.0, 2000000.0, 1000000.0,
                                                500000.0, 3000000.0, 2500000.0, 2000000.0, 400000.0, 5000000.0, 4000000.0};
    static const double kDefReliability[EG_NT] = {0.35, 0.35, 0.25, 0.25, 0.25, 0.95, 0.90, 0.85, 0.90, 0.80, 0.75, 0.95, 0.98, 0.45, 0.40};
    struct Plant { std::string id; int type, first_year, commissioning; double x, y; };
    std::vector<Plant> plants;
    const EgHostMap& m = hmap;
    for (size_t g = 0; g < m.ex.size(); g++)  // "Existing_{type}_{n}" (generators_loader.rs:190): the third id field is the row number
      plants.push_back({std::string("Existing_") + kGenNames[m.etype[g]] + "_" + std::to_string(g), m.etype[g],
                        g < htab.ex_online_year.size() && htab.ex_online_year[g] ? htab.ex_online_year[g] : 1 << 30, (int)g, m.ex[g], m.ey[g]});
    for (int y = 0; y < EG_NY; y++)
      for (int i = 0; i < traj.n_deficit[y] + traj.n_additional[y]; i++) {
        const int a = traj.actions[row[y] + i];
        if (a >= 45 || sites.site[row[y] + i] == EG_SITE_NONE) continue;
        const int year = EG_BASE_YEAR + y;
        Plant p{std::string("Gen_") + kGenNames[a / 3] + "_" + std::to_string(year) + "_" + std::to_string(plants.size()), a / 3, year, year, 0, 0};
        uint32_t h = 0;
        for (unsigned char ch : p.id) h += ch;
        p.x = 5000.0 + (double)(h % 100) / 100.0 * (50000.0 - 10000.0);
        p.y = 5000.0 + (double)((h / 100) % 100) / 100.0 * (50000.0 - 10000.0);
        plants.push_back(p);
      }
    for (int y = 0; y < EG_NY; y++) {
      const int year = EG_BASE_YEAR + y;
      for (const Plant& p : plants) {
        if (p.first_year > year) continue;
        const int t = p.type;
        const double xv = std::min(std::max(p.x, 0.0), 50000.0), yv = std::min(std::max(p.y, 0.0), 50000.0);
        const double lon = -10.6 + ((-5.9 - -10.6) * (xv / 50000.0)), lat = 51.4 + ((55.4 - 51.4) * (yv / 50000.0));
        const double power = kDefPower[t];
        const double co2 = kDefCo2PerKwh[t] == 0 ? 0.0 : power * kDefCo2PerKwh[t] * 8760.0 / 1000.0;
        const double size = t == 0 ? power / 3.0 : t == 1 ? power / 8.0 : t == 2 ? power * 8.0 : t == 3 ? power * 6.0 : t == 4 ? power * 2.0 : power / 50.0;
        const double capital = power * kDefCostPerMw[t], operating = capital * 0.03;
        double planning, construction;
        eg_host_tech_durations(t, p.commissioning, &planning, &construction);
        // efficiency 0.99 and operation 100 (get_operation_percentage, a 0..100 value that the exporter scales by 100 again)
        std::fprintf(f, "%d,%s,%s,%.6f,%.6f,%.2f,%.2f,%.2f,%.2f,true,%d,%d,%.2f,%.2f,%.2f,%.2f,%.2f,%.2f,%.2f,Normal\n", year, p.id.c_str(), kGenNames[t],
                     lon, lat, power, 0.99 * 100.0, 100.0 * 100.0, co2, p.commissioning, p.commissioning + 25, size * 100.0, capital, operating,
                     capital + operating, kDefReliability[t], planning, construction);
      }
    }
    std::fclose(f);
  }
  {  // yearly_details/carbon_offsets.csv, csv_export.rs:987-1093
    // The exporter rebuilds the offsets on a copy of the base map, whose construction delays are on and whose clock stands
    // at 2024 (multi_simulation.rs:862-888, map_handler.rs:785-811): every offset is still `Planned` when the rows are
    // written, so calc_carbon_offset is 0 in every year and the size column, derived from it (:1353-1366), is 0 as well.
    // Coordinates are thread_rng draws there (actions.rs:142-144); here a Philox stream keyed by the offset's position.
    std::FILE* f = std::fopen((dir + "/yearly_details/carbon_offsets.csv").c_str(), "w");
    if (!f) return eg_fail(EG_ERR_IO, "cannot write carbon_offsets.csv in " + dir);
    std::fprintf(f, "Year,Offset ID,Type,X,Y,Size,Capture Efficiency (%%),Power Consumption (MW),CO2 Offset (tonnes),Negative CO2 Emissions (tonnes),"
                    "Cost (\xE2\x82\xAC),Operating Cost (\xE2\x82\xAC),Total Annual Cost (\xE2\x82\xAC),Cost Per Tonne (\xE2\x82\xAC)\n");
    static const double kOffOperating[EG_N_OFFSET_TYPES] = {10000.0, 15000.0, 100000.0, 5000.0};
    static const double kOffOpTrend[EG_N_OFFSET_TYPES] = {1.0, 1.01, 0.97, 1.02};
    struct Offset { std::string id; int type, year, mult; double x, y; };
    std::vector<Offset> offs;
    for (int y = 0; y < EG_NY; y++)
      for (int i = traj.n_deficit[y]; i < traj.n_deficit[y] + traj.n_additional[y]; i++) {
        const int a = traj.actions[row[y] + i];
        if (a < 45 || a >= 57) continue;
        const int o = (a - 45) / 3, year = EG_BASE_YEAR + y;
        Offset r{std::string("Offset_") + kOffsetNames[o] + "_" + std::to_string(year) + "_" + std::to_string(offs.size()), o, year, (a - 45) % 3, 0, 0};
        r.x = csv_uniform((uint32_t)offs.size(), 0) * 50000.0;
        r.y = csv_uniform((uint32_t)offs.size(), 1) * 50000.0;
        offs.push_back(r);
      }
    for (int y = 0; y < EG_NY; y++) {
      const int year = EG_BASE_YEAR + y;
      for (const Offset& r : offs) {
        if (year < r.year) continue;
        const double lon = -10.6 + ((-5.9 - -10.6) * (r.x / 50000.0)), lat = 51.4 + ((55.4 - 51.4) * (r.y / 50000.0));
        const double cost = (T.off_base_cost[r.type] * powi(1.0 + 0.0185, y)) * T.mult[r.mult];                       // carbon_offset.rs:188-195
        const double operating = kOffOperating[r.type] * T.year[y].inflation * std::pow(kOffOpTrend[r.type], (double)y);  // :197-209
        std::fprintf(f, "%d,%s,%s,%.6f,%.6f,0,%.2f,%s,0.00,-0.00,%.2f,%.2f,%.2f,0.00\n", year, r.id.c_str(), kOffsetNames[r.type], lon, lat,
                     0.85 * 100.0, r.type == 2 ? "50" : "0", cost, operating, cost + operating);
      }
    }
    std::fclose(f);
  }
  {  // operation_logs/generator_operation_logs.csv, csv_export.rs:1096-1310: the year loop there runs over
     // commissioning_year..=min(eol, 2050) with eol a lifespan (25..60 years), an empty range, so only the header is written
    if (!mkdir_p(dir + "/operation_logs")) return eg_fail(EG_ERR_IO, "cannot create " + dir + "/operation_logs");
    std::FILE* f = std::fopen((dir + "/operation_logs/generator_operation_logs.csv").c_str(), "w");
    if (!f) return eg_fail(EG_ERR_IO, "cannot write generator_operation_logs.csv in " + dir);
    std::fprintf(f, "Year,Month,Day,Hour,Generator ID,Type,Power Output (MW),Operation %%,Actual Output (MW),Weather Factor,CO2 Emissions (tonnes)\n");
    std::fclose(f);
  }
  if (written_dir) std::snprintf(written_dir, 512, "%s", dir.c_str());
  return EG_OK;
}

int eg_write_location_analysis(const std::vector<double>& scores, int half, double step, double min_suitability, const char* cache_dir,
                               const char* text_path) {
  const int side = 2 * half + 1;
  struct Loc { double x, y; std::vector<int> types; };
  std::vector<Loc> locations;
  size_t type_counts[EG_NT] = {0};
  std::vector<size_t> type_to_locations[EG_NT];
  size_t multi = 0;
  auto clamp_map = [](double v) { return std::min(std::max(v, 0.0), 50000.0); };  // Coordinate::new, data/poi.rs:11-15
  for (int i = -half; i <= half; i++)
    for (int j = -half; j <= half; j++) {
      const double* sc = &scores[((size_t)(i + half) * side + (size_t)(j + half)) * EG_NT];
      Loc loc{clamp_map((double)i * step), clamp_map((double)j * step), {}};
      for (int t = 0; t < EG_NT; t++)
        if (sc[t] >= min_suitability) {
          loc.types.push_back(t);
          type_counts[t]++;
          type_to_locations[t].push_back(locations.size());
        }
      if (!loc.types.empty()) {
        if (loc.types.size() > 1) multi++;
        locations.push_back(loc);
      }
    }
  // scores of a stored location, by its position in the scan
  auto score_of = [&](const Loc& l, int t) {
    // locations keep their coordinates only; find the scan cell again through the coordinate (first cell with it: the
    // clamped duplicates share their scores)
    const int i = (int)(l.x / step), j = (int)(l.y / step);
    return scores[((size_t)(i + half) * side + (size_t)(j + half)) * EG_NT + t];
  };
  if (cache_dir) {
    if (!mkdir_p(cache_dir)) return eg_fail(EG_ERR_IO, std::string("cannot create ") + cache_dir);
    // serde_json::to_string_pretty(LocationAnalysis): fields in declaration order; the HashMaps (unordered in the
    // reference) are written in generator-type order
    std::string o = "{\n  \"locations\": [";
    for (size_t k = 0; k < locations.size(); k++) {
      const Loc& l = locations[k];
      o += k ? ",\n    {\n" : "\n    {\n";
      o += "      \"coordinate\": {\n        \"x\": " + egjson::fmt_double(l.x) + ",\n        \"y\": " + egjson::fmt_double(l.y) + "\n      },\n";
      o += "      \"suitability_scores\": {";
      for (size_t q = 0; q < l.types.size(); q++)
        o += std::string(q ? ",\n" : "\n") + "        \"" + kGenNames[l.types[q]] + "\": " + egjson::fmt_double(score_of(l, l.types[q]));
      o += "\n      }\n    }";
    }
    o += locations.empty() ? "],\n" : "\n  ],\n";
    auto count_map = [&](const char* name) {
      o += std::string("  \"") + name + "\": {";
      bool first = true;
      for (int t = 0; t < EG_NT; t++)
        if (type_counts[t]) {
          o += std::string(first ? "\n" : ",\n") + "    \"" + kGenNames[t] + "\": " + std::to_string(type_counts[t]);
          first = false;
        }
      o += first ? "},\n" : "\n  },\n";
    };
    count_map("type_counts");
    o += "  \"multi_type_locations\": [";
    bool first_multi = true;
    for (const Loc& l : locations) {
      if (l.types.size() < 2) continue;
      o += first_multi ? "\n    [\n" : ",\n    [\n";
      first_multi = false;
      o += "      {\n        \"x\": " + egjson::fmt_double(l.x) + ",\n        \"y\": " + egjson::fmt_double(l.y) + "\n      },\n      [";
      for (size_t q = 0; q < l.types.size(); q++) o += std::string(q ? ",\n" : "\n") + "        \"" + kGenNames[l.types[q]] + "\"";
      o += "\n      ]\n    ]";
    }
    o += first_multi ? "],\n" : "\n  ],\n";
    count_map("remaining_spaces");
    o += "  \"exhausted_types\": [],\n  \"type_to_locations\": {";
    bool first_type = true;
    for (int t = 0; t < EG_NT; t++) {
      if (type_to_locations[t].empty()) continue;
      o += std::string(first_type ? "\n" : ",\n") + "    \"" + kGenNames[t] + "\": [";
      first_type = false;
      for (size_t q = 0; q < type_to_locations[t].size(); q++) o += std::string(q ? ",\n" : "\n") + "      " + std::to_string(type_to_locations[t][q]);
      o += "\n    ]";
    }
    o += first_type ? "}\n}" : "\n  }\n}";
    const std::string path = std::string(cache_dir) + "/location_analysis.json";
    FILE* f = std::fopen(path.c_str(), "wb");
    if (!f || std::fwrite(o.data(), 1, o.size(), f) != o.size()) { if (f) std::fclose(f); return eg_fail(EG_ERR_IO, "cannot write " + path); }
    std::fclose(f);
  }
  if (text_path) {
    std::string o = "Location Analysis Results\n========================\n\n";
    o += "Total suitable locations: " + std::to_string(locations.size()) + "\nMulti-type locations: " + std::to_string(multi) + "\n\n";
    o += "Locations by Generator Type:\n--------------------------\n";
    for (int t = 0; t < EG_NT; t++)
      if (type_counts[t]) o += std::string(kGenNames[t]) + ": " + std::to_string(type_counts[t]) + "\n";
    o += "\nDetailed Location Data:\n---------------------\n";
    for (const Loc& l : locations) {
      o += "\nCoordinate: (" + rust_display(l.x) + ", " + rust_display(l.y) + ")\n";
      for (int t : l.types) o += std::string("  ") + kGenNames[t] + ": " + fixed(score_of(l, t), 3) + "\n";
    }
    FILE* f = std::fopen(text_path, "wb");
    if (!f || std::fwrite(o.data(), 1, o.size(), f) != o.size()) { if (f) std::fclose(f); return eg_fail(EG_ERR_IO, std::string("cannot write ") + text_path); }
    std::fclose(f);
  }
  return EG_OK;
}
