// host_tables.hpp — host-side map (as loaded), the small host-built tables, and the output files written from them.
#pragma once
#include <cstdint>
#include <string>
#include <vector>
#include "tables.h"

struct EgHostMap {
  std::vector<double> sx, sy;      // settlements, grid metres
  std::vector<uint32_t> spop;      // 2025 population
  std::vector<std::string> sname;  // settlement names (CSV export only; empty for maps set through eg_map_set)
  std::vector<double> ex, ey, ecap;  // plants existing before the simulation
  std::vector<uint8_t> etype;
  std::vector<double> cx, cy;      // coastline polygon
  int grid_n = 0;
  double step = 0;
};

struct EgHostTables {
  EgSmallTables small;
  std::vector<double> plant_terms;   // [EG_OPC_SIZE][2]
  std::vector<uint32_t> pop;         // [26][S]
  std::vector<double> near_factor;   // [6][r2_stride], by squared cell distance
  int r2_limit[2 * EG_N_RCLASS + 1] = {0};  // limits, compact-table offsets, compact-table size
  int r2_stride = 0;
  int kmax = 0;
  int near_geom = 0;                 // EgDeviceMap::near_geom (0 compact, 1 medium, 2 general)
  std::vector<int> ex_online_year;   // first year in which each pre-existing plant is Operational (quirk Q1); 0 = never
};

int eg_host_map_load(EgHostMap* m, const char* settlements_json, const char* generators_csv, const char* coastline_json);
int eg_host_map_set(EgHostMap* m, const eg_map_desc* d);
int eg_host_map_validate(const EgHostMap& m);
void eg_host_build_tables(const EgHostMap& m, EgHostTables* out);
// planning_duration / construction_duration of config/tech_type.rs:70-200 for a generator type registered in `year`
void eg_host_tech_durations(int type, int year, double* planning, double* construction);

// report_files.cpp: the six CSV files of the best run under <output_dir>/<timestamp>/ from its record `traj` and replay (the
// directory goes to `written_dir`, 512 bytes, unless NULL), and location_analysis.json in `cache_dir` and the text report at
// `text_path` (either may be NULL) from the scores [(2 half + 1)^2][EG_NT] of analyze_map's grid
int eg_write_best_run_csv(const char* output_dir, const eg_weights* w, const EgHostMap& hmap, const EgHostTables& htab, const eg_traj& traj,
                          const eg_result& res, const eg_yearly& yearly, const eg_sites& sites, char* written_dir);
int eg_write_location_analysis(const std::vector<double>& scores, int half, double step, double min_suitability, const char* cache_dir,
                               const char* text_path);
