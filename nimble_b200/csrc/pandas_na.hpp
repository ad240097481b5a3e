// What pandas.read_csv turns into NaN by default (check_df_from_input, nimble/__main__.py:219).  One list for the two
// routes to the counts TSV: `report` drops rows whose field is one of these (report.cpp), `align --counts` drops the
// same rows before they reach the UMI stage (stream.cpp: barcodes, engine.cu: single-feature rows).
// frontend._PANDAS_NA is the Python copy.
#pragma once
#include <string_view>

namespace nb200 {

inline bool pandas_na(std::string_view v) {
    static const char *na[] = {"", "#N/A", "#N/A N/A", "#NA", "-1.#IND", "-1.#QNAN", "-NaN", "-nan", "1.#IND", "1.#QNAN", "<NA>",
                               "N/A", "NA", "NULL", "NaN", "None", "n/a", "nan", "null"};
    for (const char *s : na) if (v == s) return true;
    return false;
}

}  // namespace nb200
