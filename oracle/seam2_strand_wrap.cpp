/* oracle/seam2_strand_wrap.cpp — TEST INFRASTRUCTURE ONLY.
 *
 * Linked (oracle/seam2_strand.mk) into _ref/seam2_cluster_driver_strand_{ref,gpu}: the unchanged
 * oracle/seam2_cluster_driver.cpp plus this file, with the driver's call of cluster_session_init redirected here by
 * -Wl,--wrap.  SEAM2_STRAND=both|plus sets Parameters::opt_strand (--strand) before the session is initialised, so that
 * tests/test_cluster_strand_gpu.py can compare the reference's clustering session with shim/cluster_session_vsg.cpp on
 * both strands.  Everything else the driver does (its keys, masking, sorting, output) is untouched.
 */
#include "vsearch_api.h"
#include "core/cluster.hpp"

#include <cstdlib>
#include <cstring>

extern "C" void __real__Z20cluster_session_initP17cluster_session_sRK10ParametersR7DbindexRK8Database(
    cluster_session_s * cs, Parameters const & parameters, Dbindex & dbindex, Database const & db);

extern "C" void __wrap__Z20cluster_session_initP17cluster_session_sRK10ParametersR7DbindexRK8Database(
    cluster_session_s * cs, Parameters const & parameters, Dbindex & dbindex, Database const & db)
{
  char const * const s = std::getenv("SEAM2_STRAND");
  if (s != nullptr) {
    // the driver's Parameters is a non-const local of its main(): writing through the reference is well defined
    const_cast<Parameters &>(parameters).opt_strand = std::strcmp(s, "both") == 0;
  }
  __real__Z20cluster_session_initP17cluster_session_sRK10ParametersR7DbindexRK8Database(cs, parameters, dbindex, db);
}
