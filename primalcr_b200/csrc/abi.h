// abi.h -- error reporting of the C ABI (include/primalcr.h), shared by engine.cu and queries.cu.
// An entry point runs its body between API_BEGIN and API_END: a pcr::Error returns its code, any other exception
// PRIMALCR_EINTERNAL, and the message stays readable through primalcr_last_error() on the calling thread.
#pragma once
#include "common.cuh"
#include "../../include/primalcr.h"

namespace pcr {
extern thread_local std::string g_last_error;     // defined in engine.cu
}

#define API_BEGIN try {
#define API_END                                                                  \
    } catch (const pcr::Error &e) { pcr::g_last_error = e.what(); return e.code; } \
    catch (const std::exception &e) { pcr::g_last_error = e.what(); return PRIMALCR_EINTERNAL; } \
    return PRIMALCR_OK;
