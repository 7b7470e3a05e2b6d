// The message cls_last_error returns: every failing call of the C ABI records it for the calling thread (capi.cpp).
#pragma once
#include <string>

namespace cls {
int set_last_error(int code, const std::string &msg);   // returns `code`
}
