// Host shim over eraytracer_b200/csrc/scene_tables.cpp: the library's own camera matrix and rotation check, for the
// CPU tests of ERT_FLAG_CAMERA_ROTATION (tests/test_camera_rotation_host.py).
#include "../../eraytracer_b200/csrc/scene_tables.h"

#include <cstring>

extern "C" {

int cr_camera_matrix(const double *rot3, double *m9) { return ert::camera_matrix(rot3, m9) ? 1 : 0; }

// the message of a non-finite rotation, or "" for a finite one
const char *cr_check_rotation(const double *rot3)
{
    static std::string msg;
    ert_camera c{};
    std::memcpy(c.rotation, rot3, sizeof c.rotation);
    c.fov = 90; c.screen_width = 4; c.screen_height = 3;
    msg = ert::check_camera_rotation(c);
    return msg.c_str();
}

}
