// formats_probe.cpp -- prints the format table of csrc/rip_formats.h for tests/test_formats.py: for every code from -1 to 64
// either "none <code>" or the row, followed by the acceptance and bytes per frame of each shape of a fixed grid.
//   row <code> <name> <layout> <channels> <bgr> <pattern> <bits> <packing> <decodes> <num> <den> <w_mul> <h_mul> <w_min> <h_min>
//   shape <code> <W> <H> <accepted> <bytes>
#include <cstdio>

#include "rip_formats.h"

int main()
{
    const int widths[] = {1, 2, 3, 4, 5, 6, 7, 8, 9, 16, 17, 684, 4096}, heights[] = {1, 2, 3, 4, 5, 1023};
    for (int code = -1; code <= 64; code++) {
        const rip::Format *f = rip::format_of(code);
        if (!f) {
            printf("none %d\n", code);
            continue;
        }
        printf("row %d %s %d %d %d %d %d %d %d %d %d %d %d %d %d\n", f->code, f->name, (int)f->layout, f->channels, (int)f->bgr,
               f->pattern, f->bits, (int)f->packing, (int)rip::decodes_to_color(code), f->bytes_num, f->bytes_den, f->w_mul,
               f->h_mul, f->w_min, f->h_min);
        for (int W : widths)
            for (int H : heights)
                printf("shape %d %d %d %d %zu\n", code, W, H, (int)rip::shape_ok(*f, W, H), rip::frame_bytes(*f, W, H));
    }
    return 0;
}
